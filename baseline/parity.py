"""CHECKER ONLY -- token-id parity of this repo's CUDA engine against the UNMODIFIED reference on the SAME GPU.

The north star asks for greedy ids "bit-exact" against the reference.  Both sides run bf16 on the B200 with the SAME
weight tensors (the reference model's parameters are re-pointed at the HF model's storage): the reference through its
own ``jacobi_greedy_search_multilevel`` (``lade/decoding.py:697-1259``), ours through ``LookaheadEngine.generate``.

What can and cannot be exact: random-init bf16 logits tie to within 0-3 bf16 ulps at a few positions of every run
(SURVEY.md App. D.8), and the two sides cannot round identically everywhere -- the reference's ids themselves change
with the cuBLAS kernel its GEMM shape selects (its lookahead run and its own plain-greedy run already differ at such
positions).  So the check is:

  * compare ids position by position;
  * at a divergence, compute the reference model's OWN next-token logits on the common prefix (its plain causal
    forward, ``LlamaModeljforward(is_prefill=True)``, ``modeling_llama.py:1108``) and record the margin between the two
    candidates and the top logit, in ulps of the model dtype (bf16, or fp16 for fp16 models) at the top logit;
  * force the reference's token (re-run ours from ``ref[:i+1]``) and continue, so EVERY position of the run is
    compared, not only the prefix up to the first near-tie.

``report["exact"]`` is True when no position diverged; ``report["ok"]`` when every divergence is a near-tie
(both candidates within ``tol_ulps`` of the reference's top logit).

The reference is not part of this repository, so the GPU tests judge against records of its runs on a B200
(``record_reference`` / ``compare_ids_to_record``, written by ``tests/golden/gen_golden_gpu_parity.py``).
"""
from __future__ import annotations

import contextlib
import hashlib
import io
import random
from typing import Callable, List, Optional, Sequence

import torch

from . import ref_loader as R


def reference_model_sharing_weights(hf_model, shape: dict):
    """Reference ``LlamaForCausalLM`` (unmodified class) whose parameters ARE the HF model's tensors (no copy)."""
    from transformers import GenerationConfig

    _, modeling = R.load_reference()
    dev = next(hf_model.parameters()).device
    cfg = R.make_llama_config(hidden=shape["hidden"], layers=shape["layers"], heads=shape["heads"],
                              kv_heads=shape.get("kv_heads") or shape["heads"], inter=shape["inter"], vocab=shape["vocab"],
                              max_pos=shape.get("max_pos", 2048), rope_theta=shape.get("rope_theta", 10000.0),
                              eps=shape.get("eps", 1e-5))
    old_dtype = torch.get_default_dtype()
    torch.set_default_dtype(next(hf_model.parameters()).dtype)
    try:
        with torch.device("meta"):
            ref = modeling.LlamaForCausalLM(cfg)
        ref = ref.to_empty(device=dev)
        src = dict(hf_model.named_parameters())
        with torch.no_grad():
            for name, p in ref.named_parameters():
                if name not in src:
                    raise RuntimeError(f"reference parameter {name} has no HF counterpart")
                p.data = src[name].data                      # shared storage (views of the fused q/k/v stay valid)
        # buffers were left uninitialised by to_empty(): rebuild the rotary tables the way __init__ does
        # (fp32 math, cached in the default dtype; modeling_llama.py:240-256)
        for mod in ref.modules():
            if hasattr(mod, "_set_cos_sin_cache") and hasattr(mod, "inv_freq"):
                with torch.device(dev):
                    inv = 1.0 / (mod.base ** (torch.arange(0, mod.dim, 2, device=dev).float() / mod.dim))
                mod.register_buffer("inv_freq", inv, persistent=False)
                mod._set_cos_sin_cache(seq_len=mod.max_position_embeddings, device=dev, dtype=torch.get_default_dtype())
    finally:
        torch.set_default_dtype(old_dtype)
    ref.eval()
    ref.generation_config = GenerationConfig(pad_token_id=0, eos_token_id=None)
    return ref


@contextlib.contextmanager
def _reference_device(dev, dtype=torch.bfloat16):
    """The reference's mask builder creates small CPU tensors (``modeling_llama.py:143-181``); a default device makes
    them land on the GPU.  The default dtype follows the model (bf16 on the GPU configs)."""
    old_dtype = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    torch.set_default_device(dev)
    try:
        yield
    finally:
        torch.set_default_dtype(old_dtype)
        torch.set_default_device("cpu")


def reference_greedy(ref_model, prompt: Sequence[int], max_new: int, W: int, N: int, G: int, py_seed: int = 0,
                     eos_token_id=None, pool_from_prompt: bool = False):
    """The reference's own greedy lookahead loop on the model's device.  Returns (ids list, n_steps)."""
    from transformers import MaxLengthCriteria, StoppingCriteriaList

    decoding, _ = R.load_reference()
    dev = next(ref_model.parameters()).device
    P = len(prompt)
    decoding.CONFIG_MAP.clear()
    decoding.CONFIG_MAP.update(dict(WINDOW_SIZE=W, LEVEL=N, GUESS_SET_SIZE=G, DEBUG=1, log=[],
                                    POOL_FROM_PROMPT=int(pool_from_prompt)))
    random.seed(py_seed)
    with _reference_device(dev, next(ref_model.parameters()).dtype), torch.no_grad(), \
            contextlib.redirect_stdout(io.StringIO()):
        ids = torch.tensor([list(prompt)], dtype=torch.long, device=dev)
        out = decoding.jacobi_greedy_search_multilevel(
            ref_model, ids, stopping_criteria=StoppingCriteriaList([MaxLengthCriteria(P + max_new)]),
            attention_mask=torch.ones_like(ids), use_cache=True, return_dict_in_generate=False,
            output_attentions=False, output_hidden_states=False, output_scores=False, pad_token_id=0,
            eos_token_id=eos_token_id)
    steps = decoding.CONFIG_MAP["log"][-1][1] if decoding.CONFIG_MAP.get("log") else None
    return out[0].tolist(), steps


def reference_next_logits(ref_model, prefix: Sequence[int]) -> torch.Tensor:
    """Next-token logits of the reference model after `prefix` (its plain causal forward), fp32 [V]."""
    dev = next(ref_model.parameters()).device
    with _reference_device(dev, next(ref_model.parameters()).dtype), torch.no_grad():
        x = torch.tensor([list(prefix)], dtype=torch.long, device=dev)
        out = ref_model.model.LlamaModeljforward(input_ids=x, is_prefill=True, level_sizes=[x.size(1) - 1], guess=None,
                                                 use_cache=False)
        h = out[0] if isinstance(out, tuple) else out.last_hidden_state
        return ref_model.lm_head(h[:, -1:, :])[0, 0].float()


def reference_self_consistency(ref_model, ref_ids: Sequence[int], n_prompt: int) -> dict:
    """The noise floor of the comparison: the reference's lookahead ids judged by the reference model's OWN plain causal
    forward over the same sequence (one teacher-forced pass, same GPU, same weights).  A position where the causal
    argmax differs from the token the reference's lookahead run emitted is a position where the reference disagrees
    with itself (its step forward of q rows and its plain forward round differently); the distance of the emitted
    token below the causal top logit, in bf16 ulps, says how wide "a tie" is on this model."""
    dev = next(ref_model.parameters()).device
    ref_ids = list(ref_ids)
    with _reference_device(dev, next(ref_model.parameters()).dtype), torch.no_grad():
        x = torch.tensor([ref_ids[:-1]], dtype=torch.long, device=dev)
        out = ref_model.model.LlamaModeljforward(input_ids=x, is_prefill=True, level_sizes=[x.size(1) - 1], guess=None,
                                                 use_cache=False)
        h = out[0] if isinstance(out, tuple) else out.last_hidden_state
        logits = ref_model.lm_head(h[0, n_prompt - 1:, :]).float()           # row i predicts token n_prompt + i
    want = torch.tensor(ref_ids[n_prompt:], device=logits.device)
    top2 = torch.topk(logits, 2, dim=-1).values
    top = top2[:, 0]
    ulp = torch.pow(2.0, torch.floor(torch.log2(top.abs().clamp_min(1e-30))) - _mant_bits(ref_model))
    chosen = logits.gather(1, want[:, None])[:, 0]
    below = (top - chosen) / ulp
    margin = (top2[:, 0] - top2[:, 1]) / ulp
    mism = below > 0
    return {"positions": int(want.numel()), "n_self_mismatch": int(mism.sum()), "worst_below_top_ulps": round(float(below.max()), 2),
            "median_top2_margin_ulps": round(float(margin.median()), 2),
            "positions_with_top2_margin_le_3_ulps": int((margin <= 3).sum()),
            "how": "reference lookahead ids vs the reference model's own teacher-forced causal forward (argmax per position)"}


def weights_digest(model) -> str:
    """sha256 over the parameter names and bytes: a record of the reference holds only for the weights it ran on."""
    h = hashlib.sha256()
    for name, p in sorted(model.named_parameters()):
        h.update(name.encode())
        h.update(p.detach().contiguous().view(torch.uint8).cpu().numpy().tobytes())
    return h.hexdigest()


def _mant_bits(model) -> int:
    """Explicit mantissa bits of the model dtype: the unit in which a logit 'tie' is measured (bf16 7, fp16 10)."""
    return {torch.bfloat16: 7, torch.float16: 10}.get(next(model.parameters()).dtype, 23)


def _bf16_ulp(x: float, mant_bits: int = 7) -> float:
    """ulp of the model dtype at |x| (bf16 by default; the name is kept for the callers of round 2's first version)."""
    import math
    ax = abs(float(x))
    if ax == 0.0:
        return 2.0 ** -133
    return 2.0 ** (math.floor(math.log2(ax)) - mant_bits)


def compare_ids(our_generate: Callable[[List[int], int], List[int]], ref_ids: Sequence[int], n_prompt: int,
                ref_model, tol_ulps: float = 3.0, max_divergences: int = 64, self_check: bool = True) -> dict:
    """Position-by-position comparison with forcing (see the module docstring).

    our_generate(prompt_ids, max_new) -> prompt + generated ids of THIS repo's engine.
    The tolerance is max(tol_ulps, the reference's own self-inconsistency on this run): a divergence no wider than
    the distance at which the reference disagrees with itself cannot be told apart from a tie."""
    ref_ids = list(ref_ids)
    self_rep = reference_self_consistency(ref_model, ref_ids, n_prompt) if self_check and len(ref_ids) - n_prompt >= 1 else None
    return _compare_on_logits(our_generate, ref_ids, n_prompt, lambda prefix: reference_next_logits(ref_model, prefix),
                              _mant_bits(ref_model), self_rep, tol_ulps, max_divergences)


def record_reference(ref_model, ref_ids: Sequence[int], n_prompt: int, top_k: int = 32) -> dict:
    """What compare_ids reads from the reference model, recorded so that the comparison can run without it: the ids,
    the self-consistency report, the mantissa bits of the model dtype and, at every generated position i, the top
    `top_k` of reference_next_logits(ref_ids[:i]) (values are model-dtype numbers, exact in fp32)."""
    ref_ids = list(ref_ids)
    top_idx, top_val = [], []
    for i in range(n_prompt, len(ref_ids)):
        t = torch.topk(reference_next_logits(ref_model, ref_ids[:i]), top_k)
        top_idx.append(t.indices.tolist())
        top_val.append(t.values.tolist())
    return {"ids": ref_ids, "n_prompt": n_prompt, "mant_bits": _mant_bits(ref_model),
            "self_consistency": reference_self_consistency(ref_model, ref_ids, n_prompt), "top_idx": top_idx,
            "top_val": top_val}


def compare_ids_to_record(our_generate: Callable[[List[int], int], List[int]], rec: dict, vocab: int,
                          tol_ulps: float = 3.0, max_divergences: int = 64) -> dict:
    """compare_ids against a record_reference() record.  A token outside the recorded top-k gets -inf as its logit:
    a divergence to it is never taken for a tie."""
    ref_ids, n_prompt = list(rec["ids"]), rec["n_prompt"]

    def next_logits(prefix):
        i = len(prefix)
        assert list(prefix) == ref_ids[:i] and n_prompt <= i < len(ref_ids), "not a recorded prefix"
        logits = torch.full((vocab,), -float("inf"))
        logits[torch.tensor(rec["top_idx"][i - n_prompt])] = torch.tensor(rec["top_val"][i - n_prompt])
        return logits
    return _compare_on_logits(our_generate, ref_ids, n_prompt, next_logits, rec["mant_bits"], rec["self_consistency"],
                              tol_ulps, max_divergences)


def _compare_on_logits(our_generate, ref_ids: List[int], n_prompt: int, next_logits: Callable[[List[int]], torch.Tensor],
                       mant_bits: int, self_rep: Optional[dict], tol_ulps: float, max_divergences: int) -> dict:
    """The loop of compare_ids; next_logits(prefix) -> the reference model's fp32 [V] logits after that prefix."""
    total = len(ref_ids)
    if self_rep is not None:
        tol_ulps = max(tol_ulps, self_rep["worst_below_top_ulps"])
    ours = list(our_generate(ref_ids[:n_prompt], total - n_prompt))
    start = n_prompt
    divergences = []
    while True:
        n = min(len(ours), total)
        i = next((k for k in range(start, n) if ours[k] != ref_ids[k]), None)
        if i is None:
            length_ok = len(ours) == total
            break
        logits = next_logits(ref_ids[:i])
        top = logits.max().item()
        ulp = _bf16_ulp(top, mant_bits)
        la, lb = logits[ours[i]].item(), logits[ref_ids[i]].item()
        srt = torch.topk(logits, 2).values
        divergences.append({"index": i - n_prompt, "ours": int(ours[i]), "ref": int(ref_ids[i]),
                            "ours_below_top_ulps": round((top - la) / ulp, 2), "ref_below_top_ulps": round((top - lb) / ulp, 2),
                            "ref_top2_margin_ulps": round((srt[0] - srt[1]).item() / ulp, 2)})
        if len(divergences) >= max_divergences or i + 1 >= total:
            length_ok = True
            break
        forced = ref_ids[: i + 1]
        ours = forced + list(our_generate(forced, total - (i + 1)))[i + 1:]
        start = i + 1
    worst = max([max(d["ours_below_top_ulps"], d["ref_below_top_ulps"]) for d in divergences], default=0.0)
    return {
        "compared_tokens": total - n_prompt,
        "exact": not divergences and length_ok,
        "exact_prefix_tokens": (divergences[0]["index"] if divergences else total - n_prompt),
        "n_divergences": len(divergences),
        "worst_candidate_below_top_ulps": worst,
        "tol_ulps": tol_ulps,
        "reference_self_consistency": self_rep,
        "ok": length_ok and worst <= tol_ulps and len(divergences) < max_divergences,
        "divergences": divergences[:8],
        "how": "ours vs the unmodified reference's jacobi_greedy_search_multilevel on the same GPU and weights; every "
               "divergence is judged on the reference model's own next-token logits, then the reference's token is "
               "forced and the comparison continues",
    }
