"""GPU token-id parity: this repo's engine against the UNMODIFIED reference run on a B200 with the same weight tensors.
The reference is not part of the repository: its runs are recorded in tests/golden/reference_gpu_parity.json.gz
(tests/golden/gen_golden_gpu_parity.py; ids, self-consistency and the top-32 next-token logits at every position,
baseline/parity.py) together with a digest of the weights they ran on.

BASELINE.json config 1 (tiny random-init Llama, W5 N3 G3 -- with head_dim 128 so the production kernel runs), the
7B-config lookahead shape W15 N5 G15 on the tiny model, and the edge shapes of tests/golden/greedy_edge_traces.json.gz
(1-token prompt, prompt shorter than N, 1 and 2 new tokens, W=1, G=1, N=3 under a wide window, EOS on the first token)
through the ENGINE (the state-machine replay of those traces is in test_gpu_state_machine.py).

Pass criterion: ids identical, or every divergence is a near-tie on the reference model's own logits (<= 3 bf16 ulps
below its top logit for both candidates); every position is compared (the reference's token is forced after a
divergence).  The report is printed (run with -s) and the exact cases are asserted exact."""
import functools
import gzip
import json
import os
import random

import pytest
import torch

from baseline import parity as PAR

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_gpu_parity.json.gz")

TINY = dict(hidden=256, layers=2, heads=2, kv_heads=2, inter=688, vocab=32000, max_pos=2048, rope_theta=10000.0, eps=1e-5)
GQA = dict(hidden=512, layers=2, heads=4, kv_heads=2, inter=688, vocab=4096, max_pos=2048, rope_theta=10000.0, eps=1e-5)
# head_dim 64 with grouped KV heads: the TinyLlama-1.1B layout (2048 / 32 heads, 4 KV heads) in miniature
D64 = dict(hidden=256, layers=2, heads=4, kv_heads=2, inter=688, vocab=4096, max_pos=2048, rope_theta=10000.0, eps=1e-5)

#        name                 shape  W   N  G   P  new pool
CASES = [("cfg1_w5n3g3",       TINY, 5,  3, 3,  64, 96, False),
         ("cfg1_w5n3g3_pool",  TINY, 5,  3, 3,  64, 96, True),
         ("w15n5g15",          TINY, 15, 5, 15, 64, 128, False),
         ("w15n5g15_pool",     TINY, 15, 5, 15, 64, 128, True),
         ("w20n7g20_pool",     TINY, 20, 7, 20, 96, 96, True),
         ("gqa_w15n5g15",      GQA,  15, 5, 15, 48, 96, False),
         ("d64_gqa_w15n5g15",  D64,  15, 5, 15, 48, 96, True),
         # a summarisation-length prompt: 21 query tiles of prefill attention, kv past 2.5 k in the decode steps
         ("long_prompt_2600",  dict(TINY, max_pos=4096), 15, 5, 15, 2600, 48, True),
         # edge shapes (tests/golden/gen_golden_edge.py)
         ("edge_p1",           TINY, 5,  3, 3,  1,  24, True),
         ("edge_p2_lt_n",      TINY, 7,  5, 7,  2,  24, True),
         ("edge_new1",         TINY, 5,  3, 3,  12, 1,  False),
         ("edge_new2",         TINY, 5,  3, 3,  12, 2,  True),
         ("edge_w1g1",         TINY, 1,  3, 1,  16, 24, True),
         ("edge_w2n4g1",       TINY, 2,  4, 1,  16, 32, True),
         ("edge_g1_w15n5",     TINY, 15, 5, 1,  32, 48, True),
         ("edge_n3_w20g20",    TINY, 20, 3, 20, 24, 48, True)]
FP16_CASES = ("cfg1_w5n3g3_pool", "w15n5g15", "gqa_w15n5g15", "d64_gqa_w15n5g15", "edge_p1")


@functools.lru_cache(maxsize=None)
def _records():
    with gzip.open(GOLDEN, "rt") as f:
        return json.load(f)["records"]


def build_recorded(key, shape, dtype=torch.bfloat16):
    """The HF model (bench.build_model, seed 0) and the record of the reference's run on those weights."""
    from bench import build_model
    hf = build_model(shape, torch.device("cuda"), seed=0)
    if dtype != torch.bfloat16:
        hf = hf.to(dtype)
    rec = _records()[key]
    assert PAR.weights_digest(hf) == rec["weights_sha256"], f"{key}: not the weights the reference was recorded on"
    return hf, rec


def engine_generate(hf, W, N, G, pool, cap, eos=(), **engine_kw):
    from lookaheaddecoding_b200 import LookaheadEngine
    eng = LookaheadEngine(hf, W, N, G, pool_from_prompt=pool, max_total_len=cap, **engine_kw)

    def gen(prompt, n_new):
        return eng.generate(prompt, n_new, eos_token_ids=eos, rng=random.Random(7))
    return eng, gen


@pytest.mark.parametrize("name,shape,W,N,G,P,new,pool", CASES, ids=[c[0] for c in CASES])
def test_engine_ids_match_reference_on_the_same_gpu(name, shape, W, N, G, P, new, pool):
    hf, rec = build_recorded(name, shape)
    assert len(rec["ids"]) == P + new and rec["n_prompt"] == P
    eng, gen = engine_generate(hf, W, N, G, pool, P + new)
    rep = PAR.compare_ids_to_record(gen, rec, shape["vocab"])
    print(f"\n{name}: exact={rep['exact']} exact_prefix={rep['exact_prefix_tokens']}/{rep['compared_tokens']} "
          f"divergences={rep['n_divergences']} worst={rep['worst_candidate_below_top_ulps']} ulp "
          f"ref_steps={rec['steps']} {rep['divergences'][:3]}")
    assert rep["ok"], rep
    eng.close()


def test_eos_on_first_token_matches_reference():
    hf, rec = build_recorded("eos_first", TINY)
    ref_ids = rec["ids"]
    prompt, eos = ref_ids[:12], ref_ids[12]
    assert len(ref_ids) == 12 + 1          # the reference stopped on the EOS it emitted first
    eng, gen = engine_generate(hf, 5, 3, 3, True, 12 + 16, eos=[eos])
    ours = gen(prompt, 16)
    if ours != ref_ids:      # only a near-tie on the very first token may differ
        rep = PAR.compare_ids_to_record(gen, rec, 32000)
        assert rep["ok"], rep
    eng.close()


def test_window_fill_step_larger_than_steady_and_host_stopping_criteria():
    """G=0, W < N-2, short prompt: a window-fill step has more rows than the steady step (buffers are sized for it, no
    silent clamp); output == the reference model's plain greedy.  Then a custom StoppingCriteria through generate()."""
    import lade
    from transformers import StoppingCriteria, StoppingCriteriaList
    hf, rec = build_recorded("plain_greedy", TINY)
    prompt = rec["ids"][:10]
    assert len(rec["ids"]) == 10 + 24
    eng, gen = engine_generate(hf, 5, 8, 0, False, 10 + 24)
    assert eng.q_nonprefill > eng.q_steady
    rep = PAR.compare_ids_to_record(gen, rec, 32000)
    assert rep["ok"], rep
    eng.close()

    class StopAfter(StoppingCriteria):
        def __call__(self, input_ids, scores, **kw):
            return torch.full((input_ids.shape[0],), input_ids.shape[1] >= 10 + 7, dtype=torch.bool, device=input_ids.device)

    import os
    hf.generation_config.pad_token_id = 0
    hf.generation_config.eos_token_id = None
    os.environ["USE_LADE"] = "1"
    lade.augment_all()
    try:
        lade.config_lade(LEVEL=4, WINDOW_SIZE=5, GUESS_SET_SIZE=5, DEBUG=0)
        ids = torch.tensor([prompt], device="cuda")
        full = hf.generate(ids, attention_mask=torch.ones_like(ids), max_new_tokens=24, do_sample=False)
        cut = hf.generate(ids, attention_mask=torch.ones_like(ids), max_new_tokens=24, do_sample=False,
                          stopping_criteria=StoppingCriteriaList([StopAfter()]))
        assert full.shape[1] == 34
        assert 17 <= cut.shape[1] <= 17 + 2                      # stops at the first step boundary past 7 new tokens
        assert cut[0].tolist() == full[0, : cut.shape[1]].tolist()
    finally:
        lade.restore_generate()
        os.environ["USE_LADE"] = "0"


@pytest.mark.parametrize("name,shape,W,N,G,P,new,pool", [c for c in CASES if c[0] in FP16_CASES],
                         ids=lambda v: v if isinstance(v, str) else None)
def test_fp16_engine_ids_match_reference_on_the_same_gpu(name, shape, W, N, G, P, new, pool):
    """fp16 models (the dtype of the reference's README / minimal.py): the *_f16 kernels against the unmodified reference
    running in fp16 on the same GPU and weights; ties are measured in fp16 ulps."""
    hf, rec = build_recorded("fp16/" + name, shape, dtype=torch.float16)
    assert rec["mant_bits"] == 10 and len(rec["ids"]) == P + new
    prompt = rec["ids"][:P]
    eng, gen = engine_generate(hf, W, N, G, pool, P + new)
    assert eng.dt == torch.float16
    rep = PAR.compare_ids_to_record(gen, rec, shape["vocab"])
    print(f"\nfp16 {name}: exact={rep['exact']} exact_prefix={rep['exact_prefix_tokens']}/{rep['compared_tokens']} "
          f"divergences={rep['n_divergences']} worst={rep['worst_candidate_below_top_ulps']} ulp(fp16) ref_steps={rec['steps']}")
    assert rep["ok"], rep
    # sampling on the fp16 logits (device verification): reproducible, in range
    a = eng.generate(prompt, min(new, 24), rng=random.Random(1), sampling={"temperature": 0.8, "top_k": 40, "seed": 5})
    b = eng.generate(prompt, min(new, 24), rng=random.Random(1), sampling={"temperature": 0.8, "top_k": 40, "seed": 5})
    assert a == b and all(0 <= t < shape["vocab"] for t in a)
    eng.close()


@pytest.mark.parametrize("name,shape,W,N,G,P,new,pool", [c for c in CASES if c[0] in ("w15n5g15_pool", "gqa_w15n5g15", "w20n7g20_pool", "edge_p1")],
                         ids=["w15n5g15_pool", "w20n7g20_pool", "gqa_w15n5g15", "edge_p1"])
def test_reference_order_attention_engine_ids(name, shape, W, N, G, P, new, pool):
    """attn_impl=3: the attention variant that rounds the probabilities like the reference, through the whole engine."""
    hf, rec = build_recorded(name, shape)
    eng, gen = engine_generate(hf, W, N, G, pool, P + new, attn_impl=3)
    rep = PAR.compare_ids_to_record(gen, rec, shape["vocab"])
    print(f"\n{name} (attn_impl=3): exact={rep['exact']} divergences={rep['n_divergences']}")
    assert rep["ok"], rep
    eng.close()


def test_reference_order_attention_refuses_contexts_it_cannot_hold():
    """attn_impl=3 keeps every S tile of a split in tensor memory: more than 3072 rows of context (3 tiles x 8 splits)
    are refused when the engine is built, never silently downgraded."""
    from bench import build_model
    from lookaheaddecoding_b200 import LookaheadEngine
    hf = build_model(dict(TINY, max_pos=8192), torch.device("cuda"), seed=0)
    with pytest.raises(Exception, match="attn_impl=3"):
        LookaheadEngine(hf, 15, 5, 15, max_total_len=4096, attn_impl=3)
    with pytest.raises(Exception, match="attn_impl=3"):
        LookaheadEngine(hf, 15, 5, 15, max_total_len=1024, attn_impl=3, attn_splits=2)
    eng = LookaheadEngine(hf, 15, 5, 15, max_total_len=1024, attn_impl=3)
    assert eng.attn_splits >= 3 and eng.attn_kv_bound <= 384 * eng.attn_splits
    eng.close()
