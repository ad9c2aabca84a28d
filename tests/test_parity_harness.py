"""CPU checks of the GPU-vs-GPU parity harness (baseline/parity.py) itself: the unmodified reference is loaded with
shared weights, its lookahead ids equal its own plain greedy ids in fp32, and the comparison loop reports / judges
divergences the way bench.py's `parity` field relies on; the judgment on a recorded reference run, which
tests/test_gpu_vs_reference.py relies on, is checked without the reference."""
import pytest
import torch

from baseline import parity as PAR
from baseline import ref_loader as R

SHAPE = dict(hidden=256, layers=2, heads=2, kv_heads=2, inter=688, vocab=4096, max_pos=512, rope_theta=10000.0, eps=1e-5)


def _hf_model(dtype):
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(hidden_size=256, num_hidden_layers=2, num_attention_heads=2, num_key_value_heads=2,
                      intermediate_size=688, vocab_size=4096, max_position_embeddings=512, rms_norm_eps=1e-5,
                      tie_word_embeddings=False, attention_bias=False,
                      rope_parameters={"rope_type": "default", "rope_theta": 10000.0})
    torch.manual_seed(0)
    m = LlamaForCausalLM(cfg).to(dtype).eval()
    return m


def _ar_greedy(ref, prompt, n):
    ids = list(prompt)
    for _ in range(n):
        ids.append(int(torch.argmax(PAR.reference_next_logits(ref, ids))))
    return ids


@pytest.mark.skipif(not R.reference_available(), reason="unmodified reference not present (baseline/_ref)")
def test_reference_shares_weights_and_lookahead_equals_plain_greedy_fp32():
    hf = _hf_model(torch.float32)
    ref = PAR.reference_model_sharing_weights(hf, SHAPE)
    src = dict(hf.named_parameters())
    for name, p in ref.named_parameters():
        assert p.data_ptr() == src[name].data_ptr(), name
    g = torch.Generator().manual_seed(1)
    prompt = torch.randint(3, 4096, (24,), generator=g).tolist()
    ids, steps = PAR.reference_greedy(ref, prompt, 32, 5, 4, 5, py_seed=0)
    assert len(ids) == 24 + 32 and steps <= 32
    assert ids == _ar_greedy(ref, prompt, 32)

    # the comparison loop: an exact "engine", then one that flips a token (not a tie -> not ok)
    rep = PAR.compare_ids(lambda p, n: _ar_greedy(ref, p, n), ids, 24, ref)
    assert rep["exact"] and rep["ok"] and rep["n_divergences"] == 0 and rep["exact_prefix_tokens"] == 32

    def flipped(p, n):
        out = _ar_greedy(ref, p, n)
        if len(p) == 24:
            out[24 + 7] = (out[24 + 7] + 1) % 4096
        return out
    rep = PAR.compare_ids(flipped, ids, 24, ref)
    assert not rep["exact"] and not rep["ok"]
    assert rep["n_divergences"] == 1 and rep["divergences"][0]["index"] == 7 and rep["exact_prefix_tokens"] == 7
    assert rep["divergences"][0]["ref_below_top_ulps"] == 0.0 and rep["divergences"][0]["ours_below_top_ulps"] > 3


def test_bf16_ulp():
    assert PAR._bf16_ulp(1.0) == 2.0 ** -7 and PAR._bf16_ulp(5.0) == 2.0 ** -5 and PAR._bf16_ulp(-0.75) == 2.0 ** -8


def test_compare_against_a_recorded_reference():
    """compare_ids_to_record judges on the recorded top-k like compare_ids on live logits; a token outside the top-k
    is never a tie."""
    rec = {"ids": [5, 6, 1, 2, 3], "n_prompt": 2, "mant_bits": 7, "self_consistency": {"worst_below_top_ulps": 0.0},
           "top_idx": [[1, 4], [2, 7], [3, 0]], "top_val": [[1.0, 1.0], [1.0, 0.5], [2.0, 1.0]]}

    def engine(first_new):
        """Emits `first_new` after the prompt, and the reference's ids after that or after a forced prefix."""
        def gen(p, n):
            out = p + first_new if len(p) == 2 else list(p)
            return (out + rec["ids"][len(out):])[:len(p) + n]
        return gen
    rep = PAR.compare_ids_to_record(engine([]), rec, 8)
    assert rep["exact"] and rep["ok"] and rep["exact_prefix_tokens"] == 3
    rep = PAR.compare_ids_to_record(engine([4]), rec, 8)                # token 4 ties the reference's token 1
    assert not rep["exact"] and rep["ok"] and rep["n_divergences"] == 1 and rep["divergences"][0]["ours_below_top_ulps"] == 0.0
    rep = PAR.compare_ids_to_record(engine([1, 7]), rec, 8)             # 0.5 below the top: 64 ulps
    assert not rep["ok"] and rep["divergences"][0]["index"] == 1 and rep["divergences"][0]["ours_below_top_ulps"] == 64.0
    rep = PAR.compare_ids_to_record(engine([1, 2, 6]), rec, 8)          # not in the recorded top-k
    assert not rep["ok"] and rep["divergences"][0]["ours_below_top_ulps"] == float("inf")
