#!/usr/bin/env python
"""Generates tests/golden/reference_gpu_parity.json.gz: runs of the UNMODIFIED reference's greedy lookahead loop
(lade/decoding.py:697, loaded by baseline/ref_loader.py) on a B200, on the weight tensors of bench.build_model (seed 0),
for every configuration of tests/test_gpu_vs_reference.py.  Each record (baseline/parity.record_reference) holds the
ids, the reference's self-consistency report and the top-32 of its next-token logits at every generated position, plus
the sha256 of the weights, so that the test can judge the engine's ids without the reference.

Needs the reference (LADE_REFERENCE_ROOT=<checkout of hao-ai-lab/LookaheadDecoding>) and a CUDA device: the ids and
logits are those of the reference's eager loop on the GPU.

  python tests/golden/gen_golden_gpu_parity.py [OUT]        (default: tests/golden/reference_gpu_parity.json.gz)
"""
import gzip
import json
import os
import sys
import warnings

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]
warnings.filterwarnings("ignore")

from baseline import parity as PAR  # noqa: E402
from bench import build_model  # noqa: E402
from test_gpu_vs_reference import CASES, FP16_CASES, TINY  # noqa: E402


def model_pair(shape, dtype=torch.bfloat16, device="cuda"):
    hf = build_model(shape, torch.device(device), seed=0)
    if dtype != torch.bfloat16:
        hf = hf.to(dtype)
    return hf, PAR.reference_model_sharing_weights(hf, shape)


def prompt_ids(vocab, P, seed):
    return torch.randint(3, vocab, (P,), generator=torch.Generator().manual_seed(seed)).tolist()


def lookahead_record(shape, W, N, G, P, new, pool, dtype=torch.bfloat16, device="cuda"):
    hf, ref = model_pair(shape, dtype, device)
    prompt = prompt_ids(shape["vocab"], P, 1)
    ids, steps = PAR.reference_greedy(ref, prompt, new, W, N, G, py_seed=0, pool_from_prompt=pool)
    assert len(ids) == P + new
    return dict(PAR.record_reference(ref, ids, P), steps=steps, weights_sha256=PAR.weights_digest(hf),
                config=dict(W=W, N=N, G=G, pool_from_prompt=pool, dtype=str(dtype)))


def eos_first_record(device="cuda"):
    """W5 N3 G3 with pool, prompt 12: the EOS is the first token the reference emits without one."""
    hf, ref = model_pair(TINY, device=device)
    prompt = prompt_ids(32000, 12, 1)
    free, _ = PAR.reference_greedy(ref, prompt, 16, 5, 3, 3, py_seed=0, pool_from_prompt=True)
    ids, steps = PAR.reference_greedy(ref, prompt, 16, 5, 3, 3, py_seed=0, eos_token_id=[free[12]], pool_from_prompt=True)
    assert ids == prompt + [free[12]]
    return dict(PAR.record_reference(ref, ids, 12), steps=steps, weights_sha256=PAR.weights_digest(hf),
                config=dict(W=5, N=3, G=3, pool_from_prompt=True, eos_token_id=free[12]))


def plain_greedy_record(device="cuda"):
    """24 tokens of the reference model's plain greedy (its causal forward) after a 10-token prompt."""
    hf, ref = model_pair(TINY, device=device)
    ids = prompt_ids(32000, 10, 3)
    for _ in range(24):
        ids.append(int(torch.argmax(PAR.reference_next_logits(ref, ids))))
    return dict(PAR.record_reference(ref, ids, 10), steps=24, weights_sha256=PAR.weights_digest(hf),
                config=dict(plain_greedy=True))


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "reference_gpu_parity.json.gz")
    assert torch.cuda.is_available(), "the records are of the reference's run on the GPU"
    recs = {}
    for (name, shape, W, N, G, P, new, pool) in CASES:
        recs[name] = lookahead_record(shape, W, N, G, P, new, pool)
        if name in FP16_CASES:
            recs["fp16/" + name] = lookahead_record(shape, W, N, G, P, new, pool, dtype=torch.float16)
    recs["eos_first"] = eos_first_record()
    recs["plain_greedy"] = plain_greedy_record()
    for k, r in recs.items():
        print(f"{k}: {len(r['ids']) - r['n_prompt']} tokens in {r['steps']} steps, self-consistency "
              f"{r['self_consistency']['n_self_mismatch']} mismatches (worst {r['self_consistency']['worst_below_top_ulps']} ulp)")
    with gzip.open(out, "wt") as f:
        json.dump(dict(device=torch.cuda.get_device_name(0), torch=torch.__version__, records=recs), f,
                  separators=(",", ":"))


if __name__ == "__main__":
    main()
