"""Lookahead parallelism on device.

(1) single GPU, bit-exact: D device contexts (one per simulated rank) are driven with the reference's own
    per-rank LP traces (tests/golden/lp_traces.json.gz, real gloo run of the unmodified reference); the
    all-gather is a concatenation of the D records.  Every rank's rows / position ids / masks, the reduced
    decision, the replicated pool and the output ids must equal the reference's.
(2) multi GPU (skipped unless >= 2 devices and launched under torchrun): the engine over NCCL produces the
    single-GPU ids."""
import ctypes as C
import gzip
import json
import os
import random

import numpy as np
import pytest
import torch

from helpers import GOLD, make_lade_config

pytestmark = pytest.mark.gpu


def load_lp_cases():
    with gzip.open(os.path.join(GOLD, "lp_traces.json.gz"), "rt") as f:
        return json.load(f)


LP_CASES = load_lp_cases()


@pytest.mark.parametrize("name", sorted(LP_CASES))
def test_lp_device_state_machine_matches_reference(name):
    from lookaheaddecoding_b200 import _cabi
    from lookaheaddecoding_b200._cabi import check

    lib = _cabi.load()
    c = LP_CASES[name]
    W, N, G, D = c["W"], c["N"], c["G"], c["D"]
    GS, WCAP = N - 1, W + N - 3
    V = c["model"]["vocab"]
    P = len(c["prompt"])
    max_length = P + c["max_new"]
    dev = torch.device("cuda")
    stream = torch.cuda.current_stream().cuda_stream
    i32 = dict(dtype=torch.int32, device=dev)
    prompt = np.asarray(c["prompt"], dtype=np.int32)
    win0 = np.asarray(_full_window0(c), dtype=np.int32)
    ctxs, cfgs = [], []
    for r in range(D):
        cfg = make_lade_config(W, N, G, V, max_length + N + 8, pool=c["pool_from_prompt"])
        cfg.dist_workers, cfg.rank = D, r
        ctx = C.c_void_p()
        check(lib.lade_ctx_create(C.byref(cfg), C.byref(ctx)), "create")
        check(lib.lade_ctx_reset(ctx, stream, prompt.ctypes.data, P, win0.ctypes.data, WCAP, max_length), "reset")
        ctxs.append(ctx)
        cfgs.append(cfg)
    torch.cuda.synchronize()
    rec_ints = lib.lade_lp_record_ints(C.byref(cfgs[0]))
    assert rec_ints == 3 + GS + WCAP
    lm_cap = 1 + WCAP + G * GS
    q_cap = P + WCAP + GS * (W + G) + 8
    n_steps = c["n_steps"]
    out_ids = list(c["prompt"])
    recs = torch.zeros(D * rec_ints, **i32)
    metas = [torch.zeros(_cabi.META_INTS, **i32) for _ in range(D)]
    res = [torch.zeros(_cabi.RES_INTS, **i32) for _ in range(D)]
    for i in range(n_steps):
        for r in range(D):
            g = c["ranks"][r]["steps"][i]
            n_in = len(g["input_ids"])
            flat = list(g["input_ids"])
            flat_pos = list(g["position_ids"])
            lst = g["position_ids"][-1]
            for ll, lvl in enumerate(g["past_tokens"][: g["fill_level"] + 1]):
                flat = flat + lvl
                if ll == 0:
                    flat_pos = flat_pos + list(range(lst + 1, lst + 1 + len(lvl)))
                else:
                    off = len(g["past_tokens"][0]) + 1 - len(lvl)
                    flat_pos = flat_pos + list(range(lst + ll + off, lst + ll + off + len(lvl)))
            gt = g["guess_tokens"] or []
            flat = flat + gt
            flat_pos = flat_pos + list(range(lst + 1, lst + 1 + GS)) * (len(gt) // GS)
            q_len = len(flat)
            bound = lib.lade_step_rows_bound(C.byref(cfgs[r]), P, i)
            assert bound >= q_len, f"rank {r} step {i}: rows bound {bound} < {q_len}"
            q_pad = bound
            ids, pos, rd = torch.zeros(q_cap, **i32), torch.zeros(q_cap, **i32), torch.zeros(q_cap, **i32)
            lm_rows = torch.zeros(lm_cap, **i32)
            mw = (q_pad + 31) // 32 + 1
            rowmask = torch.zeros(q_pad * mw, **i32)
            check(lib.lade_step_layout(ctxs[r], stream, q_pad, ids.data_ptr(), pos.data_ptr(), rd.data_ptr(),
                                       lm_rows.data_ptr(), metas[r].data_ptr(), rowmask.data_ptr(), mw), "layout")
            m = metas[r].cpu().numpy()
            assert m[_cabi.M_Q_LEN] == q_len, f"rank {r} step {i}: q_len {m[_cabi.M_Q_LEN]} != {q_len}"
            assert ids[:q_len].cpu().tolist() == flat, f"rank {r} step {i} ids"
            assert pos[:q_len].cpu().tolist() == flat_pos, f"rank {r} step {i} pos"
            assert m[_cabi.M_KV_LEN] + n_in == g["kvcache_len"] and m[_cabi.M_KV_LEN] + q_len == g["step_len"]
            if g["mask_rows"] is not None:
                from test_gpu_state_machine import _mask_from_rowdesc
                from helpers import rows_to_bool
                want = rows_to_bool(g["mask_rows"])[:, m[_cabi.M_KV_LEN]:]
                got = _mask_from_rowdesc(rd[:q_len].cpu().numpy(), q_len, int(m[_cabi.M_LEVEL_OFFSET]))
                np.testing.assert_array_equal(got, want, err_msg=f"rank {r} step {i} mask")
                if i > 0:
                    wd = rowmask.cpu().numpy().view(np.uint32).reshape(q_pad, mw)
                    bits = np.unpackbits(wd.view(np.uint8).reshape(q_pad, mw * 4), axis=-1, bitorder="little").astype(bool)
                    np.testing.assert_array_equal(bits[:q_len, :q_len], want, err_msg=f"rank {r} step {i} rowmask")
            am = np.zeros(lm_cap, dtype=np.int32)
            am[0] = g["first_guess"]
            am[1:1 + len(g["inp_tokens"])] = g["inp_tokens"]
            am[1 + WCAP:1 + WCAP + len(g["guess_results"])] = g["guess_results"]
            am_d = torch.from_numpy(am).to(dev)
            check(lib.lade_lp_verify(ctxs[r], stream, am_d.data_ptr(), metas[r].data_ptr(),
                                     recs[r * rec_ints:].data_ptr()), "lp_verify")
        for r in range(D):   # "all-gather" = every rank sees the same concatenation
            check(lib.lade_lp_commit(ctxs[r], stream, recs.data_ptr(), metas[r].data_ptr(), res[r].data_ptr()), "lp_commit")
        rs = [x.cpu().numpy() for x in res]
        for r in range(1, D):
            np.testing.assert_array_equal(rs[r][:9], rs[0][:9])      # slot 9 (n-grams verified) is rank-local
            np.testing.assert_array_equal(rs[r][_cabi.R_HITS:_cabi.R_HITS + GS], rs[0][_cabi.R_HITS:_cabi.R_HITS + GS])
        n_emit = int(rs[0][_cabi.R_N_EMIT])
        out_ids += rs[0][_cabi.R_HITS:_cabi.R_HITS + n_emit].tolist()
        if i + 1 < n_steps:
            nxt = c["ranks"][0]["steps"][i + 1]
            assert out_ids[-len(nxt["input_ids"]):] == nxt["input_ids"], f"step {i}: re-fed tokens"
            assert int(rs[0][_cabi.R_KV_LEN]) + len(nxt["input_ids"]) == nxt["kvcache_len"]
            assert not rs[0][_cabi.R_DONE]
        else:
            assert rs[0][_cabi.R_DONE]
    assert out_ids[:max_length] == c["output_ids"]
    for r in range(D):
        cnt = np.zeros(V, dtype=np.int32)
        tup = np.zeros((V, G, GS), dtype=np.int32)
        check(lib.lade_ctx_pool_snapshot(ctxs[r], stream, cnt.ctypes.data, tup.ctypes.data), "snapshot")
        got = {str(k): tup[k, : cnt[k]].tolist() for k in np.nonzero(cnt)[0]}
        assert got == c["ranks"][r]["final_pool"], f"rank {r} pool"
        lib.lade_ctx_destroy(ctxs[r])


def _full_window0(c):
    """The broadcast initial window = the last rank's level-0 input at step 0 is a prefix only; rebuild the
    full W+N-3 window from the rank that feeds all of it (the last non-empty slice ends at window_len)."""
    best = max((rk["steps"][0]["past_tokens"][0] for rk in c["ranks"]), key=len)
    assert len(best) == c["W"] + c["N"] - 3
    return best


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("world", [w for w in (2, 4, 8) if w <= max(torch.cuda.device_count(), 2)])
def test_engine_lp_over_nccl_matches_single_gpu(world):
    """Real NCCL run: torchrun x `world` ranks, lade.config_lade(DIST_WORKERS=world); ids == single-GPU ids."""
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.join(here, "lp_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "LP_WORKER_OK" in res.stdout
    print(res.stdout[-1500:])
