#!/usr/bin/env python
"""bench.py -- tokens/sec + accepted-tokens/step of lookahead decoding, Llama-2-7B shape, W=15 N=5 G=15.

One "step" of the contract = one full generate() of `--max-new` tokens from a fixed synthetic prompt
(the unit minimal.py:34-45 times).  `value` is whole-job tokens/s with the prompt ids already handed to
the engine (device timed with CUDA events); `e2e` is the same metric through the reference-facing plugin
surface (lade.augment_all(); lade.config_lade(...); model.generate(...)) with the prompt in pinned host
memory and the output read back to the host inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload 7b|13b|tiny]
                  [--dump-outputs DIR]

Extra objects on the JSON line: `roofline` (lookahead-attention kernel, HBM bound, timed live with CUDA
events), `cpu_baseline` (the oracle port of the reference's loop on the host cores, bounded sample),
`clocks`, `accepted_tokens_per_step`.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (model shape, W, N, G, prompt_len)
    "7b": (dict(hidden=4096, layers=32, heads=32, kv_heads=32, inter=11008, vocab=32000, max_pos=4096,
                rope_theta=10000.0, eps=1e-5), 15, 5, 15, 1024),
    "13b": (dict(hidden=5120, layers=40, heads=40, kv_heads=40, inter=13824, vocab=32016, max_pos=16384,
                 rope_theta=1000000.0, eps=1e-5), 20, 7, 20, 256),
    "tiny": (dict(hidden=256, layers=2, heads=2, kv_heads=2, inter=688, vocab=32000, max_pos=2048,
                  rope_theta=10000.0, eps=1e-5), 5, 3, 3, 64),
}
WORKLOAD_NAMES = {"7b": "Llama-2-7B-shaped random-init bf16, greedy", "13b": "CodeLlama-13B-shaped random-init bf16, greedy",
                  "tiny": "tiny random-init Llama (2 layers, hidden 256), greedy"}


def _positive_int(v):
    n = int(v)
    if n < 1:
        raise argparse.ArgumentTypeError(f"{v} is not >= 1")
    return n


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive_int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="7b", choices=sorted(WORKLOADS))
    ap.add_argument("--prompt-len", type=int, default=None)
    ap.add_argument("--max-new", type=int, default=256)
    ap.add_argument("--attn-impl", type=int, default=0)
    ap.add_argument("--attn-splits", type=int, default=0)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--do-sample", action="store_true",
                    help="BASELINE.json configs[2]: sampling, temperature 0.8, top_k=0, top_p=1.0 (lade/decoding.py:137)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the AR series and the extra BASELINE configs (7B sampling, 13B, periodic-text weights)")
    ap.add_argument("--weights", default="random", choices=["random", "cyclic"],
                    help="cyclic: o_proj/down_proj zeroed -> periodic text, n-gram hits (see build_model)")
    ap.add_argument("--lp-scale", action="store_true",
                    help="lookahead parallelism with WINDOW_SIZE and GUESS_SET_SIZE multiplied by the number of ranks (each "
                         "rank keeps about the single-GPU row count: the lookahead capacity grows with N, not the per-rank "
                         "work); not the BASELINE config -- the line says so in config.workload")
    ap.add_argument("--ref-budget-s", type=float, default=240.0,
                    help="--impl reference: wall-clock bound of the timed steady steps; once 3 are in, it ends the "
                         "sample before --steps (the JSON line's `steps` says how many were timed)")
    ap.add_argument("--no-reference-cuda", action="store_true",
                    help="skip timing the unmodified reference's CUDA-eager loop (needs baseline/_ref)")
    ap.add_argument("--cuda-profiler-range", action="store_true",
                    help="cudaProfilerStart/Stop around the timed region (use with ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the ids the last timed generate() returned (DIR/output_ids.npy) "
                         "and those of the last end-to-end generate() (DIR/e2e_output_ids.npy), float64, prompt included")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times a bounded sample of steps and has no outputs")
    return args


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock / throttle reasons during the timed region (B200_PROFILING.md recipe), sampled IN-PROCESS through NVML
    (nvidia_ml_py) every 0.25 s.  Round 1 spawned `nvidia-smi` every 200 ms; on the 8-GPU node each spawn enumerates
    all boards and the end-to-end leg lost half its throughput there.  Falls back to the subprocess at 1 Hz when NVML
    cannot be loaded."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index: int):
        self.index = index
        self.rows = []          # (sm_mhz, sm_max_mhz, reason_bits)
        self._stop = threading.Event()
        self._t = None
        self._h = None
        self._nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self._nv, self._h = pynvml, h
            self._max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    def _sample_nvml(self):
        nv, h = self._nv, self._h
        sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
        try:
            bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
        except Exception:
            bits = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
        self.rows.append((sm, self._max, bits))

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
            r = [x.strip() for x in out.split(",")]
            bits = 0
            for bit, v in zip((0x8, 0x40, 0x20, 0x4), r[2:6]):
                if v.lower().startswith("active"):
                    bits |= bit
            self.rows.append((float(r[0]), float(r[1]), bits))

    def _run(self):
        while not self._stop.is_set():
            try:
                if self._nv is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.25 if self._nv is not None else 1.0)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[2]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(r[1] for r in self.rows),
                "reasons": sorted(n for b, n in self.REASONS.items() if bits & b), "samples": len(sm),
                "source": "nvml" if self._nv is not None else "nvidia-smi"}


def build_model(shape, device, seed=0, weights="random", dtype=None):
    """HF LlamaForCausalLM of `shape`, random init normal(0, 0.02) (modeling_llama.py:934-943), bf16.
    weights="cyclic": o_proj and down_proj are zeroed, so every layer is the identity on the residual stream and the
    next token is a deterministic function of the last one -- the text becomes periodic, n-grams repeat, and the
    verification branch / kv_compact / pool lookups do real work.  Bytes and FLOPs per step are unchanged."""
    import torch
    from transformers import LlamaConfig, LlamaForCausalLM

    cfg = LlamaConfig(
        hidden_size=shape["hidden"], num_hidden_layers=shape["layers"], num_attention_heads=shape["heads"],
        num_key_value_heads=shape["kv_heads"], intermediate_size=shape["inter"], vocab_size=shape["vocab"],
        max_position_embeddings=shape["max_pos"], rms_norm_eps=shape["eps"], tie_word_embeddings=False,
        attention_bias=False, hidden_act="silu",
        rope_parameters={"rope_type": "default", "rope_theta": shape["rope_theta"]})
    with torch.device("meta"):
        model = LlamaForCausalLM(cfg)
    model = model.to_empty(device=device).to(torch.bfloat16)
    g = torch.Generator(device=device).manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():      # normal(0, initializer_range) as modeling_llama.py:934-943
            if p.dim() >= 2:
                p.normal_(0.0, 0.02, generator=g)
                if weights == "cyclic" and (name.endswith("o_proj.weight") or name.endswith("down_proj.weight")):
                    p.zero_()
            else:
                p.fill_(1.0)
        if hasattr(model.model, "rotary_emb"):
            re = model.model.rotary_emb
            D = cfg.hidden_size // cfg.num_attention_heads
            inv = 1.0 / (shape["rope_theta"] ** (torch.arange(0, D, 2, dtype=torch.float32) / D))
            re.inv_freq = inv.to(device)
            if hasattr(re, "original_inv_freq"):
                re.original_inv_freq = inv.to(device)
    if dtype is not None:
        import torch as _t
        if dtype != _t.bfloat16:
            model = model.to(dtype)              # same draws, rounded to the other 16-bit format
    model.eval()
    model.generation_config.pad_token_id = 0
    model.generation_config.eos_token_id = None
    return model


def attn_roofline(eng, shape, reps=5):
    """Time the lookahead-attention kernel alone, back to back over every layer's cache (L x 2 x kv rows
    > L2, so no launch re-reads a cache line of the previous ones), on the launching stream."""
    import torch
    from lookaheaddecoding_b200 import _cabi

    lib = eng.lib
    meta_now = eng.meta.cpu().tolist()
    kv_len = meta_now[_cabi.M_KV_LEN]
    # own Q / output buffers at the metric's full shape (under LP the engine's per-rank buffers are smaller)
    # full steady-state layout of the metric's shape (q = (N-1)(W+G) rows: every guess slot filled); random-init
    # weights on a random prompt rarely produce pool hits, so the live decode mostly runs with fewer rows
    W, N, G, GS = eng.W, eng.N, eng.G, eng.GS
    q_len = GS * (W + G)
    rows = q_len
    kv_len = min(kv_len, eng.kv_capacity - q_len)          # stay inside the allocated cache rows
    import numpy as np
    vis = np.zeros((q_len, q_len), dtype=bool)            # steady lookahead mask, SURVEY App. B (one GPU)
    for r in range(q_len):
        if r < GS * W:
            lvl, j = divmod(r, W)
            vis[r, : j + 1] = True                        # level-0 block, causal in the column
            for l2 in range(1, lvl + 1):
                vis[r, l2 * W + j] = True                 # same column of levels 1..lvl
        else:
            e, u = divmod(r - GS * W, GS)
            vis[r, 0] = True                              # the input token
            vis[r, GS * W + e * GS: GS * W + e * GS + u + 1] = True
    mw = (rows + 31) // 32 + 1
    bits = np.zeros((rows, mw * 32), dtype=bool)
    bits[:q_len, :q_len] = vis
    words = np.packbits(bits.reshape(rows, mw, 32), axis=-1, bitorder="little").view(np.uint32).reshape(rows, mw)
    rowmask = torch.from_numpy(words.view(np.int32).copy()).to(eng.dev)
    meta = torch.zeros(_cabi.META_INTS, dtype=torch.int32, device=eng.dev)
    for k, v in {_cabi.M_Q_LEN: q_len, _cabi.M_KV_LEN: kv_len, _cabi.M_N_INPUT: 1, _cabi.M_TINY: W,
                 _cabi.M_N_LEVELS: N - 1, _cabi.M_N_GUESS_TOK: G * GS, _cabi.M_PHASE: 2, _cabi.M_Q_PAD: rows}.items():
        meta[k] = v
    qb = torch.randn(eng.nh, rows, eng.D, device=eng.dev).to(eng.dt)
    attn_out = torch.empty(rows, eng.nh * eng.D, dtype=eng.dt, device=eng.dev)
    scratch = torch.zeros(int(lib.lade_attn_scratch_bytes(rows, eng.nh, eng.D, eng.attn_splits)), dtype=torch.uint8, device=eng.dev)
    stream = torch.cuda.current_stream(eng.dev)

    def one_pass():
        cs = torch.cuda.current_stream(eng.dev).cuda_stream
        for l in range(eng.L):
            _cabi.check(eng.k_attn_fwd(cs, qb.data_ptr(), eng.kv[l, 0].data_ptr(), eng.kv[l, 1].data_ptr(),
                                          attn_out.data_ptr(), rowmask.data_ptr(), mw, meta.data_ptr(),
                                          scratch.data_ptr(), rows, eng.nh, eng.nkv, eng.D, eng.kv_capacity,
                                          eng.kv_capacity, eng.attn_splits, eng.attn_impl))
    def timed_us(pdl):
        """us per launch, one pass over the L layer caches captured in a CUDA graph (the launch rate of a python loop,
        ~20 us per ctypes call, must not bound the kernel measurement); events on the replaying stream."""
        _cabi.check(lib.lade_debug_attn_pdl(pdl))
        for _ in range(3):
            one_pass()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=eng.dev)
        side.wait_stream(torch.cuda.current_stream(eng.dev))
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                one_pass()
        torch.cuda.current_stream(eng.dev).wait_stream(side)
        g.replay()
        torch.cuda.synchronize()
        stream = torch.cuda.current_stream(eng.dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            g.replay()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / (reps * eng.L)

    # (1) as launched in the decode step: programmatic dependent launch on -- there the kernel's set-up overlaps the
    # tail of lade_rope_append; in this loop the predecessor is the previous layer's lade_attn_fwd, which triggers its
    # dependents at entry in the same way (tools/step_ablation.py: the kernel costs the same 15 us inside the step);
    # (2) strictly serialised launches (attribute off), reported beside it
    us = timed_us(1)
    us_serial = timed_us(0)
    _cabi.check(lib.lade_debug_attn_pdl(-1))
    # algorithmic bytes per launch (SURVEY.md 8d): K,V cache read + Q read + new K,V read + O write
    Hq, Hkv, D = eng.nh, eng.nkv, eng.D
    bytes_alg = 2 * kv_len * Hkv * D * 2 + q_len * Hq * D * 2 + 2 * q_len * Hkv * D * 2 + q_len * Hq * D * 2
    peak, how = measured_peaks()
    achieved = bytes_alg / (us * 1e-6) / 1e9
    traffic = None            # DRAM bytes per launch from the committed ncu capture closest to this shape
    try:
        with open(os.path.join(ROOT, "profiles", "attn_traffic.json")) as f:
            caps = [c for c in json.load(f)["captures"] if c["q_len"] == q_len]
        if caps:
            best = min(caps, key=lambda c: abs(c["kv_len"] - kv_len))
            if abs(best["kv_len"] - kv_len) <= 64:
                traffic = best["dram_bytes"]
    except Exception:
        traffic = None
    return {"bound": "hbm", "kernel": "lade_attn_fwd", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
            "frac": round(achieved / peak, 4), "traffic": traffic, "peak_source": how, "us_per_launch": round(us, 2),
            "us_per_launch_serialized": round(us_serial, 2), "frac_serialized": round(bytes_alg / (us_serial * 1e-6) / 1e9 / peak, 4),
            "launch_mode": "programmatic dependent launch as in the decode step (set-up overlaps the predecessor's tail); "
                           "'serialized' = the same loop with the attribute off",
            "alg_bytes_per_launch": bytes_alg, "kv_len": kv_len, "q_len": q_len, "launches_timed": reps * eng.L}


def usable_cores() -> int:
    """Host cores this process may really use: affinity mask, clipped by the cgroup CPU quota (os.cpu_count() reports
    the machine, and oversubscribing a quota-limited container makes the CPU baseline slow and erratic)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except (OSError, ValueError):
        try:    # cgroup v1
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                quota = int(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                period = int(f.read())
            if quota > 0 and period > 0:
                n = max(1, min(n, quota // period))
        except (OSError, ValueError):
            pass
    return n


class _EnoughSteps(Exception):
    pass


def reference_cpu(shape, W, N, G, P, max_new, n_threads, timed_steps=8, warm_steps=2, budget_s=240.0, weights="random"):
    """The UNMODIFIED reference (baseline/_ref, loaded by baseline/ref_loader.py with the shims of SURVEY App. C)
    running its own `jacobi_greedy_search_multilevel` (lade/decoding.py:697) on the HOST cores at the full stated
    config: full depth, full widths, prompt P.  Bounded sample: the prefill step and the N-3 window-fill steps are
    timed once, then `warm_steps` untimed + up to `timed_steps` timed STEADY decode steps (all identical in shape);
    the run is aborted from a forward hook once enough steps are in (or `budget_s` is spent, never below 3 steps).
    tokens/s of the whole workload = max_new / (t_prefill + t_fill + n_steady * mean(steady step)).
    Each step time is a full loop iteration (model forward + the reference's python token selection / pool update)."""
    import statistics
    import torch
    from baseline import ref_loader as R
    from transformers import GenerationConfig, MaxLengthCriteria, StoppingCriteriaList

    if not R.reference_available():
        return {"unavailable": "baseline/_ref not present"}
    torch.set_num_threads(n_threads)
    decoding, modeling = R.load_reference()
    cfg = R.make_llama_config(hidden=shape["hidden"], layers=shape["layers"], heads=shape["heads"], kv_heads=shape["kv_heads"],
                              inter=shape["inter"], vocab=shape["vocab"], max_pos=shape["max_pos"],
                              rope_theta=shape["rope_theta"], eps=shape["eps"])
    old_dtype = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    t_build = time.perf_counter()
    try:
        with torch.device("meta"):
            model = modeling.LlamaForCausalLM(cfg)
        model = model.to_empty(device="cpu")
        # normal(0, 0.02) values are drawn ONCE (2^24 of them) and tiled into every matrix at a per-tensor offset:
        # drawing 6.7 G values with the CPU generator alone takes minutes, and GEMM time does not depend on the values
        g = torch.Generator().manual_seed(0)
        bank = (torch.randn(1 << 24, generator=g, dtype=torch.float32) * 0.02).to(torch.bfloat16)
        with torch.no_grad():
            for k, (name, p_) in enumerate(model.named_parameters()):
                if p_.dim() >= 2:
                    if weights == "cyclic" and (name.endswith("o_proj.weight") or name.endswith("down_proj.weight")):
                        p_.zero_()
                        continue
                    flat = p_.view(-1)
                    off = (k * 1000003) % (bank.numel() // 2)
                    pos = 0
                    while pos < flat.numel():
                        n = min(bank.numel() - off, flat.numel() - pos)
                        flat[pos:pos + n].copy_(bank[off:off + n])
                        pos += n
                        off = 0
                else:
                    p_.fill_(1.0)
        for mod in model.modules():          # rotary tables were left uninitialised by to_empty()
            if hasattr(mod, "_set_cos_sin_cache") and hasattr(mod, "inv_freq"):
                inv = 1.0 / (mod.base ** (torch.arange(0, mod.dim, 2).float() / mod.dim))
                mod.register_buffer("inv_freq", inv, persistent=False)
                mod._set_cos_sin_cache(seq_len=mod.max_position_embeddings, device="cpu", dtype=torch.bfloat16)
        model.eval()
        model.generation_config = GenerationConfig(pad_token_id=0, eos_token_id=None)
        t_build = time.perf_counter() - t_build
        torch.manual_seed(1)
        prompt = torch.randint(3, shape["vocab"], (1, P))
        n_pre = N - 2                                   # prefill + N-3 window-fill steps
        marks = []
        t_start = [0.0]
        inner = model.jforward_multilevel

        def hooked(*a, **k):
            now = time.perf_counter()
            marks.append(now)
            steady_done = len(marks) - 1 - n_pre - warm_steps      # completed timed steady steps
            if steady_done >= timed_steps or (steady_done >= 3 and now - t_start[0] > budget_s):
                raise _EnoughSteps()
            return inner(*a, **k)

        model.jforward_multilevel = hooked
        decoding.CONFIG_MAP.clear()
        decoding.CONFIG_MAP.update(dict(WINDOW_SIZE=W, LEVEL=N, GUESS_SET_SIZE=G, DEBUG=0, log=[]))
        random.seed(0)
        t_start[0] = time.perf_counter()
        import contextlib, io
        try:
            with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
                decoding.jacobi_greedy_search_multilevel(
                    model, prompt, stopping_criteria=StoppingCriteriaList([MaxLengthCriteria(P + max_new)]),
                    attention_mask=torch.ones_like(prompt), use_cache=True, return_dict_in_generate=False,
                    output_attentions=False, output_hidden_states=False, output_scores=False, pad_token_id=0,
                    eos_token_id=None)
            marks.append(time.perf_counter())           # the run ended by itself (short max_new)
        except _EnoughSteps:
            pass
    finally:
        torch.set_default_dtype(old_dtype)
    dur = [b - a for a, b in zip(marks[:-1], marks[1:])]           # full loop iterations
    t_prefill = dur[0]
    t_fill = sum(dur[1:n_pre])
    steady = dur[n_pre + warm_steps:]
    if len(steady) < 1:
        return {"unavailable": f"too few steps timed ({len(dur)})"}
    mean_steady = sum(steady) / len(steady)
    # random-init weights on a random prompt accept exactly 1 token per step (the GPU arm reports the same); under
    # `cyclic` weights the acceptance of the sample is not representative of the whole run, so it is not extrapolated
    n_steady = max_new - n_pre
    total_s = t_prefill + t_fill + n_steady * mean_steady
    return {"value": round(max_new / total_s, 4), "unit": "tokens/s", "cores": n_threads, "kind": "reference",
            "s_per_steady_step": round(mean_steady, 4), "steady_steps_timed": len(steady),
            "steady_min_s": round(min(steady), 4), "steady_max_s": round(max(steady), 4),
            "steady_stdev_s": round(statistics.pstdev(steady), 4), "prefill_s": round(t_prefill, 3),
            "window_fill_s": round(t_fill, 3), "model_build_s": round(t_build, 1), "accepted_tokens_per_step": 1.0,
            "sample": f"UNMODIFIED reference (baseline/_ref) jacobi_greedy_search_multilevel on {n_threads} host threads, bf16, "
                      f"full depth ({shape['layers']} layers) and widths, prompt {P}: prefill step {t_prefill:.1f}s + {n_pre - 1} "
                      f"window-fill steps {t_fill:.1f}s timed once, {warm_steps} untimed + {len(steady)} timed steady steps "
                      f"(mean {mean_steady:.3f}s, min {min(steady):.3f}, max {max(steady):.3f}); whole workload "
                      f"= {max_new} tokens / (prefill + fill + {n_steady} x mean steady step) at 1.0 accepted tokens/step"}


def reference_cuda_eager(ref_model, shape, W, N, G, prompt_list, max_new):
    """The UNMODIFIED reference (baseline/_ref) running its own eager lookahead loop on the same GPU and the SAME weight
    tensors as our engine: the denominator of BASELINE.json's ">= 1.8x over the reference's own CUDA eager lookahead".
    Returns (report, ids of the timed run)."""
    import torch
    from baseline import parity as PAR

    PAR.reference_greedy(ref_model, prompt_list, 4, W, N, G, py_seed=0)           # warm-up (minimal.py:30)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ids, steps = PAR.reference_greedy(ref_model, prompt_list, max_new, W, N, G, py_seed=0)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    toks = len(ids) - len(prompt_list)
    return {"value": round(toks / dt, 2), "unit": "tokens/s", "tokens": toks, "decode_steps": steps,
            "ms_per_decode_step": round(1e3 * dt / steps, 3), "accepted_tokens_per_step": round(toks / steps, 3),
            "source": "unmodified reference (baseline/_ref, shims of SURVEY App. C), eager attention, same GPU, same weight "
                      "tensors / prompt / seeds; wall clock around one generate after a warm-up (minimal.py:34-45)"}, ids


def time_generates(run_once, n, P, eng, dev):
    """n device-timed generate() calls; returns (tokens, steps, ms)."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    toks = steps = 0
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        out = run_once()
        toks += len(out) - P
        steps += eng.last_steps
    e1.record()
    torch.cuda.synchronize()
    return toks, steps, e0.elapsed_time(e1)


def extra_workload(name, args, dev, do_sample=False, model=None, reps=3, dtype=None):
    """One more BASELINE.json config measured in the same process (device-timed generate() calls + its own attention
    roofline): configs[2] (7B sampling, T=0.8) and configs[3] (CodeLlama-13B shape, W20 N7 G20)."""
    import torch
    from lookaheaddecoding_b200 import LookaheadEngine
    shape, W, N, G, P = WORKLOADS[name]
    own = model is None
    if own:
        model = build_model(shape, dev, dtype=dtype)
    eng = LookaheadEngine(model, W, N, G, max_total_len=P + args.max_new)
    torch.manual_seed(1)
    prompt = torch.randint(3, shape["vocab"], (1, P))[0].tolist()
    if do_sample:
        def run_once():         # verification on device (lade_sample_verify, Philox)
            return eng.generate(prompt, args.max_new, rng=random.Random(0), sampling={"temperature": 0.8, "seed": 2})
    else:
        def run_once():
            return eng.generate(prompt, args.max_new, rng=random.Random(0))
    for _ in range(2):
        run_once()
    toks, steps, ms = time_generates(run_once, reps, P, eng, dev)
    roof = attn_roofline(eng, shape)
    wname = WORKLOAD_NAMES[name] if dtype is None else WORKLOAD_NAMES[name].replace("bf16", str(dtype).replace("torch.", ""))
    rep = {"workload": f"{wname}{' -> sampling temp=0.8 top_k=0 top_p=1.0' if do_sample else ''}, W={W} N={N} "
                       f"G={G}, prompt {P}, {args.max_new} new tokens", "value": round(toks / (ms * 1e-3), 2),
           "unit": "tokens/s", "generates_timed": reps, "ms_per_decode_step": round(ms / steps, 4),
           "accepted_tokens_per_step": round(toks / steps, 3), "attn_splits": eng.attn_splits, "roofline": roof}
    eng.close()
    del eng
    if own:
        model.__dict__.pop("_lade_fused", None)
        model.__dict__.pop("_lade_engines", None)
        del model
    torch.cuda.empty_cache()
    return rep


def main():
    args = parse()
    shape, W, N, G, P = WORKLOADS[args.workload]
    if args.prompt_len:
        P = args.prompt_len
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.lp_scale and world > 1:
        W, G = W * world, G * world
    config = {"workload": f"{WORKLOAD_NAMES[args.workload]}, W={W} N={N} G={G}, prompt {P} tokens, {args.max_new} new tokens "
                          f"per generate()", "prompt_len": P, "max_new_tokens": args.max_new,
              "weights": "random-init normal(0, 0.02)" if args.weights == "random" else
              "random-init, o_proj/down_proj zeroed (periodic text: n-gram hits; same bytes/FLOPs)",
              "parallelism": "single" if world == 1 else
              f"lookahead parallelism x{world} (lade_distributed: window columns + guess n-grams sharded per rank, "
              f"one NCCL all-gather of a fixed int32 record per step; same W/G => total work fixed)",
              "l2_policy": "inputs larger than L2 (weights 13 GB/step stream through; KV of 32 layers > 126 MB)"}
    metric = "tokens/sec (wall-clock) and accepted-tokens/step, Llama-2-7B W=15 N=5 G=15" if args.workload == "7b" else \
        f"tokens/sec (wall-clock) and accepted-tokens/step, {args.workload} W={W} N={N} G={G}"

    if args.impl == "reference":
        if rank != 0:
            return
        # The reference's own implementation of the path on the host cores: the UNMODIFIED reference from baseline/_ref
        # at the stated config (full depth, P tokens of context).  One "step" of this arm = one steady decode step of
        # its loop (a bounded sample of the workload); W untimed + K timed, the whole-workload tokens/s follows from
        # prefill + window fill (timed once) + (max_new - N + 2) steady steps.
        n_threads = usable_cores()
        cb = reference_cpu(shape, W, N, G, P, args.max_new, n_threads, timed_steps=args.steps,
                           warm_steps=max(0, args.warmup), budget_s=args.ref_budget_s, weights=args.weights)
        if "unavailable" in cb:
            print(json.dumps({"impl": "reference", "unavailable": cb["unavailable"]}))
            return
        # --steps steady steps are timed unless --ref-budget-s runs out first (never below 3) or the run ends by itself
        line = {"metric": metric, "value": cb["value"], "unit": "tokens/s", "n_gpus": args.gpus,
                "steps": cb["steady_steps_timed"],
                "warmup": args.warmup, "ms_per_step": round(1e3 * cb["s_per_steady_step"], 1), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config,
                "impl": "reference", "accepted_tokens_per_step": cb["accepted_tokens_per_step"], "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import lade
    from lookaheaddecoding_b200.decoding import CONFIG_MAP, get_engine

    model = build_model(shape, dev, weights=args.weights)
    os.environ["USE_LADE"] = "1"
    lade.augment_all()
    lade.config_lade(LEVEL=N, WINDOW_SIZE=W, GUESS_SET_SIZE=G, DEBUG=0, DIST_WORKERS=world if world > 1 else None,
                     backend="nccl")
    CONFIG_MAP["MAX_TOTAL_LEN"] = P + args.max_new
    overrides = {}
    if args.attn_impl:
        overrides["attn_impl"] = args.attn_impl
    if args.attn_splits:
        overrides["attn_splits"] = args.attn_splits
    if args.no_graph:
        overrides["use_cuda_graph"] = False
    CONFIG_MAP["ENGINE_OVERRIDES"] = overrides
    torch.manual_seed(1)              # LP: every rank decodes the SAME sequence
    prompt_host = torch.randint(3, shape["vocab"], (1, P)).pin_memory()
    prompt_list = prompt_host[0].tolist()
    eng = get_engine(model, max_total_len=P + args.max_new)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also captures the steady-step CUDA graph)
    if args.do_sample:
        def run_once():         # verification on device (lade_sample_verify, Philox)
            return eng.generate(prompt_list, args.max_new, rng=random.Random(0), sampling={"temperature": 0.8, "seed": 2})
        gen_kwargs = dict(do_sample=True, temperature=0.8, top_k=0, top_p=1.0)
        config["workload"] = config["workload"].replace("greedy", "sampling temp=0.8")
    else:
        def run_once():
            return eng.generate(prompt_list, args.max_new, rng=random.Random(0))
        gen_kwargs = dict(do_sample=False)
    for _ in range(max(args.warmup, 1)):
        out_warm = run_once()
    barrier()

    # ---- device-timed: prompt already with the engine
    sampler = ClockSampler(local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    toks = steps = 0
    launches0 = eng.launches
    with sampler:
        barrier()
        if args.cuda_profiler_range:
            torch.cuda.profiler.start()
        e0.record()
        for _ in range(args.steps):
            out = run_once()
            toks += len(out) - P
            steps += eng.last_steps
        e1.record()
        barrier()
        if args.cuda_profiler_range:
            torch.cuda.profiler.stop()
        dev_ms = e0.elapsed_time(e1)
        launches = eng.launches - launches0
        # ---- end to end through the plugin surface: pinned host prompt -> generate() -> host ids
        for _ in range(2):                                     # the HF generate() path has its own first-call costs
            model.generate(prompt_host.to(dev), attention_mask=torch.ones(1, P, dtype=torch.long, device=dev),
                           max_new_tokens=8, **gen_kwargs)
        engine_s = [0.0]
        if not args.do_sample:
            inner_generate = eng.generate

            def timed_generate(*a, **k):
                t_ = time.perf_counter()
                r_ = inner_generate(*a, **k)
                engine_s[0] += time.perf_counter() - t_
                return r_
            eng.generate = timed_generate
        barrier()
        t0 = time.perf_counter()
        e2e_toks = 0
        e2e_ids = None
        for _ in range(args.steps):
            random.seed(0)
            ids = prompt_host.to(dev, non_blocking=True)
            if args.do_sample:
                torch.manual_seed(2)
            o = model.generate(ids, attention_mask=torch.ones_like(ids), max_new_tokens=args.max_new, **gen_kwargs)
            o_host = o.cpu()
            e2e_toks += o_host.shape[1] - P
            e2e_ids = o_host[0].tolist()
        barrier()
        e2e_s = time.perf_counter() - t0
        if not args.do_sample:
            eng.generate = inner_generate
    t = torch.tensor([dev_ms, e2e_s, float(toks), float(e2e_toks), float(steps), float(launches)], device=dev, dtype=torch.float64)
    lp_ids_equal = None
    if world > 1:
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms, e2e_s = mx[0].item(), mx[1].item()
        launches = sm[5].item()          # kernels launched on all ranks; tokens/steps are one shared sequence
        # ids under lookahead parallelism: every rank must hold the same sequence, and it must be the single-GPU one
        # (decoding.py:1088-1107: LP changes who verifies what, never the greedy output)
        mine = torch.tensor(out, device=dev, dtype=torch.int64)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        ranks_agree = all(bool((a_ == allr[0]).all()) for a_ in allr)
        single = None
        if rank == 0:
            from lookaheaddecoding_b200 import LookaheadEngine
            e1gpu = LookaheadEngine(model, W, N, G, max_total_len=P + args.max_new)
            single = e1gpu.generate(prompt_list, args.max_new, rng=random.Random(0))
            e1gpu.close()
            del e1gpu
            n_same = next((i for i in range(min(len(single), len(out))) if single[i] != out[i]), min(len(single), len(out)))
            lp_ids_equal = {"ranks_agree": ranks_agree, "equal_to_single_gpu": single == out,
                            "equal_prefix_tokens": n_same - P, "compared_tokens": len(out) - P}
            if single != out and n_same < min(len(single), len(out)):
                # a rank forwards 1/N of the window rows, so its GEMMs run at another M and round differently: judge the
                # first divergence on the model's own logits (stock HF forward of the common prefix, same weights)
                with torch.no_grad():
                    lg = model(torch.tensor([out[:n_same]], device=dev)).logits[0, -1].float()
                import math
                top = lg.max().item()
                ulp = 2.0 ** (math.floor(math.log2(abs(top))) - 7)
                lp_ids_equal["first_divergence"] = {
                    "index": n_same - P, "lp_token_below_top_ulps": round((top - lg[out[n_same]].item()) / ulp, 2),
                    "single_gpu_token_below_top_ulps": round((top - lg[single[n_same]].item()) / ulp, 2),
                    "how": "both candidates judged on the stock HF forward of the common prefix (bf16 ulps of the top logit)"}
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "output_ids.npy"), np.asarray(out, dtype=np.float64))
        np.save(os.path.join(args.dump_outputs, "e2e_output_ids.npy"), np.asarray(e2e_ids, dtype=np.float64))
    clocks = sampler.summary()
    roof = attn_roofline(eng, shape)

    # ---- the unmodified reference on the same GPU and weights: timing + token-id parity
    ref_cuda = parity = ar = None
    extras = {}
    if world == 1 and not args.do_sample and not args.no_reference_cuda:
        try:
            from baseline import parity as PAR
            from baseline import ref_loader as RL
            if not RL.reference_available():
                ref_cuda = {"unavailable": "baseline/_ref not present"}
            else:
                ref_model = PAR.reference_model_sharing_weights(model, shape)
                ref_cuda, ref_ids = reference_cuda_eager(ref_model, shape, W, N, G, prompt_list, args.max_new)
                parity = PAR.compare_ids(lambda p_, n_: eng.generate(p_, n_, rng=random.Random(0)), ref_ids, P, ref_model)
                parity["e2e_ids_equal_device_timed_ids"] = (e2e_ids == out)
                del ref_model
                torch.cuda.empty_cache()
        except Exception as ex:   # reporting only
            ref_cuda = ref_cuda or {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
            parity = parity or {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}

    # ---- plain autoregressive series (BASELINE.md "AR"; SURVEY 8(d)(iii)): at 1.0 accepted tokens/step lookahead is
    # pure overhead, and only this line shows it.  Ours: the same engine with the smallest window (W=1, N=3, G=0: two
    # rows per step, no verification).  Reference side: stock HF generate() on the same model (USE_LADE=0 -- what the
    # reference's greedy_search_proxy falls back to, lade/decoding.py:15-26).
    if world == 1 and not args.do_sample and not args.no_extras:
        try:
            from lookaheaddecoding_b200 import LookaheadEngine
            ar_eng = LookaheadEngine(model, 1, 3, 0, max_total_len=P + args.max_new)
            ar_run = lambda: ar_eng.generate(prompt_list, args.max_new, rng=random.Random(0))
            ar_run()
            a_toks, a_steps, a_ms = time_generates(ar_run, 2, P, ar_eng, dev)
            ar_out = ar_run()
            ar_eng.close()
            del ar_eng
            os.environ["USE_LADE"] = "0"
            ids = prompt_host.to(dev)
            am_ = torch.ones_like(ids)
            model.generate(ids, attention_mask=am_, max_new_tokens=8, do_sample=False)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            hf_out = model.generate(ids, attention_mask=am_, max_new_tokens=args.max_new, do_sample=False)
            torch.cuda.synchronize()
            hf_s = time.perf_counter() - t0
            os.environ["USE_LADE"] = "1"
            hf_list = hf_out[0].tolist()
            same = next((i for i in range(P, min(len(hf_list), len(out))) if hf_list[i] != out[i]), min(len(hf_list), len(out)))
            ar = {"ours_min_window": {"value": round(a_toks / (a_ms * 1e-3), 2), "unit": "tokens/s",
                                      "ms_per_decode_step": round(a_ms / a_steps, 4), "config": "W=1 N=3 G=0 (2 rows/step)",
                                      "ids_equal_lookahead_ids": ar_out == out},
                  "hf_generate": {"value": round((hf_out.shape[1] - P) / hf_s, 2), "unit": "tokens/s",
                                  "ms_per_decode_step": round(1e3 * hf_s / max(hf_out.shape[1] - P, 1), 3),
                                  "config": "transformers generate(), USE_LADE=0, same model object",
                                  "ids_equal_prefix_vs_lookahead": same - P},
                  "lookahead_over_own_ar": round((toks / (dev_ms * 1e-3)) / (a_toks / (a_ms * 1e-3)), 3)}
        except Exception as ex:
            os.environ["USE_LADE"] = "1"
            ar = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}

    # ---- BASELINE.json configs[2] (7B sampling) and configs[3] (13B W20 N7 G20) in the same run
    if world == 1 and args.workload == "7b" and not args.do_sample and not args.no_extras and args.weights == "random":
        for key, kw in (("7b_sampling", dict(name="7b", do_sample=True, model=model)), ("13b", dict(name="13b")),
                        ("7b_fp16", dict(name="7b", dtype=torch.float16))):     # the dtype of the reference's README / minimal.py
            try:
                extras[key] = extra_workload(args=args, dev=dev, **kw)
            except Exception as ex:
                extras[key] = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
        # ---- a workload on which lookahead DOES something (VERDICT r1 #6): zero o_proj/down_proj in place -> the next
        # token is a function of the last one, text turns periodic, n-grams hit.  Both arms, same weights.
        try:
            with torch.no_grad():
                for layer in model.model.layers:
                    layer.self_attn.o_proj.weight.zero_()
                    layer.mlp.down_proj.weight.zero_()
            run_once()
            c_toks, c_steps, c_ms = time_generates(run_once, 3, P, eng, dev)
            cyc = {"weights": "o_proj/down_proj zeroed (periodic text; bytes/FLOPs per step unchanged)",
                   "value": round(c_toks / (c_ms * 1e-3), 2), "unit": "tokens/s",
                   "accepted_tokens_per_step": round(c_toks / c_steps, 3), "ms_per_decode_step": round(c_ms / c_steps, 4),
                   "kv_compact_steps": sum(1 for r_ in eng.last_records if r_.max_hit > 0)}
            from baseline import parity as PAR
            from baseline import ref_loader as RL
            if RL.reference_available():
                ref_model = PAR.reference_model_sharing_weights(model, shape)
                rc, rids = reference_cuda_eager(ref_model, shape, W, N, G, prompt_list, args.max_new)
                cyc["reference_cuda_eager"] = {k_: rc[k_] for k_ in ("value", "accepted_tokens_per_step", "ms_per_decode_step", "decode_steps")}
                pr = PAR.compare_ids(lambda p_, n_: eng.generate(p_, n_, rng=random.Random(0)), rids, P, ref_model, max_divergences=16)
                cyc["parity"] = {k_: pr[k_] for k_ in ("exact", "ok", "exact_prefix_tokens", "compared_tokens", "n_divergences",
                                                       "worst_candidate_below_top_ulps")}
                del ref_model
            extras["7b_periodic"] = cyc
        except Exception as ex:
            extras["7b_periodic"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}

    cb = None
    if not args.no_cpu_baseline and world == 1:      # host-core baseline: rank 0 at N=1 only, bounded sample
        try:
            cb = reference_cpu(shape, W, N, G, P, args.max_new, usable_cores(), timed_steps=8, warm_steps=2, budget_s=60.0)
        except Exception as ex:  # the baseline is reporting only; never hide the GPU numbers
            cb = {"value": None, "unit": "tokens/s", "cores": usable_cores(), "kind": "reference", "sample": f"failed: {ex}"}
    value = toks / (dev_ms * 1e-3)
    line = {
        "metric": metric, "value": round(value, 2), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(dev_ms / args.steps, 3), "higher_is_better": True,
        "scaling": "weak" if world == 1 else "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config,
        "accepted_tokens_per_step": round(toks / steps, 3), "decode_steps": int(steps),
        "ms_per_decode_step": round(dev_ms / steps, 4),
        "e2e": {"value": round(e2e_toks / e2e_s, 2), "unit": "tokens/s", "h2d_bytes_per_step": P * 8,
                "d2h_bytes_per_step": (P + args.max_new) * 8 + int(steps / args.steps) * 48 * 4,
                "outside_engine_ms_per_generate": None if args.do_sample else
                round(1e3 * (e2e_s - engine_s[0]) / args.steps, 2)},
        "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cb, "reference_cuda_eager": ref_cuda,
        "parity": parity, "ar": ar, "lp_ids": lp_ids_equal, "more_configs": extras or None,
        "clocks": clocks,
        "attn_impl": eng.attn_impl, "attn_splits": eng.attn_splits, "cuda_graph": eng.use_cuda_graph,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
