"""Host-side mirror of the reference's plugin surface (lade/utils.py, lade/decoding.py proxies): CPU-only checks.

No compute is launched; these tests cover configuration plumbing, the reversible generate() patch, the loud
failures the drop-in promises (no CPU fallback, no silent oracle path) and small host helpers."""
import io
import os
import re
import contextlib

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under the product packages may import it."""
    pat = re.compile(r"^\s*(from\s+oracle\b|import\s+oracle\b|from\s+\.\.?oracle\b)", re.M)
    for pkg in ("lookaheaddecoding_b200", "lade"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, pkg)):
            for f in files:
                if f.endswith(".py"):
                    src = open(os.path.join(dirpath, f)).read()
                    assert not pat.search(src), f"{pkg}/{f} imports oracle"
                    assert "/root/reference" not in src, f"{pkg}/{f} reads the reference checkout"


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from lookaheaddecoding_b200 import _cabi, build
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(build, "LIB_PATH", str(tmp_path / "liblade_sm100.so"))
    monkeypatch.setattr(build, "is_fresh", lambda: False)

    def no_nvcc(*a, **k):
        raise RuntimeError("nvcc not found")

    monkeypatch.setattr(build, "build", no_nvcc)
    with pytest.raises(_cabi.LadeError, match="missing and could not be built"):
        _cabi.load()
    with pytest.raises(_cabi.LadeError, match="no CPU fallback"):
        _cabi.load(build_if_missing=False)


def test_cpu_model_is_rejected_not_emulated():
    from transformers import LlamaConfig, LlamaForCausalLM
    from lookaheaddecoding_b200 import LookaheadEngine, LadeError
    cfg = LlamaConfig(hidden_size=256, num_hidden_layers=1, num_attention_heads=2, num_key_value_heads=2,
                      intermediate_size=688, vocab_size=512, max_position_embeddings=256)
    model = LlamaForCausalLM(cfg).to(torch.bfloat16)
    with pytest.raises(LadeError):
        LookaheadEngine(model, 5, 3, 3)


def test_config_lade_populates_config_map_like_the_reference():
    import lade
    from lookaheaddecoding_b200.decoding import CONFIG_MAP
    CONFIG_MAP.clear()
    lade.config_lade(LEVEL=7, WINDOW_SIZE=20, GUESS_SET_SIZE=20, DEBUG=1, POOL_FROM_PROMPT=True, USE_FLASH=True,
                     ALWAYS_FWD_ONE=1, SPLIT_FLAG=0)
    assert CONFIG_MAP["LEVEL"] == 7 and CONFIG_MAP["WINDOW_SIZE"] == 20 and CONFIG_MAP["GUESS_SET_SIZE"] == 20
    assert CONFIG_MAP["POOL_FROM_PROMPT"] is True and CONFIG_MAP["USE_FLASH"] is True and CONFIG_MAP["log"] == []
    assert "DIST_WORKERS" not in CONFIG_MAP                      # only set for > 1 workers (lade/utils.py:28)
    CONFIG_MAP["log"] = [(10, 4), (6, 4)]
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        lade.log_history()
    assert "OVERALL GEN:  16" in buf.getvalue() and "STEPS:  8" in buf.getvalue() and "2.0" in buf.getvalue()
    with contextlib.redirect_stdout(io.StringIO()):
        lade.log_history(clear=True)
    assert CONFIG_MAP["log"] == []


def test_save_log_round_trip(tmp_path):
    import lade
    from lookaheaddecoding_b200.decoding import CONFIG_MAP
    CONFIG_MAP["log"] = [(5, 2)]
    path = str(tmp_path / "log.pt")
    lade.save_log(path)
    assert torch.load(path) == [(5, 2)]


def test_generate_patch_is_reversible():
    from transformers import GenerationMixin
    import lade
    from lookaheaddecoding_b200.decoding import sample_entry_proxy
    original = GenerationMixin._sample
    lade.augment_generate()
    try:
        assert GenerationMixin._sample is sample_entry_proxy
        lade.augment_generate()                                   # idempotent: the original is not lost
        assert GenerationMixin._sample is sample_entry_proxy
    finally:
        lade.restore_generate()
    assert GenerationMixin._sample is original


def test_max_length_resolution():
    from transformers import MaxLengthCriteria, StoppingCriteriaList
    from lookaheaddecoding_b200.decoding import _max_length_from
    from lookaheaddecoding_b200 import LadeError
    crit = StoppingCriteriaList([MaxLengthCriteria(40), MaxLengthCriteria(32)])
    assert _max_length_from(crit, None, 10) == 32
    assert _max_length_from(None, 5, 10) == 15
    assert _max_length_from(crit, 5, 10) == 15
    with pytest.raises(LadeError):
        _max_length_from(None, None, 10)


def test_split_warpers_and_their_validation():
    from transformers.generation.logits_process import (LogitsProcessorList, MinLengthLogitsProcessor,
                                                        RepetitionPenaltyLogitsProcessor, TemperatureLogitsWarper,
                                                        TopKLogitsWarper, TopPLogitsWarper, TypicalLogitsWarper)
    from lookaheaddecoding_b200.sampling import _check_warpers, split_warpers
    from lookaheaddecoding_b200 import LadeError
    lp = LogitsProcessorList([RepetitionPenaltyLogitsProcessor(1.1), TemperatureLogitsWarper(0.8), TopKLogitsWarper(50),
                              MinLengthLogitsProcessor(3, 2), TopPLogitsWarper(0.9)])
    procs, warpers = split_warpers(lp)
    assert [type(p).__name__ for p in procs] == ["RepetitionPenaltyLogitsProcessor", "MinLengthLogitsProcessor"]
    assert [type(w).__name__ for w in warpers] == ["TemperatureLogitsWarper", "TopKLogitsWarper", "TopPLogitsWarper"]
    _check_warpers(warpers)
    with pytest.raises(LadeError, match="top_k=0.0 and top_p=1.0"):       # lade/decoding.py:377
        _check_warpers(LogitsProcessorList([TypicalLogitsWarper(0.5)]))
    assert split_warpers(None) == (LogitsProcessorList(), LogitsProcessorList())


def test_use_lade_env_gate(monkeypatch):
    from lookaheaddecoding_b200.decoding import _use_lade
    monkeypatch.delenv("USE_LADE", raising=False)
    assert not _use_lade()
    monkeypatch.setenv("USE_LADE", "0")
    assert not _use_lade()
    monkeypatch.setenv("USE_LADE", "1")
    assert _use_lade()


def test_config_lade_joins_lookahead_workers_over_gloo(tmp_path):
    """config_lade(DIST_WORKERS=2, backend='gloo') under torchrun: process group joined, LOCAL_RANK recorded
    (lade/utils.py:28-33), get_device()/distributed() answer like lade/lade_distributed.py."""
    import subprocess
    import sys
    script = tmp_path / "join.py"
    script.write_text(
        "import os, sys\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import torch.distributed as dist\n"
        "import lade\n"
        "from lookaheaddecoding_b200.decoding import CONFIG_MAP\n"
        "lade.config_lade(LEVEL=5, WINDOW_SIZE=15, GUESS_SET_SIZE=15, DIST_WORKERS=2, backend='gloo')\n"
        "assert lade.distributed() and lade.get_device() == int(os.environ['LOCAL_RANK'])\n"
        "assert CONFIG_MAP['DIST_WORKERS'] == 2 and CONFIG_MAP['LEVEL'] == 5 and CONFIG_MAP['log'] == []\n"
        "dist.barrier()\n"
        "print('LP_JOIN_OK') if dist.get_rank() == 0 else None\n"
        "dist.destroy_process_group()\n")
    # host only: with a GPU visible every worker selects the device of its LOCAL_RANK, which a one-GPU machine lacks
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29581", str(script)],
                         capture_output=True, text=True, timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert res.returncode == 0 and "LP_JOIN_OK" in res.stdout, res.stderr[-1500:]


def test_extra_stopping_criteria_are_found_and_evaluated_on_the_host():
    """MaxLength / EOS criteria are handled on the device; anything else is called after every step (decoding.py:1215)."""
    from transformers import MaxLengthCriteria, StoppingCriteria, StoppingCriteriaList
    from lookaheaddecoding_b200.decoding import _extra_stopping_criteria, _host_stop_fn

    class StopOnToken(StoppingCriteria):
        def __call__(self, input_ids, scores, **kw):
            return torch.tensor([bool((input_ids[0] == 7).any())])

    crit = StoppingCriteriaList([MaxLengthCriteria(40), StopOnToken()])
    extra = _extra_stopping_criteria(crit)
    assert len(extra) == 1 and isinstance(extra[0], StopOnToken)
    assert _extra_stopping_criteria(StoppingCriteriaList([MaxLengthCriteria(4)])) == []
    assert _host_stop_fn([], torch.device("cpu"), torch.long) is None
    stop = _host_stop_fn(extra, torch.device("cpu"), torch.long)
    assert stop([1, 2, 3]) is False and stop([1, 7, 3]) is True


def test_device_sampling_is_chosen_for_the_warpers_generate_builds():
    from transformers.generation.logits_process import (LogitsProcessorList, TemperatureLogitsWarper, TopKLogitsWarper,
                                                        TopPLogitsWarper)
    from transformers.generation.logits_process import TypicalLogitsWarper
    from lookaheaddecoding_b200.sampling import device_sampling_params, device_temperature
    assert device_temperature(None) == 1.0 and device_temperature(LogitsProcessorList()) == 1.0
    assert abs(device_temperature(LogitsProcessorList([TemperatureLogitsWarper(0.8)])) - 0.8) < 1e-9
    assert device_temperature(LogitsProcessorList([TemperatureLogitsWarper(0.8), TopKLogitsWarper(50)])) is None
    assert device_sampling_params(None) == (1.0, 0, 1.0)
    assert device_sampling_params(LogitsProcessorList([TemperatureLogitsWarper(0.7), TopKLogitsWarper(50),
                                                       TopPLogitsWarper(0.9)])) == (0.7, 50, 0.9)
    assert device_sampling_params(LogitsProcessorList([TopPLogitsWarper(0.9)])) == (1.0, 0, 0.9)
    # not what generate() builds -> host-RNG compatibility loop: wrong order, other warpers, non-default keep / fill
    assert device_sampling_params(LogitsProcessorList([TopPLogitsWarper(0.9), TopKLogitsWarper(50)])) is None
    assert device_sampling_params(LogitsProcessorList([TypicalLogitsWarper(0.5)])) is None
    assert device_sampling_params(LogitsProcessorList([TopPLogitsWarper(0.9, min_tokens_to_keep=2)])) is None
    assert device_sampling_params(LogitsProcessorList([TopKLogitsWarper(50, filter_value=-1e4)])) is None


def test_eval_harness_bookkeeping_matches_the_reference_summary():
    """applications/eval_mtbench.py:384-389: THROUGHPUT1 = mean of per-call tokens/s, THROUGHPUT2 = tokens / seconds."""
    from lookaheaddecoding_b200.eval_harness import EvalReport, run_eval, synthetic_questions
    qs = synthetic_questions(2, 3, 5, vocab=100, seed=1)
    assert len(qs) == 2 and all(len(q) == 3 and all(len(t) == 5 for t in q) for q in qs)
    assert qs == synthetic_questions(2, 3, 5, vocab=100, seed=1) and qs != synthetic_questions(2, 3, 5, vocab=100, seed=2)

    class FakeModel(torch.nn.Module):          # echoes the prompt and appends max_new_tokens zeros
        def __init__(self):
            super().__init__()
            self.p = torch.nn.Parameter(torch.zeros(1))
            self.calls = []

        def generate(self, ids, max_new_tokens=0, **kw):
            self.calls.append((ids.shape[1], kw.get("do_sample"), kw.get("temperature")))
            return torch.cat([ids, torch.zeros(1, max_new_tokens, dtype=ids.dtype)], dim=1)

    m = FakeModel()
    rep = run_eval(m, qs, max_new_token=4, temperature=0.0, sync=lambda: None)
    assert rep.count_gen == 6 and rep.overall_gen == 24
    assert [c[0] for c in m.calls] == [5, 14, 23, 5, 14, 23]          # the conversation grows by turn + answer
    assert all(c[1] is False for c in m.calls)
    assert abs(rep.throughput_overall - rep.overall_gen / rep.overall_time) < 1e-9
    assert "AVERAGE THROUGHPUT1" in rep.summary() and "STAT" in rep.summary()
    m.calls.clear()
    run_eval(m, qs[:1], max_new_token=2, temperature=0.7, sync=lambda: None, max_context=12)
    assert all(c[1] is True and abs(c[2] - 0.7) < 1e-9 for c in m.calls)
    assert max(c[0] for c in m.calls) <= 10                            # context clipped to max_context - max_new_token
    r = EvalReport()
    assert r.throughput_overall == 0 and r.throughput_mean_of_calls == 0


def test_nccl_entry_points_degrade_without_a_communicator():
    import ctypes as C
    from lookaheaddecoding_b200 import _cabi
    lib = _cabi.load()
    assert lib.lade_nccl_available() in (0, 1)
    assert lib.lade_nccl_comm_destroy(None) == _cabi.LADE_EINVAL
    assert lib.lade_lp_exchange(None, None, None, None, None) == _cabi.LADE_EINVAL
    assert lib.lade_sample_verify(None, None, None, 0, 0, None, None, C.c_float(1.0), 0, C.c_float(1.0), None, None, None) == _cabi.LADE_EINVAL
    assert lib.lade_l2_prefetch(None, None, 0, 1, 16) == _cabi.LADE_EINVAL
