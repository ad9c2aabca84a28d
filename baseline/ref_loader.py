"""CHECKER / BASELINE INFRASTRUCTURE ONLY -- loader for the *unmodified* reference (hao-ai-lab/LookaheadDecoding).

This module imports the reference's ``lade/decoding.py`` and ``lade/models/modeling_llama.py`` as they are --
from ``baseline/_ref`` (the offline pip install of the reference: git-ignored, travels to the GPU box) or, in the
build container, from ``/root/reference`` (never copied into this repo) -- under the transformers/torch versions of
this image, using the five small shims of SURVEY.md App. C.  Users:

  * ``tests/golden/gen_golden.py`` runs the reference's own ``jacobi_greedy_search_multilevel`` /
    ``jacobi_sample_multilevel`` (``/root/reference/lade/decoding.py:697`` / ``:137``) and
    ``j_make_causal_mask_multilevel`` (``/root/reference/lade/models/modeling_llama.py:115``) to
    produce the committed golden fixtures that pin ``oracle/``;
  * CPU tests that are skipped when ``/root/reference`` is absent (e.g. on the GPU box).

  * ``bench.py``: the ``--impl reference`` arm (the unmodified reference on the host cores), the
    ``reference_cuda_eager`` leg (the same loop on the GPU: the denominator of the north star's 1.8x) and the
    ``parity`` field (token ids of our engine against the reference's on the same GPU, ``baseline/parity.py``);
  * ``tests/golden/gen_golden_gpu_parity.py``: the reference's GPU runs that the ``-m gpu`` parity tests
    (``tests/test_gpu_vs_reference.py``) are judged against.

Nothing in the product package may import this file.  ``/root/reference`` does not exist on the GPU box: there the
root is ``baseline/_ref`` (``default_reference_root()``).
"""
from __future__ import annotations

import os
import sys
import types

_HERE = os.path.dirname(os.path.abspath(__file__))


def default_reference_root() -> str:
    """LADE_REFERENCE_ROOT, else baseline/_ref (pip install --target, travels with gpurun), else /root/reference."""
    env = os.environ.get("LADE_REFERENCE_ROOT")
    if env:
        return env
    cand = os.path.join(_HERE, "_ref")
    if os.path.isfile(os.path.join(cand, "lade", "decoding.py")):
        return cand
    return "/root/reference"


REFERENCE_ROOT = default_reference_root()


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "lade", "decoding.py"))


_loaded = None


def load_reference():
    """Import the untouched reference modules; returns (decoding, modeling_llama)."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not reference_available():
        raise RuntimeError(f"reference not present at {REFERENCE_ROOT}")

    import transformers
    import transformers.utils.import_utils as iu
    import transformers.generation.utils as gu

    # shim 1: removed helper probed at import (modeling_llama.py:50)
    if not hasattr(iu, "is_torch_fx_available"):
        iu.is_torch_fx_available = lambda: False
    if not hasattr(transformers.utils, "is_torch_fx_available"):
        transformers.utils.is_torch_fx_available = lambda: False
    # shim 2: annotation-only names imported by decoding.py:8
    for name in ("GreedySearchOutput", "SampleOutput"):
        if not hasattr(gu, name):
            setattr(gu, name, type(name, (), {}))

    # shim 3: import the two hot-path modules WITHOUT executing lade/__init__.py (whose utils.py
    # touches GenerationMixin.greedy_search, gone in transformers 5.x).
    import importlib.util

    # private package names: this repo ships its own `lade` alias package, which must not be shadowed
    pkg = types.ModuleType("lade_reference")
    pkg.__path__ = [os.path.join(REFERENCE_ROOT, "lade")]
    sys.modules.setdefault("lade_reference", pkg)
    models_pkg = types.ModuleType("lade_reference.models")
    models_pkg.__path__ = [os.path.join(REFERENCE_ROOT, "lade", "models")]
    sys.modules.setdefault("lade_reference.models", models_pkg)

    def _load(modname, relpath):
        if modname in sys.modules:
            return sys.modules[modname]
        spec = importlib.util.spec_from_file_location(modname, os.path.join(REFERENCE_ROOT, relpath))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[modname] = mod
        spec.loader.exec_module(mod)
        return mod

    decoding = _load("lade_reference.decoding", "lade/decoding.py")
    modeling = _load("lade_reference.models.modeling_llama", "lade/models/modeling_llama.py")

    # shim 5: the loop calls self._update_model_kwargs_for_generation (HF mixin)
    from transformers import GenerationMixin

    if not hasattr(modeling.LlamaForCausalLM, "_update_model_kwargs_for_generation"):
        modeling.LlamaForCausalLM._update_model_kwargs_for_generation = (
            GenerationMixin._update_model_kwargs_for_generation
        )
    _loaded = (decoding, modeling)
    return _loaded


def make_llama_config(hidden=256, layers=2, heads=2, kv_heads=None, inter=688, vocab=32000,
                      max_pos=2048, rope_theta=10000.0, eps=1e-5):
    from transformers import LlamaConfig

    cfg = LlamaConfig(
        hidden_size=hidden, num_hidden_layers=layers, num_attention_heads=heads,
        num_key_value_heads=kv_heads or heads, intermediate_size=inter, vocab_size=vocab,
        max_position_embeddings=max_pos, rms_norm_eps=eps, tie_word_embeddings=False,
        attention_bias=False, hidden_act="silu",
    )
    cfg._attn_implementation = "eager"
    # shim 4: attributes the 4.36-era code reads (modeling_llama.py:416,432)
    object.__setattr__(cfg, "rope_theta", rope_theta)
    object.__setattr__(cfg, "rope_scaling", None)
    object.__setattr__(cfg, "pretraining_tp", 1)
    object.__setattr__(cfg, "attention_dropout", 0.0)
    return cfg


def build_reference_model(cfg, seed=0, dtype=None):
    """Random-init reference LlamaForCausalLM (normal(0, initializer_range))."""
    import torch
    from transformers import GenerationConfig

    _, modeling = load_reference()
    torch.manual_seed(seed)
    model = modeling.LlamaForCausalLM(cfg)
    # deterministic re-init independent of HF's lazy init machinery
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in sorted(model.named_parameters()):
            if p.dim() >= 2:
                p.copy_(torch.randn(p.shape, generator=g) * cfg.initializer_range)
            else:
                p.fill_(1.0)
    model.eval()
    if dtype is not None:
        model = model.to(dtype)
    model.generation_config = GenerationConfig(pad_token_id=0, eos_token_id=None)
    return model


def run_reference_greedy(model, prompt_ids, max_new, lade_cfg, py_seed=0, eos_token_id=None):
    """Run the reference's own greedy lookahead loop; returns LongTensor [1, P+new]."""
    import random
    import torch
    from transformers import StoppingCriteriaList, MaxLengthCriteria

    decoding, _ = load_reference()
    decoding.CONFIG_MAP.clear()
    decoding.CONFIG_MAP.update(lade_cfg)
    decoding.CONFIG_MAP.setdefault("log", [])
    random.seed(py_seed)
    P = prompt_ids.shape[1]
    with torch.no_grad():
        out = decoding.jacobi_greedy_search_multilevel(
            model, prompt_ids,
            stopping_criteria=StoppingCriteriaList([MaxLengthCriteria(P + max_new)]),
            attention_mask=torch.ones_like(prompt_ids), use_cache=True,
            return_dict_in_generate=False, output_attentions=False,
            output_hidden_states=False, output_scores=False,
            pad_token_id=0, eos_token_id=eos_token_id,
        )
    return out
