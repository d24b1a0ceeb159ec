"""TEST INFRASTRUCTURE ONLY — runtime compatibility shim for the *unmodified* reference.

Lets `/root/reference/self_speculation/*.py` (written against transformers ~4.45, pinned
4.50.0 in `/root/reference/requirements.txt:4`) import and run under the transformers 5.5
installed in this image, WITHOUT editing or copying any reference file.  Used only by
`oracle/gen_golden.py` (to produce `tests/golden/*.json`).

What is patched at run time (SURVEY.md Appendix B):
  * `colorama` is not installed            -> stub module (only used for TTY colours,
    `/root/reference/self_speculation/self_speculation_generator.py:10,160,210,212`).
  * `DynamicCache.from_legacy_cache / to_legacy_cache / __getitem__` no longer exist
    (call sites `/root/reference/self_speculation/llama_model_utils.py:169,203,229,263,308,346,385`).
  * `LlamaDecoderLayer.forward` now wants `past_key_values=` + `position_embeddings=` and
    returns a bare tensor; the reference passes `past_key_value=`/`position_ids=` and unpacks
    `(hidden, cache)` (call sites `llama_model_utils.py:193-201,253-261,354-362,375-383`).

Nothing in the product package imports this file.
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_ROOT = os.environ.get("LSK_REFERENCE_ROOT", "/root/reference")

_installed = False


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "self_speculation"))


def install() -> None:
    """Idempotently patch the process so the reference modules import."""
    global _installed
    if _installed:
        return
    if not reference_available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")

    import torch  # noqa: F401
    import transformers
    from transformers.cache_utils import DynamicCache
    from transformers.models.llama import modeling_llama

    # -- colorama stub ---------------------------------------------------------------
    if "colorama" not in sys.modules:
        class _Blank:
            def __getattr__(self, _name):
                return ""
        stub = types.ModuleType("colorama")
        stub.Fore = _Blank()
        stub.Style = _Blank()
        stub.Back = _Blank()
        sys.modules["colorama"] = stub

    # -- legacy KV tuple <-> DynamicCache ----------------------------------------------
    if not hasattr(DynamicCache, "from_legacy_cache"):
        def from_legacy_cache(cls, past_key_values=None):
            cache = cls()
            if past_key_values is not None:
                for idx, kv in enumerate(past_key_values):
                    cache.update(kv[0], kv[1], idx)
            return cache
        DynamicCache.from_legacy_cache = classmethod(from_legacy_cache)

    if not hasattr(DynamicCache, "to_legacy_cache"):
        def to_legacy_cache(self):
            out = []
            for layer in self.layers:
                if not getattr(layer, "is_initialized", False):
                    break
                out.append((layer.keys, layer.values))
            return tuple(out)
        DynamicCache.to_legacy_cache = to_legacy_cache

    if "__getitem__" not in DynamicCache.__dict__:
        def _getitem(self, idx):
            if idx < len(self.layers) and getattr(self.layers[idx], "is_initialized", False):
                return (self.layers[idx].keys, self.layers[idx].values)
            return None
        DynamicCache.__getitem__ = _getitem

    # -- decoder layer calling convention ----------------------------------------------
    layer_cls = modeling_llama.LlamaDecoderLayer
    if not getattr(layer_cls, "_lsk_shimmed", False):
        original_forward = layer_cls.forward
        rope_cache: dict = {}

        def legacy_forward(self, hidden_states, attention_mask=None, position_ids=None,
                           past_key_value=None, output_attentions=False, use_cache=False,
                           padding_mask=None, **kwargs):
            if kwargs.get("position_embeddings") is not None or "past_key_values" in kwargs:
                # native transformers-5 call (e.g. model(input_ids=...)): leave it untouched
                return original_forward(self, hidden_states, attention_mask=attention_mask,
                                        position_ids=position_ids, use_cache=use_cache, **kwargs)
            cfg = self.self_attn.config
            rope = rope_cache.get(id(cfg))
            if rope is None:
                rope = modeling_llama.LlamaRotaryEmbedding(config=cfg)
                rope_cache[id(cfg)] = rope
            pos_emb = rope(hidden_states, position_ids)
            out = original_forward(
                self, hidden_states, attention_mask=attention_mask, position_ids=position_ids,
                past_key_values=past_key_value, use_cache=use_cache,
                position_embeddings=pos_emb)
            if isinstance(out, tuple):
                out = out[0]
            return out, past_key_value

        layer_cls.forward = legacy_forward
        layer_cls._lsk_shimmed = True

    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    _installed = True
    del transformers


def load_reference():
    """Return the reference's own (unmodified) modules as a namespace."""
    install()
    from self_speculation import autoregressive_generator, generator_base
    from self_speculation import llama_model_utils, self_speculation_generator
    return types.SimpleNamespace(
        generator_base=generator_base,
        llama_model_utils=llama_model_utils,
        self_speculation_generator=self_speculation_generator,
        autoregressive_generator=autoregressive_generator,
    )
