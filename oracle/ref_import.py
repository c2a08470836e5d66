"""Import the UNMODIFIED reference classes from a checkout of the reference project ($MAPPERATORINATOR_REFERENCE).

TEST INFRASTRUCTURE. Used only by `oracle/make_golden.py` (fixture generation); the tests read the fixtures.
Follows the stub recipe of SURVEY.md §8(c): third-party modules that are not installed here
(hydra, omegaconf, slider, pydub, peft, accelerate, ...) are replaced by MagicMock modules so that
the reference's own numerics (Mapperatorinator, model_generate, DiT, create_diffusion) import unmodified.
"""
from __future__ import annotations

import importlib.machinery
import os
import sys
import types
from unittest.mock import MagicMock

REFERENCE_ROOT = os.environ.get("MAPPERATORINATOR_REFERENCE", "/root/reference")

_STUBS = [
    "slider", "slider.beatmap", "slider.mod", "slider.curve", "slider.position", "pydub",
    "hydra", "hydra.core", "hydra.core.config_store", "omegaconf", "rosu_pp_py", "peft",
    "accelerate", "accelerate.utils", "accelerate.logging", "matplotlib", "matplotlib.pyplot",
    "nnAudio", "wandb",
]


def install_stubs() -> None:
    import transformers  # noqa: F401  (must be imported before the stubs, SURVEY §8c.1)
    for name in _STUBS:
        if name in sys.modules:
            continue
        try:
            __import__(name)
            continue
        except Exception:
            pass
        m = MagicMock(name=name)
        m.__spec__ = importlib.machinery.ModuleSpec(name, None)
        m.__path__ = []
        sys.modules[name] = m
    sys.modules["omegaconf"].MISSING = "???"
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


def patch_whisper_config(d_model=768, layers=12, heads=12, ffn=3072):
    """`MapperatorinatorConfig.__init__` fetches openai/whisper-small from the hub
    (configuration_mapperatorinator.py:69-70); there is no network, so pin the dims."""
    from transformers import WhisperConfig

    def _fp(cls, name, **kw):
        return cls(d_model=d_model, encoder_layers=layers, decoder_layers=layers,
                   encoder_attention_heads=heads, decoder_attention_heads=heads,
                   encoder_ffn_dim=ffn, decoder_ffn_dim=ffn)

    WhisperConfig.from_pretrained = classmethod(_fp)


def reference_slider_path():
    """The reference's `SliderPath` class, loaded from its two numpy-only source files (slider_path.py, path_approximator.py)
    without importing the rest of the `osuT5.osuT5.inference` package."""
    import importlib.util
    base = os.path.join(REFERENCE_ROOT, "osuT5", "osuT5", "inference")
    pkg = types.ModuleType("_ref_inference")
    pkg.__path__ = [base]
    sys.modules["_ref_inference"] = pkg
    for name in ("path_approximator", "slider_path"):
        spec = importlib.util.spec_from_file_location(f"_ref_inference.{name}", os.path.join(base, f"{name}.py"))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[f"_ref_inference.{name}"] = mod
        spec.loader.exec_module(mod)
    return sys.modules["_ref_inference.slider_path"].SliderPath
