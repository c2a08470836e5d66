"""Build the UNMODIFIED reference models (needs a checkout of the reference project, see oracle/ref_import.py).

TEST INFRASTRUCTURE.  Used by oracle/make_golden.py to pin the oracle.
"""
from __future__ import annotations

import os
import re
import sys

import torch

from . import ref_import


def v29_train_config():
    """TrainConfig with the `data:`/`model:` sections of configs/train/default.yaml + v29.yaml +
    configs/model/default.yaml + whisper_small.yaml applied (Hydra itself is not installed)."""
    import yaml
    ref_import.install_stubs()
    from osuT5.osuT5.config import TrainConfig
    from osuT5.osuT5.event import ContextType
    root = ref_import.REFERENCE_ROOT
    tc = TrainConfig()

    def apply(obj, d):
        for k, v in d.items():
            if not hasattr(obj, k):
                continue
            cur = getattr(obj, k)
            if isinstance(v, dict) and not isinstance(cur, (dict, type(None))) and hasattr(cur, "__dataclass_fields__"):
                apply(cur, v)
            else:
                setattr(obj, k, v)

    def ctx(v):
        m = re.match(r"\$\{context_type:(\w+)\}", v) if isinstance(v, str) else None
        return ContextType(m.group(1)) if m else v

    for f in ("configs/train/default.yaml", "configs/train/v29.yaml"):
        y = yaml.safe_load(open(os.path.join(root, f)))
        data = y.get("data", {})
        if "context_types" in data:
            data["context_types"] = [{k: [ctx(x) for x in v] for k, v in c.items()} for c in data["context_types"]]
        apply(tc.data, data)
    for f in ("configs/model/default.yaml", "configs/model/whisper_small.yaml"):
        y = yaml.safe_load(open(os.path.join(root, f)))
        y.pop("defaults", None)
        apply(tc.model, y)
    return tc


def reference_tokenizer(tc=None, n_mappers: int = 8, n_descriptors: int = 8):
    """The reference `Tokenizer` at v29 data settings.  The MMRS metadata table (mapper ids / descriptor names) is a
    dataset artefact that is not available; it only widens the INPUT-only vocabulary tail, so it is stubbed with
    `n_mappers` / `n_descriptors` classes."""
    ref_import.install_stubs()
    from osuT5.osuT5.tokenizer import Tokenizer
    tc = tc or v29_train_config()

    class _Tok(Tokenizer):
        def _get_metadata(self, args):
            return None

        def _init_mapper_idx(self, args):
            self.mapper_idx = {i: i for i in range(n_mappers)}
            self.num_mapper_classes = n_mappers

        def _init_descriptor_idx(self, args):
            self.descriptor_idx = {f"d{i}": i for i in range(n_descriptors)}
            self.num_descriptor_classes = n_descriptors

    return _Tok(tc)


def reference_model(cfg, tok=None, tc=None, mel_impl: str = "torchaudio"):
    """`_get_model` (osuT5/osuT5/utils/model_utils.py:102-114) at the dims of `cfg` (a mapperatorinator_b200.ModelConfig);
    returns (model.eval(), tokenizer, train_config).  `mel_impl='nnAudio'` plugs the oracle's restated nnAudio transform in
    place of the (absent) package so the rest of the reference graph runs unmodified."""
    ref_import.install_stubs()
    ref_import.patch_whisper_config(cfg.d_model, cfg.encoder_layers, cfg.heads, cfg.ffn_dim)
    from osuT5.osuT5.utils.model_utils import _get_model
    tc = tc or v29_train_config()
    tc.model.spectrogram.implementation = "torchaudio" if mel_impl == "torchaudio" else "nnAudio"
    tc.model.spectrogram.n_mels = cfg.mel.n_mels
    tc.model.spectrogram.log_scale = cfg.mel.log_scale
    tc.model.spectrogram.f_min = cfg.mel.f_min
    tc.model.spectrogram.pad_mode = cfg.mel.pad_mode
    tok = tok or reference_tokenizer(tc)
    if mel_impl == "nnAudio":
        from . import mel as mel_oracle

        class _NNAudioMel(torch.nn.Module):
            def __init__(self, sr, n_fft, n_mels, hop_length, center, fmin, fmax, pad_mode):
                super().__init__()
                from mapperatorinator_b200.config import MelConfig
                self.cfg = MelConfig("nnAudio", False, sr, n_fft, n_mels, hop_length, fmin, fmax, pad_mode)

            def forward(self, x):
                return mel_oracle.nnaudio_melspectrogram(x, self.cfg)

        sys.modules["nnAudio"].features.MelSpectrogram = _NNAudioMel
    model = _get_model(tc, tok, torch.float32, "sdpa")
    model.generation_config.disable_compile = True
    return model.eval(), tok, tc


def load_state_dict_into_reference(model, sd):
    """Copy an `init_model_state_dict` dict into the reference model (strict on every key the dict names)."""
    ref_sd = model.state_dict()
    for k, v in sd.items():
        assert k in ref_sd, k
        assert tuple(ref_sd[k].shape) == tuple(v.shape), (k, ref_sd[k].shape, v.shape)
    missing = model.load_state_dict(sd, strict=False)
    return missing


def reference_dit(dcfg):
    ref_import.install_stubs()
    from osu_diffusion.utils.models import DiT
    m = DiT(in_channels=dcfg.in_channels, context_size=dcfg.context_size, hidden_size=dcfg.hidden, depth=dcfg.depth,
            num_heads=dcfg.heads, mlp_ratio=dcfg.mlp_ratio, class_size=dcfg.class_size)
    return m.eval()
