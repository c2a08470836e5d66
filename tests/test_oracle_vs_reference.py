"""The oracle against outputs of single UNMODIFIED reference functions at full v29 dimensions and on host-side helpers
(tests/golden/reference_pins.npz, produced by oracle/make_golden.py::make_pins_golden on the inputs of oracle/cases.py)."""
import dataclasses
import os

import numpy as np
import pytest
import torch

from oracle import cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def pins():
    return np.load(os.path.join(GOLDEN, "reference_pins.npz"))


def test_v29_dims_single_step_logits(pins):
    """One teacher-forced pass at full whisper-small dimensions: reference `Mapperatorinator.forward` vs the oracle (every 7th
    vocabulary column of the logits, and the argmax over the full rows)."""
    from mapperatorinator_b200 import MelConfig, v29_model_config
    from mapperatorinator_b200.weights import init_model_state_dict
    from oracle import whisper as wo
    cfg = dataclasses.replace(v29_model_config(), mel=MelConfig("torchaudio", n_mels=80))
    sd = init_model_state_dict(cfg, 0)
    pcm, ids = cases.v29_logits_case(cfg)
    with torch.no_grad():
        out = wo.forward_logits(sd, cfg, pcm, ids, ids.ne(0))
    ref = torch.from_numpy(pins["v29_logits_sample"])
    got = out[:, :, ::cases.PIN_LOGIT_STRIDE]
    assert got.shape == ref.shape
    assert torch.allclose(got, ref, rtol=1e-3, atol=1e-3), (got - ref).abs().max()
    assert torch.equal(out.argmax(-1), torch.from_numpy(pins["v29_logits_argmax"]))


def test_diffusion_host_helpers_match_reference(pins):
    """`timestep_embedding`, the seq_c layout of `events_to_sequence` (diffusion_pipeline.py:380-387) and the band mask loop
    (:146-148) — the host-side tensor preparation around stage (iii) — against the reference's own functions."""
    from mapperatorinator_b200 import diffusion as md
    seq_o, seq_d, types = cases.context_embedding_case()
    ref_time = torch.from_numpy(pins["timestep_embedding_time"])
    ref_dist = torch.from_numpy(pins["timestep_embedding_distance"])
    assert torch.equal(md.timestep_embedding(seq_o * 0.1, 128), ref_time)
    assert torch.equal(md.timestep_embedding(seq_d, 128), ref_dist)
    want = torch.cat([ref_time.T, ref_dist.T, torch.nn.functional.one_hot(types, 16).float().T], 0)
    assert torch.equal(md.build_context(seq_o, seq_d, types), want)
    # band mask: the reference fills it column by column (diffusion_pipeline.py:146-148)
    L, w = 50, 8
    ref_mask = torch.full((L, L), True, dtype=torch.bool)
    for i in range(L):
        ref_mask[max(0, i - w): min(L, i + w), i] = False
    assert torch.equal(md.band_attention_mask(L, w), ref_mask)


def test_v29_dims_bench_window_greedy_ids(pins, layout):
    """The bench workload's second window (50-token prompt, look-back + look-ahead processors, min_new_tokens) at FULL whisper-small
    dimensions through the unmodified reference `server.model_generate`, against the oracle: 10 greedy tokens, ids bit-exact.
    (The bench then asserts GPU ids == oracle ids on its CPU sample, closing the chain reference -> oracle -> engine at v29 dims.)"""
    from mapperatorinator_b200 import MelConfig, v29_model_config
    from mapperatorinator_b200.weights import init_model_state_dict
    from oracle import generate as go
    cfg = dataclasses.replace(v29_model_config(), mel=MelConfig("torchaudio", n_mels=80))
    sd = init_model_state_dict(cfg, 0)
    mk, gk, P = cases.bench_window_case(cfg)
    with torch.no_grad():
        ora_ids, _ = go.model_generate(sd, cfg, layout, mk, gk)
    ref_ids = torch.from_numpy(pins["bench_window_ids"])
    assert torch.equal(ref_ids, ora_ids), (ref_ids[0, P:].tolist(), ora_ids[0, P:].tolist())
