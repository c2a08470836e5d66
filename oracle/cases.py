"""Seeded input cases shared by oracle/make_golden.py (reference side) and the tests (oracle / CUDA side).

TEST INFRASTRUCTURE.  Everything here is regenerated from seeds with the CPU torch generator, so fixtures only store
reference outputs.
"""
from __future__ import annotations

import math

import torch

from mapperatorinator_b200 import MelConfig

MEL_CASES = {
    "torchaudio80": MelConfig("torchaudio", n_mels=80),
    "torchaudio128_log_reflect": MelConfig("torchaudio", True, n_mels=128, f_min=20, pad_mode="reflect"),
    "nnaudio388": MelConfig(),
}

MODEL_FLAVOURS = {"torchaudio": MelConfig("torchaudio", n_mels=80), "nnAudio": MelConfig()}

GK = dict(precision="fp32", do_sample=False, num_beams=1, top_p=0.9, top_k=0, cfg_scale=1.0, timeshift_bias=0, types_first=True,
          temperature=0.9, timing_temperature=0.1, mania_column_temperature=0.5, taiko_hit_temperature=0.5)


def mel_pcm(n_samples: int = 130944, B: int = 2) -> torch.Tensor:
    g = torch.Generator().manual_seed(11)
    t = torch.arange(n_samples) / 16000.0
    return 0.3 * torch.sin(2 * math.pi * 440 * t)[None] + 0.05 * torch.randn(B, n_samples, generator=g)


def model_pcm(cfg, B: int, seed: int = 0) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, cfg.samples_per_window, generator=g) * 0.1


def generate_cases():
    """name -> (prompt, negative_prompt, generate_kwargs, pcm_seed); covers first window / look-back + left pad / natural
    stop / time-shift bias + several conditional temperatures / CFG."""
    return {
        "b1_first_window": (torch.tensor([[3700, 3705, 3720, 1, 9]]), None,
                            dict(GK, max_length=5 + 40, min_new_tokens=40, lookback_time=0.0, lookahead_time=3273.6, context_type="map"), 1),
        "b2_leftpad_lookback": (torch.tensor([[0, 0, 3700, 3705, 1, 9, 3645, 30], [3700, 3701, 3702, 3703, 3704, 1, 9, 3655]]), None,
                                dict(GK, max_length=8 + 48, min_new_tokens=48, lookback_time=4092.0, lookahead_time=3273.6, context_type="map"), 2),
        "b1_eos_stop": (torch.tensor([[3700, 3705, 1, 9, 3645, 30]]), None,
                        dict(GK, max_length=64, lookback_time=4092.0, lookahead_time=3273.6, context_type="map"), 3),
        "b3_timeshift_bias": (torch.tensor([[3700, 1, 5, 3657, 100], [3701, 1, 5, 3656, 90], [3702, 1, 5, 3655, 10]]), None,
                              dict(GK, max_length=5 + 32, min_new_tokens=32, timeshift_bias=0.7, lookback_time=0.0, lookahead_time=0.0,
                                   context_type="timing"), 4),
        "b2_cfg": (torch.tensor([[3700, 3705, 3710, 1, 9, 3645, 30], [3701, 3706, 3711, 1, 9, 3648, 55]]),
                   torch.tensor([[0, 3700, 3712, 1, 9, 3645, 30], [0, 3701, 3713, 1, 9, 3648, 55]]),
                   dict(GK, cfg_scale=2.0, max_length=7 + 32, lookback_time=0.0, lookahead_time=0.0, context_type="map"), 7),
    }


def long_context_cases():
    """name -> (prompt, generate_kwargs, pcm_seed): prompts beyond 128 tokens (self-attention cache in several 64-key splits:
    3 splits at 174 tokens, 10 splits at 612), batch of 2 with left padding on row 0."""
    out = {}
    for P, new in ((150, 24), (600, 12)):
        g = torch.Generator().manual_seed(P)
        prompt = torch.randint(17, 3600, (2, P), generator=g)
        prompt[:, :4] = torch.tensor([3700, 3705, 1, 9])
        prompt[0, :7] = 0                                          # left padding on row 0
        prompt[0, 7:11] = torch.tensor([3700, 3705, 1, 9])
        gk = dict(GK, max_length=P + new, min_new_tokens=new, lookback_time=0.0, lookahead_time=0.0, context_type="map")
        out[f"long_P{P}"] = (prompt, gk, 11)
    return out


def teacher_forcing_case(cfg):
    g = torch.Generator().manual_seed(3)
    ids = torch.randint(17, cfg.vocab_size_in, (2, 21), generator=g)
    ids[1, :4] = 0
    return ids, ids.ne(0)


def processor_logits(case: str, step: int, B: int, V: int) -> torch.Tensor:
    g = torch.Generator().manual_seed(len(case) * 101 + step)
    return torch.randn(B, V, generator=g) * 3.0


def processor_cases():
    """name -> (list of input_ids per step, generate_kwargs): the processor chain applied to synthetic scores, with
    crafted histories that hit every branch (monotonic mask after/before SOS, each conditional temperature, look-back
    bias with and without a timed last token, first call without last_scores)."""
    base = dict(temperature=0.9, timing_temperature=0.1, mania_column_temperature=0.5, taiko_hit_temperature=0.5)
    seq_a = [[3700, 1, 9, 3645, 100, 900, 3648], [3701, 1, 9, 3655, 40, 3656, 3645]]
    seq_b = [[3700, 1, 9, 3645, 100, 900, 3648, 217], [3701, 1, 9, 3655, 40, 3656, 3645, 60]]
    seq_c = [[3700, 1, 9, 3645, 100, 900, 3648, 217, 3655], [3701, 1, 9, 3655, 40, 3656, 3645, 60, 1700]]
    seq_d = [[3700, 1, 9, 3645, 100, 900, 3648, 217, 3655, 230], [3701, 1, 9, 3655, 40, 3656, 3645, 60, 1700, 9]]
    lb = [torch.tensor(s) for s in (seq_a, seq_b, seq_c, seq_d)]
    mania = [torch.tensor([[3700, 1, 9, 3660, 50, 2455, 3645, 55, 2456]]), torch.tensor([[3700, 1, 9, 3660, 50, 2455, 3645, 55, 2456, 3470]])]
    scroll = [torch.tensor([[3700, 1, 11, 3662, 10, 2600]]), torch.tensor([[3700, 1, 11, 3662, 10, 2600, 3662]])]
    return {
        "lookback": (lb, dict(base, lookback_time=4092.0)),
        "nolookback_bias": (lb[:2], dict(base, lookback_time=0.0, timeshift_bias=0.7)),
        "mania": (mania, dict(base, lookback_time=0.0)),
        "scroll": (scroll, dict(base, lookback_time=0.0)),
    }


def dit_case(dc, T: int = 200, seed: int = 4):
    from oracle.dit import band_mask
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(1, 2, T, generator=g) * 2 - 1
    c = torch.randn(1, dc.context_size, T, generator=g)
    y = (torch.rand(2, dc.class_size, generator=g) < 0.1).float()
    x, c = torch.cat([x, x]), torch.cat([c, c])
    noise = torch.randn(100, 2, 2, T, generator=g)
    ip = torch.ones_like(x, dtype=torch.bool)
    ip[:, :, :40] = False
    return x, c, y, noise, ip, band_mask(T, 128)


def dit_chunk_case(dc, T: int = 300, seed: int = 8):
    """Chunked refinement case: band 32, max_seq_len 128, overlap 16 -> 3 chunks with frozen / re-noised margins."""
    g = torch.Generator().manual_seed(seed)
    seq_x = torch.rand(2, T, generator=g) * 2 - 1
    seq_c = torch.randn(dc.context_size, T, generator=g)
    y = (torch.rand(dc.class_size, generator=g) < 0.1).float()
    y_null = (torch.rand(dc.class_size, generator=g) < 0.05).float()
    return seq_x, seq_c, y, y_null, dict(train_seq_len=32, max_seq_len=128, overlap_buffer=16)


def dit_chunk_noise(k: int, shape, steps: int = 100) -> torch.Tensor:
    g = torch.Generator().manual_seed(1000 + k)
    return torch.randn(steps, *shape, generator=g)


PIN_LOGIT_STRIDE = 7      # every 7th vocabulary column of the v29 logits is stored (524 of 3667), beside the full-row argmax


def v29_logits_case(cfg):
    """One window of PCM and 12 decoder ids for a teacher-forced pass at v29 dimensions."""
    g = torch.Generator().manual_seed(0)
    pcm = torch.randn(1, cfg.samples_per_window, generator=g) * 0.1
    ids = torch.randint(17, cfg.vocab_size_in, (1, 12), generator=g)
    return pcm, ids


def context_embedding_case(T: int = 37):
    """Object times (ms), distances (px) and types of the seq_c layout (diffusion_pipeline.py:380-387)."""
    g = torch.Generator().manual_seed(4)
    seq_o = torch.rand(T, generator=g) * 180000.0
    seq_d = torch.rand(T, generator=g) * 400.0
    types = torch.randint(0, 16, (T,), generator=g)
    return seq_o, seq_d, types


def bench_window_case(cfg):
    """The bench workload's second window with 10 new tokens: (model_kwargs, generate_kwargs, prompt length)."""
    import bench
    g = torch.Generator().manual_seed(0)
    pcm = torch.randn(1, cfg.samples_per_window, generator=g) * 0.1
    prompt = torch.tensor([bench.prompt_for(1, [list(range(100, 164))])])
    P = prompt.shape[1]
    gk = bench.gen_kwargs(1, 211, P)
    gk.update(max_length=P + 10, min_new_tokens=10, precision="fp32")
    return dict(inputs=pcm, decoder_input_ids=prompt, decoder_attention_mask=prompt.ne(0)), gk, P


def slider_class_cases():
    """(curve type, control points, length) of 60 seeded sliders per curve type, some Bezier / Catmull ones with a red anchor."""
    import numpy as np
    rng = np.random.default_rng(7)
    out = []
    for typ in ("Bezier", "PerfectCurve", "Catmull", "Linear"):
        for k in range(60):
            ncp = int(rng.integers(2, 10)) if typ != "PerfectCurve" else int(rng.choice([3, 3, 4, 2]))
            cps = (rng.random((ncp, 2)) * np.array([512, 384])).astype(np.float32)
            if ncp >= 4 and k % 4 == 0:
                j = int(rng.integers(1, ncp - 2)); cps[j + 1] = cps[j]
            out.append((typ, cps, float(rng.random() * 500 + 5)))
    return out


def trim_cases(layout):
    """(tokens, trim_lookback, trim_lookahead) cases around both zones; v29 window = 8184 ms, lookback 0.5, lookahead 0.4."""
    ts, te, circle = layout.time_shift_start, layout.time_shift_end, layout.event_start["circle"]
    eos, ceos = layout.eos_id, layout.context_eos["map"]
    lb_end, la_begin = layout.lookback_end(4092.0), layout.lookback_end(4910.4)
    body = [circle, ts + 500, circle, ts + 520]
    out = []
    for tail in ([], [eos], [ceos], [ceos, eos], [eos, eos, ceos]):
        for last in (ts, lb_end - 1, lb_end, la_begin - 1, la_begin, te - 1, circle):
            for tlb in (False, True):
                for tla in (False, True):
                    out.append((body + [circle, last] + tail, tlb, tla))
    out += [([], True, True), ([eos], True, True), ([ts + 3], True, True), ([te - 1, eos], False, True)]
    return out
