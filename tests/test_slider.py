"""Slider end-point recompute of the diffusion `denoised_fn` (SURVEY §8f N2; diffusion_pipeline.py:203-222, slider_path.py, path_approximator.py).

CPU: the oracle restatement (oracle/slider.py) against tests/golden/slider_reference.npz — end points and path lengths produced by the
UNMODIFIED reference `SliderPath` on every slider of the reference's toy beatmap plus seeded random control points — and against
that class's end points on a second seeded set (tests/golden/reference_pins.npz).
GPU: the device recompute (csrc/slider.cu, through the C ABI) against the same fixture and against the oracle closure, alone and inside
the fused 100-step loop.  Tolerance: 1e-3 in normalised coordinates (north_star) = 0.256 px; measured errors are ~1e-3 px.
"""
import os

import numpy as np
import pytest
import torch

from oracle import slider as so

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMES = {v: k for k, v in so.CURVE_TYPES.items()}


@pytest.fixture(scope="module")
def gold():
    g = np.load(os.path.join(GOLDEN, "slider_reference.npz"))
    out = []
    for k in range(len(g["types"])):
        a, b = g["offsets"][k], g["offsets"][k + 1]
        out.append((NAMES[int(g["types"][k])], g["points"][a:b], float(g["lengths"][k]), float(g["max_length"][k]), g["end_pos"][k]))
    return out


def test_oracle_slider_matches_reference_fixture(gold):
    assert len(gold) >= 250 and {t for t, *_ in gold} == {"Bezier", "PerfectCurve", "Catmull", "Linear"}
    worst = 0.0
    for typ, cps, length, ml_ref, end_ref in gold:
        ml, end = so.slider_end_position(typ, cps, length)
        assert abs(ml - ml_ref) <= 1e-5 * ml_ref + 1e-4, (typ, ml, ml_ref)
        worst = max(worst, float(np.abs(end - end_ref).max()))
    assert worst <= 1e-3, worst                                   # pixels


def test_oracle_slider_matches_reference_class():
    """The oracle against the reference `SliderPath` on 60 seeded sliders per curve type (tests/golden/reference_pins.npz)."""
    from oracle import cases
    pins = np.load(os.path.join(GOLDEN, "reference_pins.npz"))
    sliders = cases.slider_class_cases()
    assert len(sliders) == len(pins["slider_class_max_length"]) == 240
    worst = 0.0
    for (typ, cps, length), ml_ref, end_ref in zip(sliders, pins["slider_class_max_length"], pins["slider_class_end_pos"]):
        if ml_ref == 0:
            continue
        ml, end = so.slider_end_position(typ, cps, length)
        worst = max(worst, float(np.abs(end - end_ref).max()))
    assert worst <= 1e-3, worst


def _layout_case(gold, n_sliders, T, seed):
    """A chunk of T points in which `n_sliders` fixture sliders are laid out back to back: [control points..., end event]."""
    rng = np.random.default_rng(seed)
    pick = rng.choice(len(gold), n_sliders, replace=False)
    pos = rng.random((T, 2)) * np.array([512, 384])
    sliders, t = [], 3
    for k in pick:
        typ, cps, length, _, _ = gold[k]
        idx = []
        for i, p in enumerate(cps):
            if i > 0 and (cps[i] == cps[i - 1]).all():
                idx.append(idx[-1])                              # red anchor: the SAME sequence index twice (diffusion_pipeline.py:412-414)
            else:
                pos[t] = p; idx.append(t); t += 1
        sliders.append(so.Slider(np.array(idx), t, typ, length)); t += 2
        assert t < T
    x = torch.from_numpy((pos / np.array([512, 384]) * 2 - 1).T.astype(np.float32))            # (2, T)
    x = torch.stack([x, x * 0.5])                                                                # conditional | null-class half
    return x, sliders, pick


@pytest.mark.gpu
def test_device_slider_recompute_matches_reference_and_oracle(gold):
    from mapperatorinator_b200 import tiny_dit_config
    from mapperatorinator_b200.diffusion import B200DiT, DiffusionSlider, InpaintDenoiser
    from mapperatorinator_b200.weights import init_dit_state_dict
    dc = tiny_dit_config()
    dit = B200DiT(dc, init_dit_state_dict(dc, 1), max_seq_len=1024)
    T = 1024
    for seed, n in ((0, 60), (1, 90), (2, 90)):
        x, sliders, pick = _layout_case(gold, n, T, seed)
        mask = torch.ones_like(x, dtype=torch.bool)
        want = so.denoised_fn_with_sliders(x, mask, x, sliders, 0, T)
        den = InpaintDenoiser(mask.cuda(), x.cuda(), [DiffusionSlider(s.seq_indices, s.end_index, s.curve_type, s.length) for s in sliders], 0, T,
                              engine=dit.engine)
        got = den(x.cuda()).cpu()
        assert got.shape == want.shape
        assert (got - want).abs().max() <= 1e-4, (got - want).abs().max()                      # normalised units (0.05 px), vs the oracle closure
        assert torch.equal(got[0], got[1])                                                       # both halves carry the conditional positions
        px = ((got[0] + 1) / 2 * torch.tensor((512.0, 384.0))[:, None]).T.numpy()
        for s, k in zip(sliders, pick):                                                          # vs the reference's own end points
            _, cps, _, ml_ref, end_ref = gold[k]
            if ml_ref > 2000:
                continue          # near-collinear "perfect curve": radius of 1e4+ px amplifies the float32 round trip of the layout above
            if len(np.unique(s.seq_indices)) == len(cps) - sum((cps[i] == cps[i - 1]).all() for i in range(1, len(cps))):
                assert np.abs(px[s.end_index] - end_ref).max() <= 0.05, (s.curve_type, px[s.end_index], end_ref)


@pytest.mark.gpu
def test_fused_loop_with_sliders_matches_oracle_closure(gold):
    """The 100-step loop with the slider closure fused on the device vs the oracle loop with the oracle closure as `denoised_fn`
    (applied to the start state first, diffusion_pipeline.py:233): 1e-3 abs."""
    from mapperatorinator_b200 import tiny_dit_config
    from mapperatorinator_b200.diffusion import B200DiT, DiffusionSlider, InpaintDenoiser, create_diffusion
    from mapperatorinator_b200.weights import init_dit_state_dict
    from oracle import cases, dit as do
    dc = tiny_dit_config()
    sd = init_dit_state_dict(dc, 1)
    dit = B200DiT(dc, sd, max_seq_len=512)
    T = 200
    _, c, y, noise, ip, am = cases.dit_case(dc, T)
    xs, sliders, _ = _layout_case(gold, 12, T, 5)
    x = torch.stack([xs[0], xs[0]])                                                              # CFG pair starts from the same state
    z0 = so.denoised_fn_with_sliders(x, ip, x, sliders, 0, T)
    closure = lambda v: so.denoised_fn_with_sliders(v, ip, z0, sliders, 0, T)
    ref = do.p_sample_loop(sd, dc, do.Schedule(), z0, c, y, 1.0, am, noise, denoised_fn=closure)
    diff = create_diffusion([100, 0, 0, 0, 0, 0, 0, 0, 0, 0], "squaredcos_cap_v2", 1000)
    mk = dict(c=c.cuda(), y=y.cuda(), cfg_scale=1.0, attn_mask=am.cuda(), key_padding_mask=None)
    den = InpaintDenoiser(ip.cuda(), x.cuda(), [DiffusionSlider(s.seq_indices, s.end_index, s.curve_type, s.length) for s in sliders], 0, T, engine=dit.engine)
    got = diff.p_sample_loop(dit.forward_with_cfg, x.shape, x.cuda(), denoised_fn=den, clip_denoised=True, model_kwargs=mk, step_noise=noise.cuda()).cpu()
    assert (got - ref).abs().max() <= 1e-3, (got - ref).abs().max()
    # and the same loop without the fused path (graph off) gives the same numbers
    dit.engine.lib.mb200_dit_set_option(dit.engine.handle, b"graph", 0)
    got2 = diff.p_sample_loop(dit.forward_with_cfg, x.shape, x.cuda(), denoised_fn=den, clip_denoised=True, model_kwargs=mk, step_noise=noise.cuda()).cpu()
    dit.engine.lib.mb200_dit_set_option(dit.engine.handle, b"graph", 1)
    assert torch.equal(got, got2)
