"""Generate tests/golden/*.npz from the UNMODIFIED reference classes (needs a checkout of the reference project, located by
oracle/ref_import.py).  The tests only read the stored outputs.

TEST INFRASTRUCTURE.  Usage:  python -m oracle.make_golden
Inputs are regenerated from seeds by the tests (torch CPU generator); only reference OUTPUTS are stored.
Weights are `init_model_state_dict(cfg, seed)` loaded into the reference model with `load_state_dict`, so no checkpoint
is stored either.  Every case records the library versions the outputs were produced with.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mapperatorinator_b200 import MelConfig, TokenLayout, tiny_dit_config, tiny_model_config  # noqa: E402
from mapperatorinator_b200.weights import init_dit_state_dict, init_model_state_dict  # noqa: E402
from oracle import cases, ref_build  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def main():
    import transformers
    meta = dict(torch=torch.__version__, transformers=transformers.__version__)
    os.makedirs(OUT, exist_ok=True)
    torch.set_grad_enabled(False)

    # ---- tokenizer layout ----
    tok = ref_build.reference_tokenizer()
    TokenLayout.from_tokenizer(tok).to_json(os.path.join(OUT, "tokenizer_v29.json"))

    # ---- stage (i): MelSpectrogram module of the reference ----
    ref_build.ref_import.install_stubs()
    from osuT5.osuT5.model.spectrogram import MelSpectrogram
    mel_out = {}
    for name, mc in cases.MEL_CASES.items():
        if mc.implementation != "torchaudio":
            continue   # nnAudio is absent: that flavour is pinned only through the restated transform (parity unpinned)
        mod = MelSpectrogram(mc.implementation, mc.log_scale, mc.sample_rate, mc.n_fft, mc.n_mels, mc.hop_length, mc.f_min, mc.f_max,
                             mc.pad_mode)
        mel_out[name] = mod(cases.mel_pcm()).numpy()[:, ::64, :]
    np.savez_compressed(os.path.join(OUT, "mel_reference.npz"), **mel_out, **{f"meta_{k}": v for k, v in meta.items()})

    # ---- stage (ii): tiny osuT5 through the reference model_generate ----
    from osuT5.osuT5.inference.server import model_generate
    gen_out = {}
    for flavour, melc in cases.MODEL_FLAVOURS.items():
        cfg = tiny_model_config(mel=melc)
        model, tok2, _ = ref_build.reference_model(cfg, tok=tok, mel_impl=melc.implementation)
        sd = init_model_state_dict(cfg, 0)
        ref_build.load_state_dict_into_reference(model, sd)
        pcm = cases.model_pcm(cfg, 3, 0)
        gen_out[f"{flavour}/encoder"] = model.get_encoder()(pcm)[0].numpy()[:, ::32, :]
        for cname, (prompt, neg, gk, seed) in cases.generate_cases().items():
            B = prompt.shape[0]
            mk = dict(inputs=cases.model_pcm(cfg, B, seed), decoder_input_ids=prompt, decoder_attention_mask=prompt.ne(0),
                      negative_prompt=neg, negative_prompt_attention_mask=None if neg is None else neg.ne(0))
            ids, stats = model_generate(model, tok2, dict(mk), dict(gk))
            gen_out[f"{flavour}/{cname}/ids"] = ids.numpy()
            gen_out[f"{flavour}/{cname}/counts"] = np.array(stats["generated_tokens_per_sample"])
        if flavour == "torchaudio":                               # long prompts: decoder-side only, one flavour is enough
            for cname, (prompt, gk, seed) in cases.long_context_cases().items():
                mk = dict(inputs=cases.model_pcm(cfg, prompt.shape[0], seed), decoder_input_ids=prompt, decoder_attention_mask=prompt.ne(0))
                ids, _ = model_generate(model, tok2, dict(mk), dict(gk))
                gen_out[f"{flavour}/{cname}/ids"] = ids.numpy()
        ids, mask = cases.teacher_forcing_case(cfg)
        out = model(frames=cases.model_pcm(cfg, 2, 1), decoder_input_ids=ids, decoder_attention_mask=mask)
        gen_out[f"{flavour}/teacher_logits"] = out.logits.float().numpy()[:, ::3, ::37]
    np.savez_compressed(os.path.join(OUT, "generate_reference.npz"), **gen_out, **{f"meta_{k}": v for k, v in meta.items()})

    # ---- logits processors in isolation (reference classes, synthetic scores) ----
    from osuT5.osuT5.inference.logit_processors import (ConditionalTemperatureLogitsWarper, LookbackBiasLogitsWarper,
                                                        MonotonicTimeShiftLogitsProcessor, TimeshiftBias, get_beat_type_tokens,
                                                        get_mania_type_tokens, get_scroll_speed_tokens)
    from osuT5.osuT5.event import EventType
    proc_out = {}
    for cname, (ids_steps, gk) in cases.processor_cases().items():
        chain = [MonotonicTimeShiftLogitsProcessor(tok)]
        if gk.get("timeshift_bias", 0) != 0:
            chain.append(TimeshiftBias(gk["timeshift_bias"], tok.event_start[EventType.TIME_SHIFT], tok.event_end[EventType.TIME_SHIFT]))
        chain.append(ConditionalTemperatureLogitsWarper(gk["temperature"], gk["timing_temperature"], gk["mania_column_temperature"],
                                                        gk["taiko_hit_temperature"], True, get_beat_type_tokens(tok),
                                                        get_mania_type_tokens(tok), get_scroll_speed_tokens(tok)))
        if gk.get("lookback_time", 0) > 0:
            chain.append(LookbackBiasLogitsWarper(gk["lookback_time"], tok, True, "cpu"))
        for step, ids in enumerate(ids_steps):
            scores = cases.processor_logits(cname, step, ids.shape[0], tok.vocab_size_out)
            for p in chain:
                scores = p(ids, scores)
            proc_out[f"{cname}/{step}"] = scores.numpy()
    np.savez_compressed(os.path.join(OUT, "processors_reference.npz"), **proc_out)

    # ---- stage (iii): tiny DiT + the reference GaussianDiffusion loop ----
    from osu_diffusion.utils.diffusion import create_diffusion
    dc = tiny_dit_config()
    dsd = init_dit_state_dict(dc, 1)
    m = ref_build.reference_dit(dc)
    m.load_state_dict(dsd, strict=True)
    dit_out = {}
    x, c, y, noise, ip, am = cases.dit_case(dc)
    t = torch.tensor([37, 37])
    dit_out["forward_with_cfg"] = m.forward_with_cfg(x, t, c, y, 1.5, attn_mask=am).numpy()
    diff = create_diffusion(timestep_respacing=[100, 0, 0, 0, 0, 0, 0, 0, 0, 0], diffusion_steps=1000, noise_schedule="squaredcos_cap_v2")
    it = iter(noise)
    orig = torch.randn_like
    torch.randn_like = lambda a: next(it)
    try:
        z0 = x.clone()
        dfn = lambda xx: torch.where(ip, xx, z0)
        dit_out["p_sample_loop"] = diff.p_sample_loop(m.forward_with_cfg, x.shape, x.clone(), denoised_fn=dfn, clip_denoised=True,
                                                      model_kwargs=dict(c=c, y=y, cfg_scale=1.0, attn_mask=am, key_padding_mask=None),
                                                      device="cpu").numpy()
    finally:
        torch.randn_like = orig
    # the chunk loop / in-paint mask / to_positions of the reference's own DiffisionPipeline.generate (diffusion_pipeline.py:111-287):
    # only the event<->tensor conversions are stubbed (they need slider + real beatmaps)
    import types as _types
    import diffusion_pipeline as dp
    seq_x, seq_c, yv, y_null, geo = cases.dit_chunk_case(dc)
    pipe = object.__new__(dp.DiffisionPipeline)
    pipe.device = "cpu"; pipe.model = m; pipe.tokenizer = None; pipe.refine_model = None
    pipe.diffusion_steps = 1000; pipe.noise_schedule = "squaredcos_cap_v2"; pipe.seq_len = geo["train_seq_len"]
    pipe.max_seq_len = geo["max_seq_len"]; pipe.overlap_buffer = geo["overlap_buffer"]; pipe.timesteps = [100, 0, 0, 0, 0, 0, 0, 0, 0, 0]
    pipe.cfg_scale = 1.0; pipe.refine_iters = 0; pipe.random_init = False; pipe.types_first = True; pipe.pad_sequence = False
    pipe.start_time = None; pipe.end_time = None; pipe.has_sv = True
    Tn = seq_x.shape[1]
    pipe.events_to_sequence = lambda events, timing, sm: (seq_x.clone(), torch.arange(Tn).float(), seq_c.clone(), Tn, {}, [])
    vecs = iter([yv.clone(), y_null.clone()])
    pipe.get_class_vector = lambda cfg_: next(vecs)
    captured = {}
    pipe.events_with_pos = lambda events, positions, idx: captured.setdefault("pos", positions.clone())
    state = {"k": -1, "it": None}
    def _randn_like(a):
        if state["it"] is None or state["left"] == 0:
            state["k"] += 1
            state["it"] = iter(cases.dit_chunk_noise(state["k"], a.shape)); state["left"] = 100
        state["left"] -= 1
        return next(state["it"])
    orig2 = torch.randn_like
    torch.randn_like = _randn_like
    try:
        gc = _types.SimpleNamespace(difficulty=None, descriptors=None, negative_descriptors=None, circle_size=None, slider_multiplier=1.4)
        pipe.generate([], gc, [], verbose=False)
    finally:
        torch.randn_like = orig2
    dit_out["chunked_positions"] = captured["pos"].numpy()
    dit_out["timestep_map"] = np.array(diff.timestep_map)
    dit_out["schedule"] = np.stack([diff.sqrt_recip_alphas_cumprod, diff.sqrt_recipm1_alphas_cumprod, diff.posterior_log_variance_clipped,
                                    np.log(diff.betas), diff.posterior_mean_coef1, diff.posterior_mean_coef2], 1)
    np.savez_compressed(os.path.join(OUT, "dit_reference.npz"), **dit_out, **{f"meta_{k}": v for k, v in meta.items()})
    make_slider_golden(meta)
    make_pins_golden(meta)
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


def make_slider_golden(meta=None):
    """Slider end points from the UNMODIFIED reference `SliderPath` (osuT5/osuT5/inference/slider_path.py) on (a) every slider of the
    reference's own toy beatmap (osu_diffusion/testing/toy_datasets/kimi_no_bouken.osu: 138 sliders, Bezier / PerfectCurve / Linear, with
    red anchors) and (b) seeded random control points for all curve types incl. Catmull.  Stored: control points (float32, as the pipeline
    feeds them), curve type, length, reference max_length and end position."""
    from oracle import ref_import, slider as so
    SP = ref_import.reference_slider_path()
    cases_ = [(t, c, l) for t, c, l in so.parse_osu_sliders(os.path.join(ref_import.REFERENCE_ROOT, "osu_diffusion", "testing", "toy_datasets", "kimi_no_bouken.osu"))]
    rng = np.random.default_rng(42)
    for typ in ("Bezier", "PerfectCurve", "Catmull"):
        for k in range(40):
            ncp = int(rng.integers(2, 9)) if typ != "PerfectCurve" else int(rng.choice([3, 3, 3, 4, 2]))
            cps = (rng.random((ncp, 2)) * np.array([512, 384])).astype(np.float32)
            if typ == "Bezier" and ncp >= 4 and k % 3 == 0:
                j = int(rng.integers(1, ncp - 2)); cps[j + 1] = cps[j]                      # red anchor
            cases_.append((typ, cps, float(rng.random() * 400 + 10)))
    types, offs, pts, lens, maxl, ends = [], [0], [], [], [], []
    for typ, cps, length in cases_:
        sp = SP(typ, cps)
        ml = float(sp.get_distance())
        if ml == 0:
            continue
        e = np.asarray(sp.position_at(length / ml), dtype=np.float64)
        types.append(so.CURVE_TYPES[typ]); offs.append(offs[-1] + len(cps)); pts.append(cps); lens.append(length); maxl.append(ml); ends.append(e)
    np.savez_compressed(os.path.join(OUT, "slider_reference.npz"), types=np.array(types, dtype=np.int32), offsets=np.array(offs, dtype=np.int32),
                        points=np.concatenate(pts).astype(np.float32), lengths=np.array(lens, dtype=np.float32), max_length=np.array(maxl),
                        end_pos=np.stack(ends), **({f"meta_{k}": v for k, v in (meta or {}).items()}))


def make_pins_golden(meta=None):
    """Outputs of single reference functions at v29 dimensions or on host-side helpers (tests/golden/reference_pins.npz):
    `Mapperatorinator.forward` logits, `server.model_generate` ids on the bench's second window, `timestep_embedding`,
    `SliderPath` end points and the token-level result of `Processor.add_predicted_tokens_to_context`."""
    import dataclasses
    import types as _types
    from mapperatorinator_b200 import v29_model_config
    from oracle import ref_import
    torch.set_grad_enabled(False)
    out = {}
    # ---- teacher-forced logits and greedy ids of the bench's second window, whisper-small dimensions ----
    cfg = dataclasses.replace(v29_model_config(), mel=MelConfig("torchaudio", n_mels=80))
    model, tok, _ = ref_build.reference_model(cfg, mel_impl="torchaudio")
    assert TokenLayout.from_tokenizer(tok) == TokenLayout.from_json(os.path.join(ROOT, "tests", "golden", "tokenizer_v29.json"))
    ref_build.load_state_dict_into_reference(model, init_model_state_dict(cfg, 0))
    pcm, ids = cases.v29_logits_case(cfg)
    logits = model(frames=pcm, decoder_input_ids=ids, decoder_attention_mask=ids.ne(0)).logits.float()
    out["v29_logits_sample"] = logits.numpy()[:, :, ::cases.PIN_LOGIT_STRIDE]
    out["v29_logits_argmax"] = logits.argmax(-1).numpy()
    from osuT5.osuT5.inference.server import model_generate
    mk, gk, _ = cases.bench_window_case(cfg)
    out["bench_window_ids"] = model_generate(model, tok, mk, gk)[0].numpy()
    del model
    # ---- timestep_embedding of the seq_c layout ----
    from osu_diffusion import timestep_embedding
    seq_o, seq_d, _ = cases.context_embedding_case()
    out["timestep_embedding_time"] = timestep_embedding(seq_o * 0.1, 128).numpy()
    out["timestep_embedding_distance"] = timestep_embedding(seq_d, 128).numpy()
    # ---- SliderPath end points (max_length 0 marks a degenerate path the test skips) ----
    SP = ref_import.reference_slider_path()
    mls, ends = [], []
    for typ, cps, length in cases.slider_class_cases():
        sp = SP(typ, cps)
        ml = float(sp.get_distance())
        mls.append(ml)
        ends.append(np.asarray(sp.position_at(length / ml), dtype=np.float64) if ml != 0 else np.zeros(2))
    out["slider_class_max_length"] = np.array(mls)
    out["slider_class_end_pos"] = np.stack(ends)
    # ---- the tokens add_predicted_tokens_to_context hands to _decode, on a stand-in `self` (processor.py:1022-1052) ----
    from osuT5.osuT5.inference import processor as rp
    from osuT5.osuT5.tokenizer import ContextType
    layout = TokenLayout.from_json(os.path.join(ROOT, "tests", "golden", "tokenizer_v29.json"))
    seen, trimmed = [], []
    fake = _types.SimpleNamespace(
        tokenizer=_types.SimpleNamespace(eos_id=layout.eos_id, context_eos={ContextType(k): v for k, v in layout.context_eos.items()}),
        lookback_time_range=range(layout.time_shift_start, layout.lookback_end(4092.0)),                 # processor.py:85
        lookahead_time_range=range(layout.lookback_end(4910.4), layout.time_shift_end),                  # processor.py:88
        types_first=True, eos_time=0.0, lookahead_max_time=4910.4,
        _decode=lambda toks, frame_time: seen.append(list(toks)) or [], _trim_events_after_time=lambda *a: None)
    old = rp.update_event_times
    rp.update_event_times = lambda *a, **k: None
    try:
        for types_first in (True, False):
            fake.types_first = types_first
            for toks, tlb, tla in cases.trim_cases(layout):
                seen.clear()
                ctx = {"context_type": ContextType("map"), "events": [], "event_times": []}
                rp.Processor.add_predicted_tokens_to_context(fake, ctx, torch.tensor(toks, dtype=torch.long).tolist(), 1234.0, tlb, tla)
                trimmed.append(seen[0])
    finally:
        rp.update_event_times = old
    out["trim_offsets"] = np.cumsum([0] + [len(s) for s in trimmed])          # types_first=True cases, then types_first=False
    out["trim_tokens"] = np.array(sum(trimmed, []), dtype=np.int64)
    np.savez_compressed(os.path.join(OUT, "reference_pins.npz"), **out, **({f"meta_{k}": v for k, v in (meta or {}).items()}))


if __name__ == "__main__":
    main()
