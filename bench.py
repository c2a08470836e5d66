#!/usr/bin/env python
"""bench.py — event tokens/sec of the Mapperatorinator inference hot path on B200 (contract: see README "Measurement").

Workload (BASELINE.json configs[1] + configs[2], SURVEY §8d rows 2a + 3): osuT5 v29 dimensions (whisper-small, 213 M params,
fp32, seeded random weights), one 180 s synthetic song as 44.1 kHz 16-bit stereo PCM -> GPU ingest (resample to 16 kHz, mono, peak-normalise) -> 211 sequential windows (stride 13 094 samples), greedy decode,
`min_new_tokens = 64`, `max_length = P + 64` (random weights have no EOS behaviour, so the token budget is pinned:
211 x 64 = 13 504 event tokens per step), real look-back / look-ahead EOS sets and logits-processor chain, prompt =
16 conditioning ids + SOS + ctx_sos(MAP) (+ the last 32 generated ids of the previous window -> sequential dependency);
THEN the osu_diffusion stage the metric names ("mel+T5+DiT"): DiT-B (131 M params, fp32, seeded weights), 1 500 hit-object
points -> chunks [0:1024] and [768:1500] (diffusion_pipeline.py:276-284), 100 denoising steps each, CFG pair, +-128 band mask.

A "step" = one full song (decode + position refinement).
  value : tokens/s with the song's file PCM (int16) and the DiT inputs already resident in HBM (engine path: GPU audio ingest + device
          segmentation, one batched mel+encoder pass over all windows, cross-K/V resident, sequential prefill + token loop per window, fused on-device 100-step loops),
          CUDA-event timed.  `value_decode_only` = the same without the DiT stage (round-1's number).
  e2e   : the same song through the reference-facing calls with HOST tensors: `audio.load_pcm` + `pipeline.segment` where the reference
          runs `load_audio_file` + `Preprocessor.segment` (host PCM in, host windows out), `server.model_generate(model, tokenizer,
          model_kwargs, generate_kwargs)` once per window (pinned PCM in, CPU LongTensor out, encoder re-run per call as the
          reference does) and `diffusion.sample_sequence` (pinned seq_x / seq_c / y in, CPU positions out) — H2D, D2H inside
          the timed region.
  --impl reference : the CPU oracle port of the reference path (same call pattern) on the host cores, bounded sample.
Multi-GPU (torchrun): one song per rank per step (weak scaling; rank r decodes song `--song-seed + r`), NCCL gather of the
token streams inside the timed region.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
import traceback

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from mapperatorinator_b200 import TokenLayout, dit_b_config, v29_model_config  # noqa: E402
from mapperatorinator_b200.pipeline import gather_token_streams, segment, segment_device  # noqa: E402
from mapperatorinator_b200.weights import init_dit_state_dict, init_model_state_dict  # noqa: E402

SONG_SECONDS = 180.0
NEW_TOKENS = 64
COND_IDS = [3667, 3680, 3700, 3710, 3730, 3798, 3810, 3870, 3965, 3975, 3992, 4006, 4100, 3862, 3863, 3864]   # 16 input-only ids
DIT_POINTS, DIT_STEPS, DIT_CLASSES = 1500, 100, 600
DIT_GEOMETRY = dict(train_seq_len=128, max_seq_len=1024, overlap_buffer=128)     # diffusion_pipeline.py defaults
METRIC = "event tokens/sec end-to-end (mel+T5+DiT)"


def synth_song(seed: int, seconds: float = SONG_SECONDS, sr: int = 16000) -> np.ndarray:
    """SURVEY §8d: 8 log-spaced sinusoids 55 Hz-7 kHz + 120 BPM click train + N(0, 0.01) noise, peak-normalised."""
    rng = np.random.default_rng(seed)
    n = int(seconds * sr)
    t = np.arange(n) / sr
    x = sum(np.sin(2 * np.pi * f * t + rng.uniform(0, 2 * np.pi)) for f in np.geomspace(55, 7000, 8)) / 8
    clicks = np.zeros(n)
    clicks[(np.arange(0, seconds, 0.5) * sr).astype(int)] = 1.0
    x = x + np.convolve(clicks, np.hanning(64), mode="same") + rng.normal(0, 0.01, n)
    return (x / np.abs(x).max()).astype(np.float32)


FILE_RATE, MODEL_RATE = 44100, 16000


def synth_song_pcm(seed: int, seconds: float = SONG_SECONDS) -> np.ndarray:
    """The song as an audio FILE holds it (BASELINE: synthetic 44.1 kHz audio): interleaved 16-bit stereo PCM, int16 [n, 2] — the same
    recipe as `synth_song` at 44.1 kHz, the right channel a slightly attenuated, phase-shifted copy."""
    rng = np.random.default_rng(seed)
    n = int(seconds * FILE_RATE)
    t = np.arange(n) / FILE_RATE
    ph = [rng.uniform(0, 2 * np.pi) for _ in range(8)]
    left = sum(np.sin(2 * np.pi * f * t + p) for f, p in zip(np.geomspace(55, 7000, 8), ph)) / 8
    right = sum(np.sin(2 * np.pi * f * t + p + 0.3) for f, p in zip(np.geomspace(55, 7000, 8), ph)) / 8 * 0.9
    clicks = np.zeros(n)
    clicks[(np.arange(0, seconds, 0.5) * FILE_RATE).astype(int)] = 1.0
    clicks = np.convolve(clicks, np.hanning(176), mode="same")
    noise = rng.normal(0, 0.01, (n, 2))
    x = np.stack([left + clicks, right + clicks], 1) + noise
    return np.clip(np.round(x / np.abs(x).max() * 30000.0), -32768, 32767).astype(np.int16)


def oracle_windows(seed: int, cfg):
    """CPU-side view of the same song for the checks / the CPU arm: the reference's ingest arithmetic (oracle.audio.ingest_reference =
    audioop.ratecv + tomono + peak normalisation, data_utils.py:80-101) and `Preprocessor.segment`."""
    from oracle import audio as audio_oracle
    return segment(audio_oracle.ingest_reference(synth_song_pcm(seed), FILE_RATE, MODEL_RATE), cfg)[0]


def prompt_for(i: int, streams) -> list:
    base = COND_IDS + [1, 9]
    return base if i == 0 else base + streams[i - 1][-32:]


def gen_kwargs(i: int, n_windows: int, P: int) -> dict:
    ms = 8184.0
    return dict(do_sample=False, num_beams=1, top_p=0.9, top_k=0, cfg_scale=1.0, timeshift_bias=0, types_first=True, temperature=0.9,
                timing_temperature=0.1, mania_column_temperature=0.5, taiko_hit_temperature=0.5, max_length=P + NEW_TOKENS,
                min_new_tokens=NEW_TOKENS, lookback_time=0.5 * ms if i > 0 else 0.0, lookahead_time=0.4 * ms if i < n_windows - 1 else 0.0,
                context_type="map")


def synth_hit_objects(seed: int, T: int = DIT_POINTS):
    """Synthetic input of the diffusion stage, shaped like `DiffisionPipeline.events_to_sequence` output (diffusion_pipeline.py:
    289-438): seq_x (2, T) start positions in [-1, 1], seq_c (272, T) = [sin/cos(time), sin/cos(distance), one-hot type], the
    class vector y and the null class vector."""
    from mapperatorinator_b200.diffusion import build_context
    g = torch.Generator().manual_seed(1000 + seed)
    seq_x = torch.rand(2, T, generator=g) * 2 - 1
    seq_o = torch.cumsum(torch.rand(T, generator=g) * 240.0, 0)                       # object times, ms
    seq_d = torch.rand(T, generator=g) * 200.0                                         # distances, osu! pixels
    types = torch.randint(0, 16, (T,), generator=g)
    seq_c = build_context(seq_o, seq_d, types)
    y = (torch.rand(DIT_CLASSES, generator=g) < 0.03).float()
    y_null = torch.zeros(DIT_CLASSES); y_null[-1] = 1.0
    return seq_x, seq_c, y, y_null


def dit_chunks(T: int = DIT_POINTS):
    ob, ms = DIT_GEOMETRY["overlap_buffer"], DIT_GEOMETRY["max_seq_len"]
    return [(i, min(i + ms, T)) for i in range(0, T - ob * 2, ms - ob * 2)]


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.rows.append(l) for l in self.proc.stdout], daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()

    def summary(self) -> dict:
        sm, mx, reasons = [], 0, set()
        for l in self.rows:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def workload_config(n_windows: int, dit: bool, songs_per_gpu: int = 1) -> dict:
    cfg = {"workload": "osuT5 v29 full-song inference, 180 s synthetic 44.1 kHz 16-bit stereo audio -> GPU ingest to 16 kHz mono (data_utils.py:80-101) -> sequential sliding windows (configs[1], SURVEY 8d 2a)"
                       + (" + osu_diffusion DiT-B 100-step position refinement (configs[2], SURVEY 8d 3)" if dit else ""),
           "windows": n_windows, "new_tokens_per_window": NEW_TOKENS, "decode": "greedy, min_new_tokens=64", "batch": songs_per_gpu,
           "weights": "seeded random init, whisper-small dims (213M) + DiT-B (131M), fp32", "songs_per_gpu_per_step": songs_per_gpu,
           "l2": "inputs larger than L2: each token streams the 464 MB fp32 decoder (L2 = 126 MB)"}
    if dit:
        cfg["dit"] = {"points": DIT_POINTS, "chunks": dit_chunks(), "steps": DIT_STEPS, "cfg_pair": True, "band": 128}
    return cfg


# ---- CPU arm (the oracle port of the reference path): bounded sample of the same workload ---------------------------------------
def cpu_sample(args, cfg, layout, windows, n_windows, sd, gpu_streams=None):
    """First `--cpu-windows` windows through the oracle's `model_generate` (reference call pattern: encoder re-run per call), plus
    the same FRACTION of the song's diffusion work (cpu_windows / n_windows of the 2 x 100 chunk-steps) through the oracle's
    `dit_forward_with_cfg`.  Returns (tokens, seconds, info)."""
    from oracle import generate as gen_oracle
    cs, toks = [], 0
    t0 = time.perf_counter()
    with torch.no_grad():
        for i in range(args.cpu_windows):
            prompt = torch.tensor([prompt_for(i, cs)])
            ids, st = gen_oracle.model_generate(sd, cfg, layout, dict(inputs=windows[i:i + 1], decoder_input_ids=prompt,
                                                                      decoder_attention_mask=prompt.ne(0)),
                                                gen_kwargs(i, n_windows, prompt.shape[1]))
            cs.append(ids[0, prompt.shape[1]:].tolist()); toks += st["generated_tokens"]
    t_dec = time.perf_counter() - t0
    info = {"decode_seconds": t_dec}
    t_dit = 0.0
    if args.dit:
        from oracle import dit as dit_oracle
        dc = dit_b_config(DIT_CLASSES)
        dsd = init_dit_state_dict(dc, 1)
        seq_x, seq_c, y, y_null = synth_hit_objects(args.song_seed)
        chunks = dit_chunks()
        share = len(chunks) * DIT_STEPS * args.cpu_windows / n_windows            # chunk-steps that belong to the sampled windows
        n_run = max(len(chunks), int(np.ceil(share)))
        am = dit_oracle.band_mask(DIT_POINTS, DIT_GEOMETRY["train_seq_len"])
        yy = torch.stack([y, y_null], 0)
        t0 = time.perf_counter()
        with torch.no_grad():
            for k in range(n_run):
                a, b = chunks[k % len(chunks)]
                x = torch.cat([seq_x[None, :, a:b]] * 2); c = torch.cat([seq_c[None, :, a:b]] * 2)
                dit_oracle.dit_forward_with_cfg(dsd, dc, x, torch.tensor([99 - k, 99 - k]), c, yy, 1.0, am[a:b, a:b])
        t_run = time.perf_counter() - t0
        t_dit = t_run * share / n_run
        info.update({"dit_steps_run": n_run, "dit_steps_charged": share, "dit_seconds_charged": t_dit})
    if gpu_streams is not None:
        info["token_ids_match_gpu"] = bool(cs == gpu_streams[:args.cpu_windows])
    sample = (f"first {args.cpu_windows} of {n_windows} sequential windows x {NEW_TOKENS} tokens, encoder re-run per call (reference call pattern)"
              + (f" + {info['dit_steps_charged']:.2f} DiT-B chunk-steps (the same fraction of the song's {len(dit_chunks()) * DIT_STEPS})" if args.dit else ""))
    return toks, t_dec + t_dit, sample, info


def run_reference(args, rank: int, world: int) -> None:
    if rank != 0:
        return
    cores = args.cpu_threads or min(os.cpu_count() or 1, 16)
    torch.set_num_threads(cores)
    cfg = v29_model_config()
    layout = TokenLayout.from_json(os.path.join(ROOT, "tests", "golden", "tokenizer_v29.json"))
    sd = init_model_state_dict(cfg, 0)
    windows = oracle_windows(args.song_seed, cfg)
    n_windows = windows.shape[0]
    for _ in range(args.warmup):
        cpu_sample(args, cfg, layout, windows, n_windows, sd)
    toks, secs = 0, 0.0
    for _ in range(args.steps):
        t, s, sample, info = cpu_sample(args, cfg, layout, windows, n_windows, sd)
        toks += t; secs += s
    v = toks / secs
    print(json.dumps({
        "impl": "reference", "metric": METRIC if args.dit else "event tokens/sec end-to-end", "value": v, "unit": "tokens/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * secs / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(n_windows, bool(args.dit)),
        "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample, **info},
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ---- whole-song parity against the oracle --------------------------------------------------------------------------------------
def oracle_song_check(cfg, layout, sd, windows, streams, which) -> dict:
    """One teacher-forced oracle pass per window (oracle.generate.teacher_forced_check): the GPU's greedy ids must be the argmax of
    the oracle's processed scores at every generated position.  `which` = window indices to check."""
    from oracle import generate as gen_oracle
    from oracle import whisper as wo
    n_windows = windows.shape[0]
    bad, min_gap, checked = None, float("inf"), 0
    t0 = time.perf_counter()
    with torch.no_grad():
        for c0 in range(0, len(which), 8):
            idx = which[c0:c0 + 8]
            enc = wo.encode(sd, cfg, windows[idx])
            for j, i in enumerate(idx):
                prompt = prompt_for(i, streams)
                rep = gen_oracle.teacher_forced_check(sd, cfg, layout, None, torch.tensor([prompt + streams[i]]), len(prompt),
                                                      gen_kwargs(i, n_windows, len(prompt)), enc=enc[j:j + 1])
                checked += rep["n_checked"]
                min_gap = min(min_gap, rep["min_gap"])
                if not rep["match"] and bad is None:
                    bad = dict(rep["first_divergence"], window=int(i), token=rep["first_divergence"]["index"] - len(prompt))
    return {"windows_checked": len(which), "of_windows": n_windows, "tokens_checked": checked, "match": bad is None, "first_divergence": bad,
            "min_top2_gap": min_gap, "seconds": time.perf_counter() - t0,
            "method": "teacher-forced oracle pass per window + processor-chain replay; GPU ids must be the argmax everywhere"}


def first_stream_divergence(a, b):
    for w, (x, y) in enumerate(zip(a, b)):
        if x != y:
            j = next((k for k in range(min(len(x), len(y))) if x[k] != y[k]), min(len(x), len(y)))
            return {"window": w, "token": j, "resident": x[j] if j < len(x) else None, "e2e": y[j] if j < len(y) else None}
    return None if len(a) == len(b) else {"window": min(len(a), len(b)), "token": 0, "resident": None, "e2e": None}


def dump_outputs(out_dir: str, streams, pos, suffix: str = "") -> None:
    """What one step of the resident path returns, as .npy files: tokens (songs, windows, new tokens) float64 generated ids (-1
    pads a window that stopped early) and, with the DiT stage, positions (songs, 2, points) float32 osu! pixels."""
    os.makedirs(out_dir, exist_ok=True)
    tokens = np.full((len(streams), len(streams[0]), max(len(w) for st in streams for w in st)), -1.0)
    for k, st in enumerate(streams):
        for i, w in enumerate(st):
            tokens[k, i, :len(w)] = w
    np.save(os.path.join(out_dir, f"tokens{suffix}.npy"), tokens)
    if pos is not None:
        np.save(os.path.join(out_dir, f"positions{suffix}.npy"), torch.stack(pos).float().cpu().numpy())


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--song-seed", type=int, default=0, help="rank r decodes synth_song(song_seed + r)")
    ap.add_argument("--songs-per-gpu", type=int, default=1,
                    help="songs decoded in lock-step per GPU per step (BASELINE configs[3]: 8 -> 64 songs on 8 GPUs); rank r takes songs "
                         "song_seed + r*S .. +S-1; window i of all S songs is one batch-S generate() call")
    ap.add_argument("--dit", type=int, default=1, help="1 = include the osu_diffusion stage the metric names (default), 0 = decode only")
    ap.add_argument("--cpu-windows", type=int, default=4, help="windows per CPU step (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--oracle-check", default="full", choices=["full", "sample", "none"],
                    help="N=1: teacher-forced oracle check of the GPU's greedy ids over the whole song / every 8th window / not at all")
    ap.add_argument("--pdl", type=int, default=int(os.environ.get("MB200_PDL", "0")))
    ap.add_argument("--windows", type=int, default=0, help="debug: truncate the song to this many windows")
    ap.add_argument("--tc", type=int, default=int(os.environ.get("MB200_TC", "1")), help="1 = tcgen05 3xTF32 GEMMs where eligible, 0 = fp32 SIMT GEMM everywhere")
    ap.add_argument("--mega", type=int, default=2, help="2 = dataflow token-loop megakernel (default), 1 = grid-barrier megakernel, 0 = CUDA-graph replay per token")
    ap.add_argument("--cpu-threads", type=int, default=int(os.environ.get("MB200_CPU_THREADS", "0")),
                    help="torch threads of the CPU arm (0 = min(cores, 16): measured best on the GPU box; 32+ threads slow a batch-1 decoder down)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--impl b200: write the token ids and DiT positions of the last timed step to DIR/tokens.npy, "
                         "DIR/positions.npy (with several ranks: tokens_rank<r>.npy, ...) to compare two builds output for output")
    args = ap.parse_args()
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from mapperatorinator_b200 import _lib
    from mapperatorinator_b200.diffusion import B200DiT, sample_sequence
    from mapperatorinator_b200.modeling import B200Mapperatorinator
    from mapperatorinator_b200.audio import load_pcm
    from mapperatorinator_b200.pipeline import SongDecoder
    from mapperatorinator_b200.server import model_generate
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(dev))
    cfg = v29_model_config()
    layout = TokenLayout.from_json(os.path.join(ROOT, "tests", "golden", "tokenizer_v29.json"))
    sd = init_model_state_dict(cfg, 0)                       # same weights on every rank
    S = max(1, args.songs_per_gpu)
    song_ids = [args.song_seed + rank * S + k for k in range(S)]      # rank r decodes songs song_seed + r*S .. + S-1
    song_id = song_ids[0]
    # the song enters as its file holds it: 44.1 kHz 16-bit stereo PCM; ingest (resample + mono + normalise) runs on the GPU (audio.load_pcm)
    pcm_host = [torch.from_numpy(synth_song_pcm(sid)).pin_memory() for sid in song_ids]
    pcm_dev = [t.to(dev) for t in pcm_host]
    songs = [segment_device(load_pcm(t, FILE_RATE, MODEL_RATE), cfg).cpu() for t in pcm_dev]
    if args.windows:
        songs = [w[:args.windows] for w in songs]
    windows = songs[0]
    n_windows = windows.shape[0]
    model = B200Mapperatorinator(cfg, sd, max_windows=S * n_windows, max_batch=max(2, S), device=dev)
    if args.pdl:
        model.engine.set_option("pdl", 1)
    model.engine.set_option("mega", args.mega)
    if os.environ.get("MB200_LL_REPS"):
        model.engine.set_option("ll_reps", int(os.environ["MB200_LL_REPS"]))
    if os.environ.get("MB200_LL_SLEEP"):
        model.engine.set_option("ll_sleep", int(os.environ["MB200_LL_SLEEP"]))
    song = SongDecoder(model, layout)
    all_windows = torch.stack(songs)                                   # (S, n_windows, samples)
    pinned = all_windows.pin_memory()
    resident = all_windows.to(dev)
    lib = _lib.load()
    lib.mb200_set_tensor_cores(int(args.tc))
    dit = None
    if args.dit:
        dc = dit_b_config(DIT_CLASSES)
        dsd = init_dit_state_dict(dc, 1)
        dit = B200DiT(dc, dsd, max_seq_len=DIT_GEOMETRY["max_seq_len"], device=dev)
        hits = [synth_hit_objects(sid) for sid in song_ids]
        seq_x, seq_c, y, y_null = hits[0]
        hit_pinned = [[t.pin_memory() for t in h] for h in hits]
        hit_resident = [[t.to(dev) for t in h] for h in hits]
        noise_gen = torch.Generator(device=dev)

    def refine(inputs, sid):
        """Stage (iii) through the public API; per-step noise drawn on the device from a seeded generator (the reference draws
        `th.randn_like` per step, gaussian_diffusion.py:454)."""
        noise_gen.manual_seed(77 + sid)
        noise = [torch.randn(DIT_STEPS, 2, 2, b - a, device=dev, generator=noise_gen) for a, b in dit_chunks()]
        return sample_sequence(dit, inputs[0], inputs[1], inputs[2], inputs[3], 1.0, step_noise=noise, **DIT_GEOMETRY)

    stage_ms = {"encode": 0.0, "decode": 0.0, "dit": 0.0}

    def step_resident():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        for k in range(S):
            w = segment_device(load_pcm(pcm_dev[k], FILE_RATE, MODEL_RATE), cfg)          # 44.1 kHz stereo int16 (resident) -> 16 kHz mono windows
            song.encode_song(w[:n_windows], slot_begin=k * n_windows)
        ev[1].record()
        if S == 1:
            streams = [song.decode_windows(n_windows, prompt_for, lambda i: gen_kwargs(i, n_windows, 18 if i == 0 else 50))]
        else:
            streams = song.decode_songs(S, n_windows, lambda k, i, st: prompt_for(i, st), lambda i: gen_kwargs(i, n_windows, 18 if i == 0 else 50))
        ev[2].record()
        pos = [refine(hit_resident[k], song_ids[k]) for k in range(S)] if dit is not None else None
        ev[3].record()
        if world > 1:
            gather_token_streams([sum(st, []) for st in streams], song_ids)
        step_resident.events.append(ev)
        return sum(len(w) for st in streams for w in st), streams, pos
    step_resident.events = []

    def step_e2e():
        streams, toks = [[] for _ in range(S)], 0
        for k in range(S):        # where the reference runs load_audio_file + Preprocessor.segment: host PCM in, host windows out
            x = load_pcm(pcm_host[k], FILE_RATE, MODEL_RATE).cpu().numpy()
            pinned[k].copy_(segment(x, cfg)[0][:n_windows])
        for i in range(n_windows):
            prompt = torch.tensor([prompt_for(i, streams[k]) for k in range(S)])
            ids, stats = model_generate(model, layout, dict(inputs=pinned[:, i], decoder_input_ids=prompt, decoder_attention_mask=prompt.ne(0)),
                                        gen_kwargs(i, n_windows, prompt.shape[1]))
            for k in range(S):
                streams[k].append(ids[k, prompt.shape[1]:].tolist())
            toks += stats["generated_tokens"]
        pos = [refine(hit_pinned[k], song_ids[k]).cpu() for k in range(S)] if dit is not None else None
        if world > 1:
            gather_token_streams([sum(st, []) for st in streams], song_ids)
        return toks, streams, pos

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        step_resident.events = []
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.mb200_launch_count()
        mstats = np.zeros(3, dtype=np.float64)
        lib.mb200_model_mega_stats(model.engine.handle, mstats.ctypes.data, 1)      # reset the megakernel event counters
        e0.record()
        toks = 0
        for _ in range(steps):
            t, streams, pos = fn()
            toks += t
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        launches = lib.mb200_launch_count() - l0
        lib.mb200_model_mega_stats(model.engine.handle, mstats.ctypes.data, 0)
        timed.mega = mstats.copy()
        if world > 1:
            tt = torch.tensor([ms, float(toks)], device=dev, dtype=torch.float64)
            mx = tt.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            sm = tt.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            ms, toks = float(mx[0]), float(sm[1])
        return ms, toks, launches, streams, pos

    with ClockSampler(local) as clk:
        ms, toks, launches, streams, pos = timed(step_resident, args.steps, args.warmup)
    clocks = clk.summary()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, streams, pos, f"_rank{rank}" if world > 1 else "")
    for ev in step_resident.events:
        stage_ms["encode"] += ev[0].elapsed_time(ev[1]); stage_ms["decode"] += ev[1].elapsed_time(ev[2]); stage_ms["dit"] += ev[2].elapsed_time(ev[3])
    n_ev = max(1, len(step_resident.events))
    stage_ms = {k: v / n_ev for k, v in stage_ms.items()}
    mega_resident, ms_resident = timed.mega, ms
    e2e_steps = max(1, args.steps // 2)
    ms_e2e, toks_e2e, _, streams2, pos2 = timed(step_e2e, e2e_steps, 1)
    # the two arms must emit the same tokens (and positions): reported, not asserted, so every rank always prints / exits cleanly
    div = None
    for k in range(S):
        dk = first_stream_divergence(streams[k], streams2[k])
        if dk is not None:
            div = dict(dk, song=song_ids[k]); break
    consistency = {"resident_equals_e2e": div is None, "first_divergence": div}
    if dit is not None:
        consistency["positions_max_abs_diff"] = max(float((a.cpu() - b).abs().max()) for a, b in zip(pos, pos2))
    all_streams, all_streams2 = streams, streams2
    streams, streams2 = all_streams[0], all_streams2[0]                # song 0 of this rank feeds the CPU / oracle checks below
    if world > 1:
        flag = torch.tensor([0 if div is None else 1], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.SUM)
        consistency["ranks_diverged"] = int(flag.item())

    # ---- roofline of the dominant kernel, timed live with CUDA events on the launching stream --------------------------------
    d, f, V, L = cfg.d_model, cfg.ffn_dim, cfg.vocab_size_out, cfg.decoder_layers
    w_bytes = 4 * (L * (3 * d * d + 2 * d * d + d * d + 2 * d * f) + V * d)                  # decoder weights streamed once per token
    ctx = 50 + NEW_TOKENS // 2
    kv_bytes = 4 * L * 2 * (cfg.max_source_positions + ctx) * d                               # cross + self K/V read per token
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    traffic, traffic_src = None, None
    try:      # per-launch DRAM bytes of the token-loop kernel from the committed `ncu --set full` capture of this round
        tr = json.load(open(os.path.join(ROOT, "profiles", "megakernel_traffic.json")))
        traffic, traffic_src = tr["dram_bytes_per_launch"], tr["source"]
    except Exception:
        pass
    mega = mega_resident
    if args.mega and mega[0] > 0:
        # persistent token-loop kernel: one launch per window decodes NEW_TOKENS-1 tokens; events recorded around every launch
        tok_per_launch = mega[2] / mega[0]
        us_per_launch = 1000.0 * mega[1] / mega[0]
        bytes_per_launch = (w_bytes + kv_bytes) * tok_per_launch
        achieved = bytes_per_launch / (us_per_launch * 1e-6) / 1e9
        roofline = {"bound": "hbm", "kernel": ("decode_megakernel_ll<1> (dataflow megakernel" if args.mega >= 2 else "decode_megakernel<1> (grid-barrier megakernel")
                              + ": persistent cooperative kernel, all layers of all tokens of one generate() call)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic if traffic and abs(tok_per_launch - 63.0) < 1e-6 else None, "traffic_source": traffic_src,
                    "peak_source": peak_src, "bytes_per_launch": bytes_per_launch, "us_per_launch": us_per_launch, "tokens_per_launch": tok_per_launch,
                    "us_per_token": us_per_launch / tok_per_launch, "bytes_per_token": w_bytes + kv_bytes,
                    "share_of_step": mega[1] / (ms_resident), "token_floor_us": (w_bytes + kv_bytes) / (peak * 1e3)}
    else:
        out_us = np.zeros(4, dtype=np.float32)
        _lib.check(lib.mb200_model_profile_step(model.engine.handle, 1, 1, 50 + NEW_TOKENS, 20, out_us.ctypes.data, torch.cuda.current_stream().cuda_stream))
        n_gemv = int(out_us[3]) // 1000000
        gemv_us = float(out_us[0])
        achieved = (w_bytes / n_gemv) / (gemv_us / n_gemv * 1e-6) / 1e9 if gemv_us > 0 else None
        roofline = {"bound": "hbm", "kernel": f"gemv_kernel<1> ({n_gemv} launches per token, CUDA-graph path; eager event timing includes launch gaps)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if achieved else None, "traffic": None,
                    "peak_source": peak_src, "bytes_per_launch": w_bytes / n_gemv, "us_per_launch": gemv_us / n_gemv,
                    "per_token_us": {"gemv": gemv_us, "attention": float(out_us[1]), "sample": float(out_us[2])},
                    "token_floor_us": (w_bytes + kv_bytes) / (peak * 1e3)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    cpu, oracle_check, dit_parity, ingest_parity = None, None, None, None
    if not args.no_cpu_baseline and world == 1:
        cores = args.cpu_threads or min(os.cpu_count() or 1, 16)
        torch.set_num_threads(cores)
        cpu_windows = oracle_windows(song_id, cfg)[:n_windows]                # the reference's ingest arithmetic + Preprocessor.segment, on the CPU
        ingest_parity = {"gpu_windows_equal_reference_ingest": bool(torch.equal(cpu_windows, windows)), "windows": int(n_windows),
                         "samples_in": int(pcm_host[0].shape[0]), "file": "44.1 kHz 16-bit stereo", "model_rate": MODEL_RATE}
        windows = cpu_windows
        ctoks, csecs, sample, info = cpu_sample(args, cfg, layout, windows, n_windows, sd, streams)
        cpu = {"value": ctoks / csecs, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample, **info}
        if args.oracle_check != "none":
            which = list(range(n_windows)) if args.oracle_check == "full" else list(range(0, n_windows, 8))
            oracle_check = oracle_song_check(cfg, layout, sd, windows, streams, which)
            if div is not None and div["song"] == song_id:      # which arm disagrees with the oracle at the point where the two arms part?
                w = div["window"]
                consistency["oracle_on_e2e_window"] = oracle_song_check(cfg, layout, sd, windows, streams2[:w + 1] + streams[w + 1:], [w])
        if dit is not None:
            # diffusion parity sample: the fused on-device 100-step loop vs the oracle's p_sample_loop on one T = 256 chunk, same
            # injected noise, north_star tolerance 1e-3 abs in normalised coordinates
            from mapperatorinator_b200.diffusion import InpaintDenoiser, band_attention_mask, create_diffusion
            from oracle import dit as dit_oracle
            Tp = 256
            g = torch.Generator().manual_seed(5)
            x = torch.cat([seq_x[None, :, :Tp]] * 2); c = torch.cat([seq_c[None, :, :Tp]] * 2); yy = torch.stack([y, y_null], 0)
            noise = torch.randn(DIT_STEPS, 2, 2, Tp, generator=g)
            ipm = torch.ones_like(x, dtype=torch.bool); ipm[:, :, :32] = False
            t0 = time.perf_counter()
            with torch.no_grad():
                ref = dit_oracle.p_sample_loop(dsd, dc, dit_oracle.Schedule(), x, c, yy, 1.0, dit_oracle.band_mask(Tp, 128), noise, inpaint_mask=ipm)
            t_ref = time.perf_counter() - t0
            diff = create_diffusion([DIT_STEPS] + [0] * 9, "squaredcos_cap_v2", 1000)
            mk = dict(c=c.to(dev), y=yy.to(dev), cfg_scale=1.0, attn_mask=band_attention_mask(Tp, 128, dev), key_padding_mask=None)
            got = diff.p_sample_loop(dit.forward_with_cfg, x.shape, x.to(dev), denoised_fn=InpaintDenoiser(ipm.to(dev), x.to(dev)), clip_denoised=True,
                                     model_kwargs=mk, step_noise=noise.to(dev)).cpu()
            err = float((got - ref).abs().max())
            dit_parity = {"chunk_points": Tp, "steps": DIT_STEPS, "max_abs_err": err, "tolerance": 1e-3, "ok": bool(err <= 1e-3), "oracle_seconds": t_ref}
    h2d = S * n_windows * cfg.samples_per_window * 4 + S * int(pcm_host[0].numel()) * 2      # per-window PCM + the file's int16 PCM for the ingest
    d2h = S * n_windows * (50 + NEW_TOKENS) * 8 + S * 4 * int(lib.mb200_audio_out_frames(int(pcm_host[0].shape[0]), FILE_RATE, MODEL_RATE))      # token ids + the ingested signal
    if dit is not None:
        h2d += S * 4 * (2 * DIT_POINTS + dc.context_size * DIT_POINTS + 2 * DIT_CLASSES)
        d2h += S * 4 * 2 * DIT_POINTS
    tok_per_song = toks / args.steps / world
    decode_only_ms = stage_ms["encode"] + stage_ms["decode"]
    print(json.dumps({
        "metric": METRIC if dit is not None else "event tokens/sec end-to-end", "value": toks / (ms / 1000), "unit": "tokens/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(n_windows, dit is not None, S), "clocks": clocks,
        "e2e": {"value": toks_e2e / (ms_e2e / 1000), "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "server.model_generate per window (host tensors in, CPU LongTensor out)"
                       + (" + diffusion.sample_sequence (host tensors in, CPU positions out)" if dit is not None else "")},
        "value_decode_only": tok_per_song * world / (decode_only_ms / 1000) if decode_only_ms > 0 else None,
        "stages_ms_per_song": {**stage_ms, "note": "rank 0, resident arm, CUDA events: audio ingest + mel+encoder (all windows, batched) | prefill + token loop "
                                                   "(all windows) | DiT refinement (2 chunks x 100 steps)"},
        "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "self_consistency": consistency, "oracle_check": oracle_check,
        "dit_parity": dit_parity, "ingest_parity": ingest_parity, "pdl": bool(args.pdl), "tensor_cores": bool(args.tc), "song_seed": args.song_seed,
        "token_stream_sha1": hashlib.sha1(json.dumps(streams).encode()).hexdigest(),
        "token_stream_sha1_all_songs": hashlib.sha1(json.dumps(all_streams).encode()).hexdigest() if S > 1 else None}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except SystemExit:
        raise
    except BaseException:
        # a rank that dies must say who it was and why, on stdout (torchrun interleaves stderr and the driver keeps stdout)
        print(json.dumps({"rank": int(os.environ.get("RANK", 0)), "error": traceback.format_exc()}), flush=True)
        sys.exit(1)
