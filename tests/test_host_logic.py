"""Host-side logic (no GPU): token layout / flag bytes, schedule tables, filterbanks, mask classification, window
segmentation, generation stats, song sharding and the world_size-2 token gather over gloo."""
import os
import sys

import numpy as np
import pytest
import torch

from mapperatorinator_b200 import MelConfig, TokenLayout, v29_model_config
from mapperatorinator_b200.filterbank import mel_filterbank
from mapperatorinator_b200.pipeline import segment, shard_songs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_layout_matches_v29_facts(layout):
    assert layout.vocab_size_out == 3667 and (layout.time_shift_start, layout.time_shift_end) == (17, 836)    # SURVEY §8
    eos = layout.eos_token_ids(4092.0, 3273.6, "map")
    assert eos[:2] == [2, 10] and eos[2] == 17 and eos[2 + 408] == 17 + 408 and eos[-1] == 835 and len(eos) == 2 + 409 + 327   # A.3
    assert layout.lookback_end(4092.0) == 17 + 409
    assert set(layout.sos_ids()) == {1, 3, 5, 7, 9, 11, 13, 15}


def test_vflags(layout):
    from mapperatorinator_b200.engine import VF_BEAT, VF_EOS, VF_LB_EOS, VF_SOS, VF_TIMED, build_vflags
    f = build_vflags(layout, layout.eos_token_ids(0.0, 0.0, "map"))
    assert f.shape == (layout.vocab_size_in,)
    assert f[2] & VF_EOS and f[10] & VF_EOS and not f[17] & VF_EOS
    assert f[1] & VF_SOS and f[9] & VF_SOS and f[10] & VF_LB_EOS
    assert f[layout.event_start["circle"]] & VF_TIMED and f[layout.event_start["beat"]] & VF_BEAT
    assert not f[layout.event_start["dist"]] & VF_TIMED


@pytest.mark.parametrize("cfg", [MelConfig(), MelConfig("torchaudio", n_mels=80), MelConfig("torchaudio", True, n_mels=128, f_min=20, pad_mode="reflect")])
def test_filterbank_matches_oracle(cfg):
    from oracle import mel as mo
    a, b = mel_filterbank(cfg), mo.mel_basis(cfg)
    assert a.shape == b.shape == (cfg.n_mels, 513)
    assert np.allclose(a, b, rtol=1e-5, atol=1e-8)
    assert ((a != 0).sum(0) <= 2).all()          # each FFT bin feeds at most two triangles (mel.cu CSR assumption is an optimisation only)


def test_schedule_rows_match_oracle():
    from mapperatorinator_b200.diffusion import create_diffusion
    from oracle import dit as do
    d = create_diffusion([100, 0, 0, 0, 0, 0, 0, 0, 0, 0], "squaredcos_cap_v2", 1000)
    s = do.Schedule()
    assert d.timestep_map == s.timestep_map == list(range(100))         # SURVEY A.4
    rows = d.schedule_rows()
    assert np.array_equal(rows[::-1, 0], np.arange(100, dtype=np.float32)) and rows[-1, 7] == 0 and rows[0, 7] == 1
    assert np.allclose(rows[::-1, 1:7], s.table()[:, 1:7], rtol=0, atol=0)


def test_mask_classification():
    from mapperatorinator_b200.diffusion import _classify_mask
    from oracle.dit import band_mask
    assert _classify_mask(None)[0] == "none"
    assert _classify_mask(band_mask(300, 128))[:2] == ("band", 128)
    assert _classify_mask(band_mask(64, 128))[0] == "band"               # fully open band when T < width
    m = band_mask(100, 16); m[3, 50] = False
    mode, _, dense = _classify_mask(m)
    assert mode == "dense" and dense.dtype == torch.uint8


def test_segment_matches_reference_arithmetic():
    cfg = v29_model_config()
    x = np.random.default_rng(0).standard_normal(2_880_000).astype(np.float32)
    w, t, length = segment(x, cfg)
    assert w.shape == (211, 130944) and length == 180000.0                # SURVEY §8a a1
    assert t[1].item() == int(13094 * 1000 / 16000) and np.array_equal(w[1, :10].numpy(), x[13094:13104])
    wp, _, _ = segment(x, cfg, parallel=True)
    assert wp.shape == (22, 130944)


def test_segment_device_equals_segment():
    """`segment_device` (windows cut from a resident signal) against `segment` on the same samples: every length class of the padding rule."""
    from mapperatorinator_b200.pipeline import segment_device
    cfg = v29_model_config()
    S, stride = cfg.samples_per_window, int(cfg.samples_per_window * (1 - 0.5 - 0.4))
    rng = np.random.default_rng(1)
    for n in (1, S - 1, S, S + 1, S + stride, S + stride + 7, 3 * S + 5):
        x = rng.standard_normal(n).astype(np.float32)
        for parallel in (False, True):
            w, _, _ = segment(x, cfg, parallel=parallel)
            wd = segment_device(torch.from_numpy(x), cfg, parallel=parallel)
            assert wd.shape == w.shape and torch.equal(wd, w), (n, parallel)


def test_generation_stats_accounting():
    from mapperatorinator_b200.server import _build_generation_stats
    res = torch.tensor([[0, 5, 6, 7, 8, 0], [4, 5, 6, 7, 0, 0]])
    mk = dict(decoder_input_ids=res[:, :3], decoder_attention_mask=res[:, :3].ne(0))
    st = _build_generation_stats(res, mk, 0, 2.0)
    assert st["generated_tokens_per_sample"] == [2, 1] and st["generated_tokens"] == 3 and st["tokens_per_second"] == 1.5


def test_shard_songs_balanced():
    lengths = [150 + (7 * i) % 61 for i in range(64)]
    shards = shard_songs(lengths, 8)
    assert sorted(sum(shards, [])) == list(range(64)) and all(len(s) == 8 for s in shards)
    loads = [sum(lengths[i] for i in s) for s in shards]
    assert max(loads) - min(loads) <= 61


def _gather_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    from mapperatorinator_b200.pipeline import gather_token_streams
    local = {0: ([[1, 2, 3], [4]], [0, 2]), 1: ([[9, 8, 7, 6, 5]], [1])}[rank]
    out = gather_token_streams(local[0], local[1])
    q.put((rank, out))
    dist.destroy_process_group()


def test_gather_token_streams_gloo_world2():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    ps = [ctx.Process(target=_gather_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in ps]
    res = dict(q.get(timeout=120) for _ in range(2))
    [p.join(60) for p in ps]
    assert res[1] is None
    assert res[0] == {0: [1, 2, 3], 2: [4], 1: [9, 8, 7, 6, 5]}


def test_product_refuses_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from mapperatorinator_b200 import tiny_model_config
    from mapperatorinator_b200.engine import ModelEngine
    with pytest.raises(RuntimeError):
        ModelEngine(tiny_model_config(), {})


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm) prints ONE JSON line with the contract's keys;
    bounded sample: one window here."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-windows", "1",
                          "--cpu-threads", "8"], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "event tokens/sec end-to-end (mel+T5+DiT)" and d["unit"] == "tokens/s"
    assert d["cpu_baseline"]["dit_steps_run"] >= 2 and 0 < d["cpu_baseline"]["dit_steps_charged"] < 1.0     # 1 of 211 windows -> 0.95 of the 200 chunk-steps
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "f32"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 8 and d["cpu_baseline"]["value"] == d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["windows"] == 211 and "workload" in d["config"]


def test_clock_sampler_parses_nvidia_smi_rows():
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    cs = bench.ClockSampler(0)
    cs.rows = ["1965, 1965, Not Active, Not Active, Not Active, Active\n", "1950, 1965, Not Active, Not Active, Not Active, Not Active\n",
               "garbage\n", "1965, 1965, Not Active, Active, Not Active, Not Active\n"]
    s = cs.summary()
    assert s["sm_mhz"] == 1965.0 and s["sm_max_mhz"] == 1965.0 and s["samples"] == 3
    assert s["reasons"] == ["hw_thermal_slowdown", "sw_power_cap"]


def test_bench_dump_outputs(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    streams = [[[5, 6, 7], [8, 9]], [[1, 2, 3], [4, 5, 6]]]
    pos = [torch.full((2, 4), 1.5), torch.full((2, 4), 2.5)]
    bench.dump_outputs(str(tmp_path / "out"), streams, pos, "_rank1")
    tok = np.load(tmp_path / "out" / "tokens_rank1.npy")
    assert tok.dtype == np.float64 and tok.shape == (2, 2, 3)
    assert tok[0].tolist() == [[5, 6, 7], [8, 9, -1]] and tok[1].tolist() == [[1, 2, 3], [4, 5, 6]]
    p = np.load(tmp_path / "out" / "positions_rank1.npy")
    assert p.dtype == np.float32 and p.shape == (2, 2, 4) and p[1].min() == 2.5
    bench.dump_outputs(str(tmp_path / "dec"), streams, None)
    assert sorted(os.listdir(tmp_path / "dec")) == ["tokens.npy"]


def test_trim_predicted_tokens_properties(layout):
    from mapperatorinator_b200.pipeline import trim_predicted_tokens
    from oracle import cases
    ts, te = layout.time_shift_start, layout.time_shift_end
    for toks, tlb, tla in cases.trim_cases(layout):
        for types_first in (True, False):
            out = trim_predicted_tokens(toks, layout, "map", 4092.0, 4910.4, tlb, tla, types_first)
            stripped = list(toks)
            while stripped and stripped[-1] in (layout.eos_id, layout.context_eos["map"]):
                stripped.pop()
            assert out == stripped[:len(out)] and len(stripped) - len(out) in (0, 1, 2)
            if len(out) != len(stripped):
                last = stripped[-1]
                assert ts <= last < te and ((tla and last >= layout.lookback_end(4910.4)) or (tlb and last < layout.lookback_end(4092.0)))
                assert len(stripped) - len(out) == min(len(stripped), 2 if types_first else 1)


def test_trim_predicted_tokens_matches_reference(layout):
    """The reference's own `Processor.add_predicted_tokens_to_context` (processor.py:1022-1052) run on a stand-in `self` that records what
    reaches `_decode` (tests/golden/reference_pins.npz) — the token-level result this repo's `trim_predicted_tokens` must reproduce."""
    from mapperatorinator_b200.pipeline import trim_predicted_tokens
    from oracle import cases
    pins = np.load(os.path.join(ROOT, "tests", "golden", "reference_pins.npz"))
    off, ref = pins["trim_offsets"], pins["trim_tokens"]
    runs = [(types_first, c) for types_first in (True, False) for c in cases.trim_cases(layout)]
    assert len(runs) == len(off) - 1
    for k, (types_first, (toks, tlb, tla)) in enumerate(runs):
        want = ref[off[k]:off[k + 1]].tolist()
        assert want == trim_predicted_tokens(toks, layout, "map", 4092.0, 4910.4, tlb, tla, types_first), (toks, tlb, tla, types_first)
