"""Host logic of bench.py (no GPU): the configurations it names are BASELINE.json's, the weak-scaling clip lengths and their
ideal efficiency follow the reference's window plan, the CPU-sample planner stays inside its size tables, and the roofline
traffic figure is read from the committed ncu summary (never a constant in the source)."""
import json
import os
import re

import bench
from upscale_a_video_b200 import sharding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_configs_are_the_baseline_configs():
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))["configs"]
    nums = [[int(x) for x in re.findall(r"\d+", c.replace("×", "x"))] for c in base]
    c2, c3, c4, c5 = bench.CONFIGS["c2"], bench.CONFIGS["c3"], bench.CONFIGS["c4"], bench.CONFIGS["c5"]
    # "8-frame 320x576 -> 1280x2304, 30 steps, guidance 6"
    assert nums[1][:3] == [8, c2["h"], c2["w"]] and bench.frames_for(1) == 8 and c2["steps"] == 30 and bench.GUIDANCE == 6.0
    assert nums[1][3:5] == [4 * c2["h"], 4 * c2["w"]]
    # "32-frame 320x576, 30 steps, propagation at [24,26,28], 4 GPUs"
    assert nums[2][:4] == [c3["frames"], c3["h"], c3["w"], c3["steps"]] and nums[2][4:7] == c3["prop"]
    # "64-frame 180x320 ... --use_video_vae"
    assert nums[3][:3] == [c4["frames"], c4["h"], c4["w"]] and c4["vae"] == "vae_video" and c4["steps"] == 30
    # "16-frame 540x960 -> 2160x3840 tile-overlap stress, 50 steps"
    assert nums[4][:3] == [c5["frames"], c5["h"], c5["w"]] and c5["tiled"] and c5["steps"] == nums[4][5] == 50


def test_weak_scaling_clip_lengths_and_ideal_efficiency():
    for n in (1, 2, 4, 8):
        T = bench.frames_for(n)
        wins = sharding.unique(sharding.unet_windows(T))
        assert len(wins) == n, (n, T, wins)                 # one 8-frame window per GPU, stride 6 (pipeline...:621-629)
        assert abs(T / (8.0 * n) - (6 * n + 2) / (8.0 * n)) < 1e-12   # frames per window-time: the `ideal_efficiency` field


def test_cpu_sample_planner_stays_inside_its_tables(monkeypatch):
    calls = []
    monkeypatch.setattr(bench, "_cpu_state", lambda: None)
    monkeypatch.setattr(bench, "_cpu_unet", lambda T, H, W: calls.append(("u", T, H, W)) or 2.0 * bench._unet_tflop(T, H, W))
    monkeypatch.setattr(bench, "_cpu_vae", lambda H, W: calls.append(("v", H, W)) or 4.0 * bench._vae_tflop(H, W))
    small = bench.cpu_plan(1e-9)
    assert small == (bench._UNET_SIZES[0], bench._VAE_SIZES[0])
    big = bench.cpu_plan(1e9)
    assert big == (bench._UNET_SIZES[-1], bench._VAE_SIZES[-1])
    us, vs = bench.cpu_plan(10.0)       # 2 s / TFLOP UNet, 4 s / TFLOP VAE
    assert bench._unet_tflop(*us) * 2.0 <= 7.5 and bench._vae_tflop(*vs) * 4.0 <= 2.5
    assert us in bench._UNET_SIZES and vs in bench._VAE_SIZES
    # FLOP models: linear in T*H*W for the UNet, conv + quadratic attention term for the VAE
    assert abs(bench._unet_tflop(8, 320, 576) - bench.UNET_TFLOP_PER_FWD_C2) < 1e-9
    assert abs(bench._vae_tflop(320, 576) - bench.VAE_TFLOP_PER_3F_C2) < 1e-9


def test_host_threads_is_bounded():
    n = bench.host_threads()
    assert 1 <= n <= 32 and n <= (os.cpu_count() or 1)


def test_dump_outputs_is_float32_bounded_and_reproducible(tmp_path, monkeypatch):
    import numpy as np
    import torch
    assert bench.DUMP_SAMPLES * 4 + 128 <= 64 << 20     # one float32 .npy (header included) per output, 64 MB in all
    monkeypatch.setattr(bench, "DUMP_SAMPLES", 1000)
    small = torch.randn(2, 3, 4, dtype=torch.float16)
    big = torch.arange(5000, dtype=torch.float64).reshape(1, 5, 1000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"small": small, "big": big})
    a_small, a_big = np.load(tmp_path / "a" / "small.npy"), np.load(tmp_path / "a" / "big.npy")
    assert a_small.dtype == np.float32 and a_small.shape == (2, 3, 4) and np.array_equal(a_small, small.float().numpy())
    assert a_big.dtype == np.float32 and a_big.shape == (1000,)
    assert np.all(np.diff(a_big) >= 0) and np.all(a_big == np.round(a_big))       # sorted positions of the flat output
    assert np.array_equal(a_big, np.load(tmp_path / "b" / "big.npy"))            # same positions on every run


def test_roofline_traffic_comes_from_the_committed_ncu_summary():
    prof = bench._ncu_profile_of_dominant_kernel()
    raw = json.load(open(os.path.join(ROOT, "profiles", "ncu_igemm_representative.json")))
    assert prof is not None and prof["dram_bytes_per_launch"] == raw["dram_bytes_read"] + raw["dram_bytes_write"]
    algorithmic = 2 * (16 * 160 * 288 * 512 * 2) + 512 * 9 * 512 * 2      # the representative launch of bench.py
    assert 0.9 < prof["dram_bytes_per_launch"] / algorithmic < 1.2         # ncu: traffic ~= algorithmic bytes
