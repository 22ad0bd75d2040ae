#!/usr/bin/env python
"""bench.py — upscaled frames/sec of the Upscale-A-Video sampling path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # uav_b200 arm (N>1: launched by torch.distributed.run)
    python bench.py --impl reference [--gpus N] ...              # reference arm: the path's own CPU implementation
    python bench.py ... --dump-outputs DIR                       # also write the last timed step's frames to DIR/*.npy

One "step" = one full pass of the hot path over one synthetic clip: `VideoUpscalePipeline.__call__` with 30 DDIM
steps (chunked UNet, CFG, step_v0, flow propagation at steps 24/26/28, step_vt) followed by the chunked VAE decode.
N=1 runs BASELINE.json configs[1] ("c2"): 8 frames 320x576 -> 1280x2304, guidance 6, fp16.  N>1 is weak scaling: the clip
has 8 + 6*(N-1) frames, i.e. exactly N unique 8-frame UNet windows per DDIM step (one per rank) and ceil(T/3) decode
chunks dealt over ranks; one NCCL all_gather per DDIM step + one at the end (upscale_a_video_b200/sharding.py).
`--config c3|c4|c5|clip64` (hidden; recorded into profiles/ by hand) select the other BASELINE configs.

`value`: frames/s with inputs resident in HBM, CUDA-event timed, max over ranks.  `e2e`: same through the public API
with pinned HOST buffers (H2D of the LR clip + flows, D2H of the decoded frames inside the timed region).
`reference_gpu` (N=1): the reference's own op sequence (oracle restatement = the same torch / cuDNN / cuBLAS calls) in the
reference's precision mode (fp16 UNet + sampler, fp32 VAE) on the same GPU, same clip, same timing window
(inference_upscale_a_video.py:205-206,335-338) — north_star's ">= 4x the reference's single-B200 fp16 path" denominator.
`cpu_baseline` / `--impl reference`: the oracle on the host cores, on a bounded sample (UNet forward + VAE decode chunk +
sampler step at reduced size), each part scaled to config 2 by its algorithmic FLOPs.
Weights are random-init (no checkpoints offline), inputs synthetic (seeded) — see `data`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

# algorithmic work (SURVEY.md §8d, BASELINE.md §3)
UNET_TFLOP_PER_FWD_C2 = 319.96     # B=2, T=8, 320x576
VAE_CONV_TFLOP_PER_3F_C2 = 85.6    # 3-frame chunk, 320x576, vae_3d: convolutions + projections
VAE_ATTN_TFLOP_PER_3F_C2 = 209.0   # ... single-head d=512 attention over 184 320 positions
VAE_TFLOP_PER_3F_C2 = VAE_CONV_TFLOP_PER_3F_C2 + VAE_ATTN_TFLOP_PER_3F_C2
GUIDANCE, NOISE_LEVEL = 6.0, 120
E2E_MAX_STEPS = 3                 # clips of the end-to-end leg (each is a full 30-step clip with H2D / D2H inside)
REFERENCE_GPU_DEADLINE_S = 480    # the reference-op-sequence leg starts only if the run is younger than this

# BASELINE.json configs (SURVEY.md §8d).  `frames=None`: weak scaling, 8 + 6 (N - 1) frames.
CONFIGS = {
    "c2": dict(frames=None, h=320, w=576, steps=30, prop=[24, 26, 28], vae="vae_3d", tiled=False),
    "c3": dict(frames=32, h=320, w=576, steps=30, prop=[24, 26, 28], vae="vae_3d", tiled=False),
    "c4": dict(frames=64, h=180, w=320, steps=30, prop=[24, 26, 28], vae="vae_video", tiled=False),
    "c5": dict(frames=16, h=540, w=960, steps=50, prop=[40, 44, 48], vae="vae_3d", tiled=True),
    "clip64": dict(frames=64, h=320, w=576, steps=30, prop=[24, 26, 28], vae="vae_3d", tiled=False),
}


def frames_for(n_gpus):
    return 8 + 6 * (n_gpus - 1)


def synth_inputs(T, H, W, device):
    g = torch.Generator().manual_seed(0)
    image = torch.rand(1, 3, T, H, W, generator=g) * 2 - 1
    yy, xx = torch.meshgrid(torch.arange(H).float(), torch.arange(W).float(), indexing="ij")
    fw = torch.stack([3.0 * torch.sin(yy / 7.0 + 0.3) + 0 * xx, 3.0 * torch.cos(xx / 5.0) + 0 * yy])
    g1 = torch.Generator().manual_seed(1)
    fw = fw[None, :, None].repeat(1, 1, T - 1, 1, 1) + 0.5 * torch.randn(1, 2, T - 1, H, W, generator=g1)
    bw = -fw + 0.4 * torch.randn(1, 2, T - 1, H, W, generator=g1)
    g2 = torch.Generator().manual_seed(2)
    pe = torch.randn(2, 77, 1024, generator=g2) * 0.3
    return image, fw, bw, pe


def _shapes(kind):
    return json.load(open(os.path.join(ROOT, "tests", "golden", f"shapes_{kind}.json")))


def _cfg(kind):
    return json.load(open(os.path.join(ROOT, "upscale_a_video_b200", "configs", f"{kind}_config.json")))


SCHED = dict(beta_schedule="scaled_linear", clip_sample=False, steps_offset=1, prediction_type="v_prediction",
             set_alpha_to_one=False)  # SD-x4-upscaler style (SURVEY.md §8a a16)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region"""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def build_pipeline(device, vae_kind="vae_3d"):
    from upscale_a_video_b200 import (AutoencoderKLVideo, DDIMScheduler, DDPMScheduler, Propagation, UNetVideoModel,
                                      VideoUpscalePipeline)
    from upscale_a_video_b200.synthetic import seeded_state_dict  # deterministic random init (no checkpoints offline)
    unet = UNetVideoModel.from_config(_cfg("unet_video"))
    unet.load_state_dict(seeded_state_dict(unet, 1234), strict=True)
    unet = unet.half().eval().to(device)
    vae = AutoencoderKLVideo.from_config(_cfg(vae_kind))
    vae.load_state_dict(seeded_state_dict(vae, 4321), strict=True)
    vae = vae.eval().to(device)
    return VideoUpscalePipeline(text_encoder=None, tokenizer=None, low_res_scheduler=DDPMScheduler(beta_schedule="scaled_linear"),
                                scheduler=DDIMScheduler(**SCHED), vae=vae, unet=unet, propagator=Propagation(4, learnable=False))


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle (CPU port of the reference path) on a bounded sample
# ------------------------------------------------------------------------------------------------
_CPU = {}
# (T, H, W) of the oracle UNet forward (B=2) and (H, W) of the 3-frame VAE decode chunk, smallest to largest
_UNET_SIZES = [(1, 16, 16), (1, 32, 32), (2, 32, 32), (2, 48, 48), (2, 64, 64), (4, 64, 64), (4, 64, 96), (4, 96, 128)]
_VAE_SIZES = [(8, 8), (16, 16), (24, 24), (32, 32), (48, 48), (64, 64)]


def _unet_tflop(T, H, W):
    # UNet work scales ~linearly in T*H*W away from the (small) self-attention term (SURVEY.md §8d)
    return UNET_TFLOP_PER_FWD_C2 * (T * H * W) / (8 * 320 * 576)


def _vae_tflop(H, W):
    r = (H * W) / (320 * 576)
    return VAE_CONV_TFLOP_PER_3F_C2 * r + VAE_ATTN_TFLOP_PER_3F_C2 * r * r


def host_threads():
    """threads for the CPU legs: the cores this process may actually use (affinity mask and cgroup quota — `os.cpu_count()`
    reports the whole host, 128 on the GPU boxes, where 128 torch threads on these small tensors ran 100x slower than 16),
    capped at 32: torch's CPU conv / GEMM kernels stop scaling there for the sample sizes that fit the time budget."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, min(n, 32))


def _cpu_state():
    if not _CPU:
        from oracle.weights import make_state_dict
        _CPU["usd"] = make_state_dict(_shapes("unet"), 1234)
        _CPU["vsd"] = make_state_dict(_shapes("vae_3d"), 4321)
        _CPU["ucfg"], _CPU["vcfg"] = _cfg("unet_video"), _cfg("vae_3d")
        torch.set_num_threads(host_threads())   # stated in `cores`
    return _CPU


def _cpu_unet(T, H, W):
    from oracle import uav_oracle as O
    st = _cpu_state()
    g = torch.Generator().manual_seed(0)
    sample, low = torch.randn(2, 4, T, H, W, generator=g), torch.randn(2, 3, T, H, W, generator=g)
    ctx = torch.randn(2, 77, 1024, generator=g) * 0.3
    t0 = time.time()
    with torch.no_grad():
        O.unet_forward(st["usd"], st["ucfg"], sample, torch.tensor(500), low, ctx, torch.tensor([120]))
    return time.time() - t0


def _cpu_vae(H, W):
    from oracle import uav_oracle as O
    st = _cpu_state()
    g = torch.Generator().manual_seed(0)
    z, img = torch.randn(1, 4, 3, H, W, generator=g), torch.rand(1, 3, 3, H, W, generator=g)
    t0 = time.time()
    with torch.no_grad():
        O.vae_decode(st["vsd"], st["vcfg"], z, img, 1.0)
    return time.time() - t0


def _cpu_sampler(T, H, W):
    """CFG + step_v0 + propagation + step_vt of one DDIM step on a (1,4,T,H,W) latent (oracle, fp32)"""
    from oracle import uav_oracle as O
    g = torch.Generator().manual_seed(0)
    lat, pred2 = torch.randn(1, 4, T, H, W, generator=g), torch.randn(2, 4, T, H, W, generator=g)
    fw, bw = torch.randn(1, 2, T - 1, H, W, generator=g), torch.randn(1, 2, T - 1, H, W, generator=g)
    s = O.DDIM(**SCHED)
    s.set_timesteps(30)
    t0 = time.time()
    with torch.no_grad():
        u, c = pred2.chunk(2)
        p = u + GUIDANCE * (c - u)
        x0 = s.step_v0(p, s.timesteps[3], lat)
        x0 = O.propagation(x0, fw, bw, "nearest", "fuse", 0.5, 0.001, 0.05)
        s.step_vt(x0, p, s.timesteps[3], lat)
    return time.time() - t0


def cpu_plan(target_s):
    """pick the largest sample sizes whose predicted time fits `target_s` (calibrated on the smallest size)"""
    _cpu_state()
    _cpu_unet(*_UNET_SIZES[0])  # warm-up (thread pool, allocator)
    tu = _cpu_unet(*_UNET_SIZES[0]) / _unet_tflop(*_UNET_SIZES[0])   # s / TFLOP
    tv = _cpu_vae(*_VAE_SIZES[0]) / _vae_tflop(*_VAE_SIZES[0])
    us = _UNET_SIZES[0]
    for s in _UNET_SIZES:   # small tensors under-use the cores, so the calibration over-predicts: conservative
        if _unet_tflop(*s) * tu <= 0.75 * target_s:
            us = s
    vs = _VAE_SIZES[0]
    for s in _VAE_SIZES:
        if _vae_tflop(*s) * tv <= 0.25 * target_s:
            vs = s
    return us, vs


def cpu_sample(plan):
    """one bounded sample; each part scaled separately by its algorithmic FLOPs to one config-2 frame"""
    (T, H, W), (hv, wv) = plan
    tu, tv, ts = _cpu_unet(T, H, W), _cpu_vae(hv, wv), _cpu_sampler(8, 64, 64)
    wu, wv_ = _unet_tflop(T, H, W), _vae_tflop(hv, wv)
    per_frame_s = (tu * (30 * UNET_TFLOP_PER_FWD_C2 / 8) / wu      # 30 UNet forwards per 8 frames
                   + tv * (VAE_TFLOP_PER_3F_C2 / 3) / wv_           # decode, per frame
                   + ts * 3 * (320 * 576) / (64 * 64) / 8)          # 3 propagation steps per clip, per frame (+ cheap rest)
    return {"value": 1.0 / per_frame_s, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
            "seconds": tu + tv + ts,
            "sample": f"oracle (fp32, {torch.get_num_threads()} threads): UNet forward B=2,T={T},{H}x{W} ({wu:.2f} TFLOP) in {tu:.1f} s"
                      f" + vae_3d decode 3x{hv}x{wv} ({wv_:.3f} TFLOP) in {tv:.1f} s + one sampler step 8x64x64 in {ts:.2f} s;"
                      f" each part scaled by its algorithmic FLOPs to config 2 ({30 * UNET_TFLOP_PER_FWD_C2 / 8:.0f} + "
                      f"{VAE_TFLOP_PER_3F_C2 / 3:.0f} TFLOP per frame)"}


def run_reference_arm(args):
    """the reference's own CPU implementation of the path (oracle port; /root/reference does not exist on the GPU box).
    Each step is ONE bounded sample, sized once so that warmup + steps samples take ~2.5 minutes in total."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    n = args.warmup + args.steps
    t_start = time.time()
    plan = cpu_plan(max(1.0, 150.0 / max(n, 1)))
    vals, secs, cb = [], [], None
    for i in range(n):
        if i > 0 and (time.time() - t_start) / i * n > 270.0:  # slower host than calibrated: fall back to the smallest sample
            plan = (_UNET_SIZES[0], _VAE_SIZES[0])
        cb = cpu_sample(plan)
        if i >= args.warmup:
            vals.append(cb["value"])
            secs.append(cb["seconds"])
    v = sum(vals) / len(vals)
    cb["value"] = v
    T = frames_for(args.gpus)
    ms = 1000.0 * sum(secs) / len(secs)
    _emit({"impl": "reference", "metric": "upscaled frames/sec (30 DDIM steps, 320x576->4x)", "value": v,
           "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms, "frames_equivalent_per_step": v * ms / 1000.0,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic, random-init weights",
           "config": {"workload": f"{T}-frame 320x576->1280x2304, 30 DDIM steps, guidance 6 — CPU: each step is one bounded "
                                  "sample (UNet forward + VAE decode chunk + sampler step at reduced size), FLOP-scaled per part; "
                                  "value = frames_equivalent_per_step / (ms_per_step / 1000)"},
           "cpu_baseline": cb,
           "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


# ------------------------------------------------------------------------------------------------
# reference on the same GPU (north_star's >= 4x denominator)
# ------------------------------------------------------------------------------------------------
def reference_gpu_leg(device, h_image, h_fw, h_bw, pe, steps, prop):
    """the reference's op sequence (oracle restatement: the same torch ops the reference modules call -> cuDNN / cuBLAS
    kernels) in the reference's precision mode: UNet + sampler fp16 (`.half()`), VAE fp32 (pipeline...:668-669) with torch's
    default TF32 convolutions; cudnn.benchmark on; the N = 184 320 VAE attention through the faster of torch's fused SDPA and
    an exact row-blocked softmax (the reference's dense score matrix is 136 GB per frame and cannot run).  ONE full clip,
    timed like inference_upscale_a_video.py:205-206,335-338 (synchronize, pipeline call, output.cpu(), synchronize).
    Favourable to the reference: no per-step empty_cache() / .item() syncs (the reference has both)."""
    from oracle import uav_oracle as O
    from oracle.weights import make_state_dict
    bench_flag = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    try:
        usd = {k: v.to(device).half() for k, v in make_state_dict(_shapes("unet"), 1234).items()}
        vsd = {k: v.to(device) for k, v in make_state_dict(_shapes("vae_3d"), 4321).items()}
        ucfg, vcfg = _cfg("unet_video"), _cfg("vae_3d")
        T, H, W = h_image.shape[2:]
        pe16 = pe.to(device).half()

        def sync():
            torch.cuda.synchronize(device)

        with torch.no_grad():
            # warm-up: cuDNN autotuning of every conv shape (UNet forward, one decode chunk per attention variant)
            lat = torch.randn(2, 4, T, H, W, device=device, dtype=torch.float16)
            low = torch.randn(2, 3, T, H, W, device=device, dtype=torch.float16)
            O.unet_forward(usd, ucfg, lat, torch.tensor(500), low, pe16, torch.tensor([NOISE_LEVEL]))
            z = torch.randn(1, 4, 3, H, W, device=device)
            img = torch.rand(1, 3, 3, H, W, device=device)
            impl_ms = {}
            for impl in ("exact", "sdpa"):
                O.ATTN_LARGE_IMPL = impl
                try:
                    O.vae_decode(vsd, vcfg, z, img, 1.0)
                    sync()
                    t0 = time.time()
                    O.vae_decode(vsd, vcfg, z, img, 1.0)
                    sync()
                    impl_ms[impl] = 1000.0 * (time.time() - t0)
                except Exception as ex:  # e.g. no fused kernel for head_dim 512 fp32 -> math fallback OOM
                    impl_ms[impl] = None
                    torch.cuda.empty_cache()
                    print(f"[reference_gpu] VAE attention impl {impl} unavailable: {type(ex).__name__}", file=sys.stderr)
            ok = {k: v for k, v in impl_ms.items() if v is not None}
            O.ATTN_LARGE_IMPL = min(ok, key=ok.get)
            del lat, low, z, img
            torch.cuda.empty_cache()
            sync()
            t0 = time.time()
            gen = torch.Generator(device=device).manual_seed(10)
            image = h_image.to(device, non_blocking=True)
            flows = [h_fw.to(device, non_blocking=True), h_bw.to(device, non_blocking=True)]
            noise = torch.randn(image.shape, generator=gen, device=device, dtype=torch.float16)
            lat0 = torch.randn(1, 4, T, H, W, generator=gen, device=device, dtype=torch.float16)
            out = O.pipeline_call(usd, ucfg, vsd, vcfg, O.DDIM(**SCHED), O.DDIM(beta_schedule="scaled_linear"), image=image,
                                  prompt_embeds=pe16, noise=noise, latents=lat0, flows_bi=flows, num_inference_steps=steps,
                                  guidance_scale=GUIDANCE, noise_level=NOISE_LEVEL, propagation_steps=prop)
            out_h = out.cpu()
            sync()
            dt = time.time() - t0
            impl = O.ATTN_LARGE_IMPL
            O.ATTN_LARGE_IMPL = "exact"
        return {"value": T / dt, "unit": "frames/s", "seconds_per_clip": dt, "clips_timed": 1, "frames": int(T),
                "kind": "reference op sequence (oracle restatement, torch -> cuDNN/cuBLAS) on the same GPU",
                "precision": "UNet + sampler fp16, VAE fp32 (TF32 convolutions: torch default), cudnn.benchmark",
                "vae_attention": impl, "vae_decode_chunk_ms": impl_ms,
                "window": "synchronize; H2D inputs; pipeline call; output.cpu(); synchronize (inference_upscale_a_video.py:205-206,335-338)",
                "output_checksum": float(out_h.double().abs().mean())}
    finally:
        torch.backends.cudnn.benchmark = bench_flag


DUMP_SAMPLES = 1 << 23   # values kept per dumped output: 32 MB of float32


def dump_outputs(dirname, outputs):
    """Write each output tensor to `dirname/<name>.npy` as float32, so that two builds run with the same arguments can be
    compared value for value.  An output of more than DUMP_SAMPLES values is stored as the values at DUMP_SAMPLES flat
    positions drawn with a fixed seed and sorted: the same positions for the same shape, on every run."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLES:
            idx = torch.randint(t.numel(), (DUMP_SAMPLES,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(dirname, f"{name}.npy"), t.float().cpu().numpy())


_REAL_STDOUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries write there too (NCCL prints its version banner on
    communicator creation), so fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved fd."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def _emit(line: dict):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


def _ncu_profile_of_dominant_kernel():
    """DRAM traffic / tensor-pipe numbers of the representative igemm launch from the committed `ncu --set full` summary
    (profiles/ncu_igemm_representative.json, written by tools/summarize_ncu.py from a capture of the same launch)."""
    p = os.path.join(ROOT, "profiles", "ncu_igemm_representative.json")
    try:
        d = json.load(open(p))
        d["source"] = "profiles/ncu_igemm_representative.json"
        return d
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="uav_b200")
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help=argparse.SUPPRESS)
    ap.add_argument("--ddim-steps", type=int, default=0, help=argparse.SUPPRESS)  # debugging only
    ap.add_argument("--no-cpu-baseline", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-reference-gpu", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-e2e", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--warmup-ddim-steps", type=int, default=0, help=argparse.SUPPRESS)  # side configs: cheap warm-up clips
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned to DIR/<name>.npy (float32; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    t_start = time.time()
    _claim_stdout()
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch.distributed as dist
    from upscale_a_video_b200 import _lib, build, ops, sharding
    build.build()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)

    cfg = CONFIGS[args.config]
    T = cfg["frames"] or frames_for(args.gpus)
    H_LR, W_LR = cfg["h"], cfg["w"]
    ddim_steps = args.ddim_steps or cfg["steps"]
    pipe = build_pipeline(device, cfg["vae"])
    image, fw, bw, pe = synth_inputs(T, H_LR, W_LR, device)
    neg, pos = pe.half().to(device).chunk(2)
    prop = [s for s in cfg["prop"] if s < ddim_steps]
    kw = dict(num_inference_steps=ddim_steps, guidance_scale=GUIDANCE, noise_level=NOISE_LEVEL, propagation_steps=prop,
              prompt_embeds=pos, negative_prompt_embeds=neg)
    d_image, d_fw, d_bw = image.to(device), fw.to(device), bw.to(device)
    h_image, h_fw, h_bw = image.pin_memory(), fw.pin_memory(), bw.pin_memory()
    h_out = torch.empty(1, 3, T, 4 * H_LR, 4 * W_LR, dtype=torch.float32).pin_memory()

    def run_pipe(img, flows, gen):
        if cfg["tiled"]:
            from upscale_a_video_b200.tiling import upscale_tiled   # inference_upscale_a_video.py:200-304
            return upscale_tiled(pipe, img, flows, generator=gen, tile_size=256, overlap=64, **kw)
        return pipe(None, image=img, flows_bi=flows, generator=gen, **kw).images

    def step_resident():
        gen = torch.Generator(device=device).manual_seed(10)  # inference_upscale_a_video.py:197
        return run_pipe(d_image, [d_fw, d_bw], gen)

    def step_e2e():
        gen = torch.Generator(device=device).manual_seed(10)
        img = h_image.to(device, non_blocking=True)
        flows = [h_fw.to(device, non_blocking=True), h_bw.to(device, non_blocking=True)]
        out = run_pipe(img, flows, gen)
        h_out.copy_(out, non_blocking=True)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        """ms of k calls of fn, and what the last call returned"""
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(k):
            out = fn()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    if args.warmup_ddim_steps:  # (hidden) warm the caches / packed weights with short clips; the timed clips are full length
        full = dict(kw)
        kw.update(num_inference_steps=args.warmup_ddim_steps, propagation_steps=[s for s in prop if s < args.warmup_ddim_steps])
    for _ in range(args.warmup):
        step_resident()
    if args.warmup_ddim_steps:
        kw.clear()
        kw.update(full)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    l0 = _lib.launch_count()
    sharding.comm_events_reset(True)
    ms_total, images = timed(step_resident, args.steps)
    comm_ms = sharding.comm_events_ms()
    sharding.comm_events_reset(False)
    launches = _lib.launch_count() - l0
    # the end-to-end leg repeats whole clips (11 s each at config 2): at most E2E_MAX_STEPS of them, so that a
    # `--steps 20 --warmup 5` run (45 clips otherwise) stays under ten minutes
    e2e_steps = min(args.steps, E2E_MAX_STEPS)
    ms_e2e = None if args.no_e2e else timed(step_e2e, e2e_steps)[0]
    clk = clocks.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"images": images})
    del images

    # roofline of the dominant kernel (tcgen05 implicit GEMM): per-launch CUDA events over one UNet forward
    roof = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        which = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PFLOP/s sustained"
        lat = torch.randn(2, 4, 8, H_LR, W_LR, device=device, dtype=torch.float16)
        lat[1] = lat[0]
        low = torch.randn(2, 3, 8, H_LR, W_LR, device=device, dtype=torch.float16)
        low[1] = low[0]
        ctx = torch.cat([neg, pos])
        ukw = dict(encoder_hidden_states=ctx, class_labels=torch.tensor([NOISE_LEVEL]), cfg_shared_input=True)
        pipe.unet(lat, 500, low, **ukw)
        with ops.Profile() as prof:
            pipe.unet(lat, 500, low, **ukw)
        summ = prof.summary()
        ig = summ.get("igemm", dict(flops=0.0, ms=1.0, launches=1))
        tot_ms = sum(d["ms"] for d in summ.values())
        achieved = ig["flops"] / ig["ms"] / 1e9
        # one representative launch of the same kernel, timed alone (CUDA events): conv3x3 512->512 on 16 x 160x288
        xr = torch.randn(16, 160, 288, 512, device=device).half()
        wr = (torch.randn(512, 3, 3, 512, device=device) * 0.02).half()
        br = torch.zeros(512, device=device)
        orr = torch.empty(16, 160, 288, 512, device=device, dtype=torch.float16)
        for _ in range(3):
            ops.conv2d(xr, wr, br, out=orr)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            ops.conv2d(xr, wr, br, out=orr)
        e1.record()
        torch.cuda.synchronize()
        rep_ms = e0.elapsed_time(e1) / 10
        rep_flops = 2.0 * 16 * 160 * 288 * 512 * 512 * 9
        burst = peaks.get("bf16_tflops", 1590.0)
        ncu = _ncu_profile_of_dominant_kernel()
        hbm = peaks.get("hbm_gbs", 6650.0)
        roof = {"bound": "tensor", "kernel": "uav::igemm_kernel (tcgen05 implicit GEMM: conv2d/conv_t/linear)",
                "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                "traffic": (ncu or {}).get("dram_bytes_per_launch"),
                "representative_launch": {"op": "conv3x3 512->512, 16 x 160x288 (3.48 TFLOP)", "ms": rep_ms,
                                          "achieved": rep_flops / rep_ms / 1e9, "peak_burst": burst,
                                          "frac_of_burst_peak": rep_flops / rep_ms / 1e9 / burst,
                                          "algorithmic_bytes": 2 * (16 * 160 * 288 * 512 * 2) + 512 * 9 * 512 * 2,
                                          "ncu": ncu},
                "peak_source": which, "launches_per_unet_forward": ig["launches"],
                "unet_forward_ms": tot_ms,
                "share_of_unet_forward_time": ig["ms"] / tot_ms,
                "per_kind_ms": {k: round(d["ms"], 3) for k, d in summ.items()},
                "hbm_bound_kinds": {k: {"GBps": round(d["bytes"] / d["ms"] / 1e6, 1), "frac_of_hbm_peak": round(d["bytes"] / d["ms"] / 1e6 / hbm, 3)}
                                    for k, d in summ.items() if d["flops"] == 0.0 and d["ms"] > 0},
                "hbm_peak_GBps": hbm}
        del lat, low, xr, wr, orr
        torch.cuda.empty_cache()

    if rank == 0:
        fps = T * args.steps / (ms_total / 1000.0)
        n_uniq = len(sharding.unique(sharding.unet_windows(T)))
        line = {"metric": "upscaled frames/sec (30 DDIM steps, 320x576->4x)", "value": fps, "unit": "frames/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
                "higher_is_better": True, "scaling": "weak" if cfg["frames"] is None else "strong", "vs_baseline": None,
                "dtype": "f16",
                "data": "synthetic (seeded LR clip, smooth flows, random prompt embeddings), random-init weights of the shipped configs",
                "config": {"workload": f"{args.config}: {T}-frame {H_LR}x{W_LR}->{4 * H_LR}x{4 * W_LR}, {ddim_steps} DDIM steps, guidance 6, "
                                       f"propagation at {prop}, {cfg['vae']} decode" + (", 256+64 px tiles" if cfg["tiled"] else ""),
                           "frames": T, "unet_windows_per_step": n_uniq, "parallelism": f"windows/chunks over {args.gpus} GPU(s)",
                           "l2": "inputs larger than L2 (activations 0.4-4.5 GB per layer)"},
                "gpu_launches": int(launches), "clocks": clk, "roofline": roof}
        if ms_e2e is not None:
            line["e2e"] = {"value": T * e2e_steps / (ms_e2e / 1000.0), "unit": "frames/s", "steps": e2e_steps,
                           "h2d_bytes_per_step": int(h_image.numel() * 4 + h_fw.numel() * 4 + h_bw.numel() * 4),
                           "d2h_bytes_per_step": int(h_out.numel() * 4)}
        if cfg["frames"] is None and args.gpus > 1:
            # the reference's 8-frame windows overlap by 2: N windows cover 6N + 2 frames, so weak scaling in FRAMES/s is
            # bounded by (6N + 2) / (8N) even with perfect window-level scaling
            line["ideal_efficiency"] = (6 * args.gpus + 2) / (8 * args.gpus)
        if world > 1:
            line["comm"] = {"collective": "NCCL all_gather_into_tensor of the windows' predictions, once per DDIM step + once after decode",
                            "ms_per_step": comm_ms / args.steps, "share_of_step": comm_ms / ms_total}
    if rank == 0 and args.gpus == 1 and args.config == "c2":
        del d_image, d_fw, d_bw
        if not args.no_reference_gpu and time.time() - t_start > REFERENCE_GPU_DEADLINE_S:
            line["reference_gpu"] = {"skipped": f"{time.time() - t_start:.0f} s into the run (the leg needs ~170 s; limit "
                                                f"{REFERENCE_GPU_DEADLINE_S} s): see profiles/r2_bench_final.json for a measured one"}
        elif not args.no_reference_gpu:
            pipe = None
            torch.cuda.empty_cache()
            try:
                line["reference_gpu"] = reference_gpu_leg(device, h_image, h_fw, h_bw, pe, ddim_steps, prop)
                line["reference_gpu"]["speedup_e2e"] = line.get("e2e", line)["value"] / line["reference_gpu"]["value"]
            except Exception as ex:  # never lose the bench line over the comparison leg
                line["reference_gpu"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
        if not args.no_cpu_baseline:
            cb = cpu_sample(cpu_plan(15.0))
            cb.pop("seconds", None)
            line["cpu_baseline"] = cb
    if rank == 0:
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
