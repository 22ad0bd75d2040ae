"""CPU tests of the host-side logic: C-ABI library loads and exports every declared symbol, header/binding
agreement, window / chunk planning, and the world_size-2 gloo path of the multi-GPU gather."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_header_symbol(uav_lib):
    from upscale_a_video_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "uav_b200.h")).read()
    declared = set(re.findall(r"\b(uav_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    for name in declared:
        assert hasattr(uav_lib, name), f"{name} declared in include/uav_b200.h but not exported"
    assert declared == set(_lib.declared_symbols()), (declared ^ set(_lib.declared_symbols()))
    assert uav_lib.uav_version().decode().startswith("uav_b200")
    if not torch.cuda.is_available():  # with a GPU, earlier tests of the session count in this process-wide counter
        assert uav_lib.uav_launch_count() == 0  # nothing may have launched on a CPU-only box


def test_no_cpu_fallback():
    """the product path must fail loudly without CUDA, never fall back"""
    from upscale_a_video_b200 import _lib, Propagation
    with pytest.raises(_lib.UavError):
        Propagation(4, learnable=False)(torch.zeros(1, 4, 2, 8, 8), torch.zeros(1, 2, 1, 8, 8), torch.zeros(1, 2, 1, 8, 8))
    src = ""
    pkg = os.path.join(ROOT, "upscale_a_video_b200")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            src += open(os.path.join(pkg, f)).read()
    assert "import oracle" not in src and "from oracle" not in src, "the product must never import the oracle"


def test_window_and_chunk_plans():
    from oracle import uav_oracle as O
    from upscale_a_video_b200 import sharding
    for T in (1, 3, 8, 9, 11, 14, 16, 26, 32, 50, 64):
        w = sharding.unet_windows(T)
        if T > 8:
            assert w == O.unet_windows(T)
            assert all(e - s == 8 for s, e in w)
        cover = set()
        for s, e in w:
            cover |= set(range(s, e))
        assert cover == set(range(T))
        ch = sharding.decode_chunks(T)
        assert sum(e - s for s, e in ch) == T and ch[0][0] == 0 and ch[-1][1] == T
    assert sharding.unique(sharding.unet_windows(14)) == [(0, 8), (6, 14)]
    assert len(sharding.unique(sharding.unet_windows(50))) == 8


WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from upscale_a_video_b200 import sharding
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
units = sharding.unique(sharding.unet_windows(26))
full = [torch.full((2, 4, 8, 3, 5), float(i + 1)) * torch.arange(5) for i in range(len(units))]
local = {i: full[i] for i in range(len(units)) if i % world == rank}
out = sharding.all_gather_units(local, len(units), (2, 4, 8, 3, 5), torch.float32, "cpu")
assert len(out) == len(units)
for a, b in zip(out, full):
    assert torch.equal(a, b)
dist.barrier()
if rank == 0:
    print("GATHER_OK")
"""


def test_all_gather_units_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29517", str(script), ROOT],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0 and "GATHER_OK" in r.stdout, r.stdout + r.stderr


def test_c_abi_error_convention(uav_lib):
    """bad arguments -> non-zero status + message, no exception / exit, nothing launched (works without a GPU)"""
    import ctypes as C
    from upscale_a_video_b200 import _lib
    n0 = uav_lib.uav_launch_count()  # process-wide: GPU tests of the same session may have launched before
    e = _lib.Epilogue()
    st = uav_lib.uav_linear(None, 4, 64, 64, None, 16, None, C.byref(e), None)
    assert st == 1 and b"null" in uav_lib.uav_last_error_string()
    st = uav_lib.uav_conv2d(None, 1, 8, 8, 64, 64, None, 64, 5, 1, 0, None, C.byref(e), None)
    assert st == 1 and b"ksize" in uav_lib.uav_last_error_string()
    st = uav_lib.uav_temporal_attention(None, None, None, None, 1, 9, 4, 8, 64, 512, 512, 512, 512, 0.125, None, None, None)
    assert st == 1
    st = uav_lib.uav_ddim_step_v0(None, None, None, 8, 7, 1.0, 0.0, 0, 1.0, 0, None)
    assert st == 1
    with pytest.raises(_lib.UavError):
        _lib.check(st, "uav_ddim_step_v0")
    assert uav_lib.uav_launch_count() == n0


def test_scheduler_host_tables_match_oracle():
    """DDIMScheduler's host-side schedule (timesteps, alphas) is plain CPU math: compare with the oracle without a GPU"""
    import json
    from oracle import uav_oracle as O
    from upscale_a_video_b200 import DDIMScheduler
    meta = json.load(open(os.path.join(ROOT, "tests", "golden", "meta.json")))
    for name, kw in meta["sched_cfgs"].items():
        a, b = DDIMScheduler(**kw), O.DDIM(**kw)
        assert torch.equal(a.alphas_cumprod, b.alphas_cumprod)
        for n in (2, 30, 50):
            a.set_timesteps(n)
            b.set_timesteps(n)
            assert a.timesteps.tolist() == b.timesteps.tolist() == a.timesteps_host
        a2 = DDIMScheduler.from_config(dict(kw, _class_name="DDIMScheduler", unknown_key=1))
        assert a2.config.prediction_type == a.config.prediction_type
    with pytest.raises(ValueError):
        DDIMScheduler().set_timesteps(2000)


def test_tile_plan_matches_reference_loop():
    """tests/golden/tiles.json was minted by executing the reference's own tile loop (oracle/make_golden_tiles.py)"""
    import json
    from upscale_a_video_b200.tiling import needs_tiling, plan_tiles
    cases = json.load(open(os.path.join(ROOT, "tests", "golden", "tiles.json")))
    assert len(cases) >= 20
    for c in cases:
        plan = plan_tiles(c["h"], c["w"], c["tile_size"])
        assert [list(t.in_box) for t in plan] == c["tiles_in"], (c["h"], c["w"], c["tile_size"])
        # replay the paste with a nearest-x4 "pipeline": must reproduce what the reference loop produced
        h, w = c["h"], c["w"]
        frame = torch.arange(h * w, dtype=torch.float32).reshape(1, 1, 1, h, w)
        out = torch.zeros(1, 1, 1, 4 * h, 4 * w)
        for t in plan:
            y0, y1, x0, x1 = t.in_box
            up = frame[..., y0:y1, x0:x1].repeat_interleave(4, -2).repeat_interleave(4, -1)
            oy0, oy1, ox0, ox1 = t.out_box
            sy0, sy1, sx0, sx1 = t.src_box
            out[..., oy0:oy1, ox0:ox1] = up[..., sy0:sy1, sx0:sx1]
        exact = torch.equal(out, frame.repeat_interleave(4, -2).repeat_interleave(4, -1))
        assert exact == c["paste_exact"], (h, w, c["tile_size"])
    assert needs_tiling(320, 576) and not needs_tiling(180, 320)


def test_ctypes_prototypes_match_header():
    """every binding in _lib.py takes exactly as many arguments as its declaration in include/uav_b200.h, with pointers /
    integers / floats in the same positions (an ABI drift here corrupts arguments silently instead of failing)"""
    import ctypes as C
    from upscale_a_video_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "uav_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", " ", hdr, flags=re.S)
    decls = dict(re.findall(r"\b(uav_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", hdr))
    assert len(decls) >= 30

    def kind(param: str) -> str:
        p = param.strip()
        if "*" in p or p.startswith("uav_stream_t"):
            return "ptr"
        base = p.rsplit(" ", 1)[0].replace("const ", "").strip()
        return {"float": "f32", "int": "i32", "int64_t": "i64", "size_t": "u64", "uint64_t": "u64",
                "uint32_t": "u32"}[base]  # LP64

    ck = {C.c_void_p: "ptr", C.c_int64: "i64", C.c_int: "i32", C.c_int32: "i32", C.c_float: "f32", C.c_size_t: "u64",
          C.c_uint64: "u64", C.c_uint32: "u32"}
    protos = dict(_lib._PROTOS)
    protos.update({k: v[1] for k, v in _lib._SPECIAL.items()})
    for name, params in decls.items():
        plist = [] if params.strip() in ("", "void") else [kind(x) for x in params.split(",")]
        got = [ck.get(t, "ptr") for t in protos[name]]  # POINTER(Epilogue) etc. count as pointers
        assert got == plist, f"{name}: header {plist} vs ctypes {got}"


TILE_WORKER = r"""
import sys, types
sys.path.insert(0, sys.argv[1])
import torch, torch.distributed as dist
from upscale_a_video_b200 import tiling
from upscale_a_video_b200.pipeline_upscale_a_video import randn_tensor
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()


class StubPipe:
    # nearest-x4 of the tile plus a signature of the noise / latents it was handed (the shared generator stream)
    def __init__(self):
        self.process_group = None
        self.vae = types.SimpleNamespace(config=types.SimpleNamespace(latent_channels=4))
        self.text_encoder = types.SimpleNamespace(dtype=torch.float32)
        self.calls = 0

    def __call__(self, image=None, flows_bi=None, noise=None, latents=None, **kw):
        assert self.process_group is None or dist.get_world_size(self.process_group) == 1  # no nested sharding
        self.calls += 1
        up = image.repeat_interleave(4, -2).repeat_interleave(4, -1).float()
        return types.SimpleNamespace(images=up + noise.mean() + 10.0 * latents.mean())


h, w, t = 300, 600, 2  # 2 x 3 tiles of 256 (+64 overlap), last column merged
image = torch.arange(3 * t * h * w, dtype=torch.float32).reshape(1, 3, t, h, w) / (3 * t * h * w)
pipe = StubPipe()
out = tiling.upscale_tiled(pipe, image, generator=torch.Generator().manual_seed(10))
plan = tiling.plan_tiles(h, w)
assert pipe.calls == len([i for i in range(len(plan)) if i % world == rank]) and pipe.process_group is None
# serial re-statement with ONE generator consumed tile by tile, as the reference loop does
g = torch.Generator().manual_seed(10)
ref = torch.zeros(1, 3, t, 4 * h, 4 * w)
for tl in plan:
    y0, y1, x0, x1 = tl.in_box
    tile = image[:, :, :, y0:y1, x0:x1]
    noise = randn_tensor(tile.shape, generator=g, device="cpu", dtype=torch.float32)
    lat = randn_tensor((1, 4, t, y1 - y0, x1 - x0), generator=g, device="cpu", dtype=torch.float32)
    res = tile.repeat_interleave(4, -2).repeat_interleave(4, -1) + noise.mean() + 10.0 * lat.mean()
    oy0, oy1, ox0, ox1 = tl.out_box
    sy0, sy1, sx0, sx1 = tl.src_box
    ref[:, :, :, oy0:oy1, ox0:ox1] = res[:, :, :, sy0:sy1, sx0:sx1]
assert torch.equal(out, ref), (out - ref).abs().max()
dist.barrier()
if rank == 0:
    print("TILES_OK", len(plan))
"""


def test_upscale_tiled_gloo_world2(tmp_path):
    """the tile driver deals tiles round-robin to ranks, keeps the reference's single generator stream, never shards
    windows inside a tile, and every rank ends with the full pasted output (one all_reduce)"""
    script = tmp_path / "tile_worker.py"
    script.write_text(TILE_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29519", str(script), ROOT],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "TILES_OK" in r.stdout, r.stdout + r.stderr


def test_raft_state_dict_keys_match_reference():
    """the RAFT parameter holders expose exactly the reference's state-dict keys and shapes (tests/golden/shapes_raft.json is
    dumped from the reference model), so `raft-things.pth` loads with strict=True"""
    import json
    from upscale_a_video_b200.raft import RAFT
    shapes = json.load(open(os.path.join(ROOT, "tests", "golden", "shapes_raft.json")))
    sd = RAFT().state_dict()
    assert {k: list(v.shape) for k, v in sd.items()} == shapes


def test_window_units_dealing():
    """whole windows unless dealing single CFG halves lowers the makespan (sharding.window_units)"""
    from upscale_a_video_b200 import sharding as S
    assert S.window_units(1, 1, True) == [(0, -1)]
    assert S.window_units(11, 1, True) == [(w, -1) for w in range(11)]
    assert S.window_units(8, 8, True) == [(w, -1) for w in range(8)]          # weak-scaling bench: one window per rank
    assert S.window_units(11, 8, False) == [(w, -1) for w in range(11)]
    u = S.window_units(11, 8, True)                                            # 64-frame clip on 8 GPUs: 22 halves, 3 rounds
    assert u == [(w, h) for w in range(11) for h in (0, 1)]
    per_rank = [sum(1 for k in range(len(u)) if k % 8 == r) for r in range(8)]
    assert max(per_rank) == 3 and max(per_rank) * S.HALF_UNIT_COST < 2
    assert S.window_units(5, 4, True) == [(w, h) for w in range(5) for h in (0, 1)]  # config 3: 10 halves on 4 ranks


def test_synthetic_weights_match_the_oracle_rule():
    """bench.py draws the product's random-init weights with upscale_a_video_b200/synthetic.py and the oracle's with
    oracle/weights.py: the two rules must give bit-identical tensors"""
    import json
    from oracle.weights import make_state_dict
    from upscale_a_video_b200.synthetic import seeded_state_dict
    for kind in ("vae_3d", "raft"):
        shapes = json.load(open(os.path.join(os.path.dirname(__file__), "golden", f"shapes_{kind}.json")))
        a, b = make_state_dict(shapes, 4321), seeded_state_dict(shapes, 4321)
        assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)


def test_pipeline_from_pretrained_local_layout(tmp_path):
    """VideoUpscalePipeline.from_pretrained(local_dir, torch_dtype) — the first call of the reference CLI
    (inference_upscale_a_video.py:101): text_encoder / low_res_scheduler / scheduler load from the shipped layout, a
    checkpoint written by an older transformers (extra `position_ids` buffer) is accepted, anything else unexpected is not"""
    import json
    from upscale_a_video_b200 import CLIPTextConfig, CLIPTextModel, DDIMScheduler, DDPMScheduler, VideoUpscalePipeline
    d = str(tmp_path)
    for sub in ("text_encoder", "low_res_scheduler", "scheduler"):
        os.makedirs(os.path.join(d, sub))
    cfg = dict(vocab_size=1000, hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4,
               max_position_embeddings=77, hidden_act="gelu", layer_norm_eps=1e-5)
    json.dump(dict(cfg, model_type="clip_text_model", architectures=["CLIPTextModel"]), open(os.path.join(d, "text_encoder", "config.json"), "w"))
    ref = CLIPTextModel(CLIPTextConfig(**cfg))
    sd = dict(ref.state_dict())
    sd["text_model.embeddings.position_ids"] = torch.arange(77)[None]
    torch.save(sd, os.path.join(d, "text_encoder", "pytorch_model.bin"))
    json.dump({"beta_schedule": "scaled_linear", "_class_name": "DDPMScheduler"}, open(os.path.join(d, "low_res_scheduler", "scheduler_config.json"), "w"))
    json.dump({"beta_schedule": "scaled_linear", "prediction_type": "v_prediction", "steps_offset": 1, "clip_sample": False,
               "set_alpha_to_one": False}, open(os.path.join(d, "scheduler", "scheduler_config.json"), "w"))
    json.dump({"max_noise_level": 300}, open(os.path.join(d, "model_index.json"), "w"))
    pipe = VideoUpscalePipeline.from_pretrained(d, torch_dtype=torch.float16)
    assert isinstance(pipe.text_encoder, CLIPTextModel) and pipe.text_encoder.dtype == torch.float16
    assert all(torch.equal(v.half(), pipe.text_encoder.state_dict()[k]) for k, v in ref.state_dict().items())
    assert isinstance(pipe.low_res_scheduler, DDPMScheduler) and isinstance(pipe.scheduler, DDIMScheduler)
    assert pipe.scheduler.config.prediction_type == "v_prediction" and pipe.config.max_noise_level == 300
    assert pipe.vae is None and pipe.unet is None and pipe.tokenizer is None
    sd["text_model.bogus.weight"] = torch.zeros(1)
    torch.save(sd, os.path.join(d, "text_encoder", "pytorch_model.bin"))
    with pytest.raises(RuntimeError):
        VideoUpscalePipeline.from_pretrained(d)
    with pytest.raises(EnvironmentError):
        VideoUpscalePipeline.from_pretrained(os.path.join(d, "nope"))
