"""GPU: non-square (height, width) images through every layer -- the ray kernels, the model-level entry with an
H != W ray map, the pipeline (V1.1-swin-Large against the fp32 oracle, including a pyramid level with partial conv
tiles and a half-empty last swin tile), CUDA-graph keys, render_stream and the sharded render.  Tolerances are the
north_star's (metrics.py: 2e-2 max relative error on HDR pixels, 45 dB log-PSNR)."""
import math
import os
import socket
import subprocess
import sys

import pytest
import torch

from oracle import renderformer_oracle as orc
from renderformer_b200 import lib as L
from renderformer_b200 import ops
from renderformer_b200.config import RenderFormerConfig
from renderformer_b200.metrics import PSNR_MIN, REL_TOL, hdr_rel_err, log_psnr
from renderformer_b200.synth import init_state_dict, make_scene

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from nonsquare_oracle import camera_rays_hw, render_hw  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_PIPES = {}


def _pipe(name, seed):
    """One resident pipeline per (config, weight seed); the Large model is built once for all its cases."""
    from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
    key = (name, seed)
    if key not in _PIPES:
        _PIPES.clear()
        cfg = RenderFormerConfig.named(name)
        sd = init_state_dict(cfg, seed)
        model = RenderFormer(cfg)
        model.load_state_dict(sd)
        pipe = RenderFormerRenderingPipeline(model)
        pipe.to(torch.device(DEV))
        _PIPES[key] = (pipe, sd, cfg)
    pipe, sd, cfg = _PIPES[key]
    pipe.cuda_graphs = False
    pipe._graphs.clear()
    return pipe, sd, cfg


def _check(img, ref, what):
    rel, psnr = hdr_rel_err(img, ref), log_psnr(img, ref)
    print(f"{what}: hdr rel {rel:.3e} log-PSNR {psnr:.1f} dB")
    assert rel <= REL_TOL and psnr >= PSNR_MIN, what


# ------------------------------------------------------------------------------------------------ ray kernels
@pytest.mark.parametrize("H,W", [(64, 192), (192, 64), (8, 24)])
def test_ray_kernels_hw(H, W):
    sc = make_scene(8, 3, seed=4)
    c2w, fov_deg = sc["c2w"][0], sc["fov"][0, :, 0]                      # [3,4,4], [3] degrees
    fov_rad = fov_deg / 180.0 * math.pi
    V = c2w.shape[0]
    # ray map: the oracle's camera (fov across the longer side), rotated into world space
    rays = ops.ray_map(c2w.to(DEV), fov_rad.to(DEV), torch.empty(V, H, W, 3, device=DEV), n_views=V, height=H, width=W)
    want = torch.einsum("vij,vhwj->vhwi", c2w[:, :3, :3], camera_rays_hw(fov_rad[:, None], H, W))
    assert (rays.cpu() - want).abs().max().item() < 2e-6
    # the square entry point is the H = W case of the same kernel
    sq = ops.ray_map(c2w.to(DEV), fov_rad.to(DEV), torch.empty(V, H, H, 3, device=DEV), n_views=V, resolution=H)
    sq_hw = ops.ray_map(c2w.to(DEV), fov_rad.to(DEV), torch.empty(V, H, H, 3, device=DEV), n_views=V, height=H, width=H)
    assert torch.equal(sq, sq_hw)
    # fused camera-space tokens (fov in degrees) vs identity-c2w ray map (radians) -> explicit-map tokens
    n_tok = (H // 8) * (W // 8)
    tok = ops.ray_tokens(fov_deg.to(DEV), torch.empty(V * n_tok, 192, dtype=torch.float16, device=DEV), n_views=V,
                         height=H, width=W)
    eye = torch.eye(4).expand(V, 4, 4).contiguous()
    cam = ops.ray_map(eye.to(DEV), fov_rad.to(DEV), torch.empty(V, H, W, 3, device=DEV), n_views=V, height=H, width=W)
    tok2 = ops.ray_map_tokens(cam, torch.empty(V * n_tok, 192, dtype=torch.float16, device=DEV), n_views=V,
                              height=H, width=W)
    a, b = tok.cpu().float(), tok2.cpu().float()
    ulp = torch.maximum(a.abs(), b.abs()).clamp_min(2.0 ** -14) * 2.0 ** -10   # one fp16 ulp at the larger value
    assert ((a - b).abs() <= ulp).all()
    # token order: row-major patch grid, feature = c*64 + p1*8 + p2 ('b (h1 p1) (w1 p2) c', view_transformer.py:105)
    grid = cam.cpu().view(V, H // 8, 8, W // 8, 8, 3).permute(0, 1, 3, 5, 2, 4).reshape(V * n_tok, 192)
    assert torch.equal(tok2.cpu(), grid.half())


def test_ray_kernels_reject_bad_sizes():
    lib = L.load()
    x = torch.empty(64 * 64 * 3, device=DEV)
    assert lib.rfb_ray_tokens_hw(x.data_ptr(), x.data_ptr(), 1, 64, 60, None) == -1
    assert lib.rfb_ray_map_tokens_hw(x.data_ptr(), x.data_ptr(), 1, 0, 64, None) == -1
    assert lib.rfb_ray_map_hw(x.data_ptr(), x.data_ptr(), x.data_ptr(), 1, 64, -8, None) == -1


# ------------------------------------------------------------------------------------------------ square via a tuple
@pytest.mark.parametrize("name,n_tris,R", [("tiny_swin", 90, 128), ("v1_1_swin_large", 512, 512)])
def test_square_tuple_is_square_int(name, n_tris, R):
    pipe, _, _ = _pipe(name, 5)
    sc = {k: v.cuda() for k, v in make_scene(n_tris, 2, seed=30).items()}
    args = (sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"])
    a = pipe(*args, resolution=R, torch_dtype=torch.bfloat16)
    b = pipe(*args, resolution=(R, R), torch_dtype=torch.bfloat16)
    assert a.shape == (1, 2, R, R, 3) and torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ model level
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("name,H,W", [("tiny_swin", 128, 192), ("tiny_swin", 192, 128), ("tiny_full", 64, 136)])
def test_model_forward_non_square_ray_map(name, H, W, dtype):
    """RenderFormer.forward with the reference's arguments and an H != W ray map rays_d [1,2,H,W,3]."""
    pipe, sd, cfg = _pipe(name, 21)
    B, V, N = 1, 2, 64
    sc = make_scene(60, V, seed=6, pad_to=N)
    tex_log = sc["texture"].clone()
    tex_log[:, :, -3:] = torch.log10(tex_log[:, :, -3:] + 1.0)
    tri_cam = orc.to_camera_space(sc["c2w"][0], sc["triangles"].expand(V, -1, -1, -1)).reshape(1, V, N, 9)
    rays = camera_rays_hw(sc["fov"][0] / 180.0 * math.pi, H, W)[None]     # [1,V,H,W,3]
    with torch.autocast("cuda", dtype=dtype):
        out = pipe.model(sc["triangles"].reshape(B, N, 9).cuda(), tex_log.cuda(), sc["mask"].cuda(),
                         sc["vn"].reshape(B, N, 9).cuda(), rays_o=torch.zeros(B, V, 3).cuda(), rays_d=rays.cuda(),
                         tri_vpos_view_tf=tri_cam.cuda())
    assert out.shape == (B, V, 3, H, W)
    hdr = (torch.pow(10.0, out) - 1.0).permute(0, 1, 3, 4, 2).cpu()
    ref = render_hw(sd, cfg, sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], (H, W))
    _check(hdr, ref, f"forward {name} {H}x{W} {dtype}")
    # the keyword form (cameras + (H, W)) renders the same rays on the device
    with torch.autocast("cuda", dtype=dtype):
        kw = pipe.model(sc["triangles"].reshape(B, N, 9).cuda(), tex_log.cuda(), sc["mask"].cuda(),
                        sc["vn"].reshape(B, N, 9).cuda(), c2w=sc["c2w"].cuda(), fov=sc["fov"].cuda(), resolution=(H, W))
    assert kw.shape == out.shape
    assert hdr_rel_err((torch.pow(10.0, kw) - 1.0).permute(0, 1, 3, 4, 2).cpu(), hdr) < 3e-3


# ------------------------------------------------------------------------------------------------ pipeline, Large
@pytest.mark.parametrize("H,W,V", [
    (576, 1024, 1),   # 72 x 128 patches: the 36-row pyramid level has partial conv tiles
    (192, 320, 1),    # 3 x 5 = 15 windows: the last 128-row swin tile is half empty
])
def test_large_pipeline_non_square(H, W, V):
    pipe, sd, cfg = _pipe("v1_1_swin_large", 5)
    sc = make_scene(512, V, seed=31)
    g = {k: v.cuda() for k, v in sc.items()}
    ref = render_hw(sd, cfg, sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], (H, W))
    for dtype in (torch.bfloat16, torch.float16):
        img = pipe(g["triangles"], g["texture"], g["mask"], g["vn"], g["c2w"], g["fov"], resolution=(H, W),
                   torch_dtype=dtype).cpu()
        assert img.shape == (1, V, H, W, 3)
        _check(img, ref, f"Large {H}x{W} {dtype}")


def test_large_pipeline_orientation_not_swapped():
    """256x512 and 512x256 (2 views) are different images and different CUDA graphs; each matches its own oracle
    image, in bf16 and fp16, eager and replayed."""
    pipe, sd, cfg = _pipe("v1_1_swin_large", 5)
    sc = make_scene(512, 2, seed=32)
    g = {k: v.cuda() for k, v in sc.items()}
    args = (g["triangles"], g["texture"], g["mask"], g["vn"], g["c2w"], g["fov"])
    refs = {hw: render_hw(sd, cfg, sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], hw)
            for hw in ((256, 512), (512, 256))}
    for dtype in (torch.bfloat16, torch.float16):
        eager = {}
        for hw, ref in refs.items():
            eager[hw] = pipe(*args, resolution=hw, torch_dtype=dtype).cpu()
            assert eager[hw].shape == (1, 2, *hw, 3)
            _check(eager[hw], ref, f"Large {hw[0]}x{hw[1]} {dtype}")
        assert hdr_rel_err(eager[(256, 512)], refs[(256, 512)]) < hdr_rel_err(eager[(256, 512)], refs[(512, 256)].transpose(2, 3))
        pipe.cuda_graphs = True
        n0 = len(pipe._graphs)
        for _ in range(2):
            for hw in refs:
                assert torch.equal(pipe(*args, resolution=hw, torch_dtype=dtype).cpu(), eager[hw])
        assert len(pipe._graphs) == n0 + 2, "(H, W) and (W, H) must be separate graphs"
        pipe.cuda_graphs = False
        pipe._graphs.clear()


# ------------------------------------------------------------------------------------------------ stream / sharded
def test_render_stream_hw_padded_ldr_reuses_one_graph():
    pipe, _, _ = _pipe("tiny_swin", 8)
    H, W = 128, 192
    counts = (61, 100)
    scenes = [make_scene(n, 2, seed=40 + i) for i, n in enumerate(counts)]
    want = []
    for sc in scenes:
        g = {k: t.cuda() for k, t in sc.items()}
        img = pipe(g["triangles"], g["texture"], g["mask"], g["vn"], g["c2w"], g["fov"], resolution=(H, W))
        want.append(pipe.hdr_to_ldr(img, "none").cpu())
    pipe.cuda_graphs = True
    host = [{k: t.pin_memory() for k, t in sc.items()} for sc in scenes]
    got = [img.clone() for img in pipe.render_stream(iter(host), resolution=(H, W), ldr="none", pad_to=128)]
    assert len(pipe._graphs) == 1, "every padded scene must replay the same graph"
    for a, b in zip(got, want):
        assert a.shape == (1, 2, H, W, 3) and a.dtype == torch.uint8
        assert (a.float() - b.float()).abs().mean().item() < 0.5  # padding moves HDR values by < 2e-3 (one graph)


def test_empty_view_slice_shape():
    pipe, _, _ = _pipe("tiny_swin", 8)
    sc = {k: v.cuda() for k, v in make_scene(20, 1, seed=2).items()}
    st = pipe.encode(sc["triangles"], sc["texture"], sc["mask"], sc["vn"])
    out = pipe.render_views(st, sc["c2w"][:, :0], sc["fov"][:, :0], (128, 192))
    assert out.shape == (1, 0, 128, 192, 3)


WORKER = r"""
import os, sys, torch
sys.path.insert(0, %(root)r)
import torch.distributed as dist
from renderformer_b200.config import RenderFormerConfig
from renderformer_b200.dist import render_sharded
from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
from renderformer_b200.synth import init_state_dict, make_scene
rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
cfg = RenderFormerConfig.named("tiny_swin")
model = RenderFormer(cfg)
model.load_state_dict(init_state_dict(cfg, 7))
pipe = RenderFormerRenderingPipeline(model)
pipe.to(dev)
pipe.view_chunk = 1  # same decoder passes in both schedules (the DPT picks its conv kernel per pass)
sc = {k: v.to(dev) for k, v in make_scene(300, 4, seed=3).items()}
args = (sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"])
single = pipe(*args, resolution=(256, 512)).clone()
ok = True
for graphs in (False, True):
    pipe.cuda_graphs = graphs
    for rep in range(2):
        out = render_sharded(pipe, *args, resolution=(256, 512), dst=0)
        if rank == 0 and not (out.shape == single.shape and torch.equal(out, single)):
            ok = False
dist.barrier()
if rank == 0:
    print("HW_SHARDED_OK" if ok else "HW_SHARDED_MISMATCH", flush=True)
pipe._graphs.clear()
torch.cuda.synchronize()
dist.barrier()
sys.stdout.flush()
os._exit(0)
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_render_sharded_hw_equals_single_gpu(tmp_path):
    worker = tmp_path / "hw_worker.py"
    worker.write_text(WORKER % {"root": ROOT})
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), str(worker)], capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "HW_SHARDED_OK" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])
