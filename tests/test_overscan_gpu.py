"""GPU: overscan -- any image size rendered on the decoder's size grid and cropped.  Covers the canvas ray-token
kernel, the cropped final DPT conv on both conv kernels (per-tap and halo tile), bit identity with the plain canvas
render where the camera's floats do not move (1080p, 720p, 4K), the fp32 oracle where they do, on-grid no-ops, CUDA
graph keys, render_stream and the sharded render.  Tolerances are the north_star's (metrics.py)."""
import math
import os
import socket
import subprocess
import sys

import pytest
import torch

from renderformer_b200 import lib as L
from renderformer_b200 import ops
from renderformer_b200.config import RenderFormerConfig, overscan_grid
from renderformer_b200.metrics import PSNR_MIN, REL_TOL, hdr_rel_err, log_psnr
from renderformer_b200.synth import init_state_dict, make_scene

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from overscan_oracle import camera_rays_overscan, render_overscan  # noqa: E402

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


def _args(sc):
    g = {k: v.to(DEV) for k, v in sc.items()}
    return g["triangles"], g["texture"], g["mask"], g["vn"], g["c2w"], g["fov"]


def _check(img, ref, what):
    rel, psnr = hdr_rel_err(img, ref), log_psnr(img, ref)
    print(f"{what}: hdr rel {rel:.3e} log-PSNR {psnr:.1f} dB")
    assert rel <= REL_TOL and psnr >= PSNR_MIN, what


# ------------------------------------------------------------------------------------------------ canvas ray tokens
@pytest.mark.parametrize("H,W,Hc,Wc,top,left", [
    (50, 150, 64, 192, 7, 21),       # odd offsets: the principal point falls on a half pixel
    (99, 150, 128, 192, 14, 21),
    (150, 99, 192, 128, 21, 14),
    (99, 150, 104, 152, 2, 1),
    (1080, 1920, 1088, 1920, 4, 0),
])
def test_canvas_ray_tokens_match_overscan_camera(H, W, Hc, Wc, top, left):
    sc = make_scene(8, 3, seed=4)
    fov_deg = sc["fov"][0, :, 0]
    V = fov_deg.shape[0]
    n_tok = (Hc // 8) * (Wc // 8)
    tok = ops.ray_tokens_canvas(fov_deg.to(DEV), torch.empty(V * n_tok, 192, dtype=torch.float16, device=DEV),
                                n_views=V, canvas_h=Hc, canvas_w=Wc, height=H, width=W, top=top, left=left)
    rays = camera_rays_overscan(fov_deg[:, None] / 180.0 * math.pi, H, W, Hc, Wc, top, left).contiguous()
    want = ops.ray_map_tokens(rays.to(DEV), torch.empty(V * n_tok, 192, dtype=torch.float16, device=DEV), n_views=V,
                              height=Hc, width=Wc)
    a, b = tok.cpu().float(), want.cpu().float()
    ulp = torch.maximum(a.abs(), b.abs()).clamp_min(2.0 ** -14) * 2.0 ** -10   # one fp16 ulp at the larger value
    assert ((a - b).abs() <= ulp).all()


@pytest.mark.parametrize("H,W", [(64, 192), (8, 24), (1088, 1920)])
def test_canvas_ray_tokens_without_border_are_ray_tokens_hw(H, W):
    fov = torch.tensor([37.5, 52.0, 80.0], device=DEV)
    n = 3 * (H // 8) * (W // 8)
    hw = ops.ray_tokens(fov, torch.empty(n, 192, dtype=torch.float16, device=DEV), n_views=3, height=H, width=W)
    cv = ops.ray_tokens_canvas(fov, torch.empty(n, 192, dtype=torch.float16, device=DEV), n_views=3, canvas_h=H,
                               canvas_w=W, height=H, width=W, top=0, left=0)
    assert torch.equal(hw, cv)


def test_canvas_ray_tokens_reject_bad_arguments():
    lib = L.load()
    x = torch.empty(64 * 64 * 3, device=DEV)
    p = x.data_ptr()
    for bad in ((60, 64, 50, 50, 0, 0),     # canvas side not a multiple of 8
                (64, 64, 60, 60, 5, 0),     # window leaves the canvas at the bottom
                (64, 64, 60, 60, 0, 5),     # ... and on the right
                (64, 64, 0, 60, 0, 0),      # empty window
                (64, 64, 60, -4, 0, 0),
                (64, 64, 60, 60, -1, 0),    # negative offset
                (0, 64, 8, 8, 0, 0)):
        assert lib.rfb_ray_tokens_canvas(p, p, 1, *bad, None) == -1, bad
    assert lib.rfb_ray_tokens_canvas(p, p, 0, 64, 64, 60, 60, 0, 0, None) == -1


# ------------------------------------------------------------------------------------------------ cropped final conv
def _final_conv_operands(B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    A = (torch.randn(B * H * W, 64, generator=g) * 0.5).half().to(DEV)
    Wt = (torch.randn(32, 9 * 64, generator=g) * 0.05).half().to(DEV)
    bias = (torch.randn(32, generator=g) * 0.1).to(DEV)
    w2 = (torch.randn(3, 32, generator=g) * 0.1).to(DEV).contiguous()
    b2 = (torch.randn(3, generator=g) * 0.1).to(DEV)
    return A, Wt, bias, w2, b2


@pytest.mark.parametrize("epi", [L.EPI_FINAL, L.EPI_FINAL_RAW], ids=["final", "final_raw"])
@pytest.mark.parametrize("B,H,W,windows", [
    # 12 super-tiles: the per-tap conv kernel (16-wide x 8-tall tiles)
    (1, 40, 56, [(37, 45, 3, 5), (40, 56, 0, 0), (1, 1, 39, 55), (24, 17, 8, 16)]),
    # 2 x 9 x 10 = 180 16 x 16 super-tiles (>= 96): the halo-tile conv kernel
    (2, 136, 152, [(123, 139, 7, 9), (136, 152, 0, 0), (99, 150, 20, 1), (9, 7, 127, 145)]),
])
def test_cropped_final_conv_is_the_slice(epi, B, H, W, windows):
    A, Wt, bias, w2, b2 = _final_conv_operands(B, H, W, 11)
    full = torch.empty(B, H, W, 3, device=DEV)
    ops.gemm(A, Wt, conv=(B, H, W, 64), epi=epi, bias=bias, w2=w2, b2=b2, out=full, ldo=3)
    for (h, w, top, left) in windows:
        crop = torch.full((B, h, w, 3), float("nan"), device=DEV)
        ops.gemm(A, Wt, conv=(B, H, W, 64), epi=epi, bias=bias, w2=w2, b2=b2, out=crop, ldo=3, crop=(h, w, top, left))
        assert torch.equal(crop, full[:, top:top + h, left:left + w]), (h, w, top, left)


def test_crop_is_rejected_outside_the_final_conv():
    B, H, W = 1, 40, 56
    A, Wt, bias, w2, b2 = _final_conv_operands(B, H, W, 12)
    out = torch.empty(B * H * W, 3, device=DEV)
    with pytest.raises(L.RfbError):   # linear A operand
        ops.gemm(A, Wt[:, :64].contiguous(), epi=L.EPI_FINAL, bias=bias, w2=w2, b2=b2, out=out, ldo=3, crop=(8, 8, 0, 0))
    with pytest.raises(L.RfbError):   # conv, but not a final epilogue
        ops.gemm(A, Wt, conv=(B, H, W, 64), out=torch.empty(B * H * W, 32, dtype=torch.float16, device=DEV),
                 crop=(8, 8, 0, 0))
    for window in ((41, 8, 0, 0), (8, 8, 0, 49), (8, 8, -1, 0), (0, 8, 0, 0)):   # window not inside the image
        with pytest.raises(L.RfbError):
            ops.gemm(A, Wt, conv=(B, H, W, 64), epi=L.EPI_FINAL, bias=bias, w2=w2, b2=b2, out=out, ldo=3, crop=window)


# ------------------------------------------------------------------------------------------------ pipeline, Large
@pytest.mark.parametrize("H,W,Hc,top", [(1080, 1920, 1088, 4), (720, 1280, 768, 24), (2160, 3840, 2176, 8)],
                         ids=["1080p", "720p", "4k"])
def test_large_overscan_is_the_canvas_render_cropped(H, W, Hc, top):
    """The longer side is on the grid: f and the principal point are the same floats as for the Hc x W image, so the
    overscan render is bit-identical to the plain canvas render, sliced.  The 4K case runs the halo conv kernel on a
    2176 x 3840 output level."""
    pipe, _, _ = _pipe("v1_1_swin_large", 5)
    args = _args(make_scene(512, 1, seed=50))
    img = pipe(*args, resolution=(H, W), torch_dtype=torch.bfloat16, overscan=True)
    assert img.shape == (1, 1, H, W, 3)
    canvas = pipe(*args, resolution=(Hc, W), torch_dtype=torch.bfloat16)
    assert torch.equal(img, canvas[:, :, top:top + H])


@pytest.mark.parametrize("name,n_tris,res", [("tiny_swin", 90, (99, 150)), ("tiny_full", 90, (99, 150)),
                                             ("v1_1_swin_large", 512, (720, 720))])
def test_overscan_against_oracle(name, n_tris, res):
    """Where the camera moves on the canvas (odd offsets, or the longer side off the grid) against the fp32 oracle
    rendered the same way."""
    pipe, sd, cfg = _pipe(name, 5)
    V = 1 if name == "v1_1_swin_large" else 2
    sc = make_scene(n_tris, V, seed=51)
    hw, canvas, offsets = overscan_grid(cfg, res)
    ref = render_overscan(sd, cfg, sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], sc["fov"], hw,
                          canvas, offsets)
    for dtype in (torch.bfloat16, torch.float16):
        img = pipe(*_args(sc), resolution=res, torch_dtype=dtype, overscan=True).cpu()
        assert img.shape == (1, V, *hw, 3)
        _check(img, ref, f"{name} {hw} on {canvas} {dtype}")


@pytest.mark.parametrize("name,res", [("v1_1_swin_large", 512), ("v1_1_swin_large", (576, 1024)),
                                      ("tiny_full", (64, 136))])
def test_overscan_on_grid_is_a_no_op(name, res):
    pipe, _, _ = _pipe(name, 5)
    args = _args(make_scene(300, 1, seed=52))
    a = pipe(*args, resolution=res, torch_dtype=torch.bfloat16, overscan=True)
    b = pipe(*args, resolution=res, torch_dtype=torch.bfloat16)
    assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ graphs / stream
def test_overscan_graphs_are_separate_entries():
    pipe, _, _ = _pipe("tiny_swin", 8)
    args = _args(make_scene(90, 2, seed=53))
    over = pipe(*args, resolution=(99, 150), overscan=True)
    plain = pipe(*args, resolution=(128, 192))
    pipe.cuda_graphs = True
    n0 = len(pipe._graphs)
    for _ in range(2):
        assert torch.equal(pipe(*args, resolution=(99, 150), overscan=True), over)
        assert torch.equal(pipe(*args, resolution=(128, 192)), plain)
    assert len(pipe._graphs) == n0 + 2, "the overscan render and its plain canvas must be separate graphs"


def test_overscan_render_stream_ldr_padded():
    pipe, _, _ = _pipe("tiny_swin", 8)
    res = (99, 150)
    counts, pad = (61, 100), 128
    pipe.cuda_graphs = True
    want = []
    for i, n in enumerate(counts):   # the same zero padding the stream applies on the device
        img = pipe(*_args(make_scene(n, 2, seed=60 + i, pad_to=pad)), resolution=res, overscan=True)
        want.append(pipe.hdr_to_ldr(img, "none").cpu())
    host = [{k: t.pin_memory() for k, t in make_scene(n, 2, seed=60 + i).items()} for i, n in enumerate(counts)]
    got = [img.clone() for img in pipe.render_stream(iter(host), resolution=res, ldr="none", pad_to=pad, overscan=True)]
    assert len(got) == 2
    for a, b in zip(got, want):
        assert a.shape == (1, 2, *res, 3) and a.dtype == torch.uint8
        assert torch.equal(a, b)


def test_overscan_empty_view_slice_shape():
    pipe, _, _ = _pipe("tiny_swin", 8)
    sc = {k: v.to(DEV) for k, v in make_scene(20, 1, seed=2).items()}
    st = pipe.encode(sc["triangles"], sc["texture"], sc["mask"], sc["vn"])
    out = pipe.render_views(st, sc["c2w"][:, :0], sc["fov"][:, :0], (99, 150), overscan=True)
    assert out.shape == (1, 0, 99, 150, 3)


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
single = pipe(*args, resolution=(99, 150), overscan=True).clone()
ok = single.shape == (1, 4, 99, 150, 3)
for graphs in (False, True):
    pipe.cuda_graphs = graphs
    for rep in range(2):
        out = render_sharded(pipe, *args, resolution=(99, 150), dst=0, overscan=True)
        if rank == 0 and not (out.shape == single.shape and torch.equal(out, single)):
            ok = False
dist.barrier()
if rank == 0:
    print("OVERSCAN_SHARDED_OK" if ok else "OVERSCAN_SHARDED_MISMATCH", flush=True)
pipe._graphs.clear()
torch.cuda.synchronize()
dist.barrier()
sys.stdout.flush()
os._exit(0)
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_render_sharded_overscan_equals_single_gpu(tmp_path):
    worker = tmp_path / "overscan_worker.py"
    worker.write_text(WORKER % {"root": ROOT})
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), str(worker)], capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "OVERSCAN_SHARDED_OK" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])
