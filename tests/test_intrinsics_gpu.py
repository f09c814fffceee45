"""GPU: per-view pinhole intrinsics (fx, fy, cx, cy) through every layer -- the intrinsics ray-token kernel on the
plain image and on an overscan canvas, the fov -> intrinsics kernel for the three sensor fits, bit identity of
`render(intrinsics=intrinsics_from_fov(fov))` with `render(fov=fov)`, the fp32 oracle with calibrated cameras, CUDA
graph keys and replays, render_stream, render_to_files and the sharded render.  Tolerances are the north_star's
(metrics.py)."""
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
from intrinsics_oracle import camera_rays_k, intrinsics_from_fov_f64, render_k  # noqa: E402

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
    return g["triangles"], g["texture"], g["mask"], g["vn"], g["c2w"]


def _check(img, ref, what):
    rel, psnr = hdr_rel_err(img, ref), log_psnr(img, ref)
    print(f"{what}: hdr rel {rel:.3e} log-PSNR {psnr:.1f} dB")
    assert rel <= REL_TOL and psnr >= PSNR_MIN, what


def _calibrated(fov_deg, H, W, sx=1.0, sy=1.0, dx=0.0, dy=0.0):
    """A calibrated-looking K [..., 4] fp32: the fov camera with its focal lengths scaled by (sx, sy) and its principal
    point moved by (dx, dy) pixels."""
    K = intrinsics_from_fov_f64(fov_deg, H, W)
    return (K * torch.tensor([sx, sy, 1.0, 1.0], dtype=torch.float64)
            + torch.tensor([0.0, 0.0, dx, dy], dtype=torch.float64)).float()


# ------------------------------------------------------------------------------------------------ ray tokens
CASES = {
    "fx_ne_fy": dict(sx=1.0, sy=1.3),
    "off_centre": dict(sx=0.9, sy=0.9, dx=17.25, dy=-9.5),
    "pp_outside": dict(sx=1.1, sy=0.8, dx=-400.0, dy=250.0),
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("H,W,Hc,Wc,top,left", [
    (64, 192, 64, 192, 0, 0),        # landscape, canvas = image
    (192, 64, 192, 64, 0, 0),        # portrait
    (99, 150, 128, 192, 14, 21),     # landscape on an overscan canvas
    (150, 99, 192, 128, 21, 14),     # portrait on an overscan canvas
    (1080, 1920, 1088, 1920, 4, 0),
])
def test_intrinsics_ray_tokens_match_camera_rays_k(case, H, W, Hc, Wc, top, left):
    fov_deg = torch.tensor([37.5, 52.0, 80.0])
    K = _calibrated(fov_deg, H, W, **CASES[case])
    V = K.shape[0]
    n_tok = (Hc // 8) * (Wc // 8)
    tok = ops.ray_tokens_intrinsics(K.to(DEV), torch.empty(V * n_tok, 192, dtype=torch.float16, device=DEV), n_views=V,
                                    canvas_h=Hc, canvas_w=Wc, height=H, width=W, top=top, left=left)
    rays = camera_rays_k(K, H, W, Hc, Wc, top, left).contiguous()
    want = ops.ray_map_tokens(rays.to(DEV), torch.empty(V * n_tok, 192, dtype=torch.float16, device=DEV), n_views=V,
                              height=Hc, width=Wc)
    a, b = tok.cpu().float(), want.cpu().float()
    ulp = torch.maximum(a.abs(), b.abs()).clamp_min(2.0 ** -14) * 2.0 ** -10   # one fp16 ulp at the larger value
    assert ((a - b).abs() <= ulp).all()


@pytest.mark.parametrize("H,W,Hc,Wc,top,left", [(64, 192, 64, 192, 0, 0), (99, 150, 128, 192, 14, 21),
                                                 (150, 99, 152, 104, 1, 2), (1080, 1920, 1088, 1920, 4, 0)])
def test_auto_fit_intrinsics_tokens_are_the_fov_tokens(H, W, Hc, Wc, top, left):
    fov = torch.tensor([20.0, 37.5, 52.0, 80.0, 120.0], device=DEV)
    V = fov.shape[0]
    K = ops.intrinsics_from_fov(fov, torch.empty(V, 4, device=DEV), n_views=V, height=H, width=W)
    n = V * (Hc // 8) * (Wc // 8)
    a = ops.ray_tokens_intrinsics(K, torch.empty(n, 192, dtype=torch.float16, device=DEV), n_views=V, canvas_h=Hc,
                                  canvas_w=Wc, height=H, width=W, top=top, left=left)
    b = ops.ray_tokens_canvas(fov, torch.empty(n, 192, dtype=torch.float16, device=DEV), n_views=V, canvas_h=Hc,
                              canvas_w=Wc, height=H, width=W, top=top, left=left)
    assert torch.equal(a, b)


@pytest.mark.parametrize("fit", ["auto", "horizontal", "vertical"])
@pytest.mark.parametrize("H,W", [(256, 512), (512, 256), (1080, 1920), (99, 150)])
def test_intrinsics_from_fov_fits(fit, H, W):
    fov = torch.tensor([10.0, 37.5, 52.0, 90.0, 150.0])
    K = ops.intrinsics_from_fov(fov.to(DEV), torch.empty(5, 4, device=DEV), n_views=5, height=H, width=W, fit=fit)
    want = intrinsics_from_fov_f64(fov, H, W, fit)
    assert torch.allclose(K.cpu().double(), want, rtol=1e-6, atol=0)
    assert torch.equal(K[:, 2:].cpu(), torch.tensor([[W / 2, H / 2]] * 5))


def test_intrinsics_kernels_reject_bad_arguments():
    lib = L.load()
    x = torch.empty(64 * 64 * 3, device=DEV)
    p = x.data_ptr()
    for bad in ((60, 64, 50, 50, 0, 0), (64, 64, 60, 60, 5, 0), (64, 64, 60, 60, 0, 5), (64, 64, 0, 60, 0, 0),
                (64, 64, 60, -4, 0, 0), (64, 64, 60, 60, -1, 0), (0, 64, 8, 8, 0, 0)):
        assert lib.rfb_ray_tokens_intrinsics(p, p, 1, *bad, None) == -1, bad
    assert lib.rfb_ray_tokens_intrinsics(p, p, 0, 64, 64, 60, 60, 0, 0, None) == -1
    assert lib.rfb_ray_tokens_intrinsics(None, p, 1, 64, 64, 64, 64, 0, 0, None) == -1
    for bad in ((1, 64, 64, 3), (1, 64, 64, -1), (0, 64, 64, 0), (1, 0, 64, 0), (1, 64, 0, 0)):
        assert lib.rfb_intrinsics_from_fov(p, p, *bad, None) == -1, bad
    with pytest.raises(ValueError):
        ops.intrinsics_from_fov(x[:1], x[:4], n_views=1, height=64, width=64, fit="diagonal")


# ------------------------------------------------------------------------------------------------ bit identity
@pytest.mark.parametrize("graphs", [False, True], ids=["eager", "graphs"])
@pytest.mark.parametrize("res,overscan", [(512, False), ((256, 512), False), ((1080, 1920), True)],
                         ids=["512", "256x512", "1080p"])
def test_auto_intrinsics_render_is_the_fov_render(res, overscan, graphs):
    pipe, _, _ = _pipe("v1_1_swin_large", 5)
    sc = make_scene(512, 2, seed=70)
    sc["fov"][0, 1, 0] = 61.0
    args = _args(sc)
    fov = sc["fov"].to(DEV)
    pipe.cuda_graphs = graphs
    K = pipe.intrinsics_from_fov(fov, res)
    assert K.shape == (1, 2, 4) and K.is_cuda
    for _ in range(2 if graphs else 1):   # the second call of a graphed render is a replay
        a = pipe(*args, fov, resolution=res, torch_dtype=torch.bfloat16, overscan=overscan)
        b = pipe(*args, resolution=res, torch_dtype=torch.bfloat16, overscan=overscan, intrinsics=K)
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ oracle
@pytest.mark.parametrize("name,n_tris,res,overscan", [("v1_1_swin_large", 512, (256, 512), False),
                                                      ("tiny_swin", 90, (99, 150), True),
                                                      ("tiny_full", 90, (99, 150), True)])
def test_intrinsics_against_oracle(name, n_tris, res, overscan):
    pipe, sd, cfg = _pipe(name, 5)
    V = 1 if name == "v1_1_swin_large" else 2
    sc = make_scene(n_tris, V, seed=71)
    H, W = res
    K = torch.stack([_calibrated(sc["fov"][0, :, 0], H, W, sx=1.0, sy=1.25, dx=23.5, dy=-11.0)])   # [1, V, 4]
    if overscan:
        hw, canvas, offsets = overscan_grid(cfg, res)
    else:
        hw, canvas, offsets = res, res, (0, 0)
    ref = render_k(sd, cfg, sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], K, hw, canvas, offsets)
    for dtype in (torch.bfloat16, torch.float16):
        img = pipe(*_args(sc), resolution=res, torch_dtype=dtype, overscan=overscan, intrinsics=K.to(DEV)).cpu()
        assert img.shape == (1, V, H, W, 3)
        _check(img, ref, f"{name} {res} on {canvas} {dtype}")


# ------------------------------------------------------------------------------------------------ graphs / stream
def test_intrinsics_graphs_are_separate_entries_and_replay_new_values():
    pipe, _, _ = _pipe("tiny_swin", 8)
    sc = make_scene(90, 2, seed=72)
    args = _args(sc)
    fov = sc["fov"].to(DEV)
    res = (128, 192)
    K1 = torch.stack([_calibrated(sc["fov"][0, :, 0], *res, sy=1.2, dx=5.0)]).to(DEV)
    K2 = torch.stack([_calibrated(sc["fov"][0, :, 0], *res, sx=0.8, dy=-30.0)]).to(DEV)
    eager = [pipe(*args, fov, resolution=res)] + [pipe(*args, resolution=res, intrinsics=k) for k in (K1, K2)]
    assert not torch.equal(eager[1], eager[2])
    pipe.cuda_graphs = True
    n0 = len(pipe._graphs)
    for _ in range(2):
        assert torch.equal(pipe(*args, fov, resolution=res), eager[0])
        assert torch.equal(pipe(*args, resolution=res, intrinsics=K1), eager[1])
        assert torch.equal(pipe(*args, resolution=res, intrinsics=K2), eager[2])   # a replay with new values
    assert len(pipe._graphs) == n0 + 2, "a fov render and an intrinsics render must be separate graphs"
    keys = list(pipe._graphs)[n0:]
    assert {"fov", "intrinsics"} <= {k for key in keys for k in key if isinstance(k, str)}


def test_intrinsics_render_views_on_a_static_state_and_empty_slice():
    pipe, _, _ = _pipe("tiny_swin", 8)
    sc = {k: v.to(DEV) for k, v in make_scene(40, 3, seed=73).items()}
    K = pipe.intrinsics_from_fov(sc["fov"], (64, 128), fit="vertical")
    st = pipe.encode(sc["triangles"], sc["texture"], sc["mask"], sc["vn"])
    want = pipe.render_views(st, sc["c2w"], resolution=(64, 128), intrinsics=K)
    assert want.shape == (1, 3, 64, 128, 3)
    assert torch.equal(want, pipe(sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], resolution=(64, 128),
                                  intrinsics=K))
    out = pipe.render_views(st, sc["c2w"][:, :0], resolution=(99, 150), overscan=True, intrinsics=K[:, :0])
    assert out.shape == (1, 0, 99, 150, 3)


def _k_scenes(counts, res, seed0):
    """Host scenes with 'intrinsics' [1, V, 4] in place of 'fov'."""
    out = []
    for i, n in enumerate(counts):
        sc = make_scene(n, 2, seed=seed0 + i)
        fov = sc.pop("fov")
        sc["intrinsics"] = torch.stack([_calibrated(fov[0, :, 0], *res, sx=1.0 + 0.1 * i, sy=0.9, dx=3.0 * i)])
        out.append(sc)
    return out


def test_intrinsics_render_stream_is_per_scene_render():
    pipe, _, _ = _pipe("tiny_swin", 8)
    res = (99, 150)
    pipe.cuda_graphs = True
    scenes = _k_scenes((61, 100), res, 80)
    want = [pipe(*_args({k: v for k, v in sc.items() if k != "intrinsics"}), resolution=res, overscan=True,
                 intrinsics=sc["intrinsics"].to(DEV)).cpu() for sc in scenes]
    host = [{k: t.pin_memory() for k, t in sc.items()} for sc in scenes]
    got = [img.clone() for img in pipe.render_stream(iter(host), resolution=res, overscan=True)]
    assert len(got) == 2
    for a, b in zip(got, want):
        assert a.shape == (1, 2, *res, 3)
        assert torch.equal(a, b)


def test_intrinsics_render_to_files(tmp_path):
    """Scenes carrying 'intrinsics' go through render_to_files; every EXR frame is the `render` image."""
    from renderformer_b200 import frame_io as fio
    pipe, _, _ = _pipe("tiny_swin", 8)
    res = (64, 128)
    scenes = _k_scenes((30, 45), res, 90)
    paths = fio.render_to_files(pipe, iter(scenes), ["a", "b"], str(tmp_path), resolution=res, workers=1)
    assert len(paths) == 4
    for name, sc in zip(("a", "b"), scenes):
        img = pipe(*_args({k: v for k, v in sc.items() if k != "intrinsics"}), resolution=res,
                   intrinsics=sc["intrinsics"].to(DEV)).cpu()
        for v in range(2):
            got = torch.from_numpy(fio.read_exr(str(tmp_path / f"{name}_view_{v}.exr"))).float()
            assert torch.equal(got, img[0, v])


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
K = pipe.intrinsics_from_fov(sc["fov"], (99, 150))
K = K * torch.tensor([1.0, 1.2, 1.0, 1.0], device=dev) + torch.tensor([0.0, 0.0, 7.5, -4.0], device=dev)
args = (sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"])
single = pipe(*args, resolution=(99, 150), overscan=True, intrinsics=K).clone()
ok = single.shape == (1, 4, 99, 150, 3)
for graphs in (False, True):
    pipe.cuda_graphs = graphs
    for rep in range(2):
        out = render_sharded(pipe, *args, resolution=(99, 150), dst=0, overscan=True, intrinsics=K)
        if rank == 0 and not (out.shape == single.shape and torch.equal(out, single)):
            ok = False
dist.barrier()
if rank == 0:
    print("INTRINSICS_SHARDED_OK" if ok else "INTRINSICS_SHARDED_MISMATCH", flush=True)
pipe._graphs.clear()
torch.cuda.synchronize()
dist.barrier()
sys.stdout.flush()
os._exit(0)
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_render_sharded_intrinsics_equals_single_gpu(tmp_path):
    worker = tmp_path / "intrinsics_worker.py"
    worker.write_text(WORKER % {"root": ROOT})
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), str(worker)], capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "INTRINSICS_SHARDED_OK" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])
