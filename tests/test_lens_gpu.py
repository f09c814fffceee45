"""GPU: lens-distorted cameras through every layer -- the lens ray-token kernel against the float64 oracle for OpenCV and
fisheye lenses on plain images and overscan canvases, bit identity of zero-coefficient OpenCV lenses with the plain
intrinsics render, finite tokens for coefficients that do not invert, the fp32 oracle with distorted cameras, CUDA
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
from renderformer_b200.config import RenderFormerConfig, overscan_grid, view_camera
from renderformer_b200.metrics import PSNR_MIN, REL_TOL, hdr_rel_err, log_psnr
from renderformer_b200.synth import init_state_dict, make_scene

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from intrinsics_oracle import intrinsics_from_fov_f64  # noqa: E402
from lens_oracle import LENS_CASES, camera_rays_lens, lens_case, render_lens  # noqa: E402

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


def _tokens(K, D, lens, Hc, Wc, H, W, top, left):
    V = K.shape[0]
    out = torch.empty(V * (Hc // 8) * (Wc // 8), 192, dtype=torch.float16, device=DEV)
    return ops.ray_tokens_lens(K.to(DEV).contiguous(), D.to(DEV).contiguous(), out, lens=lens, n_views=V, canvas_h=Hc,
                               canvas_w=Wc, height=H, width=W, top=top, left=left)


def _pad8(D):
    return torch.cat([D, torch.zeros(*D.shape[:-1], 8 - D.shape[-1], dtype=D.dtype, device=D.device)], dim=-1)


# ------------------------------------------------------------------------------------------------ ray tokens
@pytest.mark.parametrize("name", sorted(LENS_CASES))
@pytest.mark.parametrize("H,W,Hc,Wc,top,left", [
    (64, 192, 64, 192, 0, 0),        # landscape, canvas = image
    (192, 64, 192, 64, 0, 0),        # portrait
    (99, 150, 128, 192, 14, 21),     # on an overscan canvas
    (1080, 1920, 1088, 1920, 4, 0),
])
def test_lens_ray_tokens_match_the_float64_oracle(name, H, W, Hc, Wc, top, left):
    lens, K, D = lens_case(name, H, W)
    view_camera(torch.eye(4).repeat(1, K.shape[0], 1, 1), intrinsics=K[None], distortion=D[None], lens=lens,
                canvas=(Hc, Wc), window=(H, W, top, left))   # the camera passes the host check
    V = K.shape[0]
    tok = _tokens(K, D, lens, Hc, Wc, H, W, top, left)
    rays = camera_rays_lens(K.double().to(DEV), D.double().to(DEV), lens, H, W, Hc, Wc, top, left)
    want = ops.ray_map_tokens(rays.float().contiguous(), torch.empty_like(tok), n_views=V, height=Hc, width=Wc)
    a, b = tok.float(), want.float()
    ulp = torch.maximum(a.abs(), b.abs()).clamp_min(2.0 ** -14) * 2.0 ** -10   # one fp16 ulp at the larger value
    e = (a - b).abs() / ulp
    err, i = e.max().item(), e.argmax().item()
    worst = f"token {i // 192} feature {i % 192}: kernel {a.view(-1)[i].item():.6g}, oracle {b.view(-1)[i].item():.6g}"
    print(f"{name} {H}x{W} on {Hc}x{Wc}: max error {err:.2f} fp16 ulp at {worst}")
    assert torch.isfinite(a).all() and err <= 1.0, worst
    if name == "fisheye_wide":   # rays more than 100 degrees off the axis reach the kernel's corners
        assert (rays[..., 2] > 0.17).any()


@pytest.mark.parametrize("H,W,Hc,Wc,top,left", [(64, 192, 64, 192, 0, 0), (99, 150, 128, 192, 14, 21),
                                                 (150, 99, 152, 104, 1, 2), (1080, 1920, 1088, 1920, 4, 0)])
def test_zero_opencv_tokens_are_the_intrinsics_tokens(H, W, Hc, Wc, top, left):
    K = intrinsics_from_fov_f64(torch.tensor([20.0, 37.5, 52.0, 80.0, 120.0]), H, W)
    K = (K * torch.tensor([1.0, 1.13, 1.0, 1.0], dtype=torch.float64) +
         torch.tensor([0.0, 0.0, 5.25, -3.5], dtype=torch.float64)).float().to(DEV)
    V = K.shape[0]
    n = V * (Hc // 8) * (Wc // 8)
    want = ops.ray_tokens_intrinsics(K, torch.empty(n, 192, dtype=torch.float16, device=DEV), n_views=V, canvas_h=Hc,
                                     canvas_w=Wc, height=H, width=W, top=top, left=left)
    assert torch.equal(_tokens(K, torch.zeros(V, 8), "opencv", Hc, Wc, H, W, top, left), want)


def test_lens_kernel_rejects_bad_arguments():
    lib = L.load()
    x = torch.empty(64 * 64 * 3, device=DEV)
    p = x.data_ptr()
    for bad in ((60, 64, 50, 50, 0, 0), (64, 64, 60, 60, 5, 0), (64, 64, 60, 60, 0, 5), (64, 64, 0, 60, 0, 0),
                (64, 64, 60, -4, 0, 0), (64, 64, 60, 60, -1, 0), (0, 64, 8, 8, 0, 0)):
        assert lib.rfb_ray_tokens_lens(p, p, 0, p, 1, *bad, None) == -1, bad
    assert lib.rfb_ray_tokens_lens(p, p, 0, p, 0, 64, 64, 60, 60, 0, 0, None) == -1
    assert lib.rfb_ray_tokens_lens(p, p, 2, p, 1, 64, 64, 64, 64, 0, 0, None) == -1
    assert lib.rfb_ray_tokens_lens(p, p, -1, p, 1, 64, 64, 64, 64, 0, 0, None) == -1
    assert lib.rfb_ray_tokens_lens(p, None, 0, p, 1, 64, 64, 64, 64, 0, 0, None) == -1
    assert lib.rfb_ray_tokens_lens(None, p, 1, p, 1, 64, 64, 64, 64, 0, 0, None) == -1
    with pytest.raises(ValueError):
        ops.ray_tokens_lens(x[:4], x[:4], x, lens="equisolid", n_views=1, canvas_h=8, canvas_w=8, height=8, width=8)
    with pytest.raises(ValueError):   # opencv reads 8 coefficients per view
        ops.ray_tokens_lens(x[:4], x[:4], x, lens="opencv", n_views=1, canvas_h=8, canvas_w=8, height=8, width=8)


def test_device_coefficients_that_do_not_invert_give_finite_tokens():
    """Device tensors are not checked on the host: folding lenses, a vanishing denominator and a fisheye whose
    theta_d falls back towards 0 must still give finite tokens (the kernel falls back to the pinhole ray)."""
    H, W = 99, 150
    K = torch.tensor([[60.0, 60.0, 75.0, 49.5]] * 4)
    opencv = torch.tensor([[-1.5, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0],      # folds at r = 0.47
                           [0.0, 0.0, 0.0, 0.0, 0.0, -1.0, 0.0, 0.0],      # denominator 0 at r = 1
                           [5.0, -20.0, 3.0, -3.0, 40.0, -2.0, 1.0, -8.0],
                           [float("inf"), 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0]])
    fisheye = torch.tensor([[-0.5, 0.0, 0.0, 0.0], [-1.0, 0.3, -0.5, 0.1], [0.0, 0.0, 0.0, -3.0],
                            [float("nan"), 0.0, 0.0, 0.0]])
    for lens, D in (("opencv", opencv), ("fisheye", fisheye)):
        tok = _tokens(K, D, lens, 128, 192, H, W, 14, 21)
        assert torch.isfinite(tok.float()).all(), lens


# ------------------------------------------------------------------------------------------------ bit identity
@pytest.mark.parametrize("graphs", [False, True], ids=["eager", "graphs"])
@pytest.mark.parametrize("res,overscan", [(512, False), ((256, 512), False), ((1080, 1920), True)],
                         ids=["512", "256x512", "1080p"])
def test_zero_opencv_render_is_the_intrinsics_render(res, overscan, graphs):
    pipe, _, _ = _pipe("v1_1_swin_large", 5)
    sc = make_scene(512, 2, seed=70)
    args = _args(sc)
    pipe.cuda_graphs = graphs
    K = pipe.intrinsics_from_fov(sc["fov"].to(DEV), res) * torch.tensor([1.0, 1.1, 1.0, 1.0], device=DEV) + \
        torch.tensor([0.0, 0.0, 6.5, -4.25], device=DEV)
    for _ in range(2 if graphs else 1):   # the second call of a graphed render is a replay
        want = pipe(*args, resolution=res, torch_dtype=torch.bfloat16, overscan=overscan, intrinsics=K)
        for n in (8, 4, 5):
            got = pipe(*args, resolution=res, torch_dtype=torch.bfloat16, overscan=overscan, intrinsics=K,
                       distortion=torch.zeros(1, 2, n, device=DEV))
            assert torch.equal(got, want), n


# ------------------------------------------------------------------------------------------------ oracle
@pytest.mark.parametrize("name,n_tris,res,overscan,dtypes", [
    ("v1_1_swin_large", 512, (256, 512), False, (torch.bfloat16,)),
    ("tiny_swin", 90, (99, 150), True, (torch.bfloat16, torch.float16)),
    ("tiny_full", 90, (99, 150), True, (torch.bfloat16, torch.float16)),
])
@pytest.mark.parametrize("case", ["barrel", "fisheye_wide"])
def test_lens_against_oracle(name, n_tris, res, overscan, dtypes, case):
    pipe, sd, cfg = _pipe(name, 5)
    V = 1 if name == "v1_1_swin_large" else 2
    sc = make_scene(n_tris, V, seed=71)
    H, W = res
    lens, K, D = lens_case(case, H, W)
    K, D = K[None, :V], D[None, :V]
    if overscan:
        hw, canvas, offsets = overscan_grid(cfg, res)
    else:
        hw, canvas, offsets = res, res, (0, 0)
    ref = render_lens(sd, cfg, sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], K, D, lens, hw, canvas,
                      offsets)
    for dtype in dtypes:
        img = pipe(*_args(sc), resolution=res, torch_dtype=dtype, overscan=overscan, intrinsics=K, distortion=D,
                   lens=lens).cpu()   # host tensors: checked, then uploaded
        assert img.shape == (1, V, H, W, 3)
        _check(img, ref, f"{name} {case} {res} on {canvas} {dtype}")


# ------------------------------------------------------------------------------------------------ graphs / stream
def test_lens_graphs_are_separate_entries_and_replay_new_values():
    pipe, _, _ = _pipe("tiny_swin", 8)
    sc = make_scene(90, 2, seed=72)
    args = _args(sc)
    res = (128, 192)
    _, K, Db = lens_case("barrel", *res)
    _, Kf, Df = lens_case("fisheye_mild", *res)
    K, Kf = K[None].to(DEV), Kf[None].to(DEV)
    cams = [dict(intrinsics=K), dict(intrinsics=K, distortion=Db[None].to(DEV)),
            dict(intrinsics=K, distortion=(Db[None] * 0.5).to(DEV)),   # new coefficients, same graph
            dict(intrinsics=Kf, distortion=Df[None].to(DEV), lens="fisheye"),
            dict(intrinsics=Kf, distortion=(Df[None] * 2.0).to(DEV), lens="fisheye")]
    eager = [pipe(*args, resolution=res, **c) for c in cams]
    assert not torch.equal(eager[1], eager[2]) and not torch.equal(eager[3], eager[4])
    pipe.cuda_graphs = True
    n0 = len(pipe._graphs)
    for _ in range(2):
        for c, want in zip(cams, eager):
            assert torch.equal(pipe(*args, resolution=res, **c), want)
    assert len(pipe._graphs) == n0 + 3, "pinhole, opencv and fisheye renders must be separate graphs"
    keys = list(pipe._graphs)[n0:]
    assert {"intrinsics", "opencv", "fisheye"} <= {k for key in keys for k in key if isinstance(k, str)}


def test_lens_render_views_on_a_static_state():
    pipe, _, _ = _pipe("tiny_swin", 8)
    sc = {k: v.to(DEV) for k, v in make_scene(40, 2, seed=73).items()}
    lens, K, D = lens_case("fisheye_wide", 64, 128)
    K, D = K[None].to(DEV), D[None].to(DEV)
    st = pipe.encode(sc["triangles"], sc["texture"], sc["mask"], sc["vn"])
    want = pipe.render_views(st, sc["c2w"], resolution=(64, 128), intrinsics=K, distortion=D, lens=lens)
    assert want.shape == (1, 2, 64, 128, 3)
    assert torch.equal(want, pipe(sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"], resolution=(64, 128),
                                  intrinsics=K, distortion=D, lens=lens))
    out = pipe.render_views(st, sc["c2w"][:, :0], resolution=(99, 150), overscan=True, intrinsics=K[:, :0],
                            distortion=D[:, :0], lens=lens)
    assert out.shape == (1, 0, 99, 150, 3)


def _lens_scenes(counts, res, seed0, case):
    """Host scenes with 'intrinsics' [1, V, 4] and 'distortion' [1, V, n] in place of 'fov'."""
    out = []
    for i, n in enumerate(counts):
        sc = make_scene(n, 2, seed=seed0 + i)
        sc.pop("fov")
        _, K, D = lens_case(case, *res)
        sc["intrinsics"], sc["distortion"] = K[None] * (1.0 + 0.05 * i), D[None] * (1.0 - 0.2 * i)
        out.append(sc)
    return out


@pytest.mark.parametrize("case", ["rational", "fisheye_mild"])
def test_lens_render_stream_is_per_scene_render(case):
    pipe, _, _ = _pipe("tiny_swin", 8)
    res = (99, 150)
    lens = LENS_CASES[case][0]
    pipe.cuda_graphs = True
    scenes = _lens_scenes((61, 100), res, 80, case)
    want = [pipe(*_args({k: v for k, v in sc.items() if k not in ("intrinsics", "distortion")}), resolution=res,
                 overscan=True, intrinsics=sc["intrinsics"].to(DEV), distortion=sc["distortion"].to(DEV),
                 lens=lens).cpu() for sc in scenes]
    host = [{k: t.pin_memory() for k, t in sc.items()} for sc in scenes]
    got = [img.clone() for img in pipe.render_stream(iter(host), resolution=res, overscan=True, lens=lens)]
    assert len(got) == 2
    for a, b in zip(got, want):
        assert a.shape == (1, 2, *res, 3)
        assert torch.equal(a, b)


def test_lens_render_to_files(tmp_path):
    """Scenes carrying 'intrinsics' and 'distortion' go through render_to_files; every EXR frame is the `render`
    image."""
    from renderformer_b200 import frame_io as fio
    pipe, _, _ = _pipe("tiny_swin", 8)
    res = (64, 128)
    scenes = _lens_scenes((30, 45), res, 90, "fisheye_wide")
    paths = fio.render_to_files(pipe, iter(scenes), ["a", "b"], str(tmp_path), resolution=res, workers=1,
                                lens="fisheye")
    assert len(paths) == 4
    for name, sc in zip(("a", "b"), scenes):
        img = pipe(*_args({k: v for k, v in sc.items() if k not in ("intrinsics", "distortion")}), resolution=res,
                   intrinsics=sc["intrinsics"].to(DEV), distortion=sc["distortion"].to(DEV), lens="fisheye").cpu()
        for v in range(2):
            got = torch.from_numpy(fio.read_exr(str(tmp_path / f"{name}_view_{v}.exr"))).float()
            assert torch.equal(got, img[0, v])


WORKER = r"""
import os, sys, torch
sys.path.insert(0, %(root)r)
sys.path.insert(0, os.path.join(%(root)r, "tests"))
import torch.distributed as dist
from lens_oracle import lens_case
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
args = (sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"])
ok = True
for case in ("barrel", "fisheye_wide"):
    lens, K, D = lens_case(case, 99, 150)
    K = torch.cat([K, K * 1.1])[None].to(dev)   # 4 views
    D = torch.cat([D, D * 0.5])[None].to(dev)
    single = pipe(*args, resolution=(99, 150), overscan=True, intrinsics=K, distortion=D, lens=lens).clone()
    ok = ok and single.shape == (1, 4, 99, 150, 3)
    for graphs in (False, True):
        pipe.cuda_graphs = graphs
        for rep in range(2):
            out = render_sharded(pipe, *args, resolution=(99, 150), dst=0, overscan=True, intrinsics=K, distortion=D,
                                 lens=lens)
            if rank == 0 and not (out.shape == single.shape and torch.equal(out, single)):
                ok = False
    pipe.cuda_graphs = False
dist.barrier()
if rank == 0:
    print("LENS_SHARDED_OK" if ok else "LENS_SHARDED_MISMATCH", flush=True)
pipe._graphs.clear()
torch.cuda.synchronize()
dist.barrier()
sys.stdout.flush()
os._exit(0)
"""


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_render_sharded_lens_equals_single_gpu(tmp_path):
    worker = tmp_path / "lens_worker.py"
    worker.write_text(WORKER % {"root": ROOT})
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), str(worker)], capture_output=True, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0 and "LENS_SHARDED_OK" in r.stdout, (r.stdout[-1500:], r.stderr[-3000:])
