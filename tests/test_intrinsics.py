"""CPU: per-view pinhole intrinsics -- the intrinsics camera of the oracle extension (tests/intrinsics_oracle.py)
against the fov camera, the host checks of config.view_camera, the sensor-fit rule, FLOP counts (the camera does not
change the work) and the C header."""
import inspect
import math
import os
import sys

import pytest
import torch

from renderformer_b200 import flops, lib
from renderformer_b200.config import RenderFormerConfig, view_camera

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from intrinsics_oracle import camera_rays_k, intrinsics_from_fov_f64  # noqa: E402
from overscan_oracle import camera_rays_overscan  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWIN = RenderFormerConfig.named("tiny_swin")


@pytest.mark.parametrize("H,W,Hc,Wc,top,left", [(64, 64, 64, 64, 0, 0), (128, 192, 128, 192, 0, 0),
                                                 (192, 128, 192, 128, 0, 0), (99, 150, 128, 192, 14, 21),
                                                 (1080, 1920, 1088, 1920, 4, 0), (150, 99, 192, 128, 21, 14)])
def test_centred_fov_intrinsics_are_the_fov_camera(H, W, Hc, Wc, top, left):
    fov = torch.tensor([[math.radians(37.5)], [math.radians(70.0)], [0.3]])
    fl = max(H, W) / 2 / torch.tan(0.5 * fov[:, 0])
    K = torch.stack([fl, fl, torch.full_like(fl, W / 2), torch.full_like(fl, H / 2)], dim=-1)
    assert torch.equal(camera_rays_k(K, H, W, Hc, Wc, top, left), camera_rays_overscan(fov, H, W, Hc, Wc, top, left))


def test_camera_rays_k_moves_with_the_principal_point_and_focal_lengths():
    """Spot values of the convention: the ray through (cx, cy) is the optical axis, fx and fy scale x and y apart."""
    K = torch.tensor([[100.0, 50.0, 10.0, 20.0]])
    rays = camera_rays_k(K, 40, 30, 40, 30, 0, 0)[0]
    # pixel (row 19, column 9) has its centre at (9.5, 19.5): half a pixel left of and above (cx, cy)
    d = torch.tensor([-0.5 / 100.0, 0.5 / 50.0, -1.0])
    assert torch.allclose(rays[19, 9], d / d.norm(), atol=1e-7)
    # with an offset on a canvas the window's rays are the image's
    canvas = camera_rays_k(K, 40, 30, 48, 40, 3, 5)[0]
    assert torch.allclose(canvas[3:43, 5:35], rays, atol=0)


def _cams(B=1, V=3):
    return torch.eye(4).repeat(B, V, 1, 1)


def test_view_camera_accepts():
    c2w = _cams(2, 3)
    fov = torch.full((2, 3, 1), 40.0)
    assert view_camera(c2w, fov=fov) == ("fov", fov)
    K = torch.tensor([300.0, 250.0, -40.0, 600.0]).repeat(2, 3, 1)   # principal point outside the image is fine
    kind, cam = view_camera(c2w, intrinsics=K)
    assert kind == "intrinsics" and cam is K
    assert view_camera(c2w, intrinsics=K.double())[0] == "intrinsics"
    assert view_camera(c2w[:, :0], intrinsics=K[:, :0])[0] == "intrinsics"   # an empty view slice


@pytest.mark.parametrize("fov,K,what", [
    (None, None, "neither"),
    (torch.full((1, 3, 1), 40.0), torch.full((1, 3, 4), 100.0), "both"),
    (None, torch.full((1, 3, 3), 100.0), "three values"),
    (None, torch.full((1, 2, 4), 100.0), "view count"),
    (None, torch.full((2, 3, 4), 100.0), "batch"),
    (None, torch.full((3, 4), 100.0), "rank"),
    (None, torch.tensor([[[0.0, 100.0, 1.0, 1.0]] * 3]), "fx = 0"),
    (None, torch.tensor([[[100.0, -100.0, 1.0, 1.0]] * 3]), "fy < 0"),
    (None, torch.tensor([[[float("inf"), 100.0, 1.0, 1.0]] * 3]), "fx inf"),
    (None, torch.tensor([[[100.0, 100.0, float("nan"), 1.0]] * 3]), "cx nan"),
    (None, torch.full((1, 3, 4), 100, dtype=torch.int32), "integer"),
    (None, [[[100.0, 100.0, 1.0, 1.0]] * 3], "not a tensor"),
])
def test_view_camera_rejects(fov, K, what):
    with pytest.raises(ValueError):
        view_camera(_cams(1, 3), fov=fov, intrinsics=K)


@pytest.mark.parametrize("H,W", [(1080, 1920), (256, 512), (99, 150)])
def test_auto_fit_is_horizontal_on_landscape_vertical_on_portrait(H, W):
    fov = torch.tensor([20.0, 37.5, 90.0])
    assert torch.equal(intrinsics_from_fov_f64(fov, H, W, "auto"), intrinsics_from_fov_f64(fov, H, W, "horizontal"))
    assert torch.equal(intrinsics_from_fov_f64(fov, W, H, "auto"), intrinsics_from_fov_f64(fov, W, H, "vertical"))
    K = intrinsics_from_fov_f64(fov, H, W, "vertical")
    assert torch.allclose(2 * torch.atan(H / 2 / K[:, 1]) * 180 / math.pi, fov.double())   # the fov spans the height
    assert torch.equal(K[:, 2:], torch.tensor([[W / 2, H / 2]] * 3, dtype=torch.float64))


def test_flops_do_not_depend_on_the_camera():
    """The camera only changes the rays, not the work: FLOP counts take no camera argument, so a render with
    intrinsics counts what the same-size fov render counts."""
    for fn in (flops.view_flops, flops.job_flops, flops.dpt_flops, flops.scene_flops):
        params = set(inspect.signature(fn).parameters)
        assert not params & {"fov", "intrinsics", "camera"}, fn.__name__
    cfg = RenderFormerConfig.named("v1_1_swin_large")
    assert flops.view_flops(cfg, 4096, (1080, 1920), overscan=True) == flops.view_flops(cfg, 4096, (1088, 1920))


def test_header_and_bindings_declare_the_entry_points():
    with open(os.path.join(ROOT, "include", "rfb200.h")) as f:
        header = " ".join(f.read().split())
    assert ("int rfb_ray_tokens_intrinsics(const float* intr, void* out, int n_views, int canvas_h, int canvas_w, "
            "int height, int width, int top, int left, rfb_stream_t stream);") in header
    assert ("int rfb_intrinsics_from_fov(const float* fov_deg, float* out, int n_views, int height, int width, int fit, "
            "rfb_stream_t stream);") in header
    assert {"rfb_ray_tokens_intrinsics", "rfb_intrinsics_from_fov"} <= set(lib.SYMBOLS)


def test_pipeline_checks_the_camera_before_any_launch():
    """Camera errors are ValueErrors on the host, before anything reaches the kernels (which, without a GPU, would
    fail with RfbError: there is no CPU fallback)."""
    from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
    from renderformer_b200.synth import make_scene
    pipe = RenderFormerRenderingPipeline(RenderFormer(SWIN))
    sc = make_scene(8, 2)
    args = (sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"])
    K = torch.tensor([100.0, 100.0, 32.0, 32.0]).repeat(1, 2, 1)
    with pytest.raises(ValueError):
        pipe(*args, sc["fov"], resolution=64, intrinsics=K)
    with pytest.raises(ValueError):
        pipe(*args, resolution=64)
    with pytest.raises(ValueError):
        pipe(*args, resolution=64, intrinsics=K[:, :1])
    bad = K.clone()
    bad[0, 1, 1] = 0.0
    with pytest.raises(ValueError):
        pipe(*args, resolution=64, intrinsics=bad)
    with pytest.raises(ValueError):
        pipe.intrinsics_from_fov(sc["fov"], 64, fit="sensor")
    with pytest.raises(ValueError):
        pipe.intrinsics_from_fov(sc["fov"], (0, 64))
    if not torch.cuda.is_available():
        with pytest.raises(lib.RfbError):
            pipe(*args, resolution=64, intrinsics=K)
