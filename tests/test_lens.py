"""CPU: lens-distorted cameras -- the float64 lens camera of the oracle extension (tests/lens_oracle.py) against its own
forward models and the pinhole / equidistant closed forms, the host checks of config.view_camera (shapes, padding,
lens names, finiteness, invertibility on the canvas), the COLMAP text-model reader with a convention pin, FLOP counts
and the C header."""
import inspect
import math
import os
import sys

import numpy as np
import pytest
import torch

from renderformer_b200 import flops, lib
from renderformer_b200.config import RenderFormerConfig, camera_kwargs, view_camera
from renderformer_b200.scene_io import read_colmap_cameras

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from intrinsics_oracle import camera_rays_k  # noqa: E402
from lens_oracle import (LENS_CASES, camera_rays_lens, distort_fisheye, distort_opencv, lens_case,  # noqa: E402
                         lens_rays, undistort_fisheye, undistort_opencv)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWIN = RenderFormerConfig.named("tiny_swin")
# every (H, W, Hc, Wc, top, left) the GPU tests render or tokenise a LENS_CASES camera on
GPU_CANVASES = [(64, 192, 64, 192, 0, 0), (192, 64, 192, 64, 0, 0), (99, 150, 128, 192, 14, 21),
                (1080, 1920, 1088, 1920, 4, 0), (256, 512, 256, 512, 0, 0), (99, 150, 104, 152, 2, 1),
                (128, 192, 128, 192, 0, 0), (64, 128, 64, 128, 0, 0)]


def _cams(B=1, V=2):
    return torch.eye(4).repeat(B, V, 1, 1)


# ------------------------------------------------------------------------------------------------ oracle
@pytest.mark.parametrize("name", sorted(LENS_CASES))
def test_oracle_inverse_round_trips(name):
    lens, K, D = lens_case(name, 99, 150)
    rays = camera_rays_lens(K.double(), D.double(), lens, 99, 150, 128, 192, 14, 21)   # inverts every canvas pixel
    assert torch.isfinite(rays).all() and torch.allclose(rays.norm(dim=-1), torch.ones(1, dtype=torch.float64))
    g = torch.Generator().manual_seed(3)
    D = D[0].double()
    if lens == "opencv":
        x, y = torch.rand(2, 4096, generator=g, dtype=torch.float64) * 1.0 - 0.5
        xd, yd = distort_opencv(x, y, D)
        x2, y2 = undistort_opencv(xd, yd, D)
        a, b = distort_opencv(x2, y2, D)
        assert (a - xd).abs().max() <= 1e-12 and (b - yd).abs().max() <= 1e-12
        assert (x2 - x).abs().max() <= 1e-12 and (y2 - y).abs().max() <= 1e-12
    else:
        th = torch.rand(4096, generator=g, dtype=torch.float64) * 1.9
        rd = distort_fisheye(th, D)
        assert (distort_fisheye(undistort_fisheye(rd, D), D) - rd).abs().max() <= 1e-12
        assert (undistort_fisheye(rd, D) - th).abs().max() <= 1e-12


@pytest.mark.parametrize("H,W,Hc,Wc,top,left", [(64, 64, 64, 64, 0, 0), (99, 150, 128, 192, 14, 21),
                                                 (1080, 1920, 1088, 1920, 4, 0), (150, 99, 192, 128, 21, 14)])
def test_zero_opencv_rays_are_the_pinhole_rays(H, W, Hc, Wc, top, left):
    K = torch.tensor([[900.0, 910.0, W / 2 + 3.25, H / 2 - 7.5], [300.0, 280.0, -40.0, H + 5.0]], dtype=torch.float64)
    assert torch.equal(camera_rays_lens(K, torch.zeros(2, 8, dtype=torch.float64), "opencv", H, W, Hc, Wc, top, left),
                       camera_rays_k(K, H, W, Hc, Wc, top, left))


def test_zero_fisheye_rays_are_equidistant():
    K = torch.tensor([[300.0, 310.0, 75.5, 49.0]], dtype=torch.float64)
    rays = camera_rays_lens(K, torch.zeros(1, 4, dtype=torch.float64), "fisheye", 99, 150, 128, 192, 14, 21)[0]
    u = torch.arange(192, dtype=torch.float64) + 0.5 - 21
    v = torch.arange(128, dtype=torch.float64)[:, None] + 0.5 - 14
    xd, yd = (u - 75.5) / 300.0, (v - 49.0) / 310.0
    th = torch.sqrt(xd ** 2 + yd ** 2)   # equidistant: the angle off the axis is the distorted radius
    want = torch.stack([torch.sin(th) * xd / th, -torch.sin(th) * yd / th, -torch.cos(th)], dim=-1)
    assert torch.allclose(rays, want, rtol=0, atol=1e-15)
    # wide angles: rays 90 degrees and more off the axis are valid
    r = lens_rays(torch.tensor([75.5 + 300 * 2.0], dtype=torch.float64), torch.tensor([49.0], dtype=torch.float64),
                  K[0], torch.zeros(4, dtype=torch.float64), "fisheye")[0]
    assert torch.allclose(r, torch.tensor([math.sin(2.0), 0.0, -math.cos(2.0)], dtype=torch.float64), atol=1e-15)
    assert r[2] > 0


# ------------------------------------------------------------------------------------------------ validation
@pytest.mark.parametrize("name", sorted(LENS_CASES))
def test_gpu_test_cameras_pass_the_host_check(name):
    for H, W, Hc, Wc, top, left in GPU_CANVASES:
        lens, K, D = lens_case(name, H, W)
        kind, cam = view_camera(_cams(1, 2), intrinsics=K[None], distortion=D[None], lens=lens, canvas=(Hc, Wc),
                                window=(H, W, top, left))
        assert kind == lens and cam.shape == (1, 2, 4 + D.shape[-1])


@pytest.mark.parametrize("n", [4, 5, 8])
def test_opencv_coefficients_are_padded_to_eight(n):
    K = torch.tensor([[[500.0, 510.0, 32.0, 32.0]] * 2])
    D = torch.tensor([[[-0.1, 0.01, 0.001, -0.002, 0.003, 0.05, 0.004, 0.0005][:n]] * 2])
    kind, cam = view_camera(_cams(), intrinsics=K, distortion=D, canvas=(64, 64))
    assert kind == "opencv" and cam.shape == (1, 2, 12) and cam.dtype == torch.float32
    assert torch.equal(cam[..., :4], K) and torch.equal(cam[..., 4:4 + n], D)
    assert not cam[..., 4 + n:].any()
    kw = camera_kwargs(kind, cam)
    assert kw["lens"] == "opencv" and torch.equal(kw["intrinsics"], K) and kw["distortion"].shape == (1, 2, 8)
    kind, cam = view_camera(_cams(), intrinsics=K, distortion=D[..., :4], lens="fisheye", canvas=(64, 64))
    assert kind == "fisheye" and cam.shape == (1, 2, 8)
    assert view_camera(_cams(), intrinsics=K, lens="fisheye") == ("intrinsics", K)   # no distortion: the pinhole


@pytest.mark.skipif(not torch.cuda.is_available(), reason="device tensors need a GPU")
def test_padding_stays_on_the_device():
    K = torch.tensor([[[500.0, 510.0, 32.0, 32.0]] * 2], device="cuda")
    kind, cam = view_camera(_cams().cuda(), intrinsics=K, distortion=torch.full((1, 2, 4), -5.0, device="cuda"),
                            canvas=(64, 64))   # device values are not read back, so not checked
    assert cam.is_cuda and cam.shape == (1, 2, 12)


K2 = torch.tensor([[[500.0, 510.0, 32.0, 32.0]] * 2])
SHORT = torch.tensor([0.05, 0.05, 1.0, 1.0])   # focal lengths of 25 pixels: the 64 x 64 canvas reaches r = 1.3


@pytest.mark.parametrize("kw,what", [
    (dict(fov=torch.full((1, 2, 1), 40.0), distortion=torch.zeros(1, 2, 8)), "with fov"),
    (dict(distortion=torch.zeros(1, 2, 8)), "without a camera"),
    (dict(intrinsics=K2, distortion=torch.zeros(1, 2, 6)), "six opencv coefficients"),
    (dict(intrinsics=K2, distortion=torch.zeros(1, 2, 12)), "twelve"),
    (dict(intrinsics=K2, distortion=torch.zeros(1, 2, 5), lens="fisheye"), "five fisheye coefficients"),
    (dict(intrinsics=K2, distortion=torch.zeros(1, 2, 8), lens="fisheye"), "eight fisheye coefficients"),
    (dict(intrinsics=K2, distortion=torch.zeros(1, 3, 8)), "view count"),
    (dict(intrinsics=K2, distortion=torch.zeros(2, 2, 8)), "batch"),
    (dict(intrinsics=K2, distortion=torch.zeros(2, 8)), "rank"),
    (dict(intrinsics=K2, distortion=torch.zeros(1, 2, 8, dtype=torch.int32)), "integer"),
    (dict(intrinsics=K2, distortion=[[[0.0] * 8] * 2]), "not a tensor"),
    (dict(intrinsics=K2, distortion=torch.zeros(1, 2, 8), lens="kannala"), "unknown lens"),
    (dict(intrinsics=K2, lens="pinhole"), "unknown lens without distortion"),
    (dict(intrinsics=K2, distortion=torch.tensor([[[float("nan")] + [0.0] * 7] * 2])), "nan"),
    (dict(intrinsics=K2, distortion=torch.tensor([[[0.0, float("inf"), 0.0, 0.0]] * 2]), lens="fisheye"), "inf"),
    (dict(intrinsics=K2 * SHORT, distortion=torch.tensor([[[0.0, 0.0, 0.0, 0.0, 0.0, -1.5, 0.0, 0.0]] * 2])),
     "denominator reaches zero"),
    (dict(intrinsics=K2 * SHORT, distortion=torch.tensor([[[-0.3, 0.0, 0.0, 0.0]] * 2]), lens="fisheye"),
     "fisheye theta_d stops increasing"),
])
def test_view_camera_rejects(kw, what):
    with pytest.raises(ValueError):
        view_camera(_cams(), canvas=(64, 64), **kw)


def test_barrel_folding_inside_the_canvas_but_not_the_window_is_rejected():
    """r (1 + k1 r^2) peaks at r = 1/sqrt(-3 k1), at rd = 0.70 for k1 = -0.302: the 99 x 150 window reaches rd = 0.62,
    its 128 x 192 overscan canvas (which the model also sees) rd = 0.80, past the fold."""
    K = torch.tensor([[[144.0, 144.0, 75.0, 49.5]]])
    D = torch.tensor([[[-0.302, 0.0, 0.0, 0.0]]])
    view_camera(_cams(1, 1), intrinsics=K, distortion=D, canvas=(99, 150))
    with pytest.raises(ValueError, match="canvas pixel"):
        view_camera(_cams(1, 1), intrinsics=K, distortion=D, canvas=(128, 192), window=(99, 150, 14, 21))


def test_fisheye_reaching_pi_is_rejected():
    K = torch.tensor([[[40.0, 40.0, 75.0, 49.5]]])   # equidistant: the corner of 99 x 150 is at theta = 2.24
    view_camera(_cams(1, 1), intrinsics=K, distortion=torch.zeros(1, 1, 4), lens="fisheye", canvas=(99, 150))
    with pytest.raises(ValueError):   # at f = 25 the corner is at theta = 3.6 > pi
        view_camera(_cams(1, 1), intrinsics=K * torch.tensor([0.625, 0.625, 1, 1]), distortion=torch.zeros(1, 1, 4),
                    lens="fisheye", canvas=(99, 150))


def test_pipeline_checks_the_lens_before_any_launch():
    from renderformer_b200.model import RenderFormer, RenderFormerRenderingPipeline
    from renderformer_b200.synth import make_scene
    pipe = RenderFormerRenderingPipeline(RenderFormer(SWIN))
    sc = make_scene(8, 2)
    args = (sc["triangles"], sc["texture"], sc["mask"], sc["vn"], sc["c2w"])
    K = torch.tensor([100.0, 100.0, 32.0, 32.0]).repeat(1, 2, 1)
    D = torch.zeros(1, 2, 8)
    with pytest.raises(ValueError, match="intrinsics_from_fov"):
        pipe(*args, sc["fov"], resolution=64, distortion=D)
    with pytest.raises(ValueError):
        pipe(*args, resolution=64, intrinsics=K, distortion=D, lens="equisolid")
    with pytest.raises(ValueError):
        pipe(*args, resolution=64, intrinsics=K, distortion=torch.tensor([[[-2.0, 0, 0, 0]] * 2]))
    with pytest.raises(ValueError):   # the overscan canvas of 60 x 60 is 64 x 64: a barrel folding in its border
        pipe(*args, resolution=60, overscan=True, intrinsics=torch.tensor([[[52.0, 52.0, 30.0, 30.0]] * 2]),
             distortion=torch.tensor([[[-0.3, 0.0, 0.0, 0.0]] * 2]))
    if not torch.cuda.is_available():
        with pytest.raises(lib.RfbError):
            pipe(*args, resolution=64, intrinsics=K, distortion=D)


def test_flops_do_not_depend_on_the_lens():
    for fn in (flops.view_flops, flops.job_flops, flops.dpt_flops, flops.scene_flops):
        assert not set(inspect.signature(fn).parameters) & {"distortion", "lens"}, fn.__name__


def test_header_and_bindings_declare_the_entry_point():
    with open(os.path.join(ROOT, "include", "rfb200.h")) as f:
        header = " ".join(f.read().split())
    assert ("int rfb_ray_tokens_lens(const float* intr, const float* dist, int lens, void* out, int n_views, "
            "int canvas_h, int canvas_w, int height, int width, int top, int left, rfb_stream_t stream);") in header
    assert "rfb_ray_tokens_lens" in lib.SYMBOLS


# ------------------------------------------------------------------------------------------------ COLMAP
CAMERAS_TXT = """# Camera list with one line of data per camera:
#   CAMERA_ID, MODEL, WIDTH, HEIGHT, PARAMS[]
# Number of cameras: 9
1 SIMPLE_PINHOLE 640 480 500 320 240
2 PINHOLE 640 480 500 510 321.5 239.25
3 SIMPLE_RADIAL 640 480 500 320 240 -0.05
4 RADIAL 640 480 500 320 240 -0.05 0.01
5 OPENCV 640 480 500 510 321.5 239.25 -0.05 0.01 0.001 -0.002
6 FULL_OPENCV 640 480 500 510 321.5 239.25 -0.05 0.01 0.001 -0.002 0.003 0.1 0.02 0.001

7 SIMPLE_RADIAL_FISHEYE 720 540 300 360 270 0.02
8 RADIAL_FISHEYE 720 540 300 360 270 0.02 -0.003
9 OPENCV_FISHEYE 720 540 300 305 361.5 268.75 0.02 -0.003 0.001 -0.0002
"""

IMAGE_POSES = [(0.9238795, 0.0, 0.3826834, 0.0, 0.5, -0.25, 3.0), (1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0),
               (0.7071068, 0.7071068, 0.0, 0.0, -1.0, 0.5, 4.0), (0.5, 0.5, 0.5, 0.5, 0.2, 0.1, 2.5),
               (0.8660254, 0.0, 0.0, 0.5, 0.0, -1.0, 3.5), (0.6, 0.0, 0.8, 0.0, 1.5, 0.0, 5.0),
               (0.9, 0.1, -0.3, 0.2, 0.3, 0.3, 2.0), (0.1, 0.9, 0.3, -0.2, -0.4, 0.2, 2.2),
               (0.3, -0.2, 0.9, 0.1, 0.0, 0.6, 3.1)]


def _write_colmap(d):
    (d / "cameras.txt").write_text(CAMERAS_TXT)
    lines = ["# Image list with two lines of data per image:", "#   IMAGE_ID, QW, QX, QY, QZ, TX, TY, TZ, CAMERA_ID, NAME",
             "#   POINTS2D[] as (X, Y, POINT3D_ID)"]
    for i, pose in enumerate(IMAGE_POSES):
        lines.append(f"{i + 1} {' '.join(str(v) for v in pose)} {i + 1} frame_{i:03d}.jpg")
        lines.append("" if i % 2 else "100.5 200.25 7 310.0 20.0 -1")   # POINTS2D, empty for some images
    (d / "images.txt").write_text("\n".join(lines) + "\n")


def test_colmap_parameter_mapping(tmp_path):
    _write_colmap(tmp_path)
    recs = read_colmap_cameras(str(tmp_path))
    assert [r["name"] for r in recs] == [f"frame_{i:03d}.jpg" for i in range(9)]
    want = [("opencv", (500, 500, 320, 240), None),
            ("opencv", (500, 510, 321.5, 239.25), None),
            ("opencv", (500, 500, 320, 240), (-0.05, 0, 0, 0, 0, 0, 0, 0)),
            ("opencv", (500, 500, 320, 240), (-0.05, 0.01, 0, 0, 0, 0, 0, 0)),
            ("opencv", (500, 510, 321.5, 239.25), (-0.05, 0.01, 0.001, -0.002, 0, 0, 0, 0)),
            ("opencv", (500, 510, 321.5, 239.25), (-0.05, 0.01, 0.001, -0.002, 0.003, 0.1, 0.02, 0.001)),
            ("fisheye", (300, 300, 360, 270), (0.02, 0, 0, 0)),
            ("fisheye", (300, 300, 360, 270), (0.02, -0.003, 0, 0)),
            ("fisheye", (300, 305, 361.5, 268.75), (0.02, -0.003, 0.001, -0.0002))]
    for r, (lens, K, D) in zip(recs, want):
        assert r["lens"] == lens and np.array_equal(r["intrinsics"], np.array(K, dtype=np.float64))
        assert (r["distortion"] is None) if D is None else np.array_equal(r["distortion"], np.array(D, dtype=np.float64))
        assert r["resolution"] == ((480, 640) if lens == "opencv" else (540, 720))
    # the identity pose is the camera at the origin looking down COLMAP's +z, i.e. this project's -z
    assert np.array_equal(recs[1]["c2w"], np.diag([1.0, -1.0, -1.0, 1.0]))


@pytest.mark.parametrize("model,params", [("FOV", "500 500 320 240 0.9"),
                                          ("THIN_PRISM_FISHEYE", "500 500 320 240" + " 0" * 8),
                                          ("RAD_TAN_THIN_PRISM_FISHEYE", "500 500 320 240" + " 0" * 16)])
def test_colmap_unsupported_models_raise(tmp_path, model, params):
    (tmp_path / "cameras.txt").write_text(f"1 {model} 640 480 {params}\n")
    (tmp_path / "images.txt").write_text("1 1 0 0 0 0 0 0 1 a.jpg\n\n")
    with pytest.raises(NotImplementedError, match=model):
        read_colmap_cameras(str(tmp_path))


def _colmap_rotation(qw, qx, qy, qz):
    """COLMAP's quaternion -> rotation matrix (Eigen's convention), float64."""
    n = math.sqrt(qw * qw + qx * qx + qy * qy + qz * qz)
    w, x, y, z = qw / n, qx / n, qy / n, qz / n
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def _colmap_project(model, p, Xc):
    """COLMAP's CamFromWorld projection of the camera-space point Xc (x right, y down, z forward) for `model` and its
    parameter list `p`, restated in float64 from COLMAP's camera models -> pixel (u, v)."""
    a, b = Xc[0] / Xc[2], Xc[1] / Xc[2]
    f = {"SIMPLE_PINHOLE": (p[0], p[0], p[1], p[2]), "SIMPLE_RADIAL": (p[0], p[0], p[1], p[2]),
         "RADIAL": (p[0], p[0], p[1], p[2]), "SIMPLE_RADIAL_FISHEYE": (p[0], p[0], p[1], p[2]),
         "RADIAL_FISHEYE": (p[0], p[0], p[1], p[2])}.get(model, tuple(p[:4]))
    fx, fy, cx, cy = f
    if model in ("SIMPLE_PINHOLE", "PINHOLE"):
        du, dv = 0.0, 0.0
    elif model == "SIMPLE_RADIAL":
        r2 = a * a + b * b
        du, dv = a * p[3] * r2, b * p[3] * r2
    elif model == "RADIAL":
        r2 = a * a + b * b
        rad = p[3] * r2 + p[4] * r2 * r2
        du, dv = a * rad, b * rad
    elif model == "OPENCV":
        k1, k2, p1, p2 = p[4:8]
        r2 = a * a + b * b
        rad = k1 * r2 + k2 * r2 * r2
        du = a * rad + 2 * p1 * a * b + p2 * (r2 + 2 * a * a)
        dv = b * rad + 2 * p2 * a * b + p1 * (r2 + 2 * b * b)
    elif model == "FULL_OPENCV":
        k1, k2, p1, p2, k3, k4, k5, k6 = p[4:12]
        r2 = a * a + b * b
        rad = (1 + k1 * r2 + k2 * r2 ** 2 + k3 * r2 ** 3) / (1 + k4 * r2 + k5 * r2 ** 2 + k6 * r2 ** 3)
        du = a * rad + 2 * p1 * a * b + p2 * (r2 + 2 * a * a) - a
        dv = b * rad + 2 * p2 * a * b + p1 * (r2 + 2 * b * b) - b
    else:   # the fisheye models: theta_d = theta (1 + k1 theta^2 + ...)
        k = (p[3], 0, 0, 0) if model == "SIMPLE_RADIAL_FISHEYE" else ((p[3], p[4], 0, 0) if model == "RADIAL_FISHEYE"
                                                                   else tuple(p[4:8]))
        r = math.hypot(a, b)
        th = math.atan(r)
        thd = th * (1 + k[0] * th ** 2 + k[1] * th ** 4 + k[2] * th ** 6 + k[3] * th ** 8)
        du, dv = a * thd / r - a, b * thd / r - b
    return fx * (a + du) + cx, fy * (b + dv) + cy


def test_colmap_convention_pin(tmp_path):
    """A world point projected by COLMAP's own equations lands on a pixel whose oracle ray, taken to the world
    through the returned c2w, points at the point."""
    _write_colmap(tmp_path)
    recs = read_colmap_cameras(str(tmp_path))
    models = [line.split()[1] for line in CAMERAS_TXT.splitlines() if line and not line.startswith("#")]
    params = [[float(v) for v in line.split()[4:]] for line in CAMERAS_TXT.splitlines()
              if line and not line.startswith("#")]
    for rec, model, p, pose in zip(recs, models, params, IMAGE_POSES):
        R, t = _colmap_rotation(*pose[:4]), np.array(pose[4:])
        for Xc_want in ([0.3, -0.2, 2.0], [-0.6, 0.45, 1.5], [0.0, 0.0, 3.0], [0.5, 0.3, 0.8]):
            X = R.T @ (np.array(Xc_want) - t)          # the world point in front of the camera
            u, v = _colmap_project(model, p, R @ X + t)
            D = rec["distortion"] if rec["distortion"] is not None else np.zeros(8)
            ray = lens_rays(torch.tensor(u, dtype=torch.float64), torch.tensor(v, dtype=torch.float64),
                            torch.from_numpy(rec["intrinsics"]), torch.from_numpy(D), rec["lens"]).numpy()
            d_world = rec["c2w"][:3, :3] @ ray
            to_point = X - rec["c2w"][:3, 3]
            cosang = d_world @ to_point / np.linalg.norm(d_world) / np.linalg.norm(to_point)
            angle = math.atan2(np.linalg.norm(np.cross(d_world, to_point)), d_world @ to_point)
            assert cosang > 0 and angle < 1e-9, (model, Xc_want, angle)
