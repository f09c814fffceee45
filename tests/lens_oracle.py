"""TEST INFRASTRUCTURE ONLY: a float64 lens-distorted camera for the oracle -- OpenCV's radial-tangential model
(k1, k2, p1, p2, k3, k4, k5, k6) and OpenCV's fisheye model (k1, k2, k3, k4), both forward models, their inverses
solved by Newton's method to ~1e-14, the ray of a pixel at any (u, v), the rays of an overscan canvas, and the oracle
render through them (built like `intrinsics_oracle.render_k`).  Written independently of renderformer_b200; `oracle/`
itself is unchanged.

Convention: intrinsics K = (fx, fy, cx, cy) in pixels of the H x W image, pixel centres at j + 0.5; a pixel's distorted
normalized coordinates are xd = (u - cx) / fx, yd = (v - cy) / fy in COLMAP / OpenCV camera axes (x right, y down,
z forward); the ray is returned in this project's camera axes (x right, y up, looking down -z)."""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from oracle import renderformer_oracle as orc
from nonsquare_oracle import view_stage_hw


def distort_opencv(x, y, D):
    """OpenCV's forward model: undistorted normalized (x, y) -> distorted (xd, yd); D [..., 8] broadcasts."""
    k1, k2, p1, p2, k3, k4, k5, k6 = D.unbind(-1)
    r2 = x * x + y * y
    g = (1 + k1 * r2 + k2 * r2 ** 2 + k3 * r2 ** 3) / (1 + k4 * r2 + k5 * r2 ** 2 + k6 * r2 ** 3)
    return x * g + 2 * p1 * x * y + p2 * (r2 + 2 * x * x), y * g + p1 * (r2 + 2 * y * y) + 2 * p2 * x * y


def _opencv_jacobian(x, y, D):
    k1, k2, p1, p2, k3, k4, k5, k6 = D.unbind(-1)
    r2 = x * x + y * y
    n = 1 + k1 * r2 + k2 * r2 ** 2 + k3 * r2 ** 3
    d = 1 + k4 * r2 + k5 * r2 ** 2 + k6 * r2 ** 3
    g = n / d
    dg = ((k1 + 2 * k2 * r2 + 3 * k3 * r2 ** 2) * d - n * (k4 + 2 * k5 * r2 + 3 * k6 * r2 ** 2)) / d ** 2  # dg / dr2
    a = g + 2 * x * x * dg + 2 * p1 * y + 6 * p2 * x       # d xd / d x
    b = 2 * x * y * dg + 2 * p1 * x + 2 * p2 * y           # d xd / d y = d yd / d x
    c = g + 2 * y * y * dg + 6 * p1 * y + 2 * p2 * x       # d yd / d y
    return a, b, c


def undistort_opencv(xd, yd, D, iters: int = 100):
    """(x, y) with distort_opencv(x, y, D) = (xd, yd): Newton's method from (xd, yd), to ~1e-14."""
    x, y = xd.clone(), yd.clone()
    for _ in range(iters):
        ex, ey = distort_opencv(x, y, D)
        ex, ey = ex - xd, ey - yd
        a, b, c = _opencv_jacobian(x, y, D)
        det = a * c - b * b
        sx, sy = (c * ex - b * ey) / det, (a * ey - b * ex) / det
        x, y = x - sx, y - sy
        if not bool(((sx.abs() + sy.abs()) > 1e-16).any()):
            break
    return x, y


def distort_fisheye(theta, D):
    """OpenCV's fisheye model: the angle theta from the optical axis -> the distorted radius theta_d; D [..., 4]."""
    k1, k2, k3, k4 = D.unbind(-1)
    t2 = theta * theta
    return theta * (1 + k1 * t2 + k2 * t2 ** 2 + k3 * t2 ** 3 + k4 * t2 ** 4)


def undistort_fisheye(rd, D, iters: int = 100):
    """theta with distort_fisheye(theta, D) = rd: 1-D Newton from theta = rd, to ~1e-14."""
    k1, k2, k3, k4 = D.unbind(-1)
    th = rd.clone()
    for _ in range(iters):
        t2 = th * th
        step = (distort_fisheye(th, D) - rd) / (1 + 3 * k1 * t2 + 5 * k2 * t2 ** 2 + 7 * k3 * t2 ** 3 + 9 * k4 * t2 ** 4)
        th = th - step
        if not bool((step.abs() > 1e-16).any()):
            break
    return th


def lens_rays(u, v, K, D, lens: str):
    """Camera-space unit rays [..., 3] of pixel positions (u, v) for intrinsics K [..., 4] and coefficients D of
    `lens` ("opencv": [..., 8], "fisheye": [..., 4]), all broadcasting against each other."""
    fx, fy, cx, cy = K.unbind(-1)
    xd, yd = (u - cx) / fx, (v - cy) / fy
    if lens == "opencv":
        x, y = undistort_opencv(xd, yd, D)
        return F.normalize(torch.stack([x, -y, -torch.ones_like(x)], dim=-1), dim=-1, p=2)
    rd = torch.sqrt(xd * xd + yd * yd)
    th = undistort_fisheye(rd, D)
    s = torch.where(rd > 0, torch.sin(th) / torch.where(rd > 0, rd, 1.0), 0.0)
    return torch.stack([s * xd, -s * yd, -torch.cos(th)], dim=-1)


def camera_rays_lens(K, D, lens: str, H: int, W: int, Hc: int, Wc: int, top: int, left: int) -> torch.Tensor:
    """Rays of the Hc x Wc canvas [B, Hc, Wc, 3] for K [B, 4] and D [B, n] of the H x W image at canvas pixel
    (top, left), the pixel grid built as intrinsics_oracle.camera_rays_k builds it."""
    px = torch.linspace(0.5, Wc - 0.5, Wc, dtype=K.dtype, device=K.device)
    py = torch.linspace(0.5, Hc - 0.5, Hc, dtype=K.dtype, device=K.device)
    x, y = torch.meshgrid(px, py, indexing="xy")
    return lens_rays(x - left, y - top, K[:, None, None, :], D[:, None, None, :].to(K.dtype), lens)


@torch.no_grad()
def render_lens(sd, cfg, triangles, texture, mask, vn, c2w, K, D, lens: str, resolution, canvas=None,
                offsets=(0, 0), view_chunk: int = 4) -> torch.Tensor:
    """`intrinsics_oracle.render_k` through the lens: rays of camera_rays_lens (float64, then fp32) for K [B, V, 4] and
    D [B, V, n] on the (Hc, Wc) canvas (default: the image), cropped to the (H, W) window at `offsets` = (top, left)
    -> HDR [B, V, H, W, 3]."""
    H, W = resolution
    Hc, Wc = canvas if canvas is not None else resolution
    top, left = offsets
    B, V = c2w.shape[:2]
    N = triangles.shape[1]
    tex = texture.clone()
    tex[:, :, -3:] = torch.log10(tex[:, :, -3:] + 1.0)
    tri9 = triangles.reshape(B, N, 9).float()
    seq, key_mask = orc.scene_stage(sd, cfg, tri9, tex.float(), mask, vn.reshape(B, N, 9).float())
    out = []
    for b in range(B):
        imgs = []
        for v0 in range(0, V, view_chunk):
            v1 = min(V, v0 + view_chunk)
            n = v1 - v0
            tri_cam = orc.to_camera_space(c2w[b, v0:v1], triangles[b:b + 1].expand(n, -1, -1, -1)).reshape(n, N, 9)
            rays = camera_rays_lens(K[b, v0:v1].double(), D[b, v0:v1].double(), lens, H, W, Hc, Wc, top, left).float()
            imgs.append(view_stage_hw(sd, cfg, seq[b:b + 1].expand(n, -1, -1), key_mask[b:b + 1].expand(n, -1),
                                      tri_cam, mask[b:b + 1].expand(n, -1), rays))
        out.append(torch.cat(imgs, dim=0))
    log_img = torch.stack(out, dim=0).permute(0, 1, 3, 4, 2)[:, :, top:top + H, left:left + W]  # [B,V,H,W,3]
    return torch.pow(10.0, log_img) - 1.0


# Test cameras: lens -> (model, coefficients, focal rule).  An opencv camera's focal length comes from a field of view
# across the longer side (degrees, one per view), a fisheye's from the angle theta that half the longer side reaches
# (radians, one per view), as an equidistant fisheye would.  "fisheye_wide" sees more than 100 degrees off the axis in
# the image corners.  Every one inverts on every canvas the tests use.
LENS_CASES = {
    "barrel": ("opencv", (-0.12, 0.02, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0), ("fov", (40.0, 55.0))),
    "pincushion": ("opencv", (0.1, 0.03, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0), ("fov", (40.0, 55.0))),
    "rational": ("opencv", (0.3, -0.05, 0.0, 0.0, 0.01, 0.45, -0.02, 0.01), ("fov", (45.0, 60.0))),
    "tangential": ("opencv", (0.0, 0.0, 0.012, -0.009, 0.0, 0.0, 0.0, 0.0), ("fov", (40.0, 55.0))),
    "fisheye_mild": ("fisheye", (0.03, -0.006, 0.001, -0.0002), ("theta", (0.9, 1.1))),
    "fisheye_wide": ("fisheye", (-0.01, 0.001, 0.0, 0.0), ("theta", (1.75, 1.8))),
    "fisheye_equidistant": ("fisheye", (0.0, 0.0, 0.0, 0.0), ("theta", (1.2, 1.5))),
}


def lens_case(name: str, H: int, W: int):
    """(lens, K float32 [V, 4], D float32 [V, n]) of a LENS_CASES camera for an H x W image: fy = 1.02 fx and the
    principal point a few pixels off the centre, as a calibration gives them."""
    lens, coeffs, (rule, vals) = LENS_CASES[name]
    side = max(H, W) / 2
    f = torch.tensor([side / math.tan(math.radians(a) / 2) if rule == "fov" else side / a for a in vals],
                     dtype=torch.float64)
    K = torch.stack([f, 1.02 * f, torch.full_like(f, W / 2 + 3.5), torch.full_like(f, H / 2 - 2.25)], dim=-1)
    D = torch.tensor([coeffs] * len(vals), dtype=torch.float64)
    return lens, K.float(), D.float()
