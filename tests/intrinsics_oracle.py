"""TEST INFRASTRUCTURE ONLY: the H x W fp32 oracle extension (tests/nonsquare_oracle.py) with per-view pinhole
intrinsics K = (fx, fy, cx, cy) in pixels of the H x W image, on an Hc x Wc canvas that holds the image at canvas pixel
(top, left) (canvas == image: top = left = 0), cropped like `overscan_oracle.render_overscan`.  Built from the
oracle's own layer functions through `nonsquare_oracle.view_stage_hw`; `oracle/` itself is unchanged."""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from oracle import renderformer_oracle as orc
from nonsquare_oracle import view_stage_hw

FIT_SIDES = {"auto": lambda H, W: max(H, W), "horizontal": lambda H, W: W, "vertical": lambda H, W: H}


def camera_rays_k(K: torch.Tensor, H: int, W: int, Hc: int, Wc: int, top: int, left: int) -> torch.Tensor:
    """Camera-space rays of the Hc x Wc canvas [B, Hc, Wc, 3] for intrinsics K [B, 4] of the H x W image at canvas
    pixel (top, left): the centre of image pixel (row i, column j) is (u, v) = (j + 0.5, i + 0.5) and its ray is
    normalize(((u - cx) / fx, -(v - cy) / fy, -1)).  Written like overscan_oracle.camera_rays_overscan, so for the
    centred fov-derived K it is the same ops on the same floats."""
    px = torch.linspace(0.5, Wc - 0.5, Wc, dtype=K.dtype, device=K.device)
    py = torch.linspace(0.5, Hc - 0.5, Hc, dtype=K.dtype, device=K.device)
    x, y = torch.meshgrid(px, py, indexing="xy")
    fx, fy, cx, cy = (K[:, i, None, None] for i in range(4))
    u, v = x - left, y - top
    d = torch.stack([(u - cx) / fx, -(v - cy) / fy, -torch.ones_like(x).expand_as((u - cx) / fx)], dim=-1)
    return F.normalize(d, dim=-1, p=2)


def intrinsics_from_fov_f64(fov_deg, H: int, W: int, fit: str = "auto") -> torch.Tensor:
    """float64 (f, f, W/2, H/2) [..., 4] of fov in degrees [...]: f = side / 2 / tan(fov / 2), side = max(H, W) (auto),
    W (horizontal) or H (vertical)."""
    fov = torch.as_tensor(fov_deg, dtype=torch.float64)
    f = FIT_SIDES[fit](H, W) / 2 / torch.tan(0.5 * fov / 180.0 * math.pi)
    return torch.stack([f, f, torch.full_like(f, W / 2), torch.full_like(f, H / 2)], dim=-1)


@torch.no_grad()
def render_k(sd, cfg, triangles, texture, mask, vn, c2w, K, resolution, canvas=None, offsets=(0, 0),
             view_chunk: int = 4) -> torch.Tensor:
    """`nonsquare_oracle.render_hw` with the rays of camera_rays_k for K [B, V, 4] on the (Hc, Wc) canvas (default:
    the image), cropped to the (H, W) window at `offsets` = (top, left) -> HDR [B, V, H, W, 3]."""
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
            rays = camera_rays_k(K[b, v0:v1].float(), H, W, Hc, Wc, top, left)
            imgs.append(view_stage_hw(sd, cfg, seq[b:b + 1].expand(n, -1, -1), key_mask[b:b + 1].expand(n, -1),
                                      tri_cam, mask[b:b + 1].expand(n, -1), rays))
        out.append(torch.cat(imgs, dim=0))
    log_img = torch.stack(out, dim=0).permute(0, 1, 3, 4, 2)[:, :, top:top + H, left:left + W]  # [B,V,H,W,3]
    return torch.pow(10.0, log_img) - 1.0
