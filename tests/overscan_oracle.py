"""TEST INFRASTRUCTURE ONLY: the H x W fp32 oracle extension (tests/nonsquare_oracle.py) rendered with overscan.

An H x W image off the decoder's size grid is rendered on an Hc x Wc canvas that holds it at canvas pixel
(top, left), with the camera of the H x W image, and then cropped.  Built from the oracle's own layer functions
through `nonsquare_oracle.view_stage_hw`; `oracle/` itself is unchanged."""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from oracle import renderformer_oracle as orc
from nonsquare_oracle import view_stage_hw


def camera_rays_overscan(fov_rad: torch.Tensor, H: int, W: int, Hc: int, Wc: int, top: int, left: int) -> torch.Tensor:
    """Camera-space rays of the Hc x Wc canvas [B, Hc, Wc, 3] whose window [top, top + H) x [left, left + W) holds the
    H x W image of `nonsquare_oracle.camera_rays_hw`: f = max(H, W) / 2 / tan(fov / 2), principal point at the
    window's centre (left + W/2, top + H/2) in canvas pixels, pixel centres at +0.5.  For a canvas equal to the image
    the same ops in the same order as camera_rays_hw."""
    px = torch.linspace(0.5, Wc - 0.5, Wc, dtype=fov_rad.dtype, device=fov_rad.device)
    py = torch.linspace(0.5, Hc - 0.5, Hc, dtype=fov_rad.dtype, device=fov_rad.device)
    x, y = torch.meshgrid(px, py, indexing="xy")
    cx, cy = left + W / 2, top + H / 2
    fl = max(H, W) / 2 / torch.tan(0.5 * fov_rad[..., 0, None, None])
    d = torch.stack([(x - cx) / fl, -(y - cy) / fl, -torch.ones_like(x).expand_as((x - cx) / fl)], dim=-1)
    return F.normalize(d, dim=-1, p=2)


@torch.no_grad()
def render_overscan(sd, cfg, triangles, texture, mask, vn, c2w, fov, resolution, canvas, offsets,
                    view_chunk: int = 4) -> torch.Tensor:
    """`nonsquare_oracle.render_hw` on the (Hc, Wc) canvas with the rays of camera_rays_overscan, cropped to the
    (H, W) window at `offsets` = (top, left) -> HDR [B, V, H, W, 3]."""
    (H, W), (Hc, Wc), (top, left) = resolution, canvas, offsets
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
            rays = camera_rays_overscan(fov[b, v0:v1] / 180.0 * math.pi, H, W, Hc, Wc, top, left)
            imgs.append(view_stage_hw(sd, cfg, seq[b:b + 1].expand(n, -1, -1), key_mask[b:b + 1].expand(n, -1),
                                      tri_cam, mask[b:b + 1].expand(n, -1), rays))
        out.append(torch.cat(imgs, dim=0))
    log_img = torch.stack(out, dim=0).permute(0, 1, 3, 4, 2)[:, :, top:top + H, left:left + W]  # [B,V,H,W,3]
    return torch.pow(10.0, log_img) - 1.0
