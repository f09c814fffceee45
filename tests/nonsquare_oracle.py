"""TEST INFRASTRUCTURE ONLY: the fp32 oracle (oracle/renderformer_oracle.py) extended to H x W images.

The oracle itself stays square (its stored goldens pin it bit-exactly); this module adds the non-square camera and
restates `view_stage` / `render` with the patch grid taken from both sides of the ray map, built from the oracle's
own layer functions.  For H == W every function here is the oracle's, op for op (tests/test_nonsquare.py checks
`torch.equal` against it)."""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn.functional as F

from oracle import renderformer_oracle as orc


def camera_rays_hw(fov_rad: torch.Tensor, H: int, W: int) -> torch.Tensor:
    """Camera-space pinhole rays of an H x W image.  fov [B,1] -> [B,H,W,3].  Square pixels, principal point at
    the image centre, pixel centres at +0.5, fov spanning the LONGER side (Blender's "Auto" sensor fit):
    f = max(H, W) / 2 / tan(fov / 2).  For H == W the same ops in the same order as orc.camera_rays."""
    px = torch.linspace(0.5, W - 0.5, W, dtype=fov_rad.dtype, device=fov_rad.device)
    py = torch.linspace(0.5, H - 0.5, H, dtype=fov_rad.dtype, device=fov_rad.device)
    x, y = torch.meshgrid(px, py, indexing="xy")
    cx, cy = W / 2, H / 2
    fl = max(H, W) / 2 / torch.tan(0.5 * fov_rad[..., 0, None, None])
    d = torch.stack([(x - cx) / fl, -(y - cy) / fl, -torch.ones_like(x).expand_as((x - cx) / fl)], dim=-1)
    return F.normalize(d, dim=-1, p=2)


def view_stage_hw(sd, cfg, seq, key_mask, tri9_cam, mask, rays_d, taps: Optional[dict] = None):
    """orc.view_stage (models/view_transformer.py:88-127) on rays_d [BV,H,W,3]: Hp = H / 8, Wp = W / 8."""
    p = "view_transformer."
    BV = rays_d.shape[0]
    P = cfg.patch_size
    Hp, Wp = rays_d.shape[1] // P, rays_d.shape[2] // P
    dv, heads = cfg.view_transformer_latent_dim, cfg.view_transformer_n_heads
    rm = orc.nerf_encode(rays_d, cfg.vdir_num_freqs)
    # 'b (h1 p1) (w1 p2) c -> b (h1 w1) (c p1 p2)'   view_transformer.py:105
    tok = rm.view(BV, Hp, P, Wp, P, -1).permute(0, 1, 3, 5, 2, 4).reshape(BV, Hp * Wp, -1)
    x = sd[p + "ray_map_patch_token"] + orc.rms(
        F.linear(tok, sd[p + "ray_map_encoder.weight"], sd[p + "ray_map_encoder.bias"]),
        sd[p + "ray_map_encoder_norm.weight"], None)
    pos_k, _ = orc.centroid_positions(tri9_cam, mask, cfg.num_register_tokens)
    fr = sd[p + "transformer.rope_emb.freqs"]
    hd = dv // heads
    q_cs = orc.rope_tables(torch.zeros((BV, Hp * Wp, 9), device=x.device), fr, hd)  # camera origin = 0
    k_cs = orc.rope_tables(pos_k, fr, hd)
    out_layers = (list(range(cfg.view_transformer_n_layers - 4, cfg.view_transformer_n_layers))
                  if cfg.dpt_out_layers is None else list(cfg.dpt_out_layers))
    feats = []
    for i in range(cfg.view_transformer_n_layers):
        x = orc.decoder_layer(sd, p + f"transformer.layers.{i}.", x, seq, heads, key_mask, q_cs, k_cs,
                              cfg.view_transformer_use_swin_attn, 0 if i % 2 == 0 else 4, Hp, Wp)
        if i in out_layers:
            feats.append(x)
    if taps is not None:
        taps["dec_feats"] = [f.clone() for f in feats]
    img = orc.dpt_head(sd, p + "out_dpt.", feats, Hp, Wp, P)
    return F.elu(img, alpha=1e-3)  # view_transformer.py:86,122


@torch.no_grad()
def render_hw(sd, cfg, triangles, texture, mask, vn, c2w, fov, resolution, view_chunk: int = 4) -> torch.Tensor:
    """orc.render (pipelines/rendering_pipeline.py:28-125, fp32) at resolution (H, W) -> HDR [B, V, H, W, 3]."""
    H, W = resolution
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
            rays = camera_rays_hw(fov[b, v0:v1] / 180.0 * math.pi, H, W)
            imgs.append(view_stage_hw(sd, cfg, seq[b:b + 1].expand(n, -1, -1), key_mask[b:b + 1].expand(n, -1),
                                      tri_cam, mask[b:b + 1].expand(n, -1), rays))
        out.append(torch.cat(imgs, dim=0))
    log_img = torch.stack(out, dim=0).permute(0, 1, 3, 4, 2)  # [B,V,H,W,3]
    return torch.pow(10.0, log_img) - 1.0
