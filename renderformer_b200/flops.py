"""Algorithmic FLOP counts (2 x MAC) of the forward pass, SURVEY §8(d).

These formulas reproduce torch's FlopCounterMode on the reference; the hoisted decoder K/V
projections are counted once per scene (the reference pays them per view)."""
from __future__ import annotations

from .config import RenderFormerConfig, overscan_grid


def _patch_grid(resolution):
    """(H/8, W/8) of an int (square) or (H, W) resolution."""
    h, w = tuple(resolution) if isinstance(resolution, (tuple, list)) else (resolution, resolution)
    return h // 8, w // 8


def scene_flops(cfg: RenderFormerConfig, n_tris: int) -> float:
    d, f, L = cfg.latent_dim, cfg.dim_feedforward, cfg.num_layers
    nt = n_tris + cfg.num_register_tokens
    tex_in = cfg.texture_channels * cfg.texture_encode_patch_size ** 2
    vn_in = 9 + 18 * cfg.vn_pe_num_freqs
    tokens = 2.0 * n_tris * tex_in * d + 2.0 * n_tris * vn_in * d
    layer = 8.0 * nt * d * d + 4.0 * nt * nt * d + 6.0 * nt * d * f
    hoisted_kv = cfg.view_transformer_n_layers * 4.0 * nt * d * cfg.view_transformer_latent_dim
    return tokens + L * layer + hoisted_kv


def dpt_flops(cfg: RenderFormerConfig, resolution) -> float:
    dv, F = cfg.view_transformer_latent_dim, cfg.dpt_features
    C = cfg.dpt_out_channels
    hp, wp = _patch_grid(resolution)
    p = hp * wp
    fl = sum(2.0 * p * dv * c for c in C)                      # 1x1 projects
    fl += 2.0 * p * C[0] * C[0] * 16 + 2.0 * p * C[1] * C[1] * 4   # ConvT k4s4, k2s2
    fl += 2.0 * (p / 4) * 9 * C[3] * C[3]                          # 3x3 stride 2
    sizes = [16 * p, 4 * p, p, p / 4]
    fl += sum(2.0 * s * 9 * c * F for s, c in zip(sizes, C))       # layerN_rn
    conv = lambda s: 2.0 * s * 9 * F * F
    fl += 2 * conv(sizes[3]) + 2.0 * sizes[2] * F * F              # refinenet4 (+ out_conv at output res)
    fl += 4 * conv(sizes[2]) + 2.0 * sizes[1] * F * F
    fl += 4 * conv(sizes[1]) + 2.0 * sizes[0] * F * F
    fl += 4 * conv(sizes[0]) + 2.0 * 64 * p * F * F
    fl += 2.0 * 64 * p * 9 * F * (F // 2) + 2.0 * 64 * p * 9 * (F // 2) * 32 + 2.0 * 64 * p * 32 * 3
    return fl


def view_flops(cfg: RenderFormerConfig, n_tris: int, resolution, overscan: bool = False) -> float:
    """`resolution`: an int (square) or (H, W).  With `overscan` (any size, `render(..., overscan=True)`) a view
    costs the FLOPs of its canvas (config.overscan_grid): the model runs on the whole canvas, the crop is free."""
    if overscan:
        resolution = overscan_grid(cfg, resolution)[1]
    dv, fv, Lv = cfg.view_transformer_latent_dim, cfg.view_transformer_ffn_hidden_dim, cfg.view_transformer_n_layers
    nt = n_tris + cfg.num_register_tokens
    hp, wp = _patch_grid(resolution)
    nr = hp * wp
    self_keys = 64 if cfg.view_transformer_use_swin_attn else nr
    layer = 12.0 * nr * dv * dv + 4.0 * nr * nt * dv + 4.0 * nr * self_keys * dv + 6.0 * nr * dv * fv
    return 2.0 * nr * 192 * dv + Lv * layer + dpt_flops(cfg, resolution)


def job_flops(cfg: RenderFormerConfig, n_tris: int, resolution, n_scenes: int, n_views: int,
              overscan: bool = False) -> float:
    return n_scenes * (scene_flops(cfg, n_tris) + n_views * view_flops(cfg, n_tris, resolution, overscan))
