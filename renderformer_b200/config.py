"""Model hyper-parameters of the RenderFormer architecture.

Field names and defaults mirror the reference's flat config.json contract
(reference: renderformer/models/config.py:5-92) so that a reference checkpoint directory
(`config.json` + `model.safetensors`) loads unchanged.  Defaults are RenderFormer-V1-Base.
"""
from __future__ import annotations

import json
import numbers
import os
from dataclasses import asdict, dataclass, field, fields
from typing import List, Optional, Tuple

_CONFIG_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "configs")


@dataclass(frozen=True)
class RenderFormerConfig:
    # view-independent (triangle) transformer
    latent_dim: int = 768
    num_layers: int = 12
    num_heads: int = 6
    dim_feedforward: int = 3072
    num_register_tokens: int = 16
    dropout: float = 0.0
    activation: str = "swiglu"
    norm_type: str = "rms_norm"
    norm_first: bool = True
    view_indep_qk_norm: bool = True
    qk_norm: bool = True
    bias: bool = False
    # positional encoding
    pe_type: str = "rope"
    rope_type: str = "triangle"
    rope_double_max_freq: bool = False
    vertex_pe_num_freqs: int = 12
    # token encoders
    use_vn_encoder: bool = True
    vn_pe_num_freqs: int = 6
    vn_encoder_norm_type: str = "rms_norm"
    texture_encode_patch_size: int = 32
    texture_channels: int = 13
    texture_encoder_norm_type: str = "rms_norm"
    # view-dependent (ray bundle) transformer
    view_transformer_latent_dim: int = 768
    view_transformer_ffn_hidden_dim: int = 3072
    view_transformer_n_heads: int = 6
    view_transformer_n_layers: int = 6
    view_transformer_include_self_attn: bool = True
    view_transformer_use_swin_attn: bool = False
    vdir_pe_type: str = "nerf"
    vdir_num_freqs: int = 0
    patch_size: int = 8
    include_alpha: bool = False
    use_dpt_decoder: bool = True
    dpt_features: int = 128
    dpt_out_channels: List[int] = field(default_factory=lambda: [96, 192, 384, 768])
    dpt_out_layers: Optional[List[int]] = None
    turn_to_cam_coord: bool = True
    use_ldr: bool = False

    def get(self, key, default=None):
        return getattr(self, key, default)

    def to_dict(self) -> dict:
        return asdict(self)

    @classmethod
    def from_dict(cls, d: dict) -> "RenderFormerConfig":
        known = {f.name for f in fields(cls)}
        return cls(**{k: v for k, v in d.items() if k in known})

    @classmethod
    def from_json(cls, path: str) -> "RenderFormerConfig":
        with open(path) as f:
            return cls.from_dict(json.load(f))

    @classmethod
    def named(cls, name: str) -> "RenderFormerConfig":
        """Pinned configs shipped with the package: v1_base, v1_1_swin_large, tiny_swin, tiny_full."""
        return cls.from_json(os.path.join(_CONFIG_DIR, f"{name}.json"))

    # ---- derived quantities -------------------------------------------------
    @property
    def head_dim(self) -> int:
        return self.latent_dim // self.num_heads

    @property
    def view_head_dim(self) -> int:
        return self.view_transformer_latent_dim // self.view_transformer_n_heads

    @property
    def view_rope_dim(self) -> int:
        # reference: renderformer/models/view_transformer.py:34
        return min(self.vertex_pe_num_freqs, self.view_head_dim // 18 * 2)

    @property
    def out_layers(self) -> List[int]:
        # reference: renderformer/models/view_transformer.py:85
        n = self.view_transformer_n_layers
        return list(range(n - 4, n)) if self.dpt_out_layers is None else list(self.dpt_out_layers)

    def check_supported(self) -> None:
        """Branches the released configs never exercise are rejected, not emulated (SURVEY §8a)."""
        bad = []
        if self.pe_type != "rope" or self.rope_type != "triangle" or self.rope_double_max_freq:
            bad.append("pe_type/rope_type")
        if self.activation != "swiglu" or self.norm_type != "rms_norm" or not self.norm_first:
            bad.append("activation/norm")
        if self.bias or not (self.qk_norm and self.view_indep_qk_norm):
            bad.append("bias/qk_norm")
        if not self.use_vn_encoder or self.vn_encoder_norm_type != "rms_norm":
            bad.append("vn encoder")
        if self.texture_encoder_norm_type != "rms_norm" or self.texture_encode_patch_size != 32:
            bad.append("texture encoder")
        if self.vdir_num_freqs != 0 or self.patch_size != 8 or self.include_alpha:
            bad.append("view-direction encoding / patch")
        if not self.use_dpt_decoder or not self.turn_to_cam_coord or self.use_ldr:
            bad.append("decoder head / coordinate frame")
        if not self.view_transformer_include_self_attn:
            bad.append("view self-attention")
        if self.head_dim != 128 or self.view_head_dim != 128:
            bad.append("head_dim != 128")
        if self.dropout != 0.0:
            bad.append("dropout")
        if self.dpt_features != 128 or len(self.dpt_out_channels) != 4:
            bad.append("dpt_features != 128")
        # shape constraints of the kernels, spelled out here instead of an opaque 'rfb_gemm failed: bad argument'
        if len(self.out_layers) != 4 or self.view_transformer_n_layers < 4:
            bad.append("the DPT head taps exactly 4 decoder layers (dpt_out_layers)")
        if (self.view_transformer_n_layers * self.view_transformer_latent_dim) % 256 != 0:
            bad.append("view_transformer_n_layers * view_transformer_latent_dim must be a multiple of 256 "
                       "(the hoisted K | V^T of all layers leave one GEMM in 256-column tiles)")
        if 9 * (self.vertex_pe_num_freqs // 2) > 64 or 9 * (self.view_rope_dim // 2) > 64:
            bad.append("9 * rope_dim / 2 must fit the 64 rotation pairs of a 128-wide head")
        if self.num_register_tokens > 32:
            bad.append("num_register_tokens <= 32")
        if any(c % 32 for c in self.dpt_out_channels):
            bad.append("dpt_out_channels must be multiples of 32")
        if bad:
            raise NotImplementedError("unsupported RenderFormerConfig options: " + ", ".join(bad))


def _size_pair(resolution) -> Tuple[int, int]:
    """(height, width) of an int (square) or a (height, width) pair of positive ints; ValueError otherwise."""
    if isinstance(resolution, (tuple, list)):
        if len(resolution) != 2:
            raise ValueError(f"resolution must be an int or a (height, width) pair, got {resolution!r}")
        hw = tuple(resolution)
    else:
        hw = (resolution, resolution)
    if not all(isinstance(s, numbers.Integral) and not isinstance(s, bool) and s > 0 for s in hw):
        raise ValueError(f"resolution must be a positive int or a (height, width) pair of positive ints, got {resolution!r}")
    return int(hw[0]), int(hw[1])


def view_grid(cfg: RenderFormerConfig, resolution) -> Tuple[int, int]:
    """(height, width) in pixels of the images `resolution` asks for: an int is a square image, a pair is
    (height, width).  Sides must be multiples of 64 for the swin decoder (8x8 windows of 8x8-pixel patches, the
    reference's own constraint, SURVEY §8b) and multiples of the 8-pixel patch for full attention.  Raises
    ValueError before anything is launched."""
    H, W = _size_pair(resolution)
    if cfg.view_transformer_use_swin_attn and (H % 64 or W % 64):
        raise ValueError(f"image height and width must be multiples of 64 for swin attention, got {H}x{W}")
    if H % cfg.patch_size or W % cfg.patch_size:
        raise ValueError(f"image height and width must be multiples of the {cfg.patch_size}-pixel patch size, "
                         f"got {H}x{W}")
    return H, W


def overscan_grid(cfg: RenderFormerConfig, resolution) -> Tuple[Tuple[int, int], Tuple[int, int], Tuple[int, int]]:
    """Overscan geometry of an image of ANY positive size: ((H, W), (Hc, Wc), (top, left)).

    The model runs on a canvas Hc x Wc whose sides are H, W rounded up to the grid of `view_grid` (64 for swin,
    the 8-pixel patch for full attention); the requested H x W window sits at canvas pixel (top, left) =
    ((Hc - H) // 2, (Wc - W) // 2).  The camera is the one of the requested image (f from max(H, W), principal
    point at the window's centre), so every returned pixel is the model's output for a real H x W pinhole image;
    only the window is stored.  A size already on the grid is its own canvas.  Validates like `view_grid` and
    raises ValueError before anything is launched."""
    H, W = _size_pair(resolution)
    m = 64 if cfg.view_transformer_use_swin_attn else cfg.patch_size
    Hc, Wc = -(-H // m) * m, -(-W // m) * m
    return (H, W), (Hc, Wc), ((Hc - H) // 2, (Wc - W) // 2)


def view_camera(c2w, fov=None, intrinsics=None):
    """The camera of a render, as (keyword, tensor): ("fov", fov) or ("intrinsics", intrinsics).

    Exactly one of `fov` (degrees [B, V, 1]) and `intrinsics` must be given.  `intrinsics` is a [B, V, 4] tensor
    (fx, fy, cx, cy) in pixels of the returned H x W image, B and V matching c2w [B, V, 4, 4].  On the host its
    values are checked too (all finite, fx and fy > 0); a device tensor is not read back, so that the render path
    never waits for the device, and its values are the caller's responsibility.  Raises ValueError before anything
    is launched."""
    import torch
    if (fov is None) == (intrinsics is None):
        raise ValueError("pass exactly one of fov and intrinsics")
    if intrinsics is None:
        return "fov", fov
    if not isinstance(intrinsics, torch.Tensor):
        raise ValueError(f"intrinsics must be a torch.Tensor, got {type(intrinsics).__name__}")
    want = (*tuple(c2w.shape[:2]), 4)
    if tuple(intrinsics.shape) != want:
        raise ValueError(f"intrinsics must be [B, V, 4] = {list(want)} to match c2w, got {list(intrinsics.shape)}")
    if not intrinsics.is_floating_point():
        raise ValueError(f"intrinsics must be a floating-point tensor, got {intrinsics.dtype}")
    if intrinsics.device.type == "cpu":
        k = intrinsics.double()
        if not bool(torch.isfinite(k).all()):
            raise ValueError("intrinsics must be finite")
        if not bool((k[..., :2] > 0).all()):
            raise ValueError("intrinsics: fx and fy must be positive")
    return "intrinsics", intrinsics
