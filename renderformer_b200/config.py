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


# lens models of `distortion` -> the number of coefficients per view the ray kernel reads
LENS_COEFFS = {"opencv": 8, "fisheye": 4}


def view_camera(c2w, fov=None, intrinsics=None, distortion=None, lens: str = "opencv", canvas=None, window=None):
    """The camera of a render, as (kind, tensor): ("fov", fov), ("intrinsics", intrinsics), or for a lens-distorted
    camera (lens, intrinsics and coefficients [B, V, 4 + n]) with lens "opencv" (n = 8) or "fisheye" (n = 4).

    Exactly one of `fov` (degrees [B, V, 1]) and `intrinsics` must be given.  `intrinsics` is a [B, V, 4] tensor
    (fx, fy, cx, cy) in pixels of the returned H x W image, B and V matching c2w [B, V, 4, 4].  `distortion` (with
    `intrinsics` only) holds the lens coefficients per view: for lens "opencv" [B, V, 8] = (k1, k2, p1, p2, k3, k4, k5,
    k6), OpenCV's distCoeffs order, or its [B, V, 4] and [B, V, 5] prefixes (the missing coefficients are zero); for
    lens "fisheye" [B, V, 4] = (k1, k2, k3, k4) of OpenCV's fisheye model.  On the host the values are checked too:
    all finite, fx and fy > 0, and every pixel on the border of the canvas the model runs on (`canvas` = (Hc, Wc) and
    `window` = (h, w, top, left) or None, as `view_geometry` returns them; needed with `distortion`) must invert
    (`lens_check`).  A device tensor is not read back, so that the render path never waits for the device, and its
    values are the caller's responsibility.  Raises ValueError before anything is launched."""
    import torch
    if lens not in LENS_COEFFS:
        raise ValueError(f"lens must be one of {sorted(LENS_COEFFS)}, got {lens!r}")
    if (fov is None) == (intrinsics is None):
        raise ValueError("pass exactly one of fov and intrinsics")
    if distortion is not None and intrinsics is None:
        raise ValueError("distortion needs intrinsics: pass intrinsics=pipe.intrinsics_from_fov(fov, resolution) "
                         "in place of fov")
    if intrinsics is None:
        return "fov", fov
    if not isinstance(intrinsics, torch.Tensor):
        raise ValueError(f"intrinsics must be a torch.Tensor, got {type(intrinsics).__name__}")
    want = (*tuple(c2w.shape[:2]), 4)
    if tuple(intrinsics.shape) != want:
        raise ValueError(f"intrinsics must be [B, V, 4] = {list(want)} to match c2w, got {list(intrinsics.shape)}")
    if not intrinsics.is_floating_point():
        raise ValueError(f"intrinsics must be a floating-point tensor, got {intrinsics.dtype}")
    host = intrinsics.device.type == "cpu"
    if host:
        k = intrinsics.double()
        if not bool(torch.isfinite(k).all()):
            raise ValueError("intrinsics must be finite")
        if not bool((k[..., :2] > 0).all()):
            raise ValueError("intrinsics: fx and fy must be positive")
    if distortion is None:
        return "intrinsics", intrinsics
    if not isinstance(distortion, torch.Tensor):
        raise ValueError(f"distortion must be a torch.Tensor, got {type(distortion).__name__}")
    n = LENS_COEFFS[lens]
    sizes = (4, 5, 8) if lens == "opencv" else (4,)
    if distortion.dim() != 3 or tuple(distortion.shape[:2]) != want[:2] or distortion.shape[2] not in sizes:
        raise ValueError(f"distortion for lens {lens!r} must be [B, V, n] with B, V = {list(want[:2])} of c2w and "
                         f"n in {list(sizes)}, got {list(distortion.shape)}")
    if not distortion.is_floating_point():
        raise ValueError(f"distortion must be a floating-point tensor, got {distortion.dtype}")
    if distortion.device != intrinsics.device:
        raise ValueError(f"distortion ({distortion.device}) and intrinsics ({intrinsics.device}) must be on one device")
    if host:
        if not bool(torch.isfinite(distortion).all()):
            raise ValueError("distortion must be finite")
        if canvas is None:
            raise ValueError("view_camera: checking host distortion coefficients needs the canvas")
        lens_check(intrinsics.reshape(-1, 4).double().numpy(), distortion.reshape(-1, distortion.shape[2]).double()
                   .numpy(), lens, canvas, window, views=want[:2])
    pad = torch.zeros((*want[:2], n - distortion.shape[2]), dtype=torch.float32, device=distortion.device)
    return lens, torch.cat([intrinsics.float(), distortion.float(), pad], dim=-1)


def camera_kwargs(kind: str, cam) -> dict:
    """The keywords of `render` that give the camera `view_camera` returned as (kind, cam)."""
    if kind in LENS_COEFFS:
        return {"intrinsics": cam[..., :4], "distortion": cam[..., 4:], "lens": kind}
    return {kind: cam}


def lens_check(K, D, lens: str, canvas, window=None, views=None) -> None:
    """Raise ValueError unless every view's lens inverts on the border of the canvas, in float64 (numpy).

    K [n, 4] intrinsics and D [n, m] coefficients of n views (`views`, the (B, V) shape of the n views, names them in
    the message), `canvas` = (Hc, Wc), `window` = (h, w, top, left) or None as `view_camera` takes them.  The canvas,
    not the window, is checked: the model sees the overscan border too.  Each border pixel's (xd, yd) must be solved
    by Newton's method from the start the ray kernel uses, and
      opencv:  the Jacobian determinant and the denominator 1 + k4 r2 + k5 r2^2 + k6 r2^3 must stay positive on the
               segment from the optical axis to the solution (the lens must not fold back inside the canvas);
      fisheye: theta must stay below pi and d theta_d / d theta positive on [0, theta].
    A pixel farther out than the fold has no solution, so a lens that folds inside the canvas is rejected."""
    import numpy as np
    Hc, Wc = canvas
    top, left = (0, 0) if window is None else window[2:]
    px = np.concatenate([np.arange(Wc), np.arange(Wc), np.zeros(Hc), np.full(Hc, Wc - 1)])
    py = np.concatenate([np.zeros(Wc), np.full(Wc, Hc - 1), np.arange(Hc), np.arange(Hc)])
    fx, fy, cx, cy = (K[:, i, None] for i in range(4))
    xd, yd = (px - left + 0.5 - cx) / fx, (py - top + 0.5 - cy) / fy  # [n views, border pixels]
    with np.errstate(all="ignore"):
        if lens == "opencv":
            c = [col[:, None] for col in np.concatenate([D, np.zeros((len(D), 8 - D.shape[1]))], axis=1).T]
            x, y = xd.copy(), yd.copy()
            for _ in range(100):
                ex, ey, jxx, jyy, jxy, _ = _opencv_model(x, y, c)
                det = jxx * jyy - jxy * jxy
                sx, sy = (jyy * (ex - xd) - jxy * (ey - yd)) / det, (jxx * (ey - yd) - jxy * (ex - xd)) / det
                x, y = x - sx, y - sy
                if not np.nanmax(np.abs(sx) + np.abs(sy), initial=0) > 1e-15:
                    break
            ex, ey = _opencv_model(x, y, c)[:2]
            ok = (np.abs(ex - xd) <= 1e-9 * (1 + np.abs(xd))) & (np.abs(ey - yd) <= 1e-9 * (1 + np.abs(yd)))
            s = np.linspace(0, 1, 9)[1:]  # the segment from the optical axis to the solution
            _, _, jxx, jyy, jxy, den = _opencv_model(x[..., None] * s, y[..., None] * s, [a[..., None] for a in c])
            ok &= ((jxx * jyy - jxy * jxy > 0) & (den > 0)).all(axis=-1)
        else:
            k1, k2, k3, k4 = (D[:, i, None] for i in range(4))
            rd = np.hypot(xd, yd)
            th = rd.copy()
            for _ in range(100):
                t2 = th * th
                step = (th * (1 + t2 * (k1 + t2 * (k2 + t2 * (k3 + t2 * k4)))) - rd) / \
                    (1 + t2 * (3 * k1 + t2 * (5 * k2 + t2 * (7 * k3 + t2 * 9 * k4))))
                th = th - step
                if not np.nanmax(np.abs(step), initial=0) > 1e-15:
                    break
            t2 = th * th
            ok = np.abs(th * (1 + t2 * (k1 + t2 * (k2 + t2 * (k3 + t2 * k4)))) - rd) <= 1e-9 * (1 + rd)
            ok &= (th >= 0) & (th < np.pi)
            # d theta_d / d theta on [0, theta] for the largest theta of each view
            t2 = (np.nanmax(np.where(ok, th, 0), axis=1, keepdims=True) * np.linspace(0, 1, 1025)[1:]) ** 2
            ok &= (1 + t2 * (3 * k1 + t2 * (5 * k2 + t2 * (7 * k3 + t2 * 9 * k4))) > 0).all(axis=-1, keepdims=True)
    bad = np.argwhere(~ok)
    if len(bad):
        i, j = bad[0]
        view = f"view {i}" if views is None else f"view (b, v) = {tuple(int(a) for a in np.unravel_index(i, views))}"
        raise ValueError(f"distortion: the {lens} lens of {view} does not invert at canvas pixel (row {int(py[j])}, "
                         f"column {int(px[j])}) of the {Hc}x{Wc} canvas: the lens folds back (or, fisheye, reaches "
                         "theta = pi) inside the canvas")


def _opencv_model(x, y, c):
    """OpenCV's forward lens model at undistorted (x, y), coefficients c = (k1, k2, p1, p2, k3, k4, k5, k6):
    (xd, yd, dxd/dx, dyd/dy, dxd/dy = dyd/dx, denominator)."""
    k1, k2, p1, p2, k3, k4, k5, k6 = c
    x2, y2, xy = x * x, y * y, x * y
    r2 = x2 + y2
    num = 1 + r2 * (k1 + r2 * (k2 + r2 * k3))
    den = 1 + r2 * (k4 + r2 * (k5 + r2 * k6))
    g = num / den
    gp = ((k1 + r2 * (2 * k2 + r2 * 3 * k3)) * den - num * (k4 + r2 * (2 * k5 + r2 * 3 * k6))) / (den * den)
    return (x * g + 2 * p1 * xy + p2 * (r2 + 2 * x2), y * g + p1 * (r2 + 2 * y2) + 2 * p2 * xy,
            g + 2 * x2 * gp + 2 * p1 * y + 6 * p2 * x, g + 2 * y2 * gp + 6 * p1 * y + 2 * p2 * x,
            2 * xy * gp + 2 * p1 * x + 2 * p2 * y, den)
