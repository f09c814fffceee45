"""Torch-tensor front-ends of the C-ABI kernels (pointer + shape marshalling only, no math).

Every function launches on the current CUDA stream and writes into caller-provided (or
freshly `torch.empty`-allocated) buffers.  dtype mapping: fp32 <-> RFB_F32, bf16 <-> RFB_BF16,
fp16 <-> RFB_F16.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import lib as L

_DT = {torch.float32: L.F32, torch.bfloat16: L.BF16, torch.float16: L.F16}


# Optional per-launch timing (bench.py's roofline): a list that receives
# (kernel family, algorithmic flops, start event, end event) for the tensor-core launches.
PROFILE = None


# Device every launch is bound to.  The C launchers run on the CUDA context's *current* device with
# the stream they are handed, so both must belong to the tensors' device: `_need_cuda` records the
# device of the operands, `_stream` returns that device's current stream and `_timed` makes it the
# current device around the launch (a model on cuda:1 while cuda:0 is current must not launch on
# GPU0 against GPU1 pointers -- ADVICE r01).
_DEV = [None]


def _timed(kind: str, flops: float, launch, tag: str = ""):
    dev = _DEV[0]
    if dev is not None and dev.index is not None and dev.index != torch.cuda.current_device():
        with torch.cuda.device(dev):
            return _timed_on_device(kind, flops, launch, tag)
    return _timed_on_device(kind, flops, launch, tag)


def _timed_on_device(kind: str, flops: float, launch, tag: str):
    if PROFILE is None:
        return launch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(torch.cuda.current_stream())
    rc = launch()
    e1.record(torch.cuda.current_stream())
    PROFILE.append((kind, flops, e0, e1, tag))
    return rc


def _stream() -> int:
    return torch.cuda.current_stream(_DEV[0]).cuda_stream


def _p(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need_cuda(*ts):
    dev = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise L.RfbError("renderformer_b200 kernels need CUDA tensors (there is no CPU fallback)")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise L.RfbError(f"operands live on different devices ({dev} vs {t.device})")
    _DEV[0] = dev


def gemm(A: torch.Tensor, W: torch.Tensor, out: Optional[torch.Tensor] = None, *, M=None, N=None, K=None,
         bias=None, res1=None, res2=None, out_act=None, row_map=None, epi=L.EPI_STORE, out_dtype=None,
         conv=None, w2=None, b2=None, lda=None, ldw=None, ldo=None, ldres=None, bn=0,
         in_sumsq=None, in_rscale=None, scale_dim=0, norm_dim=0, norm_eps=1e-6, out_rscale=None, out_sumsq=None,
         out16=None, col_mul=None, aux_row_map=None, vt_out=None, vt_split=0, vt_rows_per_batch=0,
         crop=None) -> torch.Tensor:
    """out[M,N] = A[M,K] @ W[N,K]^T with fused epilogue.  `conv=(B,H,W,Cin)` switches A to NHWC 3x3
    implicit GEMM.  Shapes default to the tensors' 2-D shapes.  `crop=(h, w, top, left)` (conv with a final
    epilogue): only that window of the conv image is stored, as out [B, h, w, 3]."""
    _need_cuda(A, W)
    lib = L.load()
    a = L.GemmArgs()
    if conv is not None:
        Bc, Hc, Wc, Cin = conv
        a.a_mode, a.B, a.H, a.Wd, a.Cin = L.A_CONV3X3, Bc, Hc, Wc, Cin
        M = Bc * Hc * Wc if M is None else M
        K = 9 * Cin if K is None else K
        lda = Cin
    else:
        M = A.shape[0] if M is None else M
        K = A.shape[-1] if K is None else K
        lda = A.stride(0) if lda is None else lda
    N = W.shape[0] if N is None else N
    ldw = W.stride(0) if ldw is None else ldw
    a.M, a.N, a.K, a.A, a.lda, a.W, a.ldw = M, N, K, A.data_ptr(), lda, W.data_ptr(), ldw
    a.dtype = _DT[A.dtype]
    assert W.dtype == A.dtype, "operand dtypes differ"
    a.epi = epi
    if out is None and out_act is None and out16 is None:
        ncols = N // 2 if epi == L.EPI_SWIGLU else (3 if epi in (L.EPI_FINAL, L.EPI_FINAL_RAW) else N)
        rows = M if crop is None else conv[0] * crop[0] * crop[1]
        out = torch.empty((rows, ncols), dtype=out_dtype or torch.float32, device=A.device)
    ref = out if out is not None else out_act
    a.out, a.out_act = _p(out), _p(out_act)
    if ref is not None:
        a.out_dtype = _DT[ref.dtype]
        a.ldo = (ref.stride(0) if ref.dim() == 2 else ref.shape[-1]) if ldo is None else ldo
    else:
        a.out_dtype, a.ldo = L.F32, _rup8(N)
    if in_sumsq is not None:  # [rows, parts] partial sums of squares (all parts are summed)
        a.in_sumsq, a.in_sumsq_ld, a.in_sumsq_parts = in_sumsq.data_ptr(), in_sumsq.stride(0), in_sumsq.shape[1]
        a.norm_dim, a.norm_eps = norm_dim, norm_eps
    if in_rscale is not None:
        a.in_rscale, a.scale_dim = in_rscale.data_ptr(), scale_dim
    a.out_rscale = _p(out_rscale)
    if out_sumsq is not None:  # [rows, >= N/128]
        a.out_sumsq, a.out_sumsq_ld = out_sumsq.data_ptr(), out_sumsq.stride(0)
    if out16 is not None:
        a.out16, a.out16_dtype, a.ld16 = out16.data_ptr(), _DT[out16.dtype], out16.stride(0)
    a.col_mul, a.aux_row_map = _p(col_mul), _p(aux_row_map)
    if vt_out is not None:  # [dims, rows] or [batch, dims, rows_per_batch]: transposed V part (columns >= vt_split)
        a.vt_out, a.vt_dtype, a.vt_split = vt_out.data_ptr(), _DT[vt_out.dtype], vt_split
        a.vt_ld = vt_out.stride(-2)
        a.vt_rows_per_batch = vt_rows_per_batch
        a.vt_batch_stride = vt_out.stride(0) if vt_out.dim() == 3 else 0
    a.bias = _p(bias)
    if res1 is not None:
        a.res1, a.res_dtype = res1.data_ptr(), _DT[res1.dtype]
        a.ldres = (res1.stride(0) if res1.dim() == 2 else res1.shape[-1]) if ldres is None else ldres
    if res2 is not None:
        a.res2 = res2.data_ptr()
    a.row_map = _p(row_map)
    a.w2, a.b2 = _p(w2), _p(b2)
    a.bn_override = bn
    if crop is not None:
        a.crop_h, a.crop_w, a.crop_top, a.crop_left = crop
    tag = f"M={M} N={N} K={K} epi={epi} conv={int(conv is not None)} out={a.out_dtype} res={int(res1 is not None)}"
    L.check(_timed("gemm", 2.0 * M * N * K, lambda: lib.rfb_gemm(C.byref(a), _stream()), tag), "rfb_gemm")
    return out if out is not None else (out_act if out_act is not None else out16)


def _rup8(n: int) -> int:
    return (n + 7) // 8 * 8


def attention(Q, K, Vt, O, *, B, H, Nq, Nk, ldq, ldk, ldvt, ldo, q_bs=0, k_bs=0, vt_bs=0, o_bs=0,
              mask_bits=None, mask_bs=0, mode=0, group_id=None, group_period=0, scale=None,
              q_sumsq=None, k_sumsq=None, sumsq_ld=1, sumsq_parts=1, norm_dim=0, norm_eps=1e-6,
              kv_split_tiles=0, split_ws=None):
    """`kv_split_tiles` > 0 (mode 0): key chunks of that many 128-key tiles on separate CTAs + an ordered merge;
    `split_ws` = float32 scratch of at least `attention_ws_elems(...)` elements."""
    _need_cuda(Q, K, Vt, O)
    lib = L.load()
    a = L.AttnArgs()
    if kv_split_tiles > 0 and attention_ws_elems(B, H, Nq, Nk, kv_split_tiles) > 0:
        if split_ws is None or split_ws.dtype != torch.float32 or not split_ws.is_contiguous():
            raise L.RfbError("key-split attention needs a contiguous float32 scratch tensor (split_ws)")
        _need_cuda(split_ws)
        a.kv_split_tiles, a.split_ws, a.split_ws_bytes = kv_split_tiles, split_ws.data_ptr(), split_ws.numel() * 4
    a.B, a.H, a.Nq, a.Nk = B, H, Nq, Nk
    a.Q, a.ldq, a.q_batch_stride = Q.data_ptr(), ldq, q_bs
    a.K, a.ldk, a.k_batch_stride = K.data_ptr(), ldk, k_bs
    a.Vt, a.ldvt, a.vt_batch_stride = Vt.data_ptr(), ldvt, vt_bs
    a.O, a.ldo, a.o_batch_stride = O.data_ptr(), ldo, o_bs
    a.key_mask_bits, a.mask_batch_stride_words = _p(mask_bits), mask_bs
    a.mode, a.group_id, a.group_period = mode, _p(group_id), group_period
    a.scale = scale if scale is not None else 128 ** -0.5
    a.q_sumsq, a.k_sumsq = _p(q_sumsq), _p(k_sumsq)
    a.sumsq_ld, a.sumsq_parts, a.norm_dim, a.norm_eps = sumsq_ld, sumsq_parts, norm_dim, norm_eps
    if not (Q.dtype == K.dtype == Vt.dtype == O.dtype) or Q.dtype not in (torch.bfloat16, torch.float16):
        raise L.RfbError("attention operands must share one 16-bit dtype (bf16 or fp16)")
    a.dtype = _DT[Q.dtype]
    keys = 128 if mode == 1 else Nk
    L.check(_timed("attention", 4.0 * B * H * Nq * keys * 128, lambda: lib.rfb_attention(C.byref(a), _stream()),
                   f"B={B} H={H} Nq={Nq} Nk={Nk} mode={mode}"), "rfb_attention")
    return O


def qkv_post(x, w_qk, out_q, kv_ptrs, *, multicast=False, ldkv, row0, rows, d, pos=None, freqs=None, eps=1e-6):
    """Fused [q | k | v] post-processing + all-gather of the row-sharded scene stage (rfb_qkv_post): x fp32
    [rows, 3d]; q -> out_q; k | v -> row row0 + r of every [k | v] row store in `kv_ptrs` (device addresses: own
    store + peer-mapped stores, or one NVLS multicast address with `multicast`)."""
    _need_cuda(x, w_qk, out_q)
    nf = 0 if freqs is None else freqs.numel()
    arr = (C.c_void_p * len(kv_ptrs))(*[int(p) for p in kv_ptrs])
    L.check(_timed("qkv_post", 0.0, lambda: L.load().rfb_qkv_post(
        x.data_ptr(), x.stride(0), w_qk.data_ptr(), out_q.data_ptr(), out_q.stride(0), arr, len(kv_ptrs),
        1 if multicast else 0, ldkv, row0, rows, d, eps, _p(pos), _p(freqs), nf, _DT[out_q.dtype], _stream()),
        f"rows={rows} d={d} dst={len(kv_ptrs)} mc={int(bool(multicast))}"), "rfb_qkv_post")
    return out_q


def attention_ws_elems(B, H, Nq, Nk, kv_split_tiles) -> int:
    """float32 elements of scratch a key-split attention call needs (0: the call does not split)."""
    return int(L.load().rfb_attention_ws_bytes(B, H, Nq, Nk, kv_split_tiles)) // 4


def rmsnorm(x, w, out, *, rows, d, eps=1e-6, gather=None, ldx=None, ldo=None):
    _need_cuda(x, w, out)
    L.check(_timed("rmsnorm", 0.0, lambda: L.load().rfb_rmsnorm(x.data_ptr(), ldx or d, w.data_ptr(), out.data_ptr(), _DT[out.dtype],
                                 ldo or d, rows, d, eps, _p(gather), _stream())), "rfb_rmsnorm")
    return out


def rowstat(x, out16, sumsq, *, rows, d, gather=None):
    """sumsq: [rows, parts] partial-sum layout (total in part 0, the rest cleared).  Input row =
    gather[r] when `gather` (int32 [rows]) is given."""
    _need_cuda(x, out16, sumsq, gather)
    L.check(_timed("rowstat", 0.0, lambda: L.load().rfb_rowstat(
        x.data_ptr(), out16.data_ptr(), _DT[out16.dtype], out16.stride(0), sumsq.data_ptr(), sumsq.stride(0),
        sumsq.shape[1], rows, d, _p(gather),
        _stream())), "rfb_rowstat")
    return out16, sumsq


def qknorm_rope(x, w, out, *, rows, d, nseg, ldx, ldo, in_period=0, pos=None, freqs=None, eps=1e-6):
    _need_cuda(x, w, out)
    nf = 0 if freqs is None else freqs.numel()
    L.check(_timed("qknorm_rope", 0.0, lambda: L.load().rfb_qknorm_rope(x.data_ptr(), ldx, in_period, w.data_ptr(), out.data_ptr(), _DT[out.dtype], ldo, rows, d,
                                     nseg, eps, _p(pos), _p(freqs), nf, _stream()),
                   f"rows={rows} d={d} nseg={nseg} period={in_period}"), "rfb_qknorm_rope")
    return out


def qknorm_rope_table(x, w, out, *, rows, d, nseg, ldx, ldo, cos=None, sin=None, eps=1e-6):
    """QK-RMSNorm + RoPE from ready-made fp32 tables cos / sin [rows, >= 64] (None = norm only)."""
    _need_cuda(x, w, out, cos, sin)
    ldtab = 0 if cos is None else cos.stride(0)
    L.check(_timed("qknorm_rope", 0.0, lambda: L.load().rfb_qknorm_rope_table(
        x.data_ptr(), ldx, _p(w), out.data_ptr(), _DT[out.dtype], ldo, rows, d, nseg, eps, _p(cos), _p(sin), ldtab, _stream()),
        f"rows={rows} d={d} nseg={nseg} table"), "rfb_qknorm_rope_table")
    return out


def token_assemble(a, wa, b, wb, token, prefix, out, *, n_prefix, rows_in, rows_out, batch, d):
    _need_cuda(a, out)
    L.check(_timed("token_assemble", 0.0, lambda: L.load().rfb_token_assemble(a.data_ptr(), wa.data_ptr(), _p(b), _p(wb), token.data_ptr(), _p(prefix),
                                        n_prefix, out.data_ptr(), rows_in, rows_out, batch, d, _stream())), "rfb_token_assemble")
    return out


def texture_prep(tex, out, *, n_tris, channels, texels, log_channels=3):
    _need_cuda(tex, out)
    L.check(_timed("texture_prep", 0.0, lambda: L.load().rfb_texture_prep(tex.data_ptr(), out.data_ptr(), n_tris, channels, texels, log_channels,
                                      _stream())), "rfb_texture_prep")
    return out


def texture_const_prep(tex, out, *, n_tris, channels, ld, log_channels):
    _need_cuda(tex, out)
    L.check(_timed("texture_const_prep", 0.0, lambda: L.load().rfb_texture_const_prep(
        tex.data_ptr(), out.data_ptr(), n_tris, channels, ld, log_channels, _stream())), "rfb_texture_const_prep")
    return out


def vn_encode(vn, out, *, n, nfreq, ld):
    _need_cuda(vn, out)
    L.check(_timed("vn_encode", 0.0, lambda: L.load().rfb_vn_encode(vn.data_ptr(), out.data_ptr(), n, nfreq, ld, _stream())), "rfb_vn_encode")
    return out


def _image_hw(resolution, height, width):
    """(height, width) of a ray-kernel call: `height=` / `width=`, or the square `resolution=`."""
    if height is None and width is None:
        if resolution is None:
            raise ValueError("pass resolution= or height= and width=")
        return resolution, resolution
    if height is None or width is None or resolution is not None:
        raise ValueError("pass resolution= or both height= and width=, not a mix")
    return height, width


def ray_tokens(fov_deg, out, *, n_views, resolution=None, height=None, width=None):
    """Pinhole ray-bundle patch tokens f16 [V, (H/8)*(W/8), 192] from fov in degrees [V] (rfb_ray_tokens_hw)."""
    _need_cuda(fov_deg, out)
    H, W = _image_hw(resolution, height, width)
    L.check(_timed("ray_tokens", 0.0, lambda: L.load().rfb_ray_tokens_hw(fov_deg.data_ptr(), out.data_ptr(), n_views, H, W,
                                                                          _stream())), "rfb_ray_tokens_hw")
    return out


def ray_tokens_canvas(fov_deg, out, *, n_views, canvas_h, canvas_w, height, width, top, left):
    """Pinhole ray-bundle patch tokens f16 [V, (canvas_h/8)*(canvas_w/8), 192] of a canvas holding the height x width
    image at (top, left), with the image's camera (rfb_ray_tokens_canvas)."""
    _need_cuda(fov_deg, out)
    L.check(_timed("ray_tokens", 0.0, lambda: L.load().rfb_ray_tokens_canvas(
        fov_deg.data_ptr(), out.data_ptr(), n_views, canvas_h, canvas_w, height, width, top, left, _stream())),
        "rfb_ray_tokens_canvas")
    return out


def ray_tokens_intrinsics(intr, out, *, n_views, canvas_h, canvas_w, height, width, top=0, left=0):
    """Pinhole ray-bundle patch tokens f16 [V, (canvas_h/8)*(canvas_w/8), 192] from per-view intrinsics fp32 [V, 4] =
    (fx, fy, cx, cy) in pixels of the height x width image the canvas holds at (top, left)
    (rfb_ray_tokens_intrinsics)."""
    _need_cuda(intr, out)
    L.check(_timed("ray_tokens", 0.0, lambda: L.load().rfb_ray_tokens_intrinsics(
        intr.data_ptr(), out.data_ptr(), n_views, canvas_h, canvas_w, height, width, top, left, _stream())),
        "rfb_ray_tokens_intrinsics")
    return out


LENSES = {"opencv": 0, "fisheye": 1}


def ray_tokens_lens(intr, dist, out, *, lens, n_views, canvas_h, canvas_w, height, width, top=0, left=0):
    """Ray-bundle patch tokens f16 [V, (canvas_h/8)*(canvas_w/8), 192] of lens-distorted cameras: intrinsics fp32 [V, 4]
    as `ray_tokens_intrinsics` and coefficients fp32 dist [V, 8] (lens "opencv") or [V, 4] (lens "fisheye")
    (rfb_ray_tokens_lens)."""
    if lens not in LENSES:
        raise ValueError(f"lens must be one of {sorted(LENSES)}, got {lens!r}")
    if dist.numel() != n_views * (8 if lens == "opencv" else 4):
        raise ValueError(f"lens {lens!r} reads {8 if lens == 'opencv' else 4} coefficients per view: dist must have "
                         f"{n_views} x that many values, got {list(dist.shape)}")
    _need_cuda(intr, dist, out)
    L.check(_timed("ray_tokens", 0.0, lambda: L.load().rfb_ray_tokens_lens(
        intr.data_ptr(), dist.data_ptr(), LENSES[lens], out.data_ptr(), n_views, canvas_h, canvas_w, height, width, top,
        left, _stream())), "rfb_ray_tokens_lens")
    return out


FITS = {"auto": 0, "horizontal": 1, "vertical": 2}


def intrinsics_from_fov(fov_deg, out, *, n_views, height, width, fit="auto"):
    """fov in degrees fp32 [V] -> intrinsics fp32 [V, 4] = (f, f, width/2, height/2), the fov spanning the longer side
    ("auto"), the width ("horizontal") or the height ("vertical") (rfb_intrinsics_from_fov)."""
    if fit not in FITS:
        raise ValueError(f"fit must be one of {sorted(FITS)}, got {fit!r}")
    _need_cuda(fov_deg, out)
    L.check(_timed("intrinsics_from_fov", 0.0, lambda: L.load().rfb_intrinsics_from_fov(
        fov_deg.data_ptr(), out.data_ptr(), n_views, height, width, FITS[fit], _stream())), "rfb_intrinsics_from_fov")
    return out


def ray_map_tokens(rays_d, out, *, n_views, resolution=None, height=None, width=None):
    """Explicit ray map fp32 [V, H, W, 3] -> patch tokens f16 [V, (H/8)*(W/8), 192] (rfb_ray_map_tokens_hw)."""
    _need_cuda(rays_d, out)
    H, W = _image_hw(resolution, height, width)
    L.check(_timed("ray_map_tokens", 0.0, lambda: L.load().rfb_ray_map_tokens_hw(rays_d.data_ptr(), out.data_ptr(), n_views,
                                                                                 H, W, _stream())), "rfb_ray_map_tokens_hw")
    return out


def ray_map(c2w, fov_rad, out, *, n_views, resolution=None, height=None, width=None):
    """Pinhole ray map fp32 [V, H, W, 3] from c2w [V,4,4] and fov in radians [V] (rfb_ray_map_hw)."""
    _need_cuda(c2w, fov_rad, out)
    H, W = _image_hw(resolution, height, width)
    L.check(_timed("ray_map", 0.0, lambda: L.load().rfb_ray_map_hw(c2w.data_ptr(), fov_rad.data_ptr(), out.data_ptr(), n_views,
                                                                   H, W, _stream())), "rfb_ray_map_hw")
    return out


def positions(tri, mask_u8, c2w, pos, *, n, n_reg, rows_out, n_views):
    _need_cuda(tri, mask_u8, pos)
    L.check(_timed("positions", 0.0, lambda: L.load().rfb_positions(tri.data_ptr(), mask_u8.data_ptr(), _p(c2w), pos.data_ptr(), n, n_reg, rows_out,
                                   n_views, _stream())), "rfb_positions")
    return pos


def pack_mask(mask_u8, bits, *, n, n_prefix, words, batch):
    _need_cuda(mask_u8, bits)
    L.check(_timed("pack_mask", 0.0, lambda: L.load().rfb_pack_mask(mask_u8.data_ptr(), bits.data_ptr(), n, n_prefix, words, batch, _stream())), "rfb_pack_mask")
    return bits


def cast(x, out):
    _need_cuda(x, out)
    L.check(_timed("cast", 0.0, lambda: L.load().rfb_cast(x.data_ptr(), out.data_ptr(), _DT[out.dtype], x.numel(), _stream())), "rfb_cast")
    return out


def transpose16(x, out, *, rows, cols):
    """out[c, r] = x[r, c] for 16-bit 2-D (possibly strided) tensors."""
    _need_cuda(x, out)
    L.check(_timed("transpose16", 0.0, lambda: L.load().rfb_transpose16(x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0),
                                                                        rows, cols, _stream())), "rfb_transpose16")
    return out


def pixel_shuffle(x, out, *, B, h, w, s, C_):
    _need_cuda(x, out)
    L.check(_timed("pixel_shuffle", 0.0, lambda: L.load().rfb_pixel_shuffle(x.data_ptr(), out.data_ptr(), B, h, w, s, C_, _stream())), "rfb_pixel_shuffle")
    return out


def im2col_s2(x, out, *, B, H, W, C_):
    _need_cuda(x, out)
    L.check(_timed("im2col_s2", 0.0, lambda: L.load().rfb_im2col_s2(x.data_ptr(), out.data_ptr(), B, H, W, C_, _stream())), "rfb_im2col_s2")
    return out


def upsample_bilinear(x, out, *, B, Hi, Wi, Ho, Wo, C_):
    _need_cuda(x, out)
    L.check(_timed("upsample_bilinear", 0.0, lambda: L.load().rfb_upsample_bilinear(x.data_ptr(), out.data_ptr(), B, Hi, Wi, Ho, Wo, C_, _stream())), "rfb_upsample_bilinear")
    return out


TONE_MAPPERS = {"none": 0, "pbr_neutral": 1, "Khronos PBR Neutral": 1}


def ldr_quantize(hdr: torch.Tensor, tone_mapper: str = "none") -> torch.Tensor:
    """HDR fp32 [..., 3] -> uint8 [..., 3] on the device (infer.py:94-98).  'none' is the CLIs' default
    clip-and-truncate, bit-exact; 'pbr_neutral' is the published Khronos curve + sRGB OETF (unpinned)."""
    _need_cuda(hdr)
    if tone_mapper not in TONE_MAPPERS:
        raise ValueError(f"tone_mapper must be one of {sorted(TONE_MAPPERS)} (agx / filmic need OpenColorIO LUTs)")
    if hdr.dtype != torch.float32 or hdr.shape[-1] != 3:
        raise ValueError("hdr must be fp32 [..., 3]")
    hdr = hdr.contiguous()
    out = torch.empty(hdr.shape, dtype=torch.uint8, device=hdr.device)
    L.check(_timed("ldr_quantize", 0.0, lambda: L.load().rfb_ldr_quantize(
        hdr.data_ptr(), out.data_ptr(), hdr.numel() // 3, TONE_MAPPERS[tone_mapper], _stream())), "rfb_ldr_quantize")
    return out
