"""The reference's module boundaries on the sm_100a kernels.

Every class below keeps the constructor signature, parameter tree (state_dict keys) and `forward`
signature of its namesake in the reference, so code written against `renderformer.layers.*`,
`renderformer.encodings.*`, `renderformer.utils.*` and `renderformer.models.view_transformer` keeps
working; the math of every `forward` runs in the C-ABI kernels (renderformer_b200/ops.py), never in
torch.  The leaves (nn.Linear, nn.RMSNorm, nn.Conv2d, ...) are plain parameter holders.

Two tiers:
* stack-level classes -- TransformerEncoder, TransformerDecoder, DPTHead, ViewTransformer -- forward to
  the FUSED schedules of renderformer_b200.engine.Engine (the same code the pipeline runs);
* block-level classes -- FeedForwardSwiGLU, MultiHeadAttention, SwinSelfAttention, AttentionLayer -- are
  self-contained kernel sequences (norm -> GEMM -> QK-norm/RoPE -> attention -> GEMM) without the
  cross-block fusions, for callers that drive single blocks.

Only the configuration space of the released checkpoints is implemented (RMSNorm, SwiGLU, no bias,
QK-norm, triangle RoPE, head_dim 128); anything else raises NotImplementedError at construction or call
time -- there is no torch fallback.  Inference only (no autograd through the kernels).

Reference: layers/attention.py:34-57,85-202,205-370,373-527,530-590,593-688; layers/dpt.py:57-273;
models/view_transformer.py:12-127; encodings/rope.py:41-206; encodings/nerf_encoding.py:25-84;
utils/ray_generator.py:6-50; utils/transform.py:7-27.
"""
from __future__ import annotations

import math
from typing import Literal, Optional

import torch
from torch import nn

from . import lib as L
from . import ops
from .config import RenderFormerConfig

EPS = 1e-6  # layers/attention.py:16
# tensor-core operand format of modules called on their own (the reference CLIs' default precision is fp16;
# the pipeline picks the format per call from `torch_dtype`)
OPERAND_DTYPE = torch.float16


def _rup(x: int, m: int) -> int:
    return (x + m - 1) // m * m


def _need_eval(m: nn.Module, dropout: float):
    if m.training and dropout > 0:
        raise NotImplementedError("dropout > 0 in training mode: the kernels implement inference only")


class _Cached:
    """Kernel-ready weight layouts, rebuilt when a parameter changes or moves."""

    def _cached(self, build):
        params = list(self.parameters())
        key = (str(params[0].device),) + tuple((p.data_ptr(), p._version) for p in params)
        if getattr(self, "_kcache_key", None) != key:
            self._kcache, self._kcache_key = build(), key
        return self._kcache

    @property
    def _dev(self) -> torch.device:
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise L.RfbError(f"{type(self).__name__}.forward needs the module on a CUDA device (no CPU fallback)")
        return dev


def _rms_norm(dim: int, norm_type: str, eps=EPS) -> nn.Module:
    if norm_type != "rms_norm":
        raise NotImplementedError("norm_type='layer_norm' is not exercised by the released configs (SURVEY §8a)")
    return nn.RMSNorm(dim, eps=eps)


def _f32_rows(x: torch.Tensor, d: int) -> torch.Tensor:
    return x.reshape(-1, d).to(torch.float32).contiguous()


def _pack_key_mask(mask: Optional[torch.Tensor], B: int, Nk: int, dev):
    """bool [B, Nk] (True = attend) -> packed bits for rfb_attention (None = attend to everything)."""
    if mask is None:
        return None, 0
    if tuple(mask.shape) != (B, Nk):
        raise AssertionError(f"expecting key_padding_mask shape of {(B, Nk)}, but got {tuple(mask.shape)}")
    m8 = mask.to(dev).contiguous().view(torch.uint8) if mask.dtype == torch.bool else mask.to(dev, torch.uint8)
    words = 4 * ((Nk + 127) // 128)
    bits = ops.pack_mask(m8, torch.empty((B, words), dtype=torch.int32, device=dev), n=Nk, n_prefix=0, words=words, batch=B)
    return bits, words


# =============================================================================================== encodings
class NeRFEncoding(nn.Module):
    """encodings/nerf_encoding.py:25-84: [x, sin(x 2^j), sin(x 2^j + pi/2)], j = 0..F-1, no pi factor.
    The 9-dimensional case (vertex normals) runs in rfb_vn_encode (fp16 kernel output, returned as fp32);
    F = 0 is the identity (view directions)."""

    def __init__(self, in_dim: int, num_frequencies: int, min_freq_exp: float = 0.0,
                 max_freq_exp: Optional[float] = None, include_input: bool = False) -> None:
        super().__init__()
        self.in_dim, self.num_frequencies = in_dim, num_frequencies
        self.min_freq = min_freq_exp
        self.max_freq = num_frequencies - 1 if max_freq_exp is None else max_freq_exp
        self.include_input = include_input

    def get_out_dim(self) -> int:
        return self.in_dim * self.num_frequencies * 2 + (self.in_dim if self.include_input else 0)

    def forward(self, in_tensor: torch.Tensor) -> torch.Tensor:
        F_ = self.num_frequencies
        if F_ == 0:
            return in_tensor if self.include_input else in_tensor[..., :0]
        if (in_tensor.shape[-1] != 9 or not self.include_input or self.min_freq != 0 or self.max_freq != F_ - 1
                or not in_tensor.is_cuda):
            raise NotImplementedError("NeRFEncoding kernel: 9-d CUDA input, include_input, frequencies 2^0..2^(F-1)")
        x = _f32_rows(in_tensor, 9)
        ld = _rup(9 + 18 * F_, 64)
        out = ops.vn_encode(x, torch.empty((x.shape[0], ld), dtype=torch.float16, device=x.device), n=x.shape[0],
                            nfreq=F_, ld=ld)
        return out[:, :9 + 18 * F_].float().reshape(*in_tensor.shape[:-1], 9 + 18 * F_)


def rotate_half_hf(x):
    """encodings/rope.py:41-45."""
    x1, x2 = x[..., : x.shape[-1] // 2], x[..., x.shape[-1] // 2:]
    return torch.cat((-x2, x1), dim=-1)


def freqs_to_cos_sin(freqs, scale=1.0, start_index=0, head_dim=None):
    """encodings/rope.py:78-103 (table construction: host-side glue; the fused kernels never build tables,
    they take the positions -- this exists for callers of the block-level classes)."""
    if head_dim is not None:
        freqs = freqs[..., : freqs.shape[-1] // 2]
        right = head_dim // 2 - (start_index + freqs.shape[-1])
        z = lambda n: torch.zeros((*freqs.shape[:-1], n), device=freqs.device)  # noqa: E731
        freqs = torch.cat((z(start_index), freqs, z(right)), dim=-1)
        freqs = torch.cat([freqs, freqs], dim=-1)
    return freqs.cos() * scale, freqs.sin() * scale


def _rope_rows(t: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor) -> torch.Tensor:
    """(B, H, N, 128) rotated by (B, 1, N, 128) tables on rfb_qknorm_rope_table (no normalisation)."""
    B, H, N, hd = t.shape
    if hd != 128 or cos.shape[-1] != 128:
        raise NotImplementedError("RoPE kernel: head_dim 128")
    x = t.permute(0, 2, 1, 3).reshape(B * N, H * hd).to(torch.float32).contiguous()
    c = cos.expand(B, 1, N, hd).reshape(B * N, hd).to(torch.float32).contiguous()
    s = sin.expand(B, 1, N, hd).reshape(B * N, hd).to(torch.float32).contiguous()
    out = torch.empty((B * N, H * hd), dtype=OPERAND_DTYPE, device=t.device)
    ops.qknorm_rope_table(x, None, out, rows=B * N, d=H * hd, nseg=1, ldx=H * hd, ldo=H * hd, cos=c, sin=s)
    return out.view(B, N, H, hd).permute(0, 2, 1, 3).to(t.dtype)


def apply_rotary_emb_one_cossin(one_tensor, cos, sin):
    """encodings/rope.py:132-149 (result rounded to bf16 by the kernel before the cast back)."""
    return _rope_rows(one_tensor, cos, sin)


def apply_rotary_emb_cossin(q, k, cos, sin):
    """encodings/rope.py:107-129."""
    return _rope_rows(q, cos, sin), _rope_rows(k, cos, sin)


class TriangleRotaryEmbedding(nn.Module):
    """encodings/rope.py:152-206: log-spaced frequencies 2**linspace(0, log2(dim/2 - 1), dim/2), stored as a
    frozen parameter (it is in the state_dict).  The angle table is host-side glue (see freqs_to_cos_sin)."""

    def __init__(self, dim, hf_format=True, double_max_freq=False):
        super().__init__()
        if not hf_format or double_max_freq:
            raise NotImplementedError("only the hf RoPE layout without doubled frequency range")
        self.hf_format = hf_format
        max_freq = math.log(dim // 2 - 1, 2)
        self.freqs = nn.Parameter(2 ** torch.linspace(0, max_freq, dim // 2), requires_grad=False)
        self.register_buffer("dummy", torch.tensor(0), persistent=False)

    @property
    def device(self):
        return self.dummy.device

    def get_triangle_freqs(self, pos: torch.Tensor):
        f = self.forward(pos)  # [B, N, 9, F]
        f = f.reshape(f.shape[0], 1, f.shape[1], -1)
        return torch.cat([f, f], dim=-1)

    def forward(self, t: torch.Tensor, seq_len=None, offset=0):
        return t.to(self.freqs.dtype)[..., None] * self.freqs


# =============================================================================================== utils
class RayGenerator(nn.Module):
    """utils/ray_generator.py:6-50 on rfb_ray_map_hw: pinhole pixel-centre rays rotated by R(c2w), normalised.
    `img_res` is an int (square, as in the reference) or (height, width); the fov spans the longer side."""

    def forward(self, c2w, fov, img_res=256):
        batch_shape = c2w.shape[:-2]
        if not c2w.is_cuda:
            raise L.RfbError("RayGenerator.forward needs CUDA tensors (no CPU fallback)")
        H, W = tuple(img_res) if isinstance(img_res, (tuple, list)) else (img_res, img_res)
        c = c2w.reshape(-1, 4, 4).to(torch.float32).contiguous()
        f = fov.reshape(-1).to(torch.float32).contiguous()
        out = torch.empty((c.shape[0], H, W, 3), dtype=torch.float32, device=c.device)
        ops.ray_map(c, f, out, n_views=c.shape[0], height=H, width=W)
        return c2w[..., :3, 3], out.view(*batch_shape, H, W, 3)


@torch.no_grad()
def trans_to_cam_coord(c2w: torch.Tensor, triangles: torch.Tensor, vns: Optional[torch.Tensor] = None):
    """utils/transform.py:7-27 on rfb_positions: T^-1 x for every vertex (T = c2w, rigid), identity c2w back,
    and R^T n for the optional normals."""
    if not triangles.is_cuda:
        raise L.RfbError("trans_to_cam_coord needs CUDA tensors (no CPU fallback)")
    B, N = triangles.shape[:2]
    dev = triangles.device
    ones = torch.ones((N,), dtype=torch.uint8, device=dev)
    c = c2w.to(torch.float32).contiguous()

    def apply(mats, pts):
        out = torch.empty((B, N, 9), dtype=torch.float32, device=dev)
        p9 = pts.reshape(B, N, 9).to(torch.float32).contiguous()
        for b in range(B):
            ops.positions(p9[b], ones, mats[b:b + 1], out[b:b + 1], n=N, n_reg=0, rows_out=N, n_views=1)
        return out.view(B, N, 3, 3).to(triangles.dtype)
    tri_cam = apply(c, triangles)
    vn_cam = None
    if vns is not None:
        rot = c.clone()
        rot[:, :3, 3] = 0
        vn_cam = apply(rot, vns)
    return tri_cam, torch.eye(4, device=dev, dtype=triangles.dtype).repeat(c2w.shape[0], 1, 1), vn_cam


# =============================================================================================== blocks
class FeedForwardSwiGLU(nn.Module, _Cached):
    """layers/attention.py:34-57: w2(silu(w1 x) * w3 x), as two GEMMs (w1 || w3 interleaved, SwiGLU epilogue)."""

    def __init__(self, dim: int, hidden_dim: int, dropout: float = 0.1, bias: bool = True):
        super().__init__()
        self.w1 = nn.Linear(dim, hidden_dim, bias=bias)
        self.w2 = nn.Linear(hidden_dim, dim, bias=bias)
        self.w3 = nn.Linear(dim, hidden_dim, bias=bias)
        self.dropout = nn.Dropout(dropout) if dropout > 0 else nn.Identity()
        self._p_drop = dropout

    def _weights(self):
        def build():
            if self.w1.bias is not None:
                raise NotImplementedError("FeedForwardSwiGLU kernels: bias=False (released configs)")
            w1, w3 = self.w1.weight.detach().float(), self.w3.weight.detach().float()
            f, d = w1.shape
            w13 = torch.stack([w1.view(f // 16, 16, d), w3.view(f // 16, 16, d)], dim=1).reshape(2 * f, d)
            return w13.to(OPERAND_DTYPE).contiguous(), self.w2.weight.detach().to(OPERAND_DTYPE).contiguous()
        return self._cached(build)

    def _run(self, h16: torch.Tensor, residual: Optional[torch.Tensor] = None) -> torch.Tensor:
        """h16 bf16 [rows, dim] (already normalised) -> fp32 [rows, dim] (+ residual)."""
        w13, w2 = self._weights()
        g = ops.gemm(h16, w13, epi=L.EPI_SWIGLU, out_dtype=OPERAND_DTYPE)
        out = torch.empty((h16.shape[0], w2.shape[0]), dtype=torch.float32, device=h16.device)
        return ops.gemm(g, w2, out=out, res1=residual)

    def forward(self, x):
        _need_eval(self, self._p_drop)
        self._dev
        d = self.w1.in_features
        x32 = _f32_rows(x, d)
        h = ops.cast(x32, torch.empty(x32.shape, dtype=OPERAND_DTYPE, device=x32.device))
        return self._run(h).view(*x.shape[:-1], d)


class MultiHeadAttention(nn.Module, _Cached):
    """layers/attention.py:85-202.  q/k/v projections (one fused GEMM for self-attention, V produced
    transposed), QK-RMSNorm over the full width + RoPE from the given cos / sin tables in one row kernel,
    tcgen05 flash attention with the key-padding mask fused, out-projection."""

    def __init__(self, query_dim, num_heads, kv_dim=None, bias=True, qk_norm=False, norm_type="layer_norm"):
        super().__init__()
        self.apply_rope_cossin = apply_rotary_emb_cossin
        self.num_heads = num_heads
        self.is_self_attn = kv_dim is None
        kv_dim = query_dim if kv_dim is None else kv_dim
        if self.is_self_attn:
            self.in_proj = nn.Linear(query_dim, 3 * query_dim, bias=bias)
        else:
            self.q_proj = nn.Linear(query_dim, query_dim, bias=bias)
            self.k_proj = nn.Linear(kv_dim, query_dim, bias=bias)
            self.v_proj = nn.Linear(kv_dim, query_dim, bias=bias)
        self.out_proj = nn.Linear(query_dim, query_dim, bias=bias)
        if qk_norm:
            self.q_norm, self.k_norm = _rms_norm(query_dim, norm_type), _rms_norm(query_dim, norm_type)
        else:
            self.q_norm, self.k_norm = nn.Identity(), nn.Identity()
        self.query_dim = query_dim

    def _weights(self):
        def build():
            if self.out_proj.bias is not None:
                raise NotImplementedError("MultiHeadAttention kernels: bias=False (released configs)")
            if isinstance(self.q_norm, nn.Identity):
                raise NotImplementedError("MultiHeadAttention kernels: qk_norm=True (released configs)")
            if self.query_dim // self.num_heads != 128:
                raise NotImplementedError("attention kernels: head_dim 128")
            bf = OPERAND_DTYPE
            w = {"o": self.out_proj.weight.detach().to(bf).contiguous(),
                 "qn": self.q_norm.weight.detach().float().contiguous(), "kn": self.k_norm.weight.detach().float().contiguous()}
            w["qkn"] = torch.cat([w["qn"], w["kn"]])
            if self.is_self_attn:
                w["in"] = self.in_proj.weight.detach().to(bf).contiguous()
            else:
                for n in ("q", "k", "v"):
                    w[n] = getattr(self, n + "_proj").weight.detach().to(bf).contiguous()
            return w
        return self._cached(build)

    def _run(self, q16, kv16, B, Nq, Nk, mask, rope_cos, rope_sin, rope_ctx_cos, rope_ctx_sin, residual=None):
        """q16 bf16 [B*Nq, dq], kv16 bf16 [B*Nk, dkv] (already normalised) -> fp32 [B*Nq, dq] (+ residual)."""
        w = self._weights()
        d, H, dev = self.query_dim, self.num_heads, q16.device
        bf, f32 = OPERAND_DTYPE, torch.float32

        def table(t, n):
            return None if t is None else t.expand(B, 1, n, 128).reshape(B * n, 128).to(f32).contiguous()
        Nkp = _rup(Nk, 8)
        vt = torch.empty((B, d, Nkp), dtype=bf, device=dev)
        if self.is_self_attn:
            if Nk != Nkp:
                raise NotImplementedError("self-attention kernels: sequence length must be a multiple of 8")
            qk = ops.gemm(q16, w["in"], out=torch.empty((B * Nq, 2 * d), dtype=f32, device=dev), vt_out=vt, vt_split=2 * d,
                          vt_rows_per_batch=Nq)
            qkr = torch.empty((B * Nq, 2 * d), dtype=bf, device=dev)
            if rope_ctx_cos is None:
                ops.qknorm_rope_table(qk, w["qkn"], qkr, rows=B * Nq, d=d, nseg=2, ldx=2 * d, ldo=2 * d,
                                      cos=table(rope_cos, Nq), sin=table(rope_sin, Nq), eps=EPS)
            else:
                ops.qknorm_rope_table(qk, w["qn"], qkr, rows=B * Nq, d=d, nseg=1, ldx=2 * d, ldo=2 * d,
                                      cos=table(rope_cos, Nq), sin=table(rope_sin, Nq), eps=EPS)
                ops.qknorm_rope_table(qk[:, d:], w["kn"], qkr[:, d:], rows=B * Nq, d=d, nseg=1, ldx=2 * d, ldo=2 * d,
                                      cos=table(rope_ctx_cos, Nk), sin=table(rope_ctx_sin, Nk), eps=EPS)
            Q, K, ldq, ldk = qkr, qkr[:, d:], 2 * d, 2 * d
        else:
            qf = ops.gemm(q16, w["q"], out_dtype=f32)
            kf = ops.gemm(kv16, w["k"], out_dtype=f32)
            for b in range(B):  # V^T[b] = Wv . kv[b]^T : operands swapped
                ops.gemm(w["v"], kv16[b * Nk:(b + 1) * Nk], out=vt[b], N=Nk)
            Q, K = torch.empty((B * Nq, d), dtype=bf, device=dev), torch.empty((B * Nk, d), dtype=bf, device=dev)
            kc, ks = (rope_cos, rope_sin) if rope_ctx_cos is None else (rope_ctx_cos, rope_ctx_sin)
            if rope_ctx_cos is None and rope_cos is not None and Nq != Nk:
                raise ValueError("cross-attention with one rope table needs equal query / key lengths")
            ops.qknorm_rope_table(qf, w["qn"], Q, rows=B * Nq, d=d, nseg=1, ldx=d, ldo=d, cos=table(rope_cos, Nq),
                                  sin=table(rope_sin, Nq), eps=EPS)
            ops.qknorm_rope_table(kf, w["kn"], K, rows=B * Nk, d=d, nseg=1, ldx=d, ldo=d, cos=table(kc, Nk),
                                  sin=table(ks, Nk), eps=EPS)
            ldq = ldk = d
        bits, words = _pack_key_mask(mask, B, Nk, dev)
        att = torch.empty((B * Nq, d), dtype=bf, device=dev)
        ops.attention(Q, K, vt, att, B=B, H=H, Nq=Nq, Nk=Nk, ldq=ldq, ldk=ldk, ldvt=Nkp, ldo=d, q_bs=Nq * ldq,
                      k_bs=Nk * ldk, vt_bs=d * Nkp, o_bs=Nq * d, mask_bits=bits, mask_bs=words)
        out = torch.empty((B * Nq, d), dtype=f32, device=dev)
        return ops.gemm(att, w["o"], out=out, res1=residual)

    def forward(self, q, k, v, src_key_padding_mask=None, rope_cos=None, rope_sin=None, rope_ctx_cos=None,
                rope_ctx_sin=None, force_sdpa=False):
        self._dev
        if k is not v and not self.is_self_attn:
            raise NotImplementedError("MultiHeadAttention kernels: key and value share one input (kv)")
        B, Nq, Nk = q.shape[0], q.shape[1], k.shape[1]
        q32 = _f32_rows(q, q.shape[-1])
        q16 = ops.cast(q32, torch.empty(q32.shape, dtype=OPERAND_DTYPE, device=q32.device))
        if self.is_self_attn:
            kv16 = q16
        else:
            k32 = _f32_rows(k, k.shape[-1])
            kv16 = ops.cast(k32, torch.empty(k32.shape, dtype=OPERAND_DTYPE, device=k32.device))
        out = self._run(q16, kv16, B, Nq, Nk, src_key_padding_mask, rope_cos, rope_sin, rope_ctx_cos, rope_ctx_sin)
        return out.view(B, Nq, self.query_dim)


def window_partition(x, window_size):
    """layers/attention.py:205-217 (index shuffle; host-side helper, the kernels fold it into row maps)."""
    B, H, W, C = x.shape
    x = x.view(B, H // window_size, window_size, W // window_size, window_size, C)
    return x.permute(0, 1, 3, 2, 4, 5).contiguous().view(-1, window_size, window_size, C)


def window_reverse(windows, window_size, H, W):
    """layers/attention.py:220-234."""
    B = int(windows.shape[0] / (H * W / window_size / window_size))
    x = windows.view(B, H // window_size, W // window_size, window_size, window_size, -1)
    return x.permute(0, 1, 3, 2, 4, 5).contiguous().view(B, H, W, -1)


def get_swin_attn_mask(H, W, window_size, shift_size, device):
    """layers/attention.py:238-271 from the closed form of the region ids (SURVEY Appendix E3); no global
    cache (the reference's is keyed without the device)."""
    from .engine import swin_window_maps
    _, region = swin_window_maps(H, W, shift_size, window_size)
    r = region.view(-1, window_size * window_size).to(device)
    return r.unsqueeze(1) == r.unsqueeze(2)


class SwinSelfAttention(nn.Module, _Cached):
    """layers/attention.py:274-370.  roll + window partition are a row gather folded into the 16-bit cast,
    the [q|k|v] projection is one GEMM (V transposed), QK-RMSNorm is carried as partial row sums into the
    shifted-window attention kernel (block-diagonal + region-id mask), and the out-projection scatters the
    rows back through the inverse permutation."""

    def __init__(self, dim, num_heads, window_size, shift_size: int = 0, bias=True, qk_norm=False,
                 norm_type="layer_norm"):
        super().__init__()
        self.dim, self.num_heads, self.window_size, self.shift_size = dim, num_heads, window_size, shift_size
        self.in_proj = nn.Linear(dim, 3 * dim, bias=bias)
        self.out_proj = nn.Linear(dim, dim, bias=bias)
        if qk_norm:
            self.q_norm, self.k_norm = _rms_norm(dim, norm_type), _rms_norm(dim, norm_type)
        else:
            self.q_norm, self.k_norm = nn.Identity(), nn.Identity()
        self._maps = {}

    def _weights(self):
        def build():
            if self.in_proj.bias is not None or isinstance(self.q_norm, nn.Identity) or self.window_size != 8:
                raise NotImplementedError("SwinSelfAttention kernels: bias=False, qk_norm=True, 8x8 windows")
            if self.dim // self.num_heads != 128:
                raise NotImplementedError("attention kernels: head_dim 128")
            bf = OPERAND_DTYPE
            return {"in": self.in_proj.weight.detach().to(bf).contiguous(),
                    "o": self.out_proj.weight.detach().to(bf).contiguous(),
                    "qkn": torch.cat([self.q_norm.weight.detach().float(), self.k_norm.weight.detach().float()]).contiguous()}
        return self._cached(build)

    def _window_maps(self, B, H, W, dev):
        from .engine import swin_window_maps
        key = (B, H, W, str(dev))
        if key not in self._maps:
            perm, region = swin_window_maps(H, W, self.shift_size, self.window_size)
            n = H * W
            full = (perm[None, :] + (torch.arange(B, dtype=torch.int32) * n)[:, None]).reshape(-1)
            self._maps[key] = (full.to(dev).contiguous(), region.to(dev).contiguous())
        return self._maps[key]

    def _run(self, x32: torch.Tensor, B, H, W, residual=None, scale_rows=None):
        """x32 fp32 [B*H*W, dim] in token order (already normalised) -> fp32 [B*H*W, dim] (+ residual)."""
        w = self._weights()
        d, Hh, dev = self.dim, self.num_heads, x32.device
        if H % 8 or W % 8 or (H * W) % 128:
            raise ValueError("swin kernels need token grids that are multiples of 8 with H*W a multiple of 128")
        rows, P = B * H * W, d // 128
        bf, f32 = OPERAND_DTYPE, torch.float32
        perm, region = self._window_maps(B, H, W, dev)
        xw = torch.empty((rows, d), dtype=bf, device=dev)
        ops.rowstat(x32, xw, torch.empty((rows, 1), dtype=f32, device=dev), rows=rows, d=d, gather=perm)
        qkh, qksq = torch.empty((rows, 2 * d), dtype=bf, device=dev), torch.empty((rows, 2 * P), dtype=f32, device=dev)
        vt = torch.empty((d, rows), dtype=bf, device=dev)
        ops.gemm(xw, w["in"], out16=qkh, col_mul=w["qkn"], out_sumsq=qksq, vt_out=vt, vt_split=2 * d)
        att = torch.empty((rows, d), dtype=bf, device=dev)
        ops.attention(qkh, qkh[:, d:], vt, att, B=1, H=Hh, Nq=rows, Nk=rows, ldq=2 * d, ldk=2 * d, ldvt=rows, ldo=d,
                      mode=1, group_id=region, group_period=H * W, q_sumsq=qksq, k_sumsq=qksq.view(-1)[P:],
                      sumsq_ld=2 * P, sumsq_parts=P, norm_dim=d, norm_eps=EPS)
        out = torch.empty((rows, d), dtype=f32, device=dev)
        return ops.gemm(att, w["o"], out=out, res1=residual, row_map=perm)

    def forward(self, x):
        self._dev
        B, H, W, C = x.shape
        return self._run(_f32_rows(x, C), B, H, W).view(B, H, W, C)


class AttentionLayer(nn.Module, _Cached):
    """layers/attention.py:373-527: pre-norm residual block  x += MHA(norm(x), norm(kv));
    [x += SelfAttn(norm(x))];  x += FFN(norm(x)).  RMSNorm kernels feed the GEMMs in bf16, the residual adds
    are the out-projection epilogues, the residual stream stays fp32."""

    def __init__(self, query_dim: int, num_heads: int, ffn_hidden_dim: int, kv_dim: Optional[int] = None,
                 dropout: float = 0.1, bias: bool = True, bias_kv: bool = False, activation: str = "swiglu",
                 norm_type: Literal["layer_norm", "rms_norm"] = "layer_norm", disable_q_norm: bool = False,
                 disable_kv_norm: bool = False, qk_norm: bool = False, add_self_attn: bool = False,
                 use_swin_attn: bool = False, window_size: int = 8, shift_size: int = 0):
        super().__init__()
        if bias_kv:
            raise NotImplementedError("Bias for key and value is not supported for now")  # as the reference :426
        if activation != "swiglu":
            raise NotImplementedError("activation='gelu' is not exercised by the released configs (SURVEY §8a)")
        if disable_q_norm or disable_kv_norm:
            raise NotImplementedError("disable_q_norm / disable_kv_norm")
        self.multihead_attn = MultiHeadAttention(query_dim, num_heads, kv_dim, bias, qk_norm, norm_type)
        self.dropout = nn.Dropout(dropout) if dropout > 0 else nn.Identity()
        self._p_drop = dropout
        self.query_norm = _rms_norm(query_dim, norm_type)
        if not self.multihead_attn.is_self_attn:
            self.kv_norm = _rms_norm(query_dim if kv_dim is None else kv_dim, norm_type)
        self.add_self_attn, self.use_swin_attn = add_self_attn, use_swin_attn
        if add_self_attn:
            if use_swin_attn:
                self.self_attn = SwinSelfAttention(query_dim, num_heads, window_size, shift_size, bias, qk_norm, norm_type)
            else:
                self.self_attn = MultiHeadAttention(query_dim, num_heads, None, bias, qk_norm, norm_type)
            self.self_attn_norm = _rms_norm(query_dim, norm_type)
        self.ffn = FeedForwardSwiGLU(query_dim, hidden_dim=ffn_hidden_dim, dropout=dropout, bias=bias)
        self.ffn_norm = _rms_norm(query_dim, norm_type)
        self.query_dim = query_dim

    @staticmethod
    def _norm16(x32, norm: nn.RMSNorm, dtype=OPERAND_DTYPE):
        rows, d = x32.shape
        return ops.rmsnorm(x32, norm.weight.detach().float().contiguous(), torch.empty((rows, d), dtype=dtype, device=x32.device),
                           rows=rows, d=d, eps=EPS)

    def forward(self, query, kv=None, src_key_padding_mask=None, rope_cos=None, rope_sin=None, rope_ctx_cos=None,
                rope_ctx_sin=None, force_sdpa=False, patch_h=None, patch_w=None):
        _need_eval(self, self._p_drop)
        self.ffn._dev  # raises unless the module lives on a CUDA device
        B, Nq, d = query.shape
        x = _f32_rows(query, d).clone()                       # fp32 residual stream, updated by the epilogues
        q16 = self._norm16(x, self.query_norm)
        if self.multihead_attn.is_self_attn:
            kv16, Nk = q16, Nq
        else:
            kv32 = _f32_rows(kv, kv.shape[-1])
            kv16, Nk = self._norm16(kv32, self.kv_norm), kv.shape[1]
        x = self.multihead_attn._run(q16, kv16, B, Nq, Nk, src_key_padding_mask, rope_cos, rope_sin, rope_ctx_cos,
                                     rope_ctx_sin, residual=x)
        if self.add_self_attn:
            if self.use_swin_attn:
                h32 = self._norm16(x, self.self_attn_norm, torch.float32)
                x = self.self_attn._run(h32, B, patch_h, patch_w, residual=x)
            else:
                h16 = self._norm16(x, self.self_attn_norm)
                x = self.self_attn._run(h16, h16, B, Nq, Nq, None, rope_cos, rope_sin, None, None, residual=x)
        x = self.ffn._run(self._norm16(x, self.ffn_norm), residual=x)
        return x.view(B, Nq, d)


# =============================================================================================== stacks
def _stack_config(**kw) -> RenderFormerConfig:
    return RenderFormerConfig.from_dict({**RenderFormerConfig().to_dict(), **kw})


def _check_stack_args(activation, norm_type, norm_first, bias, bias_kv, qk_norm, rope_type, rope_double_max_freq, rope_dim):
    if not norm_first:
        raise AssertionError("Only support norm_first=True")
    if activation != "swiglu" or norm_type != "rms_norm" or bias or bias_kv or not qk_norm:
        raise NotImplementedError("stack kernels: swiglu, rms_norm, bias=False, qk_norm=True (released configs; SURVEY §8a)")
    if rope_type != "triangle" or rope_double_max_freq or rope_dim is None:
        raise NotImplementedError("stack kernels: rope_type='triangle' with a rope_dim")


class _EngineBacked(_Cached):
    """A stack whose forward is one of Engine's fused schedules; the engine holds the kernel-ready weights of
    THIS module's parameters only (`parts`)."""
    _parts: tuple = ()
    _prefix: str = ""

    def _engine(self):
        from .engine import Engine

        def build():
            sd = {self._prefix + k: v for k, v in self.state_dict().items()}
            return Engine(self._cfg, sd, self._dev, parts=self._parts, op_dtype=OPERAND_DTYPE)
        return self._cached(build)


class TransformerEncoder(nn.Module, _EngineBacked):
    """layers/attention.py:530-590 on Engine.encoder_layers (RMSNorm fused into the GEMMs, [q|k|v] in one
    GEMM, QK-norm + RoPE from the triangle positions in one row kernel, two-tile tcgen05 attention)."""
    _parts, _prefix = ("encoder",), "transformer."

    def __init__(self, num_layers: int, num_heads: int, hidden_dim: int, ffn_hidden_dim: int, dropout: float = 0.1,
                 bias: bool = True, bias_kv: bool = False, activation: str = "gelu",
                 norm_type: Literal["layer_norm", "rms_norm"] = "layer_norm", norm_first: bool = True,
                 rope_dim: Optional[int] = None,
                 rope_type: Literal["triangle", "triangle_learned", "triangle_mixed"] = "triangle",
                 rope_double_max_freq: bool = False, qk_norm: bool = False):
        super().__init__()
        _check_stack_args(activation, norm_type, norm_first, bias, bias_kv, qk_norm, rope_type, rope_double_max_freq, rope_dim)
        self.head_dim = hidden_dim // num_heads
        self.layers = nn.ModuleList([
            AttentionLayer(query_dim=hidden_dim, num_heads=num_heads, ffn_hidden_dim=ffn_hidden_dim, dropout=dropout,
                           bias=bias, bias_kv=bias_kv, activation=activation, norm_type=norm_type, qk_norm=qk_norm)
            for _ in range(num_layers)])
        self.rope_dim = rope_dim
        assert rope_dim % 2 == 0, "rope_dim must be even"
        assert rope_dim // 2 * 9 <= hidden_dim // num_heads, f"rope_dim {rope_dim} is too large"
        self.rope_emb = TriangleRotaryEmbedding(dim=rope_dim, double_max_freq=rope_double_max_freq)
        self._cfg = _stack_config(latent_dim=hidden_dim, num_layers=num_layers, num_heads=num_heads,
                                  dim_feedforward=ffn_hidden_dim, dropout=0.0, view_transformer_latent_dim=hidden_dim,
                                  view_transformer_n_heads=num_heads)
        self._p_drop = dropout

    def forward(self, x, src_key_padding_mask=None, triangle_pos=None):
        _need_eval(self, self._p_drop)
        assert triangle_pos is not None, "triangle_pos must be provided if rope_dim is not None"
        eng = self._engine()
        B, Nt, d = x.shape
        Ntp = _rup(Nt, 8)
        dev = eng.device
        xs = torch.zeros((B, Ntp, d), dtype=torch.float32, device=dev)
        xs[:, :Nt] = x.to(dev, torch.float32)
        pos = torch.zeros((B, Ntp, 9), dtype=torch.float32, device=dev)
        pos[:, :Nt] = triangle_pos.to(dev, torch.float32)
        mask = torch.ones((B, Nt), dtype=torch.bool, device=dev) if src_key_padding_mask is None else src_key_padding_mask
        bits, words = _pack_key_mask(mask, B, Nt, dev)
        if words * 32 < Ntp or bits.shape[1] != 4 * ((Ntp + 127) // 128):
            raise RuntimeError("mask packing mismatch")
        out, _, _ = eng.encoder_layers(xs.view(B * Ntp, d), pos, bits, words, B, Ntp)
        return out.view(B, Ntp, d)[:, :Nt]


class TransformerDecoder(nn.Module, _EngineBacked):
    """layers/attention.py:593-688 on Engine.decoder_layers.  Every batch element is an independent (context,
    ray tokens) pair, as in the reference (the pipeline's fused path additionally shares the hoisted K/V of
    one scene between its views).  `ray_pos` must be zero (camera-space rays: the query RoPE is the identity)."""
    _parts, _prefix = ("decoder",), "view_transformer.transformer."

    def __init__(self, num_layers: int, num_heads: int, hidden_dim: int, ffn_hidden_dim: int,
                 ctx_dim: Optional[int] = None, dropout: float = 0.1, include_self_attn: bool = True,
                 use_swin_attn: bool = False, window_size: int = 8, shift_size: int = 4, activation: str = "gelu",
                 norm_first: bool = True, bias: bool = True, bias_kv: bool = False,
                 norm_type: Literal["layer_norm", "rms_norm"] = "layer_norm", qk_norm: bool = False,
                 rope_dim: Optional[int] = None,
                 rope_type: Literal["triangle", "triangle_learned", "triangle_mixed"] = "triangle",
                 rope_double_max_freq: bool = False):
        super().__init__()
        _check_stack_args(activation, norm_type, norm_first, bias, bias_kv, qk_norm, rope_type, rope_double_max_freq, rope_dim)
        if not include_self_attn or window_size != 8 or shift_size != 4:
            raise NotImplementedError("decoder kernels: self-attention after cross-attention, 8x8 windows shifted by 4")
        ctx_dim = hidden_dim if ctx_dim is None else ctx_dim
        self.head_dim = hidden_dim // num_heads
        self.layers = nn.ModuleList([
            AttentionLayer(query_dim=hidden_dim, kv_dim=ctx_dim, num_heads=num_heads, ffn_hidden_dim=ffn_hidden_dim,
                           dropout=dropout, bias=bias, bias_kv=bias_kv, activation=activation, norm_type=norm_type,
                           qk_norm=qk_norm, add_self_attn=include_self_attn, use_swin_attn=use_swin_attn,
                           window_size=window_size, shift_size=0 if i % 2 == 0 else shift_size)
            for i in range(num_layers)])
        self.rope_dim = rope_dim
        assert rope_dim % 2 == 0, "rope_dim must be even"
        assert rope_dim // 2 * 9 <= hidden_dim // num_heads, f"rope_dim {rope_dim} is too large"
        self.rope_emb = TriangleRotaryEmbedding(dim=rope_dim, double_max_freq=rope_double_max_freq)
        self._cfg = _stack_config(latent_dim=ctx_dim, num_heads=ctx_dim // 128, view_transformer_latent_dim=hidden_dim,
                                  view_transformer_n_heads=num_heads, view_transformer_n_layers=num_layers,
                                  view_transformer_ffn_hidden_dim=ffn_hidden_dim, dropout=0.0,
                                  view_transformer_use_swin_attn=use_swin_attn, num_register_tokens=0)
        self._p_drop = dropout

    def forward(self, x, ctx, src_key_padding_mask=None, triangle_pos=None, ray_pos=None, out_layers=[], tf32_mode=False,
                patch_h=None, patch_w=None):
        _need_eval(self, self._p_drop)
        assert triangle_pos is not None and ray_pos is not None, "triangle_pos and ray_pos must be provided"
        if bool((ray_pos != 0).any()):
            raise NotImplementedError("decoder kernels: ray_pos must be 0 (camera-space rays)")
        eng = self._engine()
        dev = eng.device
        BV, Nr, dv = x.shape
        Nt = ctx.shape[1]
        if patch_h is None or patch_w is None:
            patch_h = patch_w = int(round(math.sqrt(Nr)))
        if patch_h * patch_w != Nr:
            raise ValueError("patch_h * patch_w must equal the number of ray tokens")
        mask = torch.ones((BV, Nt), dtype=torch.bool, device=dev) if src_key_padding_mask is None else src_key_padding_mask
        st = eng.scene_state_from_tokens(ctx, None, mask)
        want = list(out_layers) if out_layers else [len(self.layers) - 1]
        outs = [[] for _ in want]
        for b in range(BV):
            xb = x[b].to(dev, torch.float32).contiguous().clone()
            pos = torch.zeros((1, st.Ntp, 9), dtype=torch.float32, device=dev)
            pos[0, :Nt] = triangle_pos[b].to(dev, torch.float32)
            feats = eng.decoder_layers(st, b, xb, pos, 1, patch_h, patch_w, out_layers=want, want_f32=True)
            for o, f in zip(outs, feats):
                o.append(f.view(1, Nr, dv))
        outs = [torch.cat(o, dim=0) for o in outs]
        return outs[0] if not out_layers else [[o] for o in outs]


class ResidualConvUnit(nn.Module):
    """layers/dpt.py:57-92 (parameter holder; the math runs inside DPTHead's fused conv chain)."""

    def __init__(self, features, activation=None):
        super().__init__()
        self.conv1 = nn.Conv2d(features, features, kernel_size=3, stride=1, padding=1, bias=True)
        self.conv2 = nn.Conv2d(features, features, kernel_size=3, stride=1, padding=1, bias=True)
        if activation is not None:  # same attribute path as the reference (:74); the kernels apply SiLU themselves
            self.activation = activation


class FeatureFusionBlock(nn.Module):
    """layers/dpt.py:95-159 (parameter holder)."""

    def __init__(self, features, no_resconv1: bool = False):
        super().__init__()
        self.out_conv = nn.Conv2d(features, features, kernel_size=1, stride=1, padding=0, bias=True)
        act = nn.SiLU(False)  # one instance per block, shared by its units (layers/dpt.py:128-129,162-171)
        if not no_resconv1:
            self.resConvUnit1 = ResidualConvUnit(features, act)
        self.resConvUnit2 = ResidualConvUnit(features, act)


class DPTHead(nn.Module, _EngineBacked):
    """layers/dpt.py:174-273 on Engine._dpt: NHWC fp16 implicit-GEMM convolutions (halo-tile tcgen05 kernel),
    ConvTranspose(k = s) as GEMM + pixel shuffle, align_corners bilinear kernels; returns the head's own
    output [B, out_dim, H, W] (before the ELU of ViewTransformer)."""
    _parts, _prefix = ("dpt",), "view_transformer.out_dpt."

    def __init__(self, in_channels, features=256, out_channels=[256, 512, 1024, 1024], out_dim=3):
        super().__init__()
        if out_dim != 3:
            raise NotImplementedError("DPT kernels: 3 output channels (include_alpha=False)")
        oc = list(out_channels)
        self.projects = nn.ModuleList([nn.Conv2d(in_channels, c, kernel_size=1) for c in oc])
        self.resize_layers = nn.ModuleList([
            nn.ConvTranspose2d(oc[0], oc[0], kernel_size=4, stride=4, padding=0),
            nn.ConvTranspose2d(oc[1], oc[1], kernel_size=2, stride=2, padding=0),
            nn.Identity(),
            nn.Conv2d(oc[3], oc[3], kernel_size=3, stride=2, padding=1)])
        self.scratch = nn.Module()
        for i, c in enumerate(oc):
            setattr(self.scratch, f"layer{i + 1}_rn", nn.Conv2d(c, features, kernel_size=3, stride=1, padding=1, bias=False))
        self.scratch.refinenet1 = FeatureFusionBlock(features)
        self.scratch.refinenet2 = FeatureFusionBlock(features)
        self.scratch.refinenet3 = FeatureFusionBlock(features)
        self.scratch.refinenet4 = FeatureFusionBlock(features, no_resconv1=True)
        self.scratch.output_conv1 = nn.Conv2d(features, features // 2, kernel_size=3, stride=1, padding=1)
        self.scratch.output_conv2 = nn.Sequential(nn.Conv2d(features // 2, 32, kernel_size=3, stride=1, padding=1),
                                                  nn.SiLU(True), nn.Conv2d(32, out_dim, kernel_size=1))
        self._cfg = _stack_config(view_transformer_latent_dim=in_channels, view_transformer_n_heads=in_channels // 128,
                                  dpt_features=features, dpt_out_channels=oc)

    def forward(self, out_features, patch_h, patch_w, patch_size=16):
        if patch_size != 8:
            raise NotImplementedError("DPT kernels: patch_size 8 (the final resize is then the identity, SURVEY E2)")
        eng = self._engine()
        feats = [f[0] if isinstance(f, (list, tuple)) else f for f in out_features]
        B, n, dv = feats[0].shape
        f16 = []
        for f in feats:
            f32 = f.to(eng.device, torch.float32).contiguous().view(B * n, dv)
            f16.append(ops.cast(f32, torch.empty((B * n, dv), dtype=torch.float16, device=eng.device)))
        raw = eng._dpt(f16, B, patch_h, patch_w, raw_out=True)  # [B, H, W, 3]
        return raw.permute(0, 3, 1, 2)


class ViewTransformer(nn.Module, _EngineBacked):
    """models/view_transformer.py:12-127: ray map -> 8x8 patch tokens -> decoder (cross-attention to the
    triangle tokens, swin / full self-attention, SwiGLU) -> DPT head -> ELU; returns the log-encoded image
    [B, 3, H, W] (H != W within the size rules of config.view_grid).  One Engine call per batch element
    (Engine.render_views with an explicit ray map)."""
    _parts, _prefix = ("ray", "decoder", "dpt"), "view_transformer."

    def __init__(self, config: RenderFormerConfig):
        super().__init__()
        config.check_supported()
        self.config = config
        self.rope_dim = config.view_rope_dim
        dv = config.view_transformer_latent_dim
        self.ray_map_patch_token = nn.Parameter(torch.randn(1, 1, dv))
        self.vdir_pe = NeRFEncoding(in_dim=3, num_frequencies=config.vdir_num_freqs, include_input=True)
        self.ray_map_encoder = nn.Linear(self.vdir_pe.get_out_dim() * config.patch_size ** 2, dv)
        self.ray_map_encoder_norm = nn.RMSNorm(dv)
        self.transformer = TransformerDecoder(
            num_layers=config.view_transformer_n_layers, num_heads=config.view_transformer_n_heads, hidden_dim=dv,
            ctx_dim=config.latent_dim, ffn_hidden_dim=config.view_transformer_ffn_hidden_dim, dropout=config.dropout,
            activation=config.activation, norm_type=config.norm_type, norm_first=config.norm_first,
            rope_dim=self.rope_dim, rope_type=config.rope_type, rope_double_max_freq=config.rope_double_max_freq,
            qk_norm=config.qk_norm, bias=config.bias, include_self_attn=config.view_transformer_include_self_attn,
            use_swin_attn=config.view_transformer_use_swin_attn)
        self.out_dpt = DPTHead(in_channels=dv, features=config.dpt_features, out_channels=config.dpt_out_channels, out_dim=3)
        self.out_layers = config.out_layers
        self.out_proj_act = nn.ELU(alpha=1e-3)
        self._cfg = config

    def forward(self, camera_o, ray_map, tri_tokens, tri_pos, valid_mask, tf32_mode=False):
        if bool((camera_o != 0).any()):
            raise NotImplementedError("view-stage kernels: camera_o must be 0 (camera-space rays)")
        eng = self._engine()
        B, H, W = ray_map.shape[0], ray_map.shape[1], ray_map.shape[2]
        st = eng.scene_state_from_tokens(tri_tokens, None, valid_mask)
        imgs = [eng.render_views(st, b, None, None, (H, W), rays_d=ray_map[b:b + 1], pos_cam=tri_pos[b:b + 1])
                for b in range(B)]
        hdr = torch.cat(imgs, dim=0)                      # [B, H, W, 3] = 10^elu(head) - 1
        return torch.log10(hdr + 1.0).permute(0, 3, 1, 2)  # back to what the reference returns (elu(head))
