"""Host-side schedule of the RenderFormer forward pass on the sm_100a kernels.

Two stages, mirroring the reference's structure (models/renderformer.py:171-206):

* `encode_scene`  -- view-independent: token construction + triangle-token encoder, run once
  per scene; additionally hoists the decoder's per-layer K / V projections of the triangle
  tokens, which do not depend on the view (SURVEY §0.8, Appendix E5).
* `render_views`  -- view-dependent: ray-bundle tokens, decoder (cross-attention to the hoisted
  K/V with per-view K RoPE, swin or full self-attention, SwiGLU), DPT head, HDR decode.

All math runs in the C-ABI kernels (ops.py); torch provides buffers and streams only.
Precision policy: fp32 residual stream, bf16 tensor-core operands in the transformer stacks,
fp16 operands in the token encoders and the DPT head, fp32 accumulation / softmax / norms.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Callable, Dict, List, Optional

import torch

from . import lib as L
from . import ops
from .config import RenderFormerConfig, view_grid

EPS = 1e-6  # reference: layers/attention.py:16


def _rup(x: int, m: int) -> int:
    return (x + m - 1) // m * m


@dataclass
class SceneState:
    """Per-scene device state handed from the view-independent to the view-dependent stage."""
    B: int
    N: int
    Nt: int
    Ntp: int
    seq: torch.Tensor        # fp32 [B, Ntp, d]
    tri: torch.Tensor        # fp32 [B, N, 9]
    mask_u8: torch.Tensor    # uint8 [B, N]
    mask_bits: torch.Tensor  # int32 [B, words]
    k_all: torch.Tensor      # fp32 [B, Ntp, L*dv]: hoisted decoder K of every layer (pre-QK-norm, pre-RoPE)
    v_all: torch.Tensor      # bf16 [B, L*dv, Ntp]: hoisted decoder V of every layer, transposed

    dv: int = 0              # decoder width (columns of one layer inside k_all / rows inside v_all)
    static: bool = False     # buffers persist across calls (CUDA-graph output / broadcast receive buffer)

    def k_pre(self, layer: int, b: int) -> torch.Tensor:
        """fp32 [Ntp, dv] view (row stride L*dv)."""
        return self.k_all[b, :, layer * self.dv:(layer + 1) * self.dv]

    def v_t(self, layer: int, b: int) -> torch.Tensor:
        """bf16 [dv, Ntp] contiguous view."""
        return self.v_all[b, layer * self.dv:(layer + 1) * self.dv]

    def tensors(self):
        return [self.seq, self.tri, self.mask_u8, self.mask_bits, self.k_all, self.v_all]

    @property
    def complete(self) -> bool:
        """False when `seq` holds only this rank's rows (row-sharded encode without `gather_seq`)."""
        return self.seq is not None and self.seq.shape[1] == self.Ntp


@dataclass
class RowShard:
    """Partition of the triangle-token rows of the view-independent stage over `world` ranks.

    Rank r owns the contiguous rows [r*S, (r+1)*S) of the (padded) token sequence, S = shard_rows().
    Everything that is row-local (token construction, attention queries, out-projection, SwiGLU) runs
    on the own rows only; what every rank needs of the others -- the 16-bit copy of the residual stream
    and its row sums of squares, i.e. the input of the next layer's K / V projection -- is exchanged
    with ONE all-gather per layer: `all_gather(full, chunk)` fills `full` ([world*S, ld] contiguous)
    from every rank's `chunk` (= full[rank*S:(rank+1)*S], written in place).  The reference has no
    counterpart (single device, models/renderformer.py:171-206); SURVEY §8(e) derives the scheme."""
    rank: int
    world: int
    all_gather: Callable[[torch.Tensor, torch.Tensor], None]
    # optional (renderformer_b200.dist.SymmKVStore): kv_store(rows, width, dtype, device) -> peer-mapped, double-
    # buffered [k | v] row store.  With it the per-layer all-gather disappears: the kernel that produces a rank's
    # k | v rows stores them straight into every rank's memory (NVLS multicast or peer stores over NVLink,
    # rfb_qkv_post) and the ranks meet at a signal-pad barrier before the attention reads them.
    kv_store: Optional[Callable] = None

    def shard_rows(self, ntp: int) -> int:
        return _rup(-(-ntp // self.world), 8)

    def my_rows(self, ntp: int):
        s = self.shard_rows(ntp)
        r0 = min(self.rank * s, ntp)
        return r0, min(r0 + s, ntp)


def swin_window_maps(Hp: int, Wp: int, shift: int, ws: int = 8):
    """Window-order -> token-order permutation and shifted-window region ids.

    Row w of the window-major layout holds token perm[w] of the row-major (Hp x Wp) grid, i.e.
    torch.roll(-shift) followed by window_partition (layers/attention.py:205-218,334-339); region
    ids are the closed form of get_swin_attn_mask (:238-271, SURVEY Appendix E3)."""
    w = torch.arange(Hp * Wp)
    win, p = w // (ws * ws), w % (ws * ws)
    ry = (win // (Wp // ws)) * ws + p // ws
    rx = (win % (Wp // ws)) * ws + p % ws
    perm = ((ry + shift) % Hp) * Wp + (rx + shift) % Wp
    if shift > 0:
        def rid(r, n):
            return (r >= n - ws).long() + (r >= n - shift).long()
        region = 3 * rid(ry, Hp) + rid(rx, Wp)
    else:
        region = torch.zeros_like(w)
    return perm.to(torch.int32), region.to(torch.uint8)


ALL_PARTS = ("tokens", "ray", "encoder", "decoder", "dpt")


class Engine:
    def __init__(self, cfg: RenderFormerConfig, state_dict: Dict[str, torch.Tensor], device, parts=ALL_PARTS,
                 op_dtype: torch.dtype = torch.bfloat16):
        """`parts`: which sections of the state_dict are laid out for the kernels -- the whole model for
        the pipeline; a single section when one of the reference's sub-modules (renderformer.layers.*,
        ViewTransformer, DPTHead) is called on its own (renderformer_b200/modules.py).
        `op_dtype`: tensor-core operand format of the two transformer stacks, torch.bfloat16 or torch.float16
        (same tcgen05 rate; fp16 has 3 more mantissa bits: ~8x less rounding noise, DESIGN.md §3).  Token
        encoders and the DPT head always use fp16 operands."""
        cfg.check_supported()
        if op_dtype not in (torch.bfloat16, torch.float16):
            raise ValueError("op_dtype must be torch.bfloat16 or torch.float16")
        self.cfg = cfg
        self.op = op_dtype
        self.parts = tuple(parts)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.RfbError("renderformer_b200.Engine needs a CUDA device (there is no CPU fallback)")
        L.load()
        # RMSNorm is fused into the GEMMs (norm weights folded into the next projection, 1/rms applied
        # in its epilogue from partial sums of squares left by the residual GEMMs) in the scene stage
        # and in the swin decoder; the full-attention decoder (V1-Base) keeps explicit norm kernels.
        self.fused_dec = bool(cfg.view_transformer_use_swin_attn)
        self.w: Dict[str, torch.Tensor] = {}
        self._maps: Dict[tuple, tuple] = {}
        self._prepare(state_dict)

    # ------------------------------------------------------------------ weights
    def _prepare(self, sd: Dict[str, torch.Tensor]) -> None:
        cfg, dev = self.cfg, self.device
        bf, hf = self.op, torch.float16

        def g(k):
            return sd[k].detach().to(dev, torch.float32)

        def put(name, t, dt=None):
            self.w[name] = (t if dt is None else t.to(dt)).contiguous()

        def swiglu_w(p):
            w1, w3 = g(p + "w1.weight"), g(p + "w3.weight")
            f, d = w1.shape
            return torch.stack([w1.view(f // 16, 16, d), w3.view(f // 16, 16, d)], dim=1).reshape(2 * f, d)

        def conv_w(k):  # [Co, Ci, 3, 3] -> [Co, (ky*3+kx)*Ci + ci]
            w = g(k)
            return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1)

        def fold(wt, norm_key, on=True):  # RMSNorm(x) W^T = r * x (W . w)^T : fold the norm weight along K
            return wt * g(norm_key)[None, :] if on else wt

        fused_dec = self.fused_dec

        d = cfg.latent_dim
        if "tokens" in self.parts:
            self._prepare_tokens(g, put, d)
        if "ray" in self.parts:
            self._prepare_ray(g, put)
        if "encoder" in self.parts:
            self._prepare_encoder(g, put, fold, swiglu_w)
        if "decoder" in self.parts:
            self._prepare_decoder(g, put, fold, swiglu_w)
        if "dpt" in self.parts:
            self._prepare_dpt(g, put, conv_w)

    def _prepare_tokens(self, g, put, d):
        cfg, dev = self.cfg, self.device
        hf = torch.float16
        put("tri_token", g("tri_token").reshape(-1))
        put("reg_tokens", g("reg_tokens").reshape(cfg.num_register_tokens, d))
        vw = g("vn_encoding_proj.weight")
        self.vn_ld = _rup(vw.shape[1], 64)
        vwp = torch.zeros((d, self.vn_ld), device=dev)
        vwp[:, : vw.shape[1]] = vw
        put("vn.w", vwp, hf), put("vn.b", g("vn_encoding_proj.bias")), put("vn.norm", g("vn_encoder_norm.weight"))
        put("tex.w", g("texture_encoder.weight"), hf), put("tex.b", g("texture_encoder.bias"))
        # constant-texture fast path: texels of one channel share one value inside the triangular
        # texel mask x + y <= P, so the projection reduces to the texel-summed weight [d, channels]
        P_, C_ = cfg.texture_encode_patch_size, cfg.texture_channels
        ii = torch.arange(P_, device=dev)
        tmask = (ii[:, None] + ii[None, :] <= P_).to(torch.float32)
        wr = (g("texture_encoder.weight").view(d, C_, P_, P_) * tmask).sum(dim=(2, 3))
        self.texc_ld = _rup(C_, 16)
        wrp = torch.zeros((d, self.texc_ld), device=dev)
        wrp[:, :C_] = wr
        put("tex.wr", wrp, hf)
        put("tex.norm", g("texture_encoder_norm.weight"))

    def _prepare_ray(self, g, put):
        hf = torch.float16
        v = "view_transformer."
        put("ray.token", g(v + "ray_map_patch_token").reshape(-1))
        put("ray.w", g(v + "ray_map_encoder.weight"), hf), put("ray.b", g(v + "ray_map_encoder.bias"))
        put("ray.norm", g(v + "ray_map_encoder_norm.weight"))

    def _prepare_encoder(self, g, put, fold, swiglu_w):
        cfg = self.cfg
        bf = self.op
        put("enc.freqs", g("transformer.rope_emb.freqs"))
        for i in range(cfg.num_layers):
            p, o = f"transformer.layers.{i}.", f"enc{i}."
            w_in = fold(g(p + "multihead_attn.in_proj.weight"), p + "query_norm.weight")
            put(o + "wqkv", w_in, bf)  # one GEMM: q | k to fp32, v transposed (vt_out)
            put(o + "wo", g(p + "multihead_attn.out_proj.weight"), bf)
            put(o + "qkn", torch.cat([g(p + "multihead_attn.q_norm.weight"), g(p + "multihead_attn.k_norm.weight")]))
            put(o + "w13", fold(swiglu_w(p + "ffn."), p + "ffn_norm.weight"), bf)
            put(o + "w2", g(p + "ffn.w2.weight"), bf)

    def _prepare_decoder(self, g, put, fold, swiglu_w):
        cfg = self.cfg
        bf = self.op
        fused_dec = self.fused_dec
        v = "view_transformer."
        dv = cfg.view_transformer_latent_dim
        put("dec.freqs", g(v + "transformer.rope_emb.freqs"))
        for i in range(cfg.view_transformer_n_layers):
            p, o = v + f"transformer.layers.{i}.", f"dec{i}."
            put(o + "wq", fold(g(p + "multihead_attn.q_proj.weight"), p + "query_norm.weight", fused_dec), bf)
            put(o + "wk", fold(g(p + "multihead_attn.k_proj.weight"), p + "kv_norm.weight"), bf)
            put(o + "wv", fold(g(p + "multihead_attn.v_proj.weight"), p + "kv_norm.weight"), bf)
            put(o + "wout", g(p + "multihead_attn.out_proj.weight"), bf)
            put(o + "qn", g(p + "multihead_attn.q_norm.weight")), put(o + "kn", g(p + "multihead_attn.k_norm.weight"))
            put(o + "n_q", g(p + "query_norm.weight"))
            w_in = fold(g(p + "self_attn.in_proj.weight"), p + "self_attn_norm.weight", fused_dec)
            if fused_dec:
                put(o + "s.wqkv", w_in, bf)
            else:
                put(o + "s.wqk", w_in[: 2 * dv], bf), put(o + "s.wv", w_in[2 * dv:], bf)
            put(o + "s.wo", g(p + "self_attn.out_proj.weight"), bf)
            put(o + "s.qkn", torch.cat([g(p + "self_attn.q_norm.weight"), g(p + "self_attn.k_norm.weight")]))
            put(o + "n_s", g(p + "self_attn_norm.weight")), put(o + "n_f", g(p + "ffn_norm.weight"))
            put(o + "w13", fold(swiglu_w(p + "ffn."), p + "ffn_norm.weight", fused_dec), bf)
            put(o + "w2", g(p + "ffn.w2.weight"), bf)

        Lv = cfg.view_transformer_n_layers
        put("dec.kn_all", torch.cat([self.w.pop(f"dec{i}.kn") for i in range(Lv)], dim=0))
        put("dec.wkv_all", torch.cat([self.w.pop(f"dec{i}.wk") for i in range(Lv)] +
                                     [self.w.pop(f"dec{i}.wv") for i in range(Lv)], dim=0))

    def _prepare_dpt(self, g, put, conv_w):
        hf = torch.float16
        h = "view_transformer.out_dpt."
        for i in range(4):
            put(f"dpt.proj{i}.w", g(h + f"projects.{i}.weight").flatten(1), hf)
            put(f"dpt.proj{i}.b", g(h + f"projects.{i}.bias"))
            put(f"dpt.rn{i}.w", conv_w(h + f"scratch.layer{i + 1}_rn.weight"), hf)
        for i, s in ((0, 4), (1, 2)):  # ConvTranspose2d(k = s): [Ci, Co, s, s] -> [(i*s+j)*Co + co, ci]
            w = g(h + f"resize_layers.{i}.weight")
            put(f"dpt.up{i}.w", w.permute(2, 3, 1, 0).reshape(s * s * w.shape[1], w.shape[0]), hf)
            put(f"dpt.up{i}.b", g(h + f"resize_layers.{i}.bias").repeat(s * s))
        put("dpt.down3.w", conv_w(h + "resize_layers.3.weight"), hf), put("dpt.down3.b", g(h + "resize_layers.3.bias"))
        for r in (1, 2, 3, 4):
            p = h + f"scratch.refinenet{r}."
            put(f"dpt.rf{r}.out.w", g(p + "out_conv.weight").flatten(1), hf), put(f"dpt.rf{r}.out.b", g(p + "out_conv.bias"))
            for u in ((1, 2) if r != 4 else (2,)):
                for c in (1, 2):
                    put(f"dpt.rf{r}.u{u}c{c}.w", conv_w(p + f"resConvUnit{u}.conv{c}.weight"), hf)
                    put(f"dpt.rf{r}.u{u}c{c}.b", g(p + f"resConvUnit{u}.conv{c}.bias"))
        put("dpt.oc1.w", conv_w(h + "scratch.output_conv1.weight"), hf), put("dpt.oc1.b", g(h + "scratch.output_conv1.bias"))
        put("dpt.oc2.w", conv_w(h + "scratch.output_conv2.0.weight"), hf), put("dpt.oc2.b", g(h + "scratch.output_conv2.0.bias"))
        put("dpt.oc3.w", g(h + "scratch.output_conv2.2.weight").flatten(1)), put("dpt.oc3.b", g(h + "scratch.output_conv2.2.bias"))

    def _e(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    # ------------------------------------------------------------------ shared blocks
    def _ffn(self, x, rows, d, n_w, w13, w2):
        """x += w2(silu(w1 n(x)) * w3 n(x))   layers/attention.py:56-57,526."""
        h = ops.rmsnorm(x, n_w, self._e((rows, d), self.op), rows=rows, d=d, eps=EPS)
        g = ops.gemm(h, w13, epi=L.EPI_SWIGLU, out_dtype=self.op)
        ops.gemm(g, w2, out=x, res1=x)

    # ------------------------------------------------------------------ stage 1
    @torch.no_grad()
    def encode_scene(self, triangles, texture, mask, vn, texture_is_log: bool = False,
                     shard: Optional[RowShard] = None, texture_own_rows: bool = False,
                     taps: Optional[dict] = None, gather_seq: bool = False) -> SceneState:
        """View-independent stage.  With `shard` (multi-GPU) every rank passes the same scene and runs
        the row-sharded schedule `_encode_scene_sharded`; every rank returns the complete SceneState.
        `texture_own_rows`: `texture` holds only the triangles of this rank's rows
        (`own_triangles(N, shard)`), so a rank never has to upload the other ranks' texels.
        `gather_seq`: also all-gather the fp32 token sequence `SceneState.seq` (nothing downstream needs it: the
        view stage reads the hoisted K / V; without it `seq` holds this rank's own rows only)."""
        cfg, w, dev = self.cfg, self.w, self.device
        if shard is not None and shard.world > 1:
            B = triangles.shape[0]
            sts = [self._encode_scene_sharded(triangles[b:b + 1], texture[b:b + 1], mask[b:b + 1], vn[b:b + 1],
                                              texture_is_log, shard, texture_own_rows, gather_seq) for b in range(B)]
            if B == 1:
                return sts[0]
            cat = [torch.cat(ts, dim=0) for ts in zip(*(st.tensors() for st in sts))]
            return SceneState(B, sts[0].N, sts[0].Nt, sts[0].Ntp, *cat, sts[0].dv)
        x, pos, bits, words, (B, N, Nt, Ntp), tri, mask_u8 = self.construct_seq(triangles, texture, mask, vn, texture_is_log)
        return self._encode_fused(x, pos, bits, words, B, N, Nt, Ntp, tri, mask_u8, taps)

    def construct_seq(self, triangles, texture, mask, vn, texture_is_log: bool = False):
        """RenderFormer.construct_seq + process_tri_vpos_list (models/renderformer.py:103-169): token rows
        x fp32 [B*Ntp, d] (16 register tokens, then tri_token + RMSNorm(texture emb) + RMSNorm(normal emb);
        rows padded to a multiple of 8 with zeros), RoPE positions pos [B, Ntp, 9] (masked centroid for the
        register rows), packed key mask bits [B, words]."""
        cfg, w, dev = self.cfg, self.w, self.device
        B, N = triangles.shape[:2]
        d = cfg.latent_dim
        nreg = cfg.num_register_tokens
        Nt, Ntp = N + nreg, _rup(N + nreg, 8)
        tri = triangles.reshape(B, N, 9).to(dev, torch.float32).contiguous()
        vn9 = vn.reshape(B, N, 9).to(dev, torch.float32).contiguous()
        tex = texture.to(dev, torch.float32).contiguous()
        const_tex = tex.dim() == 3  # [B, N, channels]: per-triangle constants (scene_io / to_h5 scenes)
        mask_u8 = mask.to(dev).contiguous().view(torch.uint8) if mask.dtype == torch.bool else mask.to(dev, torch.uint8)
        C_, P = cfg.texture_channels, cfg.texture_encode_patch_size

        log_ch = 0 if (cfg.use_ldr or texture_is_log) else 3
        if const_tex:
            if tex.shape[2] != C_:
                raise ValueError(f"constant texture must be [B, N, {C_}], got {tuple(tex.shape)}")
            tex16 = ops.texture_const_prep(tex, self._e((B * N, self.texc_ld), torch.float16), n_tris=B * N,
                                           channels=C_, ld=self.texc_ld, log_channels=log_ch)
            tex_lin = ops.gemm(tex16, w["tex.wr"], bias=w["tex.b"], out_dtype=torch.float32)
        else:
            tex16 = ops.texture_prep(tex, self._e((B * N, C_ * P * P), torch.float16), n_tris=B * N, channels=C_,
                                     texels=P * P, log_channels=log_ch)
            tex_lin = ops.gemm(tex16, w["tex.w"], bias=w["tex.b"], out_dtype=torch.float32)
        del tex16
        vn16 = ops.vn_encode(vn9, self._e((B * N, self.vn_ld), torch.float16), n=B * N, nfreq=cfg.vn_pe_num_freqs,
                             ld=self.vn_ld)
        vn_lin = ops.gemm(vn16, w["vn.w"], bias=w["vn.b"], out_dtype=torch.float32)
        x = self._e((B * Ntp, d), torch.float32)
        ops.token_assemble(tex_lin, w["tex.norm"], vn_lin, w["vn.norm"], w["tri_token"], w["reg_tokens"], x,
                           n_prefix=nreg, rows_in=N, rows_out=Ntp, batch=B, d=d)
        pos = self._e((B, Ntp, 9), torch.float32)
        for b in range(B):
            ops.positions(tri[b], mask_u8[b], None, pos[b], n=N, n_reg=nreg, rows_out=Ntp, n_views=1)
        words = 4 * ((Ntp + 127) // 128)
        bits = ops.pack_mask(mask_u8, self._e((B, words), torch.int32), n=N, n_prefix=nreg, words=words, batch=B)
        return x, pos, bits, words, (B, N, Nt, Ntp), tri, mask_u8

    def _encode_fused(self, x, pos, bits, words, B, N, Nt, Ntp, tri, mask_u8, taps=None) -> SceneState:
        """Encoder + K/V hoist with RMSNorm fused into the GEMMs."""
        x, xb, xsq = self.encoder_layers(x, pos, bits, words, B, Ntp, taps)
        k_all, v_all = self.hoist_kv(xb, xsq, B, Ntp)
        return SceneState(B, N, Nt, Ntp, x.view(B, Ntp, self.cfg.latent_dim), tri, mask_u8, bits, k_all, v_all,
                          self.cfg.view_transformer_latent_dim)

    @staticmethod
    def enc_kv_split_tiles(Ntp: int) -> int:
        """Key-chunk length (in 128-key tiles) of the encoder's self-attention; 0 = no split.  Chunks of about 11
        tiles, at most 4: the chunks run on separate CTAs, which is what keeps the SMs busy when a rank of the
        row-sharded schedule holds a few hundred query rows.  A function of the key count ONLY, so that every
        schedule (one GPU or N ranks) does the same arithmetic per row."""
        n_tiles = (Ntp + 127) // 128
        splits = max(1, min(4, n_tiles // 11))
        return 0 if splits == 1 else -(-n_tiles // splits)

    def encoder_layers(self, x, pos, bits, words, B, Ntp, taps=None):
        """TransformerEncoder.forward (layers/attention.py:579-590) on x fp32 [B*Ntp, d] (updated in place),
        pos [B, Ntp, 9], packed key mask `bits` [B, words].  State carried between GEMMs: x (fp32 residual),
        xb (bf16 copy of x), xsq (per-row partial sums of squares of x, one per 128 columns); returns all
        three."""
        cfg, w = self.cfg, self.w
        d, H = cfg.latent_dim, cfg.num_heads
        rows = B * Ntp
        bf, f32 = self.op, torch.float32
        nrm = dict(norm_dim=d, norm_eps=EPS)
        P = d // 128
        xb, xsq = self._e((rows, d), bf), self._e((rows, P), f32)
        xb2, xsq2 = self._e((rows, d), bf), self._e((rows, P), f32)
        ops.rowstat(x, xb, xsq, rows=rows, d=d)
        if taps is not None:  # per-layer (16-bit stream, row sums) snapshots: what the sharded schedule all-gathers
            taps.setdefault("enc_stream", []).append((xb.clone(), xsq.clone()))
        kst = self.enc_kv_split_tiles(Ntp)
        ws = self._e((max(ops.attention_ws_elems(B, H, Ntp, Ntp, kst), 1),), f32) if kst else None
        for i in range(cfg.num_layers):
            o = f"enc{i}."
            vt = self._e((B, d, Ntp), bf)
            qk = ops.gemm(xb, w[o + "wqkv"], out=self._e((rows, 2 * d), f32), in_sumsq=xsq, vt_out=vt, vt_split=2 * d,
                          vt_rows_per_batch=Ntp, **nrm)
            qkr = ops.qknorm_rope(qk, w[o + "qkn"], self._e((rows, 2 * d), bf), rows=rows, d=d, nseg=2,
                                  ldx=2 * d, ldo=2 * d, pos=pos, freqs=w["enc.freqs"], eps=EPS)
            if taps is not None:  # per-layer 16-bit K (after QK-norm + RoPE) and V^T: what the sharded schedule gathers
                taps.setdefault("enc_kv", []).append((qkr[:, d:].clone(), vt.clone()))
            att = self._e((rows, d), bf)
            ops.attention(qkr, qkr[:, d:], vt, att, B=B, H=H, Nq=Ntp, Nk=Ntp, ldq=2 * d, ldk=2 * d, ldvt=Ntp, ldo=d,
                          q_bs=Ntp * 2 * d, k_bs=Ntp * 2 * d, vt_bs=d * Ntp, o_bs=Ntp * d, mask_bits=bits,
                          mask_bs=words, kv_split_tiles=kst, split_ws=ws)
            ops.gemm(att, w[o + "wo"], out=x, res1=x, out_sumsq=xsq2, out16=xb2)
            g = ops.gemm(xb2, w[o + "w13"], epi=L.EPI_SWIGLU, out_dtype=bf, in_sumsq=xsq2, **nrm)
            ops.gemm(g, w[o + "w2"], out=x, res1=x, out_sumsq=xsq, out16=xb)
            if taps is not None:
                taps["enc_stream"].append((xb.clone(), xsq.clone()))
        return x, xb, xsq

    def hoist_kv(self, xb, xsq, B, Ntp):
        """Decoder K / V projections of the triangle tokens for ALL layers in one GEMM (view independent,
        SURVEY E5; every layer's kv_norm weight is folded into its rows): k_all fp32 [B, Ntp, L*dv]
        (pre-QK-norm, pre-RoPE), v_all bf16 [B, L*dv, Ntp] (transposed)."""
        cfg, w = self.cfg, self.w
        d, dv, Lv = cfg.latent_dim, cfg.view_transformer_latent_dim, cfg.view_transformer_n_layers
        v_all = self._e((B, Lv * dv, Ntp), self.op)
        k_all = ops.gemm(xb, w["dec.wkv_all"], out=self._e((B * Ntp, Lv * dv), torch.float32), in_sumsq=xsq,
                         vt_out=v_all, vt_split=Lv * dv, vt_rows_per_batch=Ntp, norm_dim=d, norm_eps=EPS)
        return k_all.view(B, Ntp, Lv * dv), v_all

    def scene_state_from_tokens(self, seq, tri_pos_world, mask) -> SceneState:
        """SceneState from ready-made encoder output `seq` [B, Nt, d] (ViewTransformer / TransformerDecoder
        called on their own, models/view_transformer.py:88): rows are padded to a multiple of 8, the decoder
        K / V are hoisted.  `mask` [B, Nt] bool over ALL tokens (register prefix included)."""
        cfg = self.cfg
        B, Nt, d = seq.shape
        Ntp = _rup(Nt, 8)
        dev = self.device
        x = torch.zeros((B, Ntp, d), dtype=torch.float32, device=dev)
        x[:, :Nt] = seq.to(dev, torch.float32)
        P = d // 128
        xb, xsq = self._e((B * Ntp, d), self.op), self._e((B * Ntp, P), torch.float32)
        ops.rowstat(x.view(B * Ntp, d), xb, xsq, rows=B * Ntp, d=d)
        k_all, v_all = self.hoist_kv(xb, xsq, B, Ntp)
        m8 = mask.to(dev).contiguous().view(torch.uint8) if mask.dtype == torch.bool else mask.to(dev, torch.uint8)
        words = 4 * ((Ntp + 127) // 128)
        bits = ops.pack_mask(m8, self._e((B, words), torch.int32), n=Nt, n_prefix=0, words=words, batch=B)
        nreg = cfg.num_register_tokens
        return SceneState(B, Nt - nreg, Nt, Ntp, x, None, m8[:, nreg:].contiguous(), bits, k_all, v_all,
                          cfg.view_transformer_latent_dim)

    def own_triangles(self, N: int, sh: RowShard):
        """[t0, t1): the triangles whose token rows rank `sh.rank` owns."""
        nreg = self.cfg.num_register_tokens
        r0, r1 = sh.my_rows(_rup(N + nreg, 8))
        return min(max(r0 - nreg, 0), N), min(max(r1 - nreg, 0), N)

    def _encode_scene_sharded(self, triangles, texture, mask, vn, texture_is_log, sh: RowShard,
                              texture_own_rows: bool = False, gather_seq: bool = False) -> SceneState:
        """One scene, token rows split over the ranks of `sh` (see RowShard).  Per layer and rank: ONE fused
        [q|k|v] projection of the OWN rows, `rfb_qkv_post` (QK-norm + RoPE of q and k, cast of v) which writes the
        16-bit [k | v] rows into the layer's row store -- with `sh.kv_store` straight into EVERY rank's store (NVLS
        multicast or peer stores: the all-gather is fused into the producer) followed by a barrier, otherwise into the
        local buffer followed by one all-gather (16.8 MB for 4096 triangles) -- a local transpose of V, key-split
        attention of the own query rows against all keys, out-projection + SwiGLU on the own rows.  Nothing is
        computed twice; after the last layer one more gather collects the 16-bit stream + row sums that the hoisted
        decoder K / V are projected from (replicated: 0.2 TFLOP is cheaper than moving the 300 MB result).  The
        arithmetic of a row does not depend on which rank owns it or how many rows a launch holds: the result is
        bit-identical to the single-GPU schedule (tests/test_dist_gpu.py)."""
        cfg, w, dev = self.cfg, self.w, self.device
        N = triangles.shape[1]
        d, H, dv = cfg.latent_dim, cfg.num_heads, cfg.view_transformer_latent_dim
        nreg = cfg.num_register_tokens
        Nt, Ntp = N + nreg, _rup(N + nreg, 8)
        bf, f32, hf = self.op, torch.float32, torch.float16
        S = sh.shard_rows(Ntp)
        r0, r1 = sh.my_rows(Ntp)
        rows = r1 - r0
        P = d // 128
        ldx = _rup(d + 2 * P, 8)                       # bf16 elements per gathered row
        tri = triangles.reshape(1, N, 9).to(dev, f32).contiguous()
        vn9 = vn.reshape(1, N, 9).to(dev, f32).contiguous()
        mask_u8 = mask.to(dev).contiguous().view(torch.uint8) if mask.dtype == torch.bool else mask.to(dev, torch.uint8)
        C_, Pt = cfg.texture_channels, cfg.texture_encode_patch_size
        const_tex = texture.dim() == 3
        log_ch = 0 if (cfg.use_ldr or texture_is_log) else 3

        # ---- token construction of the own rows (models/renderformer.py:126-169)
        t0, t1 = self.own_triangles(N, sh)                          # own triangles
        nt = t1 - t0
        p_own = max(0, min(r1, nreg) - r0)                          # register-token rows inside the own range
        x = self._e((max(rows, 1), d), f32)
        if rows > 0:
            if nt > 0:
                tex = (texture[0] if texture_own_rows else texture[0, t0:t1]).to(dev, f32).contiguous()
                if tex.shape[0] != nt:
                    raise ValueError(f"texture holds {tex.shape[0]} triangles, this rank owns {nt}")
                if const_tex:
                    if tex.shape[1] != C_:
                        raise ValueError(f"constant texture must be [B, N, {C_}], got {tuple(texture.shape)}")
                    tex16 = ops.texture_const_prep(tex, self._e((nt, self.texc_ld), hf), n_tris=nt, channels=C_,
                                                   ld=self.texc_ld, log_channels=log_ch)
                    tex_lin = ops.gemm(tex16, w["tex.wr"], bias=w["tex.b"], out_dtype=f32)
                else:
                    tex16 = ops.texture_prep(tex, self._e((nt, C_ * Pt * Pt), hf), n_tris=nt, channels=C_,
                                             texels=Pt * Pt, log_channels=log_ch)
                    tex_lin = ops.gemm(tex16, w["tex.w"], bias=w["tex.b"], out_dtype=f32)
                del tex16, tex
                vn16 = ops.vn_encode(vn9[0, t0:t1], self._e((nt, self.vn_ld), hf), n=nt, nfreq=cfg.vn_pe_num_freqs,
                                     ld=self.vn_ld)
                vn_lin = ops.gemm(vn16, w["vn.w"], bias=w["vn.b"], out_dtype=f32)
            else:
                tex_lin = vn_lin = w["tri_token"]  # never dereferenced (rows_in = 0)
            ops.token_assemble(tex_lin, w["tex.norm"], vn_lin, w["vn.norm"], w["tri_token"],
                               w["reg_tokens"][r0:] if p_own > 0 else None, x, n_prefix=p_own, rows_in=nt,
                               rows_out=rows, batch=1, d=d)
        pos = ops.positions(tri[0], mask_u8[0], None, self._e((Ntp, 9), f32), n=N, n_reg=nreg, rows_out=Ntp, n_views=1)
        words = 4 * ((Ntp + 127) // 128)
        bits = ops.pack_mask(mask_u8, self._e((1, words), torch.int32), n=N, n_prefix=nreg, words=words, batch=1)

        # ---- per layer every rank projects, normalises and rotates ITS rows, then ONE all-gather moves the 16-bit
        # [k | v] rows of all ranks (row r of `kv` = [d k | d v]); V is transposed locally for the attention kernel
        store = sh.kv_store(sh.world * S, 2 * d, bf, dev) if sh.kv_store is not None else None
        kv_local = None if store is not None else self._e((sh.world * S, 2 * d), bf)
        nrm = dict(norm_dim=d, norm_eps=EPS)
        n_own = max(rows, 1)
        xb, xsq = self._e((n_own, d), bf), self._e((n_own, P), f32)
        xb2, xsq2 = self._e((n_own, d), bf), self._e((n_own, P), f32)
        qkv32 = self._e((n_own, 3 * d), f32)
        qr = self._e((n_own, d), bf)
        att = self._e((n_own, d), bf)
        vt = self._e((1, d, Ntp), bf)
        kst = self.enc_kv_split_tiles(Ntp)
        ws = self._e((max(ops.attention_ws_elems(1, H, n_own, Ntp, kst), 1),), f32) if kst else None
        if rows > 0:
            ops.rowstat(x, xb, xsq, rows=rows, d=d)
        for i in range(cfg.num_layers):
            o = f"enc{i}."
            # the k | v rows of layer i live in buffer i & 1 of the store: a fast rank may already push layer i + 1
            # while a slow one still attends layer i (it cannot be further ahead: one barrier per layer)
            kv = store.buf(i & 1) if store is not None else kv_local
            dsts, mc = store.dst(i & 1) if store is not None else ([kv.data_ptr()], False)
            if rows > 0:
                ops.gemm(xb[:rows], w[o + "wqkv"], out=qkv32, in_sumsq=xsq[:rows], **nrm)               # [q | k | v], fp32
                ops.qkv_post(qkv32, w[o + "qkn"], qr, dsts, multicast=mc, ldkv=2 * d, row0=r0, rows=rows, d=d,
                             pos=pos[r0:r1], freqs=w["enc.freqs"], eps=EPS)
            if store is not None:
                store.barrier()
            else:
                sh.all_gather(kv, kv[sh.rank * S:(sh.rank + 1) * S])
            ops.transpose16(kv[:Ntp, d:], vt[0], rows=Ntp, cols=d)
            if rows > 0:
                ops.attention(qr, kv, vt, att, B=1, H=H, Nq=rows, Nk=Ntp, ldq=d, ldk=2 * d, ldvt=Ntp, ldo=d,
                              mask_bits=bits, mask_bs=words, kv_split_tiles=kst, split_ws=ws)
                ops.gemm(att[:rows], w[o + "wo"], out=x, res1=x, out_sumsq=xsq2, out16=xb2, M=rows)
                g = ops.gemm(xb2[:rows], w[o + "w13"], epi=L.EPI_SWIGLU, out_dtype=bf, in_sumsq=xsq2[:rows], **nrm)
                ops.gemm(g, w[o + "w2"], out=x, res1=x, out_sumsq=xsq, out16=xb, M=rows)
        # the hoisted decoder K / V need the final 16-bit stream + row sums of ALL rows: one more gather
        # (row r of `xbs` = [d 16-bit values | d/128 fp32 partial sums | pad])
        xbs = self._e((sh.world * S, ldx), bf)
        xbs32 = xbs.view(f32)                                        # [world*S, ldx/2]
        xb_all, xsq_all = xbs[:Ntp, :d], xbs32[:Ntp, d // 2:d // 2 + P]
        if rows > 0:
            xbs[r0:r1, :d].copy_(xb[:rows])
            xbs32[r0:r1, d // 2:d // 2 + P].copy_(xsq[:rows])
        sh.all_gather(xbs, xbs[sh.rank * S:(sh.rank + 1) * S])
        # hoisted decoder K / V of ALL layers from the gathered stream, replicated on every rank (0.2 TFLOP:
        # cheaper than moving the 300 MB result over NVLink)
        k_all, v_all = self.hoist_kv(xb_all, xsq_all, 1, Ntp)
        if not gather_seq:  # the fp32 token sequence is not needed downstream: keep the own rows, skip the collective
            return SceneState(1, N, Nt, Ntp, x[:rows].view(1, rows, d), tri, mask_u8, bits, k_all, v_all, dv)
        seq = self._e((sh.world * S, d), f32)
        if rows > 0:
            seq[r0:r1].copy_(x[:rows])
        sh.all_gather(seq, seq[sh.rank * S:(sh.rank + 1) * S])
        return SceneState(1, N, Nt, Ntp, seq[:Ntp].view(1, Ntp, d), tri, mask_u8, bits, k_all, v_all, dv)

    def alloc_scene_state(self, B: int, N: int) -> SceneState:
        """Uninitialised SceneState of the right shapes (receive buffers for the NCCL broadcast)."""
        cfg = self.cfg
        d, dv = cfg.latent_dim, cfg.view_transformer_latent_dim
        Nt = N + cfg.num_register_tokens
        Ntp = _rup(Nt, 8)
        words = 4 * ((Ntp + 127) // 128)
        Lv = cfg.view_transformer_n_layers
        return SceneState(B, N, Nt, Ntp, self._e((B, Ntp, d), torch.float32), self._e((B, N, 9), torch.float32),
                          self._e((B, N), torch.uint8), self._e((B, words), torch.int32),
                          self._e((B, Ntp, Lv * dv), torch.float32), self._e((B, Lv * dv, Ntp), self.op), dv)

    # ------------------------------------------------------------------ stage 2
    def _keys_all_layers(self, st: SceneState, b: int, pos, V: int) -> torch.Tensor:
        """K-side QK-RMSNorm + camera-space RoPE of the hoisted keys of EVERY decoder layer for V
        views in one launch: bf16 [V*Ntp, L*dv]; layer i is the column slice [i*dv, (i+1)*dv)."""
        cfg = self.cfg
        dv, Lv = cfg.view_transformer_latent_dim, cfg.view_transformer_n_layers
        kall = self._e((V * st.Ntp, Lv * dv), self.op)
        ops.qknorm_rope(st.k_all[b], self.w["dec.kn_all"], kall, rows=V * st.Ntp, d=dv, nseg=Lv, ldx=Lv * dv,
                        ldo=Lv * dv, in_period=st.Ntp, pos=pos, freqs=self.w["dec.freqs"], eps=EPS)
        return kall

    def _swin_maps(self, Hp, Wp, shift, V):
        key = (Hp, Wp, shift, V)
        if key not in self._maps:
            perm, region = swin_window_maps(Hp, Wp, shift)
            n = Hp * Wp
            full = (perm[None, :] + (torch.arange(V, dtype=torch.int32) * n)[:, None]).reshape(-1)
            inv = torch.empty_like(full)
            inv[full.long()] = torch.arange(full.numel(), dtype=torch.int32)
            self._maps[key] = (full.to(self.device).contiguous(), region.to(self.device).contiguous(),
                               inv.to(self.device).contiguous())
        return self._maps[key]

    @torch.no_grad()
    def render_views(self, st: SceneState, b: int, c2w: Optional[torch.Tensor], fov_deg: Optional[torch.Tensor],
                     resolution, taps: Optional[dict] = None, rays_d: Optional[torch.Tensor] = None,
                     tri_cam: Optional[torch.Tensor] = None, pos_cam: Optional[torch.Tensor] = None,
                     raw_log: bool = False, out: Optional[torch.Tensor] = None,
                     window: Optional[tuple] = None, intrinsics: Optional[torch.Tensor] = None,
                     distortion: Optional[torch.Tensor] = None, lens: str = "opencv") -> torch.Tensor:
        """Render V views of scene `b` -> HDR fp32 [V,H,W,3]; `resolution` is an int (square) or (H, W)
        (config.view_grid).  Either cameras (c2w [V,4,4], fov_deg [V] or [V,1]; rays and camera-space triangles
        are derived on the device, fov spanning the longer image side) or, for the model-level entry
        (models/renderformer.py:171-206), an explicit camera-space ray map `rays_d` [V,H,W,3] together
        with the camera-space triangles `tri_cam` [V,N,9] -- or the ready RoPE positions `pos_cam`
        [V,Nt,9] (register centroids included) as ViewTransformer.forward receives them
        (models/view_transformer.py:88).  `raw_log`: return the head's pre-ELU output [V,H,W,3] instead
        (DPTHead.forward, layers/dpt.py:242-273).  `out`: contiguous fp32 [V,H,W,3] buffer the last kernel
        writes the image into (a slice of the caller's result tensor: no concatenation afterwards).
        `window=(h, w, top, left)` (cameras only, config.overscan_grid): `resolution` is the canvas the model runs
        on, the cameras are those of the h x w image it holds at canvas pixel (top, left), and only that window is
        stored: the result (and `out`) is [V, h, w, 3].
        `intrinsics` [V, 4] (fx, fy, cx, cy) in pixels of the returned image (the window, or the whole image) takes
        the place of `fov_deg`: a pinhole camera with those focal lengths and that principal point.  `distortion` (with
        `intrinsics`) makes it a lens-distorted camera: [V, 8] coefficients of lens "opencv" or [V, 4] of "fisheye"
        (config.view_camera's padded form)."""
        cfg, dev = self.cfg, self.device
        explicit = rays_d is not None
        if explicit and tri_cam is None and pos_cam is None:
            raise ValueError("rays_d needs tri_cam (camera-space triangle vertices) or pos_cam")
        if explicit and window is not None:
            raise ValueError("window (overscan) needs cameras; an explicit ray map covers the whole image")
        V = rays_d.shape[0] if explicit else c2w.shape[0]
        H, W = view_grid(cfg, resolution)
        Hp, Wp = H // 8, W // 8
        Ntp, N = st.Ntp, st.N
        if explicit:
            if tuple(rays_d.shape[1:]) != (H, W, 3):
                raise ValueError(f"rays_d must be [V, {H}, {W}, 3], got {tuple(rays_d.shape)}")
            rays = rays_d.to(dev, torch.float32).contiguous()
            if pos_cam is not None:
                pos = torch.zeros((V, Ntp, 9), dtype=torch.float32, device=dev)
                pos[:, :pos_cam.shape[1]] = pos_cam.to(dev, torch.float32)
            else:
                tc = tri_cam.reshape(V, N, 9).to(dev, torch.float32).contiguous()
                pos = self._e((V, Ntp, 9), torch.float32)
                for vi in range(V):  # centroid registers + vertices, already in camera space
                    ops.positions(tc[vi], st.mask_u8[b], None, pos[vi], n=N, n_reg=cfg.num_register_tokens,
                                  rows_out=Ntp, n_views=1)
            x = self.ray_tokens(V, H, W, rays=rays)
        else:
            c2w = c2w.to(dev, torch.float32).contiguous()
            if intrinsics is not None:
                fov, intr = None, intrinsics.reshape(V, 4).to(dev, torch.float32).contiguous()
            else:
                fov, intr = fov_deg.reshape(-1).to(dev, torch.float32).contiguous(), None
            if distortion is not None:
                distortion = distortion.reshape(V, -1).to(dev, torch.float32).contiguous()
            pos = ops.positions(st.tri[b], st.mask_u8[b], c2w, self._e((V, Ntp, 9), torch.float32), n=N,
                                n_reg=cfg.num_register_tokens, rows_out=Ntp, n_views=V)
            x = self.ray_tokens(V, H, W, fov=fov, window=window, intrinsics=intr, distortion=distortion, lens=lens)
        feats = self.decoder_layers(st, b, x, pos, V, Hp, Wp, taps)
        return self._dpt(feats, V, Hp, Wp, raw_out=raw_log, out=out, window=window)

    def ray_tokens(self, V: int, H: int, W: int, fov=None, rays=None, window=None, intrinsics=None, distortion=None,
                   lens: str = "opencv"):
        """Ray-bundle patch tokens x fp32 [V*(H/8)*(W/8), dv], row-major patch grid: pinhole rays
        (utils/ray_generator.py:13-50) or an explicit ray map -> 8x8 patches -> ray_map_patch_token +
        RMSNorm(Linear)  (view_transformer.py:104-108).  `window=(h, w, top, left)`: H x W is a canvas and the
        rays are those of the h x w camera whose image sits at (top, left).  `intrinsics` fp32 [V, 4] (fx, fy, cx,
        cy) in pixels of that image replaces `fov`, and `distortion` fp32 [V, 8] ("opencv") or [V, 4] ("fisheye") adds
        the `lens` model to it."""
        w = self.w
        dv = self.cfg.view_transformer_latent_dim
        rows = V * (H // 8) * (W // 8)
        rt = self._e((rows, 192), torch.float16)
        if rays is not None:
            ops.ray_map_tokens(rays, rt, n_views=V, height=H, width=W)
        elif intrinsics is not None:
            h, w_, top, left = (H, W, 0, 0) if window is None else window
            if distortion is not None:
                ops.ray_tokens_lens(intrinsics, distortion, rt, lens=lens, n_views=V, canvas_h=H, canvas_w=W, height=h,
                                    width=w_, top=top, left=left)
            else:
                ops.ray_tokens_intrinsics(intrinsics, rt, n_views=V, canvas_h=H, canvas_w=W, height=h, width=w_,
                                          top=top, left=left)
        elif window is not None:
            h, w_, top, left = window
            ops.ray_tokens_canvas(fov, rt, n_views=V, canvas_h=H, canvas_w=W, height=h, width=w_, top=top, left=left)
        else:
            ops.ray_tokens(fov, rt, n_views=V, height=H, width=W)
        lin = ops.gemm(rt, w["ray.w"], bias=w["ray.b"], out_dtype=torch.float32)
        x = self._e((rows, dv), torch.float32)
        ops.token_assemble(lin, w["ray.norm"], None, None, w["ray.token"], None, x, n_prefix=0, rows_in=rows,
                           rows_out=rows, batch=1, d=dv)
        return x

    def decoder_layers(self, st: SceneState, b: int, x, pos, V, Hp, Wp, taps=None, out_layers=None, want_f32=False):
        """TransformerDecoder.forward (layers/attention.py:673-688) for V views of scene `b`: x fp32
        [V*Hp*Wp, dv] ray tokens (updated in place), pos [V, Ntp, 9] camera-space RoPE positions of the
        triangle tokens.  Returns the feature maps of `out_layers` (default: the four DPT taps) as fp16
        [rows, dv] tensors (fp32 clones with `want_f32`)."""
        cfg, w = self.cfg, self.w
        out_layers = list(cfg.out_layers) if out_layers is None else list(out_layers)
        if self.fused_dec:
            return self._decode_fused(st, b, x, pos, V, Hp, Wp, taps, out_layers, want_f32)
        dv, Hh = cfg.view_transformer_latent_dim, cfg.view_transformer_n_heads
        Nr, Ntp = Hp * Wp, st.Ntp
        rows = V * Nr
        bf = self.op
        feats = []
        Lv = cfg.view_transformer_n_layers
        kall = self._keys_all_layers(st, b, pos, V)
        for i in range(cfg.view_transformer_n_layers):
            o = f"dec{i}."
            # cross-attention to the triangle tokens  (layers/attention.py:503-513)
            h = ops.rmsnorm(x, w[o + "n_q"], self._e((rows, dv), bf), rows=rows, d=dv, eps=EPS)
            qf = ops.gemm(h, w[o + "wq"], out_dtype=torch.float32)
            q = ops.qknorm_rope(qf, w[o + "qn"], self._e((rows, dv), bf), rows=rows, d=dv, nseg=1, ldx=dv, ldo=dv,
                                eps=EPS)  # camera-space ray origin is 0: query RoPE is the identity (E5)
            att = self._e((rows, dv), bf)
            ops.attention(q, kall[:, i * dv:], st.v_t(i, b), att, B=V, H=Hh, Nq=Nr, Nk=Ntp, ldq=dv, ldk=Lv * dv,
                          ldvt=Ntp, ldo=dv, q_bs=Nr * dv, k_bs=Ntp * Lv * dv, vt_bs=0, o_bs=Nr * dv,
                          mask_bits=st.mask_bits[b], mask_bs=0)
            ops.gemm(att, w[o + "wout"], out=x, res1=x)

            # full self-attention among ray tokens  (layers/attention.py:515-523; swin runs in _decode_fused)
            hs = ops.rmsnorm(x, w[o + "n_s"], self._e((rows, dv), bf), rows=rows, d=dv, eps=EPS)
            qk = ops.gemm(hs, w[o + "s.wqk"], out_dtype=torch.float32)
            Nrp = _rup(Nr, 8)
            vt = self._e((V, dv, Nrp), bf)
            for vi in range(V):
                ops.gemm(w[o + "s.wv"], hs[vi * Nr:(vi + 1) * Nr], out=vt[vi], N=Nr)
            qkn = ops.qknorm_rope(qk, w[o + "s.qkn"], self._e((rows, 2 * dv), bf), rows=rows, d=dv, nseg=2,
                                  ldx=2 * dv, ldo=2 * dv, eps=EPS)  # ray RoPE is the identity
            ops.attention(qkn, qkn[:, dv:], vt, att, B=V, H=Hh, Nq=Nr, Nk=Nr, ldq=2 * dv, ldk=2 * dv, ldvt=Nrp,
                          ldo=dv, q_bs=Nr * 2 * dv, k_bs=Nr * 2 * dv, vt_bs=dv * Nrp, o_bs=Nr * dv)
            ops.gemm(att, w[o + "s.wo"], out=x, res1=x)
            self._ffn(x, rows, dv, w[o + "n_f"], w[o + "w13"], w[o + "w2"])
            if i in out_layers:
                feats.append(x.clone() if want_f32 else ops.cast(x, self._e((rows, dv), torch.float16)))
                if taps is not None:
                    taps.setdefault("dec_feats", []).append(x.clone().view(V, Nr, dv))
        return feats

    def _decode_fused(self, st: SceneState, b: int, x, pos, V, Hp, Wp, taps, out_layers, want_f32=False):
        """Swin decoder with RMSNorm / QK-RMSNorm fused into the GEMMs and the attention kernels.
        Carried state: x fp32 (token order), xb bf16 copy + xsq partial row sums (token order), and
        their window-order twins xbw / xsqw written by the cross-attention out-projection."""
        cfg, w = self.cfg, self.w
        dv, Hh = cfg.view_transformer_latent_dim, cfg.view_transformer_n_heads
        Nr, Ntp = Hp * Wp, st.Ntp
        rows = V * Nr
        bf, f32 = self.op, torch.float32
        nrm = dict(norm_dim=dv, norm_eps=EPS)
        P = dv // 128
        xb, xsq = self._e((rows, dv), bf), self._e((rows, P), f32)
        xbw, xsqw = self._e((rows, dv), bf), self._e((rows, P), f32)
        qh, qsq = self._e((rows, dv), bf), self._e((rows, P), f32)
        qkh, qksq = self._e((rows, 2 * dv), bf), self._e((rows, 2 * P), f32)
        att = self._e((rows, dv), bf)
        vt = self._e((dv, rows), bf)
        Lv = cfg.view_transformer_n_layers
        kall = self._keys_all_layers(st, b, pos, V)
        ops.rowstat(x, xb, xsq, rows=rows, d=dv)
        feats = []
        for i in range(cfg.view_transformer_n_layers):
            o = f"dec{i}."
            perm, region, inv = self._swin_maps(Hp, Wp, 0 if i % 2 == 0 else 4, V)
            # cross-attention: q = (n_q(x) Wq^T) . qn / rms  -- the 1/rms goes into the softmax scale
            ops.gemm(xb, w[o + "wq"], out16=qh, col_mul=w[o + "qn"], out_sumsq=qsq, in_sumsq=xsq, **nrm)
            ops.attention(qh, kall[:, i * dv:], st.v_t(i, b), att, B=V, H=Hh, Nq=Nr, Nk=Ntp, ldq=dv, ldk=Lv * dv,
                          ldvt=Ntp, ldo=dv, q_bs=Nr * dv, k_bs=Ntp * Lv * dv, vt_bs=0, o_bs=Nr * dv,
                          mask_bits=st.mask_bits[b], mask_bs=0, q_sumsq=qsq, sumsq_ld=P, sumsq_parts=P, **nrm)
            # x += out_proj(att); bf16 copy + row sums land in window order for the swin block
            ops.gemm(att, w[o + "wout"], out=x, res1=x, out_sumsq=xsqw, out16=xbw, aux_row_map=inv)
            # shifted-window self-attention (window-major rows); q sums in parts [0,P), k sums in [P,2P)
            ops.gemm(xbw, w[o + "s.wqkv"], out16=qkh, col_mul=w[o + "s.qkn"], out_sumsq=qksq, in_sumsq=xsqw,
                     vt_out=vt, vt_split=2 * dv, **nrm)
            ops.attention(qkh, qkh[:, dv:], vt, att, B=1, H=Hh, Nq=rows, Nk=rows, ldq=2 * dv, ldk=2 * dv,
                          ldvt=rows, ldo=dv, mode=1, group_id=region, group_period=Nr,
                          q_sumsq=qksq, k_sumsq=qksq.view(-1)[P:], sumsq_ld=2 * P, sumsq_parts=P, **nrm)
            ops.gemm(att, w[o + "s.wo"], out=x, res1=x, row_map=perm, out_sumsq=xsq, out16=xb)
            # SwiGLU
            g = ops.gemm(xb, w[o + "w13"], epi=L.EPI_SWIGLU, out_dtype=bf, in_sumsq=xsq, **nrm)
            ops.gemm(g, w[o + "w2"], out=x, res1=x, out_sumsq=xsq, out16=xb)
            if i in out_layers:
                feats.append(x.clone() if want_f32 else ops.cast(x, self._e((rows, dv), torch.float16)))
                if taps is not None:
                    taps.setdefault("dec_feats", []).append(x.clone().view(V, Nr, dv))
        return feats

    # ------------------------------------------------------------------ DPT head (layers/dpt.py:242-273)
    def _conv(self, x, name, B, H, W, Cin, **kw):
        return ops.gemm(x, self.w[name + ".w"], conv=(B, H, W, Cin), **kw)

    def _rcu(self, x_raw, x_act, name, B, H, W, extra_res=None, want_act=False):
        """x + conv2(silu(conv1(silu(x))))  (+ extra_res)   layers/dpt.py:76-92,139-143."""
        F_ = self.cfg.dpt_features
        hf = torch.float16
        t = self._e((B * H * W, F_), hf)
        self._conv(x_act, name + "c1", B, H, W, F_, bias=self.w[name + "c1.b"], out=None, out_act=t)
        out = self._e((B * H * W, F_), hf)
        act = self._e((B * H * W, F_), hf) if want_act else None
        self._conv(t, name + "c2", B, H, W, F_, bias=self.w[name + "c2.b"], res1=x_raw, res2=extra_res, out=out,
                   out_act=act)
        return out, act

    def _fusion(self, r, B, H, W, Ho, Wo, x0, x1_raw=None, x1_act=None, x0_act=None):
        """FeatureFusionBlock (layers/dpt.py:133-159); the 1x1 out_conv runs before the bilinear
        resize, with which it commutes (SURVEY Appendix E1)."""
        F_ = self.cfg.dpt_features
        hf = torch.float16
        name = f"dpt.rf{r}."
        if x1_raw is not None:
            s_raw, s_act = self._rcu(x1_raw, x1_act, name + "u1", B, H, W, extra_res=x0, want_act=True)
        else:
            s_raw, s_act = x0, x0_act
        o, _ = self._rcu(s_raw, s_act, name + "u2", B, H, W)
        o = ops.gemm(o, self.w[name + "out.w"], bias=self.w[name + "out.b"], out=self._e((B * H * W, F_), hf))
        return ops.upsample_bilinear(o, self._e((B * Ho * Wo, F_), hf), B=B, Hi=H, Wi=W, Ho=Ho, Wo=Wo, C_=F_)

    def _dpt(self, feats, V, Hp, Wp, raw_out: bool = False, out: Optional[torch.Tensor] = None, window=None):
        """DPTHead.forward (layers/dpt.py:242-273) on four fp16 feature maps [V*Hp*Wp, dv] -> HDR image fp32
        [V, 8Hp, 8Wp, 3] (the head's ELU and the pipeline's 10^x - 1 are the last conv's epilogue), or with
        `raw_out` the head's own output before the ELU.  `window=(h, w, top, left)`: the last conv stores only that
        window of the image, [V, h, w, 3]."""
        cfg, w = self.cfg, self.w
        hf = torch.float16
        C = list(cfg.dpt_out_channels)
        F_ = cfg.dpt_features
        n = V * Hp * Wp
        proj = [ops.gemm(feats[i], w[f"dpt.proj{i}.w"], bias=w[f"dpt.proj{i}.b"], out=self._e((n, C[i]), hf))
                for i in range(4)]
        # resize to the 4 pyramid levels (layers/dpt.py:195-213)
        t0 = ops.gemm(proj[0], w["dpt.up0.w"], bias=w["dpt.up0.b"], out=self._e((n, 16 * C[0]), hf))
        r0 = ops.pixel_shuffle(t0, self._e((V * 16 * Hp * Wp, C[0]), hf), B=V, h=Hp, w=Wp, s=4, C_=C[0])
        t1 = ops.gemm(proj[1], w["dpt.up1.w"], bias=w["dpt.up1.b"], out=self._e((n, 4 * C[1]), hf))
        r1 = ops.pixel_shuffle(t1, self._e((V * 4 * Hp * Wp, C[1]), hf), B=V, h=Hp, w=Wp, s=2, C_=C[1])
        r2 = proj[2]
        H3, W3 = (Hp + 1) // 2, (Wp + 1) // 2
        col = ops.im2col_s2(proj[3], self._e((V * H3 * W3, 9 * C[3]), hf), B=V, H=Hp, W=Wp, C_=C[3])
        r3 = ops.gemm(col, w["dpt.down3.w"], bias=w["dpt.down3.b"], out=self._e((V * H3 * W3, C[3]), hf))
        dims = [(4 * Hp, 4 * Wp), (2 * Hp, 2 * Wp), (Hp, Wp), (H3, W3)]
        lraw, lact = [], []
        for i, (r, (H, W)) in enumerate(zip((r0, r1, r2, r3), dims)):
            raw, act = self._e((V * H * W, F_), hf), self._e((V * H * W, F_), hf)
            self._conv(r, f"dpt.rn{i}", V, H, W, C[i], out=raw, out_act=act)
            lraw.append(raw), lact.append(act)
        p4 = self._fusion(4, V, *dims[3], *dims[2], lraw[3], x0_act=lact[3])
        p3 = self._fusion(3, V, *dims[2], *dims[1], p4, lraw[2], lact[2])
        p2 = self._fusion(2, V, *dims[1], *dims[0], p3, lraw[1], lact[1])
        Ho, Wo = 8 * Hp, 8 * Wp
        p1 = self._fusion(1, V, *dims[0], Ho, Wo, p2, lraw[0], lact[0])
        # head (layers/dpt.py:266-271); F.interpolate to (8*Hp, 8*Wp) is the identity here (E2)
        o1 = self._conv(p1, "dpt.oc1", V, Ho, Wo, F_, bias=w["dpt.oc1.b"], out=self._e((V * Ho * Wo, F_ // 2), hf))
        Hs, Ws = (Ho, Wo) if window is None else window[:2]
        if out is not None and (tuple(out.shape) != (V, Hs, Ws, 3) or out.dtype != torch.float32 or not out.is_contiguous()):
            raise ValueError("out must be a contiguous fp32 [V, H, W, 3] tensor")
        img = out if out is not None else self._e((V, Hs, Ws, 3), torch.float32)
        self._conv(o1, "dpt.oc2", V, Ho, Wo, F_ // 2, bias=w["dpt.oc2.b"], epi=L.EPI_FINAL_RAW if raw_out else L.EPI_FINAL,
                   w2=w["dpt.oc3.w"], b2=w["dpt.oc3.b"], out=img, ldo=3, crop=window)
        return img
