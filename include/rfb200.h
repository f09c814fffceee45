/*
 * rfb200.h -- C ABI of the B200-native RenderFormer inference kernels.
 *
 * The reference (agwi-lab/renderformer) has no FFI layer: its hot path is Python
 * calling torch / flash-attn / cuDNN.  Each entry point below replaces one family of
 * those call sites (cited as reference file:line, relative to the reference root).
 * All pointers are device pointers unless stated; all functions are asynchronous on
 * `stream`, never allocate, and return RFB_OK (0) or a negative error code.
 * No torch types cross this boundary.
 */
#ifndef RFB200_H_
#define RFB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* rfb_stream_t; /* cudaStream_t */

enum {
  RFB_OK = 0,
  RFB_ERR_ARG = -1,    /* bad argument / unsupported shape */
  RFB_ERR_ALIGN = -2,  /* pointer or stride not 16-byte aligned */
  RFB_ERR_DRIVER = -3, /* CUDA driver entry point unavailable (no GPU driver) */
  RFB_ERR_TMAP = -4,   /* cuTensorMapEncodeTiled rejected the descriptor */
  RFB_ERR_LAUNCH = -5  /* kernel launch failed */
};

/* element types */
enum { RFB_F32 = 0, RFB_BF16 = 1, RFB_F16 = 2 };

int rfb_version(void);
/* number of kernels launched by this library since load (bench.py's gpu_launches) */
long long rfb_launch_count(void);

/* ---------------------------------------------------------------------------------
 * rfb_gemm: C[M,N] = A[M,K] * W[N,K]^T  (16-bit operands, fp32 accumulate in TMEM;
 * TMA-fed tcgen05.mma, persistent, fused epilogue).
 *
 * Replaces every nn.Linear on the path -- layers/attention.py:51-57 (SwiGLU w1,w2,w3),
 * :95-100,120-125,202 (in_proj/q_proj/k_proj/v_proj/out_proj), :300-301,343,361 (swin),
 * models/renderformer.py:49,63,139-147 (token encoders), models/view_transformer.py:45,108
 * -- and, with a_mode = RFB_A_CONV3X3, the DPT convolutions layers/dpt.py:44-52,68-71,
 * 184-240 as implicit GEMM (1x1 convs and ConvTranspose k=s are plain linear GEMMs).
 * ------------------------------------------------------------------------------- */
enum { RFB_A_LINEAR = 0, RFB_A_CONV3X3 = 1 };
enum {
  RFB_EPI_STORE = 0,  /* v = acc (+bias) (+res1) (+res2); out = v; out_act = silu(v) */
  RFB_EPI_SWIGLU = 1, /* W rows interleaved [16 gate | 16 up] per 32: out[:, n/2] = silu(g)*u */
  RFB_EPI_FINAL = 2,  /* N==32: y = w2 * silu(acc+bias) + b2 (3 ch); out = 10^elu(y) - 1, fp32 */
  RFB_EPI_FINAL_RAW = 3 /* as FINAL but out = y: DPTHead.forward's own return value (layers/dpt.py:271) */
};

typedef struct {
  int M, N, K;   /* conv: M = B*H*W output pixels, K = 9*Cin */
  const void* A; /* [M,K] row-major (lda elements) | conv: NHWC [B,H,W,Cin] */
  long long lda;
  const void* W; /* [N,K] row-major (ldw elements); conv: K index = tap*Cin + cin, tap = ky*3+kx */
  long long ldw;
  int dtype; /* operand type: RFB_BF16 or RFB_F16 */
  int a_mode;
  int B, H, Wd, Cin; /* conv geometry (stride 1, pad 1) */
  int epi;
  const float* bias; /* [N] or NULL */
  const void* res1;  /* [M, ldres] addend or NULL */
  const void* res2;
  int res_dtype;
  long long ldres;
  void* out; /* [M, ldo] or NULL */
  int out_dtype;
  long long ldo;
  void* out_act;      /* optional silu(v) copy, same dtype/ld as out */
  const int* row_map; /* optional: output/residual row = row_map[m] (swin window order -> token order) */
  const float* w2;    /* RFB_EPI_FINAL: [3,32] */
  const float* b2;    /* RFB_EPI_FINAL: [3] */
  int bn_override;    /* 0 = auto; else force the N tile (32/64/128/256) */
  int max_ctas;       /* 0 = one per SM */
  /* ---- fused RMSNorm plumbing (RFB_EPI_STORE / RFB_EPI_SWIGLU; all optional) -----------------
   * RMSNorm(x) W^T = r * (x (W . w)^T), r = rsqrt(mean(x^2) + eps): the norm weight w is folded
   * into W offline, A is the raw activation in 16 bits, and the per-row factor r is applied to
   * the accumulator here.  Row sums of squares travel between kernels as PARTIAL sums, one per
   * RFB_SUMSQ_PART_COLS (128) columns of the producing GEMM: no atomics, no clearing, and the
   * result is deterministic.  A consumer adds the first `parts` entries of its row. */
  const float* in_sumsq; /* [M][in_sumsq_ld] partial sums of x^2 of the A rows; r applied per row */
  int in_sumsq_ld;
  int in_sumsq_parts;
  const float* in_rscale; /* ready-made factors instead of in_sumsq: [M] (scale_dim 0) or [N] (scale_dim 1) */
  int scale_dim;
  int norm_dim;           /* row length the mean is taken over */
  float norm_eps;
  float* out_rscale;      /* [M] side output: the factor r derived from in_sumsq */
  float* out_sumsq;       /* [rows][out_sumsq_ld]: entry n/128 = sum over columns [128(n/128), +128) of v^2,
                             v = value stored to out; needs N % 128 == 0 (forces the 256-wide tile) */
  int out_sumsq_ld;
  void* out16;            /* extra 16-bit copy of v * col_mul[n] */
  int out16_dtype;
  long long ld16;
  const float* col_mul;   /* [N] or NULL */
  const int* aux_row_map; /* row of out16 / out_sumsq = aux_row_map ? aux_row_map[out_row] : out_row */
  /* ---- transposed side output (RFB_EPI_STORE, linear A): the V part of a fused [q | k | v] projection.
   * Columns n >= vt_split are not written to out / out16 but, multiplied by the row factor r, to
   * vt_out[b][n - vt_split][m - b*vt_rows_per_batch] (16-bit), b = m / vt_rows_per_batch (0 if that is 0):
   * V arrives transposed (keys contiguous) as rfb_attention wants it, without a second GEMM.
   * vt_split must be a multiple of 256 (a whole number of N tiles). */
  void* vt_out;
  int vt_dtype;
  int vt_split;
  int vt_rows_per_batch;
  long long vt_ld;
  long long vt_batch_stride;
  /* ---- output crop (conv A with RFB_EPI_FINAL / RFB_EPI_FINAL_RAW; all zero = none): only the pixels of the
   * window [crop_top, crop_top + crop_h) x [crop_left, crop_left + crop_w) of the H x Wd image are stored, pixel
   * (b, y, x) to row (b * crop_h + y - crop_top) * crop_w + (x - crop_left) of out [B, crop_h, crop_w, ldo].
   * The window must lie inside the image; the rest of the image is computed and discarded (overscan). */
  int crop_h, crop_w, crop_top, crop_left;
} rfb_gemm_args;

int rfb_gemm(const rfb_gemm_args* a, rfb_stream_t stream);

/* ---------------------------------------------------------------------------------
 * rfb_attention: O = softmax(scale * Q K^T + mask) V, head_dim 128, bf16 or fp16 in/out, fp32
 * softmax and accumulation (tcgen05 flash-style kernel, S and O live in TMEM).
 *
 * Replaces F.scaled_dot_product_attention / flash_attn_* at layers/attention.py:143-198
 * (encoder self-attention and decoder cross-attention, key-padding mask fused) and the
 * per-window SDPA of SwinSelfAttention at layers/attention.py:349-358 (mode 1: the
 * window partition and the shifted-window region mask become a group-id equality test).
 *
 * Layouts: Q [B][Nq][ldq], K [B][Nk][ldk] with head h in columns [h*128, h*128+128);
 * Vt [B][H*128][ldvt] = V transposed (keys contiguous).  A batch stride of 0 on K / Vt /
 * mask shares that tensor across the batch (hoisted per-scene K/V, SURVEY E5).
 * ------------------------------------------------------------------------------- */
typedef struct {
  int B, H, Nq, Nk;
  const void* Q;
  long long ldq, q_batch_stride;
  const void* K;
  long long ldk, k_batch_stride;
  const void* Vt;
  long long ldvt, vt_batch_stride;
  void* O;
  long long ldo, o_batch_stride;
  const uint32_t* key_mask_bits; /* mode 0: [B][4*ceil(Nk/128)] packed bits, 1 = attend; NULL = all */
  long long mask_batch_stride_words;
  int mode;                /* 0 = dense over all keys, 1 = block-diagonal 128-token tiles */
  const uint8_t* group_id; /* mode 1: [group_period] region ids; i,j attend iff same 64-token
                              half of the tile and equal ids */
  int group_period;
  float scale;
  /* fused QK-RMSNorm (optional): Q / K hold q*w, k*w un-normalised; logits are multiplied by
   * rsqrt(SQ(q_sumsq, b*Nq+i)/norm_dim + eps) * rsqrt(SQ(k_sumsq, b*Nk+j)/norm_dim + eps) with
   * SQ(p, r) = sum of p[r*sumsq_ld + 0 .. sumsq_parts) (partial sums left by rfb_gemm's out_sumsq).
   * k_sumsq: mode 1 only. */
  const float* q_sumsq;
  const float* k_sumsq;
  int sumsq_ld;
  int sumsq_parts;
  int norm_dim;
  float norm_eps;
  int dtype; /* operand type of Q, K, Vt and O: RFB_BF16 (also 0 = unset) or RFB_F16 */
  /* key splitting (mode 0, optional; 0 = off): the key range is cut into chunks of kv_split_tiles 128-key tiles,
   * every chunk runs on its own CTA (more CTAs when there are few query rows, e.g. one rank's rows of the
   * row-sharded scene stage) and a second kernel merges the chunks' partial softmax results in chunk order.
   * The result of a query row depends on kv_split_tiles but not on how many rows the call holds.
   * split_ws: caller-provided scratch, >= rfb_attention_ws_bytes(...) bytes, 16-byte aligned; at most 8 chunks. */
  int kv_split_tiles;
  void* split_ws;
  long long split_ws_bytes;
} rfb_attn_args;

int rfb_attention(const rfb_attn_args* a, rfb_stream_t stream);
long long rfb_attention_ws_bytes(int B, int H, int Nq, int Nk, int kv_split_tiles);

/* ---------------------------------------------------------------------------------
 * Row kernels (one warp per row, fp32 math, 128-bit accesses).
 * ------------------------------------------------------------------------------- */

/* out[r,:] = RMSNorm(x[gather ? gather[r] : r, :]) * w -- nn.RMSNorm at layers/attention.py:
 * 436-482 as used in AttentionLayer.forward :503,508,516,526.  `gather` folds torch.roll +
 * window_partition (:334-339) into the read.  out_dtype RFB_F32/BF16/F16. */
int rfb_rmsnorm(const float* x, long long ldx, const float* w, void* out, int out_dtype, long long ldo,
                int rows, int d, float eps, const int* gather, rfb_stream_t stream);

/* (input row = gather ? gather[r] : r: torch.roll + window_partition, layers/attention.py:334-339, folded into the read)
 * out16[r*ld16 + :] = cast(x[r,:]) (16-bit), sumsq[r*sumsq_ld] = sum(x[r,:]^2), sumsq[r*sumsq_ld + 1..parts) = 0:
 * seeds the fused-norm GEMM chain (the input side of nn.RMSNorm, layers/attention.py:503-526,
 * without materialising norm(x)) in the partial-sum layout rfb_gemm's out_sumsq uses. */
int rfb_rowstat(const float* x, void* out16, int out_dtype, long long ld16, float* sumsq, int sumsq_ld, int parts,
                int rows, int d, const int* gather, rfb_stream_t stream);

/* QK-RMSNorm over the full model width + triangle RoPE (layers/attention.py:128-141,
 * encodings/rope.py:78-149,152-206): fp32 [rows, nseg*d] -> 16 bit (out_dtype RFB_BF16 / RFB_F16).  Input row = r % in_period
 * when in_period > 0 (one hoisted pre-RoPE K re-rotated for every view).  pos [rows,9] or NULL. */
int rfb_qknorm_rope(const float* x, long long ldx, int in_period, const float* w, void* out, int out_dtype,
                    long long ldo, int rows, int d, int nseg, float eps, const float* pos, const float* freqs,
                    int nfreq, rfb_stream_t stream);

/* Row-sharded scene stage (multi-GPU; the reference has no counterpart, models/renderformer.py:171-206 runs on one
 * device): post-processing of ONE rank's fused [q | k | v] projection x fp32 [rows, ldx >= 3d] (RMSNorm row factor
 * applied) fused with the layer's all-gather.  q and k get the QK-RMSNorm (w_qk = [w_q | w_k]) + triangle RoPE of
 * rfb_qknorm_rope (bit-identical per row), v is cast; q goes to out_q [rows, ldq], k | v go to row row0 + r of
 * EVERY destination [*, ldkv] (columns [0,d) and [d,2d)).  kv_dst: n_dst (<= 8) device pointers -- this rank's own
 * store, plus the peer-mapped stores of the other ranks (plain NVLink stores) -- or, with multicast != 0, ONE NVLS
 * multicast address (multimem.st: the switch replicates each store into all ranks' memories).  The caller
 * synchronises the ranks afterwards (a signal-pad barrier) before anybody reads the stores. */
int rfb_qkv_post(const float* x, long long ldx, const float* w_qk, void* out_q, long long ldq, void* const* kv_dst,
                 int n_dst, int multicast, long long ldkv, long long row0, int rows, int d, float eps, const float* pos,
                 const float* freqs, int nfreq, int out_dtype, rfb_stream_t stream);

/* The same with READY-MADE rotation tables, as MultiHeadAttention.forward receives them (layers/attention.py:115:
 * rope_cos / rope_sin [rows, ldtab >= 64] fp32 from freqs_to_cos_sin, encodings/rope.py:78-103): pair (i, i+64) of
 * every head rotates by (cos_tab[r][i], sin_tab[r][i]).  NULL tables = QK-RMSNorm only; w == NULL = rotation
 * only (apply_rotary_emb_one_cossin, encodings/rope.py:132-149). */
int rfb_qknorm_rope_table(const float* x, long long ldx, const float* w, void* out, int out_dtype, long long ldo,
                          int rows, int d, int nseg, float eps, const float* cos_tab, const float* sin_tab,
                          long long ldtab, rfb_stream_t stream);

/* out[b, n_prefix + i, :] = token + RMSNorm(a[b,i]) * wa (+ RMSNorm(b[b,i]) * wb); rows
 * [0,n_prefix) = prefix; rows past n_prefix + rows_in are zero.  models/renderformer.py:139-163,
 * models/view_transformer.py:108.  eps = fp32 machine epsilon (nn.RMSNorm(eps=None)). */
int rfb_token_assemble(const float* a, const float* wa, const float* b, const float* wb, const float* token,
                       const float* prefix, int n_prefix, float* out, int rows_in, int rows_out, int batch,
                       int d, rfb_stream_t stream);

/* texture fp32 [n_tris, channels, texels] -> f16, log10(x+1) on the last log_channels channels
 * (pipelines/rendering_pipeline.py:67-68; does not touch the caller's tensor). */
int rfb_texture_prep(const float* tex, void* out, long long n_tris, int channels, int texels,
                     int log_channels, rfb_stream_t stream);

/* Constant-texture fast path (SURVEY §8f rank 2): scenes written by scene_processor/to_h5.py:37-66 hold
 * 13 per-triangle constants times a fixed triangular texel mask, so texture_encoder
 * (models/renderformer.py:145-147) collapses to a [N,13] x [13,d] product with the texel-summed weight.
 * tex fp32 [n_tris, channels] -> f16 [n_tris, ld] zero padded, log10(x+1) on the last log_channels. */
int rfb_texture_const_prep(const float* tex, void* out, long long n_tris, int channels, int ld, int log_channels,
                           rfb_stream_t stream);

/* NeRF encoding of vertex normals [n,9] -> f16 [n, ld] (encodings/nerf_encoding.py:63-84). */
int rfb_vn_encode(const float* vn, void* out, int n, int nfreq, int ld, rfb_stream_t stream);

/* Ray kernels of an H x W image (height, width multiples of 8 where patch tokens are produced).  Camera: pinhole,
 * square pixels, principal point at the image centre, pixel centres at +0.5, fov spanning the LONGER side:
 * f = max(H, W) / 2 / tan(fov / 2), d = ((px + 0.5 - W/2) / f, -(py + 0.5 - H/2) / f, -1).  Patch tokens are
 * f16 [V, (H/8)*(W/8), 192] in row-major patch-grid order (token = h1 * (W/8) + w1, feature = c*64 + p1*8 + p2,
 * models/view_transformer.py:104-107).  The `resolution` forms are the square case H = W = resolution. */

/* camera-space ray bundles -> patch tokens (utils/ray_generator.py:13-50 with identity c2w); fov in degrees. */
int rfb_ray_tokens_hw(const float* fov_deg, void* out, int n_views, int height, int width, rfb_stream_t stream);
int rfb_ray_tokens(const float* fov_deg, void* out, int n_views, int resolution, rfb_stream_t stream);
/* the same over a canvas_h x canvas_w canvas (sides multiples of 8) that holds the height x width image at canvas
 * pixel (top, left): tokens [V, (canvas_h/8)*(canvas_w/8), 192]; the camera is the image's (f from max(height,
 * width)), with the principal point at the window's centre (left + width/2, top + height/2).  rfb_ray_tokens_hw
 * is the case canvas == image, top = left = 0. */
int rfb_ray_tokens_canvas(const float* fov_deg, void* out, int n_views, int canvas_h, int canvas_w, int height,
                          int width, int top, int left, rfb_stream_t stream);
/* the same tokens for per-view pinhole intrinsics intr [V,4] = (fx, fy, cx, cy) on the device, in pixels of the
 * height x width image the canvas holds at (top, left) (canvas == image: top = left = 0).  The centre of image pixel
 * (row i, column j) is (j + 0.5, i + 0.5) (OpenCV K: add 0.5 to cx and cy); its ray is
 * normalize(((u - cx) / fx, -(v - cy) / fy, -1)).  Argument checks as rfb_ray_tokens_canvas. */
int rfb_ray_tokens_intrinsics(const float* intr, void* out, int n_views, int canvas_h, int canvas_w, int height,
                              int width, int top, int left, rfb_stream_t stream);
/* the same tokens for lens-distorted cameras: intrinsics as rfb_ray_tokens_intrinsics, and per view lens coefficients
 * on the device, dist [V,8] = (k1, k2, p1, p2, k3, k4, k5, k6) for lens 0 (OpenCV, COLMAP FULL_OPENCV) or dist [V,4]
 * = (k1, k2, k3, k4) for lens 1 (OpenCV fisheye, COLMAP OPENCV_FISHEYE).  Each pixel's distorted normalized
 * coordinates ((u - cx) / fx, (v - cy) / fy) are undistorted by Newton's method; the ray is normalize((x, -y, -1))
 * (lens 0) or (sin t * xd / rd, -sin t * yd / rd, -cos t) (lens 1).  Coefficients that do not invert give finite
 * tokens, not correct ones.  Argument checks as rfb_ray_tokens_intrinsics, and lens must be 0 or 1. */
int rfb_ray_tokens_lens(const float* intr, const float* dist, int lens, void* out, int n_views, int canvas_h,
                        int canvas_w, int height, int width, int top, int left, rfb_stream_t stream);
/* fov in degrees [V] -> intrinsics [V,4] = (f, f, width/2, height/2) of a height x width image, f = side / 2 /
 * tan(fov / 2) with side = max(height, width) (fit 0, Blender's "Auto"; the focal length rfb_ray_tokens_canvas
 * uses, bit for bit), width (fit 1, "Horizontal") or height (fit 2, "Vertical"). */
int rfb_intrinsics_from_fov(const float* fov_deg, float* out, int n_views, int height, int width, int fit,
                            rfb_stream_t stream);

/* RayGenerator.forward (utils/ray_generator.py:13-50) for callers that want the ray map itself: c2w [V,4,4],
 * fov in RADIANS [V] -> rays_d fp32 [V, H, W, 3] (rotated by R(c2w), L2-normalised). */
int rfb_ray_map_hw(const float* c2w, const float* fov_rad, float* rays_d, int n_views, int height, int width,
                   rfb_stream_t stream);
int rfb_ray_map(const float* c2w, const float* fov_rad, float* rays_d, int n_views, int resolution, rfb_stream_t stream);

/* explicit ray map fp32 [V, H, W, 3] -> patch tokens (models/view_transformer.py:104-107): the model-level entry
 * RenderFormer.forward(..., rays_d, tri_vpos_view_tf) hands rays in instead of cameras. */
int rfb_ray_map_tokens_hw(const float* rays_d, void* out, int n_views, int height, int width, rfb_stream_t stream);
int rfb_ray_map_tokens(const float* rays_d, void* out, int n_views, int resolution, rfb_stream_t stream);

/* RoPE positions [V, rows_out, 9]: register rows = masked centroid, then T_v^-1 * triangle
 * (models/renderformer.py:103-124, utils/transform.py:7-27).  c2w NULL = world space. */
int rfb_positions(const float* tri, const uint8_t* mask, const float* c2w, float* pos, int n, int n_reg,
                  int rows_out, int n_views, rfb_stream_t stream);

/* bool key mask [batch, n] -> packed bits [batch, words] behind n_prefix always-valid keys. */
int rfb_pack_mask(const uint8_t* mask, uint32_t* bits, int n, int n_prefix, int words, int batch,
                  rfb_stream_t stream);

int rfb_cast(const float* x, void* out, int out_dtype, long long n, rfb_stream_t stream);

/* out[c*ld_out + r] = in[r*ld_in + c] for 16-bit elements (cols, ld_in, ld_out even).  The row-sharded scene stage
 * (renderformer_b200/engine.py:_encode_scene_sharded) all-gathers the ranks' [k | v] rows and turns V into the
 * V^T layout rfb_attention reads; the single-GPU path never needs it (its V leaves the GEMM transposed). */
int rfb_transpose16(const void* in, long long ld_in, void* out, long long ld_out, int rows, int cols, rfb_stream_t stream);

/* ---------------------------------------------------------------------------------
 * DPT decoder helpers, NHWC f16 (layers/dpt.py:154-155,195-213).
 * ------------------------------------------------------------------------------- */
int rfb_pixel_shuffle(const void* in, void* out, int B, int h, int w, int s, int C, rfb_stream_t stream);
int rfb_im2col_s2(const void* in, void* out, int B, int H, int W, int C, rfb_stream_t stream);
int rfb_upsample_bilinear(const void* in, void* out, int B, int Hi, int Wi, int Ho, int Wo, int C,
                          rfb_stream_t stream);

/* HDR fp32 [n_pixels, 3] -> uint8 [n_pixels, 3], the step right after the path in the CLIs
 * (infer.py:94-98, batch_infer.py:153-157).  mode 0 = their default `(np.clip(hdr, 0, 1) * 255).astype(uint8)`,
 * bit-exact; mode 1 = Khronos PBR Neutral tone curve + sRGB OETF (published formula; the reference reaches
 * it through simple_ocio, which is not vendored: unpinned). */
int rfb_ldr_quantize(const float* hdr, uint8_t* out, long long n_pixels, int mode, rfb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RFB200_H_ */
