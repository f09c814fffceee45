// rfb_attention: entry point of the flash-style attention kernels (tcgen05 / TMEM, head_dim = 128, sm_100a).
//
//   O = softmax(scale * Q K^T + mask) V        per (batch, head, 128-query tile)
//
// The kernels live in attention2.cu (two query tiles per CTA), attention3.cu (one query tile per CTA, Q in
// TMEM) and attention_swin.cu (block-diagonal shifted-window mode); the arithmetic they share is in
// attention_common.cuh.  This file builds the TMA descriptors and the dense kernels' parameters, picks the
// kernel and merges key-split partial results.  Operands are bf16 or fp16 (`dtype`), V is consumed
// transposed ([head_dim, keys], keys contiguous) so every operand is K-major.
//
// mode 0: every query tile visits all key tiles; keys are masked by a packed bit mask
//         (the key-padding mask of layers/attention.py:145-161, True = attend).
// mode 1: block-diagonal -- query tile i only sees key tile i; a tile holds two 64-token swin
//         windows and tokens attend iff they sit in the same window (tile half) and carry the
//         same shifted-window region id (layers/attention.py:238-271,327-358).
#include <stdlib.h>

#include "attention_common.cuh"

namespace rfb {

// Key-split attention, second pass: one warp per (batch, head, query row) merges the chunks' partial results
// IN CHUNK ORDER (deterministic; a row's result does not depend on the grid that produced the chunks):
//   M = max_s m_s,  w_s = 2^(m_s - M),  O = sum_s w_s O_s / sum_s w_s l_s       (m_s in log2 units)
// part_o [split][B][H][Nq][128] fp32, part_ml [split][B][H][Nq][2]; O 16-bit [B][Nq][ldo], head h at column h*128.
template <bool F16>
__global__ void __launch_bounds__(256)
    attn_combine_kernel(const float* __restrict__ part_o, const float* __restrict__ part_ml, int n_splits, int B, int H,
                        int Nq, uint16_t* __restrict__ O, long long ldo, long long o_batch_stride) {
  const long long rows = (long long)B * H * Nq;
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int q = (int)(row % Nq);
  const int h = (int)((row / Nq) % H);
  const int b = (int)(row / ((long long)Nq * H));
  float m[8], l[8];
  float M = -INFINITY;
#pragma unroll
  for (int s = 0; s < 8; ++s)
    if (s < n_splits) {
      const float2 ml = *reinterpret_cast<const float2*>(part_ml + ((long long)s * rows + row) * 2);
      m[s] = ml.x, l[s] = ml.y;
      M = fmaxf(M, ml.x);
    }
  float L = 0.f;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int s = 0; s < 8; ++s)
    if (s < n_splits) {
      const float w = (m[s] == -INFINITY) ? 0.f : exp2f(m[s] - M);
      L = fmaf(w, l[s], L);
      const float4 o = *reinterpret_cast<const float4*>(part_o + ((long long)s * rows + row) * 128 + lane * 4);
      acc.x = fmaf(w, o.x, acc.x), acc.y = fmaf(w, o.y, acc.y), acc.z = fmaf(w, o.z, acc.z), acc.w = fmaf(w, o.w, acc.w);
    }
  const float inv = L > 0.f ? 1.0f / L : 0.f;
  uint2 u;
  u.x = pack16<F16>(acc.x * inv, acc.y * inv), u.y = pack16<F16>(acc.z * inv, acc.w * inv);
  *reinterpret_cast<uint2*>(O + (long long)b * o_batch_stride + (long long)q * ldo + h * 128 + lane * 4) = u;
}

// Parameters of the dense kernels (mode 0).  With n_splits > 1 the key chunks leave their results in part_o /
// part_ml (null otherwise).
static DenseAttnParams dense_attn_params(const rfb_attn_args* a, int k_batched, int v_batched, int n_splits,
                                         float* part_o, float* part_ml) {
  DenseAttnParams p{};
  p.B = a->B, p.split_tiles = n_splits > 1 ? a->kv_split_tiles : 0;
  p.part_o = part_o, p.part_ml = part_ml;
  p.Nq = a->Nq, p.Nk = a->Nk;
  p.n_kv_tiles = (a->Nk + 127) / 128;
  p.k_batched = k_batched, p.v_batched = v_batched;
  p.Q = static_cast<const uint16_t*>(a->Q), p.ldq = a->ldq;
  p.q_batch_stride = a->B > 1 ? a->q_batch_stride : 0;
  p.mask_bits = a->key_mask_bits;
  p.mask_stride_words = a->mask_batch_stride_words;
  p.O = a->O, p.ldo = a->ldo, p.o_batch_stride = a->o_batch_stride;
  p.scale_log2 = a->scale * 1.4426950408889634f;
  p.q_sumsq = a->q_sumsq, p.sumsq_ld = a->sumsq_ld > 0 ? a->sumsq_ld : 1;
  p.sumsq_parts = a->sumsq_parts > 0 ? a->sumsq_parts : 1;
  p.inv_norm_dim = a->norm_dim > 0 ? 1.0f / (float)a->norm_dim : 0.f, p.norm_eps = a->norm_eps;
  return p;
}

}  // namespace rfb

using namespace rfb;

extern "C" long long rfb_attention_ws_bytes(int B, int H, int Nq, int Nk, int kv_split_tiles) {
  if (kv_split_tiles <= 0 || B <= 0 || H <= 0 || Nq <= 0 || Nk <= 0) return 0;
  const int n_tiles = (Nk + 127) / 128;
  const int n_splits = (n_tiles + kv_split_tiles - 1) / kv_split_tiles;
  if (n_splits <= 1) return 0;
  return (long long)n_splits * B * H * Nq * (128 + 2) * 4;
}

extern "C" int rfb_attention(const rfb_attn_args* a, rfb_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!a || !a->Q || !a->K || !a->Vt || !a->O || a->B <= 0 || a->H <= 0 || a->Nq <= 0 || a->Nk <= 0)
    return RFB_ERR_ARG;
  if (a->mode == 1 && (!a->group_id || a->group_period <= 0 || a->Nq != a->Nk)) return RFB_ERR_ARG;
  if (a->ldo % 8) return RFB_ERR_ALIGN;
  if (a->dtype != 0 && a->dtype != RFB_BF16 && a->dtype != RFB_F16) return RFB_ERR_ARG;
  const int dt = a->dtype == RFB_F16 ? RFB_F16 : RFB_BF16;  // 0 (unset) = bf16

  const uint64_t hd_cols = (uint64_t)a->H * 128;
  CUtensorMap tmQ, tmK, tmV;
  int rc;
  const uint32_t box[3] = {64, 128, 1};
  {
    uint64_t dims[3] = {hd_cols, (uint64_t)a->Nq, (uint64_t)a->B};
    uint64_t st[2] = {(uint64_t)a->ldq * 2, (uint64_t)(a->B > 1 ? a->q_batch_stride : (long long)a->Nq * a->ldq) * 2};
    if ((rc = make_tmap_16b(&tmQ, dt, a->Q, 3, dims, st, box)) != RFB_OK) return rc;
  }
  const int k_batched = (a->B > 1 && a->k_batch_stride != 0);
  const int v_batched = (a->B > 1 && a->vt_batch_stride != 0);
  {
    uint64_t dims[3] = {hd_cols, (uint64_t)a->Nk, (uint64_t)(k_batched ? a->B : 1)};
    uint64_t st[2] = {(uint64_t)a->ldk * 2, (uint64_t)(k_batched ? a->k_batch_stride : (long long)a->Nk * a->ldk) * 2};
    if ((rc = make_tmap_16b(&tmK, dt, a->K, 3, dims, st, box)) != RFB_OK) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)a->Nk, hd_cols, (uint64_t)(v_batched ? a->B : 1)};
    uint64_t st[2] = {(uint64_t)a->ldvt * 2, (uint64_t)(v_batched ? a->vt_batch_stride : (long long)hd_cols * a->ldvt) * 2};
    if ((rc = make_tmap_16b(&tmV, dt, a->Vt, 3, dims, st, box)) != RFB_OK) return rc;
  }

  // key splitting (mode 0): chunks of kv_split_tiles key tiles, each on its own CTA, merged by attn_combine_kernel
  int n_splits = 1;
  float *part_o = nullptr, *part_ml = nullptr;
  if (a->kv_split_tiles < 0 || (a->kv_split_tiles > 0 && a->mode != 0)) return RFB_ERR_ARG;
  if (a->kv_split_tiles > 0) {
    const int n_tiles = (a->Nk + 127) / 128;
    n_splits = (n_tiles + a->kv_split_tiles - 1) / a->kv_split_tiles;
    if (n_splits > 8) return RFB_ERR_ARG;
    if (n_splits > 1) {
      const long long need = rfb_attention_ws_bytes(a->B, a->H, a->Nq, a->Nk, a->kv_split_tiles);
      if (!a->split_ws || a->split_ws_bytes < need || (reinterpret_cast<uintptr_t>(a->split_ws) & 15)) return RFB_ERR_ARG;
      part_o = static_cast<float*>(a->split_ws);
      part_ml = part_o + (long long)n_splits * a->B * a->H * a->Nq * 128;
    }
  }

  if (a->mode == 0) {
    static int forced = -1;  // RFB_ATTN_GEN = 2 | 3 forces one dense kernel generation (A/B runs)
    if (forced < 0) {
      const char* e = getenv("RFB_ATTN_GEN");
      forced = (e && e[0] >= '2' && e[0] <= '3') ? e[0] - '0' : 0;
    }
    int gen = forced;
    if (gen == 0) {
      // Both kernels sustain the same rate per tile; what differs is how evenly their grids fill
      // the SMs (one CTA per SM): two-tile CTAs (gen 2) vs one-tile CTAs (gen 3).
      const int sms = num_sms();
      const long long n2 = (long long)((a->Nq + 255) / 256) * a->H * a->B * n_splits;
      const long long n3 = (long long)((a->Nq + 127) / 128) * a->H * a->B * n_splits;
      const double e2 = (double)n2 / (double)(((n2 + sms - 1) / sms) * sms);
      const double e3 = (double)n3 / (double)(((n3 + sms - 1) / sms) * sms);
      gen = (e3 > e2 + 0.02) ? 3 : 2;
    }
    const DenseAttnParams p = dense_attn_params(a, k_batched, v_batched, n_splits, part_o, part_ml);
    rc = (gen == 3 ? launch_attention3 : launch_attention2)(tmQ, tmK, tmV, a, p, stream);
    if (rc != RFB_OK || n_splits <= 1) return rc;
    const long long rows = (long long)a->B * a->H * a->Nq;
    const unsigned blocks = (unsigned)((rows + 7) / 8);
    const long long obs = a->B > 1 ? a->o_batch_stride : 0;
    if (dt == RFB_F16)
      attn_combine_kernel<true><<<blocks, 256, 0, stream>>>(part_o, part_ml, n_splits, a->B, a->H, a->Nq,
                                                            static_cast<uint16_t*>(a->O), a->ldo, obs);
    else
      attn_combine_kernel<false><<<blocks, 256, 0, stream>>>(part_o, part_ml, n_splits, a->B, a->H, a->Nq,
                                                             static_cast<uint16_t*>(a->O), a->ldo, obs);
    g_launch_count++;
    return check_launch("attn_combine_kernel");
  }
  return launch_attention_swin(tmQ, tmK, tmV, a, k_batched, v_batched, stream);
}
