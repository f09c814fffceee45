// Arithmetic shared by the attention kernels: attn2_tc_kernel (attention2.cu), attn3_tc_kernel (attention3.cu)
// and, for the tile constants, the rms factor, the O store and the launch, attn_swin_kernel (attention_swin.cu).
//
// rfb_attention picks attn2 or attn3 from how evenly their grids fill the SMs, so the same query row may run
// on either kernel (a sharded render and a single-GPU render of the same job do): the two must give
// bit-identical results.  Everything they compute between the S tile in TMEM and the stored O row is defined
// here, once.  The barrier protocol around these steps differs between the kernels and stays in each kernel.
#pragma once
#include <atomic>

#include "host_util.h"
#include "ptx.cuh"

namespace rfb {

extern std::atomic<long long> g_launch_count;

constexpr uint32_t kAttnTile = 128 * 128 * 2;  // one 128 x 128 16-bit operand tile (two SW128 halves)
constexpr uint32_t kAttnHalf = 128 * 64 * 2;   // one 64-column swizzle half
// every kPolyEvery-th pair of exponentials goes to the FMA-pipe polynomial, the others to MUFU.EX2
constexpr int kPolyEvery = 4;

// Descriptor offset (16-byte units) of K step k (16 elements, 32 B) of a 128-wide K-major SW128 tile:
// four steps per 64-column half, the halves kAttnHalf apart.
__device__ __forceinline__ uint32_t sw128_kstep(int k) { return (k >> 2) * (kAttnHalf >> 4) + (k & 3) * 2; }

// 2^t for t in [-126, 0] on the FMA pipe, two lanes at a time: t = n + f, n = round(t), |f| <= 0.5,
// 2^f ~ degree-3 minimax polynomial (rel. error 7.5e-5, far below bf16 resolution of P), and 2^n is
// applied by adding n to the exponent field (r = t + 1.5*2^23 keeps n in its low mantissa bits).
__device__ __forceinline__ void exp2_poly2(uint64_t t2, float& p0, float& p1) {
  const float ta = fmaxf(lo2f(t2), -126.0f), tb = fmaxf(hi2f(t2), -126.0f);
  const uint64_t t = pack2f(ta, tb);
  const uint64_t r = fadd2(t, pack2f(12582912.0f, 12582912.0f));
  const uint64_t n = fadd2(r, pack2f(-12582912.0f, -12582912.0f));
  const uint64_t f = ffma2(n, pack2f(-1.0f, -1.0f), t);
  uint64_t p = ffma2(f, pack2f(0.0551716685f, 0.0551716685f), pack2f(0.2426111251f, 0.2426111251f));
  p = ffma2(p, f, pack2f(0.6932609677f, 0.6932609677f));
  p = ffma2(p, f, pack2f(0.9999280572f, 0.9999280572f));
  p0 = __uint_as_float(__float_as_uint(lo2f(p)) + (__float_as_uint(lo2f(r)) << 23));
  p1 = __uint_as_float(__float_as_uint(hi2f(p)) + (__float_as_uint(hi2f(r)) << 23));
}

// Fused RMSNorm: 1/rms of row `row` from its `parts` partial sums of squares (as the producing GEMM leaves them).
__device__ __forceinline__ float rms_factor(const float* sumsq, long long row, int ld, int parts, float inv_dim,
                                            float eps) {
  const float* sp = sumsq + row * ld;
  float ss = 0.f;
  for (int j = 0; j < parts; ++j) ss += sp[j];
  return rsqrtf(ss * inv_dim + eps);
}

// O row of a tile (TMEM columns tO .. tO+127 of this thread's lane) times inv_l -> 16-bit -> orow[0, 128).
template <bool F16>
__device__ __forceinline__ void store_o_row(uint32_t tO, uint16_t* orow, bool row_ok, float inv_l) {
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    uint32_t o[32];
    tmem_ld32(tO + c * 32, o);
    tmem_wait_ld();
    if (row_ok) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        uint4 u;
        u.x = pack16<F16>(__uint_as_float(o[i * 8 + 0]) * inv_l, __uint_as_float(o[i * 8 + 1]) * inv_l);
        u.y = pack16<F16>(__uint_as_float(o[i * 8 + 2]) * inv_l, __uint_as_float(o[i * 8 + 3]) * inv_l);
        u.z = pack16<F16>(__uint_as_float(o[i * 8 + 4]) * inv_l, __uint_as_float(o[i * 8 + 5]) * inv_l);
        u.w = pack16<F16>(__uint_as_float(o[i * 8 + 6]) * inv_l, __uint_as_float(o[i * 8 + 7]) * inv_l);
        *reinterpret_cast<uint4*>(orow + c * 32 + i * 8) = u;
      }
    }
  }
}

// ------------------------------ dense kernels (mode 0): attn2 and attn3 ------------------------------

struct DenseAttnParams {
  int Nq, Nk, n_kv_tiles;
  int k_batched, v_batched;
  const uint16_t* Q;  // attn3 reads Q rows directly (attn2 loads them through the Q tensor map)
  long long ldq, q_batch_stride;
  const uint32_t* mask_bits;
  long long mask_stride_words;
  void* O;
  long long ldo, o_batch_stride;
  float scale_log2;
  const float* q_sumsq;
  int sumsq_ld, sumsq_parts;
  float inv_norm_dim, norm_eps;
  // key splitting: blockIdx.z = b + B * split; split s visits key tiles [s*split_tiles, min(.., n_kv_tiles)) and
  // leaves its un-normalised result in part_o / part_ml (attention.cu: attn_combine_kernel finishes the job)
  int B, split_tiles;
  float* part_o;   // [split][B][H][Nq][128] fp32
  float* part_ml;  // [split][B][H][Nq][2]   (running max in log2 units, running sum)

  int n_splits() const { return split_tiles > 0 ? (n_kv_tiles + split_tiles - 1) / split_tiles : 1; }
};

// The key tiles of this CTA: its split, the first key tile, how many it visits, and the local index of the
// sequence's short tail tile.
struct DenseTiles {
  int split, j_begin, n_tiles;
  // Short tail: when the LAST key tile of the sequence holds <= 32 keys (16 register tokens + a multiple of 128
  // triangles is the common case) its products run 32 keys wide -- S = Q K^T with N = 32, P V with two K = 16
  // steps -- and the softmax touches one 32-column chunk instead of four.  The skipped columns are masked keys,
  // whose probabilities are exactly 0: the result is bit-identical to the full-width tile.
  int tail_local;  // local index, or -1 (never)
};
__device__ __forceinline__ DenseTiles dense_tiles(const DenseAttnParams& p) {
  DenseTiles t;
  t.split = p.split_tiles > 0 ? blockIdx.z / p.B : 0;
  t.j_begin = t.split * p.split_tiles;
  t.n_tiles = p.split_tiles > 0 ? min(p.split_tiles, p.n_kv_tiles - t.j_begin) : p.n_kv_tiles;
  t.tail_local = (p.Nk - (p.n_kv_tiles - 1) * 128 <= 32) ? p.n_kv_tiles - 1 - t.j_begin : -1;
  return t;
}

// Softmax scale of query row qrow in log2 units; the fused q RMSNorm folds the row's 1/rms into it.
__device__ __forceinline__ float dense_scale_log2(const DenseAttnParams& p, int b, int qrow) {
  float sl2 = p.scale_log2;
  if (p.q_sumsq && qrow < p.Nq)
    sl2 *= rms_factor(p.q_sumsq, static_cast<long long>(b) * p.Nq + qrow, p.sumsq_ld, p.sumsq_parts,
                      p.inv_norm_dim, p.norm_eps);
  return sl2;
}

// Keys of key tile `tile` that may be attended, bit i of word w for key tile*128 + 32w + i: the packed key mask,
// or without one every key below Nk.
__device__ __forceinline__ void key_mask_words(const DenseAttnParams& p, int b, int tile, uint32_t (&mw)[4]) {
  if (p.mask_bits) {
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(p.mask_bits + static_cast<long long>(b) * p.mask_stride_words + tile * 4));
    mw[0] = u.x, mw[1] = u.y, mw[2] = u.z, mw[3] = u.w;
  } else {
    const int rem = p.Nk - tile * 128;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const int lo = w * 32;
      mw[w] = rem <= lo ? 0u : (rem - lo >= 32 ? 0xffffffffu : ((1u << (rem - lo)) - 1u));
    }
  }
}

// Online softmax of one key tile, in three steps; the kernel orders them against its barriers.
//   (a) softmax_max:   S row (nc 32-column chunks at tS) -> registers v, masked keys -> -inf, new running max
//   (b) rescale_o:     O *= alpha (only needed when some row's max moved)
//   (c) softmax_exp:   P = 2^(s*sl2 - m*sl2) as 16-bit pairs over columns [0, 64) of S; returns the row sum
//   then l_run = fmaf(l_run, alpha, row sum) (one rounding), m_run = m_new.
struct SoftmaxMax {
  float m_new, alpha, neg_ms;
};
__device__ __forceinline__ SoftmaxMax softmax_max(uint32_t tS, int nc, const uint32_t (&mw)[4], float m_run,
                                                  float sl2, uint32_t (&v)[4][32]) {
  tmem_ld32(tS, v[0]);
  if (nc == 4) {
    tmem_ld32(tS + 32, v[1]);
    tmem_ld32(tS + 64, v[2]);
    tmem_ld32(tS + 96, v[3]);
  }
  tmem_wait_ld();

  if ((mw[0] & mw[1] & mw[2] & mw[3]) != 0xffffffffu) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      if (c < nc) {
        const uint32_t bits = mw[c];
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (!((bits >> i) & 1u)) v[c][i] = 0xff800000u;  // -inf
      }
    }
  }
  float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
  for (int c = 0; c < 4; ++c)
    if (c < nc) {
#pragma unroll
      for (int i = 0; i < 32; ++i) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(v[c][i]));
    }
  const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
  SoftmaxMax s;
  s.m_new = fmaxf(m_run, mx);
  const float m_use = (s.m_new == -INFINITY) ? 0.f : s.m_new;
  s.alpha = (m_run == -INFINITY) ? 0.f : ex2_f((m_run - m_use) * sl2);
  s.neg_ms = -m_use * sl2;
  return s;
}

__device__ __forceinline__ void rescale_o(uint32_t tO, float alpha) {
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    uint32_t o[32];
    tmem_ld32(tO + c * 32, o);
    tmem_wait_ld();
#pragma unroll
    for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
    tmem_st32(tO + c * 32, o);
  }
}

template <bool F16>
__device__ __forceinline__ float softmax_exp(const uint32_t (&v)[4][32], uint32_t tS, int nc, float sl2,
                                             float neg_ms) {
  const uint64_t sl2_2 = pack2f(sl2, sl2), nms_2 = pack2f(neg_ms, neg_ms);
  uint64_t rs2[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    if (c >= nc) continue;
    uint32_t pk[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const uint64_t t2 = ffma2(pack2f(__uint_as_float(v[c][2 * i]), __uint_as_float(v[c][2 * i + 1])), sl2_2, nms_2);
      float p0, p1;
      if (i % kPolyEvery == kPolyEvery - 1) {
        exp2_poly2(t2, p0, p1);
      } else {
        p0 = ex2_f(lo2f(t2)), p1 = ex2_f(hi2f(t2));
      }
      rs2[i & 3] = fadd2(rs2[i & 3], pack2f(p0, p1));
      pk[i] = pack16<F16>(p0, p1);
    }
    tmem_st16(tS + c * 16, pk);
  }
  const uint64_t rsum = fadd2(fadd2(rs2[0], rs2[1]), fadd2(rs2[2], rs2[3]));
  return lo2f(rsum) + hi2f(rsum);
}

// Epilogue of query row qrow (O at TMEM tO of this thread's lane): O / l as 16-bit into O, or with key splitting
// the un-normalised O (relative to m_run) and (m_run in log2 units, l_run) into part_o / part_ml.
template <bool F16>
__device__ __forceinline__ void dense_store_row(const DenseAttnParams& p, uint32_t tO, int split, int b, int h,
                                                int qrow, float m_run, float l_run, float sl2) {
  const bool row_ok = qrow < p.Nq;
  if (p.part_o) {
    const long long prow = ((static_cast<long long>(split) * p.B + b) * gridDim.y + h) * p.Nq + qrow;
    if (row_ok) {
      float2* ml = reinterpret_cast<float2*>(p.part_ml) + prow;
      *ml = make_float2(m_run * sl2, l_run);
    }
    float* po = p.part_o + prow * 128;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {
      uint32_t o[32];
      tmem_ld32(tO + c * 32, o);
      tmem_wait_ld();
      if (row_ok) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
          *reinterpret_cast<uint4*>(po + c * 32 + i * 4) = make_uint4(o[i * 4], o[i * 4 + 1], o[i * 4 + 2], o[i * 4 + 3]);
      }
    }
  } else {
    const float inv_l = (l_run > 0.f) ? 1.0f / l_run : 0.f;
    uint16_t* orow = static_cast<uint16_t*>(p.O) + static_cast<long long>(b) * p.o_batch_stride +
                     static_cast<long long>(qrow) * p.ldo + h * 128;
    store_o_row<F16>(tO, orow, row_ok, inv_l);
  }
}

// ------------------------------ host side ------------------------------

// The launchers, called by rfb_attention (attention.cu).  The dense ones share a signature; attn3 does not use tmQ.
int launch_attention2(const CUtensorMap& tmQ, const CUtensorMap& tmK, const CUtensorMap& tmV,
                      const rfb_attn_args* a, const DenseAttnParams& p, cudaStream_t stream);
int launch_attention3(const CUtensorMap& tmQ, const CUtensorMap& tmK, const CUtensorMap& tmV,
                      const rfb_attn_args* a, const DenseAttnParams& p, cudaStream_t stream);
int launch_attention_swin(const CUtensorMap& tmQ, const CUtensorMap& tmK, const CUtensorMap& tmV,
                          const rfb_attn_args* a, int k_batched, int v_batched, cudaStream_t stream);

// Launches an attention kernel: raises its dynamic shared-memory limit the first time on this device (smem_set
// is the caller's per-device flag for this kernel instance), counts the launch and checks it.
template <typename... KArgs, typename... Args>
inline int launch_attn_kernel(void (*kern)(KArgs...), const char* name, bool& smem_set, uint32_t smem, dim3 grid,
                              int threads, cudaStream_t stream, const Args&... args) {
  if (!smem_set) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess)
      return RFB_ERR_LAUNCH;
    smem_set = true;
  }
  kern<<<grid, threads, smem, stream>>>(args...);
  g_launch_count++;
  return check_launch(name);
}

}  // namespace rfb
