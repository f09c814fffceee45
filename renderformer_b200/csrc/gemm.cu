// Persistent, warp-specialised tcgen05 GEMM for sm_100a.
//
//   C[M,N] = A[M,K] * W[N,K]^T     16-bit operands (bf16 or fp16), fp32 accumulate in TMEM
//
// Roles (320 threads): warp 0 = TMA producer (one lane), warp 1 = tcgen05.mma issuer (one lane,
// also owns the TMEM allocation), warps 2..9 = epilogue (TMEM -> registers -> fused math -> HBM;
// two warps per TMEM lane quarter, alternating 32-column chunks).
// The accumulator is double-buffered in TMEM so the epilogue of tile i overlaps the main loop
// of tile i+1.  A-operand tiles come either from a 2-D tensor map (linear layers) or from a
// 4-D NHWC tensor map walked over the 9 filter taps (3x3 convolution as implicit GEMM; the
// zero padding is TMA's out-of-bounds fill, negative coordinates included).
//
// Reference call sites replaced: see include/rfb200.h (rfb_gemm).
#include <stdlib.h>

#include <atomic>

#include "host_util.h"
#include "ptx.cuh"

namespace rfb {

std::atomic<long long> g_launch_count{0};

struct GemmKParams {
  int M, N, K;
  int num_m_tiles, num_n_tiles, num_kb;
  int a_mode;
  int H, Wd, Cin, tw, th, tiles_x, tiles_y, kb_per_tap;
  uint32_t idesc;
  int epi;
  const float* bias;
  const void* res1;
  const void* res2;
  int res_dtype;
  long long ldres;
  void* out;
  int out_dtype;
  long long ldo;
  void* out_act;
  const int* row_map;
  const float* w2;
  const float* b2;
  int n_store;
  int direct_store;  // debug: thread-per-row stores instead of the smem-transposed path
  // fused RMSNorm plumbing
  const float* in_sumsq;  // per-row partial sums of squares [M][in_sumsq_ld], first in_sumsq_parts entries
  int in_sumsq_ld, in_sumsq_parts;
  const float* in_rscale;  // ready-made factors: per A row (scale_dim 0) or per output column (1)
  int scale_dim;
  float inv_norm_dim, norm_eps;
  float* out_rscale;  // [M] side output of the per-row factor derived from in_sumsq
  float* out_sumsq;   // [rows][out_sumsq_ld]: entry n/128 = sum of v^2 over that 128-column part
  int out_sumsq_ld;
  void* out16;
  int out16_dtype;
  long long ld16;
  const float* col_mul;
  const int* aux_row_map;
  // transposed side output: columns n >= vt_split go to vt_out[b][n - vt_split][row] (16-bit, x r)
  void* vt_out;
  int vt_dtype, vt_split, vt_rows_per_batch;
  long long vt_ld, vt_batch_stride;
  // conv output crop (final epilogue only; crop_w == 0: none): only pixels of the window [crop_top, +crop_h) x
  // [crop_left, +crop_w) are stored, to row (b * crop_h + y - crop_top) * crop_w + x - crop_left
  int crop_h, crop_w, crop_top, crop_left;
};

// output row of conv pixel (b, y, x); false when the pixel lies outside the image or outside the crop window
__device__ __forceinline__ bool conv_out_row(const GemmKParams& p, int b, int y, int x, long long& orow) {
  if (p.crop_w) {
    y -= p.crop_top, x -= p.crop_left;
    orow = (static_cast<long long>(b) * p.crop_h + y) * p.crop_w + x;
    return static_cast<unsigned>(y) < static_cast<unsigned>(p.crop_h) &&
           static_cast<unsigned>(x) < static_cast<unsigned>(p.crop_w);
  }
  orow = (static_cast<long long>(b) * p.H + y) * p.Wd + x;
  return (y < p.H) && (x < p.Wd);
}

constexpr int kBM = 128;
constexpr int kBK = 64;
constexpr uint32_t kABytes = kBM * kBK * 2;

// epilogue: 8 warps (two per TMEM lane quarter, alternating 32-column chunks), each with a
// 32 x 32 fp32 transposition buffer (16-byte chunks XOR-swizzled by row, no padding)
constexpr int kEpiWarps = 8;
constexpr int kGemmThreads = 64 + kEpiWarps * 32;
// EK_RESID variant: warpgroup 0 = {TMA, MMA, 2 idle warps}, warpgroups 1-2 = epilogue; setmaxnreg hands
// warpgroup 0's registers to the epilogue warps so that the residual of a warp's whole half tile
// (4 chunks x 8 row slots x 16 B) can be in flight while the main loop of the tile is still running.
constexpr int kGemmThreadsWG = 128 + kEpiWarps * 32;
constexpr int kRegsGemmWg0 = 56, kRegsGemmEpi = 224;  // 128*56 + 256*224 = 384*168
constexpr uint32_t kEpiStageBytes = kEpiWarps * 32 * 32 * 4;

template <int BN>
struct GemmCfg {
  static constexpr uint32_t kBBytes = BN * kBK * 2;
  static constexpr int kStages = (BN == 256) ? 4 : (BN == 128 ? 6 : 8);
  static constexpr uint32_t kTmemCols = (2 * BN < 32) ? 32 : 2 * BN;
  static constexpr uint32_t kSmemBytes = kStages * (kABytes + kBBytes) + 1024 + 256 + kEpiStageBytes;
};

__device__ __forceinline__ void load8(const void* base, int dtype, long long idx, float (&x)[8]) {
  if (dtype == RFB_F32) {
    const float4* p = reinterpret_cast<const float4*>(static_cast<const float*>(base) + idx);
    float4 a = p[0], b = p[1];
    x[0] = a.x, x[1] = a.y, x[2] = a.z, x[3] = a.w, x[4] = b.x, x[5] = b.y, x[6] = b.z, x[7] = b.w;
  } else {
    uint4 u = *reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(base) + idx);
    uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (dtype == RFB_BF16) {
        x[2 * i] = __uint_as_float(w[i] << 16);
        x[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
      } else {
        __half2 h = *reinterpret_cast<__half2*>(&w[i]);
        float2 f = __half22float2(h);
        x[2 * i] = f.x, x[2 * i + 1] = f.y;
      }
    }
  }
}

__device__ __forceinline__ void store8(void* base, int dtype, long long idx, const float (&x)[8]) {
  if (dtype == RFB_F32) {
    float4* p = reinterpret_cast<float4*>(static_cast<float*>(base) + idx);
    p[0] = make_float4(x[0], x[1], x[2], x[3]);
    p[1] = make_float4(x[4], x[5], x[6], x[7]);
  } else {
    uint4 u;
    if (dtype == RFB_BF16) {
      u.x = pack_bf16(x[0], x[1]), u.y = pack_bf16(x[2], x[3]);
      u.z = pack_bf16(x[4], x[5]), u.w = pack_bf16(x[6], x[7]);
    } else {
      u.x = pack_f16(x[0], x[1]), u.y = pack_f16(x[2], x[3]);
      u.z = pack_f16(x[4], x[5]), u.w = pack_f16(x[6], x[7]);
    }
    *reinterpret_cast<uint4*>(static_cast<uint16_t*>(base) + idx) = u;
  }
}

// One thread owns one output row; v = 32 consecutive accumulator columns starting at n0.
__device__ __forceinline__ void epilogue_chunk(const GemmKParams& p, long long orow, int n0,
                                               const uint32_t (&v)[32], float rs) {
  if (p.epi == RFB_EPI_STORE) {
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const int n = n0 + g * 8;
      if (n >= p.n_store) break;
      float x[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] = __uint_as_float(v[g * 8 + j]);
      if (p.bias) {
        float b[8];
        load8(p.bias, RFB_F32, n, b);
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] += b[j];
      }
      if (p.res1) {
        float r[8];
        load8(p.res1, p.res_dtype, orow * p.ldres + n, r);
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] += r[j];
      }
      if (p.res2) {
        float r[8];
        load8(p.res2, p.res_dtype, orow * p.ldres + n, r);
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] += r[j];
      }
      if (p.out) store8(p.out, p.out_dtype, orow * p.ldo + n, x);
      if (p.out_act) {
#pragma unroll
        for (int j = 0; j < 8; ++j) x[j] = silu_f(x[j]);
        store8(p.out_act, p.out_dtype, orow * p.ldo + n, x);
      }
    }
  } else if (p.epi == RFB_EPI_SWIGLU) {
    if (n0 >= p.N) return;
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      float h[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float gate = __uint_as_float(v[g * 8 + j]) * rs;
        const float up = __uint_as_float(v[16 + g * 8 + j]) * rs;
        h[j] = silu_f(gate) * up;
      }
      store8(p.out, p.out_dtype, orow * p.ldo + (n0 >> 1) + g * 8, h);
    }
  } else {  // RFB_EPI_FINAL / RFB_EPI_FINAL_RAW (N == 32, n0 == 0)
    float h[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) h[j] = silu_f(__uint_as_float(v[j]) + __ldg(p.bias + j));
    float* o = static_cast<float*>(p.out) + orow * p.ldo;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float y = __ldg(p.b2 + c);
#pragma unroll
      for (int j = 0; j < 32; ++j) y = fmaf(__ldg(p.w2 + c * 32 + j), h[j], y);
      if (p.epi == RFB_EPI_FINAL_RAW) {
        o[c] = y;                             // DPTHead.forward's own output  layers/dpt.py:271
      } else {
        y = y > 0.f ? y : 1e-3f * expm1f(y);  // ELU(alpha=1e-3)  view_transformer.py:86,122
        o[c] = exp10f(y) - 1.0f;              // rendering_pipeline.py:122-123
      }
    }
  }
}

__device__ __forceinline__ void load4(const void* base, int dtype, long long idx, float (&x)[4]) {
  if (dtype == RFB_F32) {
    const float4 a = *reinterpret_cast<const float4*>(static_cast<const float*>(base) + idx);
    x[0] = a.x, x[1] = a.y, x[2] = a.z, x[3] = a.w;
  } else {
    const uint2 u = *reinterpret_cast<const uint2*>(static_cast<const uint16_t*>(base) + idx);
    if (dtype == RFB_BF16) {
      x[0] = __uint_as_float(u.x << 16), x[1] = __uint_as_float(u.x & 0xffff0000u);
      x[2] = __uint_as_float(u.y << 16), x[3] = __uint_as_float(u.y & 0xffff0000u);
    } else {
      const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
      const float2 f1 = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
      x[0] = f0.x, x[1] = f0.y, x[2] = f1.x, x[3] = f1.y;
    }
  }
}

__device__ __forceinline__ void store4(void* base, int dtype, long long idx, const float (&x)[4]) {
  if (dtype == RFB_F32) {
    *reinterpret_cast<float4*>(static_cast<float*>(base) + idx) = make_float4(x[0], x[1], x[2], x[3]);
  } else {
    uint2 u;
    if (dtype == RFB_BF16) {
      u.x = pack_bf16(x[0], x[1]), u.y = pack_bf16(x[2], x[3]);
    } else {
      u.x = pack_f16(x[0], x[1]), u.y = pack_f16(x[2], x[3]);
    }
    *reinterpret_cast<uint2*>(static_cast<uint16_t*>(base) + idx) = u;
  }
}

// RFB_EPI_STORE through a per-warp smem transposition: the accumulator chunk arrives with one
// thread per row (TMEM lane); it leaves with 8 consecutive lanes covering 128 contiguous bytes
// of one row, so residual reads and output writes are fully coalesced (4 rows per instruction).
// Row slot `it` of a lane is tile row it*4 + (lane>>3); the per-row metadata (output row, aux
// row, 1/rms) lives in the row-owner lane and is fetched with a shuffle where it is needed, so
// the only per-chunk register arrays are the accumulator and the raw residual bits.
// Epilogue kinds: the generic one reads every feature flag at run time; the two specialised ones
// fix the flags of the decoder's hot shapes at compile time, which removes the per-row-slot
// uniform branches (the epilogue is instruction-latency bound: 2 warps per scheduler).
constexpr int EK_GENERIC = 0;
constexpr int EK_RESID = 1;   // out f32 = acc*r + res1 f32, + bf16 copy + partial sums of squares
constexpr int EK_PROJ16 = 2;  // out16 bf16 = acc*r*col_mul only, + partial sums of squares
constexpr int EK_RESID_H = 3;   // the same two with an fp16 (half) 16-bit side output
constexpr int EK_PROJ16_H = 4;
__host__ __device__ constexpr bool ek_resid(int ek) { return ek == EK_RESID || ek == EK_RESID_H; }
__host__ __device__ constexpr bool ek_fast(int ek) { return ek >= EK_RESID && ek <= EK_PROJ16_H; }
__host__ __device__ constexpr bool ek_half(int ek) { return ek == EK_RESID_H || ek == EK_PROJ16_H; }
// EK >= EK_CONV: the generic epilogue with its flags fixed at compile time for the DPT convolutions
// (fp16 in / out, 128-wide tile): EK = EK_CONV + mask, mask bits below
constexpr int EK_CONV = 16;
constexpr int CF_OUT = 1, CF_ACT = 2, CF_BIAS = 4, CF_RES1 = 8, CF_RES2 = 16;

__device__ __forceinline__ void unpack16x2(uint32_t u, int dtype, float& lo, float& hi) {
  if (dtype == RFB_BF16) {
    lo = __uint_as_float(u << 16), hi = __uint_as_float(u & 0xffff0000u);
  } else {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&u));
    lo = f.x, hi = f.y;
  }
}

// ---------------------------------------------------------------------------------------------
// Generic RFB_EPI_STORE epilogue of one warp's share [c_begin, c_end) of the tile's 32-column
// chunks; every feature is a run-time (warp-uniform) flag.  The work of a chunk is split into
// one straight-line pass over the 8 row slots per feature ("loop fission"), so a flag costs one
// uniform branch per chunk instead of one per row slot and each pass schedules as a block.
// ---------------------------------------------------------------------------------------------
template <int EK>
__device__ __forceinline__ void epilogue_generic_coalesced(const GemmKParams& p, float* stage, int lane,
                                                           uint32_t taddr0, int n0, int c_begin, int c_end,
                                                           int orow_mine, int arow_mine, float rs_mine,
                                                           uint64_t* tfull_bar, uint32_t parity) {
  const int c4 = lane & 7;
  const int g4 = lane >> 3;
  int orow[8];
  float rs[8];
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    orow[it] = __shfl_sync(0xffffffffu, orow_mine, it * 4 + g4);
    rs[it] = __shfl_sync(0xffffffffu, rs_mine, it * 4 + g4);
  }
  constexpr bool RT = EK < EK_CONV;  // flags read at run time
  constexpr int CM = RT ? 0 : EK - EK_CONV;
  const bool f_out = RT ? p.out != nullptr : (CM & CF_OUT) != 0;
  const bool f_res = RT ? p.res1 != nullptr : (CM & CF_RES1) != 0;
  const bool f_res32 = RT ? p.res_dtype == RFB_F32 : false;
  const bool f_res2 = RT ? p.res2 != nullptr : (CM & CF_RES2) != 0;
  const bool f_out16 = RT ? p.out16 != nullptr : false;
  const bool f_sumsq = RT ? p.out_sumsq != nullptr : false;
  const bool f_act = RT ? p.out_act != nullptr : (CM & CF_ACT) != 0;
  const bool f_bias = RT ? p.bias != nullptr : (CM & CF_BIAS) != 0;
  const bool f_cm = RT ? p.col_mul != nullptr : false;
  const bool f_cs = RT ? (p.in_rscale != nullptr && p.scale_dim == 1) : false;
  const int out_dtype = RT ? p.out_dtype : RFB_F16;
  const int res_dtype = RT ? p.res_dtype : RFB_F16;
  float sqp[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  uint4 cur[8], nxt[8];  // raw residual bits; 16-bit residuals: res1 in (x,y), res2 in (z,w)
  auto prefetch = [&](uint4(&r)[8], int n) {
    if (n >= p.n_store) return;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      if (orow[it] < 0) continue;
      const long long idx = (long long)orow[it] * p.ldres + n;
      if (f_res32) {
        r[it] = *reinterpret_cast<const uint4*>(static_cast<const float*>(p.res1) + idx);
      } else {
        const uint2 a = *reinterpret_cast<const uint2*>(static_cast<const uint16_t*>(p.res1) + idx);
        r[it].x = a.x, r[it].y = a.y;
        if (f_res2) {
          const uint2 b = *reinterpret_cast<const uint2*>(static_cast<const uint16_t*>(p.res2) + idx);
          r[it].z = b.x, r[it].w = b.y;
        }
      }
    }
  };
  // the first chunk's residual does not depend on the accumulator: fetch it while the main loop
  // of this tile is still running
  if (f_res && c_begin < c_end) prefetch(cur, n0 + c_begin * 32 + c4 * 4);
  mbar_wait(tfull_bar, parity);
  tc_fence_after();
#pragma unroll 1
  for (int c = c_begin; c < c_end; ++c) {
    if (n0 + c * 32 >= p.n_store) break;  // warp-uniform
    uint32_t v[32];
    tmem_ld32(taddr0 + c * 32, v);
    const int n = n0 + c * 32 + c4 * 4;
    const bool col_ok = n < p.n_store;
    if (f_res && c + 1 < c_end) prefetch(nxt, n + 32);
    tmem_wait_ld();
#pragma unroll
    for (int g = 0; g < 8; ++g)
      *reinterpret_cast<float4*>(stage + lane * 32 + ((g ^ c4) << 2)) =
          make_float4(__uint_as_float(v[g * 4]), __uint_as_float(v[g * 4 + 1]), __uint_as_float(v[g * 4 + 2]),
                      __uint_as_float(v[g * 4 + 3]));
    __syncwarp();
    float x[8][4];
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int rr = it * 4 + g4;
      const float4 a = *reinterpret_cast<const float4*>(stage + rr * 32 + ((c4 ^ (rr & 7)) << 2));
      x[it][0] = a.x * rs[it], x[it][1] = a.y * rs[it], x[it][2] = a.z * rs[it], x[it][3] = a.w * rs[it];
    }
    __syncwarp();
    if (f_cs || f_bias) {
      float cs[4] = {1.f, 1.f, 1.f, 1.f}, bias[4] = {0.f, 0.f, 0.f, 0.f};
      if (col_ok && f_cs) load4(p.in_rscale, RFB_F32, n, cs);
      if (col_ok && f_bias) load4(p.bias, RFB_F32, n, bias);
#pragma unroll
      for (int it = 0; it < 8; ++it)
#pragma unroll
        for (int j = 0; j < 4; ++j) x[it][j] = fmaf(x[it][j], cs[j], bias[j]);
    }
    if (f_res) {
      if (f_res32) {
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          x[it][0] += __uint_as_float(cur[it].x), x[it][1] += __uint_as_float(cur[it].y);
          x[it][2] += __uint_as_float(cur[it].z), x[it][3] += __uint_as_float(cur[it].w);
        }
      } else {
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          float r0, r1, r2, r3;
          unpack16x2(cur[it].x, res_dtype, r0, r1), unpack16x2(cur[it].y, res_dtype, r2, r3);
          x[it][0] += r0, x[it][1] += r1, x[it][2] += r2, x[it][3] += r3;
        }
        if (f_res2) {
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            float r0, r1, r2, r3;
            unpack16x2(cur[it].z, res_dtype, r0, r1), unpack16x2(cur[it].w, res_dtype, r2, r3);
            x[it][0] += r0, x[it][1] += r1, x[it][2] += r2, x[it][3] += r3;
          }
        }
      }
    }
    if (f_out) {
      if (out_dtype == RFB_F32) {
#pragma unroll
        for (int it = 0; it < 8; ++it)
          if (orow[it] >= 0 && col_ok) store4(p.out, RFB_F32, (long long)orow[it] * p.ldo + n, x[it]);
      } else if (out_dtype == RFB_BF16) {
#pragma unroll
        for (int it = 0; it < 8; ++it)
          if (orow[it] >= 0 && col_ok) store4(p.out, RFB_BF16, (long long)orow[it] * p.ldo + n, x[it]);
      } else {
#pragma unroll
        for (int it = 0; it < 8; ++it)
          if (orow[it] >= 0 && col_ok) store4(p.out, RFB_F16, (long long)orow[it] * p.ldo + n, x[it]);
      }
    }
    if (f_sumsq) {
#pragma unroll
      for (int it = 0; it < 8; ++it)
        if (orow[it] >= 0 && col_ok)
          sqp[it] += x[it][0] * x[it][0] + x[it][1] * x[it][1] + x[it][2] * x[it][2] + x[it][3] * x[it][3];
    }
    if (f_out16) {
      float cm[4] = {1.f, 1.f, 1.f, 1.f};
      if (col_ok && f_cm) load4(p.col_mul, RFB_F32, n, cm);
      const bool aux = p.aux_row_map != nullptr;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        int arow = orow[it];
        if (aux) arow = __shfl_sync(0xffffffffu, arow_mine, it * 4 + g4);
        if (orow[it] >= 0 && col_ok) {
          const float y[4] = {x[it][0] * cm[0], x[it][1] * cm[1], x[it][2] * cm[2], x[it][3] * cm[3]};
          store4(p.out16, p.out16_dtype, (long long)arow * p.ld16 + n, y);
        }
      }
    }
    if (f_act) {
      const bool bf = out_dtype == RFB_BF16;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        float y[4] = {silu_f(x[it][0]), silu_f(x[it][1]), silu_f(x[it][2]), silu_f(x[it][3])};
        if (orow[it] >= 0 && col_ok) {
          if (out_dtype == RFB_F32) store4(p.out_act, RFB_F32, (long long)orow[it] * p.ldo + n, y);
          else if (bf) store4(p.out_act, RFB_BF16, (long long)orow[it] * p.ldo + n, y);
          else store4(p.out_act, RFB_F16, (long long)orow[it] * p.ldo + n, y);
        }
      }
    }
    if (f_res) {
#pragma unroll
      for (int it = 0; it < 8; ++it) cur[it] = nxt[it];
    }
  }
  // BN == 256 whenever out_sumsq is set: this warp's columns are exactly one 128-column part
  if (f_sumsq && n0 + c_begin * 32 < p.n_store) {
    float mine = 0.f;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      float t = sqp[it];
      t += __shfl_xor_sync(0xffffffffu, t, 1);
      t += __shfl_xor_sync(0xffffffffu, t, 2);
      t += __shfl_xor_sync(0xffffffffu, t, 4);
      t = __shfl_sync(0xffffffffu, t, (lane & 3) * 8);
      if ((lane >> 2) == it) mine = t;
    }
    if (orow_mine >= 0) p.out_sumsq[(long long)arow_mine * p.out_sumsq_ld + ((n0 + c_begin * 32) >> 7)] = mine;
  }
}

// ---------------------------------------------------------------------------------------------
// Transposed tile: the V part of a fused [q | k | v] projection.  A thread owns one row (token) and
// 32 consecutive columns (feature dims); for a fixed column the warp's 32 lanes hold 32 consecutive
// tokens, so each column is one 64-byte store into V^T[dim][token] -- no staging needed.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void epilogue_vt_chunks(const GemmKParams& p, uint32_t taddr0, int n0, int c_begin,
                                                   int c_end, int m, bool valid, float rs, uint64_t* tfull_bar,
                                                   uint32_t parity) {
  mbar_wait(tfull_bar, parity);
  tc_fence_after();
  const int b = p.vt_rows_per_batch > 0 ? m / p.vt_rows_per_batch : 0;
  const int mrow = m - b * p.vt_rows_per_batch;
  uint16_t* base = static_cast<uint16_t*>(p.vt_out) + (long long)b * p.vt_batch_stride + mrow;
#pragma unroll 1
  for (int c = c_begin; c < c_end; ++c) {
    if (n0 + c * 32 >= p.N) break;  // warp-uniform
    uint32_t v[32];
    tmem_ld32(taddr0 + c * 32, v);
    tmem_wait_ld();
    if (valid) {
      uint16_t* col = base + (long long)(n0 + c * 32 - p.vt_split) * p.vt_ld;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        if (n0 + c * 32 + i < p.N) {
          const float x = __uint_as_float(v[i]) * rs;
          uint16_t h;
          if (p.vt_dtype == RFB_BF16) {
            h = static_cast<uint16_t>(pack_bf16(x, 0.f) & 0xffffu);
          } else {
            h = static_cast<uint16_t>(pack_f16(x, 0.f) & 0xffffu);
          }
          col[(long long)i * p.vt_ld] = h;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Specialised epilogue of one warp's half tile (4 chunks of 32 columns, BN == 256, N % 256 == 0)
// for EK_RESID / EK_PROJ16.  Everything that is constant over the tile's chunks (output rows,
// 1/rms, smem addresses) lives in registers, the chunk loop is fully unrolled so the residual
// prefetch ping-pongs between two register sets without copies, and the sums of squares are
// reduced across lanes once per tile instead of once per chunk.
// ---------------------------------------------------------------------------------------------
// x0^2 + x1^2 + x2^2 + x3^2 with the contraction pinned (the 256- and 128-wide tiles must agree bit for bit)
__device__ __forceinline__ float sq4(const float (&x)[4]) {
  return __fmaf_rn(x[3], x[3], __fmaf_rn(x[2], x[2], __fmaf_rn(x[1], x[1], __fmul_rn(x[0], x[0]))));
}

// NCHW = 32-column chunks per warp: 4 (BN == 256: the warp owns one whole 128-column sum-of-squares part) or
// 2 (BN == 128: the part is shared by the two warps of a TMEM lane quarter).  In the second case the sums are
// chained in column order -- the first-half warp (`half_idx` 0) parks its per-lane sums in its staging buffer,
// the second-half warp adds its two chunks on top -- so every partial sum is rounded exactly as in the
// one-warp case and a row's result does not depend on the tile width (small-M launches pick the narrow tile).
template <int EK, int NCHW>
__device__ __forceinline__ void epilogue_half_tile_fast(const GemmKParams& p, float* stage, int lane, uint32_t taddr,
                                                        int n_begin, int orow_mine, int arow_mine, float rs_mine,
                                                        uint64_t* tfull_bar, uint32_t parity, int half_idx, int bar_id) {
  constexpr bool RES = ek_resid(EK);
  constexpr bool O16H = ek_half(EK);
  const int c4 = lane & 7;
  const int g4 = lane >> 3;
  int orow[8], arow[8];
  float rs[8];
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    orow[it] = __shfl_sync(0xffffffffu, orow_mine, it * 4 + g4);
    arow[it] = __shfl_sync(0xffffffffu, arow_mine, it * 4 + g4);
    rs[it] = __shfl_sync(0xffffffffu, rs_mine, it * 4 + g4);
  }
  float sqp[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float sqc[NCHW == 2 ? 2 : 1][8] = {};  // second-half warp of a narrow tile: its chunks' sums, added after the first half's
  const float* res = static_cast<const float*>(p.res1);
  float* out = static_cast<float*>(p.out);
  uint16_t* out16 = static_cast<uint16_t*>(p.out16);
  // the residual of the whole half tile is requested up front (register budget: setmaxnreg), so
  // its latency hides behind the main loop of this tile
  uint4 rr4[NCHW][8];
  if (RES) {
#pragma unroll
    for (int c = 0; c < NCHW; ++c)
#pragma unroll
      for (int it = 0; it < 8; ++it)
        if (orow[it] >= 0)
          rr4[c][it] = *reinterpret_cast<const uint4*>(res + (long long)orow[it] * p.ldres + n_begin + c * 32 + c4 * 4);
  }
  mbar_wait(tfull_bar, parity);
  tc_fence_after();
#pragma unroll
  for (int c = 0; c < NCHW; ++c) {
    uint32_t v[32];
    tmem_ld32(taddr + c * 32, v);
    const int n = n_begin + c * 32 + c4 * 4;
    float cm[4] = {1.f, 1.f, 1.f, 1.f};
    if (!RES) load4(p.col_mul, RFB_F32, n, cm);
    tmem_wait_ld();
#pragma unroll
    for (int g = 0; g < 8; ++g)
      *reinterpret_cast<float4*>(stage + lane * 32 + ((g ^ c4) << 2)) =
          make_float4(__uint_as_float(v[g * 4]), __uint_as_float(v[g * 4 + 1]), __uint_as_float(v[g * 4 + 2]),
                      __uint_as_float(v[g * 4 + 3]));
    __syncwarp();
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int rr = it * 4 + g4;
      const float4 a = *reinterpret_cast<const float4*>(stage + rr * 32 + ((c4 ^ (rr & 7)) << 2));
      float x[4] = {a.x * rs[it], a.y * rs[it], a.z * rs[it], a.w * rs[it]};
      if (RES) {
        const uint4& r = rr4[c][it];
        x[0] += __uint_as_float(r.x), x[1] += __uint_as_float(r.y);
        x[2] += __uint_as_float(r.z), x[3] += __uint_as_float(r.w);
      }
      if (orow[it] >= 0) {
        if (RES) {
          const uint4 xo = make_uint4(__float_as_uint(x[0]), __float_as_uint(x[1]), __float_as_uint(x[2]),
                                      __float_as_uint(x[3]));
          *reinterpret_cast<uint4*>(out + (long long)orow[it] * p.ldo + n) = xo;
        }
        if (NCHW == 2 && half_idx == 1) sqc[NCHW == 2 ? c : 0][it] = sq4(x);
        else sqp[it] = __fadd_rn(sqp[it], sq4(x));
        uint2 u;
        u.x = pack16<O16H>(x[0] * cm[0], x[1] * cm[1]), u.y = pack16<O16H>(x[2] * cm[2], x[3] * cm[3]);
        *reinterpret_cast<uint2*>(out16 + (long long)arow[it] * p.ld16 + n) = u;
      }
    }
    __syncwarp();
  }
  if (NCHW == 2) {
    // hand-over of the first half's per-lane sums through the first-half warp's staging buffer (1 KB of it):
    // rendezvous 1 = "sums parked", rendezvous 2 = "sums read" (the buffer is free for the next tile)
    float* xch = (half_idx == 0 ? stage : stage - 4 * 32 * 32) + lane * 8;
    if (half_idx == 0) {
      *reinterpret_cast<float4*>(xch) = make_float4(sqp[0], sqp[1], sqp[2], sqp[3]);
      *reinterpret_cast<float4*>(xch + 4) = make_float4(sqp[4], sqp[5], sqp[6], sqp[7]);
    }
    bar_sync(bar_id, 64);
    if (half_idx == 1) {
      const float4 a = *reinterpret_cast<const float4*>(xch), b = *reinterpret_cast<const float4*>(xch + 4);
      const float first[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
      for (int it = 0; it < 8; ++it)
        if (orow[it] >= 0) sqp[it] = __fadd_rn(__fadd_rn(first[it], sqc[0][it]), sqc[NCHW == 2 ? 1 : 0][it]);
    }
    bar_sync(bar_id, 64);
    if (half_idx == 0) return;  // the second-half warp owns the part's write
  }
  // one 128-column part per warp: reduce the 8 column lanes of every row slot, owner lane writes
  float mine = 0.f;
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    float t = sqp[it];
    t += __shfl_xor_sync(0xffffffffu, t, 1);
    t += __shfl_xor_sync(0xffffffffu, t, 2);
    t += __shfl_xor_sync(0xffffffffu, t, 4);
    t = __shfl_sync(0xffffffffu, t, (lane & 3) * 8);
    if ((lane >> 2) == it) mine = t;
  }
  if (orow_mine >= 0) p.out_sumsq[(long long)arow_mine * p.out_sumsq_ld + (n_begin >> 7)] = mine;
}


template <int BN, int EK>
__global__ void __launch_bounds__(ek_resid(EK) ? kGemmThreadsWG : kGemmThreads, 1)
    gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const GemmKParams p) {
  using Cfg = GemmCfg<BN>;
  constexpr int STAGES = Cfg::kStages;
  constexpr uint32_t B_BYTES = Cfg::kBBytes;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * kABytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(sB + STAGES * B_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* epi_stage = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full) + 256);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr int EPI0 = ek_resid(EK) ? 4 : 2;  // first epilogue warp

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], kEpiWarps);  // one arrive per epilogue warp
    }
    fence_mbar_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int total_tiles = p.num_m_tiles * p.num_n_tiles;

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if constexpr (ek_resid(EK)) setmaxnreg_dec<kRegsGemmWg0>();
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int mt = tile / p.num_n_tiles;
        const int n0 = (tile % p.num_n_tiles) * BN;
        int m0 = mt * kBM, bi = 0, y0 = 0, x0 = 0;
        if (p.a_mode == RFB_A_CONV3X3) {
          const int per_img = p.tiles_x * p.tiles_y;
          bi = mt / per_img;
          const int r = mt % per_img;
          y0 = (r / p.tiles_x) * p.th;
          x0 = (r % p.tiles_x) * p.tw;
        }
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          mbar_expect_tx(&full[stage], kABytes + B_BYTES);
          int kw;  // K coordinate in the weight matrix
          if (p.a_mode == RFB_A_LINEAR) {
            kw = kb * kBK;
            tma_load_2d(sA + stage * kABytes, &tmA, &full[stage], kw, m0);
          } else {
            const int tap = kb / p.kb_per_tap;
            const int cb = kb % p.kb_per_tap;
            kw = tap * p.Cin + cb * kBK;
            tma_load_4d(sA + stage * kABytes, &tmA, &full[stage], cb * kBK, x0 + tap % 3 - 1,
                        y0 + tap / 3 - 1, bi);
          }
          tma_load_2d(sB + stage * B_BYTES, &tmB, &full[stage], kw, n0);
          if (++stage == STAGES) stage = 0, phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer ------------------------------
    if constexpr (ek_resid(EK)) setmaxnreg_dec<kRegsGemmWg0>();
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const int as = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        mbar_wait(&tempty[as], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint64_t ad = umma_desc_sw128(smem_u32(sA + stage * kABytes));
          const uint64_t bd = umma_desc_sw128(smem_u32(sB + stage * B_BYTES));
#pragma unroll
          for (int k = 0; k < kBK / 16; ++k)
            umma_f16(d_tmem, ad + 2 * k, bd + 2 * k, p.idesc, (kb | k) != 0);
          umma_commit(&empty[stage]);  // frees the smem stage once these MMAs retire
          if (++stage == STAGES) stage = 0, phase ^= 1;
        }
        umma_commit(&tfull[as]);  // accumulator complete -> epilogue
      }
    }
  } else if (warp < EPI0) {
    if constexpr (ek_resid(EK)) setmaxnreg_dec<kRegsGemmWg0>();  // idle warps of warpgroup 0
  } else {
    // ------------------------------ epilogue ------------------------------
    if constexpr (ek_resid(EK)) setmaxnreg_inc<kRegsGemmEpi>();
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const int as = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      const int mt = tile / p.num_n_tiles;
      const int n0 = (tile % p.num_n_tiles) * BN;
      long long orow;
      bool valid;
      if (p.a_mode == RFB_A_LINEAR) {
        const int m = mt * kBM + r;
        valid = m < p.M;
        orow = valid ? (p.row_map ? p.row_map[m] : m) : 0;
      } else {
        const int per_img = p.tiles_x * p.tiles_y;
        const int bi = mt / per_img;
        const int rr = mt % per_img;
        const int y = (rr / p.tiles_x) * p.th + r / p.tw;
        const int x = (rr % p.tiles_x) * p.tw + r % p.tw;
        valid = conv_out_row(p, bi, y, x, orow);
      }
      // fused-norm inputs of this thread's row: aux row index and 1/rms factor
      int orow_mine = valid ? static_cast<int>(orow) : -1;
      int arow_mine = orow_mine;
      float rs = 1.0f;
      if (valid) {
        if (p.aux_row_map) arow_mine = p.aux_row_map[orow];
        if (p.in_sumsq) {
          const float* sp = p.in_sumsq + static_cast<long long>(mt * kBM + r) * p.in_sumsq_ld;
          float ss = 0.f;
          if (((p.in_sumsq_parts | p.in_sumsq_ld) & 3) == 0) {
            for (int j = 0; j < p.in_sumsq_parts; j += 4) {
              const float4 t = *reinterpret_cast<const float4*>(sp + j);
              ss += (t.x + t.y) + (t.z + t.w);
            }
          } else {
            for (int j = 0; j < p.in_sumsq_parts; ++j) ss += sp[j];
          }
          rs = rsqrtf(ss * p.inv_norm_dim + p.norm_eps);
          if (p.out_rscale && n0 == 0 && warp < EPI0 + 4) p.out_rscale[mt * kBM + r] = rs;
        } else if (p.in_rscale && p.scale_dim == 0) {
          rs = p.in_rscale[mt * kBM + r];
        }
      }
      float* my_stage = epi_stage + (warp - EPI0) * 32 * 32;
      // the two warps of a TMEM lane quarter take the two contiguous halves of the tile's columns
      constexpr int NCH = BN / 32;
      constexpr int HALF = (NCH + 1) / 2;
      const int c_begin = ((warp - EPI0) >> 2) * HALF;
      const int c_end = (c_begin + HALF < NCH) ? c_begin + HALF : NCH;
      if (p.vt_out && n0 >= p.vt_split) {  // tile of the transposed (V) part: warp-uniform per tile
        epilogue_vt_chunks(p, tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN, n0, c_begin, c_end,
                           mt * kBM + r, valid, rs, &tfull[as], aph);
      } else if constexpr (ek_fast(EK)) {
        static_assert(BN == 256 || BN == 128, "specialised epilogues use the 256- or 128-wide tile");
        epilogue_half_tile_fast<EK, BN / 64>(p, my_stage, lane,
                                             tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN + c_begin * 32,
                                             n0 + c_begin * 32, orow_mine, arow_mine, rs, &tfull[as], aph,
                                             (warp - EPI0) >> 2, 1 + q);
      } else {
        const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN;
        if ((p.epi == RFB_EPI_STORE) && !p.direct_store) {
          epilogue_generic_coalesced<EK>(p, my_stage, lane, taddr0, n0, c_begin, c_end, orow_mine, arow_mine, rs,
                                     &tfull[as], aph);
        } else {
          mbar_wait(&tfull[as], aph);
          tc_fence_after();
#pragma unroll 1
          for (int c = c_begin; c < c_end; ++c) {
            if (n0 + c * 32 >= p.n_store) break;  // warp-uniform
            uint32_t v[32];
            tmem_ld32(taddr0 + c * 32, v);
            tmem_wait_ld();
            if (valid) epilogue_chunk(p, orow, n0 + c * 32, v, rs);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int BN, int EK = EK_GENERIC>
static int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmKParams& p,
                       int grid, cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  static PerDeviceFlag attr_flags;
  bool& attr_set = attr_flags.get();
  if (!attr_set) {
    if (cudaFuncSetAttribute(gemm_tc_kernel<BN, EK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             Cfg::kSmemBytes) != cudaSuccess)
      return RFB_ERR_LAUNCH;
    if (ek_resid(EK)) {  // setmaxnreg only moves registers inside the CTA's launch allocation
      cudaFuncAttributes fa;
      if (cudaFuncGetAttributes(&fa, gemm_tc_kernel<BN, EK>) != cudaSuccess) return RFB_ERR_LAUNCH;
      if (128 * kRegsGemmWg0 + 256 * kRegsGemmEpi > kGemmThreadsWG * fa.numRegs) {
        fprintf(stderr, "rfb: gemm_tc_kernel<RESID> compiled with %d registers/thread; setmaxnreg split does not fit\n",
                fa.numRegs);
        return RFB_ERR_LAUNCH;
      }
    }
    attr_set = true;
  }
  constexpr int threads = ek_resid(EK) ? kGemmThreadsWG : kGemmThreads;
  gemm_tc_kernel<BN, EK><<<grid, threads, Cfg::kSmemBytes, stream>>>(tmA, tmB, p);
  g_launch_count++;
  return check_launch("gemm_tc_kernel");
}

// =============================================================================================
// 3x3 convolution with a shared-memory halo tile.
//
// The implicit-GEMM conv above re-loads the activation tile once per filter tap (9x) and the weights
// once per 128-pixel tile; both come from L2 and the kernel ends up bound by L2->SM bandwidth.  Here a
// CTA works on a 16 x 16 pixel super-tile = two 8-wide x 16-tall UMMA tiles: per 64-channel block ONE
// 4-D TMA box brings the 18 x 18 pixel halo region into shared memory (pixel = 128-byte row, 128B
// swizzle), and the nine tap-shifted A operands of both tiles are read straight out of it by offsetting
// the UMMA descriptor: start = halo + ((dy*18 + dx + 8*tile) * 128) B, 8-row-group stride = 18 * 128 B.
// (The swizzle is a function of the shared-memory address, so any 128-byte-aligned start and any group
// stride work -- checked by selftest_halo.)  A weight stage [BN x 64] is used for both tiles, so per
// 256 output pixels and channel block 41.5 KB + 9 * BN * 128 B travel instead of 2 * 9 * (16 KB + BN*128 B).
// Accumulators: 2 tiles x 2 buffers x BN TMEM columns.  Epilogues are the GEMM's.
// =============================================================================================
constexpr int kHaloPitch = 18;                                   // pixels per halo row
constexpr uint32_t kHaloBytes = kHaloPitch * kHaloPitch * 128;   // 41472
constexpr uint32_t kHaloStride = 42 * 1024;                      // 1024-aligned slot per halo buffer

template <int BN>
struct HaloCfg {
  static constexpr uint32_t kBBytes = BN * kBK * 2;
  static constexpr int kStages = (BN == 128) ? 6 : 8;
  static constexpr uint32_t kTmemCols = (4 * BN < 32) ? 32 : 4 * BN;
  static constexpr uint32_t kSmemBytes = 2 * kHaloStride + kStages * kBBytes + 1024 + 256 + kEpiStageBytes;
};

template <int BN, int EK>
__global__ void __launch_bounds__(kGemmThreads, 1)
    conv_halo_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                     const GemmKParams p) {
  using Cfg = HaloCfg<BN>;
  constexpr int STAGES = Cfg::kStages;
  constexpr uint32_t B_BYTES = Cfg::kBBytes;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* sH = smem;                      // 2 halo buffers
  uint8_t* sB = smem + 2 * kHaloStride;    // weight stages
  uint64_t* bfull = reinterpret_cast<uint64_t*>(sB + STAGES * B_BYTES);
  uint64_t* bempty = bfull + STAGES;
  uint64_t* hfull = bempty + STAGES;
  uint64_t* hempty = hfull + 2;
  uint64_t* tfull = hempty + 2;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* epi_stage = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bfull) + 256);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) mbar_init(&bfull[i], 1), mbar_init(&bempty[i], 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&hfull[i], 1), mbar_init(&hempty[i], 1);
      mbar_init(&tfull[i], 1), mbar_init(&tempty[i], kEpiWarps);
    }
    fence_mbar_init();
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int per_img = p.tiles_x * p.tiles_y;
  const int total = p.num_m_tiles;  // super-tiles
  const int ncb = p.kb_per_tap;     // 64-channel blocks

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0, hb = 0;
      uint32_t phase = 0, hphase = 0;
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int bi = tile / per_img, rr = tile % per_img;
        const int y0 = (rr / p.tiles_x) * 16, x0 = (rr % p.tiles_x) * 16;
        for (int cb = 0; cb < ncb; ++cb) {
          mbar_wait(&hempty[hb], hphase ^ 1);
          mbar_expect_tx(&hfull[hb], kHaloBytes);
          tma_load_4d(sH + hb * kHaloStride, &tmA, &hfull[hb], cb * kBK, x0 - 1, y0 - 1, bi);
          if (++hb == 2) hb = 0, hphase ^= 1;
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(&bempty[stage], phase ^ 1);
            mbar_expect_tx(&bfull[stage], B_BYTES);
            tma_load_2d(sB + stage * B_BYTES, &tmB, &bfull[stage], tap * p.Cin + cb * kBK, 0);
            if (++stage == STAGES) stage = 0, phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int stage = 0, hb = 0, it = 0;
      uint32_t phase = 0, hphase = 0;
      for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++it) {
        const int as = it & 1;
        mbar_wait(&tempty[as], ((it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d0 = tmem_base + as * 2 * BN;
        for (int cb = 0; cb < ncb; ++cb) {
          mbar_wait(&hfull[hb], hphase);
          tc_fence_after();
          const uint32_t halo = smem_u32(sH + hb * kHaloStride);
          for (int tap = 0; tap < 9; ++tap) {
            mbar_wait(&bfull[stage], phase);
            tc_fence_after();
            const uint64_t bd = umma_desc_sw128(smem_u32(sB + stage * B_BYTES));
            const uint32_t a0 = halo + ((tap / 3) * kHaloPitch + tap % 3) * 128;
#pragma unroll
            for (int t = 0; t < 2; ++t) {
              // 8-row group g = image row y of the tile: stride = one halo row
              uint64_t ad = static_cast<uint64_t>(((a0 + t * 8 * 128) >> 4) & 0x3fff);
              ad |= static_cast<uint64_t>((kHaloPitch * 128) >> 4) << 32;
              ad |= static_cast<uint64_t>(1) << 46;
              ad |= static_cast<uint64_t>(2) << 61;
#pragma unroll
              for (int k = 0; k < kBK / 16; ++k)
                umma_f16(d0 + t * BN, ad + 2 * k, bd + 2 * k, p.idesc, (cb | tap | k) != 0);
            }
            umma_commit(&bempty[stage]);
            if (++stage == STAGES) stage = 0, phase ^= 1;
          }
          umma_commit(&hempty[hb]);
          if (++hb == 2) hb = 0, hphase ^= 1;
        }
        umma_commit(&tfull[as]);
      }
    }
  } else {
    // ------------------------------ epilogue (same code as the GEMM) ------------------------------
    const int q = warp & 3;
    const int r = q * 32 + lane;
    int it = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++it) {
      const int as = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      const int bi = tile / per_img, rr = tile % per_img;
      const int y = (rr / p.tiles_x) * 16 + (r >> 3);
      float* my_stage = epi_stage + (warp - 2) * 32 * 32;
      constexpr int NCH = BN / 32;
      constexpr int HALF = (NCH + 1) / 2;
      const int c_begin = ((warp - 2) >> 2) * HALF;
      const int c_end = (c_begin + HALF < NCH) ? c_begin + HALF : NCH;
#pragma unroll 1
      for (int t = 0; t < 2; ++t) {
        const int x = (rr % p.tiles_x) * 16 + t * 8 + (r & 7);
        long long orow;
        const bool valid = conv_out_row(p, bi, y, x, orow);
        const int orow_mine = valid ? static_cast<int>(orow) : -1;
        const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * 2 * BN + t * BN;
        if (p.epi == RFB_EPI_STORE) {
          epilogue_generic_coalesced<EK>(p, my_stage, lane, taddr0, 0, c_begin, c_end, orow_mine, orow_mine, 1.0f,
                                         &tfull[as], aph);
        } else {
          mbar_wait(&tfull[as], aph);
          tc_fence_after();
#pragma unroll 1
          for (int c = c_begin; c < c_end; ++c) {
            if (c * 32 >= p.n_store) break;
            uint32_t v[32];
            tmem_ld32(taddr0 + c * 32, v);
            tmem_wait_ld();
            if (valid) epilogue_chunk(p, orow, c * 32, v, 1.0f);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[as]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int BN, int EK = EK_GENERIC>
static int launch_conv_halo(const CUtensorMap& tmA, const CUtensorMap& tmB, const GemmKParams& p, int grid,
                            cudaStream_t stream) {
  using Cfg = HaloCfg<BN>;
  static PerDeviceFlag attr_flags;
  bool& attr_set = attr_flags.get();
  if (!attr_set) {
    if (cudaFuncSetAttribute(conv_halo_kernel<BN, EK>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             Cfg::kSmemBytes) != cudaSuccess)
      return RFB_ERR_LAUNCH;
    attr_set = true;
  }
  conv_halo_kernel<BN, EK><<<grid, kGemmThreads, Cfg::kSmemBytes, stream>>>(tmA, tmB, p);
  g_launch_count++;
  return check_launch("conv_halo_kernel");
}

}  // namespace rfb

using namespace rfb;

extern "C" int rfb_gemm(const rfb_gemm_args* a, rfb_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  if (!a || !a->A || !a->W || a->M <= 0 || a->N <= 0 || a->K <= 0) return RFB_ERR_ARG;
  if (a->dtype != RFB_BF16 && a->dtype != RFB_F16) return RFB_ERR_ARG;

  GemmKParams p{};
  p.M = a->M, p.N = a->N, p.K = a->K;
  p.a_mode = a->a_mode;
  p.epi = a->epi;
  p.bias = a->bias, p.res1 = a->res1, p.res2 = a->res2, p.res_dtype = a->res_dtype;
  p.ldres = a->ldres, p.out = a->out, p.out_dtype = a->out_dtype, p.ldo = a->ldo;
  p.out_act = a->out_act, p.row_map = a->row_map, p.w2 = a->w2, p.b2 = a->b2;

  p.in_sumsq = a->in_sumsq, p.in_sumsq_ld = a->in_sumsq_ld > 0 ? a->in_sumsq_ld : 1;
  p.in_sumsq_parts = a->in_sumsq_parts > 0 ? a->in_sumsq_parts : 1;
  p.in_rscale = a->in_rscale, p.scale_dim = a->scale_dim, p.out_rscale = a->out_rscale;
  p.inv_norm_dim = a->norm_dim > 0 ? 1.0f / (float)a->norm_dim : 0.f;
  p.norm_eps = a->norm_eps;
  p.out_sumsq = a->out_sumsq, p.out_sumsq_ld = a->out_sumsq_ld;
  p.out16 = a->out16, p.out16_dtype = a->out16_dtype, p.ld16 = a->ld16;
  p.col_mul = a->col_mul, p.aux_row_map = a->aux_row_map;
  p.vt_out = a->vt_out, p.vt_dtype = a->vt_dtype, p.vt_split = a->vt_split;
  p.vt_rows_per_batch = a->vt_rows_per_batch, p.vt_ld = a->vt_ld, p.vt_batch_stride = a->vt_batch_stride;
  if (a->vt_out) {
    if (a->a_mode != RFB_A_LINEAR || a->epi != RFB_EPI_STORE || a->row_map || a->vt_split <= 0 || a->vt_split >= a->N ||
        a->vt_split % 256 || (a->vt_dtype != RFB_BF16 && a->vt_dtype != RFB_F16) || a->vt_ld < 1 ||
        (a->in_rscale && a->scale_dim == 1))
      return RFB_ERR_ARG;
  }
  const bool fused_any = a->in_sumsq || a->in_rscale || a->out_rscale || a->out_sumsq || a->out16 || a->col_mul;
  if (a->in_sumsq && (a->norm_dim <= 0 || a->in_rscale || p.in_sumsq_parts > p.in_sumsq_ld)) return RFB_ERR_ARG;
  if (a->in_rscale && a->scale_dim != 0 && a->scale_dim != 1) return RFB_ERR_ARG;
  if (a->out_rscale && !a->in_sumsq) return RFB_ERR_ARG;
  const bool epi_final = a->epi == RFB_EPI_FINAL || a->epi == RFB_EPI_FINAL_RAW;
  if (fused_any && epi_final) return RFB_ERR_ARG;
  if (a->crop_h || a->crop_w || a->crop_top || a->crop_left) {  // the window must lie inside the conv image
    if (a->a_mode != RFB_A_CONV3X3 || !epi_final || a->crop_h <= 0 || a->crop_w <= 0 || a->crop_top < 0 ||
        a->crop_left < 0 || a->crop_h > a->H - a->crop_top || a->crop_w > a->Wd - a->crop_left)
      return RFB_ERR_ARG;
    p.crop_h = a->crop_h, p.crop_w = a->crop_w, p.crop_top = a->crop_top, p.crop_left = a->crop_left;
  }
  if (a->epi == RFB_EPI_SWIGLU && (a->out_rscale || a->out_sumsq || a->out16 || a->col_mul ||
                                   (a->in_rscale && a->scale_dim != 0)))
    return RFB_ERR_ARG;
  if (a->out16 && (a->ld16 % 8 || (a->out16_dtype != RFB_BF16 && a->out16_dtype != RFB_F16))) return RFB_ERR_ARG;
  if (a->out16 && a->N % 8) return RFB_ERR_ARG;
  const int n_plain = a->vt_out ? a->vt_split : a->N;  // columns that go through the ordinary epilogue
  if (a->out_sumsq && (n_plain % 128 || a->out_sumsq_ld < n_plain / 128)) return RFB_ERR_ARG;
  if (a->res2 && (a->res_dtype == RFB_F32 || !a->res1)) return RFB_ERR_ARG;

  // the compile-time residual-stream epilogue (EK_RESID: fp32 out = acc*r + fp32 residual, 16-bit copy, sums of
  // squares) exists for 256- and 128-wide tiles; every other user of out_sumsq needs the 256-wide one
  const bool resid_kind = a->epi == RFB_EPI_STORE && a->a_mode == RFB_A_LINEAR && a->N % 256 == 0 && a->out16 &&
                          a->out_sumsq && !a->bias && !a->res2 && !a->out_act && !a->vt_out && !a->col_mul &&
                          !(a->in_rscale && a->scale_dim == 1) && a->out && a->out_dtype == RFB_F32 && a->res1 &&
                          a->res_dtype == RFB_F32;
  const int sms = num_sms();
  const long long m_tiles_lin = (a->M + kBM - 1) / kBM;
  int bn = a->bn_override;
  if (a->vt_out) {
    if (bn != 0 && bn != 256) return RFB_ERR_ARG;
    bn = 256;  // vt_split is a whole number of 256-wide tiles
  }
  if (a->out_sumsq) {
    if (bn != 0 && bn != 256 && !(bn == 128 && resid_kind)) return RFB_ERR_ARG;
    // one epilogue warp per 128-column sum-of-squares part; a launch that cannot fill half of the SMs with
    // 256-wide tiles (the row-sharded scene stage: a few hundred rows per rank) takes the 128-wide variant,
    // whose two warps per part chain their sums in column order -- bit-identical results
    if (bn == 0) bn = (resid_kind && m_tiles_lin * (a->N / 256) * 2 <= sms) ? 128 : 256;
  }
  if (bn == 0) {
    if (a->N <= 32) bn = 32;
    else if (a->N <= 64) bn = 64;
    else if (a->N % 256 == 0) bn = 256;
    else if (a->a_mode == RFB_A_LINEAR && a->N > 1024 && ((a->N + 255) / 256) * 256 * 100 <= a->N * 110)
      bn = 256;  // ragged N: the 256-wide UMMA is ~35 % faster per FLOP, worth <= 10 % padded columns
    else bn = 128;
    // Small grids (few rows): a narrower tile puts more SMs to work.  cost = rounds of the persistent grid x
    // (tile width + a fixed per-tile share for the pipeline fill and the slower narrow UMMA); the accumulation
    // order along K does not depend on the tile width, so the result is bit-identical whichever is picked.
    if (bn == 256 && a->a_mode == RFB_A_LINEAR && (a->epi == RFB_EPI_STORE || a->epi == RFB_EPI_SWIGLU)) {
      long long best = -1;
      for (int cand = 256; cand >= 64; cand >>= 1) {
        const long long tiles = m_tiles_lin * (a->N / cand);
        const long long cost = ((tiles + sms - 1) / sms) * (cand + 64);
        if (best < 0 || cost < best) best = cost, bn = cand;
      }
    }
  }
  if (bn != 32 && bn != 64 && bn != 128 && bn != 256) return RFB_ERR_ARG;

  if (a->epi == RFB_EPI_STORE) {
    p.n_store = (n_plain + 7) & ~7;
    if (p.n_store > a->ldo) return RFB_ERR_ARG;
    if ((a->bias || a->res1 || a->res2) && (a->N % 8) != 0) return RFB_ERR_ARG;
    if (!a->out && !a->out_act && !a->out16) return RFB_ERR_ARG;
    const int align = (a->out_dtype == RFB_F32) ? 4 : 8;
    if (a->ldo % align) return RFB_ERR_ALIGN;
    if ((a->res1 || a->res2) && a->ldres % ((a->res_dtype == RFB_F32) ? 4 : 8)) return RFB_ERR_ALIGN;
  } else if (a->epi == RFB_EPI_SWIGLU) {
    if (a->N % 32 || !a->out || a->out_dtype == RFB_F32 || a->ldo % 8) return RFB_ERR_ARG;
    p.n_store = a->N;
  } else if (epi_final) {
    if (a->N != 32 || !a->out || !a->bias || !a->w2 || !a->b2) return RFB_ERR_ARG;
    bn = 32;
    p.n_store = 32;
  } else {
    return RFB_ERR_ARG;
  }

  CUtensorMap tmA, tmB;
  int rc;
  if (a->a_mode == RFB_A_LINEAR) {
    uint64_t dims[2] = {(uint64_t)a->K, (uint64_t)a->M};
    uint64_t strides[1] = {(uint64_t)a->lda * 2};
    uint32_t box[2] = {(uint32_t)kBK, (uint32_t)kBM};
    if ((rc = make_tmap_16b(&tmA, a->dtype, a->A, 2, dims, strides, box)) != RFB_OK) return rc;
    p.num_m_tiles = (a->M + kBM - 1) / kBM;
    p.num_kb = (a->K + kBK - 1) / kBK;
  } else if (a->a_mode == RFB_A_CONV3X3) {
    if (a->B <= 0 || a->H <= 0 || a->Wd <= 0 || a->Cin <= 0 || a->K != 9 * a->Cin ||
        a->M != a->B * a->H * a->Wd || a->row_map)
      return RFB_ERR_ARG;
    {
      // halo-tile kernel: whole 64-channel blocks, one N tile, enough 16 x 16 super-tiles to fill the GPU
      static int halo_on = -1;
      if (halo_on < 0) {
        const char* e = getenv("RFB_CONV_HALO");
        halo_on = (e && e[0] == '0') ? 0 : 1;
      }
      const int stx = (a->Wd + 15) / 16, sty = (a->H + 15) / 16;
      const long long n_super = (long long)a->B * stx * sty;
      if (halo_on && a->Cin % 64 == 0 && a->N == bn && (bn == 128 || bn == 64 || bn == 32) && n_super >= 96 &&
          !fused_any && !a->vt_out && !p.direct_store) {
        p.H = a->H, p.Wd = a->Wd, p.Cin = a->Cin;
        p.tw = 8, p.th = 16, p.tiles_x = stx, p.tiles_y = sty, p.kb_per_tap = a->Cin / kBK;
        p.num_m_tiles = (int)n_super, p.num_n_tiles = 1, p.num_kb = 9 * p.kb_per_tap;
        uint64_t dims[4] = {(uint64_t)a->Cin, (uint64_t)a->Wd, (uint64_t)a->H, (uint64_t)a->B};
        uint64_t strides[3] = {(uint64_t)a->Cin * 2, (uint64_t)a->Wd * a->Cin * 2, (uint64_t)a->H * a->Wd * a->Cin * 2};
        uint32_t box[4] = {(uint32_t)kBK, (uint32_t)kHaloPitch, (uint32_t)kHaloPitch, 1};
        if ((rc = make_tmap_16b(&tmA, a->dtype, a->A, 4, dims, strides, box)) != RFB_OK) return rc;
        uint64_t wd[2] = {(uint64_t)a->K, (uint64_t)a->N};
        uint64_t ws[1] = {(uint64_t)a->ldw * 2};
        uint32_t wb[2] = {(uint32_t)kBK, (uint32_t)bn};
        if ((rc = make_tmap_16b(&tmB, a->dtype, a->W, 2, wd, ws, wb)) != RFB_OK) return rc;
        p.idesc = umma_idesc_f16(a->dtype == RFB_BF16 ? 1u : 0u, kBM, bn);
        const int cap = a->max_ctas > 0 ? a->max_ctas : num_sms();
        const int grid = (int)(n_super < cap ? n_super : cap);
        if (bn == 64) return launch_conv_halo<64>(tmA, tmB, p, grid, stream);
        if (bn == 32) return launch_conv_halo<32>(tmA, tmB, p, grid, stream);
        if (a->epi == RFB_EPI_STORE && a->dtype == RFB_F16 && a->out_dtype == RFB_F16 &&
            (!a->res1 || a->res_dtype == RFB_F16)) {
          const int cm = (a->out ? CF_OUT : 0) | (a->out_act ? CF_ACT : 0) | (a->bias ? CF_BIAS : 0) |
                         (a->res1 ? CF_RES1 : 0) | (a->res2 ? CF_RES2 : 0);
          switch (cm) {
            case CF_OUT | CF_ACT: return launch_conv_halo<128, EK_CONV + (CF_OUT | CF_ACT)>(tmA, tmB, p, grid, stream);
            case CF_ACT | CF_BIAS: return launch_conv_halo<128, EK_CONV + (CF_ACT | CF_BIAS)>(tmA, tmB, p, grid, stream);
            case CF_OUT | CF_BIAS | CF_RES1:
              return launch_conv_halo<128, EK_CONV + (CF_OUT | CF_BIAS | CF_RES1)>(tmA, tmB, p, grid, stream);
            case CF_OUT | CF_ACT | CF_BIAS | CF_RES1:
              return launch_conv_halo<128, EK_CONV + (CF_OUT | CF_ACT | CF_BIAS | CF_RES1)>(tmA, tmB, p, grid, stream);
            case CF_OUT | CF_BIAS | CF_RES1 | CF_RES2:
              return launch_conv_halo<128, EK_CONV + (CF_OUT | CF_BIAS | CF_RES1 | CF_RES2)>(tmA, tmB, p, grid, stream);
            case CF_OUT | CF_ACT | CF_BIAS | CF_RES1 | CF_RES2:
              return launch_conv_halo<128, EK_CONV + (CF_OUT | CF_ACT | CF_BIAS | CF_RES1 | CF_RES2)>(tmA, tmB, p, grid,
                                                                                                   stream);
            default: break;
          }
        }
        return launch_conv_halo<128>(tmA, tmB, p, grid, stream);
      }
    }
    p.H = a->H, p.Wd = a->Wd, p.Cin = a->Cin;
    p.tw = (a->Wd >= 16) ? 16 : 8;
    p.th = kBM / p.tw;
    p.tiles_x = (a->Wd + p.tw - 1) / p.tw;
    p.tiles_y = (a->H + p.th - 1) / p.th;
    p.kb_per_tap = (a->Cin + kBK - 1) / kBK;
    uint64_t dims[4] = {(uint64_t)a->Cin, (uint64_t)a->Wd, (uint64_t)a->H, (uint64_t)a->B};
    uint64_t strides[3] = {(uint64_t)a->Cin * 2, (uint64_t)a->Wd * a->Cin * 2,
                           (uint64_t)a->H * a->Wd * a->Cin * 2};
    uint32_t box[4] = {(uint32_t)kBK, (uint32_t)p.tw, (uint32_t)p.th, 1};
    if ((rc = make_tmap_16b(&tmA, a->dtype, a->A, 4, dims, strides, box)) != RFB_OK) return rc;
    p.num_m_tiles = a->B * p.tiles_x * p.tiles_y;
    p.num_kb = 9 * p.kb_per_tap;
  } else {
    return RFB_ERR_ARG;
  }
  {
    uint64_t dims[2] = {(uint64_t)a->K, (uint64_t)a->N};
    uint64_t strides[1] = {(uint64_t)a->ldw * 2};
    uint32_t box[2] = {(uint32_t)kBK, (uint32_t)bn};
    if ((rc = make_tmap_16b(&tmB, a->dtype, a->W, 2, dims, strides, box)) != RFB_OK) return rc;
  }
  p.num_n_tiles = (a->N + bn - 1) / bn;
  p.idesc = umma_idesc_f16(a->dtype == RFB_BF16 ? 1u : 0u, kBM, bn);

  {
    static int direct = -1;
    if (direct < 0) {
      const char* e = getenv("RFB_EPI_DIRECT");
      direct = (e && e[0] == '1') ? 1 : 0;
    }
    p.direct_store = direct;
  }
  if (p.direct_store && fused_any) p.direct_store = 0;
  const long long total = (long long)p.num_m_tiles * p.num_n_tiles;
  int cap = a->max_ctas > 0 ? a->max_ctas : num_sms();
  int grid = (int)(total < cap ? total : cap);

  if (bn == 128 && a->out_sumsq) {  // narrow residual-stream tile (resid_kind checked above)
    if (p.direct_store) return RFB_ERR_ARG;
    return a->out16_dtype == RFB_F16 ? launch_gemm<128, EK_RESID_H>(tmA, tmB, p, grid, stream)
                                     : launch_gemm<128, EK_RESID>(tmA, tmB, p, grid, stream);
  }
  if (bn == 256 && a->N % 256 == 0 && a->epi == RFB_EPI_STORE && !p.direct_store && a->out16 &&
      a->out_sumsq && !a->bias && !a->res2 && !a->out_act && !(a->in_rscale && a->scale_dim == 1)) {
    const bool half = a->out16_dtype == RFB_F16;
    if (a->out && a->out_dtype == RFB_F32 && a->res1 && a->res_dtype == RFB_F32 && !a->col_mul)
      return half ? launch_gemm<256, EK_RESID_H>(tmA, tmB, p, grid, stream)
                  : launch_gemm<256, EK_RESID>(tmA, tmB, p, grid, stream);
    if (!a->out && !a->res1 && a->col_mul)
      return half ? launch_gemm<256, EK_PROJ16_H>(tmA, tmB, p, grid, stream)
                  : launch_gemm<256, EK_PROJ16>(tmA, tmB, p, grid, stream);
  }
  if (bn == 128 && a->a_mode == RFB_A_CONV3X3 && a->epi == RFB_EPI_STORE && !p.direct_store && !fused_any && !a->vt_out &&
      a->dtype == RFB_F16 && a->out_dtype == RFB_F16 && (!a->res1 || a->res_dtype == RFB_F16) && a->N % 128 == 0) {
    const int cm = (a->out ? CF_OUT : 0) | (a->out_act ? CF_ACT : 0) | (a->bias ? CF_BIAS : 0) | (a->res1 ? CF_RES1 : 0) |
                   (a->res2 ? CF_RES2 : 0);
    switch (cm) {  // the flag sets the DPT head uses (layers/dpt.py:57-92,133-159,195-240)
      case CF_OUT | CF_ACT: return launch_gemm<128, EK_CONV + (CF_OUT | CF_ACT)>(tmA, tmB, p, grid, stream);
      case CF_ACT | CF_BIAS: return launch_gemm<128, EK_CONV + (CF_ACT | CF_BIAS)>(tmA, tmB, p, grid, stream);
      case CF_OUT | CF_BIAS | CF_RES1:
        return launch_gemm<128, EK_CONV + (CF_OUT | CF_BIAS | CF_RES1)>(tmA, tmB, p, grid, stream);
      case CF_OUT | CF_ACT | CF_BIAS | CF_RES1:
        return launch_gemm<128, EK_CONV + (CF_OUT | CF_ACT | CF_BIAS | CF_RES1)>(tmA, tmB, p, grid, stream);
      case CF_OUT | CF_BIAS | CF_RES1 | CF_RES2:
        return launch_gemm<128, EK_CONV + (CF_OUT | CF_BIAS | CF_RES1 | CF_RES2)>(tmA, tmB, p, grid, stream);
      case CF_OUT | CF_ACT | CF_BIAS | CF_RES1 | CF_RES2:
        return launch_gemm<128, EK_CONV + (CF_OUT | CF_ACT | CF_BIAS | CF_RES1 | CF_RES2)>(tmA, tmB, p, grid, stream);
      default: break;
    }
  }
  switch (bn) {
    case 32: return launch_gemm<32>(tmA, tmB, p, grid, stream);
    case 64: return launch_gemm<64>(tmA, tmB, p, grid, stream);
    case 128: return launch_gemm<128>(tmA, tmB, p, grid, stream);
    default: return launch_gemm<256>(tmA, tmB, p, grid, stream);
  }
}

extern "C" int rfb_version(void) { return 102; }
extern "C" long long rfb_launch_count(void) { return g_launch_count.load(); }
