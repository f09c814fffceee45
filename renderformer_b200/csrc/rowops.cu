// Bandwidth-bound row kernels around the tensor-core GEMMs: RMSNorm, QK-RMSNorm + 3-D vertex
// RoPE, token assembly, input preparation (texture / vertex-normal / ray-bundle tokens),
// camera-space triangle positions, key-mask packing, fp32 -> 16-bit casts.
// One warp per row, 128-bit coalesced accesses, fp32 math.
#include <atomic>

#include "host_util.h"
#include "ptx.cuh"

namespace rfb {

extern std::atomic<long long> g_launch_count;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void store4_16(void* base, int dtype, long long idx, float a, float b,
                                          float c, float d) {
  uint2 u;
  if (dtype == RFB_BF16) {
    u.x = pack_bf16(a, b), u.y = pack_bf16(c, d);
  } else {
    u.x = pack_f16(a, b), u.y = pack_f16(c, d);
  }
  *reinterpret_cast<uint2*>(static_cast<uint16_t*>(base) + idx) = u;
}

constexpr int kMaxVec = 16;  // d <= 16 * 128 = 2048

// ---------------------------------------------------------------------------------------------
// out[r, :] = rmsnorm(x[src(r), :]) * w      (nn.RMSNorm, layers/attention.py:436-482,503-526)
// ---------------------------------------------------------------------------------------------
__global__ void rmsnorm_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ w,
                               void* __restrict__ out, int out_dtype, long long ldo, int rows, int d,
                               float eps, const int* __restrict__ gather) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const long long src = gather ? gather[row] : row;
  const float4* xr = reinterpret_cast<const float4*>(x + src * ldx);
  const int nvec = d >> 7;  // float4 per lane
  float4 v[kMaxVec];
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxVec; ++j)
    if (j < nvec) {
      v[j] = xr[j * 32 + lane];
      ss += v[j].x * v[j].x + v[j].y * v[j].y + v[j].z * v[j].z + v[j].w * v[j].w;
    }
  ss = warp_sum(ss);
  const float r = rsqrtf(ss / d + eps);
  const float4* wr = reinterpret_cast<const float4*>(w);
#pragma unroll
  for (int j = 0; j < kMaxVec; ++j)
    if (j < nvec) {
      const float4 g = __ldg(wr + j * 32 + lane);
      const long long idx = (long long)row * ldo + (j * 32 + lane) * 4;
      if (out_dtype == RFB_F32)
        *reinterpret_cast<float4*>(static_cast<float*>(out) + idx) =
            make_float4(v[j].x * r * g.x, v[j].y * r * g.y, v[j].z * r * g.z, v[j].w * r * g.w);
      else
        store4_16(out, out_dtype, idx, v[j].x * r * g.x, v[j].y * r * g.y, v[j].z * r * g.z,
                  v[j].w * r * g.w);
    }
}

// ---------------------------------------------------------------------------------------------
// Row statistics for the fused-norm GEMMs: out16[r,:] = cast(x[r,:]), sumsq[r] = sum(x[r,:]^2).
// (Seeds the (16-bit copy, sum of squares) pair that the residual GEMM epilogues then maintain.)
// ---------------------------------------------------------------------------------------------
__global__ void rowstat_kernel(const float* __restrict__ x, void* __restrict__ out16, int out_dtype, long long ld16,
                               float* __restrict__ sumsq, int sumsq_ld, int parts, int rows, int d,
                               const int* __restrict__ gather) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float4* xr = reinterpret_cast<const float4*>(x + (long long)(gather ? gather[row] : row) * d);
  const int nvec = d >> 7;
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxVec; ++j)
    if (j < nvec) {
      const float4 v = xr[j * 32 + lane];
      ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
      store4_16(out16, out_dtype, (long long)row * ld16 + (j * 32 + lane) * 4, v.x, v.y, v.z, v.w);
    }
  ss = warp_sum(ss);
  if (lane < parts) sumsq[(long long)row * sumsq_ld + lane] = lane == 0 ? ss : 0.f;
}

// ---------------------------------------------------------------------------------------------
// QK-RMSNorm over the full width (all heads) + triangle RoPE, fp32 in -> bf16 out.
//   layers/attention.py:128-141, encodings/rope.py:78-149,152-206.
// A row holds `nseg` segments of width d (e.g. [q | k]), each normalised with its own weight.
// RoPE pairs are (i, i+64) inside every 128-wide head; pair i < 9*nfreq rotates by
// pos[i / nfreq] * freq[i % nfreq], the remaining pairs are the identity.
// Input row = r % in_period (lets V views re-rotate one shared pre-RoPE K), position row = r.
// ---------------------------------------------------------------------------------------------
// sin/cos with an explicit two-constant reduction to [-pi, pi] followed by the SFU approximations
// (abs. error ~1e-6 for the |angle| < 100 rad seen here; the result is rounded to bf16 anyway).
// Keeps the kernels free of the slow-path code of sincosf and its register footprint.
__device__ __forceinline__ void fast_sincos(float x, float& s, float& c) {
  const float k = rintf(x * 0.15915494309189535f);
  float r = fmaf(k, -6.28318548202514648f, x);
  r = fmaf(k, 1.74845553146951715e-7f, r);
  __sincosf(r, &s, &c);
}

// cos / sin of the four rotation pairs [o, o+4) a lane owns inside every head (pair i < 9*nfreq rotates by
// pos[i / nfreq] * freq[i % nfreq], the rest are the identity); `prow` = the row's 9 position floats or NULL
__device__ __forceinline__ void rope_lane_cs(const float* __restrict__ prow, const float* __restrict__ freqs, int nfreq,
                                             const float* __restrict__ ctab, const float* __restrict__ stab, int o,
                                             float (&cs)[4], float (&sn)[4]) {
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    cs[e] = 1.f, sn[e] = 0.f;
    const int i = o + e;
    if (ctab) {  // ready-made cos / sin tables (pair i rotates by entry i; entries 64.. duplicate 0..63)
      cs[e] = ctab[i], sn[e] = stab[i];
    } else if (prow && i < 9 * nfreq) {
      const float ang = prow[i / nfreq] * __ldg(freqs + i % nfreq);
      fast_sincos(ang, sn[e], cs[e]);
    }
  }
}

// One (row, segment) per warp: RMSNorm over the segment's d values (weight ws; NULL = rotation only) and the
// rotation of every head's pairs (i, i+64); st(base, ra, rb) receives the rotated values of columns
// [base, base+4) and [base+64, base+68).  Shared by every kernel that applies the QK-norm + RoPE, so that a
// row comes out bit-identical whichever launch produced it.
template <class St>
__device__ __forceinline__ void qknorm_rope_segment(const float* __restrict__ xs, const float* __restrict__ ws, int d,
                                                    float eps, const float (&cs)[4], const float (&sn)[4], int o, int lane,
                                                    St&& st) {
  const int units = d >> 3;  // (head, float4-pair) units per segment = H * 16
  float4 lo[kMaxVec / 2], hi[kMaxVec / 2];
  float ss = 0.f;
#pragma unroll
  for (int it = 0; it < kMaxVec / 2; ++it) {
    const int u = it * 32 + lane;
    if (u < units) {
      const int base = (u >> 4) * 128 + o;
      lo[it] = *reinterpret_cast<const float4*>(xs + base);
      hi[it] = *reinterpret_cast<const float4*>(xs + base + 64);
      ss += lo[it].x * lo[it].x + lo[it].y * lo[it].y + lo[it].z * lo[it].z + lo[it].w * lo[it].w;
      ss += hi[it].x * hi[it].x + hi[it].y * hi[it].y + hi[it].z * hi[it].z + hi[it].w * hi[it].w;
    }
  }
  ss = warp_sum(ss);
  const float r = ws ? rsqrtf(ss / d + eps) : 1.0f;  // ws == NULL: rotation only (apply_rotary_emb_one_cossin)
#pragma unroll
  for (int it = 0; it < kMaxVec / 2; ++it) {
    const int u = it * 32 + lane;
    if (u < units) {
      const int base = (u >> 4) * 128 + o;
      const float4 one4 = make_float4(1.f, 1.f, 1.f, 1.f);
      const float4 wl = ws ? __ldg(reinterpret_cast<const float4*>(ws + base)) : one4;
      const float4 wh = ws ? __ldg(reinterpret_cast<const float4*>(ws + base + 64)) : one4;
      const float a[4] = {lo[it].x * r * wl.x, lo[it].y * r * wl.y, lo[it].z * r * wl.z, lo[it].w * r * wl.w};
      const float b[4] = {hi[it].x * r * wh.x, hi[it].y * r * wh.y, hi[it].z * r * wh.z, hi[it].w * r * wh.w};
      float ra[4], rb[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        ra[e] = a[e] * cs[e] - b[e] * sn[e];
        rb[e] = b[e] * cs[e] + a[e] * sn[e];
      }
      st(base, ra, rb);
    }
  }
}

// warp-per-row variant (no view fan-out): in_period == 0
__global__ void __launch_bounds__(256, 3)
    qknorm_rope_rows_kernel(const float* __restrict__ x, long long ldx, int in_period,
                                   const float* __restrict__ w, void* __restrict__ out, long long ldo,
                                   int rows, int d, int nseg, float eps, const float* __restrict__ pos,
                                   const float* __restrict__ freqs, int nfreq, int out_dtype,
                                   const float* __restrict__ ctab = nullptr, const float* __restrict__ stab = nullptr,
                                   long long ldtab = 0) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const long long src = in_period > 0 ? (row % in_period) : row;
  const int o = (lane & 15) * 4;  // pair offset inside a head (0..60)
  float cs[4], sn[4];
  rope_lane_cs(pos ? pos + (long long)row * 9 : nullptr, freqs, nfreq, ctab ? ctab + (long long)row * ldtab : nullptr,
               ctab ? stab + (long long)row * ldtab : nullptr, o, cs, sn);
  const int s = blockIdx.y;  // one (row, segment) per warp: twice the warps, no serial segment loop
  qknorm_rope_segment(x + src * ldx + (long long)s * d, w ? w + (long long)s * d : nullptr, d, eps, cs, sn, o, lane,
                      [&](int base, const float (&ra)[4], const float (&rb)[4]) {
                        const long long idx = (long long)row * ldo + (long long)s * d + base;
                        store4_16(out, out_dtype, idx, ra[0], ra[1], ra[2], ra[3]);
                        store4_16(out, out_dtype, idx + 64, rb[0], rb[1], rb[2], rb[3]);
                      });
}

// ---------------------------------------------------------------------------------------------
// Row-sharded scene stage: what follows a rank's fused [q | k | v] projection (fp32 [rows, 3d], the RMSNorm
// row factor already applied) -- and the all-gather of the layer, fused into the producer:
//   segment 0: q -> QK-RMSNorm + RoPE -> out_q [rows, ldq]                          (this rank's queries)
//   segment 1: k -> QK-RMSNorm + RoPE -> row row0 + r, columns [0, d)   of EVERY destination
//   segment 2: v -> cast              -> row row0 + r, columns [d, 2d)  of EVERY destination
// The destinations are the [k | v] row stores of all ranks: either n_dst peer-mapped pointers (plain stores
// over NVLink) or ONE NVLS multicast address (multimem.st: the NVSwitch replicates every store into all
// ranks' memories, so a rank sends its rows once instead of once per peer).
// ---------------------------------------------------------------------------------------------
struct KvDst {
  void* p[8];
};

__device__ __forceinline__ void store_kv8(const KvDst& dst, int n_dst, int multicast, long long idx, uint2 u) {
  if (multicast) {
    uint16_t* a = static_cast<uint16_t*>(dst.p[0]) + idx;
    asm volatile("multimem.st.weak.global.v2.f32 [%0], {%1, %2};" ::"l"(a), "f"(__uint_as_float(u.x)),
                 "f"(__uint_as_float(u.y))
                 : "memory");
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i)  // static indices: the pointers stay in the kernel's parameter bank
      if (i < n_dst) {
        uint16_t* a = static_cast<uint16_t*>(dst.p[i]) + idx;
        asm volatile("st.global.v2.b32 [%0], {%1, %2};" ::"l"(a), "r"(u.x), "r"(u.y) : "memory");
      }
  }
}

__device__ __forceinline__ uint2 pack4_16(int dtype, float a, float b, float c, float d) {
  uint2 u;
  if (dtype == RFB_BF16) u.x = pack_bf16(a, b), u.y = pack_bf16(c, d);
  else u.x = pack_f16(a, b), u.y = pack_f16(c, d);
  return u;
}

__global__ void __launch_bounds__(256, 3)
    qkv_post_kernel(const float* __restrict__ x, long long ldx, const float* __restrict__ w_qk,
                    void* __restrict__ out_q, long long ldq, const __grid_constant__ KvDst dst, int n_dst, int multicast, long long ldkv,
                    long long row0, int rows, int d, float eps, const float* __restrict__ pos,
                    const float* __restrict__ freqs, int nfreq, int out_dtype) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int s = blockIdx.y;
  const float* xs = x + (long long)row * ldx + (long long)s * d;
  const long long kv_row = (row0 + row) * ldkv;
  if (s == 2) {
    const int nvec = d >> 7;
#pragma unroll
    for (int j = 0; j < kMaxVec; ++j)
      if (j < nvec) {
        const float4 v = *reinterpret_cast<const float4*>(xs + (j * 32 + lane) * 4);
        store_kv8(dst, n_dst, multicast, kv_row + d + (j * 32 + lane) * 4, pack4_16(out_dtype, v.x, v.y, v.z, v.w));
      }
    return;
  }
  const int o = (lane & 15) * 4;
  float cs[4], sn[4];
  rope_lane_cs(pos ? pos + (long long)row * 9 : nullptr, freqs, nfreq, nullptr, nullptr, o, cs, sn);
  qknorm_rope_segment(xs, w_qk + (long long)s * d, d, eps, cs, sn, o, lane,
                      [&](int base, const float (&ra)[4], const float (&rb)[4]) {
                        if (s == 0) {
                          const long long idx = (long long)row * ldq + base;
                          store4_16(out_q, out_dtype, idx, ra[0], ra[1], ra[2], ra[3]);
                          store4_16(out_q, out_dtype, idx + 64, rb[0], rb[1], rb[2], rb[3]);
                        } else {
                          store_kv8(dst, n_dst, multicast, kv_row + base, pack4_16(out_dtype, ra[0], ra[1], ra[2], ra[3]));
                          store_kv8(dst, n_dst, multicast, kv_row + base + 64,
                                    pack4_16(out_dtype, rb[0], rb[1], rb[2], rb[3]));
                        }
                      });
}


constexpr int kRopeViews = 4;  // views rotated per pass over one source row (= warps per block)

__global__ void __launch_bounds__(kRopeViews * 32, 6)
    qknorm_rope_kernel(const float* __restrict__ x, long long ldx, int in_period, const float* __restrict__ w,
                       void* __restrict__ out, long long ldo, int rows, int d, int nseg, float eps,
                       const float* __restrict__ pos, const float* __restrict__ freqs, int nfreq, int out_dtype) {
  // One block (4 warps) per SOURCE row.  With in_period > 0 the same source row feeds
  // rows / in_period output rows (one per view, each with its own positions): warp v computes the
  // rotation table of view v once into shared memory, then the warps split the row's segments and
  // rotate each normalised segment for all views of the group from registers.
  __shared__ float s_cs[kRopeViews][64], s_sn[kRopeViews][64];
  const int src_rows = in_period > 0 ? in_period : rows;
  const int nv = in_period > 0 ? rows / in_period : 1;
  const int src = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int o = (lane & 15) * 4;  // pair offset inside a head (0..60)
  const int units = d >> 3;       // (head, float4-pair) units per segment = H * 16

  for (int v0 = 0; v0 < nv; v0 += kRopeViews) {
    __syncthreads();
    if (v0 + warp < nv) {
      const long long row = (long long)(v0 + warp) * src_rows + src;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int i = lane * 2 + e;  // pair index 0..63
        float c = 1.f, sn = 0.f;
        if (pos && i < 9 * nfreq) fast_sincos(pos[row * 9 + i / nfreq] * __ldg(freqs + i % nfreq), sn, c);
        s_cs[warp][i] = c, s_sn[warp][i] = sn;
      }
    }
    __syncthreads();
    for (int s = warp; s < nseg; s += kRopeViews) {
      const float* xs = x + (long long)src * ldx + (long long)s * d;
      const float* ws = w + (long long)s * d;
      float4 lo[kMaxVec / 2], hi[kMaxVec / 2];
      float ss = 0.f;
#pragma unroll
      for (int it = 0; it < kMaxVec / 2; ++it) {
        const int u = it * 32 + lane;
        if (u < units) {
          const int base = (u >> 4) * 128 + o;
          lo[it] = *reinterpret_cast<const float4*>(xs + base);
          hi[it] = *reinterpret_cast<const float4*>(xs + base + 64);
          ss += lo[it].x * lo[it].x + lo[it].y * lo[it].y + lo[it].z * lo[it].z + lo[it].w * lo[it].w;
          ss += hi[it].x * hi[it].x + hi[it].y * hi[it].y + hi[it].z * hi[it].z + hi[it].w * hi[it].w;
        }
      }
      ss = warp_sum(ss);
      const float r = rsqrtf(ss / d + eps);
#pragma unroll
      for (int it = 0; it < kMaxVec / 2; ++it) {
        const int u = it * 32 + lane;
        if (u < units) {
          const int base = (u >> 4) * 128 + o;
          const float4 wl = __ldg(reinterpret_cast<const float4*>(ws + base));
          const float4 wh = __ldg(reinterpret_cast<const float4*>(ws + base + 64));
          const float a[4] = {lo[it].x * r * wl.x, lo[it].y * r * wl.y, lo[it].z * r * wl.z, lo[it].w * r * wl.w};
          const float b[4] = {hi[it].x * r * wh.x, hi[it].y * r * wh.y, hi[it].z * r * wh.z, hi[it].w * r * wh.w};
          for (int vv = 0; vv < kRopeViews && v0 + vv < nv; ++vv) {
            const float4 c4 = *reinterpret_cast<const float4*>(&s_cs[vv][o]);
            const float4 s4 = *reinterpret_cast<const float4*>(&s_sn[vv][o]);
            const float cs[4] = {c4.x, c4.y, c4.z, c4.w}, sn[4] = {s4.x, s4.y, s4.z, s4.w};
            float ra[4], rb[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              ra[e] = a[e] * cs[e] - b[e] * sn[e];
              rb[e] = b[e] * cs[e] + a[e] * sn[e];
            }
            const long long idx = ((long long)(v0 + vv) * src_rows + src) * ldo + (long long)s * d + base;
            store4_16(out, out_dtype, idx, ra[0], ra[1], ra[2], ra[3]);
            store4_16(out, out_dtype, idx + 64, rb[0], rb[1], rb[2], rb[3]);
          }
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// out[r, :] = token + rmsnorm(a[r]) * wa (+ rmsnorm(b[r]) * wb)   (eps = fp32 machine eps)
//   models/renderformer.py:139-159 (tri_token + texture emb + normal emb),
//   models/view_transformer.py:108 (ray_map_patch_token + ray emb).
// Rows [0, n_prefix) of every batch item are copied from `prefix` (register tokens, :151,163).
// ---------------------------------------------------------------------------------------------
__global__ void token_assemble_kernel(const float* __restrict__ a, const float* __restrict__ wa,
                                      const float* __restrict__ b, const float* __restrict__ wb,
                                      const float* __restrict__ token, const float* __restrict__ prefix,
                                      int n_prefix, float* __restrict__ out, int rows_in, int rows_out,
                                      int batch, int d, float eps) {
  const int gr = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (gr >= batch * rows_out) return;
  const int lane = threadIdx.x & 31;
  const int bi = gr / rows_out, r = gr % rows_out;
  float4* orow = reinterpret_cast<float4*>(out + (long long)gr * d);
  const int nvec = d >> 7;
  if (r < n_prefix) {
    const float4* p = reinterpret_cast<const float4*>(prefix + (long long)r * d);
    for (int j = 0; j < nvec; ++j) orow[j * 32 + lane] = p[j * 32 + lane];
    return;
  }
  const int ri = r - n_prefix;
  if (ri >= rows_in) {  // padding rows
    for (int j = 0; j < nvec; ++j) orow[j * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  const float4* ar = reinterpret_cast<const float4*>(a + ((long long)bi * rows_in + ri) * d);
  const float4* br = b ? reinterpret_cast<const float4*>(b + ((long long)bi * rows_in + ri) * d) : nullptr;
  float4 va[kMaxVec], vb[kMaxVec];
  float sa = 0.f, sb = 0.f;
#pragma unroll
  for (int j = 0; j < kMaxVec; ++j)
    if (j < nvec) {
      va[j] = ar[j * 32 + lane];
      sa += va[j].x * va[j].x + va[j].y * va[j].y + va[j].z * va[j].z + va[j].w * va[j].w;
      if (br) {
        vb[j] = br[j * 32 + lane];
        sb += vb[j].x * vb[j].x + vb[j].y * vb[j].y + vb[j].z * vb[j].z + vb[j].w * vb[j].w;
      }
    }
  sa = warp_sum(sa), sb = warp_sum(sb);
  const float ra = rsqrtf(sa / d + eps), rb = rsqrtf(sb / d + eps);
#pragma unroll
  for (int j = 0; j < kMaxVec; ++j)
    if (j < nvec) {
      const int c = j * 32 + lane;
      const float4 t = __ldg(reinterpret_cast<const float4*>(token) + c);
      const float4 ga = __ldg(reinterpret_cast<const float4*>(wa) + c);
      float4 o = make_float4(t.x + va[j].x * ra * ga.x, t.y + va[j].y * ra * ga.y,
                             t.z + va[j].z * ra * ga.z, t.w + va[j].w * ra * ga.w);
      if (br) {
        const float4 gb = __ldg(reinterpret_cast<const float4*>(wb) + c);
        o.x += vb[j].x * rb * gb.x, o.y += vb[j].y * rb * gb.y;
        o.z += vb[j].z * rb * gb.z, o.w += vb[j].w * rb * gb.w;
      }
      orow[c] = o;
    }
}

// texture fp32 [n, C*P*P] -> f16, log10(x+1) on the last 3 channels (rendering_pipeline.py:67-68)
__global__ void texture_prep_kernel(const float* __restrict__ tex, uint16_t* __restrict__ out,
                                    long long n_vec4, int per_tri_vec4, int log_from_vec4) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec4;
       i += (long long)gridDim.x * blockDim.x) {
    float4 v = __ldg(reinterpret_cast<const float4*>(tex) + i);
    if ((int)(i % per_tri_vec4) >= log_from_vec4) {
      v.x = log10f(v.x + 1.f), v.y = log10f(v.y + 1.f), v.z = log10f(v.z + 1.f), v.w = log10f(v.w + 1.f);
    }
    store4_16(out, RFB_F16, i * 4, v.x, v.y, v.z, v.w);
  }
}

// per-triangle constant texture [n, C] fp32 -> f16 [n, ld] (zero padded), log10(x+1) on the last
// `log_channels` channels: the input of the reduced texture projection (constant-texture fast path)
__global__ void texture_const_prep_kernel(const float* __restrict__ tex, uint16_t* __restrict__ out, long long n,
                                          int channels, int ld, int log_channels) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * ld) return;
  const long long row = t / ld;
  const int c = (int)(t % ld);
  float v = 0.f;
  if (c < channels) {
    v = tex[row * channels + c];
    if (c >= channels - log_channels) v = log10f(v + 1.f);
  }
  out[t] = __half_as_ushort(__float2half_rn(v));
}

// vertex normals [n, 9] -> NeRF encoding [n, 128] f16 (117 used: x | sin(x 2^j) | cos(x 2^j), zero pad)
//   encodings/nerf_encoding.py:63-84 with F frequencies, input-major / frequency-minor order.
__global__ void vn_encode_kernel(const float* __restrict__ vn, uint16_t* __restrict__ out, int n, int nf,
                                 int ld) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * ld) return;
  const int row = t / ld, c = t % ld;
  float v = 0.f;
  const float* x = vn + (long long)row * 9;
  if (c < 9) {
    v = x[c];
  } else if (c < 9 + 9 * nf) {
    const int k = c - 9;
    v = sinf(x[k / nf] * exp2f((float)(k % nf)));
  } else if (c < 9 + 18 * nf) {
    const int k = c - 9 - 9 * nf;
    v = sinf(x[k / nf] * exp2f((float)(k % nf)) + 1.5707963267948966f);
  }
  __half h = __float2half(v);
  out[t] = *reinterpret_cast<uint16_t*>(&h);
}

// Pinhole camera of an H x W image: square pixels, principal point at the image centre, the field of view
// spanning the LONGER side (Blender's "Auto" sensor fit), so f = max(H, W) / 2 / tan(fov / 2); pixel centres at
// +0.5.  For H == W this is utils/ray_generator.py:13-50, evaluated in the same float order.
__device__ __forceinline__ float pinhole_focal(int H, int W, float fov_rad) {
  return (max(H, W) * 0.5f) / tanf(0.5f * fov_rad);
}

// Ray-bundle patch tokens for V pinhole cameras in camera space:
//   utils/ray_generator.py:13-50 (c2w = identity) + models/view_transformer.py:104-107.
// out [V, (Hc/8)*(Wc/8), 192] f16 over an Hc x Wc canvas, feature = c*64 + p1*8 + p2, token = h1*(Wc/8) + w1
// (row-major patch grid).  The camera is the one of the H x W image the canvas holds at (top, left): f from
// max(H, W), principal point (cx, cy) = (left + W/2, top + H/2) in canvas pixels.  Canvas == image is the plain
// H x W camera (cx = W * 0.5 is the same exact float the subtraction used before).
__global__ void ray_tokens_kernel(const float* __restrict__ fov_deg, uint16_t* __restrict__ out, int V, int Hc,
                                  int Wc, int H, int W, float cx, float cy) {
  const int P = 8, Tw = Wc / P;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_view = (long long)(Hc / P) * Tw * 192;
  if (t >= V * per_view) return;
  const int v = t / per_view;
  const int rem = t % per_view;
  const int tok = rem / 192, f = rem % 192;
  const int c = f >> 6, p1 = (f >> 3) & 7, p2 = f & 7;
  const int py = (tok / Tw) * P + p1, px = (tok % Tw) * P + p2;
  const float fov = fov_deg[v] / 180.f * 3.14159265358979323846f;
  const float fl = pinhole_focal(H, W, fov);
  const float dx = ((px + 0.5f) - cx) / fl;
  const float dy = -((py + 0.5f) - cy) / fl;
  const float inv = 1.0f / fmaxf(sqrtf(dx * dx + dy * dy + 1.f), 1e-12f);
  const float val = (c == 0 ? dx : (c == 1 ? dy : -1.f)) * inv;
  __half h = __float2half(val);
  out[t] = *reinterpret_cast<uint16_t*>(&h);
}

// The same tokens for V cameras with user-set pinhole intrinsics intr [V, 4] = (fx, fy, cx, cy) in pixels of the
// H x W image the canvas holds at (top, left); pixel (row i, column j) of the image has its centre at (j + 0.5,
// i + 0.5) and the ray normalize(((u - cx) / fx, -(v - cy) / fy, -1)).  With the intrinsics of rfb_intrinsics_from_fov
// (auto fit) u - cx and (px + 0.5) - (left + W/2) are the same exact float, so the tokens equal ray_tokens_kernel's.
// The normalisation repeats ray_tokens_kernel's expressions verbatim: moving them into a shared inline function
// reschedules that kernel's compiled code.
__global__ void ray_tokens_intrinsics_kernel(const float* __restrict__ intr, uint16_t* __restrict__ out, int V,
                                             int Hc, int Wc, int top, int left) {
  const int P = 8, Tw = Wc / P;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_view = (long long)(Hc / P) * Tw * 192;
  if (t >= V * per_view) return;
  const int v = t / per_view;
  const int rem = t % per_view;
  const int tok = rem / 192, f = rem % 192;
  const int c = f >> 6, p1 = (f >> 3) & 7, p2 = f & 7;
  const int py = (tok / Tw) * P + p1, px = (tok % Tw) * P + p2;
  const float fx = intr[4 * v], fy = intr[4 * v + 1], cx = intr[4 * v + 2], cy = intr[4 * v + 3];
  const float u = (float)(px - left) + 0.5f, vv = (float)(py - top) + 0.5f;
  const float dx = (u - cx) / fx;
  const float dy = -(vv - cy) / fy;
  const float inv = 1.0f / fmaxf(sqrtf(dx * dx + dy * dy + 1.f), 1e-12f);
  const float val = (c == 0 ? dx : (c == 1 ? dy : -1.f)) * inv;
  __half h = __float2half(val);
  out[t] = *reinterpret_cast<uint16_t*>(&h);
}

// The same tokens for V lens-distorted cameras: intrinsics intr [V, 4] as ray_tokens_intrinsics_kernel, and per view
// dist [V, 8] = (k1, k2, p1, p2, k3, k4, k5, k6) (lens 0, OpenCV / COLMAP FULL_OPENCV) or dist [V, 4] = (k1, k2, k3,
// k4) (lens 1, OpenCV fisheye / COLMAP OPENCV_FISHEYE).  A pixel's distorted normalized coordinates are
// (xd, yd) = ((u - cx) / fx, (v - cy) / fy) in COLMAP's axes (y down).
//   lens 0: Newton's method with the analytic 2x2 Jacobian, from (xd, yd), solves
//           xd = x g + 2 p1 x y + p2 (r2 + 2 x^2),  yd = y g + p1 (r2 + 2 y^2) + 2 p2 x y,
//           g = (1 + k1 r2 + k2 r2^2 + k3 r2^3) / (1 + k4 r2 + k5 r2^2 + k6 r2^3),  r2 = x^2 + y^2,
//           and the ray is normalize((x, -y, -1)).
//   lens 1: 1-D Newton in fp64 from theta = rd = |(xd, yd)| solves rd = theta (1 + k1 t2 + k2 t2^2 + k3 t2^3 + k4 t2^4),
//           t2 = theta^2, and the ray is (sin theta xd / rd, -sin theta yd / rd, -cos theta) ((0, 0, -1) at rd = 0).
// One thread per pixel: the solve is ~20x the pinhole's arithmetic, so it runs once and writes the three channels.
// Threads are ordered (view, token, p1, p2) so that a warp stores 64 contiguous bytes per channel.  With all
// coefficients zero the first residual is exactly 0, so (x, -y) are ray_tokens_intrinsics_kernel's (dx, dy) and the
// normalisation below repeats its expressions, with the contraction its SASS shows (fma(dx, dx, dy * dy) + 1) pinned:
// the tokens are that kernel's, bit for bit.  A pixel that does not converge keeps its last iterate; a non-finite one
// (coefficients that fold or a vanishing denominator, which the host checks only for host tensors) falls back to the
// pinhole ray normalize((xd, -yd, -1)), so no token is ever non-finite for finite intrinsics.
__global__ void ray_tokens_lens_kernel(const float* __restrict__ intr, const float* __restrict__ dist, int lens,
                                       uint16_t* __restrict__ out, int V, int Hc, int Wc, int top, int left) {
  const int P = 8, Tw = Wc / P;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_view = (long long)Hc * Wc;
  if (t >= V * per_view) return;
  const int v = t / per_view;
  const int rem = t % per_view;
  const int tok = rem / 64, p1 = (rem >> 3) & 7, p2 = rem & 7;
  const int py = (tok / Tw) * P + p1, px = (tok % Tw) * P + p2;
  const float fx = intr[4 * v], fy = intr[4 * v + 1], cx = intr[4 * v + 2], cy = intr[4 * v + 3];
  const float u = (float)(px - left) + 0.5f, vv = (float)(py - top) + 0.5f;
  const float xd = (u - cx) / fx;
  const float yd = (vv - cy) / fy;
  float o0, o1, o2;
  bool pinhole = true;
  if (lens == 0) {
    const float* k = dist + 8 * v;
    const float k1 = k[0], k2 = k[1], q1 = k[2], q2 = k[3], k3 = k[4], k4 = k[5], k5 = k[6], k6 = k[7];
    float x = xd, y = yd;
    for (int it = 0; it < 20; ++it) {
      const float x2 = x * x, y2 = y * y, xy = x * y, r2 = x2 + y2;
      const float num = 1.f + r2 * (k1 + r2 * (k2 + r2 * k3));
      const float den = 1.f + r2 * (k4 + r2 * (k5 + r2 * k6));
      const float g = num / den;
      const float gp = ((k1 + r2 * (2.f * k2 + r2 * 3.f * k3)) * den - num * (k4 + r2 * (2.f * k5 + r2 * 3.f * k6))) /
                       (den * den);  // dg / dr2
      const float ex = x * g + 2.f * q1 * xy + q2 * (r2 + 2.f * x2) - xd;
      const float ey = y * g + q1 * (r2 + 2.f * y2) + 2.f * q2 * xy - yd;
      const float jxx = g + 2.f * x2 * gp + 2.f * q1 * y + 6.f * q2 * x;
      const float jyy = g + 2.f * y2 * gp + 6.f * q1 * y + 2.f * q2 * x;
      const float jxy = 2.f * xy * gp + 2.f * q1 * x + 2.f * q2 * y;
      const float det = jxx * jyy - jxy * jxy;
      const float sx = (jyy * ex - jxy * ey) / det, sy = (jxx * ey - jxy * ex) / det;
      x -= sx;
      y -= sy;
      if (!(fabsf(sx) + fabsf(sy) > 1e-7f * (1.f + fabsf(x) + fabsf(y)))) break;  // converged, or NaN
    }
    if (isfinite(x) && isfinite(y)) {
      const float dx = x;
      const float dy = -y;
      const float inv = 1.0f / fmaxf(sqrtf(__fadd_rn(__fmaf_rn(dx, dx, __fmul_rn(dy, dy)), 1.f)), 1e-12f);
      o0 = dx * inv;
      o1 = dy * inv;
      o2 = -1.f * inv;
      pinhole = false;
    }
  } else {
    // in fp64: -cos theta crosses zero at 90 degrees, and near there an fp32 theta (or fp32 (xd, yd)) cannot resolve it
    // to an fp16 ulp of the token
    const float* k = dist + 4 * v;
    const double k1 = k[0], k2 = k[1], k3 = k[2], k4 = k[3];
    const double x = ((double)u - cx) / fx, y = ((double)vv - cy) / fy;
    const double rd = sqrt(x * x + y * y);
    double th = rd;
    for (int it = 0; it < 20; ++it) {
      const double t2 = th * th;
      const double poly = 1.0 + t2 * (k1 + t2 * (k2 + t2 * (k3 + t2 * k4)));
      const double dpoly = 1.0 + t2 * (3.0 * k1 + t2 * (5.0 * k2 + t2 * (7.0 * k3 + t2 * 9.0 * k4)));
      const double s = (th * poly - rd) / dpoly;
      th -= s;
      if (!(fabs(s) > 1e-12 * (1.0 + th))) break;  // converged (the next step would be ~1e-24), or NaN
    }
    if (isfinite(th)) {
      double sn, cs;
      sincos(th, &sn, &cs);
      const double q = rd > 0.0 ? sn / rd : 0.0;
      o0 = (float)(q * x);
      o1 = (float)(-q * y);
      o2 = rd > 0.0 ? (float)-cs : -1.f;
      pinhole = false;
    }
  }
  if (pinhole) {
    const float inv = 1.0f / fmaxf(sqrtf(xd * xd + yd * yd + 1.f), 1e-12f);
    o0 = xd * inv;
    o1 = -yd * inv;
    o2 = -inv;
  }
  uint16_t* o = out + ((long long)v * (Hc / P) * Tw + tok) * 192 + p1 * 8 + p2;
  o[0] = __half_as_ushort(__float2half(o0));
  o[64] = __half_as_ushort(__float2half(o1));
  o[128] = __half_as_ushort(__float2half(o2));
}

// fov in degrees [V] -> intrinsics [V, 4] = (f, f, W/2, H/2) of an H x W image, the fov spanning the longer side
// (fit 0, "auto": ray_tokens_kernel's own focal length, bit for bit), the width (1) or the height (2).
__global__ void intrinsics_from_fov_kernel(const float* __restrict__ fov_deg, float* __restrict__ out, int V, int H,
                                           int W, int fit) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= V) return;
  const float fov = fov_deg[v] / 180.f * 3.14159265358979323846f;
  const int side = fit == 1 ? W : (fit == 2 ? H : max(H, W));
  const float fl = pinhole_focal(side, side, fov);
  out[4 * v] = fl;
  out[4 * v + 1] = fl;
  out[4 * v + 2] = W * 0.5f;
  out[4 * v + 3] = H * 0.5f;
}

// explicit ray map [V, H, W, 3] fp32 -> patch tokens (same layout as ray_tokens_kernel): the model-level
// entry RenderFormer.forward(..., rays_d, ...) (models/renderformer.py:171-206) hands the rays in
__global__ void ray_map_tokens_kernel(const float* __restrict__ rays, uint16_t* __restrict__ out, int V, int H,
                                      int W) {
  const int P = 8, Tw = W / P;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_view = (long long)(H / P) * Tw * 192;
  if (t >= V * per_view) return;
  const int v = t / per_view;
  const int rem = t % per_view;
  const int tok = rem / 192, f = rem % 192;
  const int c = f >> 6, p1 = (f >> 3) & 7, p2 = f & 7;
  const int py = (tok / Tw) * P + p1, px = (tok % Tw) * P + p2;
  __half h = __float2half(rays[(((long long)v * H + py) * W + px) * 3 + c]);
  out[t] = *reinterpret_cast<uint16_t*>(&h);
}

// Pinhole ray map of V cameras: rays_d [V, H, W, 3] fp32 = normalize(R_v * ((x - cx) / f, -(y - cy) / f, -1)),
// the camera of pinhole_focal, fov in RADIANS as RayGenerator.forward takes it (utils/ray_generator.py:13-50).
// One thread per pixel, 12-byte stores.
__global__ void ray_map_kernel(const float* __restrict__ c2w, const float* __restrict__ fov_rad, float* __restrict__ out,
                               int V, int H, int W) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)V * H * W) return;
  const int v = t / ((long long)H * W);
  const int rem = t % ((long long)H * W);
  const int py = rem / W, px = rem % W;
  const float fl = pinhole_focal(H, W, fov_rad[v]);
  const float d[3] = {((px + 0.5f) - W * 0.5f) / fl, -((py + 0.5f) - H * 0.5f) / fl, -1.0f};
  const float* m = c2w + (long long)v * 16;
  float r[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) r[i] = m[i * 4] * d[0] + m[i * 4 + 1] * d[1] + m[i * 4 + 2] * d[2];
  const float inv = 1.0f / fmaxf(sqrtf(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]), 1e-12f);
  out[t * 3] = r[0] * inv, out[t * 3 + 1] = r[1] * inv, out[t * 3 + 2] = r[2] * inv;
}

// RoPE positions: pos[v, 0:n_reg] = masked vertex centroid (x3), pos[v, n_reg + i] = T_v^-1 tri_i.
//   models/renderformer.py:103-124, utils/transform.py:7-27.  One block per view; c2w == NULL
//   keeps world coordinates (the view-independent stage).
__global__ void positions_kernel(const float* __restrict__ tri, const uint8_t* __restrict__ mask,
                                 const float* __restrict__ c2w, float* __restrict__ pos, int n, int n_reg,
                                 int rows_out) {
  const int v = blockIdx.x;
  float R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, tr[3] = {0, 0, 0};
  if (c2w) {
    const float* m = c2w + (long long)v * 16;
    for (int i = 0; i < 3; ++i) {
      for (int j = 0; j < 3; ++j) R[i * 3 + j] = m[i * 4 + j];
      tr[i] = m[i * 4 + 3];
    }
  }
  float* pv = pos + (long long)v * rows_out * 9;
  float acc[3] = {0.f, 0.f, 0.f};
  float cnt = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const float* t = tri + (long long)i * 9;
    float o[9];
    for (int k = 0; k < 3; ++k) {
      const float x = t[k * 3] - tr[0], y = t[k * 3 + 1] - tr[1], z = t[k * 3 + 2] - tr[2];
      // x_cam = R^T (x - t)
      o[k * 3 + 0] = R[0] * x + R[3] * y + R[6] * z;
      o[k * 3 + 1] = R[1] * x + R[4] * y + R[7] * z;
      o[k * 3 + 2] = R[2] * x + R[5] * y + R[8] * z;
    }
    for (int k = 0; k < 9; ++k) pv[(long long)(n_reg + i) * 9 + k] = o[k];
    if (mask[i]) {
      cnt += 1.f;
      for (int k = 0; k < 3; ++k) acc[k] += o[k] + o[3 + k] + o[6 + k];
    }
  }
  for (int i = n_reg + n + threadIdx.x; i < rows_out; i += blockDim.x)
    for (int k = 0; k < 9; ++k) pv[(long long)i * 9 + k] = 0.f;
  __shared__ float red[4][32];
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  float vals[4] = {acc[0], acc[1], acc[2], cnt};
  for (int k = 0; k < 4; ++k) {
    vals[k] = warp_sum(vals[k]);
    if (lane == 0) red[k][wp] = vals[k];
  }
  __syncthreads();
  if (wp == 0) {
    for (int k = 0; k < 4; ++k) {
      float s = lane < (blockDim.x >> 5) ? red[k][lane] : 0.f;
      vals[k] = warp_sum(s);
    }
    if (lane < n_reg) {
      const float inv = 1.0f / (vals[3] + 1e-5f) / 3.0f;
      for (int k = 0; k < 9; ++k) pv[(long long)lane * 9 + k] = vals[k % 3] * inv;
    }
  }
}

// key mask bytes [B, n] -> packed bits [B, words] with n_prefix always-valid keys in front
__global__ void pack_mask_kernel(const uint8_t* __restrict__ mask, uint32_t* __restrict__ bits, int n,
                                 int n_prefix, int words, int batch) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= batch * words) return;
  const int b = t / words, w = t % words;
  uint32_t out = 0;
  for (int i = 0; i < 32; ++i) {
    const int k = w * 32 + i;
    bool ok = k < n_prefix;
    if (!ok && k - n_prefix < n) ok = mask[(long long)b * n + (k - n_prefix)] != 0;
    out |= (ok ? 1u : 0u) << i;
  }
  bits[t] = out;
}

__global__ void cast_kernel(const float* __restrict__ x, void* __restrict__ out, int dtype, long long n_vec4) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_vec4;
       i += (long long)gridDim.x * blockDim.x) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(x) + i);
    store4_16(out, dtype, i * 4, v.x, v.y, v.z, v.w);
  }
}

// 16-bit matrix transpose out[c][r] = in[r][c] through a padded 64 x 64 shared-memory tile: 32-bit (two-element)
// accesses on both sides, 128 contiguous bytes per warp row.  Used by the row-sharded scene stage: V arrives
// row-major from the all-gather of the ranks' [k | v] rows and the attention kernels want V^T (keys contiguous).
__global__ void __launch_bounds__(256) transpose16_kernel(const uint16_t* __restrict__ in, long long ld_in,
                                                          uint16_t* __restrict__ out, long long ld_out, int rows, int cols) {
  __shared__ uint16_t tile[64][66];
  const int r0 = blockIdx.y * 64, c0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = r0 + ty + i * 8, c = c0 + tx * 2;
    uint32_t v = 0;
    if (r < rows && c < cols) v = *reinterpret_cast<const uint32_t*>(in + (long long)r * ld_in + c);  // cols even
    tile[ty + i * 8][tx * 2] = static_cast<uint16_t>(v & 0xffffu);
    tile[ty + i * 8][tx * 2 + 1] = static_cast<uint16_t>(v >> 16);
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = c0 + ty + i * 8, r = r0 + tx * 2;  // output row = input column
    if (c < cols && r < rows) {
      const uint32_t v = static_cast<uint32_t>(tile[tx * 2][ty + i * 8]) |
                         (static_cast<uint32_t>(tile[tx * 2 + 1][ty + i * 8]) << 16);
      if (r + 1 < rows) *reinterpret_cast<uint32_t*>(out + (long long)c * ld_out + r) = v;
      else out[(long long)c * ld_out + r] = static_cast<uint16_t>(v & 0xffffu);
    }
  }
}

}  // namespace rfb

using namespace rfb;

#define RFB_LAUNCHED(name) \
  g_launch_count++;        \
  return check_launch(name)

extern "C" int rfb_rmsnorm(const float* x, long long ldx, const float* w, void* out, int out_dtype,
                           long long ldo, int rows, int d, float eps, const int* gather,
                           rfb_stream_t stream) {
  if (!x || !w || !out || rows <= 0 || d % 128 || d > kMaxVec * 128 || ldx % 4 || ldo % 4) return RFB_ERR_ARG;
  const int wpb = 8;
  rmsnorm_kernel<<<(rows + wpb - 1) / wpb, wpb * 32, 0, (cudaStream_t)stream>>>(x, ldx, w, out, out_dtype, ldo,
                                                                               rows, d, eps, gather);
  RFB_LAUNCHED("rmsnorm_kernel");
}

extern "C" int rfb_rowstat(const float* x, void* out16, int out_dtype, long long ld16, float* sumsq, int sumsq_ld,
                           int parts, int rows, int d, const int* gather, rfb_stream_t stream) {
  if (!x || !out16 || !sumsq || rows <= 0 || d % 128 || d > kMaxVec * 128 || ld16 < d || ld16 % 4) return RFB_ERR_ARG;
  if (parts < 1 || parts > 32 || sumsq_ld < parts) return RFB_ERR_ARG;
  const int wpb = 8;
  rowstat_kernel<<<(rows + wpb - 1) / wpb, wpb * 32, 0, (cudaStream_t)stream>>>(x, out16, out_dtype, ld16, sumsq, sumsq_ld, parts, rows, d, gather);
  RFB_LAUNCHED("rowstat_kernel");
}

extern "C" int rfb_qknorm_rope(const float* x, long long ldx, int in_period, const float* w, void* out, int out_dtype,
                               long long ldo, int rows, int d, int nseg, float eps, const float* pos,
                               const float* freqs, int nfreq, rfb_stream_t stream) {
  if (!x || !w || !out || rows <= 0 || d % 128 || d > kMaxVec * 128 || ldx % 4 || ldo % 4 || nseg < 1)
    return RFB_ERR_ARG;
  if (out_dtype != RFB_BF16 && out_dtype != RFB_F16) return RFB_ERR_ARG;
  if (pos && (!freqs || nfreq < 1 || 9 * nfreq > 64)) return RFB_ERR_ARG;
  const int wpb = 8;
  if (in_period > 0 && rows % in_period) return RFB_ERR_ARG;
  const int src_rows = in_period > 0 ? in_period : rows;
  if (in_period == 0) {
    qknorm_rope_rows_kernel<<<dim3((rows + wpb - 1) / wpb, nseg), wpb * 32, 0, (cudaStream_t)stream>>>(
        x, ldx, in_period, w, out, ldo, rows, d, nseg, eps, pos, freqs, nfreq, out_dtype);
    RFB_LAUNCHED("qknorm_rope_rows_kernel");
  }
  qknorm_rope_kernel<<<src_rows, kRopeViews * 32, 0, (cudaStream_t)stream>>>(
      x, ldx, in_period, w, out, ldo, rows, d, nseg, eps, pos, freqs, nfreq, out_dtype);
  RFB_LAUNCHED("qknorm_rope_kernel");
}

extern "C" int rfb_qkv_post(const float* x, long long ldx, const float* w_qk, void* out_q, long long ldq,
                            void* const* kv_dst, int n_dst, int multicast, long long ldkv, long long row0, int rows,
                            int d, float eps, const float* pos, const float* freqs, int nfreq, int out_dtype,
                            rfb_stream_t stream) {
  if (!x || !w_qk || !out_q || !kv_dst || rows <= 0 || d % 128 || d > kMaxVec * 128 || ldx % 4 || ldx < 3LL * d ||
      ldq % 4 || ldq < d || ldkv % 4 || ldkv < 2LL * d || row0 < 0 || n_dst < 1 || n_dst > 8 || (multicast && n_dst != 1))
    return RFB_ERR_ARG;
  if (out_dtype != RFB_BF16 && out_dtype != RFB_F16) return RFB_ERR_ARG;
  if (pos && (!freqs || nfreq < 1 || 9 * nfreq > 64)) return RFB_ERR_ARG;
  KvDst dst{};
  for (int i = 0; i < n_dst; ++i) {
    if (!kv_dst[i] || (reinterpret_cast<uintptr_t>(kv_dst[i]) & 7)) return RFB_ERR_ALIGN;
    dst.p[i] = kv_dst[i];
  }
  const int wpb = 8;
  qkv_post_kernel<<<dim3((rows + wpb - 1) / wpb, 3), wpb * 32, 0, (cudaStream_t)stream>>>(
      x, ldx, w_qk, out_q, ldq, dst, n_dst, multicast, ldkv, row0, rows, d, eps, pos, freqs, nfreq, out_dtype);
  RFB_LAUNCHED("qkv_post_kernel");
}

extern "C" int rfb_transpose16(const void* in, long long ld_in, void* out, long long ld_out, int rows, int cols,
                               rfb_stream_t stream) {
  if (!in || !out || rows <= 0 || cols <= 0 || cols % 2 || ld_in % 2 || ld_out % 2 || ld_in < cols || ld_out < rows)
    return RFB_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 3) return RFB_ERR_ALIGN;
  transpose16_kernel<<<dim3((cols + 63) / 64, (rows + 63) / 64), 256, 0, (cudaStream_t)stream>>>(
      static_cast<const uint16_t*>(in), ld_in, static_cast<uint16_t*>(out), ld_out, rows, cols);
  RFB_LAUNCHED("transpose16_kernel");
}

extern "C" int rfb_qknorm_rope_table(const float* x, long long ldx, const float* w, void* out, int out_dtype,
                                     long long ldo, int rows, int d, int nseg, float eps, const float* cos_tab,
                                     const float* sin_tab, long long ldtab, rfb_stream_t stream) {
  if (out_dtype != RFB_BF16 && out_dtype != RFB_F16) return RFB_ERR_ARG;
  if (!x || !out || rows <= 0 || d % 128 || d > kMaxVec * 128 || ldx % 4 || ldo % 4 || nseg < 1) return RFB_ERR_ARG;
  if ((cos_tab == nullptr) != (sin_tab == nullptr) || (cos_tab && ldtab < 64)) return RFB_ERR_ARG;
  const int wpb = 8;
  qknorm_rope_rows_kernel<<<dim3((rows + wpb - 1) / wpb, nseg), wpb * 32, 0, (cudaStream_t)stream>>>(
      x, ldx, 0, w, out, ldo, rows, d, nseg, eps, nullptr, nullptr, 0, out_dtype, cos_tab, sin_tab, ldtab);
  RFB_LAUNCHED("qknorm_rope_rows_kernel");
}

extern "C" int rfb_token_assemble(const float* a, const float* wa, const float* b, const float* wb,
                                  const float* token, const float* prefix, int n_prefix, float* out,
                                  int rows_in, int rows_out, int batch, int d, rfb_stream_t stream) {
  if (!a || !wa || !token || !out || d % 128 || d > kMaxVec * 128 || (n_prefix > 0 && !prefix) || (b && !wb))
    return RFB_ERR_ARG;
  const int wpb = 8;
  const int total = batch * rows_out;
  token_assemble_kernel<<<(total + wpb - 1) / wpb, wpb * 32, 0, (cudaStream_t)stream>>>(
      a, wa, b, wb, token, prefix, n_prefix, out, rows_in, rows_out, batch, d, 1.1920928955078125e-07f);
  RFB_LAUNCHED("token_assemble_kernel");
}

extern "C" int rfb_texture_prep(const float* tex, void* out, long long n_tris, int channels, int texels,
                                int log_channels, rfb_stream_t stream) {
  if (!tex || !out || n_tris <= 0 || texels % 4) return RFB_ERR_ARG;
  const int per = channels * texels / 4;
  const long long n = n_tris * per;
  const int blocks = (int)((n + 255) / 256 < 148 * 16 ? (n + 255) / 256 : 148 * 16);
  texture_prep_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(tex, (uint16_t*)out, n, per,
                                                                (channels - log_channels) * texels / 4);
  RFB_LAUNCHED("texture_prep_kernel");
}

extern "C" int rfb_texture_const_prep(const float* tex, void* out, long long n_tris, int channels, int ld,
                                      int log_channels, rfb_stream_t stream) {
  if (!tex || !out || n_tris <= 0 || channels <= 0 || ld < channels || ld % 8 || log_channels > channels)
    return RFB_ERR_ARG;
  const long long total = n_tris * ld;
  texture_const_prep_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      tex, (uint16_t*)out, n_tris, channels, ld, log_channels);
  RFB_LAUNCHED("texture_const_prep_kernel");
}

extern "C" int rfb_vn_encode(const float* vn, void* out, int n, int nfreq, int ld, rfb_stream_t stream) {
  if (!vn || !out || n <= 0 || ld < 9 + 18 * nfreq) return RFB_ERR_ARG;
  const long long total = (long long)n * ld;
  vn_encode_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(vn, (uint16_t*)out, n,
                                                                                      nfreq, ld);
  RFB_LAUNCHED("vn_encode_kernel");
}

extern "C" int rfb_ray_tokens_canvas(const float* fov_deg, void* out, int n_views, int canvas_h, int canvas_w,
                                     int height, int width, int top, int left, rfb_stream_t stream) {
  if (!fov_deg || !out || n_views <= 0 || canvas_h <= 0 || canvas_w <= 0 || canvas_h % 8 || canvas_w % 8 ||
      height <= 0 || width <= 0 || top < 0 || left < 0 || height > canvas_h - top || width > canvas_w - left)
    return RFB_ERR_ARG;
  // principal point of the window in canvas pixels: integers + halves, exact in fp32 for any image size here
  const float cx = (float)left + (float)width * 0.5f, cy = (float)top + (float)height * 0.5f;
  const long long total = (long long)n_views * (canvas_h / 8) * (canvas_w / 8) * 192;
  ray_tokens_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      fov_deg, (uint16_t*)out, n_views, canvas_h, canvas_w, height, width, cx, cy);
  RFB_LAUNCHED("ray_tokens_kernel");
}

extern "C" int rfb_ray_tokens_intrinsics(const float* intr, void* out, int n_views, int canvas_h, int canvas_w,
                                         int height, int width, int top, int left, rfb_stream_t stream) {
  if (!intr || !out || n_views <= 0 || canvas_h <= 0 || canvas_w <= 0 || canvas_h % 8 || canvas_w % 8 ||
      height <= 0 || width <= 0 || top < 0 || left < 0 || height > canvas_h - top || width > canvas_w - left)
    return RFB_ERR_ARG;
  const long long total = (long long)n_views * (canvas_h / 8) * (canvas_w / 8) * 192;
  ray_tokens_intrinsics_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      intr, (uint16_t*)out, n_views, canvas_h, canvas_w, top, left);
  RFB_LAUNCHED("ray_tokens_intrinsics_kernel");
}

extern "C" int rfb_ray_tokens_lens(const float* intr, const float* dist, int lens, void* out, int n_views,
                                   int canvas_h, int canvas_w, int height, int width, int top, int left,
                                   rfb_stream_t stream) {
  if (!intr || !dist || !out || lens < 0 || lens > 1 || n_views <= 0 || canvas_h <= 0 || canvas_w <= 0 ||
      canvas_h % 8 || canvas_w % 8 || height <= 0 || width <= 0 || top < 0 || left < 0 || height > canvas_h - top ||
      width > canvas_w - left)
    return RFB_ERR_ARG;
  const long long total = (long long)n_views * canvas_h * canvas_w;  // one thread per pixel
  ray_tokens_lens_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      intr, dist, lens, (uint16_t*)out, n_views, canvas_h, canvas_w, top, left);
  RFB_LAUNCHED("ray_tokens_lens_kernel");
}

extern "C" int rfb_intrinsics_from_fov(const float* fov_deg, float* out, int n_views, int height, int width, int fit,
                                       rfb_stream_t stream) {
  if (!fov_deg || !out || n_views <= 0 || height <= 0 || width <= 0 || fit < 0 || fit > 2) return RFB_ERR_ARG;
  intrinsics_from_fov_kernel<<<(n_views + 127) / 128, 128, 0, (cudaStream_t)stream>>>(fov_deg, out, n_views, height,
                                                                                      width, fit);
  RFB_LAUNCHED("intrinsics_from_fov_kernel");
}

extern "C" int rfb_ray_tokens_hw(const float* fov_deg, void* out, int n_views, int height, int width,
                                 rfb_stream_t stream) {
  return rfb_ray_tokens_canvas(fov_deg, out, n_views, height, width, height, width, 0, 0, stream);
}

extern "C" int rfb_ray_tokens(const float* fov_deg, void* out, int n_views, int resolution,
                              rfb_stream_t stream) {
  return rfb_ray_tokens_hw(fov_deg, out, n_views, resolution, resolution, stream);
}

extern "C" int rfb_ray_map_hw(const float* c2w, const float* fov_rad, float* rays_d, int n_views, int height, int width,
                              rfb_stream_t stream) {
  if (!c2w || !fov_rad || !rays_d || n_views <= 0 || height <= 0 || width <= 0) return RFB_ERR_ARG;
  const long long total = (long long)n_views * height * width;
  ray_map_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(c2w, fov_rad, rays_d, n_views,
                                                                                    height, width);
  RFB_LAUNCHED("ray_map_kernel");
}

extern "C" int rfb_ray_map(const float* c2w, const float* fov_rad, float* rays_d, int n_views, int resolution,
                           rfb_stream_t stream) {
  return rfb_ray_map_hw(c2w, fov_rad, rays_d, n_views, resolution, resolution, stream);
}

extern "C" int rfb_ray_map_tokens_hw(const float* rays_d, void* out, int n_views, int height, int width,
                                     rfb_stream_t stream) {
  if (!rays_d || !out || n_views <= 0 || height <= 0 || width <= 0 || height % 8 || width % 8) return RFB_ERR_ARG;
  const long long total = (long long)n_views * (height / 8) * (width / 8) * 192;
  ray_map_tokens_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rays_d, (uint16_t*)out,
                                                                                           n_views, height, width);
  RFB_LAUNCHED("ray_map_tokens_kernel");
}

extern "C" int rfb_ray_map_tokens(const float* rays_d, void* out, int n_views, int resolution, rfb_stream_t stream) {
  return rfb_ray_map_tokens_hw(rays_d, out, n_views, resolution, resolution, stream);
}

extern "C" int rfb_positions(const float* tri, const uint8_t* mask, const float* c2w, float* pos, int n,
                             int n_reg, int rows_out, int n_views, rfb_stream_t stream) {
  if (!tri || !mask || !pos || n <= 0 || n_reg > 32 || rows_out < n + n_reg || n_views <= 0) return RFB_ERR_ARG;
  positions_kernel<<<n_views, 256, 0, (cudaStream_t)stream>>>(tri, mask, c2w, pos, n, n_reg, rows_out);
  RFB_LAUNCHED("positions_kernel");
}

extern "C" int rfb_pack_mask(const uint8_t* mask, uint32_t* bits, int n, int n_prefix, int words, int batch,
                             rfb_stream_t stream) {
  if (!mask || !bits || words % 4 || words * 32 < n + n_prefix) return RFB_ERR_ARG;
  const int total = batch * words;
  pack_mask_kernel<<<(total + 127) / 128, 128, 0, (cudaStream_t)stream>>>(mask, bits, n, n_prefix, words, batch);
  RFB_LAUNCHED("pack_mask_kernel");
}

extern "C" int rfb_cast(const float* x, void* out, int out_dtype, long long n, rfb_stream_t stream) {
  if (!x || !out || n % 4 || (out_dtype != RFB_BF16 && out_dtype != RFB_F16)) return RFB_ERR_ARG;
  const long long nv = n / 4;
  const int blocks = (int)((nv + 255) / 256 < 148 * 16 ? (nv + 255) / 256 : 148 * 16);
  cast_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, out, out_dtype, nv);
  RFB_LAUNCHED("cast_kernel");
}
