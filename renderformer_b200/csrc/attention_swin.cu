// Shifted-window self-attention among ray tokens (rfb_attention mode 1), one CTA per 128-token
// tile (two 64-token windows, window-major token order), looping over ALL heads of that tile.
//
//   warp 0 = TMA producer, warp 1 = tcgen05.mma issuer, warps 2..5 = softmax + epilogue
//   (one thread per query row).
//
// A window only attends to itself, so per (tile, head) there is exactly one 128 x 128 S = Q K^T and
// one O = P V: the work per head is tiny (8.4 MFLOP) and the kernel is bound by how fast Q, K, V
// tiles stream in and O streams out.  Hence the head loop: the three operand tiles of head h+1 are
// in flight (2-stage smem ring, 96 KB per stage) while head h is computed, S and O are
// double-buffered in TMEM so QK(h+1) overlaps softmax(h) and the O epilogue of head h-1 overlaps
// PV(h), and the TMEM allocation / barrier set-up is paid once per tile instead of once per
// (tile, head).  P is written back over S as packed bf16 (tcgen05.mma with a TMEM A operand).
// Each softmax warp only touches the 64 keys of its own window (the other window's logits are
// masked by construction); shifted layers add the region mask as a per-token region id.
//
// Replaces the per-window SDPA of SwinSelfAttention.forward, layers/attention.py:349-358, incl.
// window_partition / get_swin_attn_mask (:205-271).
#include "attention_common.cuh"

namespace rfb {

struct SwinParams {
  int N, H;
  int k_batched, v_batched;
  const uint8_t* group_id;
  int group_period;
  void* O;
  long long ldo, o_batch_stride;
  float scale_log2;
  const float* q_sumsq;
  const float* k_sumsq;
  int sumsq_ld, sumsq_parts;
  float inv_norm_dim, norm_eps;
};

constexpr uint32_t kSwStage = 3 * kAttnTile;  // Q, K, V^T of one head
constexpr int kSwThreads = 64 + 128;
constexpr uint32_t kSwSmem = 2 * kSwStage + 1024 + 1024;

template <bool F16>
__global__ void __launch_bounds__(kSwThreads, 1)
    attn_swin_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                     const __grid_constant__ CUtensorMap tmV, const SwinParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * kSwStage);
  uint64_t* full = bars;          // 2: Q, K, V of a stage have landed
  uint64_t* empty = full + 2;     // 2: P.V of that stage retired
  uint64_t* s_full = empty + 2;   // 2: S buffer written
  uint64_t* p_full = s_full + 2;  // 2: P written over S by the 4 softmax warps
  uint64_t* o_full = p_full + 2;  // 2: O buffer complete
  uint64_t* o_empty = o_full + 2; // 2: O buffer drained by the 4 epilogue warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_empty + 2);
  uint8_t* s_gid = reinterpret_cast<uint8_t*>(tmem_slot + 2);  // 128 region ids
  float* s_rk = reinterpret_cast<float*>(s_gid + 128);         // 128 per-key 1/rms factors

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int q0 = blockIdx.x * 128;

  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&full[i], 1), mbar_init(&empty[i], 1), mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4), mbar_init(&o_full[i], 1), mbar_init(&o_empty[i], 4);
    }
    fence_mbar_init();
    tma_prefetch_desc(&tmQ), tma_prefetch_desc(&tmK), tma_prefetch_desc(&tmV);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  if (threadIdx.x >= 64) {
    const int i = threadIdx.x - 64;
    s_gid[i] = p.group_id[(q0 + i) % p.group_period];
    float rk = 1.0f;
    if (p.k_sumsq && q0 + i < p.N)
      rk = rms_factor(p.k_sumsq, static_cast<long long>(b) * p.N + q0 + i, p.sumsq_ld, p.sumsq_parts, p.inv_norm_dim,
                      p.norm_eps);
    s_rk[i] = rk;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;  // S0 [0,128) S1 [128,256) O0 [256,384) O1 [384,512)
  const int H = p.H;
  const int kb = p.k_batched ? b : 0, vb = p.v_batched ? b : 0;

  if (warp == 0) {
    if (lane == 0) {
      for (int h = 0; h < H; ++h) {
        const int s = h & 1;
        uint8_t* st = smem + s * kSwStage;
        mbar_wait(&empty[s], ((h >> 1) & 1) ^ 1);
        mbar_expect_tx(&full[s], kSwStage);
        tma_load_3d(st, &tmQ, &full[s], h * 128, q0, b);
        tma_load_3d(st + kAttnHalf, &tmQ, &full[s], h * 128 + 64, q0, b);
        tma_load_3d(st + kAttnTile, &tmK, &full[s], h * 128, q0, kb);
        tma_load_3d(st + kAttnTile + kAttnHalf, &tmK, &full[s], h * 128 + 64, q0, kb);
        tma_load_3d(st + 2 * kAttnTile, &tmV, &full[s], q0, h * 128, vb);
        tma_load_3d(st + 2 * kAttnTile + kAttnHalf, &tmV, &full[s], q0 + 64, h * 128, vb);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_f16(F16 ? 0u : 1u, 128, 128);
      auto issue_qk = [&](int h) {  // S[h&1] = Q_h K_h^T  (the buffer's previous P was consumed by PV(h-2),
        const int s = h & 1;        //  issued earlier: tcgen05 operations of one thread retire in order)
        mbar_wait(&full[s], (h >> 1) & 1);
        tc_fence_after();
        const uint64_t ad = umma_desc_sw128(smem_u32(smem + s * kSwStage));
        const uint64_t bd = umma_desc_sw128(smem_u32(smem + s * kSwStage + kAttnTile));
#pragma unroll
        for (int k = 0; k < 8; ++k) umma_f16(tmem_base + s * 128, ad + sw128_kstep(k), bd + sw128_kstep(k), idesc, k != 0);
        umma_commit(&s_full[s]);
      };
      auto issue_pv = [&](int h) {  // O[h&1] = P_h V_h  (A operand: packed bf16 P in S[h&1] columns [0,64))
        const int s = h & 1;
        mbar_wait(&p_full[s], (h >> 1) & 1);
        mbar_wait(&o_empty[s], ((h >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint64_t bd = umma_desc_sw128(smem_u32(smem + s * kSwStage + 2 * kAttnTile));
#pragma unroll
        for (int k = 0; k < 8; ++k)
          umma_f16_ts(tmem_base + 256 + s * 128, tmem_base + s * 128 + k * 8, bd + sw128_kstep(k), idesc, k != 0);
        umma_commit(&o_full[s]);
        umma_commit(&empty[s]);
      };
      issue_qk(0);
      for (int h = 0; h < H; ++h) {
        if (h + 1 < H) issue_qk(h + 1);
        issue_pv(h);
      }
    }
  } else {
    // ------------------------------ softmax + epilogue warps ------------------------------
    const int q = warp & 3;  // TMEM lane quarter
    const int r = q * 32 + lane;
    const int half = r >> 6;  // window inside the tile; the warp's rows all share it
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    const bool row_ok = q0 + r < p.N;
    float sl2 = p.scale_log2;
    if (p.q_sumsq && row_ok)
      sl2 *= rms_factor(p.q_sumsq, static_cast<long long>(b) * p.N + q0 + r, p.sumsq_ld, p.sumsq_parts, p.inv_norm_dim,
                        p.norm_eps);
    // keys of the own window this row may attend: same region id, inside the sequence
    uint32_t mw[2];
    {
      const uint8_t g = s_gid[r];
#pragma unroll
      for (int w = 0; w < 2; ++w) {
        uint32_t bits = 0;
        for (int i = 0; i < 32; ++i) {
          const int key = half * 64 + w * 32 + i;
          bits |= ((s_gid[key] == g && q0 + key < p.N) ? 1u : 0u) << i;
        }
        mw[w] = bits;
      }
    }
    const bool all_valid = (mw[0] & mw[1]) == 0xffffffffu;
    float rk[64];
    const bool k_scaled = p.k_sumsq != nullptr;
    if (k_scaled) {
#pragma unroll
      for (int i = 0; i < 64; ++i) rk[i] = s_rk[half * 64 + i];
    }
    uint16_t* obase = static_cast<uint16_t*>(p.O) + static_cast<long long>(b) * p.o_batch_stride +
                      static_cast<long long>(q0 + r) * p.ldo;
    float inv_l_prev = 0.f;

    auto epilogue = [&](int g, float inv_l) {  // O[g&1] / l -> bf16 -> global
      const int s = g & 1;
      mbar_wait(&o_full[s], (g >> 1) & 1);
      tc_fence_after();
      store_o_row<F16>(tmem_base + 256 + s * 128 + lane_addr, obase + g * 128, row_ok, inv_l);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&o_empty[s]);
    };

    for (int h = 0; h < H; ++h) {
      const int s = h & 1;
      const uint32_t tS = tmem_base + s * 128 + lane_addr;
      mbar_wait(&s_full[s], (h >> 1) & 1);
      tc_fence_after();
      uint32_t v[2][32];
      tmem_ld32(tS + half * 64, v[0]);
      tmem_ld32(tS + half * 64 + 32, v[1]);
      tmem_wait_ld();
      if (k_scaled) {
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
          for (int i = 0; i < 32; ++i) v[c][i] = __float_as_uint(__uint_as_float(v[c][i]) * rk[c * 32 + i]);
      }
      if (!all_valid) {
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
          for (int i = 0; i < 32; ++i)
            if (!((mw[c] >> i) & 1u)) v[c][i] = 0xff800000u;  // -inf
      }
      float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
      for (int c = 0; c < 2; ++c)
#pragma unroll
        for (int i = 0; i < 32; ++i) mx4[i & 3] = fmaxf(mx4[i & 3], __uint_as_float(v[c][i]));
      const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      const float m_use = (mx == -INFINITY) ? 0.f : mx;
      const uint64_t sl2_2 = pack2f(sl2, sl2), nms_2 = pack2f(-m_use * sl2, -m_use * sl2);
      uint64_t rs2[2] = {0ull, 0ull};
      uint32_t zero[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) zero[i] = 0u;
      tmem_st16(tS + (half ^ 1) * 32, zero);
      tmem_st16(tS + (half ^ 1) * 32 + 16, zero);
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const uint64_t t2 =
              ffma2(pack2f(__uint_as_float(v[c][2 * i]), __uint_as_float(v[c][2 * i + 1])), sl2_2, nms_2);
          const float p0 = ex2_f(lo2f(t2)), p1 = ex2_f(hi2f(t2));
          rs2[i & 1] = fadd2(rs2[i & 1], pack2f(p0, p1));
          pk[i] = pack16<F16>(p0, p1);
        }
        tmem_st16(tS + half * 32 + c * 16, pk);
      }
      const uint64_t rsum = fadd2(rs2[0], rs2[1]);
      const float l = lo2f(rsum) + hi2f(rsum);
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[s]);
      if (h > 0) epilogue(h - 1, inv_l_prev);
      inv_l_prev = l > 0.f ? 1.0f / l : 0.f;
    }
    epilogue(H - 1, inv_l_prev);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// called by rfb_attention (attention.cu) for mode 1; Q/K maps have box {64,128,1}, V^T map {64,128,1}
int launch_attention_swin(const CUtensorMap& tmQ, const CUtensorMap& tmK, const CUtensorMap& tmV,
                          const rfb_attn_args* a, int k_batched, int v_batched, cudaStream_t stream) {
  SwinParams p{};
  p.N = a->Nq, p.H = a->H;
  p.k_batched = k_batched, p.v_batched = v_batched;
  p.group_id = a->group_id, p.group_period = a->group_period;
  p.O = a->O, p.ldo = a->ldo, p.o_batch_stride = a->o_batch_stride;
  p.scale_log2 = a->scale * 1.4426950408889634f;
  p.q_sumsq = a->q_sumsq, p.k_sumsq = a->k_sumsq;
  p.sumsq_ld = a->sumsq_ld > 0 ? a->sumsq_ld : 1, p.sumsq_parts = a->sumsq_parts > 0 ? a->sumsq_parts : 1;
  p.inv_norm_dim = a->norm_dim > 0 ? 1.0f / (float)a->norm_dim : 0.f, p.norm_eps = a->norm_eps;
  const bool f16 = a->dtype == RFB_F16;
  static PerDeviceFlag attr_flags[2];
  const dim3 grid((a->Nq + 127) / 128, a->B);
  return launch_attn_kernel(f16 ? attn_swin_kernel<true> : attn_swin_kernel<false>, "attn_swin_kernel",
                            attr_flags[f16].get(), kSwSmem, grid, kSwThreads, stream, tmQ, tmK, tmV, p);
}

}  // namespace rfb
