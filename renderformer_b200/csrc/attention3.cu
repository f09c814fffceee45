// Dense flash attention, third generation: ONE 128-query tile per CTA, BOTH products take their A
// operand from tensor memory.
//
//   warp 0 = TMA producer (K / V^T tiles, 3-stage rings), warp 1 = tcgen05.mma issuer,
//   warps 2..5 = softmax + epilogue (one thread per query row).
//
// Why: a 128 x 128 x 16 UMMA with both operands in shared memory needs 8 KB per 64 clk = the whole
// 128 B/clk of the SM's shared-memory read bandwidth, so S = Q K^T could never run at the tensor
// rate in the two-tile kernel (attention2.cu).  Here the softmax warps copy the Q tile into TMEM once
// (64 columns of packed bf16 pairs) and Q K^T is issued with a TMEM A operand like P V already was:
// only K and V stream through shared memory (64 B/clk).  TMEM map: S0 [0,128) S1 [128,256)
// O [256,384) Q [384,448).  S is double-buffered, so Q K_{j+1}^T runs while the softmax of tile j is
// exponentiating; P_j overwrites the first 64 columns of S_{j&1}.  One tile per CTA also gives
// Nq/128 * H * B CTAs (1024 for 4 views: 6.9 waves instead of 3.46 of the two-tile kernel).
//
// O rescale: Q K_{j+1}^T is issued before P_{j-1} V_{j-1}... so "S_j ready" does not imply that the
// previous P V retired; the (rare) rescale waits on an explicit pv_done barrier first.
//
// Used for mode 0 (encoder self-attention, decoder cross-attention, key-padding mask, fused query
// RMSNorm), like attn2_tc_kernel (attention2.cu), which must give bit-identical results: the softmax
// steps, the epilogues and the key-tile range of a CTA are shared with it in attention_common.cuh;
// this file holds the Q copy into TMEM, the TMA producer, the MMA issuer and the barrier protocol
// around the softmax.  Reference call sites: include/rfb200.h.
#include "attention_common.cuh"

namespace rfb {

constexpr int kStg3 = 3;
constexpr int kAttn3Threads = 64 + 128;
constexpr uint32_t kAttn3Smem = kAttnTile * 2 * kStg3 + 1024 + 256;

template <bool F16>
__global__ void __launch_bounds__(kAttn3Threads, 1)
    attn3_tc_kernel(const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                    const DenseAttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* sK = smem;                       // kStg3 tiles
  uint8_t* sV = sK + kStg3 * kAttnTile;     // kStg3 tiles
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + kStg3 * kAttnTile);
  uint64_t* k_full = bars;              // kStg3
  uint64_t* k_empty = k_full + kStg3;   // kStg3
  uint64_t* v_full = k_empty + kStg3;   // kStg3
  uint64_t* v_empty = v_full + kStg3;   // kStg3
  uint64_t* s_full = v_empty + kStg3;   // 2
  uint64_t* p_full = s_full + 2;        // 2 (4 softmax warps each)
  uint64_t* pv_done = p_full + 2;       // 1
  uint64_t* q_ready = pv_done + 1;      // 1 (4 softmax warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(q_ready + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int h = blockIdx.y;
  const DenseTiles tiles = dense_tiles(p);
  const int split = tiles.split, j_begin = tiles.j_begin, n_tiles = tiles.n_tiles, tail_local = tiles.tail_local;
  const int b = blockIdx.z - split * p.B;
  const int q0 = blockIdx.x * 128;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kStg3; ++i) {
      mbar_init(&k_full[i], 1), mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1), mbar_init(&v_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) mbar_init(&s_full[i], 1), mbar_init(&p_full[i], 4);
    mbar_init(pv_done, 1);
    mbar_init(q_ready, 4);
    fence_mbar_init();
    tma_prefetch_desc(&tmK), tma_prefetch_desc(&tmV);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tO = tmem_base + 256, tQ = tmem_base + 384;
  const int kb = p.k_batched ? b : 0;
  const int vb = p.v_batched ? b : 0;

  if (warp == 0) {
    if (lane == 0) {
      for (int j = 0; j < n_tiles; ++j) {
        const int s = j % kStg3;
        const uint32_t ph = (j / kStg3) & 1;
        mbar_wait(&k_empty[s], ph ^ 1);
        mbar_expect_tx(&k_full[s], kAttnTile);
        const int key0 = (j_begin + j) * 128;
        tma_load_3d(sK + s * kAttnTile, &tmK, &k_full[s], h * 128, key0, kb);
        tma_load_3d(sK + s * kAttnTile + kAttnHalf, &tmK, &k_full[s], h * 128 + 64, key0, kb);
        mbar_wait(&v_empty[s], ph ^ 1);
        mbar_expect_tx(&v_full[s], kAttnTile);
        tma_load_3d(sV + s * kAttnTile, &tmV, &v_full[s], key0, h * 128, vb);
        tma_load_3d(sV + s * kAttnTile + kAttnHalf, &tmV, &v_full[s], key0 + 64, h * 128, vb);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_f16(F16 ? 0u : 1u, 128, 128);
      const uint32_t idesc_tail = umma_idesc_f16(F16 ? 0u : 1u, 128, 32);
      auto issue_qk = [&](int j) {  // S[j&1] = Q K_j^T, A operand = Q in TMEM (packed bf16 pairs)
        const int s = j % kStg3;
        mbar_wait(&k_full[s], (j / kStg3) & 1);
        tc_fence_after();
        const uint64_t bd = umma_desc_sw128(smem_u32(sK + s * kAttnTile));
        const uint32_t id = (j == tail_local) ? idesc_tail : idesc;
#pragma unroll
        for (int k = 0; k < 8; ++k) umma_f16_ts(tmem_base + (j & 1) * 128, tQ + k * 8, bd + sw128_kstep(k), id, k != 0);
        umma_commit(&k_empty[s]);
        umma_commit(&s_full[j & 1]);
      };
      auto issue_pv = [&](int j) {  // O += P_j V_j, A operand = P in S[j&1] columns [0,64)
        const int s = j % kStg3;
        mbar_wait(&v_full[s], (j / kStg3) & 1);
        mbar_wait(&p_full[j & 1], (j >> 1) & 1);
        tc_fence_after();
        const uint64_t bd = umma_desc_sw128(smem_u32(sV + s * kAttnTile));
        const int ksteps = (j == tail_local) ? 2 : 8;  // short tail: 32 keys = two K = 16 steps
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k < ksteps) umma_f16_ts(tO, tmem_base + (j & 1) * 128 + k * 8, bd + sw128_kstep(k), idesc, (j | k) != 0);
        umma_commit(&v_empty[s]);
        umma_commit(pv_done);
      };
      mbar_wait(q_ready, 0);
      tc_fence_after();
      issue_qk(0);
      for (int j = 0; j < n_tiles; ++j) {
        if (j + 1 < n_tiles) issue_qk(j + 1);
        issue_pv(j);
      }
    }
  } else {
    // ------------------------------ softmax warps ------------------------------
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    const int qrow = q0 + r;
    const bool row_ok = qrow < p.Nq;

    // Q row -> TMEM (64 packed columns); rows past Nq are zero
    {
      const uint16_t* qsrc = p.Q + static_cast<long long>(b) * p.q_batch_stride + static_cast<long long>(qrow) * p.ldq + h * 128;
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t w[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          uint4 u = make_uint4(0u, 0u, 0u, 0u);
          if (row_ok) u = __ldg(reinterpret_cast<const uint4*>(qsrc + half * 64 + i * 8));
          w[i * 4] = u.x, w[i * 4 + 1] = u.y, w[i * 4 + 2] = u.z, w[i * 4 + 3] = u.w;
        }
        tmem_st32(tQ + lane_addr + half * 32, w);
      }
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(q_ready);
    }

    const float sl2 = dense_scale_log2(p, b, qrow);
    float m_run = -INFINITY, l_run = 0.f;
    const uint32_t tOl = tO + lane_addr;

    for (int j = 0; j < n_tiles; ++j) {
      uint32_t mw[4];
      key_mask_words(p, b, j_begin + j, mw);
      const uint32_t tS = tmem_base + (j & 1) * 128 + lane_addr;
      mbar_wait(&s_full[j & 1], (j >> 1) & 1);
      tc_fence_after();
      const int nc = (j == tail_local) ? 1 : 4;  // 32-column chunks of S that exist (short tail: one)
      uint32_t v[4][32];
      const SoftmaxMax sm = softmax_max(tS, nc, mw, m_run, sl2, v);
      if (j > 0 && __any_sync(0xffffffffu, sm.alpha != 1.0f)) {
        mbar_wait(pv_done, (j - 1) & 1);  // P_{j-1} V_{j-1} retired: O is stable
        tc_fence_after();
        rescale_o(tOl, sm.alpha);
      }
      l_run = fmaf(l_run, sm.alpha, softmax_exp<F16>(v, tS, nc, sl2, sm.neg_ms));
      m_run = sm.m_new;

      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      // A parity wait can only tell the current phase of a barrier from the one before it.  S is double-buffered,
      // so a fast warp may get here a whole tile ahead of the slowest one: P_{j-1} V_{j-1} is then not even issued
      // and pv_done still sits in phase j-1 -- the epilogue's wait for phase j (same parity as phase j-2, which HAS
      // completed) would fall through and read O two products early.  Seeing phase j-1 complete first makes the
      // epilogue's wait unambiguous (S_j ready => phase j-2 complete, and phase j cannot start before this warp's
      // arrive below).
      if (j == n_tiles - 1 && j > 0) mbar_wait(pv_done, (j - 1) & 1);
      if (lane == 0) mbar_arrive(&p_full[j & 1]);
    }

    mbar_wait(pv_done, (n_tiles - 1) & 1);
    tc_fence_after();
    dense_store_row<F16>(p, tOl, split, b, h, qrow, m_run, l_run, sl2);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

int launch_attention3(const CUtensorMap&, const CUtensorMap& tmK, const CUtensorMap& tmV, const rfb_attn_args* a,
                      const DenseAttnParams& p, cudaStream_t stream) {
  if (a->ldq % 8 || (reinterpret_cast<uintptr_t>(a->Q) & 15) || (a->B > 1 && a->q_batch_stride % 8)) return RFB_ERR_ALIGN;
  const bool f16 = a->dtype == RFB_F16;
  static PerDeviceFlag attr_flags[2];
  const dim3 grid((a->Nq + 127) / 128, a->H, a->B * p.n_splits());
  return launch_attn_kernel(f16 ? attn3_tc_kernel<true> : attn3_tc_kernel<false>, "attn3_tc_kernel",
                            attr_flags[f16].get(), kAttn3Smem, grid, kAttn3Threads, stream, tmK, tmV, p);
}

}  // namespace rfb
