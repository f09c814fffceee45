// Dense flash attention, second generation: two 128-query tiles per CTA sharing one K/V stream,
// P kept in tensor memory.
//
//   warpgroup 0: warp 0 = TMA producer, warp 1 = tcgen05.mma issuer, warps 2-3 idle (they exist so
//   that setmaxnreg can hand the group's registers to the softmax warpgroups);
//   warpgroup 1 (warps 4-7) = softmax of query tile A, warpgroup 2 (warps 8-11) = softmax of query
//   tile B, one thread per query row.
//
// The softmax is the co-critical resource next to the tensor pipe (128 x 128 exponentials per
// 2 x 4.2 MFLOP tile pair: the 16/clk/SM MUFU rate equals the tensor time), so its inner loop uses
// packed fp32x2 arithmetic (FFMA2 / FADD2) and evaluates a quarter of the exponentials with a
// degree-3 polynomial on the FMA pipe (Cody-Waite split, exponent inserted with an integer add)
// instead of MUFU.EX2.
//
// TMEM map (512 columns): S_A [0,128)  S_B [128,256)  O_A [256,384)  O_B [384,512).
// After the softmax has pulled its whole S row into registers it writes P (bf16 pairs) back into
// the first 64 columns of the same S region; the P.V product then takes its A operand straight
// from TMEM (tcgen05.mma with a TMEM A descriptor), so P never touches shared memory and the
// only smem traffic of the second GEMM is V.  The MMA issue order
//     PV_A(j), QK_A(j+1), PV_B(j), QK_B(j+1)
// lets the tensor pipe work on one query tile while the other tile's softmax runs.  Because
// tcgen05 operations of one thread complete in order, "S_t(j) is ready" already implies
// "PV_t(j-1) is done", so the (rare) O rescale needs no extra barrier.
//
// Used for mode 0 (encoder self-attention, decoder cross-attention, key-padding mask, fused query
// RMSNorm), like attn3_tc_kernel (attention3.cu), which must give bit-identical results: the softmax
// steps, the epilogues and the key-tile range of a CTA are shared with it in attention_common.cuh;
// this file holds the TMA producer, the MMA issuer and the barrier protocol around the softmax.
// Reference call sites: include/rfb200.h.
#include "attention_common.cuh"

namespace rfb {

constexpr int kStg = 2;
constexpr int kAttn2Threads = 3 * 128;
constexpr int kRegsWg0 = 56, kRegsSoftmax = 224;  // setmaxnreg targets (128*56 + 256*224 = 384*168)
constexpr uint32_t kAttn2Smem = kAttnTile * (2 + 2 * kStg) + 1024 + 256;

template <bool F16>
__global__ void __launch_bounds__(kAttn2Threads, 1)
    attn2_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                    const __grid_constant__ CUtensorMap tmV, const DenseAttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* sQ = smem;                 // 2 tiles
  uint8_t* sK = sQ + 2 * kAttnTile;     // kStg tiles
  uint8_t* sV = sK + kStg * kAttnTile;  // kStg tiles
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + kStg * kAttnTile);
  uint64_t* q_full = bars;            // 1
  uint64_t* k_full = q_full + 1;      // kStg
  uint64_t* k_empty = k_full + kStg;  // kStg
  uint64_t* v_full = k_empty + kStg;  // kStg
  uint64_t* v_empty = v_full + kStg;  // kStg
  uint64_t* s_full = v_empty + kStg;  // 2 (per query tile)
  uint64_t* p_full = s_full + 2;      // 2
  uint64_t* o_done = p_full + 2;      // 2
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_done + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int h = blockIdx.y;
  const DenseTiles tiles = dense_tiles(p);
  const int split = tiles.split, j_begin = tiles.j_begin, n_tiles = tiles.n_tiles, tail_local = tiles.tail_local;
  const int b = blockIdx.z - split * p.B;
  const int q0 = blockIdx.x * 256;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int i = 0; i < kStg; ++i) {
      mbar_init(&k_full[i], 1), mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1), mbar_init(&v_empty[i], 1);
    }
    for (int t = 0; t < 2; ++t) mbar_init(&s_full[t], 1), mbar_init(&p_full[t], 4), mbar_init(&o_done[t], 1);
    fence_mbar_init();
    tma_prefetch_desc(&tmQ), tma_prefetch_desc(&tmK), tma_prefetch_desc(&tmV);
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int kb = p.k_batched ? b : 0;
  const int vb = p.v_batched ? b : 0;

  if (warp == 0) {
    setmaxnreg_dec<kRegsWg0>();
    if (lane == 0) {
      mbar_expect_tx(q_full, 2 * kAttnTile);
      for (int t = 0; t < 2; ++t) {
        tma_load_3d(sQ + t * kAttnTile, &tmQ, q_full, h * 128, q0 + t * 128, b);
        tma_load_3d(sQ + t * kAttnTile + kAttnHalf, &tmQ, q_full, h * 128 + 64, q0 + t * 128, b);
      }
      for (int j = 0; j < n_tiles; ++j) {
        const int s = j % kStg;
        const uint32_t ph = (j / kStg) & 1;
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
    setmaxnreg_dec<kRegsWg0>();
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_f16(F16 ? 0u : 1u, 128, 128);
      const uint32_t idesc_tail = umma_idesc_f16(F16 ? 0u : 1u, 128, 32);
      auto issue_qk = [&](int t, int j) {  // S_t = Q_t K_j^T
        const int s = j % kStg;
        const uint64_t ad = umma_desc_sw128(smem_u32(sQ + t * kAttnTile));
        const uint64_t bd = umma_desc_sw128(smem_u32(sK + s * kAttnTile));
        const uint32_t id = (j == tail_local) ? idesc_tail : idesc;
#pragma unroll
        for (int k = 0; k < 8; ++k) umma_f16(tmem_base + t * 128, ad + sw128_kstep(k), bd + sw128_kstep(k), id, k != 0);
        umma_commit(&s_full[t]);
      };
      auto issue_pv = [&](int t, int j) {  // O_t += P_t V_j   (A operand from TMEM)
        const int s = j % kStg;
        mbar_wait(&p_full[t], j & 1);
        tc_fence_after();
        const uint64_t bd = umma_desc_sw128(smem_u32(sV + s * kAttnTile));
        const int ksteps = (j == tail_local) ? 2 : 8;  // short tail: 32 keys = two K = 16 steps
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if (k < ksteps)
            umma_f16_ts(tmem_base + 256 + t * 128, tmem_base + t * 128 + k * 8, bd + sw128_kstep(k), idesc, (j | k) != 0);
      };
      mbar_wait(q_full, 0);
      mbar_wait(&k_full[0], 0);
      tc_fence_after();
      issue_qk(0, 0);
      issue_qk(1, 0);
      umma_commit(&k_empty[0]);
      for (int j = 0; j < n_tiles; ++j) {
        const int s = j % kStg;
        const bool more = j + 1 < n_tiles;
        const int s1 = (j + 1) % kStg;
        mbar_wait(&v_full[s], (j / kStg) & 1);
        issue_pv(0, j);
        if (more) {
          mbar_wait(&k_full[s1], ((j + 1) / kStg) & 1);
          tc_fence_after();
          issue_qk(0, j + 1);
        }
        issue_pv(1, j);
        umma_commit(&v_empty[s]);
        if (more) {
          issue_qk(1, j + 1);
          umma_commit(&k_empty[s1]);
        }
      }
      umma_commit(&o_done[0]);
      umma_commit(&o_done[1]);
    }
  } else if (warp < 4) {
    setmaxnreg_dec<kRegsWg0>();  // idle warps of warpgroup 0
  } else {
    // ------------------------------ softmax warps ------------------------------
    setmaxnreg_inc<kRegsSoftmax>();
    const int t = (warp - 4) >> 2;  // query tile of this warp group
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t tS = tmem_base + t * 128 + lane_addr;
    const uint32_t tO = tmem_base + 256 + t * 128 + lane_addr;
    const int qrow = q0 + t * 128 + r;
    const float sl2 = dense_scale_log2(p, b, qrow);
    float m_run = -INFINITY, l_run = 0.f;

    for (int j = 0; j < n_tiles; ++j) {
      uint32_t mw[4];
      key_mask_words(p, b, j_begin + j, mw);
      mbar_wait(&s_full[t], j & 1);
      tc_fence_after();
      const int nc = (j == tail_local) ? 1 : 4;  // 32-column chunks of S that exist (short tail: one)
      uint32_t v[4][32];
      const SoftmaxMax sm = softmax_max(tS, nc, mw, m_run, sl2, v);
      // S_t(j) ready implies PV_t(j-1) retired (in-order tcgen05 pipe): O_t may be rescaled now
      if (j > 0 && __any_sync(0xffffffffu, sm.alpha != 1.0f)) rescale_o(tO, sm.alpha);
      l_run = fmaf(l_run, sm.alpha, softmax_exp<F16>(v, tS, nc, sl2, sm.neg_ms));
      m_run = sm.m_new;

      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[t]);
    }

    mbar_wait(&o_done[t], 0);
    tc_fence_after();
    dense_store_row<F16>(p, tO, split, b, h, qrow, m_run, l_run, sl2);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

int launch_attention2(const CUtensorMap& tmQ, const CUtensorMap& tmK, const CUtensorMap& tmV,
                      const rfb_attn_args* a, const DenseAttnParams& p, cudaStream_t stream) {
  const bool f16 = a->dtype == RFB_F16;
  auto kern = f16 ? attn2_tc_kernel<true> : attn2_tc_kernel<false>;
  static PerDeviceFlag attr_flags[2];
  bool& attr_set = attr_flags[f16].get();
  if (!attr_set) {
    // setmaxnreg moves registers inside the CTA's launch allocation only: the softmax warpgroups'
    // request must be covered by what warpgroup 0 gives back, or the kernel would wait forever
    cudaFuncAttributes fa;
    if (cudaFuncGetAttributes(&fa, kern) != cudaSuccess) return RFB_ERR_LAUNCH;
    if (128 * kRegsWg0 + 256 * kRegsSoftmax > kAttn2Threads * fa.numRegs) {
      fprintf(stderr, "rfb: attn2_tc_kernel compiled with %d registers/thread; setmaxnreg split %d/%d does not fit\n",
              fa.numRegs, kRegsWg0, kRegsSoftmax);
      return RFB_ERR_LAUNCH;
    }
  }
  const dim3 grid((a->Nq + 255) / 256, a->H, a->B * p.n_splits());
  return launch_attn_kernel(kern, "attn2_tc_kernel", attr_set, kAttn2Smem, grid, kAttn2Threads, stream, tmQ, tmK, tmV, p);
}

}  // namespace rfb
