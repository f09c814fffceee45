// Standalone GPU self-test + micro-benchmark of rfb_attention (no torch).
#include <stdlib.h>
#include <string.h>

#include "selftest_common.h"

// operand format under test: bf16, or fp16 with RFB_TEST_F16=1 in the environment
static int g_dt = RFB_BF16;
__device__ int d_f16 = 0;
__device__ __forceinline__ float bf2f(uint16_t u) {
  return d_f16 ? __half2float(*reinterpret_cast<const __half*>(&u)) : __uint_as_float((uint32_t)u << 16);
}

// one thread per (b, h, q): fp32 online softmax over all permitted keys
__global__ void ref_attn(const uint16_t* Q, long long ldq, long long qbs, const uint16_t* K,
                         long long ldk, long long kbs, const uint16_t* Vt, long long ldvt,
                         long long vbs, float* O, int B, int H, int Nq, int Nk,
                         const uint32_t* mask, long long mstride, int mode, const uint8_t* gid,
                         int period, float scale, const float* rq, const float* rk) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)B * H * Nq) return;
  const int qi = t % Nq, h = (t / Nq) % H, b = t / ((long long)Nq * H);
  const uint16_t* q = Q + b * qbs + (long long)qi * ldq + h * 128;
  float m = -INFINITY, l = 0.f, acc[128];
  for (int d = 0; d < 128; ++d) acc[d] = 0.f;
  int k_lo = 0, k_hi = Nk;
  if (mode == 1) k_lo = (qi / 128) * 128, k_hi = min(Nk, k_lo + 128);
  for (int k = k_lo; k < k_hi; ++k) {
    if (mode == 0 && mask && !((mask[b * mstride + k / 32] >> (k % 32)) & 1u)) continue;
    if (mode == 1 && (gid[qi % period] != gid[k % period] || qi / 64 != k / 64)) continue;
    const uint16_t* kr = K + b * kbs + (long long)k * ldk + h * 128;
    float s = 0.f;
    for (int d = 0; d < 128; ++d) s = fmaf(bf2f(q[d]), bf2f(kr[d]), s);
    s *= scale;
    if (rq) s *= rq[(long long)b * Nq + qi];
    if (rk) s *= rk[(long long)b * Nk + k];
    const float mn = fmaxf(m, s);
    const float a = expf(m - mn), pexp = expf(s - mn);
    l = l * a + pexp;
    const uint16_t* vc = Vt + b * vbs + (long long)h * 128 * ldvt + k;
    for (int d = 0; d < 128; ++d) acc[d] = acc[d] * a + pexp * bf2f(vc[(long long)d * ldvt]);
    m = mn;
  }
  float* o = O + ((long long)b * Nq + qi) * H * 128 + h * 128;
  for (int d = 0; d < 128; ++d) o[d] = l > 0.f ? acc[d] / l : 0.f;
}

// 64-bit FNV-1a of the output bytes, printed per correctness case: runs under RFB_ATTN_GEN=2 and =3 must print the
// same hashes, because the two dense kernels are meant to give bit-identical results
static void print_hash(const char* name, const std::vector<uint16_t>& out) {
  uint64_t h = 14695981039346656037ull;
  const unsigned char* p = reinterpret_cast<const unsigned char*>(out.data());
  for (size_t i = 0; i < out.size() * sizeof(uint16_t); ++i) h = (h ^ p[i]) * 1099511628211ull;
  printf("[HASH] %-46s %016llx\n", name, (unsigned long long)h);
}

struct ACase {
  const char* name;
  int B, H, Nq, Nk, mode, masked, shareKV, period;
  int fused = 0;  // 1: q_sumsq partial sums (fused q RMSNorm); 2: q and k sums (mode 1)
  int split = 0;  // kv_split_tiles: key chunks of this many 128-key tiles + ordered merge
};

static void run(const ACase& c, bool timing_only = false) {
  const int D = c.H * 128;
  const long long ldvt = (c.Nk + 7) & ~7;
  const int Bkv = c.shareKV ? 1 : c.B;
  const size_t nq = (size_t)c.B * c.Nq * D, nk = (size_t)Bkv * c.Nk * D, nv = (size_t)Bkv * D * ldvt;
  DevBuf<uint16_t> dQ(nq), dK(nk), dV(nv), dO(nq);
  if (!timing_only) {
    dQ.up(rand16(nq, 1, 2.0f, g_dt));
    dK.up(rand16(nk, 2, 2.0f, g_dt));
    dV.up(rand16(nv, 3, 1.0f, g_dt));
  } else {
    CK(cudaMemset(dQ.p, 0x3c, nq * 2));
    CK(cudaMemset(dK.p, 0x3c, nk * 2));
    CK(cudaMemset(dV.p, 0x3c, nv * 2));
  }
  dO.fill_byte(0xff);
  const int words = 4 * ((c.Nk + 127) / 128);
  std::vector<uint32_t> hm((size_t)c.B * words, 0);
  for (int b = 0; b < c.B; ++b)
    for (int k = 0; k < c.Nk; ++k) {
      bool ok = true;
      if (c.masked == 1) ok = k < c.Nk - 37 * (b + 1);                  // prefix (padding) mask
      if (c.masked == 2) ok = (hash_u32(k * 31 + b) % 3) != 0 || k < 16;  // arbitrary mask
      if (c.masked == 3) ok = k < 200 - 70 * b;                         // whole key chunks without a valid key
      if (ok) hm[(size_t)b * words + k / 32] |= 1u << (k % 32);
    }
  DevBuf<uint32_t> dM(hm.size());
  dM.up(hm);
  std::vector<uint8_t> hg(c.period > 0 ? c.period : 1);
  for (size_t i = 0; i < hg.size(); ++i) hg[i] = (uint8_t)(hash_u32(i / 8) % 3);
  DevBuf<uint8_t> dG(hg.size());
  dG.up(hg);

  // fused QK-RMSNorm inputs: interleaved [q parts | k parts] partial sums per row, as rfb_gemm leaves them
  const int parts = 3, sq_ld = 2 * parts, norm_dim = 384;
  const float eps = 1e-6f;
  const size_t nrows = (size_t)c.B * (c.Nq > c.Nk ? c.Nq : c.Nk);
  std::vector<float> hsq(nrows * sq_ld), hrq(nrows, 1.f), hrk(nrows, 1.f);
  for (size_t r = 0; r < nrows; ++r) {
    float tq = 0.f, tk = 0.f;
    for (int j = 0; j < parts; ++j) {
      hsq[r * sq_ld + j] = 40.f + 80.f * (0.5f + 0.5f * hval(71, (uint32_t)(r * 8 + j)));
      hsq[r * sq_ld + parts + j] = 30.f + 90.f * (0.5f + 0.5f * hval(72, (uint32_t)(r * 8 + j)));
      tq += hsq[r * sq_ld + j], tk += hsq[r * sq_ld + parts + j];
    }
    hrq[r] = 1.0f / sqrtf(tq / norm_dim + eps), hrk[r] = 1.0f / sqrtf(tk / norm_dim + eps);
  }
  DevBuf<float> dsq(hsq.size()), drq(nrows), drk(nrows);
  dsq.up(hsq), drq.up(hrq), drk.up(hrk);

  rfb_attn_args a;
  memset(&a, 0, sizeof(a));
  a.B = c.B, a.H = c.H, a.Nq = c.Nq, a.Nk = c.Nk;
  if (c.fused) {
    a.q_sumsq = dsq.p, a.sumsq_ld = sq_ld, a.sumsq_parts = parts, a.norm_dim = norm_dim, a.norm_eps = eps;
    if (c.fused == 2) a.k_sumsq = dsq.p + parts;
  }
  a.Q = dQ.p, a.ldq = D, a.q_batch_stride = (long long)c.Nq * D;
  a.K = dK.p, a.ldk = D, a.k_batch_stride = c.shareKV ? 0 : (long long)c.Nk * D;
  a.Vt = dV.p, a.ldvt = ldvt, a.vt_batch_stride = c.shareKV ? 0 : (long long)D * ldvt;
  a.O = dO.p, a.ldo = D, a.o_batch_stride = (long long)c.Nq * D;
  a.key_mask_bits = c.masked ? dM.p : nullptr, a.mask_batch_stride_words = words;
  a.mode = c.mode, a.group_id = dG.p, a.group_period = c.period;
  a.scale = 0.08838834764831845f;
  a.dtype = g_dt;
  const long long ws_bytes = rfb_attention_ws_bytes(c.B, c.H, c.Nq, c.Nk, c.split);
  DevBuf<float> dws((size_t)(ws_bytes / 4 + 4));
  if (c.split) a.kv_split_tiles = c.split, a.split_ws = dws.p, a.split_ws_bytes = ws_bytes;

  if (timing_only) {
    for (int i = 0; i < 3; ++i) rfb_attention(&a, 0);
    CK(cudaDeviceSynchronize());
    GpuTimer t;
    const int iters = 10;
    t.start();
    for (int i = 0; i < iters; ++i) rfb_attention(&a, 0);
    float ms = t.stop() / iters;
    double keys = c.mode == 1 ? 128.0 : c.Nk;
    double tf = 4.0 * c.B * c.H * (double)c.Nq * keys * 128 / (ms * 1e-3) / 1e12;
    printf("[BENCH] %-44s %.3f ms  %.1f TFLOP/s\n", c.name, ms, tf);
    fflush(stdout);
    return;
  }

  int rc = rfb_attention(&a, 0);
  cudaError_t e = cudaDeviceSynchronize();
  if (rc != RFB_OK || e != cudaSuccess) {
    printf("[FAIL] %-46s rc=%d cuda=%s\n", c.name, rc, cudaGetErrorString(e));
    g_fail++;
    if (e != cudaSuccess) exit(3);
    return;
  }
  DevBuf<float> dref(nq);
  long long nthreads = (long long)c.B * c.H * c.Nq;
  ref_attn<<<(unsigned)((nthreads + 63) / 64), 64>>>(
      dQ.p, D, (long long)c.Nq * D, dK.p, D, a.k_batch_stride, dV.p, ldvt, a.vt_batch_stride, dref.p,
      c.B, c.H, c.Nq, c.Nk, c.masked ? dM.p : nullptr, words, c.mode, dG.p, c.period > 0 ? c.period : 1,
      a.scale, c.fused ? drq.p : nullptr, c.fused == 2 ? drk.p : nullptr);
  CK(cudaDeviceSynchronize());
  std::vector<float> ref = dref.down();
  std::vector<uint16_t> ho = dO.down();
  print_hash(c.name, ho);
  std::vector<float> got(nq);
  for (size_t i = 0; i < nq; ++i) got[i] = h162f(ho[i], g_dt);
  report(c.name, got, ref, 1.5e-2, 2e-2, D);
}

// A query row's result must not depend on how many rows the call holds (which decides the kernel generation and
// the grid): rows [r0, r0 + n) of a full-length call vs a call on those rows alone, bit for bit.
static void run_row_invariance(const char* name, int H, int N, int r0, int n, int split) {
  const int D = H * 128;
  const long long ldvt = (N + 7) & ~7;
  const size_t nq = (size_t)N * D, nv = (size_t)D * ldvt;
  DevBuf<uint16_t> dQ(nq), dK(nq), dV(nv), dO(nq), dO2((size_t)n * D);
  dQ.up(rand16(nq, 41, 2.0f, g_dt)), dK.up(rand16(nq, 42, 2.0f, g_dt)), dV.up(rand16(nv, 43, 1.0f, g_dt));
  dO.fill_byte(0xff), dO2.fill_byte(0xee);
  const int words = 4 * ((N + 127) / 128);
  std::vector<uint32_t> hm(words, 0);
  for (int k = 0; k < N - 29; ++k) hm[k / 32] |= 1u << (k % 32);
  DevBuf<uint32_t> dM(hm.size());
  dM.up(hm);
  std::vector<uint16_t> got[2];
  for (int w = 0; w < 2; ++w) {
    const int Nq = w == 0 ? N : n;
    const long long ws_bytes = rfb_attention_ws_bytes(1, H, Nq, N, split);
    DevBuf<float> dws((size_t)(ws_bytes / 4 + 4));
    rfb_attn_args a;
    memset(&a, 0, sizeof(a));
    a.B = 1, a.H = H, a.Nq = Nq, a.Nk = N;
    a.Q = w == 0 ? dQ.p : dQ.p + (size_t)r0 * D, a.ldq = D;
    a.K = dK.p, a.ldk = D, a.Vt = dV.p, a.ldvt = ldvt;
    a.O = w == 0 ? dO.p : dO2.p, a.ldo = D;
    a.key_mask_bits = dM.p, a.mask_batch_stride_words = words;
    a.scale = 0.08838834764831845f, a.dtype = g_dt;
    if (split) a.kv_split_tiles = split, a.split_ws = dws.p, a.split_ws_bytes = ws_bytes;
    int rc = rfb_attention(&a, 0);
    cudaError_t e = cudaDeviceSynchronize();
    if (rc != RFB_OK || e != cudaSuccess) {
      printf("[FAIL] %-46s rc=%d cuda=%s\n", name, rc, cudaGetErrorString(e));
      g_fail++;
      if (e != cudaSuccess) exit(3);
      return;
    }
    got[w] = w == 0 ? dO.down() : dO2.down();
  }
  const bool same = !memcmp(got[0].data() + (size_t)r0 * D, got[1].data(), (size_t)n * D * 2);
  printf("[%s] %-46s rows %d..%d of %d vs alone: %s\n", same ? " ok " : "FAIL", name, r0, r0 + n, N,
         same ? "bit-identical" : "DIFFERENT");
  if (!same) g_fail++;
}

int main(int argc, char** argv) {
  const bool only_bench = argc > 1 && !strcmp(argv[1], "bench");
  if (const char* e = getenv("RFB_TEST_F16")) {
    if (e[0] == '1') {
      g_dt = RFB_F16;
      const int one = 1;
      CK(cudaMemcpyToSymbol(d_f16, &one, sizeof(int)));
      printf("selftest_attn: fp16 operands\n");
    }
  }
  if (!only_bench) {
    std::vector<ACase> cases = {
        {"1 tile  B1 H1 Nq128 Nk128", 1, 1, 128, 128, 0, 0, 0, 0},
        {"2 kv tiles B1 H1 Nq128 Nk256", 1, 1, 128, 256, 0, 0, 0, 0},
        {"5 kv tiles B1 H2 Nq256 Nk640", 1, 2, 256, 640, 0, 0, 0, 0},
        {"ragged B2 H2 Nq300 Nk400 (no mask)", 2, 2, 300, 400, 0, 0, 0, 0},
        {"prefix mask B2 H2 Nq300 Nk400", 2, 2, 300, 400, 0, 1, 0, 0},
        {"random mask B3 H1 Nq200 Nk1000", 3, 1, 200, 1000, 0, 2, 0, 0},
        {"shared KV B4 H2 Nq256 Nk272 prefix mask", 4, 2, 256, 272, 0, 1, 1, 0},
        {"enc-like B1 H8 N4112", 1, 8, 4112, 4112, 0, 1, 0, 0},
        {"swin mode1 B1 H2 N1024 period 256", 1, 2, 1024, 1024, 1, 0, 0, 256},
        {"swin mode1 B1 H8 N8192 period 4096", 1, 8, 8192, 8192, 1, 0, 0, 4096},
        {"fused q-norm B3 H2 Nq300 Nk400 shared KV", 3, 2, 300, 400, 0, 1, 1, 0, 1},
        {"fused q+k-norm swin mode1 B1 H2 N1024", 1, 2, 1024, 1024, 1, 0, 0, 256, 2},
        // short tail (last key tile <= 32 keys runs 32 wide): 16 / 32 keys, 33 keys (full-width path), with masks and splits
        {"short tail 16: random mask B3 H1 Nq200 Nk1040", 3, 1, 200, 1040, 0, 2, 0, 0},
        {"short tail 32: prefix mask B2 H2 Nq300 Nk1056", 2, 2, 300, 1056, 0, 1, 0, 0},
        {"tail 33 (full width) B2 H2 Nq300 Nk1057", 2, 2, 300, 1057, 0, 0, 0, 0},
        {"short tail 1 key, no mask B1 H2 Nq130 Nk129", 1, 2, 130, 129, 0, 0, 0, 0},
        {"short tail 16 + key split 3, random mask Nk1040", 3, 1, 200, 1040, 0, 2, 0, 0, 0, 3},
        {"short tail alone in its chunk: split 4, Nk1040", 2, 2, 300, 1040, 0, 1, 0, 0, 0, 4},
        {"key split 2 B3 H1 Nq200 Nk1000 random mask", 3, 1, 200, 1000, 0, 2, 0, 0, 0, 2},
        {"key split 3 (3,3,2) B2 H2 Nq300 Nk1000 prefix", 2, 2, 300, 1000, 0, 1, 0, 0, 0, 3},
        {"key split 1: chunks with no valid key", 2, 2, 300, 600, 0, 3, 0, 0, 0, 1},
        {"key split 2 fused q-norm shared KV B3 Nk700", 3, 2, 300, 700, 0, 1, 1, 0, 1, 2},
        {"key split 11 enc-like B1 H8 N4112", 1, 8, 4112, 4112, 0, 1, 0, 0, 0, 11},
        {"key split 11 one rank of 8: Nq520 Nk4112", 1, 8, 520, 4112, 0, 1, 0, 0, 0, 11},
    };
    for (auto& c : cases) run(c);
    run_row_invariance("row invariance, key split 11, H8 N4112", 8, 4112, 1040, 520, 11);
    run_row_invariance("row invariance, no split, H8 N4112", 8, 4112, 1040, 520, 0);
    run_row_invariance("row invariance, key split 3, H2 N1500 (ragged)", 2, 1500, 256, 200, 3);
    printf("selftest_attn: %d failure(s)\n", g_fail);
    if (g_fail) return 1;
  }
  run({"enc self  B1 H8 N4112", 1, 8, 4112, 4112, 0, 0, 0, 0}, true);
  run({"enc self  B1 H8 N4112, key split 11", 1, 8, 4112, 4112, 0, 0, 0, 0, 0, 11}, true);
  run({"one rank of 8: Nq520 Nk4112", 1, 8, 520, 4112, 0, 0, 0, 0}, true);
  run({"one rank of 8: Nq520 Nk4112, key split 11", 1, 8, 520, 4112, 0, 0, 0, 0, 0, 11}, true);
  run({"one rank of 2: Nq2056 Nk4112, key split 11", 1, 8, 2056, 4112, 0, 0, 0, 0, 0, 11}, true);
  run({"cross     B8 H8 Nq4096 Nk4112 sharedKV", 8, 8, 4096, 4112, 0, 1, 1, 0}, true);
  run({"swin      B1 H8 N32768 mode1", 1, 8, 32768, 32768, 1, 0, 0, 4096}, true);
  return g_fail ? 1 : 0;
}
