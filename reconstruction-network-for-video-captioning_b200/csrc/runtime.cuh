// Host-side runtime shared by the sequence drivers: precision dispatch of the GEMM provider, split-K policy,
// workspace carving.  T = float (RECNET_PREC_FP32, FFMA sgemm) or bf16 (RECNET_PREC_BF16, tcgen05 GEMM).
#pragma once
#include "attention.cuh"
#include "common.cuh"
#include "gemm_tc.cuh"
#include "losses.cuh"
#include "lstm_cell.cuh"
#include "misc.cuh"
#include "sgemm.cuh"
#include <stdlib.h>

namespace rt {

constexpr int NUM_SMS = 148;

struct Bump {
  uint8_t* base;
  size_t off;
  explicit Bump(void* b) : base(reinterpret_cast<uint8_t*>(b)), off(0) {}
  template <typename T> T* take(size_t n) {
    off = (off + 255) & ~(size_t)255;
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

template <typename T> struct Prec;
template <> struct Prec<float> { static constexpr int id = RECNET_PREC_FP32; static constexpr int kpad = 4; };
template <> struct Prec<bf16> { static constexpr int id = RECNET_PREC_BF16; static constexpr int kpad = 64; };

// ---- side stream for the batched work around the time loops (default on; RECNET_SIDE=0 puts everything on `main`) -------------
// Before and after each time loop a driver issues a dozen mutually independent batched kernels (weight-gradient GEMMs, column
// sums, operand staging); several of them are small grids (the 128-row attention weight gradients run on 32-64 CTAs) or end in
// a partial wave.  fork() hands out a second stream ordered after everything issued so far on `main`; the driver splits the
// independent work between the two and join()s before it returns, so nothing outlives the call and the pattern is a plain
// fork/join inside a captured CUDA graph.  Concurrent split-K GEMMs / column sums use separate scratch (Ws::splitk2).
// History: r1 measured this SLOWER (2.781 -> 2.839 ms, profiles/r1_g_side_stream.md) -- the one-tile-per-CTA GEMMs of that round each
// filled the machine with 200-400 CTAs, so two of them side by side only shared the L2.  The persistent GEMMs of r2 (gemm_tc2.cuh) launch
// min(tiles, 148) CTAs: a 72- or 96-tile GEMM leaves SMs free and its neighbour on the other stream takes them.  r2: 2.276 -> 2.232 ms.
struct Side {
  cudaStream_t s = nullptr;
  cudaEvent_t fork_ev = nullptr, join_ev = nullptr;
  int dev = -1;
  static bool enabled() {
    static const int on = rn_env_int("RECNET_SIDE", 1);
    return on != 0;
  }
  int fork(cudaStream_t main, cudaStream_t* out) {
    *out = main;
    if (!enabled()) return 0;
    int cur = 0;
    RN_CUDA_OK(cudaGetDevice(&cur));
    if (cur != dev) {               // one process drives one GPU; re-create if a test switches devices
      RN_CUDA_OK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
      RN_CUDA_OK(cudaEventCreateWithFlags(&fork_ev, cudaEventDisableTiming));
      RN_CUDA_OK(cudaEventCreateWithFlags(&join_ev, cudaEventDisableTiming));
      dev = cur;
    }
    RN_CUDA_OK(cudaEventRecord(fork_ev, main));
    RN_CUDA_OK(cudaStreamWaitEvent(s, fork_ev, 0));
    *out = s;
    return 0;
  }
  int join(cudaStream_t main, cudaStream_t side_stream) {
    if (side_stream == main) return 0;
    RN_CUDA_OK(cudaEventRecord(join_ev, side_stream));
    RN_CUDA_OK(cudaStreamWaitEvent(main, join_ev, 0));
    return 0;
  }
};
inline Side& side() { static Side x; return x; }

// ---- split-K / tile policy ---------------------------------------------------------------------------
struct GemmPlan { int bn; int splits; };
template <typename T> static inline GemmPlan plan_gemm(int M, int N, int K);
template <> inline GemmPlan plan_gemm<bf16>(int M, int N, int K) {
  GemmPlan p;
  p.bn = (N >= 1024) ? 128 : 64;
  const int nkb0 = rn_cdiv(K, tc::BK);
  if (nkb0 >= 16 && rn_cdiv(M, tc::BM) * rn_cdiv(N, 64) >= 2 * NUM_SMS) {
    // Batched GEMMs (weight gradients, hoisted projections).  r1 ncu: the main loop is bound by what one SM can pull from L2
    // (~50 B/clk), not by the tensor pipe, so wider N tiles (fewer A re-reads per MMA) win unless they cost a whole extra wave.
    // cost per k-block ~ max(MMA cycles = 2 bn, (A 12.8 KB + B 128 bn bytes) / 50 B/clk); total ~ waves * cost.
    float best = 1e30f;
    for (int bn = 64; bn <= 256; bn *= 2) {
      const int tiles = rn_cdiv(M, tc::BM) * rn_cdiv(N, bn);
      const float per = fmaxf(2.f * bn, (12800.f + 128.f * bn) / 50.f);
      const float cost = (float)rn_cdiv(tiles, NUM_SMS) * per;
      if (cost < best * 0.97f) { best = cost; p.bn = bn; }
    }
    p.splits = 1;
    return p;
  }
  const int tiles = rn_cdiv(M, tc::BM) * rn_cdiv(N, p.bn);
  const int nkb = rn_cdiv(K, tc::BK);
  int s = NUM_SMS / tiles;
  if (s < 1) s = 1;
  if (s > nkb) s = nkb;
  const int kb_per = rn_cdiv(nkb, s);
  p.splits = rn_cdiv(nkb, kb_per);
  return p;
}
template <> inline GemmPlan plan_gemm<float>(int M, int N, int K) {
  GemmPlan p;
  p.bn = 0;
  const int tiles = rn_cdiv(M, sg::BM) * rn_cdiv(N, sg::BN);
  int s = (2 * NUM_SMS) / tiles;
  const int maxs = K / 64 > 0 ? K / 64 : 1;
  if (s < 1) s = 1;
  if (s > maxs) s = maxs;
  const int k_per = rn_cdiv(rn_cdiv(K, s), sg::BK) * sg::BK;
  p.splits = rn_cdiv(K, k_per);
  return p;
}

// ---- raw GEMM provider -----------------------------------------------------------------------------------
static inline int gemm_raw(const float* A, long long lda, int tA, const float* B, long long ldb, int tB, float* C,
                           long long ldc, const float* bias, int M, int N, int K, GemmPlan p, long long split_stride,
                           int accumulate, cudaStream_t st) {
  return sg::launch(A, lda, tA, B, ldb, tB, C, ldc, bias, M, N, K, p.splits, split_stride, accumulate, st);
}
static inline int gemm_raw(const bf16* A, long long lda, int tA, const bf16* B, long long ldb, int tB, float* C,
                           long long ldc, const float* bias, int M, int N, int K, GemmPlan p, long long split_stride,
                           int accumulate, cudaStream_t st) {
  return tc::launch(A, lda, tA, B, ldb, tB, C, ldc, nullptr, 0, bias, M, N, K, p.splits, split_stride, accumulate,
                    p.bn, st);
}

__global__ void splitk_reduce_kernel(const float* __restrict__ P, int splits, long long split_stride, long long ldp,
                                     float* __restrict__ out, long long ldo, int M, int N, const float* __restrict__ bias,
                                     int accumulate) {
  const long long total = (long long)M * N;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int m = (int)(i / N), n = (int)(i % N);
    float s = bias ? bias[n] : 0.f;
    for (int k = 0; k < splits; ++k) s += P[k * split_stride + (long long)m * ldp + n];
    float* o = out + (long long)m * ldo + n;
    *o = accumulate ? *o + s : s;
  }
}
static inline int splitk_reduce(const float* P, int splits, long long split_stride, long long ldp, float* out,
                                long long ldo, int M, int N, const float* bias, int accumulate, cudaStream_t st) {
  const long long total = (long long)M * N;
  if (total <= 0) return 0;
  int blocks = (int)min((long long)NUM_SMS * 8, (total + 255) / 256);
  if (rn_background_ctas() > 0) blocks = min(blocks, rn_background_ctas());       // grid-stride loop: fewer CTAs, same result
  ProfScope prof(KC_REDUCE, M, N, splits, st);
  splitk_reduce_kernel<<<blocks, 256, 0, st>>>(P, splits, split_stride, ldp, out, ldo, M, N, bias, accumulate);
  RN_LAUNCH_OK();
  return 0;
}

constexpr size_t SPLITK_SCRATCH_FLOATS = (size_t)NUM_SMS * 2 * 128 * 128;   // enough for any plan with splits > 1

// ---- tile / split-K plan of the BATCHED GEMMs (gemm_full: weight gradients, hoisted projections, vocabulary projection) ----------
template <typename T> static inline GemmPlan plan_gemm_full(int M, int N, int K) { return plan_gemm<T>(M, N, K); }
// Cost model fitted to a sweep of every batched GEMM of the MSVD train step over (N-tile width, split count) on the B200
// (tools/gemm_sweep.py, profiles/r1_g_gemm_sweep.md).  What the sweep showed: the main loop is bound by L2 -> SM delivery, not by
// the tensor pipe.  With all 148 SMs pulling, one k-block (64 deep) costs ~857 / 1030 / 1240 cycles for 64 / 128 / 256-wide tiles
// (24 / 32 / 48 KB ingested per CTA: ~5.7 KB/clk chip-wide); a partially filled wave is bound per SM instead (~745 / 857 / 944
// cycles); every wave pays prologue + epilogue (~2000 + 16 bn cycles); a split-K plan adds the reduce pass (~5 us + bytes at
// 3.5 TB/s).  Wider tiles win whenever they do not cost an extra wave; split-K only pays for GEMMs with a handful of tiles.
// Candidates are visited from the simplest plan up and must beat the incumbent by 5 % (the fit is good to about +-4 us).
template <> inline GemmPlan plan_gemm_full<bf16>(int M, int N, int K) {
  static const float CF[3] = {857.f, 1030.f, 1240.f}, FL[3] = {745.f, 857.f, 944.f};
  static const int SPL[6] = {1, 2, 3, 4, 6, 8};
  const int mt = rn_cdiv(M, tc::BM), nkb = rn_cdiv(K, tc::BK);
  const long long Np = round_up(N, 4);
  GemmPlan best{64, 1};
  float best_us = 1e30f;
  for (int si = 0; si < 6; ++si) {
    const int s = SPL[si];
    if (s > nkb) break;
    if (s > 1 && (size_t)s * M * Np > SPLITK_SCRATCH_FLOATS) break;
    for (int bi = 0; bi < 3; ++bi) {
      const int bn = 64 << bi;
      if (s > 1 && bn == 256) continue;                  // split plans stay on the 64 / 128-wide kernels
      if (bn > 64 && N <= bn / 2) continue;              // more than half of the tile would be padding
      const long long ctas = (long long)mt * rn_cdiv(N, bn) * s;
      if (rn_background_ctas() > 0 && s > 1 && ctas > rn_background_ctas()) continue;      // background lane: stay within the CTA budget
      const int kb = rn_cdiv(nkb, s);
      const long long full = ctas / NUM_SMS;
      const int rem = (int)(ctas % NUM_SMS);
      const float wave = 2000.f + 16.f * bn;
      float clk = (float)full * (kb * CF[bi] + wave);
      if (rem) clk += kb * fmaxf(FL[bi], CF[bi] * rem / NUM_SMS) + wave;
      float us = clk / 1965.f;
      if (s > 1) us += 5.f + (float)(s + 1) * M * N * 4.f / 3.5e6f;
      if (us < best_us * 0.95f) { best_us = us; best.bn = bn; best.splits = s; }
    }
  }
  if (best.splits > 1) {                                   // every slice gets >= 1 k-block (same rounding as plan_gemm)
    const int kb_per = rn_cdiv(nkb, best.splits);
    best.splits = rn_cdiv(nkb, kb_per);
  }
  // r2: the persistent kernel of gemm_tc2.cuh (bn = 1000 + width: single CTAs, 2000 + width: CTA pairs) for everything that is not
  // skinny -- sweep in profiles/r2_h_gemm_sweep.md: it wins or ties on every batched GEMM with M, N >= 256; the four 128-row
  // attention weight gradients and the 128-column key projections stay on the split-K / 64-wide plans above.  256-wide tiles once
  // they fill 2/3 of the SMs; CTA pairs (half the B traffic per SM) only for long K loops with at least 1.5 rounds of pair tiles.
  static const int persist = rn_env_int("RECNET_GEMM_PERSIST", 1);
  if (persist && M >= 256 && N >= 256) {
    const int t256 = mt * rn_cdiv(N, 256);
    const int pairs = rn_cdiv(M, 256) * rn_cdiv(N, 256);
    best.splits = 1;
    if (t256 < 96) best.bn = 1128;
    else best.bn = (nkb >= 16 && 2 * pairs >= 3 * (NUM_SMS / 2)) ? 2256 : 1256;
  }
  return best;
}

// Full GEMM into a dense destination: splits the K loop when the tile grid alone cannot fill the GPU,
// reducing the partials with one extra pass.  `scratch` holds SPLITK_SCRATCH_FLOATS floats.
template <typename T>
static int gemm_full(const T* A, long long lda, int tA, const T* B, long long ldb, int tB, float* C, long long ldc,
                     const float* bias, int M, int N, int K, int accumulate, float* scratch, cudaStream_t st) {
  GemmPlan p = plan_gemm_full<T>(M, N, K);
  const int Np = round_up(N, 4);
  if (p.splits > 1 && (size_t)p.splits * M * Np > SPLITK_SCRATCH_FLOATS) p.splits = 1;
  if (p.splits <= 1) {
    p.splits = 1;
    return gemm_raw(A, lda, tA, B, ldb, tB, C, ldc, bias, M, N, K, p, 0, accumulate, st);
  }
  RN_TRY(gemm_raw(A, lda, tA, B, ldb, tB, scratch, Np, nullptr, M, N, K, p, (long long)M * Np, 0, st));
  return splitk_reduce(scratch, p.splits, (long long)M * Np, Np, C, ldc, M, N, bias, accumulate, st);
}

// Per-step GEMM that leaves split-K partials for the consumer kernel to sum: out [splits][M, N] (ld = N).
template <typename T>
static int gemm_partials(const T* A, long long lda, int tA, const T* B, long long ldb, int tB, float* P, int M, int N,
                         int K, GemmPlan p, cudaStream_t st) {
  return gemm_raw(A, lda, tA, B, ldb, tB, P, N, nullptr, M, N, K, p, (long long)M * N, 0, st);
}

template <typename T>
static int zero_async(T* p, size_t n, cudaStream_t st) {
  RN_CUDA_OK(cudaMemsetAsync(p, 0, n * sizeof(T), st));
  return 0;
}
}  // namespace rt
