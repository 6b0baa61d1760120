// Weight-resident persistent time loop of the LOCAL reconstructor (forward), one cooperative launch for all S steps.
//   reference: models/local_reconstructor.py:37-55 called S times from train.py:122-124
//
// Why (profiles/r2_a_segments.md): as a chain of 4 kernels per step (query GEMM, attention, gate GEMM, cell) the loop costs
// ~22 us per step, of which ~1.3 us is tensor-pipe time; the rest is kernel boundaries and the 25 MB [W_ih | W_hh] operand being
// re-pulled from L2 every step.  Here the weights are loaded ONCE into the shared memory of UG x KS CTAs and stay there:
//
//   CTA (ug, ks):  32 hidden units x 4 gates (128 accumulator columns)  x  K-slice ks of [x_t ; h_{t-1}]   (<= 11 k-blocks = 176 KB)
//
// Per step:  [h_{t-1} visible] -> recurrent half of the gate GEMM (tcgen05, accumulates in TMEM) runs while 8 warps of the
// first B CTAs do the attention of one sample each -> [x_t visible] -> input half of the GEMM into the same accumulator ->
// fp32 K-slice partials exchanged through L2 inside the unit group (KS CTAs, one flag) -> cell update, h_t written as next
// step's operand row, and the partial attention query  Wh_{t+1}[b, :] += h_t[b, units] . W_a[:, units]^T  of these 32 units
// (CUDA cores, W_a slice in registers) -> [h_t visible].  Two grid-wide flag waits + one unit-group flag per step; nothing
// else leaves the SM.  The stash (x_t / h_t operand rows, Wh, scores, activated gates, c) is laid out exactly as the
// kernel-per-phase path leaves it, so the batched GEMMs around the loop and the BPTT run unchanged behind it.
//
// Every spin is bounded (clock64 timeout -> error flag in the workspace, all later waits fall through), so a protocol bug
// surfaces as RECNET_ERR_* instead of a hung GPU.
#pragma once
#include "runtime.cuh"

namespace rp {
using namespace tc;

constexpr int THREADS = 448;          // warps 0-3 epilogue, 4 TMA producer, 5 MMA issuer, 6-13 attention
constexpr int MAX_STAGES = 8;         // activation ring (B rows x 64 k per stage): as deep as the shared memory left by the resident weights allows
constexpr int UNITS = 32;             // hidden units per CTA
constexpr int NCOL = 4 * UNITS;       // accumulator columns (gate g, unit u) -> column g*32 + u
constexpr int MAX_KB = 11;            // resident k-blocks per CTA (16 KB each)
constexpr int WTILE = NCOL * BK * 2;  // 16384
constexpr int NWORK = 12;             // warps in the cell / query phase
constexpr int MAX_UG = 64;
constexpr int HS_LD = 40;             // bf16 elements per hs row (80 B: conflict-free fragment loads)
constexpr long long TIMEOUT = 600000000LL;      // ~0.3 s of SM clocks

struct FwdParams {
  int B, S, R, H, A, L, KX, UG, KS, NHB, NXB;
  int nst, res_kb;                    // ring stages / resident k-blocks per CTA (set by the launcher)
  float inv_L, p_drop;
  bf16* X;                            // [(S+1)*B, KX] operand rows [x_t | h_{t-1}]
  const bf16* Hd;                     // [L*B, H] decoder states (attention values)
  const float* Uv;                    // [L, B, A]
  const bf16* Wa;                     // [A, R]
  const float *attn_b, *attn_w, *b_ih, *b_hh;
  float* Wh;                          // [S, B, A] stash (query without the bias)
  float* beta;                        // [S, B, L] stash (scores; alpha with the softmax attention)
  bf16* gates;                        // [S*B, 4R] activated gates
  float* c;                           // [(S+1)*B, R]
  float* XP;                          // [UG][KS][B][128] K-slice partials of the pre-activations
  float* WhP;                         // [UG][B][A] unit-group partials of the next step's query
  unsigned* sync;                     // [0] h-ready counter, [32] x-ready counter, [64 + 32*ug] exchange flags (zeroed before launch)
  int* err;
  const unsigned long long* rng;
  unsigned site;
  // GLOBAL reconstructor mode (models/global_reconstructor.py:30-46): no attention, H = 0 (operand rows hold h only); the hoisted
  // input projection Gx [S*B, 4R] (b_ih folded in) is added in the cell update instead
  int global_mode;
  const float* Gx;
};

__device__ __forceinline__ unsigned ld_acq(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_rel(unsigned* p) { asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(p) : "memory"); }
__device__ __forceinline__ void proxy_fence() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void nbar(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// bounded waits; once *abort is set every later wait falls through (all bar.sync's are still executed -> no CTA-level hang)
__device__ __forceinline__ void wait_flag(const unsigned* f, unsigned target, int* err, volatile int* abort_) {
  if (*abort_) return;
  const long long t0 = clock64();
  unsigned spins = 0;
  while (ld_acq(f) < target) {
    if ((++spins & 31u) == 0) {
      if (*reinterpret_cast<volatile int*>(err) != 0) { *abort_ = 1; return; }
      if (clock64() - t0 > TIMEOUT) { atomicExch(err, 3); *abort_ = 1; return; }
    }
  }
}
__device__ __forceinline__ void wait_mbar(uint32_t bar, uint32_t parity, int* err, volatile int* abort_) {
  if (*abort_) return;
  const long long t0 = clock64();
  uint32_t ok;
  for (;;) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return;
    if (clock64() - t0 > TIMEOUT) { atomicExch(err, 2); *abort_ = 1; return; }
    if (*abort_) return;
  }
}
// developer timeline: any single thread of block 0 (atomic slot)
__device__ __forceinline__ void stamp(int tag) {
  if (g_timeline != nullptr && blockIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    const unsigned int i = atomicAdd(&g_timeline_n, 1u);
    if (i < 4000) g_timeline[i] = (t & 0x00FFFFFFFFFFFFFFull) | ((unsigned long long)tag << 56);
  }
}

// ---- TMEM as a per-warp register file extension: 32 lanes x n columns (32-bit) of the warp's own lane quarter ----
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]),
        "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]),
        "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// loads WITHOUT the wait (several can be in flight); tmem_ld_wait() before the registers are read
__device__ __forceinline__ void tmem_ld32_nw(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16_nw(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
constexpr int TMEM_COLS = 256;        // [0,128) gate accumulator, [128, 224) attention operands parked by the attention warps

struct Smem {                // offsets from the 1024-aligned base
  int ring, wres, bars, e, whred, hs, total;
};
__host__ __device__ inline Smem smem_layout(int B, int KS, int nst, int res_kb) {
  Smem s;
  const int stage = ((B + 7) & ~7) * 128;
  s.ring = 0;
  s.wres = (nst * stage + 1023) & ~1023;
  s.bars = s.wres + res_kb * WTILE;               // full[8] empty[8] tmem wload | tmem slot | abort
  s.e = s.bars + 256;
  s.whred = s.e + 128;                            // [8][128] floats
  s.hs = s.whred + 8 * 128 * 4;                   // [48][HS_LD] bf16: h_t of this CTA's cells, A operand of the query mma
  s.total = s.hs + 4 * NWORK * HS_LD * 2 + 1024;  // + alignment slack
  return s;
}

// per-thread constants of the cell / query phase
struct CellCtx {
  int ww, lane, ug, ks, ns, j, tid, cta;
  float bi, bf_, bg, bo;
  uint32_t wb[8];                     // W_a fragments (B operand of mma.m16n8k16) of a-tiles 2ww, 2ww+1 over this CTA's 32 units
};

// cell update of this CTA's (sample, unit) cells + partial attention query of the next step + stash; all NWORK warps
template <int KS>
__device__ __forceinline__ void cell_query_phase(const FwdParams& p, const CellCtx& cq, int t, float (&creg)[4], bf16* hs) {
  const int ww = cq.ww, lane = cq.lane, ug = cq.ug, ks = cq.ks, ns = cq.ns, j = cq.j, tid = cq.tid, cta = cq.cta;
  const int B = p.B, S = p.S, R = p.R, H = p.H, A = p.A, KX = p.KX;
  const float bi = cq.bi, bf_ = cq.bf_, bg = cq.bg, bo = cq.bo;
  unsigned* barA = p.sync;
      nbar(2, NWORK * 32);
      if (cta == 0 && tid == 0) stamp(7);
      // ---------------- cell update of (sample, unit): lane = unit, warp ww takes sample slots i = ww + 12 r ----------------
      uint32_t gp_if[4], gp_go[4];                        // activated gates packed as bf16 pairs (i,f) (g,o): what the stash keeps
#pragma unroll
      for (int r0 = 0; r0 < 4; r0 += 2) {
        float pre[2][4];
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          const int r3 = r0 + rr;
          const int i = min(ww + r3 * NWORK, ns - 1), b = ks + KS * i;
          const float* q = p.XP + ((long long)ug * KS * B + b) * NCOL + lane;
          float part[KS][4];
#pragma unroll
          for (int k2 = 0; k2 < KS; ++k2)
#pragma unroll
            for (int g = 0; g < 4; ++g) part[k2][g] = q[(long long)k2 * B * NCOL + g * UNITS];
          float gxv[4] = {0.f, 0.f, 0.f, 0.f};
          if (p.global_mode) {
#pragma unroll
            for (int g = 0; g < 4; ++g) gxv[g] = p.Gx[((long long)t * B + b) * 4 * R + (long long)g * R + j];
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float s = part[0][g];
#pragma unroll
            for (int k2 = 1; k2 < KS; ++k2) s += part[k2][g];
            pre[rr][g] = s + gxv[g];
          }
        }
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          const int r3 = r0 + rr;
          const int i = ww + r3 * NWORK;
          const float gi = act_sigmoid<true>(pre[rr][0] + bi), gf = act_sigmoid<true>(pre[rr][1] + bf_);
          const float gg = act_tanh<true>(pre[rr][2] + bg), go = act_sigmoid<true>(pre[rr][3] + bo);
          { const __nv_bfloat162 x = __floats2bfloat162_rn(gi, gf), y = __floats2bfloat162_rn(gg, go);
            gp_if[r3] = *reinterpret_cast<const uint32_t*>(&x); gp_go[r3] = *reinterpret_cast<const uint32_t*>(&y); }
          if (i < ns) {
            const int b = ks + KS * i;
            creg[r3] = fmaf(gf, creg[r3], gi * gg);
            const bf16 hb = __float2bfloat16_rn(go * act_tanh<true>(creg[r3]));
            p.X[((long long)(t + 1) * B + b) * KX + H + j] = hb;          // next step's operand row
            hs[i * HS_LD + lane] = hb;
          }
        }
        if (ww + (r0 + 2) * NWORK >= ns) break;                          // warp-uniform: no further sample slots
      }
      if (cta == 0 && tid == 0) stamp(8);
      nbar(3, NWORK * 32);
      // ---------------- partial attention query of the next step over this CTA's 32 units ----------------
      // WhP[ug][b, a] = sum_u h_t[b, u] W_a[a, u]: [ns x 32] . [32 x 128] on mma.sync m16n8k16 (bf16 in, fp32 out); warp ww < 8 owns
      // a-tiles 2ww, 2ww+1 (its W_a fragments live in registers), loops over the sample tiles; rows >= ns are never stored
      if (t + 1 < S && ww < 8 && !p.global_mode) {
        const int gid = lane >> 2, tig = lane & 3;
        for (int mt = 0; mt * 16 < ns; ++mt) {
          uint32_t af[2][4];
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const bf16* r0 = hs + (mt * 16 + gid) * HS_LD + 16 * k + tig * 2;
            af[k][0] = *reinterpret_cast<const uint32_t*>(r0);
            af[k][1] = *reinterpret_cast<const uint32_t*>(r0 + 8 * HS_LD);
            af[k][2] = *reinterpret_cast<const uint32_t*>(r0 + 8);
            af[k][3] = *reinterpret_cast<const uint32_t*>(r0 + 8 * HS_LD + 8);
          }
#pragma unroll
          for (int nt = 0; nt < 2; ++nt) {
            float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
            for (int k = 0; k < 2; ++k)
              asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                           : "+f"(d0), "+f"(d1), "+f"(d2), "+f"(d3)
                           : "r"(af[k][0]), "r"(af[k][1]), "r"(af[k][2]), "r"(af[k][3]), "r"(cq.wb[4 * nt + 2 * k]), "r"(cq.wb[4 * nt + 2 * k + 1]));
            const int a = 16 * ww + 8 * nt + tig * 2;
            const int i0 = mt * 16 + gid, i1 = i0 + 8;
            if (i0 < ns) *reinterpret_cast<float2*>(p.WhP + ((long long)ug * B + (ks + KS * i0)) * A + a) = make_float2(d0, d1);
            if (i1 < ns) *reinterpret_cast<float2*>(p.WhP + ((long long)ug * B + (ks + KS * i1)) * A + a) = make_float2(d2, d3);
          }
        }
      }
      if (cta == 0 && tid == 0) stamp(9);
      nbar(4, NWORK * 32);
      if (tid == 0) { if (cta == 0) stamp(15); red_rel(barA); if (cta == 0) stamp(6); }
      // ---------------- stash for the BPTT (activated gates, c): only has to land by the end of the kernel ----------------
#pragma unroll
      for (int r3 = 0; r3 < 4; ++r3) {
        const int i = ww + r3 * NWORK;
        if (i < ns) {
          const int b = ks + KS * i;
          p.c[((long long)(t + 1) * B + b) * R + j] = creg[r3];
          unsigned short* gs = reinterpret_cast<unsigned short*>(p.gates + ((long long)t * B + b) * 4 * R + j);
          gs[0] = (unsigned short)(gp_if[r3] & 0xFFFFu); gs[R] = (unsigned short)(gp_if[r3] >> 16);
          gs[2 * R] = (unsigned short)(gp_go[r3] & 0xFFFFu); gs[3 * R] = (unsigned short)(gp_go[r3] >> 16);
        }
      }
}

// SM = true: the paper's softmax attention (opt-in) -- alpha over the Ln <= 32 scores in every attention warp's registers, weighted sum
// with scale 1 (the host passes inv_L = 1), alpha stashed in `beta`
template <int KS, bool SM>
__global__ void __launch_bounds__(THREADS, 1)
local_fwd_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW, const FwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const Smem L_ = smem_layout(p.B, KS, p.nst, p.res_kb);
  const uint32_t STAGES = (uint32_t)p.nst;
  const int stage_bytes = ((p.B + 7) & ~7) * 128;
  const uint32_t ring = base + L_.ring, wres = base + L_.wres;
  const uint32_t bar_full = base + L_.bars, bar_empty = bar_full + 8 * MAX_STAGES, bar_tmem = bar_empty + 8 * MAX_STAGES, bar_w = bar_tmem + 8;
  const uint32_t tmem_slot = bar_w + 8;
  volatile int* abort_ = reinterpret_cast<volatile int*>(gen + L_.bars + 192);
  float* e_s = reinterpret_cast<float*>(gen + L_.e);
  float* whred = reinterpret_cast<float*>(gen + L_.whred);
  bf16* hs = reinterpret_cast<bf16*>(gen + L_.hs);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cta = blockIdx.x;
  const int ug = cta / KS, ks = cta % KS;
  const int B = p.B, S = p.S, R = p.R, H = p.H, A = p.A, Ln = p.L, KX = p.KX;
  const int hb0 = (p.NHB * ks) / KS, hb1 = (p.NHB * (ks + 1)) / KS, nh = hb1 - hb0;
  const int xb0 = (p.NXB * ks) / KS, xb1 = (p.NXB * (ks + 1)) / KS, nx = xb1 - xb0;
  const int nkb = nh + nx;
  const unsigned ncta = gridDim.x;
  unsigned* barA = p.sync;
  unsigned* barB = p.sync + 32;
  unsigned* flagX = p.sync + 64 + 32 * ug;

  if (tid == 0) {
    for (int s = 0; s < MAX_STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    mbar_init(bar_tmem, 1);
    mbar_init(bar_w, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    *abort_ = 0;
  }
  if (warp == 5) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 4) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmX)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW)) : "memory");
      // resident weights: k-block i of this CTA = 4 boxes {64 k, 32 rows} (gate g rows g*R + ug*32 ..) -> tile rows g*32 + u
      mbar_expect_tx(bar_w, (uint32_t)nkb * WTILE);
      for (int i = 0; i < nkb; ++i) {
        const int kcol = (i < nh ? p.NXB + hb0 + i : xb0 + (i - nh)) * BK;
#pragma unroll
        for (int g = 0; g < 4; ++g) tma_load_2d(wres + i * WTILE + g * (UNITS * 128), &tmW, bar_w, kcol, g * R + ug * UNITS);
      }
      uint32_t it = 0;
      const uint32_t tx = (uint32_t)B * 128u;
      for (int t = 0; t < S; ++t) {
        if (t > 0) wait_flag(barA, ncta * (unsigned)t, p.err, abort_);          // h_{t-1} rows of every unit group are visible
        proxy_fence();
        if (cta == 0) stamp(1);
        for (int i = 0; i < nh; ++i, ++it) {
          const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
          wait_mbar(bar_empty + 8 * s, ph ^ 1u, p.err, abort_);
          if (*abort_) break;                                                     // never issue bulk copies into a CTA that is draining
          mbar_expect_tx(bar_full + 8 * s, tx);
          tma_load_2d(ring + s * stage_bytes, &tmX, bar_full + 8 * s, (p.NXB + hb0 + i) * BK, t * B);
        }
        if (nx == 0) continue;                                                   // global mode: the input projection is hoisted
        wait_flag(barB, (unsigned)B * (unsigned)(t + 1), p.err, abort_);       // x_t of every sample is visible
        proxy_fence();
        if (cta == 0) stamp(2);
        for (int i = 0; i < nx; ++i, ++it) {
          const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
          wait_mbar(bar_empty + 8 * s, ph ^ 1u, p.err, abort_);
          if (*abort_) break;
          mbar_expect_tx(bar_full + 8 * s, tx);
          tma_load_2d(ring + s * stage_bytes, &tmX, bar_full + 8 * s, (xb0 + i) * BK, t * B);
        }
      }
    }
  } else if (warp == 5) {
    // ================================ MMA issuer ================================
    // D[n = gate row g*32 + u (M = 128), b = sample (N = NB)] += W[n, k] . act[b, k]: weights are the M-side operand, so every accumulator
    // row is useful and an epilogue warp (TMEM lane quarter) holds ONE gate of 32 consecutive units for all samples -> its stores
    // to the exchange buffer are 128-byte rows (the sample-on-M orientation needed 512-byte-strided stores: 2.2 us per step)
    const int NB = (B + 15) & ~15;
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NB >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    wait_mbar(bar_w, 0, p.err, abort_);
    uint32_t it = 0;
    for (int t = 0; t < S; ++t) {
      for (int i = 0; i < nkb; ++i, ++it) {
        const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
        wait_mbar(bar_full + 8 * s, ph, p.err, abort_);
        tc_fence_after();
        if (lane == 0 && !*abort_) {
          const uint32_t sact = ring + s * stage_bytes, sw = wres + i * WTILE;
#pragma unroll
          for (int kk = 0; kk < BK / UMMA_K; ++kk)
            umma_bf16(tmem_base, umma_smem_desc(sw + kk * (UMMA_K * 2), 16, 1024), umma_smem_desc(sact + kk * (UMMA_K * 2), 16, 1024), idesc,
                      (i > 0 || kk > 0) ? 1u : 0u);
          umma_commit(bar_empty + 8 * s);
          if (i == nkb - 1) umma_commit(bar_tmem);
        }
        __syncwarp();
      }
    }
  } else {
    // ================================ worker warps ================================
    // two separate loops (epilogue warps 0-3 / attention warps 6-13) that meet in cell_query_phase: the attention warps keep
    // their time-invariant operands in registers for the whole kernel, the epilogue warps need theirs for tcgen05.ld
    const bool is_epi = warp < 4;
    CellCtx cq;
    cq.ww = is_epi ? warp : warp - 2;                      // 0..11 in the cell / query phase
    cq.lane = lane; cq.ug = ug; cq.ks = ks; cq.tid = tid; cq.cta = cta;
    cq.ns = (B - ks + KS - 1) / KS;                        // samples b = ks + KS*i owned by this CTA in the cell phase (<= 4 * NWORK)
    cq.j = ug * UNITS + lane;                              // this lane's hidden unit
    {
      const int j = cq.j;
      const float ih = p.global_mode ? 0.f : 1.f;            // global mode: b_ih is already inside Gx
      cq.bi = ih * p.b_ih[j] + p.b_hh[j]; cq.bf_ = ih * p.b_ih[R + j] + p.b_hh[R + j];
      cq.bg = ih * p.b_ih[2 * R + j] + p.b_hh[2 * R + j]; cq.bo = ih * p.b_ih[3 * R + j] + p.b_hh[3 * R + j];
      // W_a fragments of the query mma (B operand, col-major k x n): a = 16 ww + 8 nt + lane/4, units 16 k + 2 (lane%4) (+8)
      if (cq.ww < 8 && !p.global_mode) {
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            const bf16* src = p.Wa + (long long)min(16 * cq.ww + 8 * nt + (lane >> 2), A - 1) * R + ug * UNITS + 16 * k + (lane & 3) * 2;
            cq.wb[4 * nt + 2 * k] = *reinterpret_cast<const uint32_t*>(src);
            cq.wb[4 * nt + 2 * k + 1] = *reinterpret_cast<const uint32_t*>(src + 8);
          }
      }
    }
    float creg[4] = {0.f, 0.f, 0.f, 0.f};                  // cell state of this thread's (sample slot r, unit) cells: never re-read from memory

    if (is_epi) {
      for (int t = 0; t < S; ++t) {
        // ---------------- accumulator -> K-slice partials (warp q holds gate q of the 32 units, all samples) ----------------
        wait_mbar(bar_tmem, (uint32_t)t & 1u, p.err, abort_);
        tc_fence_after();
        if (cta == 0 && tid == 0) stamp(4);
        float* dst = p.XP + ((long long)ug * KS + ks) * B * NCOL + warp * UNITS + lane;
#pragma unroll 1
        for (int c0 = 0; c0 < B; c0 += 64) {                // two 32-column chunks in flight per wait
          uint32_t r[64];
          tmem_ld32_nw(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, r);
          tmem_ld32_nw(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(c0 + 32), r + 32);
          tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 64; ++q)
            if (c0 + q < B) dst[(long long)(c0 + q) * NCOL] = __uint_as_float(r[q]);
        }
        tc_fence_before();
        if (cta == 0 && tid == 0) stamp(10);
        nbar(1, 128);
        if (tid == 0) {
          red_rel(flagX);
          if (cta == 0) stamp(11);
          wait_flag(flagX, (unsigned)KS * (unsigned)(t + 1), p.err, abort_);     // all KS slices of this unit group have landed
          if (cta == 0) stamp(5);
        }
        cell_query_phase<KS>(p, cq, t, creg, hs);
      }
    } else if (cta >= B || p.global_mode) {
      for (int t = 0; t < S; ++t) cell_query_phase<KS>(p, cq, t, creg, hs);
    } else {
      // ---------------- attention of sample b_att = cta (warps 6-13 of the first B CTAs) ----------------
      const int aw = warp - 6, b_att = cta;
      // operands that do not change over the S steps stay in registers: the L value rows of this lane's column pair, U.v of this
      // warp's frames, attn_b / attn_w chunks (lane owns a-chunk [4 lane, 4 lane + 4) of the score dot product)
      const int col = 2 * (aw * 32 + lane);
      const bool col_ok = col < H;
      const float4 ab4 = reinterpret_cast<const float4*>(p.attn_b)[lane], aw4 = reinterpret_cast<const float4*>(p.attn_w)[lane];
      // ... parked in tensor memory (this warp's lane quarter, columns 128 + 48*(aw/4) ..): 48 registers per thread that would
      // otherwise be live across the whole loop; tcgen05.ld brings them back each step (64 B/clk, off the critical loads)
      const uint32_t t_park = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + 128u + 48u * (uint32_t)(aw >> 2);
      {
        uint32_t v[32];
        const bf16* vb = p.Hd + (long long)b_att * H + (col_ok ? col : 0);
#pragma unroll
        for (int l = 0; l < 32; ++l) v[l] = *reinterpret_cast<const uint32_t*>(vb + (long long)min(l, Ln - 1) * B * H);
        tmem_st32(t_park, v);
        uint32_t u[16];
#pragma unroll
        for (int f = 0; f < 4; ++f) {
          float4 x = reinterpret_cast<const float4*>(p.Uv + ((long long)min(aw + 8 * f, Ln - 1) * B + b_att) * A)[lane];
          x = attn::l4_add(x, ab4);                           // attn_b folded in once
          u[4 * f] = __float_as_uint(x.x); u[4 * f + 1] = __float_as_uint(x.y); u[4 * f + 2] = __float_as_uint(x.z); u[4 * f + 3] = __float_as_uint(x.w);
        }
        tmem_st16(t_park + 32u, u);
        tmem_st_wait();
      }
      float dr0 = 1.f, dr1 = 1.f;                          // dropout scales of this lane's two x_t columns for the coming step
      auto draw_dropout = [&](int t) {
        if (p.p_drop > 0.f && col_ok) {
          const uint64_t idx = (uint64_t)((long long)t * B + b_att) * (uint64_t)H + (uint64_t)col;
          const float4 d4 = dropout_scale4(p.rng, p.site, idx & ~3ull, p.p_drop);
          if ((idx & 3ull) == 0) { dr0 = d4.x; dr1 = d4.y; } else { dr0 = d4.z; dr1 = d4.w; }
        }
      };
      draw_dropout(0);
      for (int t = 0; t < S; ++t) {
        float4 wh = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t > 0) {
          if (aw == 0 && lane == 0) { wait_flag(barA, ncta * (unsigned)t, p.err, abort_); if (cta == 0) stamp(12); }
          nbar(5, 256);
          // query = sum of the unit-group partials the cell phase of step t-1 left: warp aw takes groups aw, aw + 8, ..
#pragma unroll
          for (int i0 = 0; i0 < 8; i0 += 4) {
            float4 q[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) q[i] = reinterpret_cast<const float4*>(p.WhP + ((long long)min(aw + 8 * (i0 + i), p.UG - 1) * B + b_att) * A)[lane];
#pragma unroll
            for (int i = 0; i < 4; ++i) if (aw + 8 * (i0 + i) < p.UG) wh = attn::l4_add(wh, q[i]);
          }
        }
        reinterpret_cast<float4*>(whred + aw * 128)[lane] = wh;
        nbar(5, 256);
        wh = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 8; ++i) wh = attn::l4_add(wh, reinterpret_cast<const float4*>(whred + i * 128)[lane]);
        if (aw == 0) reinterpret_cast<float4*>(p.Wh + ((long long)t * B + b_att) * A)[lane] = wh;
        if (cta == 0 && aw == 0 && lane == 0) stamp(13);
        float sc[4];
        uint32_t v[32];
        {
          uint32_t u[16];
          tmem_ld16_nw(t_park + 32u, u);
          tmem_ld32_nw(t_park, v);
          tmem_ld_wait();
#pragma unroll
          for (int f = 0; f < 4; ++f) {
            float s = aw4.x * act_tanh<true>(wh.x + __uint_as_float(u[4 * f]));
            s = fmaf(aw4.y, act_tanh<true>(wh.y + __uint_as_float(u[4 * f + 1])), s);
            s = fmaf(aw4.z, act_tanh<true>(wh.z + __uint_as_float(u[4 * f + 2])), s);
            sc[f] = fmaf(aw4.w, act_tanh<true>(wh.w + __uint_as_float(u[4 * f + 3])), s);
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
          for (int f = 0; f < 4; ++f) sc[f] += __shfl_xor_sync(0xffffffffu, sc[f], o);
        if (lane < 4) {
          const float s = lane == 0 ? sc[0] : lane == 1 ? sc[1] : lane == 2 ? sc[2] : sc[3];
          const int l = aw + 8 * lane;
          if (l < Ln) { e_s[l] = s; if (!SM) p.beta[((long long)t * B + b_att) * Ln + l] = s; }
        }
        nbar(5, 256);
        float al = 0.f;                                     // SM: lane l holds alpha[l]
        if constexpr (SM) {
          al = warp_softmax<true>(e_s[lane], lane < Ln);
          if (aw == 0 && lane < Ln) p.beta[((long long)t * B + b_att) * Ln + lane] = al;
        }
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int l = 0; l < 32; l += 2) {
          if (l < Ln) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v[l]));
            const float e = SM ? __shfl_sync(0xffffffffu, al, l) : e_s[l];
            a0 = fmaf(e, f.x, a0); a1 = fmaf(e, f.y, a1);
          }
          if (l + 1 < Ln) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v[l + 1]));
            const float e = SM ? __shfl_sync(0xffffffffu, al, l + 1) : e_s[l + 1];
            a2 = fmaf(e, f.x, a2); a3 = fmaf(e, f.y, a3);
          }
        }
        if (col_ok)
          *reinterpret_cast<__nv_bfloat162*>(p.X + ((long long)t * B + b_att) * KX + col) =
              __floats2bfloat162_rn((a0 + a2) * p.inv_L * dr0, (a1 + a3) * p.inv_L * dr1);
        if (cta == 0 && aw == 0 && lane == 0) stamp(14);
        nbar(5, 256);                                       // all of x_t[b] written (also protects e_s / whred for the next step)
        if (aw == 0 && lane == 0) { red_rel(barB); if (cta == 0) stamp(3); }
        if (t + 1 < S) draw_dropout(t + 1);                 // Philox for the next step, off the critical path
        cell_query_phase<KS>(p, cq, t, creg, hs);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc(tmem_base, TMEM_COLS);
}

// ---- host side ---------------------------------------------------------------------------------------------------
static inline bool persist_enabled() {
  static const int v = rn_env_int("RECNET_PERSIST", 1);
  return v != 0;
}
static inline int sm_count() {
  static int n = 0;
  if (!n) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); if (n <= 0) n = rt::NUM_SMS; }
  return n;
}
// K-split that keeps every CTA's weight slice resident (<= MAX_KB k-blocks) with UG*KS CTAs co-resident; 0 = shape not covered
static inline int pick_ks(int R, int H) {
  if (R % 64 || H % 64) return 0;
  const int UG = R / UNITS, NHB = R / BK, NXB = H / BK;
  for (int ks = 1; ks <= 4; ++ks) {
    int worst = 0;
    for (int k = 0; k < ks; ++k) {
      const int n = ((NHB * (k + 1)) / ks - (NHB * k) / ks) + ((NXB * (k + 1)) / ks - (NXB * k) / ks);
      worst = n > worst ? n : worst;
    }
    if (worst <= MAX_KB && UG * ks <= sm_count()) return ks;
  }
  return 0;
}
struct Shape { int B, S, R, H, A, L; };
// deepest ring that fits next to res_kb resident k-blocks (at least 2, at most MAX_STAGES); 0 = does not fit
static inline int pick_stages_fwd(int B, int ks, int res_kb) {
  for (int n = MAX_STAGES; n >= 2; --n) if (smem_layout(B, ks, n, res_kb).total <= 227 * 1024) return n;
  return 0;
}
static inline int max_res_kb_fwd(int R, int H, int ks) {
  const int NHB = R / BK, NXB = H / BK;
  int worst = 0;
  for (int k = 0; k < ks; ++k) {
    const int n = ((NHB * (k + 1)) / ks - (NHB * k) / ks) + ((NXB * (k + 1)) / ks - (NXB * k) / ks);
    worst = n > worst ? n : worst;
  }
  return worst;
}
static inline bool global_fwd_ok(int B, int S, int R) {
  if (!persist_enabled()) return false;
  const int ks = pick_ks(R, 0);
  return ks && B >= ks && B <= 128 && S >= 1 && R / UNITS <= MAX_UG && (B + ks - 1) / ks <= 4 * NWORK && pick_stages_fwd(B, ks, max_res_kb_fwd(R, 0, ks)) > 0;
}
static inline bool local_fwd_ok(const Shape& s) {
  if (!persist_enabled()) return false;
  const int ks = pick_ks(s.R, s.H);
  if (!ks) return false;
  const int UG = s.R / UNITS;
  return s.A == 128 && s.B >= ks && s.B <= 128 && s.B <= UG * ks && s.L >= 1 && s.L <= 32 && s.H <= 512 && UG <= MAX_UG && s.S >= 1 &&
         (s.B + ks - 1) / ks <= 4 * NWORK && pick_stages_fwd(s.B, ks, max_res_kb_fwd(s.R, s.H, ks)) > 0;
}
static inline size_t xp_floats(const Shape& s) { const int ks = pick_ks(s.R, s.H); return ks ? (size_t)(s.R / UNITS) * ks * s.B * NCOL : 4; }
static inline size_t whp_floats(const Shape& s) { return (size_t)(s.R / UNITS + 1) * s.B * s.A; }
constexpr int SYNC_WORDS = 64 + 32 * MAX_UG;

template <int KS, bool SM>
static int launch_ks(const CUtensorMap& mx, const CUtensorMap& mw, const FwdParams& p, cudaStream_t st) {
  auto kern = local_fwd_kernel<KS, SM>;
  const int smem = smem_layout(p.B, KS, p.nst, p.res_kb).total;
  static int attr_smem = 0;
  if (attr_smem < smem) {
    RN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_smem = smem;
  }
  void* args[] = {(void*)&mx, (void*)&mw, (void*)&p};
  ProfScope prof(KC_LOOP, p.S, p.UG * KS, 0, st);
  RN_CUDA_OK(cudaLaunchCooperativeKernel((const void*)kern, dim3(p.UG * KS), dim3(THREADS), args, (size_t)smem, st));
  RN_LAUNCH_OK();
  return 0;
}

// X / Wrec as the kernel-per-phase path stages them; sync must be zeroed (SYNC_WORDS words) before the launch
// softmax: the paper's attention (p.inv_L must then be 1)
static int launch_local_fwd(FwdParams p, const bf16* Wrec, bool softmax, cudaStream_t st) {
  p.KS = pick_ks(p.R, p.H);
  p.UG = p.R / UNITS; p.NHB = p.R / BK; p.NXB = p.H / BK; p.KX = p.H + p.R;
  p.res_kb = max_res_kb_fwd(p.R, p.H, p.KS); p.nst = pick_stages_fwd(p.B, p.KS, p.res_kb);
  if (p.nst <= 0) return RECNET_ERR_UNSUPPORTED;
  CUtensorMap mx, mw;
  RN_TRY(make_map(&mx, p.X, (long long)(p.S + 1) * p.B, p.KX, p.KX, BK, p.B));
  RN_TRY(make_map(&mw, Wrec, 4LL * p.R, p.KX, p.KX, BK, UNITS));
  switch (p.KS) {
    case 1: return softmax ? launch_ks<1, true>(mx, mw, p, st) : launch_ks<1, false>(mx, mw, p, st);
    case 2: return softmax ? launch_ks<2, true>(mx, mw, p, st) : launch_ks<2, false>(mx, mw, p, st);
    case 3: return softmax ? launch_ks<3, true>(mx, mw, p, st) : launch_ks<3, false>(mx, mw, p, st);
    case 4: return softmax ? launch_ks<4, true>(mx, mw, p, st) : launch_ks<4, false>(mx, mw, p, st);
  }
  return RECNET_ERR_UNSUPPORTED;
}
// =====================================================================================================================
// BPTT of the same loop, one cooperative launch for all S steps (mirrors local_fwd_kernel).
//   per step t = S-1 .. 0 (reference: autograd of models/local_reconstructor.py:37-55):
//     C  cell backward of (sample, unit) cells          -> dG_t (bf16 operand rows)                      [all CTAs, 12 warps]
//        dh = dHext_t + dX_{t+1}[:, H + j] (sum of the NS K-slice partials) + dWh_{t+1} . W_a (mma.sync, W_a fragments in registers)
//     G  dX_t = dG_t . [W_ih | W_hh]: CTA (cg, ns) keeps the 128 output columns cg x gate-row slice ns of the weight resident
//        (MN-major A operand, <= 11 k-blocks = 176 KB) and leaves its fp32 partial in DP[cg][ns]             [TMA + tcgen05]
//     A  attention backward of one sample: dctx = mask . sum_ns DP[x columns] -> d e -> dWh_t, dU.v, dw     [first B CTAs, 8 warps]
//   three grid-wide flag waits per step (dG ready / partials ready / dWh ready); dU.v and dw accumulate in registers over
//   all steps; V rows and U.v + b of the sample are parked in tensor memory.  Leaves dG, dx, dWh, dWh_op, dUv, dw_acc exactly
//   as the kernel-per-phase path does, so the batched weight-gradient GEMMs after the loop run unchanged.
struct BwdParams {
  int B, S, R, H, A, L, KX, CG, NS, NB4, UG, KT;
  int nst, res_kb;                    // ring stages / resident k-blocks per CTA (set by the launcher)
  float inv_L, p_drop;
  const bf16* Hd; const float* Uv; const bf16* Wa;
  const float *attn_b, *attn_w;
  const float* Wh;                    // [S, B, A]
  const bf16* gates;                  // [S*B, 4R]
  const float* c;                     // [(S+1)*B, R]
  const float* dHext;                 // [S*B, R]
  bf16* dG;                           // [S*B, 4R]
  float* dx;                          // [S, B, H]
  float* dWh; bf16* dWh_op;           // [S, B, A]
  float* dUv;                         // [L, B, A]
  float* dw_acc;                      // [B, A]
  float* DP;                          // [CG][NS][B][128]
  unsigned* sync;                     // [0] dG ready, [32] partials ready, [64] dWh ready
  int* err;
  const unsigned long long* rng;
  unsigned site;
  int global_mode;                    // GLOBAL reconstructor: no attention / query path, H = 0 (dX = dG . W_hh only)
  const float* alpha;                 // [S, B, L] softmax weights of the forward (nullable = the reference's mean)
};
constexpr int MAX_NS = 12;

struct SmemB { int ring, wres, bars, dctx, red, total; };
__host__ __device__ inline SmemB smem_layout_bwd(int B, int nst, int res_kb) {
  SmemB s;
  const int stage = ((B + 7) & ~7) * 128;
  s.ring = 0;
  s.wres = (nst * stage + 1023) & ~1023;
  s.bars = s.wres + res_kb * WTILE;
  s.dctx = s.bars + 256;                           // [512] floats
  s.red = s.dctx + 512 * 4;                        // [8][128] floats
  s.total = s.red + 8 * 128 * 4 + 1024;
  return s;
}

// SM = true: softmax attention (p.alpha, inv_L = 1): d e = alpha (d alpha - sum_l alpha[l] d alpha[l]) before the score backward
template <bool SM>
__global__ void __launch_bounds__(THREADS, 1)
local_bwd_kernel(const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmW, const BwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (base - smem_u32(smem_raw));
  const SmemB L_ = smem_layout_bwd(p.B, p.nst, p.res_kb);
  const uint32_t STAGES = (uint32_t)p.nst;
  const int stage_bytes = ((p.B + 7) & ~7) * 128;
  const uint32_t ring = base + L_.ring, wres = base + L_.wres;
  const uint32_t bar_full = base + L_.bars, bar_empty = bar_full + 8 * MAX_STAGES, bar_tmem = bar_empty + 8 * MAX_STAGES, bar_w = bar_tmem + 8;
  const uint32_t tmem_slot = bar_w + 8;
  volatile int* abort_ = reinterpret_cast<volatile int*>(gen + L_.bars + 192);
  float* dctx_s = reinterpret_cast<float*>(gen + L_.dctx);
  float* red = reinterpret_cast<float*>(gen + L_.red);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cta = blockIdx.x;
  const int B = p.B, S = p.S, R = p.R, H = p.H, A = p.A, Ln = p.L, NS = p.NS;
  const int cg = cta / NS, ns_i = cta % NS;
  const int nb0 = (p.NB4 * ns_i) / NS, nb1 = (p.NB4 * (ns_i + 1)) / NS, nkb = nb1 - nb0;
  const unsigned ncta = gridDim.x;
  unsigned* bar1 = p.sync;            // dG_t of every cell is visible
  unsigned* bar2 = p.sync + 32;       // partials of dX_t are visible
  unsigned* bar3 = p.sync + 64;       // dWh_t of every sample is visible

  if (tid == 0) {
    for (int s = 0; s < MAX_STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    mbar_init(bar_tmem, 1);
    mbar_init(bar_w, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    *abort_ = 0;
  }
  if (warp == 5) tmem_alloc(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 4) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmG)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmW)) : "memory");
      // resident weight slice as an MN-major operand: k-block i = gate rows (nb0+i)*64 .., two boxes {64 columns, 64 rows}
      mbar_expect_tx(bar_w, (uint32_t)nkb * WTILE);
      for (int i = 0; i < nkb; ++i)
#pragma unroll
        for (int jb = 0; jb < 2; ++jb) tma_load_2d(wres + i * WTILE + jb * (BK * 128), &tmW, bar_w, cg * 128 + jb * 64, (nb0 + i) * BK);
      uint32_t it = 0;
      const uint32_t tx = (uint32_t)B * 128u;
      for (int t = S - 1; t >= 0; --t) {
        wait_flag(bar1, ncta * (unsigned)(S - t), p.err, abort_);
        proxy_fence();
        if (cta == 0) stamp(1);
        for (int i = 0; i < nkb; ++i, ++it) {
          const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
          wait_mbar(bar_empty + 8 * s, ph ^ 1u, p.err, abort_);
          if (*abort_) break;
          mbar_expect_tx(bar_full + 8 * s, tx);
          tma_load_2d(ring + s * stage_bytes, &tmG, bar_full + 8 * s, (nb0 + i) * BK, t * B);
        }
      }
    }
  } else if (warp == 5) {
    // ================================ MMA issuer ================================
    // D[m = output column (128), b = sample] += W[n, cg*128 + m] . dG[b, n]   (A MN-major, B K-major)
    const int NB = (B + 15) & ~15;
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | ((uint32_t)(NB >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    wait_mbar(bar_w, 0, p.err, abort_);
    uint32_t it = 0;
    for (int t = S - 1; t >= 0; --t) {
      for (int i = 0; i < nkb; ++i, ++it) {
        const uint32_t s = it % STAGES, ph = (it / STAGES) & 1u;
        wait_mbar(bar_full + 8 * s, ph, p.err, abort_);
        tc_fence_after();
        if (lane == 0 && !*abort_) {
          const uint32_t sact = ring + s * stage_bytes, sw = wres + i * WTILE;
#pragma unroll
          for (int kk = 0; kk < BK / UMMA_K; ++kk)
            umma_bf16(tmem_base, umma_smem_desc(sw + kk * (UMMA_K * 128), BK * 128, 1024), umma_smem_desc(sact + kk * (UMMA_K * 2), 16, 1024), idesc,
                      (i > 0 || kk > 0) ? 1u : 0u);
          umma_commit(bar_empty + 8 * s);
          if (i == nkb - 1) umma_commit(bar_tmem);
        }
        __syncwarp();
      }
    }
  } else {
    // ================================ worker warps ================================
    const bool is_epi = warp < 4;
    const bool glob = p.global_mode != 0;
    const bool do_attn = !is_epi && cta < B && !glob;
    const int ww = is_epi ? warp : warp - 2;               // 0..11 in the cell phase
    const int aw = warp - 6;                                // 0..7 in the attention phase
    const int gid = lane >> 2, tig = lane & 3;
    // ---- cell-phase role: unit group ug, sample class kt (samples b = kt + KT*i); warp (mt, nt) owns the mma tile of sample slots
    //      16 mt .. +15 x units 8 nt .. +7; thread cells: slots i0 = 16 mt + gid, i1 = i0 + 8, units 8 nt + 2 tig (+1)
    const int KT = p.KT, ug = cta / KT, kt = cta % KT;
    const int nsl = (B - kt + KT - 1) / KT;                 // sample slots of this CTA (<= 48)
    const int mt = ww >> 2, nt = ww & 3;
    const int i0 = 16 * mt + gid, i1 = i0 + 8;
    const bool ok0 = i0 < nsl, ok1 = i1 < nsl;
    const int b0 = kt + KT * min(i0, nsl - 1), b1 = kt + KT * min(i1, nsl - 1);
    const int j = ug * UNITS + 8 * nt + 2 * tig;            // first of this thread's two units
    const int kcol = H + j, cgj = kcol >> 7, colj = kcol & 127;
    // W_a fragments (B operand of mma.m16n8k16, k = a, n = unit): b0b1 = W_a[16 ks + 2 tig (+1)][unit 8 nt + gid], b2b3 = rows + 8
    uint32_t wb[16];
    if (glob) {
#pragma unroll
      for (int i = 0; i < 16; ++i) wb[i] = 0u;
    } else {
      const unsigned short* W = reinterpret_cast<const unsigned short*>(p.Wa) + ug * UNITS + 8 * nt + gid;
#pragma unroll
      for (int ks8 = 0; ks8 < 8; ++ks8) {
        const int a0 = 16 * ks8 + 2 * tig;
        wb[2 * ks8] = (uint32_t)W[(long long)min(a0, A - 1) * R] | ((uint32_t)W[(long long)min(a0 + 1, A - 1) * R] << 16);
        wb[2 * ks8 + 1] = (uint32_t)W[(long long)min(a0 + 8, A - 1) * R] | ((uint32_t)W[(long long)min(a0 + 9, A - 1) * R] << 16);
      }
    }
    float dcc[4] = {0.f, 0.f, 0.f, 0.f};                    // carry dc of this thread's 4 cells (rows 0/1 x units 0/1)
    // ---- attention role (warps 6-13 of the first B CTAs): sample b_att = cta; warp aw owns frames aw + 8 f; lane owns 16-byte
    //      chunks lane, lane + 32 of the value rows and a-chunk [4 lane, +4) of the score
    const int b_att = cta;
    float4 aw4 = make_float4(0.f, 0.f, 0.f, 0.f);
    float duv[4][4], dww[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int f = 0; f < 4; ++f) { duv[f][0] = duv[f][1] = duv[f][2] = duv[f][3] = 0.f; }
    const uint32_t t_park = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + 128u + 48u * (uint32_t)(max(aw, 0) >> 2);
    const int acol = 2 * (aw * 32 + lane);                  // this thread's pair of dctx columns
    float dr0 = 1.f, dr1 = 1.f;
    auto draw_dropout = [&](int t) {
      if (p.p_drop > 0.f && acol < H) {
        const uint64_t idx = (uint64_t)((long long)t * B + b_att) * (uint64_t)H + (uint64_t)acol;
        const float4 d4 = dropout_scale4(p.rng, p.site, idx & ~3ull, p.p_drop);
        if ((idx & 3ull) == 0) { dr0 = d4.x; dr1 = d4.y; } else { dr0 = d4.z; dr1 = d4.w; }
      }
    };
    if (do_attn) {
      aw4 = reinterpret_cast<const float4*>(p.attn_w)[lane];
      const float4 ab4 = reinterpret_cast<const float4*>(p.attn_b)[lane];
      uint32_t v[32];
      const int nch = H >> 3;
#pragma unroll
      for (int f = 0; f < 4; ++f)
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int ch = lane + 32 * u;
          uint4 raw = *reinterpret_cast<const uint4*>(p.Hd + ((long long)min(aw + 8 * f, Ln - 1) * B + b_att) * H + (long long)min(ch, nch - 1) * 8);
          if (ch >= nch || aw + 8 * f >= Ln) raw = make_uint4(0u, 0u, 0u, 0u);
          v[8 * f + 4 * u] = raw.x; v[8 * f + 4 * u + 1] = raw.y; v[8 * f + 4 * u + 2] = raw.z; v[8 * f + 4 * u + 3] = raw.w;
        }
      tmem_st32(t_park, v);
      uint32_t u16[16];
#pragma unroll
      for (int f = 0; f < 4; ++f) {
        float4 x = reinterpret_cast<const float4*>(p.Uv + ((long long)min(aw + 8 * f, Ln - 1) * B + b_att) * A)[lane];
        x = attn::l4_add(x, ab4);
        u16[4 * f] = __float_as_uint(x.x); u16[4 * f + 1] = __float_as_uint(x.y); u16[4 * f + 2] = __float_as_uint(x.z); u16[4 * f + 3] = __float_as_uint(x.w);
      }
      tmem_st16(t_park + 32u, u16);
      tmem_st_wait();
      draw_dropout(S - 1);
    }

    for (int t = S - 1; t >= 0; --t) {
      const bool last = (t == S - 1);
      // ======================= C: cell backward of step t =======================
      {
        const long long r0 = (long long)t * B + b0, r1 = (long long)t * B + b1;
        float dh[2][2];
        uint32_t gq[2][4];
        float2 cp[2], cn[2];
        if (!last) {
          // partials of dX_{t+1} are visible once bar2 of step t+1 completed (attention warps of the first B CTAs saw that already)
          if (is_epi) { if (tid == 0) wait_flag(bar2, ncta * (unsigned)(S - 1 - t), p.err, abort_); nbar(1, 128); }
          else if (!do_attn) { if (aw == 0 && lane == 0) wait_flag(bar2, ncta * (unsigned)(S - 1 - t), p.err, abort_); nbar(5, 256); }
        }
        // everything that does not depend on dWh_{t+1}: issued before the wait for it
        {
          const float2 e0 = *reinterpret_cast<const float2*>(p.dHext + r0 * R + j), e1 = *reinterpret_cast<const float2*>(p.dHext + r1 * R + j);
          dh[0][0] = e0.x; dh[0][1] = e0.y; dh[1][0] = e1.x; dh[1][1] = e1.y;
          const bf16* g0 = p.gates + r0 * 4 * R + j; const bf16* g1 = p.gates + r1 * 4 * R + j;
#pragma unroll
          for (int g = 0; g < 4; ++g) { gq[0][g] = *reinterpret_cast<const uint32_t*>(g0 + (long long)g * R); gq[1][g] = *reinterpret_cast<const uint32_t*>(g1 + (long long)g * R); }
          cp[0] = *reinterpret_cast<const float2*>(p.c + r0 * R + j); cp[1] = *reinterpret_cast<const float2*>(p.c + r1 * R + j);
          cn[0] = *reinterpret_cast<const float2*>(p.c + (r0 + B) * R + j); cn[1] = *reinterpret_cast<const float2*>(p.c + (r1 + B) * R + j);
          if (!last) {
            const float* q0 = p.DP + ((long long)cgj * NS * B + b0) * 128 + colj;
            const float* q1 = p.DP + ((long long)cgj * NS * B + b1) * 128 + colj;
            float2 pa[MAX_NS], pb[MAX_NS];
#pragma unroll
            for (int s = 0; s < MAX_NS; ++s) {
              pa[s] = *reinterpret_cast<const float2*>(q0 + (long long)min(s, NS - 1) * B * 128);
              pb[s] = *reinterpret_cast<const float2*>(q1 + (long long)min(s, NS - 1) * B * 128);
            }
#pragma unroll
            for (int s = 0; s < MAX_NS; ++s)
              if (s < NS) { dh[0][0] += pa[s].x; dh[0][1] += pa[s].y; dh[1][0] += pb[s].x; dh[1][1] += pb[s].y; }
          }
        }
        if (!last && !glob) {
          // dWh_{t+1} . W_a over this CTA's 32 units: [slots x 128 a] . [128 a x 32 units], A fragments straight from dWh_op (L2)
          if (is_epi) { if (tid == 0) wait_flag(bar3, (unsigned)B * (unsigned)(S - 1 - t), p.err, abort_); nbar(1, 128); }
          else { if (aw == 0 && lane == 0) wait_flag(bar3, (unsigned)B * (unsigned)(S - 1 - t), p.err, abort_); nbar(5, 256); }
          if (cta == 0 && tid == 0) stamp(7);
          const bf16* a0p = p.dWh_op + ((long long)(t + 1) * B + b0) * A + 2 * tig;
          const bf16* a1p = p.dWh_op + ((long long)(t + 1) * B + b1) * A + 2 * tig;
          uint32_t af[8][4];
#pragma unroll
          for (int k8 = 0; k8 < 8; ++k8) {
            af[k8][0] = *reinterpret_cast<const uint32_t*>(a0p + 16 * k8);
            af[k8][1] = *reinterpret_cast<const uint32_t*>(a1p + 16 * k8);
            af[k8][2] = *reinterpret_cast<const uint32_t*>(a0p + 16 * k8 + 8);
            af[k8][3] = *reinterpret_cast<const uint32_t*>(a1p + 16 * k8 + 8);
          }
          float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
          for (int k8 = 0; k8 < 8; ++k8)
            asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                         : "+f"(d0), "+f"(d1), "+f"(d2), "+f"(d3)
                         : "r"(af[k8][0]), "r"(af[k8][1]), "r"(af[k8][2]), "r"(af[k8][3]), "r"(wb[2 * k8]), "r"(wb[2 * k8 + 1]));
          dh[0][0] += d0; dh[0][1] += d1; dh[1][0] += d2; dh[1][1] += d3;
        }
        // cell backward (lstm_cell.cuh:lstm_cell_bwd_body), 2 sample rows x 2 units
#pragma unroll
        for (int r = 0; r < 2; ++r) {
          const bool ok = r == 0 ? ok0 : ok1;
          const long long row = r == 0 ? r0 : r1;
          uint32_t og[4];
          const float cpx[2] = {cp[r].x, cp[r].y}, cnx[2] = {cn[r].x, cn[r].y};
          float o4[4][2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const float gi = __bfloat162float(__ushort_as_bfloat16((unsigned short)(u ? gq[r][0] >> 16 : gq[r][0] & 0xFFFFu)));
            const float gf = __bfloat162float(__ushort_as_bfloat16((unsigned short)(u ? gq[r][1] >> 16 : gq[r][1] & 0xFFFFu)));
            const float gg = __bfloat162float(__ushort_as_bfloat16((unsigned short)(u ? gq[r][2] >> 16 : gq[r][2] & 0xFFFFu)));
            const float go = __bfloat162float(__ushort_as_bfloat16((unsigned short)(u ? gq[r][3] >> 16 : gq[r][3] & 0xFFFFu)));
            const float dhv = dh[r][u];
            const float tc = act_tanh<true>(cnx[u]);
            const float dc = fmaf(dhv * go, 1.f - tc * tc, last ? 0.f : dcc[2 * r + u]);
            dcc[2 * r + u] = dc * gf;
            o4[0][u] = dc * gg * gi * (1.f - gi);
            o4[1][u] = dc * cpx[u] * gf * (1.f - gf);
            o4[2][u] = dc * gi * (1.f - gg * gg);
            o4[3][u] = dhv * tc * go * (1.f - go);
          }
#pragma unroll
          for (int g = 0; g < 4; ++g) { const __nv_bfloat162 x = __floats2bfloat162_rn(o4[g][0], o4[g][1]); og[g] = *reinterpret_cast<const uint32_t*>(&x); }
          if (ok) {
            bf16* dg = p.dG + row * 4 * R + j;
#pragma unroll
            for (int g = 0; g < 4; ++g) *reinterpret_cast<uint32_t*>(dg + (long long)g * R) = og[g];
          }
        }
        if (cta == 0 && tid == 0) stamp(8);
        nbar(4, NWORK * 32);
        if (tid == 0) { red_rel(bar1); if (cta == 0) stamp(9); }
      }
      // ======================= G epilogue: accumulator -> DP[cg][ns] (warp q: columns 32 q + lane, all samples) =======================
      if (is_epi) {
        wait_mbar(bar_tmem, (uint32_t)(S - 1 - t) & 1u, p.err, abort_);
        tc_fence_after();
        if (cta == 0 && tid == 0) stamp(4);
        float* dst = p.DP + ((long long)cg * NS + ns_i) * B * 128 + warp * 32 + lane;
#pragma unroll 1
        for (int c0 = 0; c0 < B; c0 += 64) {
          uint32_t r[64];
          tmem_ld32_nw(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, r);
          tmem_ld32_nw(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(c0 + 32), r + 32);
          tmem_ld_wait();
#pragma unroll
          for (int q = 0; q < 64; ++q)
            if (c0 + q < B) dst[(long long)(c0 + q) * 128] = __uint_as_float(r[q]);
        }
        tc_fence_before();
        nbar(1, 128);
        if (tid == 0) { red_rel(bar2); if (cta == 0) stamp(5); }
      }
      // ======================= A: attention backward of sample b_att, step t =======================
      if (do_attn) {
        float al[4];
        if constexpr (SM) {
#pragma unroll
          for (int f = 0; f < 4; ++f) al[f] = aw + 8 * f < Ln ? p.alpha[((long long)t * B + b_att) * Ln + aw + 8 * f] : 0.f;
        }
        if (aw == 0 && lane == 0) { wait_flag(bar2, ncta * (unsigned)(S - t), p.err, abort_); if (cta == 0) stamp(12); }
        nbar(5, 256);
        const float4 wh = reinterpret_cast<const float4*>(p.Wh + ((long long)t * B + b_att) * A)[lane];
        // dctx = dropout mask . sum of the NS partials of the x columns (2 columns per thread)
        if (acol < H) {
          const float* q = p.DP + ((long long)(acol >> 7) * NS * B + b_att) * 128 + (acol & 127);
          float2 pa[MAX_NS];
#pragma unroll
          for (int s = 0; s < MAX_NS; ++s) pa[s] = *reinterpret_cast<const float2*>(q + (long long)min(s, NS - 1) * B * 128);
          float sx = 0.f, sy = 0.f;
#pragma unroll
          for (int s = 0; s < MAX_NS; ++s) if (s < NS) { sx += pa[s].x; sy += pa[s].y; }
          sx *= dr0; sy *= dr1;
          *reinterpret_cast<float2*>(dctx_s + acol) = make_float2(sx, sy);
          *reinterpret_cast<float2*>(p.dx + ((long long)t * B + b_att) * H + acol) = make_float2(sx, sy);
        }
        nbar(5, 256);
        // d e[l] = (1/L) <dctx, v_l> for this warp's frames
        float de[4] = {0.f, 0.f, 0.f, 0.f};
        uint32_t u16[16];
        {
          uint32_t v[32];
          tmem_ld32_nw(t_park, v);
          tmem_ld16_nw(t_park + 32u, u16);
          tmem_ld_wait();
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const float4 x0 = *reinterpret_cast<const float4*>(dctx_s + (lane + 32 * u) * 8), x1 = *reinterpret_cast<const float4*>(dctx_s + (lane + 32 * u) * 8 + 4);
#pragma unroll
            for (int f = 0; f < 4; ++f) {
              const float2 p0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v[8 * f + 4 * u]));
              const float2 p1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v[8 * f + 4 * u + 1]));
              const float2 p2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v[8 * f + 4 * u + 2]));
              const float2 p3 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v[8 * f + 4 * u + 3]));
              float a = de[f];
              a = fmaf(x0.x, p0.x, a); a = fmaf(x0.y, p0.y, a); a = fmaf(x0.z, p1.x, a); a = fmaf(x0.w, p1.y, a);
              a = fmaf(x1.x, p2.x, a); a = fmaf(x1.y, p2.y, a); a = fmaf(x1.z, p3.x, a); a = fmaf(x1.w, p3.y, a);
              de[f] = a;
            }
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
          for (int f = 0; f < 4; ++f) de[f] += __shfl_xor_sync(0xffffffffu, de[f], o);
        if constexpr (SM) {           // de = d alpha so far; the sum over all frames meets in `red` (free here: last read before the previous barrier)
          float s1 = 0.f;
#pragma unroll
          for (int f = 0; f < 4; ++f) s1 = fmaf(al[f], de[f], s1);
          if (lane == 0) red[aw] = s1;
          nbar(5, 256);
          float tot = 0.f;
#pragma unroll
          for (int i = 0; i < 8; ++i) tot += red[i];
          nbar(5, 256);               // every warp has read red before it is rewritten below
#pragma unroll
          for (int f = 0; f < 4; ++f) de[f] = al[f] * (de[f] - tot);
        }
        // score backward of the same frames (tanh recomputed)
        float4 dwh = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int f = 0; f < 4; ++f) {
          if (aw + 8 * f < Ln) {
            const float g = de[f] * p.inv_L;
            const float tx = act_tanh<true>(wh.x + __uint_as_float(u16[4 * f])), ty = act_tanh<true>(wh.y + __uint_as_float(u16[4 * f + 1]));
            const float tz = act_tanh<true>(wh.z + __uint_as_float(u16[4 * f + 2])), tw = act_tanh<true>(wh.w + __uint_as_float(u16[4 * f + 3]));
            const float sx = g * aw4.x * (1.f - tx * tx), sy = g * aw4.y * (1.f - ty * ty), sz = g * aw4.z * (1.f - tz * tz), sw_ = g * aw4.w * (1.f - tw * tw);
            dwh.x += sx; dwh.y += sy; dwh.z += sz; dwh.w += sw_;
            dww[0] = fmaf(g, tx, dww[0]); dww[1] = fmaf(g, ty, dww[1]); dww[2] = fmaf(g, tz, dww[2]); dww[3] = fmaf(g, tw, dww[3]);
            duv[f][0] += sx; duv[f][1] += sy; duv[f][2] += sz; duv[f][3] += sw_;
          }
        }
        reinterpret_cast<float4*>(red + aw * 128)[lane] = dwh;
        nbar(5, 256);
        if (aw == 0) {
          float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 8; ++i) sum = attn::l4_add(sum, reinterpret_cast<const float4*>(red + i * 128)[lane]);
          reinterpret_cast<float4*>(p.dWh + ((long long)t * B + b_att) * A)[lane] = sum;
          const __nv_bfloat162 lo = __floats2bfloat162_rn(sum.x, sum.y), hi = __floats2bfloat162_rn(sum.z, sum.w);
          *reinterpret_cast<uint2*>(p.dWh_op + ((long long)t * B + b_att) * A + 4 * lane) =
              make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
        }
        nbar(5, 256);
        if (aw == 0 && lane == 0) { red_rel(bar3); if (cta == 0) stamp(3); }
        if (t > 0) draw_dropout(t - 1);
      }
    }
    // ---- accumulated over all steps: dU.v of this warp's frames, dw of the sample (summed over the 8 warps) ----
    if (do_attn) {
#pragma unroll
      for (int f = 0; f < 4; ++f)
        if (aw + 8 * f < Ln)
          reinterpret_cast<float4*>(p.dUv + ((long long)(aw + 8 * f) * B + b_att) * A)[lane] = make_float4(duv[f][0], duv[f][1], duv[f][2], duv[f][3]);
      nbar(5, 256);
      reinterpret_cast<float4*>(red + aw * 128)[lane] = make_float4(dww[0], dww[1], dww[2], dww[3]);
      nbar(5, 256);
      if (aw == 0) {
        float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 8; ++i) sum = attn::l4_add(sum, reinterpret_cast<const float4*>(red + i * 128)[lane]);
        reinterpret_cast<float4*>(p.dw_acc + (long long)b_att * A)[lane] = sum;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) tmem_dealloc(tmem_base, TMEM_COLS);
}

// gate-row split that keeps every CTA's weight slice resident with CG*NS CTAs co-resident; 0 = shape not covered
static inline int pick_ns(int R, int H) {
  const int KX = R + H;
  if (KX % 128 || R % 64 || R % UNITS) return 0;
  const int CG = KX / 128, NB4 = 4 * R / BK, UG = R / UNITS;
  for (int ns = MAX_NS; ns >= 1; --ns)                      // as many CTAs as fit: shortest gate-row slice per CTA
    if ((NB4 + ns - 1) / ns <= MAX_KB && CG * ns <= sm_count() && (CG * ns) % UG == 0) return ns;
  return 0;
}
static inline int pick_stages_bwd(int B, int res_kb) {
  for (int n = MAX_STAGES; n >= 2; --n) if (smem_layout_bwd(B, n, res_kb).total <= 227 * 1024) return n;
  return 0;
}
static inline bool global_bwd_ok(int B, int S, int R) {
  if (!persist_enabled()) return false;
  const int ns = pick_ns(R, 0);
  if (!ns) return false;
  const int KT = (R / 128) * ns / (R / UNITS);
  return B >= KT && B <= 128 && S >= 1 && (B + KT - 1) / KT <= 48 && pick_stages_bwd(B, (4 * R / BK + ns - 1) / ns) > 0;
}
static inline bool local_bwd_ok(const Shape& s) {
  if (!persist_enabled()) return false;
  const int ns = pick_ns(s.R, s.H);
  if (!ns || s.R % UNITS) return false;
  const int G = (s.R + s.H) / 128 * ns, UG = s.R / UNITS;
  if (G % UG) return false;
  const int KT = G / UG;
  return s.A == 128 && s.B >= KT && s.B <= 128 && s.B <= G && s.L >= 1 && s.L <= 32 && s.H <= 512 && s.H % 8 == 0 && s.S >= 1 &&
         (s.B + KT - 1) / KT <= 48 && pick_stages_bwd(s.B, (4 * s.R / BK + ns - 1) / ns) > 0;
}
static inline size_t dp_floats(const Shape& s) { const int ns = pick_ns(s.R, s.H); return ns ? (size_t)((s.R + s.H) / 128) * ns * s.B * 128 : 4; }

// dG / Wrec as the kernel-per-phase path lays them out; sync must be zeroed (SYNC_WORDS words) before the launch
template <bool SM>
static int launch_local_bwd_sm(BwdParams p, const bf16* Wrec, cudaStream_t st) {
  p.KX = p.H + p.R; p.NS = pick_ns(p.R, p.H); p.CG = p.KX / 128; p.NB4 = 4 * p.R / BK; p.UG = p.R / UNITS; p.KT = p.CG * p.NS / p.UG;
  CUtensorMap mg, mw;
  RN_TRY(make_map(&mg, p.dG, (long long)p.S * p.B, 4LL * p.R, 4LL * p.R, BK, p.B));
  RN_TRY(make_map(&mw, Wrec, 4LL * p.R, p.KX, p.KX, 64, BK));
  p.res_kb = (p.NB4 + p.NS - 1) / p.NS; p.nst = pick_stages_bwd(p.B, p.res_kb);
  if (p.nst <= 0) return RECNET_ERR_UNSUPPORTED;
  const int smem = smem_layout_bwd(p.B, p.nst, p.res_kb).total;
  static int attr_smem = 0;
  if (attr_smem < smem) {
    RN_CUDA_OK(cudaFuncSetAttribute(local_bwd_kernel<SM>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_smem = smem;
  }
  void* args[] = {(void*)&mg, (void*)&mw, (void*)&p};
  ProfScope prof(KC_LOOP, p.S, p.CG * p.NS, 1, st);
  RN_CUDA_OK(cudaLaunchCooperativeKernel((const void*)local_bwd_kernel<SM>, dim3(p.CG * p.NS), dim3(THREADS), args, (size_t)smem, st));
  RN_LAUNCH_OK();
  return 0;
}
// p.alpha != nullptr: softmax attention (p.inv_L must then be 1)
static int launch_local_bwd(const BwdParams& p, const bf16* Wrec, cudaStream_t st) {
  return p.alpha ? launch_local_bwd_sm<true>(p, Wrec, st) : launch_local_bwd_sm<false>(p, Wrec, st);
}
}  // namespace rp
