// Persistent tcgen05 GEMM for the BATCHED products of a train step (hoisted projections, vocabulary projection, weight gradients).
//
//   C[m,n] (+)= sum_k A(m,k) * B(n,k) (+ bias[n])          same operand conventions and epilogue options as gemm_tc.cuh (no split-K)
//
// What differs from tc::gemm_tc_kernel (one tile per CTA, kept for the per-step and split-K GEMMs):
//   * static persistent schedule: one CTA (or CTA pair) per SM walks tiles t = unit, unit + n_units, ...; the TMA ring keeps running
//     across tile boundaries, so the prologue latency (tensormap fetch, first TMA round trip) is paid once per CTA, not once per tile;
//   * two TMEM accumulators (2 x BN columns): the four epilogue warps drain tile j while the MMA thread already accumulates tile j+1;
//   * the epilogue never touches global memory with thread stores: each warp moves its 32 rows x 128 bytes of the accumulator from
//     TMEM to a swizzled shared-memory pad (8 st.shared.v4 per lane) and one lane hands the pad to the TMA store engine
//     (cp.async.bulk.tensor, or cp.reduce...add for accumulate), which also clips the M / N edges.  ~50 instructions per block instead
//     of ~360: with ONE epilogue warp per SM sub-partition every dependent instruction's latency is exposed, and the r1 epilogue
//     (scattered 16-byte stores, 8192 LSU wavefronts per 128 x 256 tile) took longer than the tile's MMAs at K = 512;
//   * CTAS = 2: the two CTAs of a cluster (one TPC) share a 256 x BN tile through tcgen05.mma.cta_group::2 -- each loads its own 128
//     rows of A and HALF of the B tile, the leader's MMA reads both halves.  Per CTA and 64-deep k-block that is 16 + BN/4 KB instead
//     of 16 + BN/2 KB for the same tensor work: the batched main loops are L2->SM delivery bound (profiles/r1_g_gemm_sweep.md).
// Warp roles: 0 = TMA producer, 1 = TMEM allocator + MMA issuer (leader CTA only), 2..5 = epilogue.
#pragma once
#include "gemm_tc.cuh"

namespace tc2 {
using tc::BK;
using tc::BM;
using tc::UMMA_K;
using tc::EpiArgs;
using tc::mbar_init;
using tc::mbar_wait;
using tc::mbar_expect_tx;
using tc::smem_u32;
using tc::tc_fence_after;
using tc::tc_fence_before;
using tc::umma_smem_desc;
constexpr int THREADS = 192;
constexpr int TC2_SMS = 148;          // B200: one CTA (or half a pair) per SM

__device__ __forceinline__ uint32_t mapa0(uint32_t addr) {           // same offset in CTA 0 of the cluster
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, 0;" : "=r"(r) : "r"(addr));
  return r;
}
template <int CTAS>
__device__ __forceinline__ void tma_load(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  if (CTAS == 1) {
    tc::tma_load_2d(dst, map, bar, c0, c1);
  } else {           // both CTAs of the pair complete their bytes on the LEADER's barrier
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
  }
}
template <int CTAS>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  if (CTAS == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int CTAS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if (CTAS == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
template <int CTAS>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  if (CTAS == 1) {
    tc::umma_bf16(tmem_d, adesc, bdesc, idesc, accum);
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
        : "memory");
  }
}
template <int CTAS>
__device__ __forceinline__ void commit(uint32_t bar) {       // CTAS = 2: arrives on the barrier at this offset in BOTH CTAs
  if (CTAS == 1) {
    tc::umma_commit(bar);
  } else {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"((uint16_t)3) : "memory");
  }
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive_local(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t* r) {
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
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

template <int BN, int STAGES, int CTAS>
struct Smem {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = (BN / CTAS) * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int PAD_OFF = STAGES * STAGE_BYTES;              // 4 epilogue warps x 2 x 4 KB store pads (32 rows x 128 B, swizzled)
  static constexpr int BAR_OFF = PAD_OFF + 8 * 4096;
  static constexpr int TOTAL = BAR_OFF + (2 * STAGES + 4) * 8 + 16 + 1024;
};

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1, bool add) {
  if (!add)
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1) : "memory");
  else
    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(map)), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16(uint32_t lo, uint32_t hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(__uint_as_float(lo), __uint_as_float(hi));
  return *reinterpret_cast<uint32_t*>(&v);
}
// r[0..31] += bias[n .. n+31] (columns >= N untouched: the TMA store clips them)
__device__ __forceinline__ void add_bias32(uint32_t* r, const float* __restrict__ bias, int n, int N, int vec_ok) {
  if (vec_ok && n + 32 <= N) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 b4 = __ldg(reinterpret_cast<const float4*>(bias + n) + j);
      r[4 * j] = __float_as_uint(__uint_as_float(r[4 * j]) + b4.x);
      r[4 * j + 1] = __float_as_uint(__uint_as_float(r[4 * j + 1]) + b4.y);
      r[4 * j + 2] = __float_as_uint(__uint_as_float(r[4 * j + 2]) + b4.z);
      r[4 * j + 3] = __float_as_uint(__uint_as_float(r[4 * j + 3]) + b4.w);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (n + j < N) r[j] = __float_as_uint(__uint_as_float(r[j]) + __ldg(bias + n + j));
  }
}

template <int BN, int STAGES, bool TA, bool TB, int CTAS, bool OUTB>
__global__ void __launch_bounds__(THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
                EpiArgs ep, int M, int N, int K, int tiles_m, int tiles_n) {
  using L = Smem<BN, STAGES, CTAS>;
  constexpr int BNL = BN / CTAS;                       // B rows this CTA loads
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = base + L::BAR_OFF;
  const uint32_t bar_empty = bar_full + 8 * STAGES;
  const uint32_t bar_tfull = bar_empty + 8 * STAGES;   // [2] accumulator a complete   (MMA -> epilogue, every CTA of the pair)
  const uint32_t bar_tempty = bar_tfull + 16;          // [2] accumulator a drained    (epilogue warps of the pair -> leader's MMA thread)
  const uint32_t tmem_slot = bar_tempty + 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = CTAS == 2 ? (int)tc::cluster_rank() : 0;
  const int unit = blockIdx.x / CTAS, n_units = gridDim.x / CTAS;
  const int n_tiles = tiles_m * tiles_n;
  const int nkb = (K + BK - 1) / BK;

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmC)) : "memory");
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + 8 * a, 1); mbar_init(bar_tempty + 8 * a, 4 * CTAS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc<CTAS>(tmem_slot, 2 * BN);
  tc_fence_before();
  if (CTAS == 2) tc::cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    if (lane == 0) {
      int it = 0;
      for (int t = unit; t < n_tiles; t += n_units) {
        const int m0 = ((t / tiles_n) * CTAS + rank) * BM;
        const int n0 = (t % tiles_n) * BN + rank * BNL;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(bar_empty + 8 * s, (((uint32_t)(it / STAGES)) & 1u) ^ 1u);
          const uint32_t fb = CTAS == 2 ? mapa0(bar_full + 8 * s) : bar_full + 8 * s;
          if (rank == 0) mbar_expect_tx(bar_full + 8 * s, L::STAGE_BYTES * CTAS);
          const uint32_t sa = base + s * L::STAGE_BYTES, sb = sa + L::A_BYTES;
          const int k = kb * BK;
          if (!TA) {
            tma_load<CTAS>(sa, &tmA, fb, k, m0);                                  // box {64 k, 128 m}
          } else {
#pragma unroll
            for (int j = 0; j < BM / 64; ++j) tma_load<CTAS>(sa + j * (BK * 128), &tmA, fb, m0 + j * 64, k);   // boxes {64 m, 64 k}
          }
          if (!TB) {
            tma_load<CTAS>(sb, &tmB, fb, k, n0);                                  // box {64 k, BNL n}
          } else {
#pragma unroll
            for (int j = 0; j < BNL / 64; ++j) tma_load<CTAS>(sb + j * (BK * 128), &tmB, fb, n0 + j * 64, k);  // boxes {64 n, 64 k}
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      // instruction descriptor: D=f32, A=B=bf16, majors, N>>3 @17, M>>4 @24 (M = 128 per CTA: 256 for the pair)
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((TA ? 1u : 0u) << 15) | ((TB ? 1u : 0u) << 16) |
                             ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((BM * CTAS) >> 4) << 24);
      int it = 0, j = 0;
      for (int t = unit; t < n_tiles; t += n_units, ++j) {
        const int a = j & 1;
        mbar_wait(bar_tempty + 8 * a, (((uint32_t)(j >> 1)) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t acc = tmem_base + (uint32_t)(a * BN);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          mbar_wait(bar_full + 8 * s, ((uint32_t)(it / STAGES)) & 1u);
          tc_fence_after();
          const uint32_t sa = base + s * L::STAGE_BYTES, sb = sa + L::A_BYTES;
#pragma unroll
          for (int kk = 0; kk < BK / UMMA_K; ++kk) {
            const uint64_t ad = TA ? umma_smem_desc(sa + kk * (UMMA_K * 128), BK * 128, 1024)
                                   : umma_smem_desc(sa + kk * (UMMA_K * 2), 16, 1024);
            const uint64_t bd = TB ? umma_smem_desc(sb + kk * (UMMA_K * 128), BK * 128, 1024)
                                   : umma_smem_desc(sb + kk * (UMMA_K * 2), 16, 1024);
            umma<CTAS>(acc, ad, bd, idesc, (kb > 0 || kk > 0) ? 1u : 0u);
          }
          commit<CTAS>(bar_empty + 8 * s);
        }
        commit<CTAS>(bar_tfull + 8 * a);
      }
    }
    __syncwarp();
  } else {
    // ---- epilogue: warp w owns TMEM lanes (w % 4) * 32 .. +31 == 32 rows of the tile ----
    constexpr int CW = OUTB ? 64 : 32;                 // output columns per staged block: 128 bytes per row either way
    const int q = warp & 3;
    const uint32_t pad = base + L::PAD_OFF + (uint32_t)(warp - 2) * 8192u;
    const uint32_t te = CTAS == 2 ? mapa0(bar_tempty) : bar_tempty;
    const uint32_t prow = (uint32_t)lane * 128u;
    const int sw = lane & 7;
    const bool add = ep.accumulate != 0;
    int j = 0, blk = 0;
    for (int t = unit; t < n_tiles; t += n_units, ++j) {
      const int a = j & 1;
      const int m0 = ((t / tiles_n) * CTAS + rank) * BM + q * 32;
      const int n0 = (t % tiles_n) * BN;
      mbar_wait(bar_tfull + 8 * a, ((uint32_t)(j >> 1)) & 1u);
      tc_fence_after();
      const uint32_t tsrc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(a * BN);
      uint32_t r[32], r2[OUTB ? 32 : 1];
      tmem_ld32_nowait(tsrc, r);
      if (OUTB) tmem_ld32_nowait(tsrc + 32u, r2);
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += CW, ++blk) {
        const uint32_t pb = pad + (uint32_t)(blk & 1) * 4096u + prow;
        if (lane == 0) bulk_wait_read1();              // the store that last read this pad (two blocks ago) has drained it
        __syncwarp();
        tmem_wait_ld();
        if (ep.bias) {
          add_bias32(r, ep.bias, n0 + c0, N, ep.vec_ok);
          if (OUTB) add_bias32(r2, ep.bias, n0 + c0 + 32, N, ep.vec_ok);
        }
        // lane = row; 16-byte piece p of the row's 128 bytes goes to slot p ^ (row & 7)  (= the TMA 128-byte swizzle)
        if (!OUTB) {
#pragma unroll
          for (int p = 0; p < 8; ++p) sts128(pb + (uint32_t)((p ^ sw) << 4), r[4 * p], r[4 * p + 1], r[4 * p + 2], r[4 * p + 3]);
        } else {
#pragma unroll
          for (int p = 0; p < 4; ++p)
            sts128(pb + (uint32_t)((p ^ sw) << 4), pack_bf16(r[8 * p], r[8 * p + 1]), pack_bf16(r[8 * p + 2], r[8 * p + 3]),
                   pack_bf16(r[8 * p + 4], r[8 * p + 5]), pack_bf16(r[8 * p + 6], r[8 * p + 7]));
#pragma unroll
          for (int p = 0; p < 4; ++p)
            sts128(pb + (uint32_t)(((p + 4) ^ sw) << 4), pack_bf16(r2[8 * p], r2[8 * p + 1]), pack_bf16(r2[8 * p + 2], r2[8 * p + 3]),
                   pack_bf16(r2[8 * p + 4], r2[8 * p + 5]), pack_bf16(r2[8 * p + 6], r2[8 * p + 7]));
        }
        if (c0 + CW < BN) {                            // next block's TMEM read flies under the store hand-off below
          tmem_ld32_nowait(tsrc + (uint32_t)(c0 + CW), r);
          if (OUTB) tmem_ld32_nowait(tsrc + (uint32_t)(c0 + CW + 32), r2);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          if (m0 < M && n0 + c0 < N) tma_store_2d(&tmC, pb, n0 + c0, m0, add);
          bulk_commit();       // ALWAYS one group per block (empty when the block lies outside C): bulk_wait_read1 counts groups, and
                               // "at most one pending" must mean "the store that read THIS pad two blocks ago is done"
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { if (CTAS == 2) mbar_arrive_cluster(te + 8 * a); else mbar_arrive_local(te + 8 * a); }
    }
    if (lane == 0) bulk_wait_all();
    __syncwarp();
  }
  tc_fence_before();
  if (CTAS == 2) tc::cluster_sync_all(); else __syncthreads();
  if (warp == 1) tmem_dealloc<CTAS>(tmem_base, 2 * BN);
}

// ---- host side -----------------------------------------------------------------------------------
// output tensor [rows, cols] row-major (ld elements): fp32 boxes of 32 x 32, bf16 boxes of 32 rows x 64 columns -- 128-byte rows
static inline int make_out_map(CUtensorMap* map, const void* ptr, long long rows, long long cols, long long ld, bool is_bf16) {
  tc::EncodeTiledFn enc = tc::get_encode_fn();
  if (!enc) return RECNET_ERR_DRIVER;
  const int esz = is_bf16 ? 2 : 4;
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || ((ld * esz) & 15)) return RECNET_ERR_ALIGNMENT;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * esz};
  cuuint32_t box[2] = {(cuuint32_t)(is_bf16 ? 64 : 32), 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, is_bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims,
                   strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : RECNET_ERR_DRIVER;
}

// the persistent kernel covers: one output (fp32 or bf16), 16-byte aligned output rows, no split-K; anything else stays on tc::
static inline bool supported(const float* Cf, long long ldc, const bf16* Cb, long long ldcb, int accumulate) {
  if ((Cf != nullptr) == (Cb != nullptr)) return false;
  if (Cf) return !(reinterpret_cast<uintptr_t>(Cf) & 15) && !((ldc * 4) & 15);
  return !accumulate && !(reinterpret_cast<uintptr_t>(Cb) & 15) && !((ldcb * 2) & 15);
}

template <int BN, int STAGES, bool TA, bool TB, int CTAS, bool OUTB>
static int launch_cfg(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mc, const EpiArgs& ep, int M, int N, int K,
                      cudaStream_t st) {
  using L = Smem<BN, STAGES, CTAS>;
  static_assert(L::TOTAL <= 232448, "shared memory");
  auto kern = gemm_tc2_kernel<BN, STAGES, TA, TB, CTAS, OUTB>;
  static bool attr_set = false;
  if (!attr_set) {
    RN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
    attr_set = true;
  }
  const int tiles_m = rn_cdiv(M, BM * CTAS), tiles_n = rn_cdiv(N, BN);
  int units = min(tiles_m * tiles_n, TC2_SMS / CTAS);
  if (rn_background_ctas() > 0) units = min(units, max(1, rn_background_ctas() / CTAS));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(units * CTAS);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = (size_t)L::TOTAL;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CTAS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = CTAS == 2 ? 1 : 0;
  ProfScope prof(KC_GEMM_TC, M, N, K, st);
  RN_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, ma, mb, mc, ep, M, N, K, tiles_m, tiles_n));
  RN_LAUNCH_OK();
  return 0;
}

template <int BN, int STAGES, int CTAS, bool OUTB>
static int launch_bn(int transA, int transB, const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mc, const EpiArgs& ep,
                     int M, int N, int K, cudaStream_t st) {
  if (!transA && !transB) return launch_cfg<BN, STAGES, false, false, CTAS, OUTB>(ma, mb, mc, ep, M, N, K, st);
  if (!transA && transB) return launch_cfg<BN, STAGES, false, true, CTAS, OUTB>(ma, mb, mc, ep, M, N, K, st);
  if (transA && !transB) return launch_cfg<BN, STAGES, true, false, CTAS, OUTB>(ma, mb, mc, ep, M, N, K, st);
  return launch_cfg<BN, STAGES, true, true, CTAS, OUTB>(ma, mb, mc, ep, M, N, K, st);
}
template <int BN, int STAGES, int CTAS>
static int launch_out(bool outb, int transA, int transB, const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mc,
                      const EpiArgs& ep, int M, int N, int K, cudaStream_t st) {
  return outb ? launch_bn<BN, STAGES, CTAS, true>(transA, transB, ma, mb, mc, ep, M, N, K, st)
              : launch_bn<BN, STAGES, CTAS, false>(transA, transB, ma, mb, mc, ep, M, N, K, st);
}

// BN in {128, 256}; ctas in {1, 2}
static inline int launch(const bf16* A, long long lda, int transA, const bf16* B, long long ldb, int transB, float* Cf, long long ldc,
                         bf16* Cb, long long ldcb, const float* bias, int M, int N, int K, int accumulate, int BN, int ctas,
                         cudaStream_t st) {
  if (M <= 0 || N <= 0 || K <= 0) return RECNET_ERR_BAD_SHAPE;
  if ((BN != 128 && BN != 256) || (ctas != 1 && ctas != 2)) return RECNET_ERR_BAD_SHAPE;
  if (!supported(Cf, ldc, Cb, ldcb, accumulate)) return RECNET_ERR_UNSUPPORTED;
  const int bnl = BN / ctas;
  const bool outb = Cb != nullptr;
  CUtensorMap ma, mb, mc;
  if (!transA) { RN_TRY(tc::make_map(&ma, A, M, K, lda, BK, BM)); } else { RN_TRY(tc::make_map(&ma, A, K, M, lda, 64, BK)); }
  if (!transB) { RN_TRY(tc::make_map(&mb, B, N, K, ldb, BK, bnl)); } else { RN_TRY(tc::make_map(&mb, B, K, N, ldb, 64, BK)); }
  RN_TRY(make_out_map(&mc, outb ? (const void*)Cb : (const void*)Cf, M, N, outb ? ldcb : ldc, outb));
  EpiArgs ep;
  ep.Cf = Cf; ep.ldc = ldc; ep.split_stride = 0; ep.Cb = Cb; ep.ldcb = ldcb; ep.bias = bias;
  ep.accumulate = accumulate;
  ep.vec_ok = (bias && (reinterpret_cast<uintptr_t>(bias) & 15)) ? 0 : 1;
  if (BN == 256) return ctas == 1 ? launch_out<256, 4, 1>(outb, transA, transB, ma, mb, mc, ep, M, N, K, st)
                                  : launch_out<256, 6, 2>(outb, transA, transB, ma, mb, mc, ep, M, N, K, st);
  return ctas == 1 ? launch_out<128, 6, 1>(outb, transA, transB, ma, mb, mc, ep, M, N, K, st)
                   : launch_out<128, 8, 2>(outb, transA, transB, ma, mb, mc, ep, M, N, K, st);
}
}  // namespace tc2
