// tcgen05 / TMEM / TMA GEMM for sm_100a (bf16 operands, fp32 accumulate in tensor memory).
//
//   C[m,n] (+)= sum_k A(m,k) * B(n,k) (+ bias[n])           one 128 x BN tile per CTA, optional split-K
//
// Operand storage (no transposed copies are ever materialised):
//   transA = 0 : A is [M,K] row-major (K-major UMMA operand)   transA = 1 : A is [K,M] row-major (MN-major)
//   transB = 0 : B is [N,K] row-major (nn.Linear weight)       transB = 1 : B is [K,N] row-major (MN-major)
// Tiles are brought in by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle), consumed from shared memory by a
// single elected thread issuing tcgen05.mma.cta_group::1.kind::f16 (UMMA 128 x BN x 16), accumulators live in
// TMEM and are read back by four epilogue warps with tcgen05.ld.  Warp roles: 0 = TMA producer,
// 1 = TMEM allocator + MMA issuer, 2..5 = epilogue.  The smem ring is STAGES deep with full/empty mbarriers.
#pragma once
#include "common.cuh"

namespace tc {

constexpr int BM = 128;
constexpr int BK = 64;          // 64 bf16 = 128 bytes = one swizzle row
constexpr int UMMA_K = 16;
constexpr int THREADS = 192;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
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
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA shared-memory matrix descriptor, 128B swizzle (layout_type = 2), descriptor version 1 (Blackwell).
//   K-major : rows of 128 B, 8-row groups SBO = 1024 B apart (LBO unused, canonical value 1).
//   MN-major: 64-element (128 B) MN blocks LBO bytes apart, 8-k-row groups SBO = 1024 B apart.
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

struct EpiArgs {
  float* Cf; long long ldc; long long split_stride;     // fp32 output (nullable)
  bf16* Cb; long long ldcb;                              // bf16 output (nullable, split 0 only)
  const float* bias;                                     // [N] nullable, added in split 0
  int accumulate;                                        // Cf += result
  int vec_ok;                                            // 16-byte aligned rows -> float4 stores
};

template <int BN, int STAGES>
struct SmemLayout {
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFF + (2 * STAGES + 1) * 8 + 16 + 1024;   // + alignment slack
};

template <int BN, int STAGES, bool TA, bool TB>
__global__ void __launch_bounds__(THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, EpiArgs ep,
               int M, int N, int K, int kb_per_split) {
  using L = SmemLayout<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = base + L::BAR_OFF;
  const uint32_t bar_empty = bar_full + 8 * STAGES;
  const uint32_t bar_tmem = bar_empty + 8 * STAGES;
  const uint32_t tmem_slot = bar_tmem + 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int nkb_total = (K + BK - 1) / BK;
  const int kb0 = blockIdx.z * kb_per_split;
  const int nkb = max(0, min(nkb_total, kb0 + kb_per_split) - kb0);

  // one producer step: expect-tx + the TMA boxes of k-block i into ring slot i % STAGES
  auto produce = [&](int i) {
    const int s = i % STAGES;
    mbar_expect_tx(bar_full + 8 * s, L::STAGE_BYTES);
    const uint32_t sa = base + s * L::STAGE_BYTES, sb = sa + L::A_BYTES;
    const int k = (kb0 + i) * BK;
    if (!TA) {
      tma_load_2d(sa, &tmA, bar_full + 8 * s, k, m0);                       // box {64 k, 128 m}
    } else {
#pragma unroll
      for (int j = 0; j < BM / 64; ++j)                                     // boxes {64 m, 64 k}
        tma_load_2d(sa + j * (BK * 128), &tmA, bar_full + 8 * s, m0 + j * 64, k);
    }
    if (!TB) {
      tma_load_2d(sb, &tmB, bar_full + 8 * s, k, n0);                       // box {64 k, BN n}
    } else {
#pragma unroll
      for (int j = 0; j < BN / 64; ++j)                                     // boxes {64 n, 64 k}
        tma_load_2d(sb + j * (BK * 128), &tmB, bar_full + 8 * s, n0 + j * 64, k);
    }
  };
  const int n_early = nkb < STAGES ? nkb : STAGES;
  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    for (int s = 0; s < STAGES; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    mbar_init(bar_tmem, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // The per-step GEMMs have 1-11 k-blocks and are pure latency chains (launch -> TMA -> UMMA -> tcgen05.ld -> store): the
    // first pass through the ring needs no empty-slot wait, so its loads are issued right here, by the thread that just
    // initialised the barriers, while warp 1 is still allocating TMEM and the CTA has not yet met at the barrier below.
    pdl_wait();
    pdl_launch_next();
    for (int i = 0; i < n_early; ++i) produce(i);
  }
  if (warp == 1) tmem_alloc(tmem_slot, BN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();          // everything above overlapped the previous kernel's tail; operands / outputs are touched only below
  pdl_launch_next();   // after the wait: the next kernel may be scheduled now, but it cannot trigger ITS dependents before we finish
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    if (lane == 0) {
      for (int i = n_early; i < nkb; ++i) {
        const int s = i % STAGES;
        const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
        mbar_wait(bar_empty + 8 * s, ph ^ 1u);
        produce(i);
      }
    }
  } else if (warp == 1) {
    // instruction descriptor: D=f32 (bits4-5=1), A=B=bf16 (bits7-9, 10-12 = 1), majors, N>>3 @17, M>>4 @24
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((TA ? 1u : 0u) << 15) | ((TB ? 1u : 0u) << 16) |
                           ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
    for (int i = 0; i < nkb; ++i) {
      const int s = i % STAGES;
      const uint32_t ph = (uint32_t)(i / STAGES) & 1u;
      mbar_wait(bar_full + 8 * s, ph);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t sa = base + s * L::STAGE_BYTES, sb = sa + L::A_BYTES;
#pragma unroll
        for (int kk = 0; kk < BK / UMMA_K; ++kk) {
          const uint64_t ad = TA ? umma_smem_desc(sa + kk * (UMMA_K * 128), BK * 128, 1024)
                                 : umma_smem_desc(sa + kk * (UMMA_K * 2), 16, 1024);
          const uint64_t bd = TB ? umma_smem_desc(sb + kk * (UMMA_K * 128), BK * 128, 1024)
                                 : umma_smem_desc(sb + kk * (UMMA_K * 2), 16, 1024);
          umma_bf16(tmem_base, ad, bd, idesc, (i > 0 || kk > 0) ? 1u : 0u);
        }
        umma_commit(bar_empty + 8 * s);
        if (i == nkb - 1) umma_commit(bar_tmem);
      }
      __syncwarp();
    }
  } else {
    // ---- epilogue: warp w owns TMEM lanes (w % 4) * 32 .. +31  == rows of the tile ----
    const int q = warp & 3;
    const int m = m0 + q * 32 + lane;
    if (nkb > 0) {
      mbar_wait(bar_tmem, 0);
      tc_fence_after();
    }
    const bool z0 = (blockIdx.z == 0);
    float* crow = ep.Cf ? ep.Cf + (long long)blockIdx.z * ep.split_stride + (long long)m * ep.ldc : nullptr;
    bf16* brow = (ep.Cb && z0) ? ep.Cb + (long long)m * ep.ldcb : nullptr;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t r[32];
      if (nkb > 0) {
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, r);   // warp-collective: outside row guard
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) r[j] = 0u;
      }
      if (m < M) {
        const int n = n0 + c0;
        if (ep.vec_ok && n + 32 <= N) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            float4 v = make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]),
                                   __uint_as_float(r[j + 3]));
            if (ep.bias && z0) {
              const float4 b4 = *reinterpret_cast<const float4*>(ep.bias + n + j);
              v.x += b4.x; v.y += b4.y; v.z += b4.z; v.w += b4.w;
            }
            if (crow) {
              float4* p = reinterpret_cast<float4*>(crow + n + j);
              if (ep.accumulate) { const float4 o = *p; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
              *p = v;
            }
            if (brow) {
              __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
              uint2 pk = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
              *reinterpret_cast<uint2*>(brow + n + j) = pk;
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (n + j < N) {
              float v = __uint_as_float(r[j]);
              if (ep.bias && z0) v += ep.bias[n + j];
              if (crow) { if (ep.accumulate) v += crow[n + j]; crow[n + j] = v; }
              if (brow) brow[n + j] = __float2bfloat16_rn(v);
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, BN);
}

// ---- host side -----------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || !p) return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// 2-D bf16 row-major tensor [rows, cols] with leading dimension ld (elements); box = {box_cols, box_rows}.
static inline int make_map(CUtensorMap* map, const void* ptr, long long rows, long long cols, long long ld,
                           int box_cols, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return RECNET_ERR_DRIVER;
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || ((ld * 2) & 15)) return RECNET_ERR_ALIGNMENT;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : RECNET_ERR_DRIVER;
}

template <int BN, int STAGES, bool TA, bool TB>
static int launch_cfg(const CUtensorMap& ma, const CUtensorMap& mb, const EpiArgs& ep, int M, int N, int K, int splits,
                      int kb_per, cudaStream_t st) {
  using L = SmemLayout<BN, STAGES>;
  auto kern = gemm_tc_kernel<BN, STAGES, TA, TB>;
  static bool attr_set = false;
  if (!attr_set) {
    RN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
    attr_set = true;
  }
  dim3 grid(rn_cdiv(N, BN), rn_cdiv(M, BM), splits);
  ProfScope prof(KC_GEMM_TC, M, N, K, st);
  RN_CUDA_OK(launch_pdl(kern, grid, dim3(THREADS), (size_t)L::TOTAL, st, ma, mb, ep, M, N, K, kb_per));
  RN_LAUNCH_OK();
  return 0;
}

template <int BN, int STAGES>
static int launch_bn(int transA, int transB, const CUtensorMap& ma, const CUtensorMap& mb, const EpiArgs& ep, int M,
                     int N, int K, int splits, int kb_per, cudaStream_t st) {
  if (!transA && !transB) return launch_cfg<BN, STAGES, false, false>(ma, mb, ep, M, N, K, splits, kb_per, st);
  if (!transA && transB) return launch_cfg<BN, STAGES, false, true>(ma, mb, ep, M, N, K, splits, kb_per, st);
  if (transA && !transB) return launch_cfg<BN, STAGES, true, false>(ma, mb, ep, M, N, K, splits, kb_per, st);
  return launch_cfg<BN, STAGES, true, true>(ma, mb, ep, M, N, K, splits, kb_per, st);
}

}  // namespace tc
namespace tc2 {
static inline int launch(const bf16* A, long long lda, int transA, const bf16* B, long long ldb, int transB, float* Cf, long long ldc,
                         bf16* Cb, long long ldcb, const float* bias, int M, int N, int K, int accumulate, int BN, int ctas,
                         cudaStream_t st);
static inline bool supported(const float* Cf, long long ldc, const bf16* Cb, long long ldcb, int accumulate);
}
namespace tc {
// bn_hint: 0 = auto, else 64/128/256 (this file's one-tile-per-CTA kernel), or 1000 + {128,256} / 2000 + {128,256}: the persistent
// kernel of gemm_tc2.cuh with single CTAs / CTA pairs (splits must be 1).  splits >= 1; every slice gets >= 1 k-block.
static inline int launch(const bf16* A, long long lda, int transA, const bf16* B, long long ldb, int transB, float* Cf,
                         long long ldc, bf16* Cb, long long ldcb, const float* bias, int M, int N, int K, int splits,
                         long long split_stride, int accumulate, int bn_hint, cudaStream_t st) {
  if (M <= 0 || N <= 0 || K <= 0) return RECNET_ERR_BAD_SHAPE;
  if (bn_hint >= 1000 && (splits > 1 || !tc2::supported(Cf, ldc, Cb, ldcb, accumulate))) bn_hint %= 1000;   // not covered: this file's kernel
  if (bn_hint >= 1000) {
    return tc2::launch(A, lda, transA, B, ldb, transB, Cf, ldc, Cb, ldcb, bias, M, N, K, accumulate, bn_hint % 1000, bn_hint / 1000, st);
  }
  int BN = bn_hint;
  if (BN == 0) BN = (N >= 1024 && (long long)rn_cdiv(M, BM) * rn_cdiv(N, 128) >= 96) ? 128 : 64;
  if (BN != 64 && BN != 128 && BN != 256) return RECNET_ERR_BAD_SHAPE;
  const int nkb = rn_cdiv(K, BK);
  if (splits < 1) splits = 1;
  if (splits > nkb) splits = nkb;
  int kb_per = rn_cdiv(nkb, splits);
  splits = rn_cdiv(nkb, kb_per);
  CUtensorMap ma, mb;
  if (!transA) { RN_TRY(make_map(&ma, A, M, K, lda, BK, BM)); } else { RN_TRY(make_map(&ma, A, K, M, lda, 64, BK)); }
  if (!transB) { RN_TRY(make_map(&mb, B, N, K, ldb, BK, BN)); } else { RN_TRY(make_map(&mb, B, K, N, ldb, 64, BK)); }
  EpiArgs ep;
  ep.Cf = Cf; ep.ldc = ldc; ep.split_stride = split_stride; ep.Cb = Cb; ep.ldcb = ldcb; ep.bias = bias;
  ep.accumulate = accumulate;
  ep.vec_ok = 1;
  if (Cf && ((reinterpret_cast<uintptr_t>(Cf) & 15) || (ldc & 3) || (split_stride & 3))) ep.vec_ok = 0;
  if (Cb && ((reinterpret_cast<uintptr_t>(Cb) & 7) || (ldcb & 3))) ep.vec_ok = 0;
  if (bias && (reinterpret_cast<uintptr_t>(bias) & 15)) ep.vec_ok = 0;
  // short K loops (the per-step split-K GEMMs) use a shallow ring (<= 97 KB smem) so that two CTAs share an SM; long K
  // loops (batched GEMMs) use the deep ring.
  static const int shallow_kb = rn_env_int("RECNET_GEMM_SHALLOW_KB", 12);
  const bool shallow = kb_per <= shallow_kb;
  if (BN == 64) return shallow ? launch_bn<64, 4>(transA, transB, ma, mb, ep, M, N, K, splits, kb_per, st)
                               : launch_bn<64, 8>(transA, transB, ma, mb, ep, M, N, K, splits, kb_per, st);
  if (BN == 128) return shallow ? launch_bn<128, 3>(transA, transB, ma, mb, ep, M, N, K, splits, kb_per, st)
                                : launch_bn<128, 6>(transA, transB, ma, mb, ep, M, N, K, splits, kb_per, st);
  return launch_bn<256, 4>(transA, transB, ma, mb, ep, M, N, K, splits, kb_per, st);
}
}  // namespace tc
#include "gemm_tc2.cuh"
