// Shared device/host helpers for the recnet_b200 kernels (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/recnet_b200.h"

// Descriptors as the drivers see them: the entry points split RECNET_ATTN_SOFTMAX off the public `cell` field once, so `cell` holds the
// plain recnet_cell value and `softmax` says whether the attention is the paper's softmax (true) or the reference's mean (false).
struct DecDesc : recnet_decoder_desc { bool softmax = false; };
struct LocalDesc : recnet_local_desc { bool softmax = false; };

typedef __nv_bfloat16 bf16;

#define RN_CUDA_OK(expr)                                  \
  do {                                                    \
    cudaError_t _e = (expr);                              \
    if (_e != cudaSuccess) return (int)_e;                \
  } while (0)

// ---- launch accounting + optional per-launch timing (bench.py's roofline leg) -------------------------------
// Every kernel launch in the library goes through RN_LAUNCH_OK(), which bumps g_launches.  When profiling is on
// (recnet_profile_enable), launch sites wrapped in a ProfScope also record a CUDA-event pair on the launching
// stream, tagged with a kernel class and the problem shape; recnet_profile_collect returns per-launch durations.
enum KernelClass { KC_OTHER = 0, KC_GEMM_TC = 1, KC_SGEMM = 2, KC_ATTN_FWD = 3, KC_ATTN_BWD = 4, KC_CELL_FWD = 5,
                   KC_CELL_BWD = 6, KC_CE = 7, KC_REDUCE = 8, KC_LOOP = 9, KC_PF_FWD = 10, KC_PF_BWD = 11 };
struct ProfRecord { int cls, M, N, K; cudaEvent_t e0, e1; };
struct ProfState {
  long long launches = 0;
  int enabled = 0;
  int n = 0, cap = 0;
  ProfRecord* rec = nullptr;
};
inline ProfState& prof_state() { static ProfState s; return s; }

struct ProfScope {
  cudaStream_t st; int idx;
  ProfScope(int cls, int M, int N, int K, cudaStream_t s) : st(s), idx(-1) {
    ProfState& p = prof_state();
    if (!p.enabled || p.n >= p.cap) return;
    idx = p.n++;
    ProfRecord& r = p.rec[idx];
    r.cls = cls; r.M = M; r.N = N; r.K = K;
    if (!r.e0) { cudaEventCreate(&r.e0); cudaEventCreate(&r.e1); }
    cudaEventRecord(r.e0, st);
  }
  ~ProfScope() { if (idx >= 0) cudaEventRecord(prof_state().rec[idx].e1, st); }
};

#define RN_LAUNCH_OK()                                    \
  do {                                                    \
    prof_state().launches++;                              \
    cudaError_t _e = cudaGetLastError();                  \
    if (_e != cudaSuccess) return (int)_e;                \
  } while (0)

#define RN_TRY(expr)                                      \
  do {                                                    \
    int _r = (expr);                                      \
    if (_r != 0) return _r;                               \
  } while (0)

static inline int rn_cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// The RECNET_* environment switches (INTEGRATION.md) are read through this: the integer value of `name`, or `dflt` when it is unset.
// The call sites keep the value in a function-local `static const`, so each switch is read once per process.
inline int rn_env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

// ---- type conversion -------------------------------------------------------------------------
// Upper bound on the CTAs of ONE launch of the batched kernels (0 = none): set by a trainer around work it runs on a second stream UNDERNEATH a
// latency-bound foreground kernel sequence (recnet_set_background_ctas; functional.py "background lane").  Persistent GEMMs, split-K plans and the
// split-K reduce and the column sums honour it.
inline int& rn_background_ctas() { static int v = 0; return v; }

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<bf16>(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f32<bf16>(float v) { return __float2bfloat16_rn(v); }

// 16-byte vector of T: 4 floats or 8 bf16
template <typename T> struct Vec16;
template <> struct Vec16<float> {
  static constexpr int N = 4;
  float4 raw;
  __device__ __forceinline__ void load(const float* p) { raw = *reinterpret_cast<const float4*>(p); }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float4*>(p) = raw; }
  __device__ __forceinline__ void get(float* f) const { f[0] = raw.x; f[1] = raw.y; f[2] = raw.z; f[3] = raw.w; }
  __device__ __forceinline__ void set(const float* f) { raw = make_float4(f[0], f[1], f[2], f[3]); }
};
template <> struct Vec16<bf16> {
  static constexpr int N = 8;
  uint4 raw;
  __device__ __forceinline__ void load(const bf16* p) { raw = *reinterpret_cast<const uint4*>(p); }
  __device__ __forceinline__ void store(bf16* p) const { *reinterpret_cast<uint4*>(p) = raw; }
  __device__ __forceinline__ void get(float* f) const {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 t = __bfloat1622float2(h[i]); f[2 * i] = t.x; f[2 * i + 1] = t.y; }
  }
  __device__ __forceinline__ void set(const float* f) {
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&raw);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  }
};

// ---- reductions ------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// block-wide sum; `red` is >= 32 floats of shared memory; every thread gets the result.
__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : 0.f;
  r = warp_sum(r);
  return r;
}
__device__ __forceinline__ float block_max(float v, float* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : -INFINITY;
  r = warp_max(r);
  return r;
}

// developer timeline (recnet_debug_set_timeline): block 0 / thread 0 appends (tag << 56 | %globaltimer ns) records
__device__ unsigned long long* g_timeline = nullptr;
__device__ unsigned int g_timeline_n = 0;
// (compiled in only with -DRECNET_PROBES for the intra-body points; the loop kernel's phase-level stamps are always on)
__device__ __forceinline__ void probe(int tag, int tid) {
  if (g_timeline != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && tid == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    const unsigned int i = g_timeline_n++;
    if (i < 4000) g_timeline[i] = (t & 0x00FFFFFFFFFFFFFFull) | ((unsigned long long)tag << 56);
  }
}

// ---- Programmatic Dependent Launch --------------------------------------------------------------------------------
// The time loops are chains of ~470 small dependent kernels.  With PDL a kernel's CTAs are scheduled, and its prologue
// (barrier init, TMEM allocation, descriptor prefetch, index math) runs, while the previous kernel is still draining;
// pdl_wait() blocks until the previous grid has completed and its writes are visible, so it must precede the first
// global-memory access.  pdl_launch_next() lets the next kernel in the stream start its own launch early.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_next() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

inline bool pdl_enabled() {
  static const int v = rn_env_int("RECNET_PDL", 0);   // measured: 4.53 ms/step with PDL vs 4.14 without -> opt-in
  return v != 0;
}
// launch with the programmatic-stream-serialization attribute (falls back to a plain launch when RECNET_PDL=0)
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

#ifdef RECNET_PROBES
#define RN_PROBE(tag, tid) probe(tag, tid)
#else
#define RN_PROBE(tag, tid) ((void)0)
#endif

// sync of one 256-thread (sub-)block: bar 0 = the whole CTA (stand-alone kernels), bar 1..15 = a named barrier shared by
// the 256 threads of one sub-block of the persistent loop kernel
__device__ __forceinline__ void blk_sync(int bar_id) {
  if (bar_id == 0) __syncthreads();
  else asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// Activation math by build: FAST (bf16 build) = one MUFU.TANH per call (tanh.approx.f32, max rel err ~2^-11, far below
// bf16 operand rounding); accurate libm (fp32 parity build, 1e-3 / bit-exact greedy).  r1 profile: with libm tanhf/expf the
// cell kernels ran ~570 instructions per element and were issue-bound.
template <bool FAST> __device__ __forceinline__ float act_tanh(float x) {
  if (FAST) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
  return tanhf(x);
}
template <bool FAST> __device__ __forceinline__ float act_sigmoid(float x) {
  if (FAST) return fmaf(0.5f, act_tanh<true>(0.5f * x), 0.5f);
  return 1.f / (1.f + expf(-x));
}
template <bool FAST> __device__ __forceinline__ float act_exp(float x) { return FAST ? __expf(x) : expf(x); }
template <typename T> struct FastMath { static constexpr bool value = false; };
template <> struct FastMath<bf16> { static constexpr bool value = true; };
// max-subtracted softmax of a row of <= 32 scores held one per lane (valid = lane < row length; invalid lanes return 0)
template <bool FAST> __device__ __forceinline__ float warp_softmax(float x, bool valid) {
  const float m = warp_max(valid ? x : -INFINITY);
  const float p = valid ? act_exp<FAST>(x - m) : 0.f;
  return p / warp_sum(p);
}

// ---- Philox4x32-10 counter RNG (Salmon et al. 2011), used for in-kernel dropout masks --------
struct Philox {
  uint32_t key[2];
  __device__ __forceinline__ Philox(uint64_t seed) { key[0] = (uint32_t)seed; key[1] = (uint32_t)(seed >> 32); }
  __device__ __forceinline__ uint4 operator()(uint64_t ctr, uint64_t stream) const {
    uint32_t c0 = (uint32_t)ctr, c1 = (uint32_t)(ctr >> 32), c2 = (uint32_t)stream, c3 = (uint32_t)(stream >> 32);
    uint32_t k0 = key[0], k1 = key[1];
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
      k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
};
// keep-mask scale for element `idx` of dropout site `site`: 0 or 1/(1-p).  rng = {seed, offset}.
__device__ __forceinline__ float dropout_scale(const unsigned long long* rng, uint32_t site, uint64_t idx, float p) {
  if (p <= 0.f) return 1.f;
  Philox ph(rng[0]);
  const uint4 r = ph(idx >> 2, (rng[1] << 8) | site);
  const uint32_t w = ((idx & 3) == 0) ? r.x : ((idx & 3) == 1) ? r.y : ((idx & 3) == 2) ? r.z : r.w;
  const float u = (float)(w >> 8) * (1.0f / 16777216.0f);
  return (u >= p) ? 1.f / (1.f - p) : 0.f;
}
// the four scales of elements idx4 .. idx4 + 3 (idx4 a multiple of 4) from ONE Philox call; identical to dropout_scale()
__device__ __forceinline__ float4 dropout_scale4(const unsigned long long* rng, uint32_t site, uint64_t idx4, float p) {
  if (p <= 0.f) return make_float4(1.f, 1.f, 1.f, 1.f);
  Philox ph(rng[0]);
  const uint4 r = ph(idx4 >> 2, (rng[1] << 8) | site);
  const float k = 1.f / (1.f - p), sc = 1.0f / 16777216.0f;
  return make_float4(((float)(r.x >> 8) * sc >= p) ? k : 0.f, ((float)(r.y >> 8) * sc >= p) ? k : 0.f,
                     ((float)(r.z >> 8) * sc >= p) ? k : 0.f, ((float)(r.w >> 8) * sc >= p) ? k : 0.f);
}
