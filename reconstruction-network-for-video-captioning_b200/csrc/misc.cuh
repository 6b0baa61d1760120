// Small data-movement kernels around the hot loops: operand staging (fp32 -> bf16 with K padding),
// embedding gather / scatter-add (models/decoder.py:46-48), bias-gradient column sums, the global
// reconstructor's mean-pool (models/global_reconstructor.py:33-37) and the multi-tensor L2-norm
// regulariser (train.py:69,101,127).  All HBM-bound, coalesced along the contiguous dimension.
#pragma once
#include "common.cuh"

namespace misc {

// dst[r, 0:cols] = (TO) src[r, 0:cols] ; dst[r, cols:cols_pad] = 0
template <typename TO>
__global__ void cast_pad_kernel(const float* __restrict__ src, long long ld_src, TO* __restrict__ dst, long long ld_dst,
                                long long rows, int cols, int cols_pad) {
  const long long total = rows * cols_pad;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols_pad; const int c = (int)(i % cols_pad);
    dst[r * ld_dst + c] = from_f32<TO>(c < cols ? src[r * ld_src + c] : 0.f);
  }
}
template <typename TO> struct Store4;
template <> struct Store4<float> {
  static __device__ __forceinline__ void st(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
};
template <> struct Store4<bf16> {
  static __device__ __forceinline__ void st(bf16* p, float4 v) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
  }
};
// 4 elements per thread, 32-bit index math (r1 launch list: the scalar version with a 64-bit divide per element ran at
// 1.9 TB/s on the 6144 x 1536 recurrent weight; these casts re-stage ~29 M weights every step)
template <typename TO>
__global__ void cast_pad4_kernel(const float* __restrict__ src, unsigned ld_src, TO* __restrict__ dst, unsigned ld_dst,
                                 unsigned total4, unsigned cols4, unsigned cp4) {
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += gridDim.x * blockDim.x) {
    const unsigned r = i / cp4, c4 = i - r * cp4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c4 < cols4) v = *reinterpret_cast<const float4*>(src + (size_t)r * ld_src + 4 * c4);
    Store4<TO>::st(dst + (size_t)r * ld_dst + 4 * c4, v);
  }
}
template <typename TO>
static int cast_pad(const float* src, long long ld_src, TO* dst, long long ld_dst, long long rows, int cols, int cols_pad,
                    cudaStream_t st) {
  const long long total = rows * cols_pad;
  if (total == 0) return 0;
  const bool vec = !(cols & 3) && !(cols_pad & 3) && !(ld_src & 3) && !(ld_dst & 3) && !(reinterpret_cast<uintptr_t>(src) & 15) &&
                   !(reinterpret_cast<uintptr_t>(dst) & 15) && total / 4 < (1ll << 31) && ld_src < (1ll << 31) && ld_dst < (1ll << 31);
  if (vec) {
    const unsigned total4 = (unsigned)(total / 4);
    const int blocks = (int)min((long long)148 * 16, ((long long)total4 + 255) / 256);
    cast_pad4_kernel<TO><<<blocks, 256, 0, st>>>(src, (unsigned)ld_src, dst, (unsigned)ld_dst, total4, (unsigned)cols / 4, (unsigned)cols_pad / 4);
  } else {
    int blocks = (int)min((long long)148 * 16, (total + 255) / 256);
    cast_pad_kernel<TO><<<blocks, 256, 0, st>>>(src, ld_src, dst, ld_dst, rows, cols, cols_pad);
  }
  RN_LAUNCH_OK();
  return 0;
}

// ---- multi-tensor operand staging ------------------------------------------------------------------------------------
// Every sequence forward re-stages the operand copies of its weights / inputs (the optimiser moves the fp32 masters) and clears
// a few state buffers: 7 casts + 3 memsets in the decoder, 6 + 3 in the local reconstructor -- each a node of a captured graph
// whose cost is its launch latency, not its bytes.  A Stager collects them and issues ONE kernel (table passed by value):
//   dst[r', 0:cols] = (TO) src[r, 0:cols], dst[r', cols:cols_pad] = 0;   r' = r, or for interleave_H > 0 the unit-interleaved
//   order  dst row 4j+g <- src row g*H+j  (W_ctx, makes the VW GEMM emit [.., H, 4]);   src == nullptr -> zero fill.
// Items that cannot take 16-byte vectors fall back to a scalar launch of their own.
struct StageItem { const float* src; void* dst; unsigned ld_src, ld_dst, rows, cols4, cp4, interleave_H; };
constexpr int STAGE_MAX = 12;
struct StageTable { StageItem it[STAGE_MAX]; unsigned blk0[STAGE_MAX + 1]; int n; };

template <typename TO>
__global__ void stage_multi_kernel(const StageTable t) {
  int e = 0;
  while (e + 1 < t.n && blockIdx.x >= t.blk0[e + 1]) ++e;
  const StageItem it = t.it[e];
  const unsigned nb = t.blk0[e + 1] - t.blk0[e], lb = blockIdx.x - t.blk0[e];
  const unsigned total4 = it.rows * it.cp4;
  TO* dst = reinterpret_cast<TO*>(it.dst);
  for (unsigned i = lb * blockDim.x + threadIdx.x; i < total4; i += nb * blockDim.x) {
    const unsigned r = i / it.cp4, c4 = i - r * it.cp4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (it.src && c4 < it.cols4) {
      const unsigned sr = it.interleave_H ? (r & 3u) * it.interleave_H + (r >> 2) : r;
      v = *reinterpret_cast<const float4*>(it.src + (size_t)sr * it.ld_src + 4 * c4);
    }
    Store4<TO>::st(dst + (size_t)r * it.ld_dst + 4 * c4, v);
  }
}
// scalar fallback for one item (any alignment, any column count)
template <typename TO>
__global__ void stage_scalar_kernel(const float* __restrict__ src, long long ld_src, TO* __restrict__ dst, long long ld_dst, long long rows,
                                    int cols, int cols_pad, int interleave_H) {
  const long long total = rows * cols_pad;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols_pad; const int c = (int)(i % cols_pad);
    const long long sr = interleave_H ? (r & 3) * interleave_H + (r >> 2) : r;
    dst[r * ld_dst + c] = from_f32<TO>((src && c < cols) ? src[sr * ld_src + c] : 0.f);
  }
}

template <typename TO>
struct Stager {
  StageTable t;
  struct Scalar { const float* src; long long ld_src; TO* dst; long long ld_dst, rows; int cols, cols_pad, interleave_H; };
  Scalar sc[STAGE_MAX];
  int n_sc = 0;
  bool overflow = false;
  Stager() { t.n = 0; t.blk0[0] = 0; }
  // dst[rows, cols_pad] <- src[rows, cols]  (see above); src == nullptr: zero fill
  void add(const float* src, long long ld_src, TO* dst, long long ld_dst, long long rows, int cols, int cols_pad, int interleave_H = 0) {
    if (rows <= 0 || cols_pad <= 0) return;
    const long long total = rows * cols_pad;
    const bool vec = !(cols & 3) && !(cols_pad & 3) && !(ld_dst & 3) && !(reinterpret_cast<uintptr_t>(dst) & 15) &&
                     (!src || (!(ld_src & 3) && !(reinterpret_cast<uintptr_t>(src) & 15))) && total / 4 < (1ll << 31) &&
                     ld_src < (1ll << 31) && ld_dst < (1ll << 31) && rows < (1ll << 31);
    if (vec && t.n < STAGE_MAX) {
      StageItem& it = t.it[t.n];
      it.src = src; it.dst = dst; it.ld_src = (unsigned)ld_src; it.ld_dst = (unsigned)ld_dst; it.rows = (unsigned)rows;
      it.cols4 = (unsigned)cols / 4; it.cp4 = (unsigned)cols_pad / 4; it.interleave_H = (unsigned)interleave_H;
      const long long total4 = total / 4;
      long long nb = (total4 + 256 * 8 - 1) / (256 * 8);
      if (nb > 148 * 8) nb = 148 * 8;
      t.blk0[t.n + 1] = t.blk0[t.n] + (unsigned)nb;
      ++t.n;
    } else if (n_sc < STAGE_MAX) {
      sc[n_sc++] = Scalar{src, ld_src, dst, ld_dst, rows, cols, cols_pad, interleave_H};
    } else {
      overflow = true;
    }
  }
  // zero `bytes` bytes at p (a multiple of 4 elements of TO, 16-byte aligned -- every workspace slice is)
  void zero(void* p, size_t bytes) { add(nullptr, 0, reinterpret_cast<TO*>(p), (long long)(bytes / sizeof(TO)), 1, 0, (int)(bytes / sizeof(TO))); }
  int launch(cudaStream_t st) {
    if (overflow) return RECNET_ERR_BAD_SHAPE;
    if (t.n > 0) {
      stage_multi_kernel<TO><<<t.blk0[t.n], 256, 0, st>>>(t);
      RN_LAUNCH_OK();
    }
    for (int i = 0; i < n_sc; ++i) {
      const Scalar& x = sc[i];
      const long long total = x.rows * x.cols_pad;
      const int blocks = (int)min((long long)148 * 16, (total + 255) / 256);
      stage_scalar_kernel<TO><<<blocks, 256, 0, st>>>(x.src, x.ld_src, x.dst, x.ld_dst, x.rows, x.cols, x.cols_pad, x.interleave_H);
      RN_LAUNCH_OK();
    }
    return 0;
  }
};

// Xe[r, c] = emb[tok[r], c] * scale * dropmask   (c < EMB), 0 for the K padding.  The mask of row r is that of row row0 + r of the
// site's tensor: a decode loop gathers one step of B rows at a time, row0 = t * B.
template <typename TO>
__global__ void embed_gather_kernel(const float* __restrict__ emb, const long long* __restrict__ tok, TO* __restrict__ out,
                                    long long ld_out, int rows, int EMB, int EMBp, int V, float scale, float p_drop,
                                    const unsigned long long* rng, unsigned int site, long long row0 = 0) {
  const int r = blockIdx.x;
  long long t = tok[r];
  if (t < 0 || t >= V) t = 0;
  for (int c = threadIdx.x; c < EMBp; c += blockDim.x) {
    float v = 0.f;
    if (c < EMB) {
      v = emb[t * EMB + c] * scale;
      if (p_drop > 0.f) v *= dropout_scale(rng, site, (uint64_t)(row0 + r) * EMB + c, p_drop);
    }
    out[(long long)r * ld_out + c] = from_f32<TO>(v);
  }
}
// dEmb[tok[r], c] += dXe[r, c] * scale * dropmask
__global__ void embed_scatter_kernel(float* __restrict__ demb, const long long* __restrict__ tok, const float* __restrict__ dxe,
                                     long long ld, int rows, int EMB, int V, float scale, float p_drop,
                                     const unsigned long long* rng, unsigned int site) {
  const int r = blockIdx.x;
  long long t = tok[r];
  if (t < 0 || t >= V) return;
  for (int c = threadIdx.x; c < EMB; c += blockDim.x) {
    float v = dxe[(long long)r * ld + c] * scale;
    if (p_drop > 0.f) v *= dropout_scale(rng, site, (uint64_t)r * EMB + c, p_drop);
    atomicAdd(demb + t * EMB + c, v);
  }
}

// out[n] (+)= sum_m X[m*ld + n]      block = 32 columns x 8 row-lanes; blockIdx.y = row chunk (two-stage, fixed order)
template <typename T>
__global__ void colsum_kernel(const T* __restrict__ X, long long ld, int M, int N, int rows_per_chunk, float* __restrict__ out,
                              int accumulate, float* __restrict__ out2 = nullptr) {
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int n = blockIdx.x * 32 + tx;
  const int m_lo = blockIdx.y * rows_per_chunk, m_hi = min(M, m_lo + rows_per_chunk);
  float s = 0.f;
  if (n < N) {
    int m = m_lo + ty;
    for (; m + 24 < m_hi; m += 32) {       // 4 independent row loads in flight
      const float v0 = to_f32<T>(X[(long long)m * ld + n]), v1 = to_f32<T>(X[(long long)(m + 8) * ld + n]);
      const float v2 = to_f32<T>(X[(long long)(m + 16) * ld + n]), v3 = to_f32<T>(X[(long long)(m + 24) * ld + n]);
      s += (v0 + v1) + (v2 + v3);
    }
    for (; m < m_hi; m += 8) s += to_f32<T>(X[(long long)m * ld + n]);
  }
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][tx];
    float* o = out + (long long)blockIdx.y * N + n;
    const float r = (accumulate && gridDim.y == 1) ? *o + t : t;
    *o = r;
    if (out2 && gridDim.y == 1) out2[n] = r;
  }
}
__global__ void colsum_finish_kernel(const float* __restrict__ part, int chunks, int N, float* __restrict__ out, int accumulate,
                                     float* __restrict__ out2 = nullptr) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float s = 0.f;
  for (int c = 0; c < chunks; ++c) s += part[(long long)c * N + n];
  const float r = accumulate ? out[n] + s : s;
  out[n] = r;
  if (out2) out2[n] = r;
}
// Vectorised variant: a thread owns VEC = 16 / sizeof(T) consecutive columns (one 16-byte load per row), block = 32 column groups x 8 row lanes.
template <typename T>
__global__ void colsum_vec_kernel(const T* __restrict__ X, long long ld, int M, int N, int rows_per_chunk, float* __restrict__ out,
                                  int accumulate, float* __restrict__ out2) {
  constexpr int VEC = 16 / (int)sizeof(T);
  __shared__ float red[8][32 * VEC + 1];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int n0 = (blockIdx.x * 32 + tx) * VEC;
  const int m_lo = blockIdx.y * rows_per_chunk, m_hi = min(M, m_lo + rows_per_chunk);
  float s[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) s[j] = 0.f;
  if (n0 < N) {                                   // the last group may reach into the row padding (round_up(N, VEC) <= ld, checked by the launcher)
    auto add = [&](const uint4& v) {
      const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
      for (int j = 0; j < VEC; ++j) s[j] += to_f32<T>(e[j]);
    };
    int m = m_lo + ty;
    for (; m + 56 < m_hi; m += 64) {              // 8 independent 16-byte loads in flight (at most 48 CTAs run: memory-level parallelism per SM matters)
      uint4 v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = *reinterpret_cast<const uint4*>(X + (long long)(m + 8 * u) * ld + n0);
#pragma unroll
      for (int u = 0; u < 8; ++u) add(v[u]);
    }
    for (; m < m_hi; m += 8) add(*reinterpret_cast<const uint4*>(X + (long long)m * ld + n0));
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j) red[ty][tx * VEC + j] = s[j];
  __syncthreads();
  for (int c = threadIdx.x; c < 32 * VEC; c += blockDim.x) {
    const int n = blockIdx.x * 32 * VEC + c;
    if (n >= N) continue;
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][c];
    float* o = out + (long long)blockIdx.y * N + n;
    const float r = (accumulate && gridDim.y == 1) ? *o + t : t;
    *o = r;
    if (out2 && gridDim.y == 1) out2[n] = r;
  }
}
// scratch: >= 64 * N floats (only used when M is large enough to be worth a second stage)
// out2 (optional): a second copy of the result (b_hh gets the same gradient as b_ih in an LSTM: one node instead of a memcpy)
template <typename T>
static int colsum(const T* X, long long ld, int M, int N, float* out, int accumulate, float* scratch, cudaStream_t st,
                  float* out2 = nullptr) {
  constexpr int VEC = 16 / (int)sizeof(T);
  const bool vec = ((N + VEC - 1) / VEC * VEC <= ld) && !(reinterpret_cast<uintptr_t>(X) & 15) && !((ld * (long long)sizeof(T)) & 15) && M >= 64;
  int chunks;
  if (vec) {
    // 16-byte loads.  On a trainer's background lane (rn_background_ctas() > 0) never more CTAs than that budget: the sums run underneath
    // the decoder's backward loop, whose CTAs need whole SMs; elsewhere ~2 CTAs per SM (next to GEMMs on the side stream, a 48-CTA sum over
    // 34 MB crawled: 87 us)
    const int cb = rn_cdiv(N, 32 * VEC);
    const int budget = rn_background_ctas() > 0 ? rn_background_ctas() : 296;
    chunks = scratch ? budget / cb : 1;
    if (chunks > M / 64) chunks = M / 64;
    if (chunks > 64) chunks = 64;
    if (chunks < 1) chunks = 1;
    const int rpc = (M + chunks - 1) / chunks;
    chunks = (M + rpc - 1) / rpc;
    colsum_vec_kernel<T><<<dim3(cb, chunks), 256, 0, st>>>(X, ld, M, N, rpc, chunks > 1 ? scratch : out, accumulate, chunks > 1 ? nullptr : out2);
  } else {
    chunks = (scratch && M >= 512) ? (M + 127) / 128 : 1;
    if (chunks > 64) chunks = 64;
    const int rpc = (M + chunks - 1) / chunks;
    dim3 grid(rn_cdiv(N, 32), chunks);
    colsum_kernel<T><<<grid, 256, 0, st>>>(X, ld, M, N, rpc, chunks > 1 ? scratch : out, accumulate, chunks > 1 ? nullptr : out2);
  }
  RN_LAUNCH_OK();
  if (chunks > 1) {
    colsum_finish_kernel<<<rn_cdiv(N, 256), 256, 0, st>>>(scratch, chunks, N, out, accumulate, out2);
    RN_LAUNCH_OK();
  }
  return 0;
}

// mp[b,j] = (sum_l Hd[l,b,j]) * scale          (global reconstructor mean-pool, scale = cap / L^2 for one decoder layer)
__global__ void pool_time_kernel(const float* __restrict__ Hd, int L, long long n, float scale, float* __restrict__ mp) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int l = 0; l < L; ++l) s += Hd[(long long)l * n + i];
  mp[i] = s * scale;
}
// dHd[l,b,j] (+)= dmp[b,j] * scale   for every l
__global__ void pool_time_bwd_kernel(const float* __restrict__ dmp, int L, long long n, float scale, float* __restrict__ dHd,
                                     int accumulate) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float g = dmp[i] * scale;
  for (int l = 0; l < L; ++l) {
    float* p = dHd + (long long)l * n + i;
    *p = accumulate ? *p + g : g;
  }
}

// Global reconstructor operand rows: Xg[t,b,:] = [Hd[t,b,:], mp[b,:] * dropmask(t,b,:)]   (TO)
// Hd is (L, NLd, B, H): the per-step input is the LAYER-0 state (global_reconstructor.py:40 `input[0]`)
template <typename TO>
__global__ void global_x_kernel(const float* __restrict__ Hd, const float* __restrict__ mp, TO* __restrict__ X, int L, int B,
                                int H, int NLd, float p_drop, const unsigned long long* rng, unsigned int site) {
  const long long total = (long long)L * B * 2 * H;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % (2 * H));
    const long long tb = i / (2 * H);
    const int b = (int)(tb % B);
    const long long t = tb / B;
    float v;
    if (c < H) v = Hd[((t * NLd) * B + b) * H + c];
    else {
      v = mp[(long long)b * H + (c - H)];
      if (p_drop > 0.f) v *= dropout_scale(rng, site, (uint64_t)(tb * H + (c - H)), p_drop);
    }
    X[i] = from_f32<TO>(v);
  }
}
// dmp[b,j] = sum_t dXg[t,b,H+j] * dropmask ; dHd[t,b,j] (+)= dXg[t,b,j]
__global__ void global_x_bwd_kernel(const float* __restrict__ dX, float* __restrict__ dHd, float* __restrict__ dmp, int L, int B,
                                    int H, int NLd, int accumulate, float p_drop, const unsigned long long* rng, unsigned int site) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * H) return;
  const int b = (int)(i / H), j = (int)(i % H);
  float s = 0.f;
  for (int t = 0; t < L; ++t) {
    const long long tb = (long long)t * B + b;
    float g = dX[tb * 2 * H + H + j];
    if (p_drop > 0.f) g *= dropout_scale(rng, site, (uint64_t)(tb * H + j), p_drop);
    s += g;
    float* p = dHd + (((long long)t * NLd) * B + b) * H + j;          // layer-0 slice of (L, NLd, B, H)
    const float d = dX[tb * 2 * H + j];
    *p = accumulate ? *p + d : d;
    if (!accumulate)
      for (int l = 1; l < NLd; ++l) dHd[(((long long)t * NLd + l) * B + b) * H + j] = 0.f;   // other layers: only the pooled term
  }
  dmp[i] = s;
}

// ---- teacher-forcing inputs of train.forward_decoder (train.py:25,44-45,54-60,68) in one launch -------------------------------
//   tokens_in[0, :] = <SOS>; tokens_in[t, :] = targets[t-1, :]
//   ce_weight[t, b] = [targets[t,b] > <PAD>] / (max(n_t, 1) * sum_t n_t),  n_t = #{b : targets[t,b] > <PAD>}
// (mean over the n_t live samples of step t, then the division by sum_t n_t).  One block; L*B is a few thousand.
__global__ void tf_prep_kernel(const long long* __restrict__ targets, int L, int B, long long pad, long long sos,
                               long long* __restrict__ tokens_in, float* __restrict__ ce_weight) {
  extern __shared__ float n_t[];          // [L] + 1
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int t = warp; t < L; t += nw) {
    float c = 0.f;
    for (int b = lane; b < B; b += 32) c += targets[(long long)t * B + b] > pad ? 1.f : 0.f;
    c = warp_sum(c);
    if (lane == 0) n_t[t] = c;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int t = 0; t < L; ++t) tot += n_t[t];
    n_t[L] = tot;
  }
  __syncthreads();
  const float tot = n_t[L];
  for (int i = threadIdx.x; i < L * B; i += blockDim.x) {
    const int t = i / B;
    const float m = targets[i] > pad ? 1.f : 0.f;
    ce_weight[i] = m / (fmaxf(n_t[t], 1.f) * tot);
    tokens_in[i] = t == 0 ? sos : targets[i - B];
  }
}

// ---- multi-tensor L2 norm regulariser: reg = sum_p ||p||_2 ; grad_p (+)= g * p / ||p|| -------------------------
constexpr int MT_CHUNK = 16384;
// table: ptrs[n] (device addresses), sizes[n]; blk_tensor[nb], blk_chunk[nb] map a block to a chunk of one tensor
__global__ void mt_sumsq_kernel(const long long* __restrict__ ptrs, const long long* __restrict__ sizes,
                                const int* __restrict__ blk_tensor, const int* __restrict__ blk_chunk, float* __restrict__ partial) {
  __shared__ float red[32];
  const int t = blk_tensor[blockIdx.x];
  const float* p = reinterpret_cast<const float*>(ptrs[t]);
  const long long n = sizes[t], lo = (long long)blk_chunk[blockIdx.x] * MT_CHUNK, hi = min(n, lo + MT_CHUNK);
  float s = 0.f;
  if (!(reinterpret_cast<uintptr_t>(p) & 15)) {           // chunk offsets are multiples of 4 elements: 16-byte loads
    const long long hi4 = lo + ((hi - lo) & ~3ll);
    for (long long i = lo + 4 * threadIdx.x; i < hi4; i += 4 * blockDim.x) {
      const float4 v = *reinterpret_cast<const float4*>(p + i);
      s += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
    }
    for (long long i = hi4 + threadIdx.x; i < hi; i += blockDim.x) { const float v = p[i]; s += v * v; }
  } else {
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) { const float v = p[i]; s += v * v; }
  }
  s = block_sum(s, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;          // fixed-order two-stage reduction: bitwise reproducible
}
// warp t sums tensor t's block partials (lane-strided, fixed order => reproducible), then reg = sum_t sqrt(sumsq[t])
__global__ void mt_norm_finalize_kernel(const float* __restrict__ partial, const int* __restrict__ blk_tensor, int n_blocks,
                                        float* __restrict__ sumsq, int n, float* __restrict__ out, const float* __restrict__ base = nullptr,
                                        const float* __restrict__ lambda_dev = nullptr, float* __restrict__ fused_out = nullptr) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int t = warp; t < n; t += nw) {
    float s = 0.f;
    for (int b = lane; b < n_blocks; b += 32) if (blk_tensor[b] == t) s += partial[b];
    s = warp_sum(s);
    if (lane == 0) sumsq[t] = s;
  }
  __syncthreads();                      // sumsq[] written by this block is visible to thread 0 (any number of tensors)
  if (threadIdx.x == 0) {
    float r = 0.f;
    for (int t = 0; t < n; ++t) r += sqrtf(sumsq[t]);
    out[0] = r;
    // loss assembly of train.py:70,102,128 folded in: fused = base + lambda * reg (saves two elementwise graph nodes per module)
    if (fused_out) fused_out[0] = (base ? base[0] : 0.f) + (lambda_dev ? lambda_dev[0] : 1.f) * r;
  }
}
__global__ void mt_reg_grad_kernel(const long long* __restrict__ ptrs, const long long* __restrict__ gptrs,
                                   const long long* __restrict__ sizes, const int* __restrict__ blk_tensor,
                                   const int* __restrict__ blk_chunk, const float* __restrict__ sumsq,
                                   const float* __restrict__ gscale, float lambda, int accumulate,
                                   const float* __restrict__ lambda_dev = nullptr) {
  const int t = blk_tensor[blockIdx.x];
  const float* p = reinterpret_cast<const float*>(ptrs[t]);
  float* g = reinterpret_cast<float*>(gptrs[t]);
  const long long n = sizes[t], lo = (long long)blk_chunk[blockIdx.x] * MT_CHUNK, hi = min(n, lo + MT_CHUNK);
  const float nrm = sqrtf(sumsq[t]);
  const float k = (nrm > 0.f) ? lambda * (gscale ? *gscale : 1.f) * (lambda_dev ? *lambda_dev : 1.f) / nrm : 0.f;
  if (!((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g)) & 15)) {
    const long long hi4 = lo + ((hi - lo) & ~3ll);
    for (long long i = lo + 4 * threadIdx.x; i < hi4; i += 4 * blockDim.x) {
      const float4 v = *reinterpret_cast<const float4*>(p + i);
      float4 o = accumulate ? *reinterpret_cast<const float4*>(g + i) : make_float4(0.f, 0.f, 0.f, 0.f);
      o.x = fmaf(k, v.x, o.x); o.y = fmaf(k, v.y, o.y); o.z = fmaf(k, v.z, o.z); o.w = fmaf(k, v.w, o.w);
      *reinterpret_cast<float4*>(g + i) = o;
    }
    for (long long i = hi4 + threadIdx.x; i < hi; i += blockDim.x) g[i] = fmaf(k, p[i], accumulate ? g[i] : 0.f);
  } else {
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) g[i] = fmaf(k, p[i], accumulate ? g[i] : 0.f);
  }
}
// x[r, c] = x[r, c] * scale + bias[c]   (hoisted embedding projection table of the greedy decoder)
__global__ void scale_add_bias_kernel(float* __restrict__ x, long long total, int cols, float scale, const float* __restrict__ bias) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    x[i] = fmaf(x[i], scale, bias[(int)(i % cols)]);
}
}  // namespace misc
