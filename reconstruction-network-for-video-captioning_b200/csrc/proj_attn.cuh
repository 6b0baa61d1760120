// Projected-feature attention fused with the LSTM cell (decoder hot path, models/decoder.py:50-66).
//
// The reference's attention has NO softmax: ctx_t[b] = (1/T) sum_tau e_t[b,tau] * v[b,tau]  (decoder.py:57-62) and the
// context only ever enters the step through the LSTM input projection ctx_t W_ctx^T (decoder.py:64-66).  Both are
// linear, so    ctx_t[b] W_ctx^T = (1/T) sum_tau e_t[b,tau] * (v[b,tau] W_ctx^T) = (1/T) sum_tau e_t[b,tau] * VW[b,tau]
// with VW = feats W_ctx^T computed ONCE per sequence (one 2800 x 2048 x 1536 tensor-core GEMM) instead of a
// [100 x 1536] x [1536 x 2048] GEMM in every one of the 31 steps.  What is left per step:
//   K1  h_{t-1} [W_a ; W_hh]^T          one split-K tcgen05 GEMM, K = H = 512 (attention query + recurrent gates together)
//   K2  pf_fwd_kernel                   scores e_t, the 28-frame weighted sum of VW, gate activations, c_t, h_t  (this file)
// and in BPTT
//   K3  pf_bwd_kernel                   cell backward -> dG_t, d e_t = <dG_t, VW>, score backward -> dWh_t, dUv, dw
//   K4  [dWh_t | dG_t] [W_a ; W_hh]     one split-K GEMM, K = A + 4H -> dh_{t-1}
// i.e. 2 + 2 dependent kernels per step instead of 4 + 4, and the per-step weight traffic drops from 8.4 MB to 2.2 MB.
// dW_ctx = dG^T ctx with ctx_t[b] = (1/T) sum_tau e_t[b,tau] v[b,tau] (pf_escore_kernel<.., true>, in the forward pass next to the vocabulary GEMM).
// The paper's softmax attention (SM = true, opt-in) keeps all of this: alpha_t = softmax_tau(e_t) takes the place of e_t and the scale is
// 1 instead of 1/T (the drivers pass inv_T = 1); the e stash holds alpha, and the backward turns d alpha into d e with
// d e[tau] = alpha[tau] (d alpha[tau] - sum_s alpha[s] d alpha[s]) before the unchanged score backward.
//
// VW and the gate stash are stored "unit-interleaved": [.., H, 4] (the 4 gate columns i,f,g,o of one hidden unit
// adjacent) so that one thread fetches its unit's 4 columns of a frame with ONE 8-byte (bf16) / 16-byte (fp32) load.
#pragma once
#include "common.cuh"

namespace pf {
constexpr int THREADS = 256;
constexpr int UPB = 128;        // hidden units per forward CTA (2 frame-halves x 128 units = 256 threads)
constexpr int MAX_T = 64;       // frames
constexpr int MAX_A = 256;      // attention size (<= 2 float4 chunks per lane)
constexpr int NW = THREADS / 32;

template <typename T> struct Quad;
template <> struct Quad<float> {
  float4 r;
  __device__ __forceinline__ void load(const float* p) { r = *reinterpret_cast<const float4*>(p); }
  __device__ __forceinline__ void get(float* f) const { f[0] = r.x; f[1] = r.y; f[2] = r.z; f[3] = r.w; }
  static __device__ __forceinline__ void store(float* p, float a, float b, float c, float d) {
    *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
  }
};
template <> struct Quad<bf16> {
  uint2 r;
  __device__ __forceinline__ void load(const bf16* p) { r = *reinterpret_cast<const uint2*>(p); }
  __device__ __forceinline__ void get(float* f) const {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
    const float2 a = __bfloat1622float2(h[0]), b = __bfloat1622float2(h[1]);
    f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y;
  }
  static __device__ __forceinline__ void store(bf16* p, float a, float b, float c, float d) {
    __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
    *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
  }
};

__device__ __forceinline__ float4 f4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

// Split-K partial sums.  These kernels are latency-bound: every load of a batch is issued before the first add
// (a plain `for (s) acc += q[s * stride]` loop costs one L2 round trip PER SPLIT -- measured 17 us for 17 splits).
__device__ __forceinline__ float sum_splits(const float* __restrict__ q, int n, long long stride) {
  float s = 0.f;
  int p = 0;
  for (; p + 8 <= n; p += 8) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = q[i * stride];
    s += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
    q += 8 * stride;
  }
  if (p + 4 <= n) {
    const float v0 = q[0], v1 = q[stride], v2 = q[2 * stride], v3 = q[3 * stride];
    s += (v0 + v1) + (v2 + v3);
    q += 4 * stride; p += 4;
  }
  if (p + 2 <= n) { const float v0 = q[0], v1 = q[stride]; s += v0 + v1; q += 2 * stride; p += 2; }
  if (p < n) s += q[0];
  return s;
}
__device__ __forceinline__ float4 sum_splits4(const float* __restrict__ q, int n, long long stride) {
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  int p = 0;
  for (; p + 4 <= n; p += 4) {
    const float4 v0 = *reinterpret_cast<const float4*>(q), v1 = *reinterpret_cast<const float4*>(q + stride);
    const float4 v2 = *reinterpret_cast<const float4*>(q + 2 * stride), v3 = *reinterpret_cast<const float4*>(q + 3 * stride);
    s = f4_add(s, f4_add(f4_add(v0, v1), f4_add(v2, v3)));
    q += 4 * stride;
  }
  for (; p < n; ++p) { s = f4_add(s, *reinterpret_cast<const float4*>(q)); q += stride; }
  return s;
}

// ---- forward -----------------------------------------------------------------------------------------------------
struct FwdArgs {
  const float* P; int n_p; long long p_stride; int NP;   // split-K partials of h_{t-1} [W_a ; W_hh]^T: [n_p][B, NP = A + 4H]; n_p = 0 at t = 0
  const float* Uv;                                        // [B, Tn, A]   hoisted U v + attn_b
  const float* attn_w;                                    // [A]
  const void* VW;                                         // [B, Tn, H, 4] TV   hoisted v W_ctx^T, unit-interleaved
  const float* Gx;                                        // [B, 4H]  hoisted embedding projection + b_ih (gate-block order)
  const long long* gx_rows;                               // nullable: row of Gx to use for sample b (greedy decoding: Gx = table over the vocabulary, rows = fed-back tokens)
  const float* b_hh;                                      // [4H]
  const float* c_prev;                                    // [B, H]
  int B, Tn, A, H; float inv_T;
  float* Wh_out; float* e_out;                            // [B, A], [B, Tn]  stash for BPTT (nullable); e_out holds alpha when SM
  void* gates_out;                                        // [B, H, 4] TO      activated gates, unit-interleaved (nullable)
  float* c_out; float* h_out;                             // [B, H] fp32
  void* h_op;                                             // [B, H] TO: next step's GEMM operand row / vocabulary-projection row
};

// NCH = float4 chunks of the attention axis per lane: 1 (A <= 128) or 2 (A <= 256).
// Index math is 32-bit unsigned on purpose (r1 ncu: 42% of the first version's instructions were 64-bit address arithmetic);
// the drivers check that every tensor has < 2^31 elements.  `Uv` already contains the attention bias (folded in at the hoist).
template <typename TV, typename TO, int NCH, int MINB, bool SM>
__global__ void __launch_bounds__(THREADS, MINB) pf_fwd_kernel(FwdArgs a) {
  constexpr bool FAST = FastMath<TO>::value;
  pdl_wait();
  pdl_launch_next();
  __shared__ __align__(16) float e_s[2][MAX_T / 2];     // e_s[tau & 1][tau >> 1]; zero for tau >= Tn
  __shared__ float4 red[UPB];
  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned b = blockIdx.y, u = tid & (UPB - 1), half = tid >> 7;
  const unsigned Tn = a.Tn, H = a.H, A = a.A, row = 4u * H;
  const unsigned j = blockIdx.x * UPB + u;
  const bool unit_ok = j < H;
  const unsigned jc = unit_ok ? j : H - 1;
  // (1) this thread's projected-feature quads of the first 32 frames (frames 2k + half): issued before anything else.
  // (loads are UNCONDITIONAL on clamped indices: a predicated `if (ok) v[k].load()` compiles to load-into-temp + predicated
  //  move and ptxas then keeps only two loads in flight -- measured 18 us instead of 5 for the backward kernel)
  const TV* vw = reinterpret_cast<const TV*>(a.VW) + ((size_t)b * Tn * H + jc) * 4;
  Quad<TV> v[16];
#pragma unroll
  for (unsigned k = 0; k < 16; ++k) v[k].load(vw + min(2 * k + half, Tn - 1) * row);
  if (tid < MAX_T && tid >= Tn) e_s[tid & 1][tid >> 1] = 0.f;
  // (2) the unit's gate pre-activations that do not depend on the attention: half 0 (which owns the cell update) fetches
  //     the hoisted embedding projection, bias and c_{t-1}; half 1 sums the split-K partials of h_{t-1} W_hh^T
  float pre[4] = {0.f, 0.f, 0.f, 0.f};
  float cp = 0.f;
  if (half == 0) {
    const float* gx = a.Gx + (size_t)(a.gx_rows ? (unsigned)a.gx_rows[b] : b) * row + jc;
    const float* bh = a.b_hh + jc;
#pragma unroll
    for (unsigned g = 0; g < 4; ++g) pre[g] = gx[g * H] + bh[g * H];
    cp = a.c_prev[b * H + jc];
  } else {
    const float* q = a.P + (size_t)b * a.NP + A + jc;
    const unsigned ps = (unsigned)a.p_stride;
    int s = 0;
    for (; s + 4 <= a.n_p; s += 4) {             // 16 independent loads in flight
      float x[4][4];
#pragma unroll
      for (unsigned i = 0; i < 4; ++i)
#pragma unroll
        for (unsigned g = 0; g < 4; ++g) x[i][g] = q[i * ps + g * H];
#pragma unroll
      for (int g = 0; g < 4; ++g) pre[g] += (x[0][g] + x[1][g]) + (x[2][g] + x[3][g]);
      q += 4 * ps;
    }
    for (; s < a.n_p; ++s) {
#pragma unroll
      for (unsigned g = 0; g < 4; ++g) pre[g] += q[g * H];
      q += ps;
    }
  }
  // (3) scores e[tau] = w . tanh(W h + (U v_tau + b)): warp w takes frames w, w + 8, ..; a lane takes float4 chunks lane, lane + 32 of A
  const unsigned nchunk = A >> 2;
  const float4* uvb = reinterpret_cast<const float4*>(a.Uv + (size_t)b * Tn * A);
  float4 uv[4][NCH];
#pragma unroll
  for (unsigned f = 0; f < 4; ++f)
#pragma unroll
    for (unsigned i = 0; i < NCH; ++i) uv[f][i] = uvb[min(warp + f * NW, Tn - 1) * nchunk + min(lane + 32 * i, nchunk - 1)];
  float4 wh[NCH], ww[NCH];
#pragma unroll
  for (unsigned i = 0; i < NCH; ++i) {
    const unsigned c = min(lane + 32 * i, nchunk - 1);
    ww[i] = reinterpret_cast<const float4*>(a.attn_w)[c];
    wh[i] = sum_splits4(a.P + (size_t)b * a.NP + 4 * c, a.n_p, a.p_stride);
    if (blockIdx.x == 0 && warp == 0 && a.Wh_out && lane + 32 * i < nchunk) reinterpret_cast<float4*>(a.Wh_out + (size_t)b * A)[c] = wh[i];
  }
  for (unsigned f0 = 0;;) {
#pragma unroll
    for (unsigned f = 0; f < 4; ++f) {
      const unsigned tau = warp + (f0 + f) * NW;
      if (tau < Tn) {               // warp-uniform
        float s = 0.f;
#pragma unroll
        for (unsigned i = 0; i < NCH; ++i) {
          if (NCH == 1 || lane + 32 * i < nchunk) {
            const float4 x = uv[f][i];
            s = fmaf(ww[i].x, act_tanh<FAST>(wh[i].x + x.x), s);
            s = fmaf(ww[i].y, act_tanh<FAST>(wh[i].y + x.y), s);
            s = fmaf(ww[i].z, act_tanh<FAST>(wh[i].z + x.z), s);
            s = fmaf(ww[i].w, act_tanh<FAST>(wh[i].w + x.w), s);
          }
        }
        if (NCH == 1 && lane >= nchunk) s = 0.f;
        s = warp_sum(s);
        if (lane == 0) {
          e_s[tau & 1][tau >> 1] = s;
          if (!SM && blockIdx.x == 0 && a.e_out) a.e_out[b * Tn + tau] = s;
        }
      }
    }
    f0 += 4;
    if (warp + f0 * NW >= Tn) break;
#pragma unroll
    for (unsigned f = 0; f < 4; ++f)
#pragma unroll
      for (unsigned i = 0; i < NCH; ++i) uv[f][i] = uvb[min(warp + (f0 + f) * NW, Tn - 1) * nchunk + min(lane + 32 * i, nchunk - 1)];
  }
  __syncthreads();
  if constexpr (SM) {             // softmax over the (<= 64) frames: warp 0, lane owns frames lane and lane + 32
    if (warp == 0) {
      const unsigned t1 = lane + 32;
      const bool ok0 = lane < Tn, ok1 = t1 < Tn;
      const float x0 = ok0 ? e_s[lane & 1][lane >> 1] : -INFINITY, x1 = ok1 ? e_s[t1 & 1][t1 >> 1] : -INFINITY;
      const float m = warp_max(fmaxf(x0, x1));
      const float p0 = ok0 ? act_exp<FAST>(x0 - m) : 0.f, p1 = ok1 ? act_exp<FAST>(x1 - m) : 0.f;
      const float z = warp_sum(p0 + p1);
      if (ok0) { e_s[lane & 1][lane >> 1] = p0 / z; if (blockIdx.x == 0 && a.e_out) a.e_out[b * Tn + lane] = p0 / z; }
      if (ok1) { e_s[t1 & 1][t1 >> 1] = p1 / z; if (blockIdx.x == 0 && a.e_out) a.e_out[b * Tn + t1] = p1 / z; }
    }
    __syncthreads();
  }
  // (4) weighted sum over this thread's frames (weights of frames >= Tn are zero, their clamped quads are finite)
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (unsigned t0 = 0;;) {
    const float4* e4 = reinterpret_cast<const float4*>(&e_s[half][t0 >> 1]);
#pragma unroll
    for (unsigned k4 = 0; k4 < 4; ++k4) {
      const float4 e = e4[k4];
      const float ev[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
      for (unsigned kk = 0; kk < 4; ++kk) {
        float f[4];
        v[4 * k4 + kk].get(f);
#pragma unroll
        for (int g = 0; g < 4; ++g) acc[g] = fmaf(ev[kk], f[g], acc[g]);
      }
    }
    t0 += 32;
    if (t0 >= Tn) break;
#pragma unroll
    for (unsigned k = 0; k < 16; ++k) v[k].load(vw + min(t0 + 2 * k + half, Tn - 1) * row);
  }
  if (half == 1)
    red[u] = make_float4(fmaf(acc[0], a.inv_T, pre[0]), fmaf(acc[1], a.inv_T, pre[1]), fmaf(acc[2], a.inv_T, pre[2]),
                         fmaf(acc[3], a.inv_T, pre[3]));
  __syncthreads();
  if (half == 0 && unit_ok) {
    const float4 o = red[u];
    const float pi = fmaf(acc[0], a.inv_T, pre[0]) + o.x, pf_ = fmaf(acc[1], a.inv_T, pre[1]) + o.y;
    const float pg = fmaf(acc[2], a.inv_T, pre[2]) + o.z, po = fmaf(acc[3], a.inv_T, pre[3]) + o.w;
    const float gi = act_sigmoid<FAST>(pi), gf = act_sigmoid<FAST>(pf_), gg = act_tanh<FAST>(pg), go = act_sigmoid<FAST>(po);
    const float cn = fmaf(gf, cp, gi * gg);
    const float hn = go * act_tanh<FAST>(cn);
    const unsigned o1 = b * H + j;
    a.c_out[o1] = cn;
    a.h_out[o1] = hn;
    reinterpret_cast<TO*>(a.h_op)[o1] = from_f32<TO>(hn);
    if (a.gates_out) Quad<TO>::store(reinterpret_cast<TO*>(a.gates_out) + (size_t)o1 * 4, gi, gf, gg, go);
  }
}

// ---- backward ----------------------------------------------------------------------------------------------------
struct BwdArgs {
  const float* dh_ext; const float* dh_ext2;            // [B, H] each (nullable): vocabulary-projection path, reconstructor path
  const float* dhP; int n_p; long long p_stride;        // split-K partials of [dWh | dG]_{t+1} [W_a ; W_hh]: [n_p][B, H] (nullable at the last step)
  float* dc; int first;                                 // [B, H] in/out; first => treated as 0
  const void* gates;                                    // [B, H, 4] TO
  const float* c_prev; const float* c_new;              // [B, H]
  const void* VW;                                       // [B, Tn, H, 4] TV
  const float* Wh; const float* Uv; const float* attn_w;  // Uv = hoisted U v + attn_b
  int B, Tn, A, H; float inv_T;
  void* dGW; long long dgw_ld;                          // [B, A + 4H] TO: [dWh | dG (gate-block order)]  -> operand of K4 and of the weight-gradient GEMMs
  float* dWh_out;                                       // [B, A] fp32 (attn_b gradient)
  float* dUv_acc; int uv_first;                         // [B, Tn, A] accumulated over steps
  float* dw_acc; int dw_first;                          // [B, A]     accumulated over steps
  const float* alpha;                                   // [B, Tn] softmax weights of the step (SM only)
};

// sum over the 32 lanes of v[k] for every k; lane l ends up with the total of v[l] (31 shuffles instead of 160)
__device__ __forceinline__ float warp_transpose_sum32(float (&v)[32], int lane) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) {
    const bool upper = (lane & s) != 0;
#pragma unroll
    for (int i = 0; i < s; ++i) {
      const float send = upper ? v[i] : v[i + s];
      const float keep = upper ? v[i + s] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
    }
  }
  return v[0];
}

constexpr int MAXS = 12;        // split-K partials summed with one batch of loads (the drivers plan <= MAXS splits)

// operands of one hidden unit's cell backward, all fetched before the first use
template <typename TO>
struct CellIn {
  Quad<TO> gq; float cp, cn, dcn, dhe, dhe2; float part[MAXS];
  __device__ __forceinline__ void load(const BwdArgs& a, long long o1) {
    gq.load(reinterpret_cast<const TO*>(a.gates) + o1 * 4);
    cp = a.c_prev[o1]; cn = a.c_new[o1];
    dcn = a.first ? 0.f : a.dc[o1];
    dhe = a.dh_ext ? a.dh_ext[o1] : 0.f;
    dhe2 = a.dh_ext2 ? a.dh_ext2[o1] : 0.f;
    if (a.dhP) {                                     // uniform branch; clamped split index -> unconditional loads
#pragma unroll
      for (int s = 0; s < MAXS; ++s) part[s] = a.dhP[o1 + (long long)min(s, a.n_p - 1) * a.p_stride];
    } else {
#pragma unroll
      for (int s = 0; s < MAXS; ++s) part[s] = 0.f;
    }
  }
  __device__ __forceinline__ float dh(const BwdArgs& a, long long o1) const {
    float d = dhe + dhe2;
    if (a.dhP) {
#pragma unroll
      for (int s = 0; s < MAXS; ++s) d += (s < a.n_p) ? part[s] : 0.f;
      if (a.n_p > MAXS) d += sum_splits(a.dhP + o1 + (long long)MAXS * a.p_stride, a.n_p - MAXS, a.p_stride);
    }
    return d;
  }
};

// cell backward of one unit (same math as cell::lstm_cell_bwd_body); returns the operand-rounded gate gradients
template <typename TO, bool FAST>
__device__ __forceinline__ float4 cell_bwd_unit(const BwdArgs& a, const CellIn<TO>& in, int b, int j, bool ok) {
  const long long o1 = (long long)b * a.H + j;
  float g[4];
  in.gq.get(g);
  const float dh = in.dh(a, o1);
  const float tc = act_tanh<FAST>(in.cn);
  const float dc = fmaf(dh * g[3], 1.f - tc * tc, in.dcn);
  const float di = dc * g[2] * g[0] * (1.f - g[0]);
  const float df = dc * in.cp * g[1] * (1.f - g[1]);
  const float dgg = dc * g[0] * (1.f - g[2] * g[2]);
  const float dO = dh * tc * g[3] * (1.f - g[3]);
  const TO r0 = from_f32<TO>(di), r1 = from_f32<TO>(df), r2 = from_f32<TO>(dgg), r3 = from_f32<TO>(dO);
  if (!ok) return make_float4(0.f, 0.f, 0.f, 0.f);
  a.dc[o1] = dc * g[1];
  TO* o = reinterpret_cast<TO*>(a.dGW) + (long long)b * a.dgw_ld + a.A + j;
  o[0] = r0; o[a.H] = r1; o[2 * a.H] = r2; o[3 * a.H] = r3;
  // the score gradient sees exactly what the GEMMs see: the operand-rounded values
  return make_float4(to_f32<TO>(r0), to_f32<TO>(r1), to_f32<TO>(r2), to_f32<TO>(r3));
}

// One CTA of 512 threads per sample.  r1 ncu of the first version (256 threads, thread-owns-unit, 28 partial sums per
// thread transposed across the warp): 2600 instructions per warp at 2 warps per scheduler -> instruction-latency bound,
// 10 us.  Now: (A) the cell backward runs one unit per thread and leaves the (operand-rounded) gate gradients in shared
// memory; (B) warp w owns the frames w, w + 16, ..: its lanes stream whole VW rows against the shared gate gradients, one
// warp_sum per frame gives d e[tau] in every lane, and (C) the same warp does the score backward of its frames.  Every
// load that does not depend on a previous phase is issued at kernel entry.
// dynamic shared memory: H float4 (gate gradients) + 2 * BNW * A floats (per-warp dWh / dw partials)
constexpr int BTHREADS = 512;
constexpr int BNW = BTHREADS / 32;
template <typename TV, typename TO, int NF, int NCH, bool SM>
__global__ void __launch_bounds__(BTHREADS) pf_bwd_kernel(BwdArgs a) {
  constexpr bool FAST = FastMath<TO>::value;
  constexpr int QP = 32 / NF;                           // VW quads per lane, frame and pass (32 quads = 64 registers in flight)
  pdl_wait();
  pdl_launch_next();
  extern __shared__ float4 dg_s[];                      // [H]
  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned b = blockIdx.x, Tn = a.Tn, H = a.H, A = a.A, row = 4u * H, nchunk = A >> 2;
  float* part = reinterpret_cast<float*>(dg_s + H);     // [2][BNW][A]
  const TV* vwb = reinterpret_cast<const TV*>(a.VW) + (size_t)b * Tn * row;
  unsigned tauc[NF];
#pragma unroll
  for (unsigned f = 0; f < NF; ++f) tauc[f] = min(warp + f * BNW, Tn - 1);
  // ---- issue: cell operands of unit tid, the first VW pass of this warp's frames, the score operands
  CellIn<TO> in;
  in.load(a, (long long)(b * H + min(tid, H - 1)));
  Quad<TV> v[NF][QP];
#pragma unroll
  for (unsigned f = 0; f < NF; ++f)
#pragma unroll
    for (unsigned q = 0; q < QP; ++q) v[f][q].load(vwb + tauc[f] * row + min(lane + 32 * q, H - 1) * 4);
  const float4* uvb = reinterpret_cast<const float4*>(a.Uv + (size_t)b * Tn * A);
  float4* dub = reinterpret_cast<float4*>(a.dUv_acc + (size_t)b * Tn * A);
  float4 uv[NF][NCH], old[NF][NCH], wh[NCH], ww[NCH];
#pragma unroll
  for (unsigned i = 0; i < NCH; ++i) {
    const unsigned cc = min(lane + 32 * i, nchunk - 1);
    wh[i] = reinterpret_cast<const float4*>(a.Wh + (size_t)b * A)[cc];          // Uv already contains attn_b
    ww[i] = reinterpret_cast<const float4*>(a.attn_w)[cc];
#pragma unroll
    for (unsigned f = 0; f < NF; ++f) uv[f][i] = uvb[tauc[f] * nchunk + cc];
  }
  float al[NF];
  if constexpr (SM) {
#pragma unroll
    for (unsigned f = 0; f < NF; ++f) al[f] = warp + f * BNW < Tn ? a.alpha[b * Tn + warp + f * BNW] : 0.f;
  }
  // ---- (A) LSTM cell backward, one unit per thread and pass
  for (unsigned j0 = 0; j0 < H; j0 += BTHREADS) {
    const unsigned j = j0 + tid;
    if (j0 != 0) in.load(a, (long long)(b * H + min(j, H - 1)));
    const float4 dg = cell_bwd_unit<TO, FAST>(a, in, b, min(j, H - 1), j < H);
    if (j < H) dg_s[j] = dg;
  }
#pragma unroll
  for (unsigned i = 0; i < NCH; ++i)
#pragma unroll
    for (unsigned f = 0; f < NF; ++f)
      old[f][i] = a.uv_first ? make_float4(0.f, 0.f, 0.f, 0.f) : dub[tauc[f] * nchunk + min(lane + 32 * i, nchunk - 1)];
  __syncthreads();
  // ---- (B) d e[tau] = (1/T) <dG, VW[tau]> for this warp's frames
  float de[NF];
#pragma unroll
  for (unsigned f = 0; f < NF; ++f) de[f] = 0.f;
  for (unsigned q0 = 0; q0 < H; q0 += 32 * QP) {
    if (q0 != 0) {
#pragma unroll
      for (unsigned f = 0; f < NF; ++f)
#pragma unroll
        for (unsigned q = 0; q < QP; ++q) v[f][q].load(vwb + tauc[f] * row + min(q0 + lane + 32 * q, H - 1) * 4);
    }
#pragma unroll
    for (unsigned q = 0; q < QP; ++q) {
      const unsigned unit = q0 + lane + 32 * q;
      float4 dg = dg_s[min(unit, H - 1)];
      if (unit >= H) dg = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (unsigned f = 0; f < NF; ++f) {
        float x[4];
        v[f][q].get(x);
        de[f] = fmaf(dg.x, x[0], fmaf(dg.y, x[1], fmaf(dg.z, x[2], fmaf(dg.w, x[3], de[f]))));
      }
    }
  }
#pragma unroll
  for (unsigned f = 0; f < NF; ++f) de[f] = warp_sum(de[f]) * a.inv_T;
  if constexpr (SM) {             // de = d alpha so far: d e = alpha (d alpha - sum_s alpha[s] d alpha[s]), the sum over every warp's frames
    __shared__ float sad[BNW];
    float s1 = 0.f;
#pragma unroll
    for (unsigned f = 0; f < NF; ++f) s1 = fmaf(al[f], de[f], s1);
    if (lane == 0) sad[warp] = s1;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (unsigned w = 0; w < BNW; ++w) tot += sad[w];
#pragma unroll
    for (unsigned f = 0; f < NF; ++f) de[f] = al[f] * (de[f] - tot);
  }
  // ---- (C) score backward of the same frames: ds = de * w * (1 - tanh^2); dWh = sum_tau ds; dUv[tau] += ds; dw += de * tanh
  float4 dwh[NCH], dww[NCH];
#pragma unroll
  for (unsigned i = 0; i < NCH; ++i) dwh[i] = dww[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (unsigned f = 0; f < NF; ++f) {
    const unsigned tau = warp + f * BNW;
    if (tau < Tn) {                                     // warp-uniform
      const float g = de[f];
#pragma unroll
      for (unsigned i = 0; i < NCH; ++i) {
        const unsigned c = lane + 32 * i;
        if (c < nchunk) {
          const float4 x = uv[f][i];
          const float tx = act_tanh<FAST>(wh[i].x + x.x), ty = act_tanh<FAST>(wh[i].y + x.y);
          const float tz = act_tanh<FAST>(wh[i].z + x.z), tw = act_tanh<FAST>(wh[i].w + x.w);
          const float4 ds = make_float4(g * ww[i].x * (1.f - tx * tx), g * ww[i].y * (1.f - ty * ty), g * ww[i].z * (1.f - tz * tz),
                                        g * ww[i].w * (1.f - tw * tw));
          dwh[i] = f4_add(dwh[i], ds);
          dww[i] = f4_add(dww[i], make_float4(g * tx, g * ty, g * tz, g * tw));
          dub[tau * nchunk + c] = f4_add(ds, old[f][i]);
        }
      }
    }
  }
#pragma unroll
  for (unsigned i = 0; i < NCH; ++i) {
    const unsigned c = lane + 32 * i;
    if (c < nchunk) {
      reinterpret_cast<float4*>(part + warp * A)[c] = dwh[i];
      reinterpret_cast<float4*>(part + (BNW + warp) * A)[c] = dww[i];
    }
  }
  __syncthreads();
  for (unsigned x = tid; x < A; x += BTHREADS) {
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (unsigned w = 0; w < BNW; ++w) { s0 += part[w * A + x]; s1 += part[(BNW + w) * A + x]; }
    a.dWh_out[b * A + x] = s0;
    reinterpret_cast<TO*>(a.dGW)[(size_t)b * a.dgw_ld + x] = from_f32<TO>(s0);
    float* pw = a.dw_acc + b * A + x;
    *pw = a.dw_first ? s1 : *pw + s1;
  }
}

// 256 threads x 2 adjacent columns, float4 broadcast reads of the scores from shared memory (the first version read e one float at a time and was
// LDS-issue bound, 53 us)
template <typename T> struct Pair;
template <> struct Pair<float> {
  static __device__ __forceinline__ float2 load(const float* p) { return *reinterpret_cast<const float2*>(p); }
  static __device__ __forceinline__ void store(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
};
template <> struct Pair<bf16> {
  static __device__ __forceinline__ float2 load(const bf16* p) { return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p)); }
  static __device__ __forceinline__ void store(bf16* p, float a, float b) { *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(a, b); }
};
// Small per-sample products with the attention scores e[t, b, tau] (L steps x Tn frames), 2 output columns per thread, grid (N / 512, B):
//   CTX = false:  out[b, tau, n] = inv_T sum_t   e[t, b, tau] X[(t, b), n]       (dVW: gradient of the projected features; rows of X = steps)
//   CTX = true :  out[t, b, n]   = inv_T sum_tau e[t, b, tau] X[(b, tau), n]     (the attention context of every step; rows of X = frames)
// S = number of summed rows (L resp. Tn), K = number of output rows per sample (Tn resp. L).  e is staged in shared memory as [S][Kp].
template <typename TO, bool CTX>
__global__ void __launch_bounds__(256) pf_escore_kernel(const float* __restrict__ e, const TO* __restrict__ X, long long ld, int col0,
                                                        TO* __restrict__ out, int L, int B, int Tn, int N, float inv_T, int spc) {
  // spc = samples per CTA (blockIdx.y covers samples [y * spc, (y + 1) * spc)): the launcher keeps the grid within ONE wave, so that a
  // persistent GEMM launched next to it never queues behind a second wave of these CTAs (CTAs are dispatched in launch order)
  extern __shared__ float4 e_sm4[];                     // [round_up(S, 16)][Kp], zero beyond S / K
  float* e_sm = reinterpret_cast<float*>(e_sm4);
  const int S = CTX ? Tn : L, K = CTX ? L : Tn;
  const int Kp = (K + 3) & ~3, Sp = (S + 15) & ~15;
  const int n = (blockIdx.x * 256 + threadIdx.x) * 2;
  for (int b = blockIdx.y * spc; b < min(B, (int)(blockIdx.y + 1) * spc); ++b) {
  __syncthreads();                                      // the previous sample's scores are no longer read
  for (int i = threadIdx.x; i < Sp * Kp; i += 256) {
    const int s_ = i / Kp, k = i - s_ * Kp;
    const int t = CTX ? k : s_, tau = CTX ? s_ : k;
    e_sm[i] = (s_ < S && k < K) ? e[((long long)t * B + b) * Tn + tau] : 0.f;
  }
  __syncthreads();
  if (n >= N) continue;
  for (int k0 = 0; k0 < K; k0 += 32) {
    float acc[32][2];
#pragma unroll
    for (int k = 0; k < 32; ++k) acc[k][0] = acc[k][1] = 0.f;
    for (int s0 = 0; s0 < S; s0 += 16) {
      float2 x[16];                                     // 16 summed rows of this column pair in flight at once
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const int s_ = min(s0 + k, S - 1);
        const long long row = CTX ? (long long)b * Tn + s_ : (long long)s_ * B + b;
        x[k] = Pair<TO>::load(X + row * ld + col0 + n);
      }
#pragma unroll
      for (int ss = 0; ss < 16; ++ss) {                 // rows >= S carry zero weights
        const float4* er = e_sm4 + ((s0 + ss) * Kp + k0) / 4;
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) {
          if (k0 + 4 * k4 < K) {
            const float4 e4 = er[k4];
            acc[4 * k4 + 0][0] = fmaf(e4.x, x[ss].x, acc[4 * k4 + 0][0]); acc[4 * k4 + 0][1] = fmaf(e4.x, x[ss].y, acc[4 * k4 + 0][1]);
            acc[4 * k4 + 1][0] = fmaf(e4.y, x[ss].x, acc[4 * k4 + 1][0]); acc[4 * k4 + 1][1] = fmaf(e4.y, x[ss].y, acc[4 * k4 + 1][1]);
            acc[4 * k4 + 2][0] = fmaf(e4.z, x[ss].x, acc[4 * k4 + 2][0]); acc[4 * k4 + 2][1] = fmaf(e4.z, x[ss].y, acc[4 * k4 + 2][1]);
            acc[4 * k4 + 3][0] = fmaf(e4.w, x[ss].x, acc[4 * k4 + 3][0]); acc[4 * k4 + 3][1] = fmaf(e4.w, x[ss].y, acc[4 * k4 + 3][1]);
          }
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 32; ++k)
      if (k0 + k < K) {
        const long long row = CTX ? (long long)(k0 + k) * B + b : (long long)b * Tn + k0 + k;
        Pair<TO>::store(out + row * N + n, acc[k][0] * inv_T, acc[k][1] * inv_T);
      }
  }
  }   // samples of this CTA
}
// samples per CTA so that the grid (ceil(N / 512) column blocks x ceil(B / spc)) fits one wave of `sms` CTAs
static inline int escore_spc(int N, int B, int sms) {
  const int cb = (N + 511) / 512;
  int spc = (cb * B + sms - 1) / sms;
  return spc < 1 ? 1 : spc;
}
static inline size_t escore_smem(int L, int Tn, bool ctx) {
  const int S = ctx ? Tn : L, K = ctx ? L : Tn;
  return (size_t)((S + 15) & ~15) * ((K + 3) & ~3) * sizeof(float);
}

// dst[(4j + g), :] = (TO) src[(g H + j), :]   -- W_ctx rows in unit-interleaved order (makes the VW GEMM emit [.., H, 4])
// one block per destination row, float4 groups per thread when cols % 4 == 0 (grid = 4H blocks)
template <typename TO>
__global__ void interleave_rows_kernel(const float* __restrict__ src, long long ld_src, TO* __restrict__ dst, int H, int cols) {
  const int r = blockIdx.x, j = r >> 2, g = r & 3;
  const float* s = src + ((long long)g * H + j) * ld_src;
  TO* d = dst + (long long)r * cols;
  if (!(cols & 3) && !(ld_src & 3) && !(reinterpret_cast<uintptr_t>(src) & 15)) {
    for (int c4 = threadIdx.x; c4 < (cols >> 2); c4 += blockDim.x) {
      const float4 v = reinterpret_cast<const float4*>(s)[c4];
      Quad<TO>::store(d + 4 * c4, v.x, v.y, v.z, v.w);
    }
  } else {
    for (int c = threadIdx.x; c < cols; c += blockDim.x) d[c] = from_f32<TO>(s[c]);
  }
}

static inline int check_shape(int Tn, int A, int H) {
  if (Tn < 1 || Tn > MAX_T || A < 4 || A > MAX_A || (A & 3) || H < 1) return RECNET_ERR_BAD_SHAPE;
  return 0;
}

// sm = softmax attention (a.inv_T must then be 1)
template <typename TV, typename TO, bool SM = false>
static int launch_fwd(const FwdArgs& a, cudaStream_t st) {
  RN_TRY(check_shape(a.Tn, a.A, a.H));
  ProfScope prof(KC_PF_FWD, a.B, a.Tn, a.H, st);
  static const int minb = rn_env_int("RECNET_PF_MINB", 3);
  const dim3 grid(rn_cdiv(a.H, UPB), a.B);
  if (a.A <= 128 && minb == 3) RN_CUDA_OK(launch_pdl(pf_fwd_kernel<TV, TO, 1, 3, SM>, grid, dim3(THREADS), 0, st, a));
  else if (a.A <= 128) RN_CUDA_OK(launch_pdl(pf_fwd_kernel<TV, TO, 1, 2, SM>, grid, dim3(THREADS), 0, st, a));
  else RN_CUDA_OK(launch_pdl(pf_fwd_kernel<TV, TO, 2, 2, SM>, grid, dim3(THREADS), 0, st, a));
  RN_LAUNCH_OK();
  return 0;
}
template <typename TV, typename TO>
static int launch_fwd(const FwdArgs& a, bool softmax, cudaStream_t st) {
  return softmax ? launch_fwd<TV, TO, true>(a, st) : launch_fwd<TV, TO, false>(a, st);
}
static inline size_t bwd_smem_bytes(int H, int A) { return (size_t)H * sizeof(float4) + (size_t)2 * BNW * A * sizeof(float); }
// a.alpha != nullptr: softmax attention (a.inv_T must then be 1)
template <typename TV, typename TO, bool SM>
static int launch_bwd_sm(const BwdArgs& a, cudaStream_t st) {
  RN_TRY(check_shape(a.Tn, a.A, a.H));
  const size_t smem = bwd_smem_bytes(a.H, a.A);
  if (smem > 46 * 1024) return RECNET_ERR_BAD_SHAPE;
  const bool nf2 = a.Tn <= 2 * BNW, ch1 = a.A <= 128;
  ProfScope prof(KC_PF_BWD, a.B, a.Tn, a.H, st);
  if (nf2 && ch1) RN_CUDA_OK(launch_pdl(pf_bwd_kernel<TV, TO, 2, 1, SM>, dim3(a.B), dim3(BTHREADS), smem, st, a));
  else if (nf2) RN_CUDA_OK(launch_pdl(pf_bwd_kernel<TV, TO, 2, 2, SM>, dim3(a.B), dim3(BTHREADS), smem, st, a));
  else if (ch1) RN_CUDA_OK(launch_pdl(pf_bwd_kernel<TV, TO, 4, 1, SM>, dim3(a.B), dim3(BTHREADS), smem, st, a));
  else RN_CUDA_OK(launch_pdl(pf_bwd_kernel<TV, TO, 4, 2, SM>, dim3(a.B), dim3(BTHREADS), smem, st, a));
  RN_LAUNCH_OK();
  return 0;
}
template <typename TV, typename TO>
static int launch_bwd(const BwdArgs& a, cudaStream_t st) {
  return a.alpha ? launch_bwd_sm<TV, TO, true>(a, st) : launch_bwd_sm<TV, TO, false>(a, st);
}
}  // namespace pf
