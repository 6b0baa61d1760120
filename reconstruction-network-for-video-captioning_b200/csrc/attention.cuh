// Fused additive temporal "attention" of RecNet (reference models/decoder.py:50-62 and
// models/local_reconstructor.py:38-50):
//     e[b,tau] = w . tanh(Wh[b] + Uv[b,tau] + bias)          (NO softmax in the reference)
//     ctx[b,:] = (1/Tn) * sum_tau e[b,tau] * V[b,tau,:]       (mean over frames)
// with Uv = V U^T hoisted out of the time loop and Wh = h W^T arriving as split-K partials of the
// tensor-core GEMM.  HBM/L2-bound: V is streamed once with 16-byte coalesced loads, scores live in
// shared memory, the weighted sum accumulates in registers.  normalize = 1 turns the scores into a max-subtracted
// softmax over frames and the mean into the weighted sum (the paper's attention, opt-in: attn_softmax); e_out then
// holds alpha, and the backward takes it (BwdArgs::alpha) instead of recomputing the softmax.
#pragma once
#include "common.cuh"

namespace attn {

constexpr int FWD_THREADS = 256;
constexpr int BWD_THREADS = 256;
constexpr int MAX_T = 64;       // frames (28 / 40) or decoder steps (<= 31)

// All three kernels are latency-bound (a few MB that live in L2, ~100 CTAs): every phase issues its loads in
// batches before the first use so that a thread has 8-28 independent requests in flight (r1 profile: the first
// version with serial per-frame loops took 13-20 us per launch).

struct FwdArgs {
  const float* WhP; int n_whp; long long whp_stride;   // Wh partials [n_whp][B,A]
  const float* Uv; long long uv_bs, uv_ts;             // Uv[b*uv_bs + tau*uv_ts + a]
  const float* attn_b; const float* attn_w;            // [A]
  const void* V; long long v_bs, v_ts;                 // V[b*v_bs + tau*v_ts + d]   (TV)
  int B, Tn, A, D; float inv_T; int normalize; int d_slice;   // d_slice: columns of D per blockIdx.x (set by launch_fwd)
  float* Wh_out;                                       // [B,A]   saved for backward (nullable)
  float* e_out;                                        // [B,Tn]  saved for backward (nullable)
  void* ctx_out; long long ctx_ld;                     // ctx[b*ctx_ld + d]   (TO) GEMM operand slot
  float p_drop; const unsigned long long* rng; unsigned int site; long long drop_base;  // dropout on ctx (train)
};

// body: one virtual block (bx = D-slice index, b = sample); 256 threads; sm = fwd_smem_floats() floats.
// Latency structure (each dependent L2 round trip costs ~0.6 us here, r1 timeline): every global load of the block --
// the V rows for the weighted sum, the Uv rows for the scores, the Wh partials -- is issued at entry, before anything
// is consumed; the frames of a column group are split over FP threads whose partial sums meet in shared memory.
template <typename TV, typename TO>
__device__ __forceinline__ void attn_fwd_body(const FwdArgs& a, int bx, int b, float* sm, int tid, int bar_id) {
  constexpr bool FAST = FastMath<TV>::value;
  constexpr int VN = Vec16<TV>::N, NW = FWD_THREADS / 32, NPRE = 16;
  float* Wh = sm;              // [A] (bias folded in)
  float* wv = sm + a.A;        // [A] attn_w
  float* e = sm + 2 * a.A;     // [Tn]
  float* red = e + a.Tn;       // [FWD_THREADS * VN] partial context sums (only when FP > 1)
  const int lane = tid & 31, warp = tid >> 5;
  const int d_lo = bx * a.d_slice, d_hi = min(a.D, d_lo + a.d_slice);
  const int G = (d_hi - d_lo) / VN;                    // 16-byte column groups of this slice (<= 256)
  int FP = 1;
  while (FP < 8 && G * FP * 2 <= FWD_THREADS) FP *= 2;  // frame partitions per column group
  const bool active = tid < G * FP;
  const int cg = active ? tid % G : 0, fp = active ? tid / G : 0;
  const int d = d_lo + cg * VN;
  const TV* Vb = reinterpret_cast<const TV*>(a.V) + (long long)b * a.v_bs + d;

  RN_PROBE(20, tid);
  // ---- issue every load up front ----
  Vec16<TV> v[NPRE];
  if (active) {
#pragma unroll
    for (int k = 0; k < NPRE; ++k) {
      const int f = fp + k * FP;
      if (f < a.Tn) v[k].load(Vb + (long long)f * a.v_ts);
    }
  }
  float u[4][4];
  const float* Ub = a.Uv + (long long)b * a.uv_bs;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int tau = warp + k * NW;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int i = lane + 32 * q;
      u[k][q] = (tau < a.Tn && i < a.A) ? __ldg(Ub + (long long)tau * a.uv_ts + i) : 0.f;
    }
  }
  for (int i = tid; i < a.A; i += FWD_THREADS) {
    float s = 0.f;
    for (int p0 = 0; p0 < a.n_whp; p0 += 8) {
      float t8[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) t8[k] = (p0 + k < a.n_whp) ? __ldg(a.WhP + (long long)(p0 + k) * a.whp_stride + (long long)b * a.A + i) : 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) s += t8[k];
    }
    Wh[i] = s + a.attn_b[i];
    wv[i] = a.attn_w[i];
    if (a.Wh_out && bx == 0) a.Wh_out[(long long)b * a.A + i] = s;
  }
  RN_PROBE(21, tid);
  blk_sync(bar_id);
  RN_PROBE(22, tid);
  // ---- scores: warp w owns frames w, w+8, w+16, w+24 (preloaded); anything beyond 32 frames / 128 units on demand ----
  {
    float sc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int i = lane + 32 * q;
      if (i < a.A) {
        const float whi = Wh[i], wi = wv[i];
#pragma unroll
        for (int k = 0; k < 4; ++k) sc[k] += wi * act_tanh<FAST>(whi + u[k][q]);
      }
    }
    for (int i = lane + 128; i < a.A; i += 32) {          // A > 128 (not the reference sizes)
      const float whi = Wh[i], wi = wv[i];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int tau = warp + k * NW;
        if (tau < a.Tn) sc[k] += wi * act_tanh<FAST>(whi + __ldg(Ub + (long long)tau * a.uv_ts + i));
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float r = warp_sum(sc[k]);
      if (lane == 0 && warp + k * NW < a.Tn) e[warp + k * NW] = r;
    }
    for (int tau = warp + 4 * NW; tau < a.Tn; tau += NW) {  // Tn > 32
      float s1 = 0.f;
      for (int i = lane; i < a.A; i += 32) s1 += wv[i] * act_tanh<FAST>(Wh[i] + __ldg(Ub + (long long)tau * a.uv_ts + i));
      s1 = warp_sum(s1);
      if (lane == 0) e[tau] = s1;
    }
  }
  blk_sync(bar_id);
  if (a.normalize) {   // softmax over frames (paper variant): alpha replaces e
    if (warp == 0) {
      float m = -INFINITY;
      for (int t = lane; t < a.Tn; t += 32) m = fmaxf(m, e[t]);
      m = warp_max(m);
      float z = 0.f;
      for (int t = lane; t < a.Tn; t += 32) z += act_exp<FAST>(e[t] - m);
      z = warp_sum(z);
      for (int t = lane; t < a.Tn; t += 32) e[t] = act_exp<FAST>(e[t] - m) / z;
    }
    blk_sync(bar_id);
  }
  if (a.e_out && bx == 0)
    for (int t = tid; t < a.Tn; t += FWD_THREADS) a.e_out[(long long)b * a.Tn + t] = e[t];

  RN_PROBE(23, tid);
  // ---- weighted sum over this thread's frames ----
  float acc[VN];
#pragma unroll
  for (int j = 0; j < VN; ++j) acc[j] = 0.f;
  if (active) {
#pragma unroll
    for (int k = 0; k < NPRE; ++k) {
      const int f = fp + k * FP;
      if (f < a.Tn) {
        float fv[VN]; v[k].get(fv);
        const float ek = e[f];
#pragma unroll
        for (int j = 0; j < VN; ++j) acc[j] += ek * fv[j];
      }
    }
    for (int f = fp + NPRE * FP; f < a.Tn; f += FP) {       // more than NPRE frames per thread: second round
      Vec16<TV> vv; vv.load(Vb + (long long)f * a.v_ts);
      float fv[VN]; vv.get(fv);
      const float ek = e[f];
#pragma unroll
      for (int j = 0; j < VN; ++j) acc[j] += ek * fv[j];
    }
  }
  if (FP > 1) {
    if (active && fp > 0) {
#pragma unroll
      for (int j = 0; j < VN; ++j) red[(fp * G + cg) * VN + j] = acc[j];
    }
    blk_sync(bar_id);
    if (active && fp == 0) {
      for (int q = 1; q < FP; ++q)
#pragma unroll
        for (int j = 0; j < VN; ++j) acc[j] += red[(q * G + cg) * VN + j];
    }
  }
  if (active && fp == 0) {
    TO* out = reinterpret_cast<TO*>(a.ctx_out) + (long long)b * a.ctx_ld + d;
    const float scl = a.normalize ? 1.f : a.inv_T;
#pragma unroll
    for (int j = 0; j < VN; ++j) {
      float r = acc[j] * scl;
      if (a.p_drop > 0.f) r *= dropout_scale(a.rng, a.site, (uint64_t)(a.drop_base + (long long)b * a.D + d + j), a.p_drop);
      out[j] = from_f32<TO>(r);
    }
  }
  RN_PROBE(24, tid);
}

template <typename TV, typename TO>
__global__ void __launch_bounds__(FWD_THREADS) attn_fwd_kernel(FwdArgs a) {
  extern __shared__ float sm[];
  pdl_wait();            // prerequisites complete ...
  pdl_launch_next();     // ... only then let the NEXT kernel be scheduled (depth-1 look-ahead, no cascade of resident waiters)
  attn_fwd_body<TV, TO>(a, blockIdx.x, blockIdx.y, sm, threadIdx.x, 0);
}

// Backward.  One CTA per sample:
//   dctx = sum of split-K partials of d[ctx;h] (first D columns)      (x dropout mask in train)
//   de[tau] = inv_T * dctx . V[b,tau,:]
//     softmax (alpha != null, inv_T = 1): d alpha[tau] = dctx . V[b,tau,:];  de[tau] = alpha[tau] (d alpha[tau] - sum_s alpha[s] d alpha[s])
//   ds[tau,a] = de[tau] * w[a] * (1 - s^2),  s = tanh(Wh + Uv + b)   (recomputed, not stored)
//   dWh[b,a] = sum_tau ds ; dUv[b,tau,a] += ds ; dw_acc[b,a] += sum_tau de[tau]*s
struct BwdArgs {
  const float* dXp; int n_p; long long p_stride; long long p_ld;      // partials [n_p][B, p_ld], cols [0,D)
  const void* V; long long v_bs, v_ts;
  const float* Wh; const float* Uv; long long uv_bs, uv_ts;
  const float* attn_b; const float* attn_w;
  int B, Tn, A, D; float inv_T;
  float* dWh_out;                      // [B,A] fp32
  void* dWh_op;                        // [B,A] operand type (nullable): A-operand of the dWh @ attn_W GEMM
  float* dUv_acc; int uv_first;        // same strides as Uv; first => overwrite instead of +=
  float* dw_acc; int dw_first;         // [B,A] += ; dw_first => overwrite
  int dwh_acc;                         // dWh_out += (several attentions share one query: stacked-decoder pseudo-steps)
  float* dctx_out;                     // [B,D] fp32 (nullable): summed/masked dctx, for the deferred dV pass
  float* de_out;                       // [B,Tn] (nullable)
  const float* alpha;                  // [B,Tn] softmax weights of the forward (nullable = the reference's mean, no softmax)
  float p_drop; const unsigned long long* rng; unsigned int site; long long drop_base;
};

// body: one virtual block = sample b; sm = (D + Tn + 2*256) floats; 256 threads.
// Same latency discipline as the forward: the Uv / dUv rows of the score backward and the first V rows of the de dot
// products are requested at entry; the split-K partial sum of dctx runs as 16-byte loads, all partials in flight.
template <typename TV, typename TO>
__device__ __forceinline__ void attn_bwd_body(const BwdArgs& a, int b, float* sm, int tid, int bar_id) {
  constexpr bool FAST = FastMath<TV>::value;
  constexpr int VN = Vec16<TV>::N, NW = BWD_THREADS / 32, MAXP = 12, NF = 14;
  float* dctx = sm;                 // [D]
  float* de = sm + a.D;             // [Tn]
  float* red = de + a.Tn;           // [2 * BWD_THREADS]
  const int lane = tid & 31, warp = tid >> 5;
  const TV* Vb = reinterpret_cast<const TV*>(a.V) + (long long)b * a.v_bs;

  // ---- prefetch for the score backward: thread (i, part) owns attention unit i and frames part, part+nparts, ... ----
  const int per = (a.A <= BWD_THREADS && BWD_THREADS % a.A == 0) ? a.A : BWD_THREADS;   // threads per frame partition
  const int nparts = BWD_THREADS / per;
  const int i3 = tid % per, part = tid / per;
  const bool pre3 = (per == a.A);                         // the common case (A divides 256): everything preloaded
  float u3[NF], o3[NF];
  const float* Ub = a.Uv + (long long)b * a.uv_bs + i3;
  float* dUb = a.dUv_acc + (long long)b * a.uv_bs + i3;
  if (pre3) {
#pragma unroll
    for (int k = 0; k < NF; ++k) {
      const int tau = part + k * nparts;
      u3[k] = (tau < a.Tn) ? __ldg(Ub + (long long)tau * a.uv_ts) : 0.f;
      o3[k] = (tau < a.Tn && !a.uv_first) ? dUb[(long long)tau * a.uv_ts] : 0.f;
    }
  }
  // ---- prefetch the V rows of this warp's first two frames (the dot products need dctx, which is not ready yet) ----
  constexpr int NV = 8;                                    // 16-byte vectors per lane per frame held in registers
  Vec16<TV> v0[NV], v1[NV];
  const int tau0 = warp, tau1 = warp + NW;
#pragma unroll
  for (int q = 0; q < NV; ++q) {
    const int d = (lane + 32 * q) * VN;
    if (d < a.D) {
      if (tau0 < a.Tn) v0[q].load(Vb + (long long)tau0 * a.v_ts + d);
      if (tau1 < a.Tn) v1[q].load(Vb + (long long)tau1 * a.v_ts + d);
    }
  }
  // ---- dctx = sum of split-K partials (x dropout mask), float4 at a time, all partials of a float4 in flight ----
  const float* Pb = a.dXp + (long long)b * a.p_ld;
  for (int d4 = tid * 4; d4 < a.D; d4 += BWD_THREADS * 4) {
    float4 t[MAXP];
#pragma unroll
    for (int p = 0; p < MAXP; ++p)
      t[p] = (p < a.n_p) ? *reinterpret_cast<const float4*>(Pb + (long long)p * a.p_stride + d4) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int p = 0; p < MAXP; ++p) { s4.x += t[p].x; s4.y += t[p].y; s4.z += t[p].z; s4.w += t[p].w; }
    for (int p = MAXP; p < a.n_p; ++p) {
      const float4 x = *reinterpret_cast<const float4*>(Pb + (long long)p * a.p_stride + d4);
      s4.x += x.x; s4.y += x.y; s4.z += x.z; s4.w += x.w;
    }
    float r[4] = {s4.x, s4.y, s4.z, s4.w};
    if (a.p_drop > 0.f) {
#pragma unroll
      for (int j = 0; j < 4; ++j) r[j] *= dropout_scale(a.rng, a.site, (uint64_t)(a.drop_base + (long long)b * a.D + d4 + j), a.p_drop);
    }
    *reinterpret_cast<float4*>(dctx + d4) = make_float4(r[0], r[1], r[2], r[3]);
    if (a.dctx_out) *reinterpret_cast<float4*>(a.dctx_out + (long long)b * a.D + d4) = make_float4(r[0], r[1], r[2], r[3]);
  }
  blk_sync(bar_id);
  // ---- de[tau] = inv_T * dctx . V[b,tau,:] ----
  auto dot_pre = [&](const Vec16<TV>* vv) {
    float s1 = 0.f;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
      const int d = (lane + 32 * q) * VN;
      if (d < a.D) {
        float f[VN]; vv[q].get(f);
#pragma unroll
        for (int j = 0; j < VN; ++j) s1 += f[j] * dctx[d + j];
      }
    }
    return s1;
  };
  auto dot_tail = [&](int tau) {          // columns beyond the NV preloaded vectors per lane (D > 32*NV*VN)
    float s1 = 0.f;
    for (int d = (lane + 32 * NV) * VN; d < a.D; d += 32 * VN) {
      Vec16<TV> x; x.load(Vb + (long long)tau * a.v_ts + d);
      float f[VN]; x.get(f);
#pragma unroll
      for (int j = 0; j < VN; ++j) s1 += f[j] * dctx[d + j];
    }
    return s1;
  };
  if (tau0 < a.Tn) {
    const float r = warp_sum(dot_pre(v0) + dot_tail(tau0)) * a.inv_T;
    if (lane == 0) { de[tau0] = r; if (a.de_out) a.de_out[(long long)b * a.Tn + tau0] = r; }
  }
  if (tau1 < a.Tn) {
    const float r = warp_sum(dot_pre(v1) + dot_tail(tau1)) * a.inv_T;
    if (lane == 0) { de[tau1] = r; if (a.de_out) a.de_out[(long long)b * a.Tn + tau1] = r; }
  }
  for (int t0 = warp + 2 * NW; t0 < a.Tn; t0 += 2 * NW) {     // remaining frames: two rows in flight per round
    const int t1 = t0 + NW;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
      const int d = (lane + 32 * q) * VN;
      if (d < a.D) {
        v0[q].load(Vb + (long long)t0 * a.v_ts + d);
        if (t1 < a.Tn) v1[q].load(Vb + (long long)t1 * a.v_ts + d);
      }
    }
    const float r0 = warp_sum(dot_pre(v0) + dot_tail(t0)) * a.inv_T;
    if (lane == 0) { de[t0] = r0; if (a.de_out) a.de_out[(long long)b * a.Tn + t0] = r0; }
    if (t1 < a.Tn) {
      const float r1 = warp_sum(dot_pre(v1) + dot_tail(t1)) * a.inv_T;
      if (lane == 0) { de[t1] = r1; if (a.de_out) a.de_out[(long long)b * a.Tn + t1] = r1; }
    }
  }
  blk_sync(bar_id);
  if (a.alpha) {       // softmax backward: de holds d alpha; de_out (if any) keeps d alpha
    if (warp == 0) {
      const float* al = a.alpha + (long long)b * a.Tn;
      float s1 = 0.f;
      for (int t = lane; t < a.Tn; t += 32) s1 += al[t] * de[t];
      s1 = warp_sum(s1);
      for (int t = lane; t < a.Tn; t += 32) de[t] = al[t] * (de[t] - s1);
    }
    blk_sync(bar_id);
  }
  // ---- ds / dWh / dUv / dw ----
  for (int i0 = 0; i0 < a.A; i0 += per) {
    const int i = i0 + i3;
    float dwh = 0.f, dw = 0.f;
    if (i < a.A) {
      const float wh = a.Wh[(long long)b * a.A + i] + a.attn_b[i];
      const float w = a.attn_w[i];
      if (pre3) {
#pragma unroll
        for (int k = 0; k < NF; ++k) {
          const int tau = part + k * nparts;
          if (tau < a.Tn) {
            const float sv = act_tanh<FAST>(wh + u3[k]);
            const float g = de[tau] * w * (1.f - sv * sv);
            dwh += g;
            dw += de[tau] * sv;
            dUb[(long long)tau * a.uv_ts] = o3[k] + g;
          }
        }
      }
      for (int tau = pre3 ? part + NF * nparts : part; tau < a.Tn; tau += nparts) {   // not preloaded (odd A or Tn > 14*nparts)
        const long long off = (long long)b * a.uv_bs + (long long)tau * a.uv_ts + i;
        const float sv = act_tanh<FAST>(wh + a.Uv[off]);
        const float g = de[tau] * w * (1.f - sv * sv);
        dwh += g;
        dw += de[tau] * sv;
        a.dUv_acc[off] = a.uv_first ? g : a.dUv_acc[off] + g;
      }
    }
    if (nparts > 1) {     // combine the frame partitions
      red[tid] = dwh; red[BWD_THREADS + tid] = dw;
      blk_sync(bar_id);
      if (part == 0 && i < a.A) {
        for (int q = 1; q < nparts; ++q) { dwh += red[q * per + tid]; dw += red[BWD_THREADS + q * per + tid]; }
      }
      blk_sync(bar_id);
    }
    if (part == 0 && i < a.A) {
      if (a.dwh_acc) dwh += a.dWh_out[(long long)b * a.A + i];
      a.dWh_out[(long long)b * a.A + i] = dwh;
      if (a.dWh_op) reinterpret_cast<TO*>(a.dWh_op)[(long long)b * a.A + i] = from_f32<TO>(dwh);
      float* pw = a.dw_acc + (long long)b * a.A + i;
      *pw = a.dw_first ? dw : *pw + dw;
    }
  }
}

template <typename TV, typename TO>
__global__ void __launch_bounds__(BWD_THREADS) attn_bwd_kernel(BwdArgs a) {
  extern __shared__ float sm[];
  pdl_wait();            // prerequisites complete ...
  pdl_launch_next();     // ... only then let the NEXT kernel be scheduled (depth-1 look-ahead, no cascade of resident waiters)
  attn_bwd_body<TV, TO>(a, blockIdx.x, sm, threadIdx.x, 0);
}

// Deferred value-gradient of the local reconstructor's attention (values = decoder hiddens, which need grad):
//   dV[l,b,:] (+)= inv_T * sum_t beta_t[b,l] * dx_t[b,:]        one pass after the time loop instead of Tsteps RMWs
// (softmax attention: beta = alpha, inv_T = 1)
// beta [S,B,Tn] fp32, dx [S,B,D] fp32, dV[b*dv_bs + l*dv_ts + d] fp32.
// step_mul / step_off: stash row of outer step t is t * step_mul + step_off (pseudo-steps of a stacked decoder)
__global__ void attn_dv_kernel(const float* __restrict__ beta, const float* __restrict__ dx, float* __restrict__ dV,
                               long long dv_bs, long long dv_ts, int S, int B, int Tn, int D, float inv_T, int accumulate,
                               int step_mul, int step_off) {
  const int b = blockIdx.y, l = blockIdx.x;
  extern __shared__ float bt[];   // [S]
  for (int t = threadIdx.x; t < S; t += blockDim.x) bt[t] = beta[((long long)(t * step_mul + step_off) * B + b) * Tn + l];
  __syncthreads();
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    float s = 0.f;
    for (int t = 0; t < S; ++t) s += bt[t] * dx[((long long)(t * step_mul + step_off) * B + b) * D + d];
    float* p = dV + (long long)b * dv_bs + (long long)l * dv_ts + d;
    s *= inv_T;
    *p = accumulate ? *p + s : s;
  }
}

// Same result, one pass over dx: a block owns (sample b, 256 columns) and accumulates ALL Tn frames in registers; the S step
// values of a column are fetched with independent loads up front (the kernel above re-reads dx once per frame: 31 x 5.7 MB of
// L2 traffic, 37 us).  grid (ceil(D / 256), B), 256 threads, dynamic smem round_up(S, 32) * round_up(Tn, 4) floats.  Tn <= 64.
__global__ void __launch_bounds__(256) attn_dv2_kernel(const float* __restrict__ beta, const float* __restrict__ dx, float* __restrict__ dV,
                                                       long long dv_bs, long long dv_ts, int S, int B, int Tn, int D, float inv_T,
                                                       int accumulate, int step_mul, int step_off) {
  extern __shared__ float4 bt4[];
  float* bt = reinterpret_cast<float*>(bt4);
  const int Tnp = (Tn + 3) & ~3, Sp = (S + 31) & ~31;
  const int b = blockIdx.y, d = blockIdx.x * 256 + threadIdx.x;
  for (int i = threadIdx.x; i < Sp * Tnp; i += 256) {        // zero rows beyond S / columns beyond Tn
    const int t = i / Tnp, l = i - t * Tnp;
    bt[i] = (t < S && l < Tn) ? beta[((long long)(t * step_mul + step_off) * B + b) * Tn + l] : 0.f;
  }
  __syncthreads();
  if (d >= D) return;
  for (int l0 = 0; l0 < Tn; l0 += 32) {
    float acc[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) acc[k] = 0.f;
    for (int t0 = 0; t0 < S; t0 += 32) {
      float g[32];
#pragma unroll
      for (int k = 0; k < 32; ++k) g[k] = dx[((long long)(min(t0 + k, S - 1) * step_mul + step_off) * B + b) * D + d];
#pragma unroll
      for (int tt = 0; tt < 32; ++tt) {                        // rows >= S carry zero weights
        const float4* br = bt4 + ((t0 + tt) * Tnp + l0) / 4;
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) {
          if (l0 + 4 * k4 < Tn) {
            const float4 e4 = br[k4];
            acc[4 * k4 + 0] = fmaf(e4.x, g[tt], acc[4 * k4 + 0]);
            acc[4 * k4 + 1] = fmaf(e4.y, g[tt], acc[4 * k4 + 1]);
            acc[4 * k4 + 2] = fmaf(e4.z, g[tt], acc[4 * k4 + 2]);
            acc[4 * k4 + 3] = fmaf(e4.w, g[tt], acc[4 * k4 + 3]);
          }
        }
      }
    }
    float old[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) old[k] = accumulate ? dV[(long long)b * dv_bs + (long long)min(l0 + k, Tn - 1) * dv_ts + d] : 0.f;
#pragma unroll
    for (int k = 0; k < 32; ++k)
      if (l0 + k < Tn) dV[(long long)b * dv_bs + (long long)(l0 + k) * dv_ts + d] = fmaf(acc[k], inv_T, old[k]);
  }
}
// picks the one-pass kernel when its alignment requirements hold
static inline int launch_dv(const float* beta, const float* dx, float* dV, long long dv_bs, long long dv_ts, int S, int B, int Tn, int D,
                            float inv_T, int accumulate, int step_mul, int step_off, cudaStream_t st) {
  const size_t smem2 = (size_t)((S + 31) & ~31) * ((Tn + 3) & ~3) * sizeof(float);
  if (Tn <= 64 && smem2 <= 40 * 1024) {
    attn_dv2_kernel<<<dim3(rn_cdiv(D, 256), B), 256, smem2, st>>>(beta, dx, dV, dv_bs, dv_ts, S, B, Tn, D, inv_T, accumulate, step_mul, step_off);
  } else {
    attn_dv_kernel<<<dim3(Tn, B), 128, (size_t)S * sizeof(float), st>>>(beta, dx, dV, dv_bs, dv_ts, S, B, Tn, D, inv_T, accumulate, step_mul, step_off);
  }
  RN_LAUNCH_OK();
  return 0;
}

// validates, fills a.d_slice and returns the number of D-slices (grid.x) through *slices_out
template <typename TV>
static int prepare_fwd(FwdArgs& a, int* slices_out) {
  if (a.Tn > MAX_T || a.Tn < 1) return RECNET_ERR_BAD_SHAPE;
  constexpr int VN = Vec16<TV>::N;
  if (a.D % VN || a.v_ts % VN || a.v_bs % VN) return RECNET_ERR_ALIGNMENT;
  // enough CTAs to cover the SMs (~150), each thread owning at most one 16-byte column group when possible
  int slices = rn_cdiv(150, a.B);
  const int min_slices = rn_cdiv(a.D, FWD_THREADS * VN);
  if (slices < min_slices) slices = min_slices;
  if (slices > a.D / VN) slices = a.D / VN;
  int slice = rn_cdiv(rn_cdiv(a.D, slices), VN) * VN;
  slices = rn_cdiv(a.D, slice);
  a.d_slice = slice;
  *slices_out = slices;
  return 0;
}
static inline size_t fwd_smem_bytes(const FwdArgs& a) { return (size_t)(2 * a.A + a.Tn + FWD_THREADS * 8) * sizeof(float); }
static inline size_t bwd_smem_bytes(const BwdArgs& a) { return (size_t)(a.D + a.Tn + 2 * BWD_THREADS) * sizeof(float); }

}  // namespace attn
#include "attention_lean.cuh"
namespace attn {

template <typename TV, typename TO>
static int launch_fwd(FwdArgs a, cudaStream_t st) {
  if (!a.normalize && lean_ok<TV>(a.Tn, a.A, a.D, a.v_bs, a.v_ts, a.uv_bs, a.uv_ts)) return launch_lean_fwd<TV, TO>(a, st);
  int slices = 1;
  RN_TRY(prepare_fwd<TV>(a, &slices));
  dim3 grid(slices, a.B);
  const size_t smem = fwd_smem_bytes(a);
  ProfScope prof(KC_ATTN_FWD, a.B, a.Tn, a.D, st);
  RN_CUDA_OK(launch_pdl(attn_fwd_kernel<TV, TO>, grid, dim3(FWD_THREADS), smem, st, a));
  RN_LAUNCH_OK();
  return 0;
}

template <typename TV, typename TO>
static int launch_bwd(const BwdArgs& a, cudaStream_t st) {
  if (!a.alpha && lean_ok<TV>(a.Tn, a.A, a.D, a.v_bs, a.v_ts, a.uv_bs, a.uv_ts) && a.p_ld % 2 == 0 && a.p_stride % 2 == 0 && a.D <= 6144)
    return launch_lean_bwd<TV, TO>(a, st);
  if (a.Tn > MAX_T || a.Tn < 1) return RECNET_ERR_BAD_SHAPE;
  constexpr int VN = Vec16<TV>::N;
  if (a.D % VN || a.v_ts % VN || a.v_bs % VN) return RECNET_ERR_ALIGNMENT;
  const size_t smem = (size_t)(a.D + a.Tn + 2 * BWD_THREADS) * sizeof(float);
  ProfScope prof(KC_ATTN_BWD, a.B, a.Tn, a.D, st);
  RN_CUDA_OK(launch_pdl(attn_bwd_kernel<TV, TO>, dim3(a.B), dim3(BWD_THREADS), smem, st, a));
  RN_LAUNCH_OK();
  return 0;
}
}  // namespace attn
