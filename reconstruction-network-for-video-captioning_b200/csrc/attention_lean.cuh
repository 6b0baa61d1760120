// Lean additive-attention kernels (same contract and argument structs as attention.cuh; used by the reconstructor loops,
// models/local_reconstructor.py:38-50).  r1 ncu (profiles/r1_e_*): the general kernels execute ~1400-1900 instructions
// per warp with 2 warps per scheduler -- they are instruction-latency bound, not memory bound.  Here the work is laid
// out so that nothing has to be exchanged between the score and the weighted-sum phases:
//     warp  w  owns frames  w, w + 8, w + 16, ..      lane owns 16 bytes of columns (weighted sum) / one float4 of A (scores)
// A warp computes the score e[tau] of its own frames (warp_sum leaves it in every lane) and immediately uses it as the
// weight of its own V rows; the only block-level exchange is the final sum over the 8 frame groups.
// All loads are unconditional on clamped indices and issued before the first use (see proj_attn.cuh on why).
#pragma once
#include "common.cuh"

namespace attn {
constexpr int LEAN_THREADS = 256;
constexpr int LEAN_NW = LEAN_THREADS / 32;
constexpr int LEAN_MAX_A = 256;
constexpr int LEAN_MAXS = 12;

__device__ __forceinline__ float4 l4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

// sum of n float4 partials, stride apart; batches of 8 loads in flight
__device__ __forceinline__ float4 sum_partials4(const float* __restrict__ q, int n, long long stride) {
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int p = 0; p < n; p += 8) {
    float4 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = *reinterpret_cast<const float4*>(q + (long long)min(p + i, n - 1) * stride);
#pragma unroll
    for (int i = 0; i < 8; ++i) if (p + i < n) s = l4_add(s, v[i]);
  }
  return s;
}

static inline bool lean_enabled() {
  static const int v = rn_env_int("RECNET_LEAN_ATTN", 1);
  return v != 0;
}

// ---- forward: grid (ceil(D / (32 VN)), B) -----------------------------------------------------------------------------
// NF = frames per warp (Tn <= 8 NF), NCH = float4 chunks of A per lane (A <= 128 NCH)
template <typename TV, typename TO, int NF, int NCH>
__global__ void __launch_bounds__(LEAN_THREADS) lean_fwd_kernel(FwdArgs a) {
  constexpr bool FAST = FastMath<TV>::value;
  constexpr int VN = Vec16<TV>::N;
  pdl_wait();
  pdl_launch_next();
  __shared__ float red[LEAN_NW][32 * VN];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.y, Tn = a.Tn, A = a.A, D = a.D;
  const int col = (blockIdx.x * 32 + lane) * VN;
  const bool col_ok = col < D;
  const TV* vb = reinterpret_cast<const TV*>(a.V) + (long long)b * a.v_bs + (col_ok ? col : 0);
  Vec16<TV> v[NF];
#pragma unroll
  for (int f = 0; f < NF; ++f) v[f].load(vb + (long long)min(warp + f * LEAN_NW, Tn - 1) * a.v_ts);
  const int nchunk = A >> 2;
  const float* uvb = a.Uv + (long long)b * a.uv_bs;
  float4 uv[NF][NCH], wh[NCH], ww[NCH];
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int cc = min(lane + 32 * i, nchunk - 1);
#pragma unroll
    for (int f = 0; f < NF; ++f) uv[f][i] = reinterpret_cast<const float4*>(uvb + (long long)min(warp + f * LEAN_NW, Tn - 1) * a.uv_ts)[cc];
    ww[i] = reinterpret_cast<const float4*>(a.attn_w)[cc];
    const float4 bb = reinterpret_cast<const float4*>(a.attn_b)[cc];
    wh[i] = a.n_whp > 0 ? sum_partials4(a.WhP + (long long)b * A + 4 * cc, a.n_whp, a.whp_stride) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (blockIdx.x == 0 && warp == 0 && a.Wh_out && lane + 32 * i < nchunk) reinterpret_cast<float4*>(a.Wh_out + (long long)b * A)[cc] = wh[i];
    wh[i] = l4_add(wh[i], bb);
  }
  float acc[VN];
#pragma unroll
  for (int i = 0; i < VN; ++i) acc[i] = 0.f;
#pragma unroll
  for (int f = 0; f < NF; ++f) {
    const int tau = warp + f * LEAN_NW;
    if (tau < Tn) {                                    // warp-uniform
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        if (lane + 32 * i < nchunk) {
          const float4 x = uv[f][i];
          s = fmaf(ww[i].x, act_tanh<FAST>(wh[i].x + x.x), s);
          s = fmaf(ww[i].y, act_tanh<FAST>(wh[i].y + x.y), s);
          s = fmaf(ww[i].z, act_tanh<FAST>(wh[i].z + x.z), s);
          s = fmaf(ww[i].w, act_tanh<FAST>(wh[i].w + x.w), s);
        }
      }
      s = warp_sum(s);                                 // every lane now holds e[tau]
      if (blockIdx.x == 0 && lane == 0 && a.e_out) a.e_out[(long long)b * Tn + tau] = s;
      float fv[VN];
      v[f].get(fv);
#pragma unroll
      for (int i = 0; i < VN; ++i) acc[i] = fmaf(s, fv[i], acc[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < VN; ++i) red[warp][lane * VN + i] = acc[i];
  __syncthreads();
  // one column per thread: sum over the 8 frame groups, scale, dropout, store in the operand precision
  for (int c = tid; c < 32 * VN; c += LEAN_THREADS) {
    const int d = blockIdx.x * 32 * VN + c;
    if (d < D) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < LEAN_NW; ++w) s += red[w][c];
      s *= a.inv_T;
      if (a.p_drop > 0.f) s *= dropout_scale(a.rng, a.site, (uint64_t)(a.drop_base + (long long)b * D + d), a.p_drop);
      reinterpret_cast<TO*>(a.ctx_out)[(long long)b * a.ctx_ld + d] = from_f32<TO>(s);
    }
  }
}

// ---- backward: one CTA per sample; dynamic smem D floats ----------------------------------------------------------------
template <typename TV, typename TO, int NF, int NCH>
__global__ void __launch_bounds__(LEAN_THREADS) lean_bwd_kernel(BwdArgs a) {
  constexpr bool FAST = FastMath<TV>::value;
  constexpr int VN = Vec16<TV>::N;
  pdl_wait();
  pdl_launch_next();
  extern __shared__ float dx_s[];                       // [D]
  __shared__ float part[2][LEAN_NW][LEAN_MAX_A];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x, Tn = a.Tn, A = a.A, D = a.D;
  const int ncg = D / VN;                               // 16-byte column groups per V row
  const TV* vb = reinterpret_cast<const TV*>(a.V) + (long long)b * a.v_bs;
  // V rows of this warp's frames, first two column groups of the lane
  Vec16<TV> v[2][NF];
#pragma unroll
  for (int u = 0; u < 2; ++u)
#pragma unroll
    for (int f = 0; f < NF; ++f)
      v[u][f].load(vb + (long long)min(warp + f * LEAN_NW, Tn - 1) * a.v_ts + (long long)min(lane + 32 * u, ncg - 1) * VN);
  // score operands of this warp's frames
  const int nchunk = A >> 2;
  const float* uvb = a.Uv + (long long)b * a.uv_bs;
  float* dub = a.dUv_acc + (long long)b * a.uv_bs;
  float4 uv[NF][NCH], old[NF][NCH], wh[NCH], ww[NCH], dwh[NCH], dww[NCH];
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int cc = min(lane + 32 * i, nchunk - 1);
    dwh[i] = dww[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    wh[i] = l4_add(reinterpret_cast<const float4*>(a.Wh + (long long)b * A)[cc], reinterpret_cast<const float4*>(a.attn_b)[cc]);
    ww[i] = reinterpret_cast<const float4*>(a.attn_w)[cc];
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      const long long off = (long long)min(warp + f * LEAN_NW, Tn - 1) * a.uv_ts;
      uv[f][i] = reinterpret_cast<const float4*>(uvb + off)[cc];
      old[f][i] = a.uv_first ? make_float4(0.f, 0.f, 0.f, 0.f) : reinterpret_cast<const float4*>(dub + off)[cc];
    }
  }
  // ---- dctx = dropout-mask * sum of the split-K partials (two adjacent columns per thread and pass)
  for (int c0 = 2 * tid; c0 < D; c0 += 2 * LEAN_THREADS) {
    float2 pv[LEAN_MAXS];
    const float* q = a.dXp + (long long)b * a.p_ld + c0;
#pragma unroll
    for (int s = 0; s < LEAN_MAXS; ++s) pv[s] = *reinterpret_cast<const float2*>(q + (long long)min(s, a.n_p - 1) * a.p_stride);
    float sx = 0.f, sy = 0.f;
#pragma unroll
    for (int s = 0; s < LEAN_MAXS; ++s) if (s < a.n_p) { sx += pv[s].x; sy += pv[s].y; }
    for (int s = LEAN_MAXS; s < a.n_p; ++s) { const float2 t = *reinterpret_cast<const float2*>(q + (long long)s * a.p_stride); sx += t.x; sy += t.y; }
    if (a.p_drop > 0.f) {
      sx *= dropout_scale(a.rng, a.site, (uint64_t)(a.drop_base + (long long)b * D + c0), a.p_drop);
      sy *= dropout_scale(a.rng, a.site, (uint64_t)(a.drop_base + (long long)b * D + c0 + 1), a.p_drop);
    }
    dx_s[c0] = sx; dx_s[c0 + 1] = sy;
    if (a.dctx_out) *reinterpret_cast<float2*>(a.dctx_out + (long long)b * D + c0) = make_float2(sx, sy);
  }
  __syncthreads();
  // ---- d e[tau] = (1/T) <dctx, v_tau> for this warp's frames (whole rows: no cross-warp reduction)
  float de[NF];
#pragma unroll
  for (int f = 0; f < NF; ++f) de[f] = 0.f;
  for (int cg0 = 0; cg0 < ncg; cg0 += 64) {
    if (cg0 != 0) {
#pragma unroll
      for (int u = 0; u < 2; ++u)
#pragma unroll
        for (int f = 0; f < NF; ++f)
          v[u][f].load(vb + (long long)min(warp + f * LEAN_NW, Tn - 1) * a.v_ts + (long long)min(cg0 + lane + 32 * u, ncg - 1) * VN);
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int cg = cg0 + lane + 32 * u;
      if (cg < ncg) {
        float dxr[VN];
#pragma unroll
        for (int i = 0; i < VN; i += 4) {
          const float4 t = *reinterpret_cast<const float4*>(dx_s + cg * VN + i);
          dxr[i] = t.x; dxr[i + 1] = t.y; dxr[i + 2] = t.z; dxr[i + 3] = t.w;
        }
#pragma unroll
        for (int f = 0; f < NF; ++f) {
          float fv[VN];
          v[u][f].get(fv);
#pragma unroll
          for (int i = 0; i < VN; ++i) de[f] = fmaf(dxr[i], fv[i], de[f]);
        }
      }
    }
  }
#pragma unroll
  for (int f = 0; f < NF; ++f) de[f] = warp_sum(de[f]) * a.inv_T;
  // ---- score backward for the same frames
#pragma unroll
  for (int f = 0; f < NF; ++f) {
    const int tau = warp + f * LEAN_NW;
    if (tau < Tn) {
      const float g = de[f];
      if (lane == 0 && a.de_out) a.de_out[(long long)b * Tn + tau] = g;
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int c = lane + 32 * i;
        if (c < nchunk) {
          const float4 x = uv[f][i];
          const float tx = act_tanh<FAST>(wh[i].x + x.x), ty = act_tanh<FAST>(wh[i].y + x.y);
          const float tz = act_tanh<FAST>(wh[i].z + x.z), tw = act_tanh<FAST>(wh[i].w + x.w);
          const float4 ds = make_float4(g * ww[i].x * (1.f - tx * tx), g * ww[i].y * (1.f - ty * ty), g * ww[i].z * (1.f - tz * tz),
                                        g * ww[i].w * (1.f - tw * tw));
          dwh[i] = l4_add(dwh[i], ds);
          dww[i] = l4_add(dww[i], make_float4(g * tx, g * ty, g * tz, g * tw));
          reinterpret_cast<float4*>(dub + (long long)tau * a.uv_ts)[c] = l4_add(ds, old[f][i]);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < NCH; ++i) {
    const int c = lane + 32 * i;
    if (c < nchunk) {
      reinterpret_cast<float4*>(&part[0][warp][0])[c] = dwh[i];
      reinterpret_cast<float4*>(&part[1][warp][0])[c] = dww[i];
    }
  }
  __syncthreads();
  for (int x = tid; x < A; x += LEAN_THREADS) {
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int w = 0; w < LEAN_NW; ++w) { s0 += part[0][w][x]; s1 += part[1][w][x]; }
    if (a.dwh_acc) s0 += a.dWh_out[(long long)b * A + x];
    a.dWh_out[(long long)b * A + x] = s0;
    if (a.dWh_op) reinterpret_cast<TO*>(a.dWh_op)[(long long)b * A + x] = from_f32<TO>(s0);
    float* pw = a.dw_acc + (long long)b * A + x;
    *pw = a.dw_first ? s1 : *pw + s1;
  }
}

template <typename TV>
static inline bool lean_ok(int Tn, int A, int D, long long v_bs, long long v_ts, long long uv_bs, long long uv_ts) {
  constexpr int VN = Vec16<TV>::N;
  return lean_enabled() && Tn >= 1 && Tn <= 64 && A >= 4 && A <= LEAN_MAX_A && A % 4 == 0 && D % VN == 0 && D % 4 == 0 && v_bs % VN == 0 &&
         v_ts % VN == 0 && uv_bs % 4 == 0 && uv_ts % 4 == 0;
}

template <typename TV, typename TO>
static int launch_lean_fwd(const FwdArgs& a, cudaStream_t st) {
  constexpr int VN = Vec16<TV>::N;
  const dim3 grid(rn_cdiv(a.D, 32 * VN), a.B);
  const bool nf4 = a.Tn <= 4 * LEAN_NW, ch1 = a.A <= 128;
  ProfScope prof(KC_ATTN_FWD, a.B, a.Tn, a.D, st);
  if (nf4 && ch1) RN_CUDA_OK(launch_pdl(lean_fwd_kernel<TV, TO, 4, 1>, grid, dim3(LEAN_THREADS), 0, st, a));
  else if (nf4) RN_CUDA_OK(launch_pdl(lean_fwd_kernel<TV, TO, 4, 2>, grid, dim3(LEAN_THREADS), 0, st, a));
  else if (ch1) RN_CUDA_OK(launch_pdl(lean_fwd_kernel<TV, TO, 8, 1>, grid, dim3(LEAN_THREADS), 0, st, a));
  else RN_CUDA_OK(launch_pdl(lean_fwd_kernel<TV, TO, 8, 2>, grid, dim3(LEAN_THREADS), 0, st, a));
  RN_LAUNCH_OK();
  return 0;
}
template <typename TV, typename TO>
static int launch_lean_bwd(const BwdArgs& a, cudaStream_t st) {
  const size_t smem = (size_t)a.D * sizeof(float);
  if (smem > 24 * 1024) return RECNET_ERR_BAD_SHAPE;
  const bool nf4 = a.Tn <= 4 * LEAN_NW, ch1 = a.A <= 128;
  ProfScope prof(KC_ATTN_BWD, a.B, a.Tn, a.D, st);
  if (nf4 && ch1) RN_CUDA_OK(launch_pdl(lean_bwd_kernel<TV, TO, 4, 1>, dim3(a.B), dim3(LEAN_THREADS), smem, st, a));
  else if (nf4) RN_CUDA_OK(launch_pdl(lean_bwd_kernel<TV, TO, 4, 2>, dim3(a.B), dim3(LEAN_THREADS), smem, st, a));
  else if (ch1) RN_CUDA_OK(launch_pdl(lean_bwd_kernel<TV, TO, 8, 1>, dim3(a.B), dim3(LEAN_THREADS), smem, st, a));
  else RN_CUDA_OK(launch_pdl(lean_bwd_kernel<TV, TO, 8, 2>, dim3(a.B), dim3(LEAN_THREADS), smem, st, a));
  RN_LAUNCH_OK();
  return 0;
}
}  // namespace attn
