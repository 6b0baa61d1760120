// Decoder time loops (projected-feature form, seq_decoder_pf.cuh / proj_attn.cuh) as ONE persistent kernel each, forward and BPTT,
// made of independent 16-CTA thread-block clusters -- no grid-wide synchronisation at all.
//   reference: models/decoder.py:45-70 called L times from train.py:41-66, and its autograd
//
// Samples are independent through the loop, and the per-step weight [W_a ; W_hh] is only 2176 x 512 bf16 = 2.2 MB, so it fits the
// distributed shared memory of ONE cluster: cluster q owns samples [13 q, 13 q + 13) for all L steps, CTA r of the cluster keeps the
// 136 weight rows of "its" 32 hidden units (4 gates) + 8 attention rows resident (139 KB).  What made the kernel-per-phase loop
// expensive disappears:
//   * the projected features VW[b, tau, unit, 4 gates] do not depend on the step: thread (sample w, unit lane) loads its 28 quads
//     ONCE and keeps them in 56 registers for the whole sequence (the per-step kernels re-read 11.5 MB of VW from L2 every step);
//   * U.v of the two frames a CTA scores stays in shared memory;
//   * the three exchanges of a step (W.h all-gather, scores all-gather, h_t all-gather; in BPTT three reduce-scatters) are DSMEM
//     stores + barrier.cluster (hardware, ~0.2 us) instead of kernel boundaries or L2 flags.
// The per-step GEMM is [16 samples x 512] . [512 x 136] per CTA on mma.sync m16n8k16 (ldmatrix-fed; 17 n-tiles): at 13 samples per
// cluster the tensor work is ~0.3 us per step and not the bottleneck, the exchanges are.  tcgen05 needs M >= 64 rows of one operand
// per CTA, which a 13-sample x 136-row slice cannot fill either way round, hence the warp-level MMA here (the batched GEMMs around
// the loop and the reconstructor loops use tcgen05).
//
// SM = true: the paper's softmax attention (opt-in): after barrier #2 every sample warp holds its whole score row (Tn <= 32) and turns it
// into alpha with one warp max / sum-exp; the context sum takes alpha with scale 1 (the host passes inv_T = 1) and the e stash holds alpha.
// Stash layout = what pf_fwd_kernel / pf_bwd_kernel leave (Hop, c, hiddens, Wh, e, gates; dGW, dWh, dUv, dw_acc), so either loop
// implementation can run in front of / behind the other and the batched GEMMs after the loop are unchanged.
#pragma once
#include <stdio.h>

#include "proj_attn.cuh"

namespace dcl {
constexpr int CS = 16;             // CTAs per cluster (non-portable size: one cluster per GPC)
constexpr int THREADS = 512;       // 16 warps: warp w <-> sample w of the cluster in the per-sample phases
constexpr int NWARP = THREADS / 32;
constexpr int MAX_MS = 16;         // samples per cluster <= warps per CTA (chosen at launch: ceil(B / co-resident clusters))
constexpr int MT = 16;             // MMA M tile (samples padded)
constexpr int H_ = 512, A_ = 128, UPC = 32, APC = 8, NR = APC + 4 * UPC;      // the shape this kernel is written for
constexpr int NRP = 144;           // weight rows padded to a multiple of 16 (K of the BPTT GEMM)
constexpr int PITCH = H_ + 8;      // bf16 elements per smem row: 1040 B -> conflict-free ldmatrix
constexpr int MAXF = 2;            // frames scored per CTA (Tn <= 32)
constexpr int MAXT = 32;

// ---- cluster / DSMEM primitives --------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cta_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t cluster_id() { uint32_t r; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_barrier() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t mapa(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_c_f32(uint32_t a, float v) { asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void st_c_f32x2(uint32_t a, float x, float y) { asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(x), "f"(y) : "memory"); }
__device__ __forceinline__ void st_c_f32x4(uint32_t a, float4 v) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_c_u32x4(uint32_t a, uint4 v) {
  asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// developer timeline (recnet_debug_set_timeline): thread 0 of block 0
__device__ __forceinline__ void stamp(int tag) {
  if (g_timeline != nullptr && blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    const unsigned int i = atomicAdd(&g_timeline_n, 1u);
    if (i < 4000) g_timeline[i] = (t & 0x00FFFFFFFFFFFFFFull) | ((unsigned long long)tag << 56);
  }
}
// ---- warp-level MMA --------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2(uint32_t (&r)[2], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2_t(uint32_t (&r)[2], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}
__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// global row of Wcat ([A + 4H, H]: rows [0, A) = W_a, row A + g H + j = W_hh gate g of unit j) held at local row lr of CTA r:
// local rows [0, 8) = attention rows 8 r .., local row 8 + 32 g + u = gate g of unit 32 r + u
__device__ __forceinline__ int wcat_row(int lr, int r) {
  return lr < APC ? r * APC + lr : A_ + ((lr - APC) / UPC) * H_ + r * UPC + (lr - APC) % UPC;
}

struct FwdArgs {
  const bf16* Wcat;               // [A + 4H, H]
  const float* Uv;                // [B, Tn, A]   U v + attn_b
  const float* attn_w;            // [A]
  const bf16* VW;                 // [B, Tn, H, 4] unit-interleaved projected features
  const float* Gx;                // [L B, 4H]    embedding projection + b_ih (gate-block order)
  const float* b_hh;              // [4H]
  float* c;                       // [(L+1) B, H] fp32 cell states, row block 0 = zeros
  float* hiddens;                 // [L B, H] fp32
  bf16* Hop;                      // [(L+1) B, H] operand rows, row block 0 = zeros
  float* Wh; float* e;            // [L B, A], [L B, Tn] stash (alpha when SM)
  bf16* gates;                    // [L B, H, 4] stash
  int B, L, Tn, MS;               // MS = samples per cluster
  float inv_T;
};

struct SmemF { int Ws, hs, og, whs, uvs, es, hst, part, total; };
__host__ __device__ inline SmemF smem_fwd() {
  SmemF s;
  s.Ws = 0;
  s.hs = s.Ws + NR * PITCH * 2;                   // [16][PITCH] bf16: h_{t-1} of the cluster's samples (rows >= nb stay zero)
  s.og = s.hs + MT * PITCH * 2;                   // [16][NR] f32: this CTA's columns of h_{t-1} [W_a ; W_hh]^T
  s.whs = s.og + MT * NR * 4;                     // [16][A] f32: gathered W h of every sample
  s.uvs = s.whs + MT * A_ * 4;                    // [MAXF][16][A] f32: U v + b of this CTA's frames
  s.es = s.uvs + MAXF * MT * A_ * 4;              // [16][MAXT] f32: gathered scores
  s.hst = s.es + MT * MAXT * 4;                   // [16 warps][32] bf16: staging of h_t for the 16-byte DSMEM stores
  s.part = s.hst + NWARP * 32 * 2;                // [16 warps][16][8] f32: K-split partials of the attention tile
  s.total = s.part + NWARP * MT * APC * 4 + 16;
  return s;
}

// NQ = frames held in registers per thread (a multiple of 4 >= Tn)
template <int NQ, bool SM>
__global__ void __launch_bounds__(THREADS, 1) decoder_fwd_cluster_kernel(const FwdArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  const SmemF S = smem_fwd();
  bf16* Ws = reinterpret_cast<bf16*>(smem + S.Ws);
  bf16* hs = reinterpret_cast<bf16*>(smem + S.hs);
  float* og = reinterpret_cast<float*>(smem + S.og);
  float* whs = reinterpret_cast<float*>(smem + S.whs);
  float* uvs = reinterpret_cast<float*>(smem + S.uvs);
  float* es = reinterpret_cast<float*>(smem + S.es);
  bf16* hst = reinterpret_cast<bf16*>(smem + S.hst);
  float* part = reinterpret_cast<float*>(smem + S.part);
  const int r = (int)cta_rank(), q = (int)cluster_id();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int B = a.B, Tn = a.Tn;
  const int b0 = q * a.MS, nb = min(a.MS, B - b0);            // this cluster's samples (whole cluster exits together if none)
  if (nb <= 0) return;

  // ---- one-time: weight rows, U.v of this CTA's frames, zero h_{-1}; per-thread constants
  for (int i = tid; i < NR * (H_ / 8); i += THREADS) {
    const int lr = i / (H_ / 8), c8 = i - lr * (H_ / 8);
    *reinterpret_cast<uint4*>(Ws + (size_t)lr * PITCH + 8 * c8) = *reinterpret_cast<const uint4*>(a.Wcat + (size_t)wcat_row(lr, r) * H_ + 8 * c8);
  }
  for (int i = tid; i < MT * PITCH / 2; i += THREADS) reinterpret_cast<uint32_t*>(hs)[i] = 0u;
  for (int i = tid; i < MAXF * MT * (A_ / 4); i += THREADS) {
    const int f = i / (MT * (A_ / 4)), rem = i - f * (MT * (A_ / 4)), s = rem / (A_ / 4), c4 = rem - s * (A_ / 4);
    const int tau = r + CS * f;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tau < Tn && s < nb) v = reinterpret_cast<const float4*>(a.Uv + ((size_t)(b0 + s) * Tn + tau) * A_)[c4];
    reinterpret_cast<float4*>(uvs)[i] = v;
  }
  for (int i = tid; i < MT * MAXT; i += THREADS) es[i] = 0.f;
  for (int i = tid; i < MT * A_; i += THREADS) whs[i] = 0.f;
  for (int i = tid; i < MT * NR; i += THREADS) og[i] = 0.f;
  // per-sample phases: warp <-> sample (clamped for idle warps), lane <-> unit of this CTA's slice / a-chunk of the score
  const bool act = warp < nb;
  const int s_w = min(warp, nb - 1), b = b0 + s_w;
  const int j = r * UPC + lane;
  pf::Quad<bf16> v[NQ];                                         // projected features of (sample, unit): resident for all L steps
  {
    const bf16* vw = a.VW + ((size_t)b * Tn * H_ + j) * 4;
#pragma unroll
    for (int k = 0; k < NQ; ++k) v[k].load(vw + (size_t)min(k, Tn - 1) * 4 * H_);
  }
  float bh[4];
#pragma unroll
  for (int g = 0; g < 4; ++g) bh[g] = a.b_hh[g * H_ + j];
  const float4 aw4 = reinterpret_cast<const float4*>(a.attn_w)[lane];
  float cstate = 0.f;
  __syncthreads();
  cluster_barrier();                                            // every CTA of the cluster is set up before the first remote store

  const uint32_t whs_sa = smem_addr(whs), es_sa = smem_addr(es), hs_sa = smem_addr(hs);
  const int gid = lane >> 2, tig = lane & 3;
  for (int t = 0; t < a.L; ++t) {
    // operands of the cell that do not depend on h_{t-1}: issued before anything else
    float gx[4];
    {
      const float* gp = a.Gx + ((size_t)t * B + b) * 4 * H_ + j;
#pragma unroll
      for (int g = 0; g < 4; ++g) gx[g] = gp[g * H_];
    }
    stamp(20);
    if (t > 0) {
      cluster_wait();                                           // #3 of the previous step: h_{t-1} is in every CTA's hs
      const uint32_t a_addr = hs_sa + (uint32_t)(((lane & 15) * PITCH + (lane >> 4) * 8) * 2);
      const uint32_t w_addr = smem_addr(Ws) + (uint32_t)(((lane & 7) * PITCH + ((lane >> 3) & 1) * 8) * 2);
      // ---- P1a: the 8 attention columns first (they gate the scores): K split over the 16 warps, partials summed through smem
      {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int kk = 0; kk < 2; ++kk) {
          uint32_t af[4], bfr[2];
          ldsm_x4(af, a_addr + (32 * warp + 16 * kk) * 2);
          ldsm_x2(bfr, w_addr + (32 * warp + 16 * kk) * 2);
          mma16816(acc, af, bfr);
        }
        float* pw = part + warp * (MT * APC);
        *reinterpret_cast<float2*>(pw + gid * APC + 2 * tig) = make_float2(acc[0], acc[1]);
        *reinterpret_cast<float2*>(pw + (gid + 8) * APC + 2 * tig) = make_float2(acc[2], acc[3]);
      }
      __syncthreads();
      // W.h all-gather: value (sample s, column c) summed over the 16 partials -> every CTA's whs[s][8 r + c]; thread = (item, 4 destinations)
      {
        const int item = tid & 127, grp = tid >> 7, s_ = item >> 3, c_ = item & 7;
        float sum = 0.f;
#pragma unroll
        for (int w2 = 0; w2 < NWARP; ++w2) sum += part[w2 * (MT * APC) + item];
        const uint32_t dst_off = whs_sa + (uint32_t)((s_ * A_ + r * APC + c_) * 4);
#pragma unroll
        for (int i = 0; i < 4; ++i) st_c_f32(mapa(dst_off, (uint32_t)(grp * 4 + i)), sum);
      }
      stamp(27);
      cluster_arrive();                                         // #1 (its latency hides behind the gate columns)
      // ---- P1b: the 128 gate columns, one 8-row n-tile per warp
      {
        float acc0[4] = {0.f, 0.f, 0.f, 0.f}, acc1[4] = {0.f, 0.f, 0.f, 0.f};        // two independent accumulation chains
        const uint32_t b_addr = w_addr + (uint32_t)((APC + warp * 8) * PITCH * 2);
#pragma unroll 2
        for (int k0 = 0; k0 < H_; k0 += 32) {
          uint32_t af[4], bfr[2], af2[4], bfr2[2];
          ldsm_x4(af, a_addr + k0 * 2);
          ldsm_x2(bfr, b_addr + k0 * 2);
          ldsm_x4(af2, a_addr + (k0 + 16) * 2);
          ldsm_x2(bfr2, b_addr + (k0 + 16) * 2);
          mma16816(acc0, af, bfr);
          mma16816(acc1, af2, bfr2);
        }
        const int n = APC + warp * 8 + 2 * tig;
        *reinterpret_cast<float2*>(og + gid * NR + n) = make_float2(acc0[0] + acc1[0], acc0[1] + acc1[1]);
        *reinterpret_cast<float2*>(og + (gid + 8) * NR + n) = make_float2(acc0[2] + acc1[2], acc0[3] + acc1[3]);
      }
      stamp(21);
      cluster_wait();                                           // #1: every sample's W.h is complete in whs
      stamp(22);
    }
    // ---- P2: scores of (sample warp, frames r and r + 16): lane owns a-chunk [4 lane, 4 lane + 4)
    {
      const float4 wh = reinterpret_cast<const float4*>(whs + s_w * A_)[lane];
      if (r == 0 && act) reinterpret_cast<float4*>(a.Wh + ((size_t)t * B + b) * A_)[lane] = wh;
      float sc[MAXF];
#pragma unroll
      for (int f = 0; f < MAXF; ++f) {
        const float4 u = reinterpret_cast<const float4*>(uvs + (f * MT + s_w) * A_)[lane];
        float s = aw4.x * act_tanh<true>(wh.x + u.x);
        s = fmaf(aw4.y, act_tanh<true>(wh.y + u.y), s);
        s = fmaf(aw4.z, act_tanh<true>(wh.z + u.z), s);
        sc[f] = fmaf(aw4.w, act_tanh<true>(wh.w + u.w), s);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int f = 0; f < MAXF; ++f) sc[f] += __shfl_xor_sync(0xffffffffu, sc[f], o);
      // all-gather: lane -> (destination CTA lane / 2, frame slot lane % 2)
      const int f = lane & 1, tau = r + CS * f;
      const float val = f ? sc[1] : sc[0];
      if (act && tau < Tn) {
        st_c_f32(mapa(es_sa + (uint32_t)((s_w * MAXT + tau) * 4), (uint32_t)(lane >> 1)), val);
        if (!SM && lane < 2) a.e[((size_t)t * B + b) * Tn + tau] = val;
      }
    }
    stamp(23);
    cluster_barrier();                                          // #2 (also orders this step's og writes before the reads below)
    stamp(24);
    if constexpr (SM) {       // this warp's row only: the next remote stores into es come after barrier #1 of the next step
      float* er = es + s_w * MAXT;
      const float al = warp_softmax<true>(er[lane], lane < Tn);
      __syncwarp();
      if (act) {
        if (lane < Tn) er[lane] = al;
        if (r == 0 && lane < Tn) a.e[((size_t)t * B + b) * Tn + lane] = al;
      }
      __syncwarp();
    }
    // ---- P3: context sum over the frames (features from registers), gates, c_t, h_t
    {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      const float4* e4 = reinterpret_cast<const float4*>(es + s_w * MAXT);
#pragma unroll
      for (int k4 = 0; k4 < NQ / 4; ++k4) {
        const float4 e = e4[k4];
        const float ev[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          float f[4];
          v[4 * k4 + kk].get(f);
#pragma unroll
          for (int g = 0; g < 4; ++g) acc[g] = fmaf(ev[kk], f[g], acc[g]);      // es is zero for tau >= Tn
        }
      }
      float pre[4];
#pragma unroll
      for (int g = 0; g < 4; ++g) pre[g] = gx[g] + bh[g] + og[s_w * NR + APC + g * UPC + lane] + acc[g] * a.inv_T;
      const float gi = act_sigmoid<true>(pre[0]), gf = act_sigmoid<true>(pre[1]), gt = act_tanh<true>(pre[2]), go = act_sigmoid<true>(pre[3]);
      const float cn = fmaf(gf, cstate, gi * gt);
      const float hn = go * act_tanh<true>(cn);
      const bf16 hb = __float2bfloat16_rn(hn);
      // h_t all-gather: the warp's 32 units (64 bytes) into row s_w of every CTA's hs, as 16-byte DSMEM stores
      hst[warp * 32 + lane] = hb;
      __syncwarp();
      if (act) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          const int item = lane * 2 + i, dst = item >> 2, chunk = item & 3;
          const uint4 val = *reinterpret_cast<const uint4*>(hst + warp * 32 + chunk * 8);
          st_c_u32x4(mapa(hs_sa + (uint32_t)((s_w * PITCH + r * UPC + chunk * 8) * 2), (uint32_t)dst), val);
        }
      }
      cluster_arrive();                                         // #3 (waited for at the top of the next step)
      if (act) {                                                // stash for the BPTT / the vocabulary projection: off the critical path
        cstate = cn;
        const size_t o1 = ((size_t)t * B + b) * H_ + j;
        a.c[o1 + (size_t)B * H_] = cn;
        a.hiddens[o1] = hn;
        a.Hop[o1 + (size_t)B * H_] = hb;
        pf::Quad<bf16>::store(a.gates + o1 * 4, gi, gf, gt, go);
      }
    }
    stamp(25);
  }
  cluster_wait();                                               // #3 of the last step: no CTA exits while a peer may still store into it
}

static inline bool cluster_enabled() {
  static const int v = rn_env_int("RECNET_DEC_CLUSTER", 1);
  return v != 0;
}
// shapes the cluster kernels are written for (MSVD decoder); everything else runs the kernel-per-phase loop
static inline bool cluster_ok(int B, int Tn, int A, int H) {
  return cluster_enabled() && H == H_ && A == A_ && Tn >= 1 && Tn <= MAXT && B >= 1 && B <= 8 * MAX_MS;
}

template <typename K>
static int launch_cluster(K kern, size_t smem, int B, cudaStream_t st, const void* args_struct_ptr, bool* configured) {
  (void)args_struct_ptr;
  if (!*configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) { cudaGetLastError(); return RECNET_ERR_UNSUPPORTED; }
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { cudaGetLastError(); return RECNET_ERR_UNSUPPORTED; }
    *configured = true;
  }
  return 0;
}

// samples per cluster such that all clusters are co-resident (one wave): ceil(B / max active clusters); 0 = not possible
template <typename K>
static int pick_ms(K kern, size_t smem, int B) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(8 * CS, 1, 1);
  cfg.blockDim = dim3(THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  int n = 0;
  if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
  n = rn_env_int("RECNET_DEC_CLUSTERS", n);          // developer override
  if (rn_env_int("RECNET_DEBUG_CLUSTERS", 0)) fprintf(stderr, "[recnet] decoder cluster kernel: max active %d-CTA clusters = %d\n", CS, n);
  if (n < 1) return 0;
  const int ms = (B + n - 1) / n;
  return ms <= MAX_MS ? ms : 0;
}

template <int NQ, bool SM>
static int launch_fwd_nq(FwdArgs a, cudaStream_t st) {
  auto kern = decoder_fwd_cluster_kernel<NQ, SM>;
  const size_t smem = smem_fwd().total;
  static bool configured = false;
  static int ms_cache_B = -1, ms_cache = 0;
  RN_TRY(launch_cluster(kern, smem, a.B, st, nullptr, &configured));
  if (ms_cache_B != a.B) { ms_cache = pick_ms(kern, smem, a.B); ms_cache_B = a.B; }
  if (ms_cache <= 0) return RECNET_ERR_UNSUPPORTED;               // the device cannot host enough clusters at once: kernel-per-phase loop
  a.MS = ms_cache;
  const int ncl = (a.B + a.MS - 1) / a.MS;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(ncl * CS, 1, 1);
  cfg.blockDim = dim3(THREADS, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  ProfScope prof(KC_LOOP, a.L, ncl * CS, 2, st);
  RN_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, a));
  RN_LAUNCH_OK();
  return 0;
}
// softmax: the paper's attention (a.inv_T must then be 1)
static int launch_fwd(const FwdArgs& a, bool softmax, cudaStream_t st) {
  if (softmax) return a.Tn <= 28 ? launch_fwd_nq<28, true>(a, st) : launch_fwd_nq<32, true>(a, st);
  return a.Tn <= 28 ? launch_fwd_nq<28, false>(a, st) : launch_fwd_nq<32, false>(a, st);
}
}  // namespace dcl
