// Decoder sequence driver, projected-feature formulation (single-layer LSTM decoder -- the BASELINE benchmark config).
// Same contract as dec::forward / dec::backward (train.py:17-75 over models/decoder.py:45-70); see proj_attn.cuh for
// the algebra.  Per step: ONE split-K GEMM on h_{t-1} (K = H) + ONE fused attention/cell kernel; BPTT: one fused
// cell/attention backward kernel + ONE split-K GEMM (K = A + 4H).
//   hoisted once per sequence: U v, VW = feats W_ctx^T (unit-interleaved, operand precision), embedding projection Gx
//   after the loop: vocabulary projection + CE + the per-step attention contexts (forward); all weight gradients as batched GEMMs (backward)
#pragma once
#include "proj_attn.cuh"
#include "seq_decoder.cuh"
#include "seq_decoder_cluster.cuh"

namespace dec {

template <typename T>
struct PfWs {
  int EMBp, Vp, Vld, NP;
  GemmPlan pl_h, pl_dh;
  T *Wemb, *WctxI, *Wcat, *U, *Wout, *feats;
  float* Uv; T* VW; T* Xe; float* Gx; T* Hop; float* P; float* Wh; float* e; T* gates; float* c;
  float *logits, *lse, *row_loss;
  T* dlogits; float* dHext; T* dGW; float* dhP; float* dWh; float* dUv; T* dUv_op; float* dw_acc; float* dc; float* dXe; T* ctx;
  float* splitk; float* splitk2; float* splitk3; int* err;      // splitk2: scratch of the side stream (runtime.cuh:Side), splitk3: of phase 4 alone
  size_t bytes;
};

// eligibility of the projected-feature path; everything else runs the general drivers (seq_decoder.cuh)
static inline bool pf_enabled() {
  static const int v = rn_env_int("RECNET_PF", 1);
  return v != 0;
}
static inline bool pf_ok(const recnet_decoder_desc& d) {
  if (!pf_enabled() || d.cell != RECNET_CELL_LSTM || d.n_layers > 1) return false;
  const int al = d.precision == RECNET_PREC_BF16 ? 8 : 4;
  if ((long long)d.B * d.T * 4 * d.H >= (1ll << 31) || (long long)d.L * d.B * (d.A + 4 * d.H) >= (1ll << 31)) return false;   // 32-bit index math
  if ((d.E & 1) || pf::escore_smem(d.L, d.T, true) > 46 * 1024) return false;          // pf_escore_kernel: column pairs, e[L x T] in shared memory
  return d.T >= 1 && d.T <= pf::MAX_T && d.A >= 4 && d.A <= pf::MAX_A && d.A % al == 0 && d.H % al == 0 &&
         pf::bwd_smem_bytes(d.H, d.A) <= 46 * 1024;
}
// the training driver a descriptor runs: projected-feature (here) or general (seq_decoder.cuh, single-layer and stacked)
enum class DecPath { PF, GENERAL };
static inline DecPath dec_path(const recnet_decoder_desc& d) {
  return pf_ok(d) ? DecPath::PF : DecPath::GENERAL;
}

template <typename T>
static PfWs<T> plan_pf(const recnet_decoder_desc& d, void* base) {
  PfWs<T> w;
  const int B = d.B, L = d.L, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T;
  w.EMBp = round_up(d.EMB, Prec<T>::kpad);
  w.Vp = round_up(V, 8);
  w.Vld = round_up(V, 4);
  w.NP = A + 4 * H;
  w.pl_h = plan_gemm<T>(B, w.NP, H);
  w.pl_dh = plan_gemm<T>(B, H, w.NP);
  if (Prec<T>::id == RECNET_PREC_BF16) {
    // K = H is only 8 k-blocks: 64-wide N tiles x few splits (34 x 4 CTAs at H = 512) instead of 128-wide x 8 -- half the
    // partial traffic for the fused kernel to sum
    w.pl_h.bn = 64;
    const int tiles = rn_cdiv(B, tc::BM) * rn_cdiv(w.NP, 64), nkb = rn_cdiv(H, tc::BK);
    int sp = NUM_SMS / tiles; if (sp < 1) sp = 1; if (sp > nkb) sp = nkb;
    w.pl_h.splits = rn_cdiv(nkb, rn_cdiv(nkb, sp));
    // dh GEMM (N = H, K = A + 4H): at most pf::MAXS splits so the fused backward kernel sums them with one batch of loads
    const int nkb2 = rn_cdiv(w.NP, tc::BK);
    if (w.pl_dh.splits > pf::MAXS) w.pl_dh.splits = rn_cdiv(nkb2, rn_cdiv(nkb2, pf::MAXS));
    // tuning overrides (tools/ sweeps): RECNET_PF_SPLITS_H / RECNET_PF_SPLITS_DH / RECNET_PF_BN_H
    static const int eh = rn_env_int("RECNET_PF_SPLITS_H", 0);
    static const int edh = rn_env_int("RECNET_PF_SPLITS_DH", 0);
    static const int ebn = rn_env_int("RECNET_PF_BN_H", 0);
    if (ebn == 64 || ebn == 128) w.pl_h.bn = ebn;
    if (eh > 0) w.pl_h.splits = rn_cdiv(nkb, rn_cdiv(nkb, eh > nkb ? nkb : eh));
    if (edh > 0) w.pl_dh.splits = rn_cdiv(nkb2, rn_cdiv(nkb2, edh > nkb2 ? nkb2 : edh));
  }
  Bump m(base);
  w.Wemb = m.take<T>((size_t)4 * H * w.EMBp);
  w.WctxI = m.take<T>((size_t)4 * H * E);
  w.Wcat = m.take<T>((size_t)w.NP * H);
  w.U = m.take<T>((size_t)A * E);
  w.Wout = m.take<T>((size_t)V * H);
  w.feats = m.take<T>((size_t)B * Tn * E);
  w.Uv = m.take<float>((size_t)B * Tn * A);
  w.VW = m.take<T>((size_t)B * Tn * 4 * H);
  w.Xe = m.take<T>((size_t)L * B * w.EMBp);
  w.Gx = m.take<float>((size_t)L * B * 4 * H);
  w.Hop = m.take<T>((size_t)(L + 1) * B * H);
  w.P = m.take<float>((size_t)w.pl_h.splits * B * w.NP);
  w.Wh = m.take<float>((size_t)L * B * A);
  w.e = m.take<float>((size_t)L * B * Tn);
  w.gates = m.take<T>((size_t)L * B * 4 * H);
  w.c = m.take<float>((size_t)(L + 1) * B * H);
  w.logits = m.take<float>((size_t)L * B * w.Vld);
  w.lse = m.take<float>((size_t)L * B);
  w.row_loss = m.take<float>((size_t)L * B);
  w.dlogits = m.take<T>((size_t)L * B * w.Vp);
  w.dHext = m.take<float>((size_t)L * B * H);
  w.dGW = m.take<T>((size_t)L * B * w.NP);
  w.dhP = m.take<float>((size_t)w.pl_dh.splits * B * H);
  w.dWh = m.take<float>((size_t)L * B * A);
  w.dUv = m.take<float>((size_t)B * Tn * A);
  w.dUv_op = m.take<T>((size_t)B * Tn * A);
  w.dw_acc = m.take<float>((size_t)B * A);
  w.dc = m.take<float>((size_t)B * H);
  w.dXe = m.take<float>((size_t)L * B * w.EMBp);
  w.ctx = m.take<T>((size_t)L * B * E);          // attention context of every step (forward, training calls): B-operand of dW_ctx
  w.splitk = m.take<float>(SPLITK_SCRATCH_FLOATS);
  w.splitk2 = m.take<float>(SPLITK_SCRATCH_FLOATS);
  w.splitk3 = m.take<float>(SPLITK_SCRATCH_FLOATS);
  w.err = m.take<int>(64);
  w.bytes = m.off + 256;
  return w;
}

// C (operand type) = A B^T, written straight in the operand precision
static inline int gemm_to_operand(const float* A, long long lda, const float* B, long long ldb, float* C, long long ldc, int M,
                                  int N, int K, float* scratch, cudaStream_t st) {
  return gemm_full<float>(A, lda, 0, B, ldb, 0, C, ldc, nullptr, M, N, K, 0, scratch, st);
}
static inline int gemm_to_operand(const bf16* A, long long lda, const bf16* B, long long ldb, bf16* C, long long ldc, int M, int N,
                                  int K, float*, cudaStream_t st) {
  GemmPlan p = plan_gemm_full<bf16>(M, N, K);
  if (p.splits > 1) p = plan_gemm<bf16>(M, N, K);          // the operand-typed epilogue needs the whole K range in one CTA
  return tc::launch(A, lda, 0, B, ldb, 0, nullptr, 0, C, ldc, nullptr, M, N, K, 1, 0, 0, p.bn, st);
}

template <typename T>
static int forward_pf(const DecDesc& d, const recnet_decoder_tensors& p, const float* feats, const long long* tokens_in,
                      const long long* targets, const float* ce_weight, const unsigned long long* rng, void* ws, long long ws_bytes,
                      float* hiddens, float* ce_out, cudaStream_t st, int phases = 3) {
  // phases (recnet_decoder_fwd_phase): 1 = staging, hoisted projections and the time loop (-> hiddens), 2 = vocabulary projection, per-step
  // attention contexts, CE (-> ce_out; needs 1).  Nothing after the loop feeds the reconstructor, so a trainer may run 2 on another stream.
  RN_TRY(check(d));
  PfWs<T> w = plan_pf<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, L = d.L, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T, EMB = d.EMB;
  const float p_emb = d.train ? d.p_emb_drop : 0.f, p_out = d.train ? d.p_out_drop : 0.f;
  const float inv_T = d.softmax ? 1.f : 1.f / Tn;             // softmax: alpha weights, summed without the 1/T of the mean
  const long long ldih = EMB + E;
  if (phases & 1) {
  // operand copies of the weights / features (the optimiser changes the fp32 masters every step)
  // operand copies of the weights / features + cleared initial state: ONE multi-tensor staging kernel (misc.cuh:Stager)
  // (the embedding gather needs neither: it starts on the second stream right away, next to the staging kernel)
  cudaStream_t s2;
  RN_TRY(side().fork(st, &s2));
  misc::embed_gather_kernel<T><<<L * B, 128, 0, s2>>>(p.embedding, tokens_in, w.Xe, w.EMBp, L * B, EMB, w.EMBp, V, d.embedding_scale,
                                                      p_emb, rng, SITE_EMB);
  RN_LAUNCH_OK();
  misc::Stager<T> sg;
  sg.add(feats, E, w.feats, E, (long long)B * Tn, E, E);
  sg.add(p.attn_U, E, w.U, E, A, E, E);
  sg.add(p.w_ih, ldih, w.Wemb, w.EMBp, 4 * H, EMB, w.EMBp);
  sg.add(p.w_ih + EMB, ldih, w.WctxI, E, 4 * H, E, E, H);                 // W_ctx rows in unit-interleaved order
  sg.add(p.attn_W, H, w.Wcat, H, A, H, H);
  sg.add(p.w_hh, H, w.Wcat + (size_t)A * H, H, 4 * H, H, H);
  sg.add(p.out_w, H, w.Wout, H, V, H, H);
  sg.zero(w.Hop, (size_t)B * H * sizeof(T));
  sg.zero(w.c, (size_t)B * H * sizeof(float));
  sg.zero(w.err, 64 * sizeof(int));
  RN_TRY(sg.launch(st));
  // hoisted projections (runtime.cuh:Side): the key projection and the time-batched embedding half of the gate projection run on the
  // second stream next to the projected-feature GEMM; the second fork orders that stream after the staging kernel.
  RN_TRY(side().fork(st, &s2));
  RN_TRY(gemm_full<T>(w.feats, E, 0, w.U, E, 0, w.Uv, A, p.attn_b, B * Tn, A, E, 0, w.splitk2, s2));      // U v + b (bias folded in)
  RN_TRY(gemm_full<T>(w.Xe, w.EMBp, 0, w.Wemb, w.EMBp, 0, w.Gx, 4 * H, p.b_ih, L * B, 4 * H, w.EMBp, 0, w.splitk2, s2));
  RN_TRY(gemm_to_operand(w.feats, E, w.WctxI, E, w.VW, 4 * H, B * Tn, 4 * H, E, w.splitk, st));
  RN_TRY(side().join(st, s2));
  bool clustered = false;
  if constexpr (std::is_same<T, bf16>::value) {
    if (dcl::cluster_ok(B, Tn, A, H)) {
      // the whole time loop as ONE kernel of independent 16-CTA clusters, [W_a ; W_hh] resident in distributed shared memory
      dcl::FwdArgs ca{};
      ca.Wcat = w.Wcat; ca.Uv = w.Uv; ca.attn_w = p.attn_w; ca.VW = w.VW; ca.Gx = w.Gx; ca.b_hh = p.b_hh; ca.c = w.c; ca.hiddens = hiddens;
      ca.Hop = w.Hop; ca.Wh = w.Wh; ca.e = w.e; ca.gates = w.gates; ca.B = B; ca.L = L; ca.Tn = Tn; ca.inv_T = inv_T;
      const int rc = dcl::launch_fwd(ca, d.softmax, st);
      if (rc == 0) clustered = true;
      else if (rc != RECNET_ERR_UNSUPPORTED) return rc;
    }
  }
  for (int t = 0; t < L && !clustered; ++t) {
    const size_t r = (size_t)t * B;
    if (t > 0)      // h_{-1} = 0: no query, no recurrent term
      RN_TRY(gemm_partials<T>(w.Hop + r * H, H, 0, w.Wcat, H, 0, w.P, B, w.NP, H, w.pl_h, st));
    pf::FwdArgs fa{};
    fa.P = w.P; fa.n_p = t > 0 ? w.pl_h.splits : 0; fa.p_stride = (long long)B * w.NP; fa.NP = w.NP;
    fa.Uv = w.Uv; fa.attn_w = p.attn_w; fa.VW = w.VW;
    fa.Gx = w.Gx + r * 4 * H; fa.b_hh = p.b_hh; fa.c_prev = w.c + r * H;
    fa.B = B; fa.Tn = Tn; fa.A = A; fa.H = H; fa.inv_T = inv_T;
    fa.Wh_out = w.Wh + r * A; fa.e_out = w.e + r * Tn; fa.gates_out = w.gates + r * 4 * H;
    fa.c_out = w.c + (r + B) * H; fa.h_out = hiddens + r * H; fa.h_op = w.Hop + (r + B) * H;
    RN_TRY((pf::launch_fwd<T, T>(fa, d.softmax, st)));
  }
  }   // phases & 1
  if (!(phases & 2)) return 0;
  // Training calls: the attention context of every step, ctx_t[b] = (1/T) sum_tau e_t[b,tau] v[b,tau] (decoder.py:57-62).  The forward pass never
  // needs it (the projected features carry it), but dW_ctx = sum_t dG_t^T ctx_t does, and HERE it costs nothing: its 256-thread CTAs share the
  // SMs with the vocabulary GEMM's.  (Until r2_i backward formed dVW[b,tau] = (1/T) sum_t e_t[b,tau] dG_t[b] after its loop instead: 29-52 us on
  // the critical path.)
  const bool training = targets && ce_weight && ce_out;
  cudaStream_t s3 = st;
  if (training) RN_TRY(side().fork(st, &s3));
  // vocabulary projection over all steps, then the masked CE (train.py:54-60,68)
  RN_TRY(gemm_full<T>(w.Hop + (size_t)B * H, H, 0, w.Wout, H, 0, w.logits, w.Vld, p.out_b, L * B, V, H, 0, w.splitk, st));
  if (training) {
    // launched after the GEMM: CTAs are dispatched in launch order (inside a captured graph sibling branches may still start in either order)
    // (one sample per CTA = two waves of CTAs.  A one-wave grid -- pf::escore_spc, three samples per CTA -- lets the GEMM start at once
    // when the graph happens to launch this branch first, but its long-lived CTAs then slow the GEMM they share the SMs with: 65 vs 34 us,
    // measured; the two-wave grid costs the GEMM a 20 us late start at worst)
    const int spc = 1;
    pf::pf_escore_kernel<T, true><<<dim3(rn_cdiv(E, 512), rn_cdiv(B, spc)), 256, pf::escore_smem(L, Tn, true), s3>>>(w.e, w.feats, E, 0, w.ctx, L, B,
                                                                                                               Tn, E, inv_T, spc);
    RN_LAUNCH_OK();
  }
  if (targets && ce_weight && ce_out) {
    ProfScope prof(KC_CE, L * B, V, 0, st);
    loss::ce_fwd_kernel<<<L * B, loss::CE_THREADS, 0, st>>>(w.logits, w.Vld, targets, ce_weight, V, p_out, rng, SITE_LOGITS, w.lse,
                                                            w.row_loss);
    RN_LAUNCH_OK();
    loss::sum_kernel<<<1, 1024, 0, st>>>(w.row_loss, L * B, ce_out, 1.f);
    RN_LAUNCH_OK();
  }
  if (training) RN_TRY(side().join(st, s3));
  return 0;
}

template <typename T>
static int backward_pf(const DecDesc& d, const recnet_decoder_tensors& p, const float* feats, const long long* tokens_in,
                       const long long* targets, const float* ce_weight, const unsigned long long* rng, void* ws, long long ws_bytes,
                       const float* g_ce, const float* g_hiddens, const recnet_decoder_tensors& g, cudaStream_t st, int phases = 15) {
  // phases (recnet_decoder_bwd_phase): 1 = CE backward + gradient wrt the states through the vocabulary projection, 2 = the BPTT loop,
  // 4 = the vocabulary projection's own gradients (need only phase 1), 8 = every other parameter gradient (needs the loop)
  RN_TRY(check(d));
  PfWs<T> w = plan_pf<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, L = d.L, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T, EMB = d.EMB;
  const float p_emb = d.train ? d.p_emb_drop : 0.f, p_out = d.train ? d.p_out_drop : 0.f;
  const int LB = L * B, NP = w.NP;
  const T* Hall = w.Hop + (size_t)B * H;          // h_t rows
  // ---- CE backward and the vocabulary projection
  if (phases & 1) {
    {
      ProfScope prof(KC_CE, LB, V, 1, st);
      loss::ce_bwd_kernel<T><<<LB, loss::CE_THREADS, 0, st>>>(w.logits, w.Vld, targets, ce_weight, w.lse, g_ce, V, w.Vp, p_out, rng,
                                                              SITE_LOGITS, w.dlogits, w.Vp);
    }
    RN_LAUNCH_OK();
    RN_TRY(gemm_full<T>(w.dlogits, w.Vp, 0, w.Wout, H, 1, w.dHext, H, nullptr, LB, H, V, 0, w.splitk, st));
  }
  // (the vocabulary projection's own gradients do not feed the loop: phase 4)
  // ---- BPTT
  for (int t = L - 1; t >= 0 && (phases & 2); --t) {
    const bool last = (t == L - 1);
    const size_t r = (size_t)t * B;
    pf::BwdArgs ba{};
    ba.dh_ext = w.dHext + r * H; ba.dh_ext2 = g_hiddens ? g_hiddens + r * H : nullptr;
    ba.dhP = last ? nullptr : w.dhP; ba.n_p = w.pl_dh.splits; ba.p_stride = (long long)B * H;
    ba.dc = w.dc; ba.first = last ? 1 : 0;
    ba.gates = w.gates + r * 4 * H; ba.c_prev = w.c + r * H; ba.c_new = w.c + (r + B) * H;
    ba.VW = w.VW; ba.Wh = w.Wh + r * A; ba.Uv = w.Uv; ba.attn_w = p.attn_w;
    ba.B = B; ba.Tn = Tn; ba.A = A; ba.H = H; ba.inv_T = d.softmax ? 1.f : 1.f / Tn; ba.alpha = d.softmax ? w.e + r * Tn : nullptr;
    ba.dGW = w.dGW + r * NP; ba.dgw_ld = NP; ba.dWh_out = w.dWh + r * A;
    ba.dUv_acc = w.dUv; ba.uv_first = last ? 1 : 0; ba.dw_acc = w.dw_acc; ba.dw_first = last ? 1 : 0;
    RN_TRY((pf::launch_bwd<T, T>(ba, st)));
    // dh_{t-1} = [dWh_t | dG_t] [W_a ; W_hh]  (attention-query path and recurrent path in one K-concatenated GEMM)
    if (t > 0) RN_TRY(gemm_partials<T>(w.dGW + r * NP, NP, 0, w.Wcat, H, 1, w.dhP, B, H, NP, w.pl_dh, st));
  }
  // ---- batched weight gradients over the stashed operands, two streams (runtime.cuh:Side)
  const long long ldih = EMB + E;
  const T* dG = w.dGW + A;                       // [LB, 4H] gate gradients, ld = NP
  if (phases == 4) {                               // on its own (a trainer's background lane): the 13 GFLOP weight gradient only -- the bias
    RN_TRY(gemm_full<T>(w.dlogits, w.Vp, 1, Hall, H, 1, g.out_w, H, nullptr, V, H, LB, 0, w.splitk3, st));      // gradient (a 26 MB column
    return 0;                                      // sum: 93 us within the lane's CTA budget, 10 us without) belongs to phase 8
  }
  if (!(phases & 8)) return 0;
  cudaStream_t s2;
  RN_TRY(side().fork(st, &s2));
  // side: vocabulary projection, embedding path, attention query weights
  if (phases & 4) RN_TRY(gemm_full<T>(w.dlogits, w.Vp, 1, Hall, H, 1, g.out_w, H, nullptr, V, H, LB, 0, w.splitk2, s2));
  RN_TRY(misc::colsum<T>(w.dlogits, w.Vp, LB, V, g.out_b, 0, w.splitk2, s2));
  RN_TRY(gemm_full<T>(dG, NP, 1, w.Xe, w.EMBp, 1, g.w_ih, ldih, nullptr, 4 * H, EMB, LB, 0, w.splitk2, s2));               // dW_emb
  RN_TRY(gemm_full<T>(dG, NP, 0, w.Wemb, w.EMBp, 1, w.dXe, w.EMBp, nullptr, LB, EMB, 4 * H, 0, w.splitk2, s2));            // dXe
  RN_CUDA_OK(cudaMemsetAsync(g.embedding, 0, (size_t)V * EMB * sizeof(float), s2));
  misc::embed_scatter_kernel<<<LB, 128, 0, s2>>>(g.embedding, tokens_in, w.dXe, w.EMBp, LB, EMB, V, d.embedding_scale, p_emb, rng,
                                                 SITE_EMB);
  RN_LAUNCH_OK();
  RN_TRY(gemm_full<T>(w.dGW, NP, 1, w.Hop, H, 1, g.attn_W, H, nullptr, A, H, LB, 0, w.splitk2, s2));                       // dW_a = dWh^T h_{t-1}
  // st: gate biases, context weights (dW_ctx = dG^T ctx, the contexts stashed by the forward pass), recurrent weights, keys
  RN_TRY(misc::colsum<T>(dG, NP, LB, 4 * H, g.b_ih, 0, w.splitk, st, g.b_hh));            // b_ih and b_hh get the same gradient
  RN_TRY(gemm_full<T>(dG, NP, 1, w.ctx, E, 1, g.w_ih + EMB, ldih, nullptr, 4 * H, E, LB, 0, w.splitk, st));            // dW_ctx = dG^T ctx
  RN_TRY(gemm_full<T>(dG, NP, 1, w.Hop, H, 1, g.w_hh, H, nullptr, 4 * H, H, LB, 0, w.splitk, st));                        // dW_hh = dG^T h_{t-1}
  RN_TRY(misc::cast_pad<T>(w.dUv, A, w.dUv_op, A, (long long)B * Tn, A, A, st));
  RN_TRY(gemm_full<T>(w.dUv_op, A, 1, w.feats, E, 1, g.attn_U, E, nullptr, A, E, B * Tn, 0, w.splitk, st));               // dU = dUv^T v
  RN_TRY(misc::colsum<float>(w.dWh, A, LB, A, g.attn_b, 0, w.splitk, st));
  RN_TRY(misc::colsum<float>(w.dw_acc, A, B, A, g.attn_w, 0, w.splitk, st));
  RN_TRY(side().join(st, s2));
  return 0;
}
// ---- greedy decoding (eval.greedy_search, eval.py:19-33) on the projected-feature kernels: bf16 build -----------------------------
// 4 launches per step instead of 8: the embedding half of the gate projection is a GATHER from EW = Embedding . W_emb^T + b_ih
// (one [V x 4H x EMB] GEMM per call; eval mode has no dropout), the context half is the hoisted VW (as in training), so a step is
//   h_{t-1} [W_a ; W_hh]^T  ->  pf_fwd_kernel (scores, context, cell; Gx row = fed-back token)  ->  vocabulary projection  ->  argmax feedback.
// The fp32 build keeps the general path (seq_decoder.cuh:decode): its summation order is the one the bit-exact id tests pin.
// The arguments passed check_decode; the <SOS> fill, the arg-max feedback and the stop step are those of decode.
template <typename T>
struct GreedyPfWs {
  int EMBp, Vld, NP;
  GemmPlan pl_h;
  T *Wemb, *WctxI, *Wcat, *U, *Wout, *feats, *Emb;
  float* Uv; T* VW; float* EW; T* Hop; float* P; float* c; float* hid; float* logits; long long* tok; int* nonpad; float* splitk;
  size_t bytes;
};
template <typename T>
static GreedyPfWs<T> plan_greedy_pf(const recnet_decoder_desc& d, void* base, int max_steps) {
  GreedyPfWs<T> w;
  const int B = d.B, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T;
  w.EMBp = round_up(d.EMB, Prec<T>::kpad);
  w.Vld = round_up(V, 4);
  w.NP = A + 4 * H;
  w.pl_h = plan_gemm<T>(B, w.NP, H);
  Bump m(base);
  w.Wemb = m.take<T>((size_t)4 * H * w.EMBp);
  w.WctxI = m.take<T>((size_t)4 * H * E);
  w.Wcat = m.take<T>((size_t)w.NP * H);
  w.U = m.take<T>((size_t)A * E);
  w.Wout = m.take<T>((size_t)V * H);
  w.feats = m.take<T>((size_t)B * Tn * E);
  w.Emb = m.take<T>((size_t)V * w.EMBp);
  w.Uv = m.take<float>((size_t)B * Tn * A);
  w.VW = m.take<T>((size_t)B * Tn * 4 * H);
  w.EW = m.take<float>((size_t)V * 4 * H);
  w.Hop = m.take<T>((size_t)2 * B * H);
  w.P = m.take<float>((size_t)w.pl_h.splits * B * w.NP);
  w.c = m.take<float>((size_t)2 * B * H);
  w.hid = m.take<float>((size_t)B * H);
  w.logits = m.take<float>((size_t)B * w.Vld);
  w.tok = m.take<long long>(B);
  w.nonpad = m.take<int>(max_steps);
  w.splitk = m.take<float>(SPLITK_SCRATCH_FLOATS);
  w.bytes = m.off + 256;
  return w;
}
static inline bool greedy_pf_ok(const recnet_decoder_desc& d) {
  static const int on = rn_env_int("RECNET_GREEDY_PF", 1);
  return on && d.precision == RECNET_PREC_BF16 && pf_ok(d) && (long long)d.V * 4 * d.H < (1ll << 31);
}

static int greedy_pf(const DecDesc& d0, const recnet_decoder_tensors& p, const float* feats, int max_steps, void* ws,
                     long long ws_bytes, long long* ids_out, int* n_steps_out, cudaStream_t st) {
  typedef bf16 T;
  DecDesc d = d0; d.L = 1; d.train = 0;
  GreedyPfWs<T> w = plan_greedy_pf<T>(d, ws, max_steps);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T, EMB = d.EMB;
  const long long ldih = EMB + E;
  misc::Stager<T> sg;
  sg.add(feats, E, w.feats, E, (long long)B * Tn, E, E);
  sg.add(p.attn_U, E, w.U, E, A, E, E);
  sg.add(p.w_ih, ldih, w.Wemb, w.EMBp, 4 * H, EMB, w.EMBp);
  sg.add(p.w_ih + EMB, ldih, w.WctxI, E, 4 * H, E, E, H);                 // W_ctx rows in unit-interleaved order
  sg.add(p.attn_W, H, w.Wcat, H, A, H, H);
  sg.add(p.w_hh, H, w.Wcat + (size_t)A * H, H, 4 * H, H, H);
  sg.add(p.out_w, H, w.Wout, H, V, H, H);
  sg.add(p.embedding, EMB, w.Emb, w.EMBp, V, EMB, w.EMBp);
  sg.zero(w.Hop, (size_t)2 * B * H * sizeof(T));
  sg.zero(w.c, (size_t)2 * B * H * sizeof(float));
  sg.zero(w.nonpad, (size_t)max_steps * sizeof(int));
  RN_TRY(sg.launch(st));
  // hoisted once per call: U v + b, VW = feats W_ctx^T, EW = (embedding_scale * Embedding) W_emb^T + b_ih
  RN_TRY(gemm_full<T>(w.feats, E, 0, w.U, E, 0, w.Uv, A, p.attn_b, B * Tn, A, E, 0, w.splitk, st));
  RN_TRY(gemm_to_operand(w.feats, E, w.WctxI, E, w.VW, 4 * H, B * Tn, 4 * H, E, w.splitk, st));
  RN_TRY(gemm_full<T>(w.Emb, w.EMBp, 0, w.Wemb, w.EMBp, 0, w.EW, 4 * H, nullptr, V, 4 * H, w.EMBp, 0, w.splitk, st));
  misc::scale_add_bias_kernel<<<NUM_SMS * 4, 256, 0, st>>>(w.EW, (long long)V * 4 * H, 4 * H, d.embedding_scale, p.b_ih);
  RN_LAUNCH_OK();
  fill_tokens_kernel<<<rn_cdiv(B, 128), 128, 0, st>>>(w.tok, B, 1 /* <SOS> */);
  RN_LAUNCH_OK();
  for (int t = 0; t < max_steps; ++t) {
    T* h_p = w.Hop + (size_t)(t & 1) * B * H;
    T* h_n = w.Hop + (size_t)((t + 1) & 1) * B * H;
    float* c_p = w.c + (size_t)(t & 1) * B * H;
    float* c_n = w.c + (size_t)((t + 1) & 1) * B * H;
    if (t > 0) RN_TRY(gemm_partials<T>(h_p, H, 0, w.Wcat, H, 0, w.P, B, w.NP, H, w.pl_h, st));
    pf::FwdArgs fa{};
    fa.P = w.P; fa.n_p = t > 0 ? w.pl_h.splits : 0; fa.p_stride = (long long)B * w.NP; fa.NP = w.NP;
    fa.Uv = w.Uv; fa.attn_w = p.attn_w; fa.VW = w.VW;
    fa.Gx = w.EW; fa.gx_rows = w.tok; fa.b_hh = p.b_hh; fa.c_prev = c_p;
    fa.B = B; fa.Tn = Tn; fa.A = A; fa.H = H; fa.inv_T = d.softmax ? 1.f : 1.f / Tn;
    fa.Wh_out = nullptr; fa.e_out = nullptr; fa.gates_out = nullptr;
    fa.c_out = c_n; fa.h_out = w.hid; fa.h_op = h_n;
    RN_TRY((pf::launch_fwd<T, T>(fa, d.softmax, st)));
    RN_TRY(gemm_full<T>(h_n, H, 0, w.Wout, H, 0, w.logits, w.Vld, p.out_b, B, V, H, 0, w.splitk, st));
    argmax_feedback_kernel<<<B, 256, 0, st>>>(w.logits, w.Vld, V, ids_out + (size_t)t * B, w.tok, w.nonpad + t);
    RN_LAUNCH_OK();
  }
  greedy_finalize_kernel<<<1, 1, 0, st>>>(w.nonpad, max_steps, n_steps_out);
  RN_LAUNCH_OK();
  return 0;
}
}  // namespace dec
