// Stacked (n_layers > 1) LSTM decoder: models/decoder.py:36-40,66 with num_layers = NL.  Layer 0 is the single-layer
// step (input [emb ; ctx]); layer l >= 1 consumes h^{l-1}_t (inter-layer dropout in train mode) and its own h^l_{t-1} as
// ONE K-concatenated GEMM over operand rows X_l[t] = [h^{l-1}_t ; h^l_{t-1}].  The attention query and the vocabulary
// projection use the TOP layer (decoder.py:51,68); `hiddens` returns every layer, (L, NL, B, H) (train.py:61-64).
// One kernel per phase (no persistent-loop variant for the stacked case).
#pragma once
#include "seq_decoder.cuh"

namespace dec {

enum : unsigned { SITE_LAYER0 = 16 };     // dropout site of the input of layer l = SITE_LAYER0 + l

template <typename T>
static int forward_ml(const DecDesc& d, const recnet_decoder_tensors& p, const float* feats, const long long* tokens_in,
                      const long long* targets, const float* ce_weight, const unsigned long long* rng, void* ws, long long ws_bytes,
                      float* hiddens, float* ce_out, cudaStream_t st) {
  RN_TRY(check(d));
  Ws<T> w = plan<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, L = d.L, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T, NL = w.NL, top = NL - 1;
  const float p_emb = d.train ? d.p_emb_drop : 0.f, p_out = d.train ? d.p_out_drop : 0.f, p_lay = d.train ? d.p_layer_drop : 0.f;
  RN_TRY(prepare<T>(d, p, feats, w, st));
  for (int l = 1; l < NL; ++l) {
    RN_TRY(misc::cast_pad<T>(p.w_ih_x[l - 1], H, w.Wrec_x[l - 1], 2 * H, 4 * H, H, H, st));
    RN_TRY(misc::cast_pad<T>(p.w_hh_x[l - 1], H, w.Wrec_x[l - 1] + H, 2 * H, 4 * H, H, H, st));
  }
  RN_TRY(gemm_full<T>(w.feats, E, 0, w.U, E, 0, w.Uv, A, nullptr, B * Tn, A, E, 0, w.splitk, st));
  misc::embed_gather_kernel<T><<<L * B, 128, 0, st>>>(p.embedding, tokens_in, w.Xe, w.EMBp, L * B, d.EMB, w.EMBp, V,
                                                      d.embedding_scale, p_emb, rng, SITE_EMB);
  RN_LAUNCH_OK();
  RN_TRY(gemm_full<T>(w.Xe, w.EMBp, 0, w.Wemb, w.EMBp, 0, w.Gx, 4 * H, p.b_ih, L * B, 4 * H, w.EMBp, 0, w.splitk, st));
  RN_CUDA_OK(cudaMemsetAsync(w.X, 0, (size_t)B * w.KX * sizeof(T), st));
  RN_CUDA_OK(cudaMemsetAsync(w.c, 0, (size_t)B * H * sizeof(float), st));
  RN_CUDA_OK(cudaMemsetAsync(w.err, 0, sizeof(int), st));
  for (int l = 1; l < NL; ++l) {
    RN_CUDA_OK(cudaMemsetAsync(w.X_x[l - 1], 0, (size_t)B * 2 * H * sizeof(T), st));
    RN_CUDA_OK(cudaMemsetAsync(w.c_x[l - 1], 0, (size_t)B * H * sizeof(float), st));
  }
  T* Xtop = w.X_x[top - 1];
  for (int t = 0; t < L; ++t) {
    T* x0 = w.X + (size_t)t * B * w.KX;
    // attention with the top layer's previous state as query
    int n_whp = 0;
    if (t > 0) {
      RN_TRY(gemm_partials<T>(Xtop + (size_t)t * B * 2 * H + H, 2 * H, 0, w.Wa, H, 0, w.WhP, B, A, H, w.pl_wh, st));
      n_whp = w.pl_wh.splits;
    }
    attn::FwdArgs fa{};
    fa.WhP = w.WhP; fa.n_whp = n_whp; fa.whp_stride = (long long)B * A;
    fa.Uv = w.Uv; fa.uv_bs = (long long)Tn * A; fa.uv_ts = A; fa.attn_b = p.attn_b; fa.attn_w = p.attn_w;
    fa.V = w.feats; fa.v_bs = (long long)Tn * E; fa.v_ts = E; fa.B = B; fa.Tn = Tn; fa.A = A; fa.D = E;
    fa.inv_T = d.softmax ? 1.f : 1.f / Tn; fa.normalize = d.softmax;
    fa.Wh_out = w.Wh + (size_t)t * B * A; fa.e_out = w.e + (size_t)t * B * Tn; fa.ctx_out = x0; fa.ctx_ld = w.KX;
    RN_TRY((attn::launch_fwd<T, T>(fa, st)));
    for (int l = 0; l < NL; ++l) {
      const int K = l == 0 ? w.KX : 2 * H;
      T* xl = l == 0 ? x0 : w.X_x[l - 1] + (size_t)t * B * 2 * H;
      const T* Wl = l == 0 ? w.Wrec : w.Wrec_x[l - 1];
      const GemmPlan pl = l == 0 ? w.pl_gate : w.pl_gate_x;
      RN_TRY(gemm_partials<T>(xl, K, 0, Wl, K, 0, w.P, B, 4 * H, K, pl, st));
      float* cl = l == 0 ? w.c : w.c_x[l - 1];
      cell::FwdArgs ca{};
      ca.P = w.P; ca.n_p = pl.splits; ca.p_stride = (long long)B * 4 * H; ca.p_ld = 4 * H;
      if (l == 0) { ca.Gx = w.Gx + (size_t)t * B * 4 * H; ca.gx_ld = 4 * H; ca.b1 = nullptr; ca.b2 = p.b_hh; }
      else { ca.Gx = nullptr; ca.b1 = p.b_ih_x[l - 1]; ca.b2 = p.b_hh_x[l - 1]; }
      ca.c_prev = cl + (size_t)t * B * H; ca.c_out = cl + (size_t)(t + 1) * B * H; ca.B = B; ca.H = H;
      ca.gates_out = (l == 0 ? w.gates : w.gates_x[l - 1]) + (size_t)t * B * 4 * H;
      ca.h_out = hiddens + ((size_t)t * NL + l) * B * H; ca.h_ld = H;
      ca.h_op = xl + (size_t)B * K + (l == 0 ? E : H); ca.hop_ld = K;                    // own recurrent slot of step t+1
      if (l < top) {                                                                       // input slot of the layer above, same t
        ca.h_op2 = w.X_x[l] + (size_t)t * B * 2 * H; ca.hop2_ld = 2 * H;
        ca.op2_drop = p_lay; ca.rng = rng; ca.site = SITE_LAYER0 + l + 1; ca.drop_base = (long long)t * B * H;
      }
      RN_TRY((cell::launch_fwd<T, T>(ca, st)));
    }
  }
  RN_TRY(gemm_full<T>(Xtop + (size_t)B * 2 * H + H, 2 * H, 0, w.Wout, H, 0, w.logits, w.Vld, p.out_b, L * B, V, H, 0, w.splitk, st));
  if (targets && ce_weight && ce_out) {
    loss::ce_fwd_kernel<<<L * B, loss::CE_THREADS, 0, st>>>(w.logits, w.Vld, targets, ce_weight, V, p_out, rng, SITE_LOGITS, w.lse, w.row_loss);
    RN_LAUNCH_OK();
    loss::sum_kernel<<<1, 1024, 0, st>>>(w.row_loss, L * B, ce_out, 1.f);
    RN_LAUNCH_OK();
  }
  return 0;
}

template <typename T>
static int backward_ml(const DecDesc& d, const recnet_decoder_tensors& p, const float* feats, const long long* tokens_in,
                       const long long* targets, const float* ce_weight, const unsigned long long* rng, void* ws, long long ws_bytes,
                       const float* g_ce, const float* g_hiddens, const recnet_decoder_tensors& g, cudaStream_t st) {
  RN_TRY(check(d));
  Ws<T> w = plan<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, L = d.L, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T, EMB = d.EMB, NL = w.NL, top = NL - 1;
  const float p_emb = d.train ? d.p_emb_drop : 0.f, p_out = d.train ? d.p_out_drop : 0.f, p_lay = d.train ? d.p_layer_drop : 0.f;
  const int LB = L * B;
  T* Xtop = w.X_x[top - 1];
  const T* Htop = Xtop + (size_t)B * 2 * H + H;                      // h^top_t rows, ld = 2H
  {
    ProfScope prof(KC_CE, LB, V, 1, st);
    loss::ce_bwd_kernel<T><<<LB, loss::CE_THREADS, 0, st>>>(w.logits, w.Vld, targets, ce_weight, w.lse, g_ce, V, w.Vp, p_out, rng,
                                                            SITE_LOGITS, w.dlogits, w.Vp);
  }
  RN_LAUNCH_OK();
  RN_TRY(gemm_full<T>(w.dlogits, w.Vp, 0, w.Wout, H, 1, w.dHext, H, nullptr, LB, H, V, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dlogits, w.Vp, 1, Htop, 2 * H, 1, g.out_w, H, nullptr, V, H, LB, 0, w.splitk, st));
  RN_TRY(misc::colsum<T>(w.dlogits, w.Vp, LB, V, g.out_b, 0, w.splitk, st));
  for (int t = L - 1; t >= 0; --t) {
    const bool last = (t == L - 1);
    for (int l = top; l >= 0; --l) {
      const int K = l == 0 ? w.KX : 2 * H;
      float* dXl = l == 0 ? w.dXp : w.dXp_x[l - 1];
      const GemmPlan pl = l == 0 ? w.pl_dx : w.pl_dx_x;
      cell::BwdArgs cb{};
      if (l == top) { cb.dh_ext = w.dHext + (size_t)t * B * H; cb.dh_ld = H; }
      cb.dh_ext2 = g_hiddens ? g_hiddens + ((size_t)t * NL + l) * B * H : nullptr; cb.dh2_ld = H;
      // own recurrent path: h-part of this layer's dgrad at step t+1
      cb.dXp = last ? nullptr : dXl; cb.n_p = pl.splits; cb.p_stride = (long long)B * K; cb.p_ld = K; cb.col0 = l == 0 ? E : H;
      if (l == top) {          // attention query of step t+1
        cb.dQp = last ? nullptr : w.dQp; cb.n_q = w.pl_dq.splits; cb.q_stride = (long long)B * H; cb.q_ld = H;
      } else {                 // input of the layer above at the SAME step (x-part of its dgrad), through the inter-layer dropout
        cb.dQp = w.dXp_x[l]; cb.n_q = w.pl_dx_x.splits; cb.q_stride = (long long)B * 2 * H; cb.q_ld = 2 * H;
        cb.q_drop = p_lay; cb.rng = rng; cb.q_site = SITE_LAYER0 + l + 1; cb.q_base = (long long)t * B * H;
      }
      cb.dc = l == 0 ? w.dc : w.dc_x[l - 1]; cb.first = last ? 1 : 0;
      cb.gates = (l == 0 ? w.gates : w.gates_x[l - 1]) + (size_t)t * B * 4 * H;
      const float* cl = l == 0 ? w.c : w.c_x[l - 1];
      cb.c_prev = cl + (size_t)t * B * H; cb.c_new = cl + (size_t)(t + 1) * B * H;
      cb.B = B; cb.H = H;
      T* dGl = (l == 0 ? w.dG : w.dG_x[l - 1]) + (size_t)t * B * 4 * H;
      cb.dG = dGl; cb.dg_ld = 4 * H;
      RN_TRY((cell::launch_bwd<T, T>(cb, st)));
      const T* Wl = l == 0 ? w.Wrec : w.Wrec_x[l - 1];
      RN_TRY(gemm_partials<T>(dGl, 4 * H, 0, Wl, K, 1, dXl, B, K, 4 * H, pl, st));
    }
    attn::BwdArgs ab{};
    ab.dXp = w.dXp; ab.n_p = w.pl_dx.splits; ab.p_stride = (long long)B * w.KX; ab.p_ld = w.KX;
    ab.V = w.feats; ab.v_bs = (long long)Tn * E; ab.v_ts = E;
    ab.Wh = w.Wh + (size_t)t * B * A; ab.Uv = w.Uv; ab.uv_bs = (long long)Tn * A; ab.uv_ts = A;
    ab.attn_b = p.attn_b; ab.attn_w = p.attn_w; ab.B = B; ab.Tn = Tn; ab.A = A; ab.D = E;
    ab.inv_T = d.softmax ? 1.f : 1.f / Tn; ab.alpha = d.softmax ? w.e + (size_t)t * B * Tn : nullptr;
    ab.dWh_out = w.dWh + (size_t)t * B * A; ab.dWh_op = w.dWh_op + (size_t)t * B * A; ab.dUv_acc = w.dUv;
    ab.uv_first = last ? 1 : 0; ab.dw_first = last ? 1 : 0; ab.dw_acc = w.dw_acc;
    RN_TRY((attn::launch_bwd<T, T>(ab, st)));
    if (t > 0) RN_TRY(gemm_partials<T>(w.dWh_op + (size_t)t * B * A, A, 0, w.Wa, H, 1, w.dQp, B, H, A, w.pl_dq, st));
  }
  // ---- weight gradients ----
  const long long ldih = EMB + E;
  RN_TRY(misc::colsum<T>(w.dG, 4 * H, LB, 4 * H, g.b_ih, 0, w.splitk, st));
  RN_CUDA_OK(cudaMemcpyAsync(g.b_hh, g.b_ih, (size_t)4 * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
  RN_TRY(gemm_full<T>(w.dG, 4 * H, 1, w.X, w.KX, 1, g.w_ih + EMB, ldih, nullptr, 4 * H, E, LB, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dG, 4 * H, 1, w.X + E, w.KX, 1, g.w_hh, H, nullptr, 4 * H, H, LB, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dG, 4 * H, 1, w.Xe, w.EMBp, 1, g.w_ih, ldih, nullptr, 4 * H, EMB, LB, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dG, 4 * H, 0, w.Wemb, w.EMBp, 1, w.dXe, w.EMBp, nullptr, LB, EMB, 4 * H, 0, w.splitk, st));
  RN_CUDA_OK(cudaMemsetAsync(g.embedding, 0, (size_t)V * EMB * sizeof(float), st));
  misc::embed_scatter_kernel<<<LB, 128, 0, st>>>(g.embedding, tokens_in, w.dXe, w.EMBp, LB, EMB, V, d.embedding_scale, p_emb, rng, SITE_EMB);
  RN_LAUNCH_OK();
  for (int l = 1; l < NL; ++l) {
    const T* dGl = w.dG_x[l - 1];
    const T* Xl = w.X_x[l - 1];
    RN_TRY(misc::colsum<T>(dGl, 4 * H, LB, 4 * H, g.b_ih_x[l - 1], 0, w.splitk, st));
    RN_CUDA_OK(cudaMemcpyAsync(g.b_hh_x[l - 1], g.b_ih_x[l - 1], (size_t)4 * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
    RN_TRY(gemm_full<T>(dGl, 4 * H, 1, Xl, 2 * H, 1, g.w_ih_x[l - 1], H, nullptr, 4 * H, H, LB, 0, w.splitk, st));
    RN_TRY(gemm_full<T>(dGl, 4 * H, 1, Xl + H, 2 * H, 1, g.w_hh_x[l - 1], H, nullptr, 4 * H, H, LB, 0, w.splitk, st));
  }
  RN_TRY(gemm_full<T>(w.dWh_op, A, 1, Xtop + H, 2 * H, 1, g.attn_W, H, nullptr, A, H, LB, 0, w.splitk, st));      // dW_a = dWh^T h^top_{t-1}
  RN_TRY(misc::cast_pad<T>(w.dUv, A, w.dUv_op, A, (long long)B * Tn, A, A, st));
  RN_TRY(gemm_full<T>(w.dUv_op, A, 1, w.feats, E, 1, g.attn_U, E, nullptr, A, E, B * Tn, 0, w.splitk, st));
  RN_TRY(misc::colsum<float>(w.dWh, A, LB, A, g.attn_b, 0, w.splitk, st));
  RN_TRY(misc::colsum<float>(w.dw_acc, A, B, A, g.attn_w, 0, w.splitk, st));
  return 0;
}
}  // namespace dec
