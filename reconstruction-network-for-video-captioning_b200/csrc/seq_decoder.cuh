// Decoder sequence driver: the whole teacher-forced loop of train.forward_decoder (train.py:17-75) over
// Decoder.forward (models/decoder.py:45-70), forward and BPTT, restructured for B200:
//   * U.v hoisted out of the loop (the reference recomputes it 31x, decoder.py:54)        -> 1 batched GEMM
//   * W_ih split into [W_emb | W_ctx]: the embedding half is time-batched (M = L*B)        -> 1 batched GEMM
//   * per step: [ctx_t ; h_{t-1}] @ [W_ctx | W_hh]^T as ONE K-concatenated tensor-core GEMM (no torch.cat,
//     decoder.py:64), split-K partials summed inside the fused cell kernel
//   * vocabulary projection batched over all steps (M = L*B), fused CE forward/backward over stacked logits
//   * BPTT mirrors it; all weight gradients are batched GEMMs over the stashed operands after the loop.
// Stacked (n_layers = NL > 1, LSTM only): models/decoder.py:36-40,66 with num_layers = NL.  Layer 0 is the step above (input
// [emb ; ctx]); layer l >= 1 consumes h^{l-1}_t (inter-layer dropout in train mode) and its own h^l_{t-1} as ONE K-concatenated GEMM
// over operand rows X_l[t] = [h^{l-1}_t ; h^l_{t-1}].  The attention query and the vocabulary projection use the TOP layer
// (decoder.py:51,68); `hiddens` returns every layer, (L, NL, B, H) (train.py:61-64).
#pragma once
#include "gru_cell.cuh"
#include "runtime.cuh"

namespace dec {
using namespace rt;

enum : unsigned { SITE_EMB = 1, SITE_LOGITS = 2, SITE_LAYER0 = 16 };   // dropout site of the input of layer l = SITE_LAYER0 + l
enum : unsigned { SITE_SAMPLE = 5 };                                     // Gumbel noise of the sampler (its own (seed, offset) pair)

template <typename T>
struct Ws {
  // geometry
  int EMBp, KX, Vp, Vld;
  int G;                             // gates per unit: 4 (LSTM) or 3 (GRU)
  GemmPlan pl_wh, pl_gate, pl_dx, pl_dq;
  GemmPlan pl_gx, pl_gh, pl_dxx, pl_dxh;   // GRU: x-part / h-part kept separate (n gate)
  // operand copies of the weights / inputs (rebuilt every forward: the optimiser changes the masters)
  T *Wemb, *Wrec, *U, *Wa, *Wout, *feats;
  // forward state kept for BPTT
  float* Uv; T* Xe; float* Gx; T* X; float* WhP; float* Wh; float* e; float* P; float* P2; T* gates; float* c;
  float *logits, *lse, *row_loss;
  // backward scratch
  T* dlogits; float* dHext; T* dG; T* dG2; float* dXp; float* dXp2; float* dQp; float* dWh; T* dWh_op; float* dUv; T* dUv_op; float* dw_acc;
  float* dc; float* dXe; float* splitk;
  int* err;                          // error flag (recnet_decoder_error_offset)
  // layers 1 .. NL-1 of a stacked decoder (index l-1): operand rows X_l[t] = [h^{l-1}_t ; h^l_{t-1}], K = 2H
  int NL;
  GemmPlan pl_gate_x, pl_dx_x;
  T* Wrec_x[RECNET_MAX_LAYERS - 1]; T* X_x[RECNET_MAX_LAYERS - 1]; T* gates_x[RECNET_MAX_LAYERS - 1]; float* c_x[RECNET_MAX_LAYERS - 1];
  T* dG_x[RECNET_MAX_LAYERS - 1]; float* dXp_x[RECNET_MAX_LAYERS - 1]; float* dc_x[RECNET_MAX_LAYERS - 1];
  size_t bytes;
};

template <typename T>
static Ws<T> plan(const recnet_decoder_desc& d, void* base) {
  Ws<T> w;
  const int B = d.B, L = d.L, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T;
  w.EMBp = round_up(d.EMB, Prec<T>::kpad);
  w.KX = E + H;
  w.Vp = round_up(V, 8);
  w.Vld = round_up(V, 4);
  w.pl_wh = plan_gemm<T>(B, A, H);
  w.pl_gate = plan_gemm<T>(B, 4 * H, w.KX);
  w.pl_dx = plan_gemm<T>(B, w.KX, 4 * H);
  w.pl_dq = plan_gemm<T>(B, H, A);
  w.G = d.cell == RECNET_CELL_GRU ? 3 : 4;
  w.pl_gx = plan_gemm<T>(B, 3 * H, E);
  w.pl_gh = plan_gemm<T>(B, 3 * H, H);
  w.pl_dxx = plan_gemm<T>(B, E, 3 * H);
  w.pl_dxh = plan_gemm<T>(B, H, 3 * H);
  const bool gru_ = d.cell == RECNET_CELL_GRU;
  Bump m(base);
  w.Wemb = m.take<T>((size_t)4 * H * w.EMBp);
  w.Wrec = m.take<T>((size_t)4 * H * w.KX);
  w.U = m.take<T>((size_t)A * E);
  w.Wa = m.take<T>((size_t)A * H);
  w.Wout = m.take<T>((size_t)V * H);
  w.feats = m.take<T>((size_t)B * Tn * E);
  w.Uv = m.take<float>((size_t)B * Tn * A);
  w.Xe = m.take<T>((size_t)L * B * w.EMBp);
  w.Gx = m.take<float>((size_t)L * B * 4 * H);
  w.X = m.take<T>((size_t)(L + 1) * B * w.KX);
  w.WhP = m.take<float>((size_t)w.pl_wh.splits * B * A);
  w.Wh = m.take<float>((size_t)L * B * A);
  w.e = m.take<float>((size_t)L * B * Tn);
  w.P = m.take<float>((size_t)(gru_ ? w.pl_gx.splits : w.pl_gate.splits) * B * 4 * H + (size_t)16 * B * 4 * H);
  w.P2 = m.take<float>(gru_ ? (size_t)w.pl_gh.splits * B * 3 * H : 1);
  w.gates = m.take<T>((size_t)L * B * 4 * H);
  w.c = m.take<float>((size_t)(L + 1) * B * H);
  w.logits = m.take<float>((size_t)L * B * w.Vld);
  w.lse = m.take<float>((size_t)L * B);
  w.row_loss = m.take<float>((size_t)L * B);
  w.dlogits = m.take<T>((size_t)L * B * w.Vp);
  w.dHext = m.take<float>((size_t)L * B * H);
  w.dG = m.take<T>((size_t)L * B * 4 * H);
  w.dXp = m.take<float>((size_t)(gru_ ? w.pl_dxx.splits : w.pl_dx.splits) * B * w.KX);
  w.dXp2 = m.take<float>(gru_ ? (size_t)w.pl_dxh.splits * B * H : 1);
  w.dG2 = m.take<T>(gru_ ? (size_t)L * B * 3 * H : 1);
  w.dQp = m.take<float>((size_t)w.pl_dq.splits * B * H);
  w.dWh = m.take<float>((size_t)L * B * A);
  w.dWh_op = m.take<T>((size_t)L * B * A);
  w.dUv = m.take<float>((size_t)B * Tn * A);
  w.dUv_op = m.take<T>((size_t)B * Tn * A);
  w.dw_acc = m.take<float>((size_t)B * A);
  w.dc = m.take<float>((size_t)B * H);
  w.dXe = m.take<float>((size_t)L * B * w.EMBp);
  w.splitk = m.take<float>(SPLITK_SCRATCH_FLOATS);
  w.err = m.take<int>(64);
  w.NL = d.n_layers < 1 ? 1 : d.n_layers;
  w.pl_gate_x = plan_gemm<T>(B, 4 * H, 2 * H);
  w.pl_dx_x = plan_gemm<T>(B, 2 * H, 4 * H);
  for (int l = 1; l < w.NL && l < RECNET_MAX_LAYERS; ++l) {
    w.Wrec_x[l - 1] = m.take<T>((size_t)4 * H * 2 * H);
    w.X_x[l - 1] = m.take<T>((size_t)(L + 1) * B * 2 * H);
    w.gates_x[l - 1] = m.take<T>((size_t)L * B * 4 * H);
    w.c_x[l - 1] = m.take<float>((size_t)(L + 1) * B * H);
    w.dG_x[l - 1] = m.take<T>((size_t)L * B * 4 * H);
    w.dXp_x[l - 1] = m.take<float>((size_t)w.pl_dx_x.splits * B * 2 * H);
    w.dc_x[l - 1] = m.take<float>((size_t)B * H);
  }
  w.bytes = m.off + 256;
  return w;
}

static inline int check(const recnet_decoder_desc& d) {
  if (d.B < 1 || d.T < 1 || d.L < 1 || d.V < 3 || d.EMB < 1 || d.T > attn::MAX_T) return RECNET_ERR_BAD_SHAPE;
  if (d.cell != RECNET_CELL_LSTM && d.cell != RECNET_CELL_GRU) return RECNET_ERR_UNSUPPORTED;
  if (d.n_layers > RECNET_MAX_LAYERS) return RECNET_ERR_UNSUPPORTED;
  if (d.n_layers > 1 && d.cell != RECNET_CELL_LSTM) return RECNET_ERR_UNSUPPORTED;      // stacked GRU: not built
  const int al = d.precision == RECNET_PREC_BF16 ? 8 : 4;
  if (d.E % al || d.H % al || d.A % 4) return RECNET_ERR_ALIGNMENT;
  return 0;
}

// Build the operand-typed copies of weights and features.
template <typename T>
static int prepare(const recnet_decoder_desc& d, const recnet_decoder_tensors& p, const float* feats, Ws<T>& w, cudaStream_t st) {
  const int H = d.H, E = d.E, A = d.A, V = d.V, EMB = d.EMB;
  const long long ldih = EMB + E;
  const int GH = w.G * H;
  RN_TRY(misc::cast_pad<T>(p.w_ih, ldih, w.Wemb, w.EMBp, GH, EMB, w.EMBp, st));
  RN_TRY(misc::cast_pad<T>(p.w_ih + EMB, ldih, w.Wrec, w.KX, GH, E, E, st));
  RN_TRY(misc::cast_pad<T>(p.w_hh, H, w.Wrec + E, w.KX, GH, H, H, st));
  RN_TRY(misc::cast_pad<T>(p.attn_U, E, w.U, E, A, E, E, st));
  RN_TRY(misc::cast_pad<T>(p.attn_W, H, w.Wa, H, A, H, H, st));
  RN_TRY(misc::cast_pad<T>(p.out_w, H, w.Wout, H, V, H, H, st));
  if (feats) RN_TRY(misc::cast_pad<T>(feats, E, w.feats, E, (long long)d.B * d.T, E, E, st));
  for (int l = 1; l < w.NL; ++l) {    // stacked layers: [W_ih | W_hh] of layer l side by side, K = 2H
    RN_TRY(misc::cast_pad<T>(p.w_ih_x[l - 1], H, w.Wrec_x[l - 1], 2 * H, 4 * H, H, H, st));
    RN_TRY(misc::cast_pad<T>(p.w_hh_x[l - 1], H, w.Wrec_x[l - 1] + H, 2 * H, 4 * H, H, H, st));
  }
  return 0;
}

// Where the top layer's h rows live: block t (B rows of ld *ld) holds h^top_{t-1}, block 0 the zero initial state.  The attention
// query, the vocabulary GEMMs and the attn_W gradient read from here.
template <typename T>
static const T* top_h(const recnet_decoder_desc& d, const Ws<T>& w, long long* ld) {
  if (w.NL == 1) { *ld = w.KX; return w.X + d.E; }
  *ld = 2 * d.H;
  return w.X_x[w.NL - 2] + d.H;
}

// one decoder step: attention -> gate GEMM -> layer-0 cell.  Pointer arguments are the row-0 addresses of step t; q_t (ld q_ld) holds
// the attention query h^top_{t-1}.  In a stack, up_t is layer 1's input slot X_1[t], written through the inter-layer dropout.
template <typename T>
static int step(const DecDesc& d, const recnet_decoder_tensors& p, Ws<T>& w, int t, const T* q_t, long long q_ld, const float* gx_t,
                T* x_t, T* x_next, float* Wh_t, float* e_t, T* gates_t, const float* c_prev, float* c_next, float* h_out, cudaStream_t st,
                T* up_t = nullptr, const unsigned long long* rng = nullptr) {
  const int B = d.B, H = d.H, E = d.E, A = d.A, Tn = d.T;
  int n_whp = 0;
  if (t > 0) {   // h_{-1} = 0 -> W h = 0, skip the GEMM
    RN_TRY(gemm_partials<T>(q_t, q_ld, 0, w.Wa, H, 0, w.WhP, B, A, H, w.pl_wh, st));
    n_whp = w.pl_wh.splits;
  }
  attn::FwdArgs fa{};
  fa.WhP = w.WhP; fa.n_whp = n_whp; fa.whp_stride = (long long)B * A;
  fa.Uv = w.Uv; fa.uv_bs = (long long)Tn * A; fa.uv_ts = A;
  fa.attn_b = p.attn_b; fa.attn_w = p.attn_w;
  fa.V = w.feats; fa.v_bs = (long long)Tn * E; fa.v_ts = E;
  fa.B = B; fa.Tn = Tn; fa.A = A; fa.D = E; fa.inv_T = d.softmax ? 1.f : 1.f / Tn; fa.normalize = d.softmax;
  fa.Wh_out = Wh_t; fa.e_out = e_t;
  fa.ctx_out = x_t; fa.ctx_ld = w.KX; fa.p_drop = 0.f;
  RN_TRY((attn::launch_fwd<T, T>(fa, st)));
  if (d.cell == RECNET_CELL_GRU) {
    // x-part: ctx_t @ W_ctx^T (K = E) ; h-part: h_{t-1} @ W_hh^T (K = H): same operand rows, same weight copy, two column ranges
    RN_TRY(gemm_partials<T>(x_t, w.KX, 0, w.Wrec, w.KX, 0, w.P, B, 3 * H, E, w.pl_gx, st));
    if (t > 0) RN_TRY(gemm_partials<T>(x_t + E, w.KX, 0, w.Wrec + E, w.KX, 0, w.P2, B, 3 * H, H, w.pl_gh, st));
    gru::FwdArgs ga{};
    ga.Px = w.P; ga.n_px = w.pl_gx.splits; ga.px_stride = (long long)B * 3 * H; ga.px_ld = 3 * H;
    ga.Ph = t > 0 ? w.P2 : nullptr; ga.n_ph = t > 0 ? w.pl_gh.splits : 0; ga.ph_stride = (long long)B * 3 * H; ga.ph_ld = 3 * H;
    ga.Gx = gx_t; ga.gx_ld = 3 * H; ga.b_ih = nullptr; ga.b_hh = p.b_hh;
    ga.h_prev = c_prev; ga.hp_ld = H; ga.B = B; ga.H = H;
    ga.stash = gates_t;
    ga.h_out = h_out; ga.h_ld = H;
    ga.h_op = x_next + E; ga.hop_ld = w.KX;
    return gru::launch_fwd<T, T>(ga, st);
  }
  RN_TRY(gemm_partials<T>(x_t, w.KX, 0, w.Wrec, w.KX, 0, w.P, B, 4 * H, w.KX, w.pl_gate, st));
  cell::FwdArgs ca{};
  ca.P = w.P; ca.n_p = w.pl_gate.splits; ca.p_stride = (long long)B * 4 * H; ca.p_ld = 4 * H;
  ca.Gx = gx_t; ca.gx_ld = 4 * H; ca.b1 = nullptr; ca.b2 = p.b_hh;
  ca.c_prev = c_prev; ca.B = B; ca.H = H;
  ca.gates_out = gates_t; ca.c_out = c_next;
  ca.h_out = h_out; ca.h_ld = H;
  ca.h_op = x_next + E; ca.hop_ld = w.KX; ca.h_op2 = nullptr;
  if (up_t) {
    ca.h_op2 = up_t; ca.hop2_ld = 2 * H;
    ca.op2_drop = d.train ? d.p_layer_drop : 0.f; ca.rng = rng; ca.site = SITE_LAYER0 + 1; ca.drop_base = (long long)t * B * H;
  }
  return cell::launch_fwd<T, T>(ca, st);
}

// layers 1 .. NL-1 of one stacked step (LSTM): per layer, the K-concatenated gate GEMM over its operand rows [h^{l-1}_t ; h^l_{t-1}]
// (block rd of X_x[l-1]) and the cell, which reads c^l_{t-1} from block rd of c_x[l-1] and writes c^l_t and h^l_t into block wr (h into
// the own recurrent slot, second half) and h^l_t into the input slot of the layer above (block rd of X_x[l], through the inter-layer
// dropout).  The sequence forward passes rd = t, wr = t + 1 and h_t = the (NL, B, H) rows of step t in `hiddens`, which also turns on
// the gate stash for BPTT; the decode loops ping-pong two blocks and pass h_t = nullptr (neither is kept).
template <typename T>
static int upper_layers(const DecDesc& d, const recnet_decoder_tensors& p, Ws<T>& w, int t, int rd, int wr, float* h_t, float p_lay,
                        const unsigned long long* rng, cudaStream_t st) {
  const int B = d.B, H = d.H, NL = w.NL;
  for (int l = 1; l < NL; ++l) {
    T* xl = w.X_x[l - 1] + (size_t)rd * B * 2 * H;
    RN_TRY(gemm_partials<T>(xl, 2 * H, 0, w.Wrec_x[l - 1], 2 * H, 0, w.P, B, 4 * H, 2 * H, w.pl_gate_x, st));
    cell::FwdArgs ca{};
    ca.P = w.P; ca.n_p = w.pl_gate_x.splits; ca.p_stride = (long long)B * 4 * H; ca.p_ld = 4 * H;
    ca.b1 = p.b_ih_x[l - 1]; ca.b2 = p.b_hh_x[l - 1];
    ca.c_prev = w.c_x[l - 1] + (size_t)rd * B * H; ca.c_out = w.c_x[l - 1] + (size_t)wr * B * H; ca.B = B; ca.H = H;
    ca.gates_out = h_t ? w.gates_x[l - 1] + (size_t)rd * B * 4 * H : nullptr;
    ca.h_out = h_t ? h_t + (size_t)l * B * H : nullptr; ca.h_ld = H;
    ca.h_op = w.X_x[l - 1] + (size_t)wr * B * 2 * H + H; ca.hop_ld = 2 * H;          // own recurrent slot of the next step
    if (l + 1 < NL) {                                                                   // input slot of the layer above, same t
      ca.h_op2 = w.X_x[l] + (size_t)rd * B * 2 * H; ca.hop2_ld = 2 * H;
      ca.op2_drop = p_lay; ca.rng = rng; ca.site = SITE_LAYER0 + l + 1; ca.drop_base = (long long)t * B * H;
    }
    RN_TRY((cell::launch_fwd<T, T>(ca, st)));
  }
  return 0;
}

template <typename T>
static int forward(const DecDesc& d, const recnet_decoder_tensors& p, const float* feats, const long long* tokens_in,
                   const long long* targets, const float* ce_weight, const unsigned long long* rng, void* ws, long long ws_bytes,
                   float* hiddens, float* ce_out, cudaStream_t st) {
  RN_TRY(check(d));
  Ws<T> w = plan<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, L = d.L, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T, NL = w.NL;
  const float p_emb = d.train ? d.p_emb_drop : 0.f, p_out = d.train ? d.p_out_drop : 0.f, p_lay = d.train ? d.p_layer_drop : 0.f;
  RN_TRY(prepare<T>(d, p, feats, w, st));
  long long ldq;
  const T* Htop = top_h(d, w, &ldq);
  // hoisted projections
  RN_TRY(gemm_full<T>(w.feats, E, 0, w.U, E, 0, w.Uv, A, nullptr, B * Tn, A, E, 0, w.splitk, st));
  misc::embed_gather_kernel<T><<<L * B, 128, 0, st>>>(p.embedding, tokens_in, w.Xe, w.EMBp, L * B, d.EMB, w.EMBp, V,
                                                      d.embedding_scale, p_emb, rng, SITE_EMB);
  RN_LAUNCH_OK();
  const int GH = w.G * H;
  const bool is_gru = d.cell == RECNET_CELL_GRU;
  RN_TRY(gemm_full<T>(w.Xe, w.EMBp, 0, w.Wemb, w.EMBp, 0, w.Gx, GH, p.b_ih, L * B, GH, w.EMBp, 0, w.splitk, st));
  // initial state: h_{-1} = 0 (operand slot of X[0]), c_{-1} = 0
  RN_CUDA_OK(cudaMemsetAsync(w.X, 0, (size_t)B * w.KX * sizeof(T), st));
  RN_CUDA_OK(cudaMemsetAsync(w.c, 0, (size_t)B * H * sizeof(float), st));
  // time loop: one kernel per phase
  RN_CUDA_OK(cudaMemsetAsync(w.err, 0, sizeof(int), st));
  for (int l = 1; l < NL; ++l) {
    RN_CUDA_OK(cudaMemsetAsync(w.X_x[l - 1], 0, (size_t)B * 2 * H * sizeof(T), st));
    RN_CUDA_OK(cudaMemsetAsync(w.c_x[l - 1], 0, (size_t)B * H * sizeof(float), st));
  }
  for (int t = 0; t < L; ++t) {
    T* x_t = w.X + (size_t)t * B * w.KX;
    // LSTM: c_{t-1} -> c_t live in w.c; GRU: the fp32 state is h itself (previous row of `hiddens`, zeros = w.c at t = 0)
    const float* s_prev = is_gru ? (t == 0 ? w.c : hiddens + (size_t)(t - 1) * B * H) : w.c + (size_t)t * B * H;
    RN_TRY(step<T>(d, p, w, t, Htop + (size_t)t * B * ldq, ldq, w.Gx + (size_t)t * B * GH, x_t, x_t + (size_t)B * w.KX,
                   w.Wh + (size_t)t * B * A, w.e + (size_t)t * B * Tn, w.gates + (size_t)t * B * 4 * H, s_prev,
                   w.c + (size_t)(t + 1) * B * H, hiddens + (size_t)t * NL * B * H, st,
                   NL > 1 ? w.X_x[0] + (size_t)t * B * 2 * H : nullptr, rng));
    RN_TRY(upper_layers<T>(d, p, w, t, t, t + 1, hiddens + (size_t)t * NL * B * H, p_lay, rng, st));
  }
  // vocabulary projection over all steps, then the masked CE (train.py:54-60,68)
  RN_TRY(gemm_full<T>(Htop + (size_t)B * ldq, ldq, 0, w.Wout, H, 0, w.logits, w.Vld, p.out_b, L * B, V, H, 0, w.splitk, st));
  if (targets && ce_weight && ce_out) {
    ProfScope prof(KC_CE, L * B, V, 0, st);
    loss::ce_fwd_kernel<<<L * B, loss::CE_THREADS, 0, st>>>(w.logits, w.Vld, targets, ce_weight, V, p_out, rng, SITE_LOGITS,
                                                            w.lse, w.row_loss);
    RN_LAUNCH_OK();
    loss::sum_kernel<<<1, 1024, 0, st>>>(w.row_loss, L * B, ce_out, 1.f);
    RN_LAUNCH_OK();
  }
  return 0;
}

template <typename T>
static int backward(const DecDesc& d, const recnet_decoder_tensors& p, const float* feats, const long long* tokens_in,
                    const long long* targets, const float* ce_weight, const unsigned long long* rng, void* ws, long long ws_bytes,
                    const float* g_ce, const float* g_hiddens, const float* hiddens_fp32, const recnet_decoder_tensors& g,
                    cudaStream_t st) {
  RN_TRY(check(d));
  Ws<T> w = plan<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, L = d.L, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T, EMB = d.EMB, NL = w.NL, top = NL - 1;
  const float p_emb = d.train ? d.p_emb_drop : 0.f, p_out = d.train ? d.p_out_drop : 0.f, p_lay = d.train ? d.p_layer_drop : 0.f;
  const int LB = L * B;
  long long ldq;
  const T* Htop = top_h(d, w, &ldq);
  // ---- CE backward and the vocabulary projection --------------------------------------------------------
  {
    ProfScope prof(KC_CE, LB, V, 1, st);
    loss::ce_bwd_kernel<T><<<LB, loss::CE_THREADS, 0, st>>>(w.logits, w.Vld, targets, ce_weight, w.lse, g_ce, V, w.Vp, p_out, rng,
                                                            SITE_LOGITS, w.dlogits, w.Vp);
  }
  RN_LAUNCH_OK();
  RN_TRY(gemm_full<T>(w.dlogits, w.Vp, 0, w.Wout, H, 1, w.dHext, H, nullptr, LB, H, V, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dlogits, w.Vp, 1, Htop + (size_t)B * ldq, ldq, 1, g.out_w, H, nullptr, V, H, LB, 0, w.splitk, st));
  RN_TRY(misc::colsum<T>(w.dlogits, w.Vp, LB, V, g.out_b, 0, w.splitk, st));
  // ---- BPTT: one kernel per phase -------------------------------------------------------------------------
  const bool is_gru = d.cell == RECNET_CELL_GRU;
  const int GH = w.G * H;
  for (int t = L - 1; t >= 0; --t) {
    const bool last = (t == L - 1);
    const size_t r = (size_t)t * B;                // first (t, b) row of step t
    if (is_gru) {
      float* dXx = w.dXp;                          // x-part dgrad partials [splits][B, E]
      float* dXh = w.dXp2;                         // h-part dgrad partials [splits][B, H]
      gru::BwdArgs gb{};
      gb.dh_ext = w.dHext + r * H; gb.dh_ld = H;
      gb.dh_ext2 = g_hiddens ? g_hiddens + r * H : nullptr; gb.dh2_ld = H;
      gb.dHp = last ? nullptr : dXh; gb.n_p = w.pl_dxh.splits; gb.p_stride = (long long)B * H; gb.p_ld = H;
      gb.dQp = last ? nullptr : w.dQp; gb.n_q = w.pl_dq.splits; gb.q_stride = (long long)B * H; gb.q_ld = H;
      gb.carry = w.dc; gb.first = last ? 1 : 0;
      gb.stash = w.gates + r * 4 * H;
      gb.h_prev = t == 0 ? w.c : hiddens_fp32 + (size_t)(t - 1) * B * H; gb.hp_ld = H;
      gb.B = B; gb.H = H; gb.dGi = w.dG + r * 3 * H; gb.dGh = w.dG2 + r * 3 * H; gb.dg_ld = 3 * H;
      RN_TRY((gru::launch_bwd<T, T>(gb, st)));
      RN_TRY(gemm_partials<T>(w.dG + r * 3 * H, 3 * H, 0, w.Wrec, w.KX, 1, dXx, B, E, 3 * H, w.pl_dxx, st));           // dctx = dGi @ W_ctx
      if (t > 0) RN_TRY(gemm_partials<T>(w.dG2 + r * 3 * H, 3 * H, 0, w.Wrec + E, w.KX, 1, dXh, B, H, 3 * H, w.pl_dxh, st));  // dh += dGh @ W_hh
      attn::BwdArgs ab{};
      ab.dXp = dXx; ab.n_p = w.pl_dxx.splits; ab.p_stride = (long long)B * E; ab.p_ld = E;
      ab.V = w.feats; ab.v_bs = (long long)Tn * E; ab.v_ts = E;
      ab.Wh = w.Wh + r * A; ab.Uv = w.Uv; ab.uv_bs = (long long)Tn * A; ab.uv_ts = A;
      ab.attn_b = p.attn_b; ab.attn_w = p.attn_w; ab.B = B; ab.Tn = Tn; ab.A = A; ab.D = E; ab.inv_T = d.softmax ? 1.f : 1.f / Tn;
      ab.dWh_out = w.dWh + r * A; ab.dWh_op = w.dWh_op + r * A; ab.dUv_acc = w.dUv;
      ab.uv_first = last ? 1 : 0; ab.dw_first = last ? 1 : 0; ab.dw_acc = w.dw_acc;
      ab.dctx_out = nullptr; ab.de_out = nullptr; ab.p_drop = 0.f; ab.alpha = d.softmax ? w.e + r * Tn : nullptr;
      RN_TRY((attn::launch_bwd<T, T>(ab, st)));
      if (t > 0) RN_TRY(gemm_partials<T>(w.dWh_op + r * A, A, 0, w.Wa, H, 1, w.dQp, B, H, A, w.pl_dq, st));
      continue;
    }
    for (int l = top; l >= 0; --l) {     // operand rows: [ctx ; h_{t-1}] for layer 0, [h^{l-1}_t ; h^l_{t-1}] above
      const int K = l == 0 ? w.KX : 2 * H;
      const GemmPlan pl = l == 0 ? w.pl_dx : w.pl_dx_x;
      float* dXl = l == 0 ? w.dXp : w.dXp_x[l - 1];
      T* dGl = (l == 0 ? w.dG : w.dG_x[l - 1]) + r * 4 * H;
      const float* cl = l == 0 ? w.c : w.c_x[l - 1];
      cell::BwdArgs cb{};
      if (l == top) { cb.dh_ext = w.dHext + r * H; cb.dh_ld = H; }
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
      cb.gates = (l == 0 ? w.gates : w.gates_x[l - 1]) + r * 4 * H;
      cb.c_prev = cl + r * H; cb.c_new = cl + (size_t)(t + 1) * B * H;
      cb.B = B; cb.H = H; cb.dG = dGl; cb.dg_ld = 4 * H;
      RN_TRY((cell::launch_bwd<T, T>(cb, st)));
      // d[x ; h_{t-1}] = dG_t @ W_rec of layer l ([W_ctx | W_hh] for layer 0)
      RN_TRY(gemm_partials<T>(dGl, 4 * H, 0, l == 0 ? w.Wrec : w.Wrec_x[l - 1], K, 1, dXl, B, K, 4 * H, pl, st));
    }
    attn::BwdArgs ab{};
    ab.dXp = w.dXp; ab.n_p = w.pl_dx.splits; ab.p_stride = (long long)B * w.KX; ab.p_ld = w.KX;
    ab.V = w.feats; ab.v_bs = (long long)Tn * E; ab.v_ts = E;
    ab.Wh = w.Wh + r * A; ab.Uv = w.Uv; ab.uv_bs = (long long)Tn * A; ab.uv_ts = A;
    ab.attn_b = p.attn_b; ab.attn_w = p.attn_w; ab.B = B; ab.Tn = Tn; ab.A = A; ab.D = E; ab.inv_T = d.softmax ? 1.f : 1.f / Tn;
    ab.dWh_out = w.dWh + r * A; ab.dWh_op = w.dWh_op + r * A; ab.dUv_acc = w.dUv;
    ab.uv_first = last ? 1 : 0; ab.dw_first = last ? 1 : 0; ab.dw_acc = w.dw_acc;
    ab.dctx_out = nullptr; ab.de_out = nullptr; ab.p_drop = 0.f; ab.alpha = d.softmax ? w.e + r * Tn : nullptr;
    RN_TRY((attn::launch_bwd<T, T>(ab, st)));
    // attention-query path into h_{t-1}: dWh_t @ attn_W, consumed (as split-K partials) by the next cell backward
    if (t > 0) RN_TRY(gemm_partials<T>(w.dWh_op + r * A, A, 0, w.Wa, H, 1, w.dQp, B, H, A, w.pl_dq, st));
  }
  // ---- batched weight gradients over the stashed operands ----------------------------------------------------
  const long long ldih = EMB + E;
  // LSTM: one gate-gradient matrix dG [LB,4H]; GRU: dGi (input side) in w.dG and dGh (hidden side, n column scaled by r) in w.dG2
  const T* dGh = is_gru ? w.dG2 : w.dG;
  RN_TRY(misc::colsum<T>(w.dG, GH, LB, GH, g.b_ih, 0, w.splitk, st));
  if (is_gru) { RN_TRY(misc::colsum<T>(dGh, GH, LB, GH, g.b_hh, 0, w.splitk, st)); }
  else RN_CUDA_OK(cudaMemcpyAsync(g.b_hh, g.b_ih, (size_t)GH * sizeof(float), cudaMemcpyDeviceToDevice, st));
  RN_TRY(gemm_full<T>(w.dG, GH, 1, w.X, w.KX, 1, g.w_ih + EMB, ldih, nullptr, GH, E, LB, 0, w.splitk, st));            // dW_ctx
  RN_TRY(gemm_full<T>(dGh, GH, 1, w.X + E, w.KX, 1, g.w_hh, H, nullptr, GH, H, LB, 0, w.splitk, st));                   // dW_hh
  RN_TRY(gemm_full<T>(w.dG, GH, 1, w.Xe, w.EMBp, 1, g.w_ih, ldih, nullptr, GH, EMB, LB, 0, w.splitk, st));              // dW_emb
  RN_TRY(gemm_full<T>(w.dG, GH, 0, w.Wemb, w.EMBp, 1, w.dXe, w.EMBp, nullptr, LB, EMB, GH, 0, w.splitk, st));           // dXe
  RN_CUDA_OK(cudaMemsetAsync(g.embedding, 0, (size_t)V * EMB * sizeof(float), st));
  misc::embed_scatter_kernel<<<LB, 128, 0, st>>>(g.embedding, tokens_in, w.dXe, w.EMBp, LB, EMB, V, d.embedding_scale, p_emb, rng,
                                                 SITE_EMB);
  RN_LAUNCH_OK();
  for (int l = 1; l < NL; ++l) {
    const T* dGl = w.dG_x[l - 1];
    const T* Xl = w.X_x[l - 1];
    RN_TRY(misc::colsum<T>(dGl, 4 * H, LB, 4 * H, g.b_ih_x[l - 1], 0, w.splitk, st));
    RN_CUDA_OK(cudaMemcpyAsync(g.b_hh_x[l - 1], g.b_ih_x[l - 1], (size_t)4 * H * sizeof(float), cudaMemcpyDeviceToDevice, st));
    RN_TRY(gemm_full<T>(dGl, 4 * H, 1, Xl, 2 * H, 1, g.w_ih_x[l - 1], H, nullptr, 4 * H, H, LB, 0, w.splitk, st));
    RN_TRY(gemm_full<T>(dGl, 4 * H, 1, Xl + H, 2 * H, 1, g.w_hh_x[l - 1], H, nullptr, 4 * H, H, LB, 0, w.splitk, st));
  }
  // attention parameters
  RN_TRY(gemm_full<T>(w.dWh_op, A, 1, Htop, ldq, 1, g.attn_W, H, nullptr, A, H, LB, 0, w.splitk, st));                 // dW_a = dWh^T h^top_{t-1}
  RN_TRY(misc::cast_pad<T>(w.dUv, A, w.dUv_op, A, (long long)B * Tn, A, A, st));
  RN_TRY(gemm_full<T>(w.dUv_op, A, 1, w.feats, E, 1, g.attn_U, E, nullptr, A, E, B * Tn, 0, w.splitk, st));             // dU = dUv^T v
  RN_TRY(misc::colsum<float>(w.dWh, A, LB, A, g.attn_b, 0, w.splitk, st));
  RN_TRY(misc::colsum<float>(w.dw_acc, A, B, A, g.attn_w, 0, w.splitk, st));
  return 0;
}

// ---- decoding: greedy, beam search and sampling as device loops ------------------------------------------------------------------
// One butterfly step (lane distance o) of a warp's arg-max over (value, index) pairs: the larger value wins, the lower index on ties
// (like topk(1)).  *carry, if given, moves with the winning pair.
__device__ __forceinline__ void argmax_shfl(float& best, int& bi, int o, float* carry = nullptr) {
  const float ob = __shfl_xor_sync(0xffffffffu, best, o);
  const float oc = carry ? __shfl_xor_sync(0xffffffffu, *carry, o) : 0.f;
  const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
  if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; if (carry) *carry = oc; }
}

// greedy (eval.py:19-33): argmax over the vocabulary (lowest index wins ties), fed back as the next token.
__global__ void argmax_feedback_kernel(const float* __restrict__ logits, long long ld, int V, long long* __restrict__ ids_out,
                                       long long* __restrict__ next_tok, int* __restrict__ nonpad_count) {
  __shared__ float sv[32];
  __shared__ int si[32];
  const int b = blockIdx.x;
  const float* z = logits + (long long)b * ld;
  float best = -INFINITY; int bi = 0x7fffffff;
  for (int v = threadIdx.x; v < V; v += blockDim.x) {
    const float x = z[v];
    if (x > best || (x == best && v < bi)) { best = x; bi = v; }
  }
  for (int o = 16; o > 0; o >>= 1) argmax_shfl(best, bi, o);
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if (lane == 0) { sv[wp] = best; si[wp] = bi; }
  __syncthreads();
  if (wp == 0) {
    best = lane < nw ? sv[lane] : -INFINITY; bi = lane < nw ? si[lane] : 0x7fffffff;
    for (int o = 16; o > 0; o >>= 1) argmax_shfl(best, bi, o);
    if (lane == 0) {
      ids_out[b] = bi; next_tok[b] = bi;
      if (bi != 0) atomicAdd(nonpad_count, 1);
    }
  }
}
// n_steps = first step (1-based) after which every fed-back token was <PAD> (eval.py:30), else max_steps
__global__ void greedy_finalize_kernel(const int* __restrict__ nonpad, int max_steps, int* __restrict__ n_steps) {
  int n = max_steps;
  for (int t = 0; t < max_steps; ++t) if (nonpad[t] == 0) { n = t + 1; break; }
  *n_steps = n;
}
__global__ void fill_tokens_kernel(long long* tok, int n, long long v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) tok[i] = v;
}

// ---- beam search (eval.beam_search, eval.py:36-120) -----------------------------------------------------------------------------
// Rows of every per-step tensor are (beam k, sample b) -> k * B0 + b; the caller passes the features tiled K times.  Per step: the
// decoder step on all K * B0 rows (same kernels as greedy), then ONE selection kernel per sample -- scores log(sigmoid(logit)) +
// cum / len^0.7 (eval.py:53-61: the running score is divided by the length at EVERY step; len = position of the last <EOS> + 1 once
// the beam has emitted one, else t + 1), top-K over the K_cur * V candidates, sequence / <EOS> / score bookkeeping -- and one gather
// kernel that moves the recurrent state of the source beams into place.  The loop freezes on the device once every fed-back token of a
// step is <PAD> (eval.py:116); the host never reads anything back until the end.
constexpr int BEAM_MAX_K = 8;
constexpr int BEAM_THREADS = 256;

__global__ void beam_select_kernel(const float* __restrict__ logits, long long ld, int V, int B0, int K, int t, int max_steps, long long eos,
                                   const float* __restrict__ cum_in, float* __restrict__ cum_out, const int* __restrict__ eos_in,
                                   int* __restrict__ eos_out, const int* __restrict__ seq_in, int* __restrict__ seq_out,
                                   long long* __restrict__ tok_out, int* __restrict__ src_out, int* __restrict__ nonpad) {
  if (t > 0 && nonpad[t - 1] == 0) return;                  // frozen: every token fed back at the previous step was <PAD>
  __shared__ float sv[BEAM_THREADS / 32];
  __shared__ int si[BEAM_THREADS / 32];
  __shared__ int chosen[BEAM_MAX_K];
  __shared__ float base[BEAM_MAX_K];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int Kc = t == 0 ? 1 : K;                            // one live beam before the first expansion
  if (tid < Kc) {
    const int le = eos_in[b * K + tid];
    const float len = le >= 0 ? (float)(le + 1) : (float)(t + 1);
    base[tid] = cum_in[tid * B0 + b] / powf(len, 0.7f);
  }
  __syncthreads();
  const int total = Kc * V;
  int n_nonpad = 0;
  for (int k = 0; k < K; ++k) {
    float best = -INFINITY; int bi = 0x7fffffff;
    for (int f = tid; f < total; f += BEAM_THREADS) {
      bool taken = false;
      for (int q = 0; q < k; ++q) taken |= (chosen[q] == f);
      if (taken) continue;
      const int i = f / V, v = f - i * V;
      const float x = logits[(long long)(i * B0 + b) * ld + v];
      const float sc = logf(1.f / (1.f + expf(-x))) + base[i];
      if (sc > best || (sc == best && f < bi)) { best = sc; bi = f; }
    }
    for (int o = 16; o > 0; o >>= 1) argmax_shfl(best, bi, o);
    if (lane == 0) { sv[warp] = best; si[warp] = bi; }
    __syncthreads();
    if (warp == 0) {
      best = lane < BEAM_THREADS / 32 ? sv[lane] : -INFINITY; bi = lane < BEAM_THREADS / 32 ? si[lane] : 0x7fffffff;
      for (int o = 16; o > 0; o >>= 1) argmax_shfl(best, bi, o);
      if (lane == 0) {
        chosen[k] = bi;
        const int i = bi / V, v = bi - i * V;
        tok_out[k * B0 + b] = v;
        src_out[b * K + k] = i;
        cum_out[k * B0 + b] = best;
        eos_out[b * K + k] = (v == (int)eos) ? t : eos_in[b * K + i];
        if (v != 0) ++n_nonpad;
      }
    }
    __syncthreads();
  }
  // sequences: beam k continues beam src[k]
  for (int x = tid; x < K * (t + 1); x += BEAM_THREADS) {
    const int k = x / (t + 1), pos = x - k * (t + 1);
    const int f = chosen[k], i = f / V, v = f - i * V;
    seq_out[(b * K + k) * max_steps + pos] = pos < t ? seq_in[(b * K + i) * max_steps + pos] : v;
  }
  if (tid == 0 && n_nonpad) atomicAdd(nonpad + t, n_nonpad);
}

// recurrent state of row (k, b) <- state of row (src[b][k], b), every layer in one launch: layer 0's h rows (ld KX) and c, layer l's
// h (second half of the X_x[l-1] rows, ld 2H) and c_x[l-1].  The input-slot halves need no gather: every step rewrites them before it
// reads them.
template <typename T>
struct BeamStateRows {
  const T* h_src[RECNET_MAX_LAYERS]; T* h_dst[RECNET_MAX_LAYERS]; long long ld[RECNET_MAX_LAYERS];
  const float* c_src[RECNET_MAX_LAYERS]; float* c_dst[RECNET_MAX_LAYERS];
  int n;
};
template <typename T>
__global__ void beam_gather_layers_kernel(BeamStateRows<T> s, int H, int B0, int K, const int* __restrict__ src,
                                          const int* __restrict__ nonpad, int t) {
  if (t > 0 && nonpad[t - 1] == 0) return;                  // frozen (see beam_select_kernel)
  const int row = blockIdx.x, k = row / B0, b = row - k * B0;
  const int srow = src[b * K + k] * B0 + b;
#pragma unroll
  for (int l = 0; l < RECNET_MAX_LAYERS; ++l) {
    if (l >= s.n) break;
    for (int j = threadIdx.x; j < H; j += blockDim.x) {
      s.h_dst[l][(long long)row * s.ld[l] + j] = s.h_src[l][(long long)srow * s.ld[l] + j];
      s.c_dst[l][(long long)row * H + j] = s.c_src[l][(long long)srow * H + j];
    }
  }
}
__global__ void beam_finalize_kernel(const int* __restrict__ nonpad, int max_steps, int B0, int K, const int* __restrict__ seq0,
                                     const int* __restrict__ seq1, long long* __restrict__ out, int* __restrict__ n_steps) {
  int n = max_steps;
  for (int t = 0; t < max_steps; ++t) if (nonpad[t] == 0) { n = t + 1; break; }
  const int* seq = (n & 1) ? seq1 : seq0;                   // step t wrote buffer (t + 1) & 1; the last executed step is n - 1
  for (int x = threadIdx.x; x < B0 * max_steps; x += blockDim.x) {
    const int b = x / max_steps, pos = x - b * max_steps;
    out[x] = pos < n ? seq[(b * K) * max_steps + pos] : -1;   // top-1 beam (eval.py:118-119)
  }
  if (threadIdx.x == 0) *n_steps = n;
}
__global__ void beam_init_kernel(float* cum, int* eos, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { cum[i] = 0.f; eos[i] = -1; }                  // log(1.) ; no <EOS> yet
}

// ---- sampling (Gumbel-max): stochastic decoding and the sampling half of self-critical training ---------------------------------
// Per step: the decoder step on all rows (the kernels of greedy, plus the training-mode dropout masks when desc.train is set), then
// ONE selection kernel that draws a token per row from softmax(z' / tau) by Gumbel-max, z' = the logits after their dropout.  Every
// dropout mask is drawn at the element index the sequence forward (dec::forward) uses for row t * B + row, so a teacher-forced pass
// over the sampled tokens with the same dropout pair differentiates the logits the sampler drew from.  A row finishes once it emits
// <EOS> or <PAD>; after that it emits and feeds back <PAD> with log-prob 0, so a row of samples has the shape of a `targets` column.
constexpr int SAMPLE_THREADS = 256;

// -log(u) for u = ((w >> 8) + 0.5) 2^-24 in (0, 1), without rounding u itself: for u >= 1/2, 1 - u is exact in fp32 but u is not
// (u = 1 - 2^-25 would round to 1 and make the Gumbel noise -log(-log u) infinite).
__device__ __forceinline__ float neg_log_uniform(uint32_t w) {
  const uint32_t k = w >> 8;
  if (k < (1u << 23)) return -logf(((float)k + 0.5f) * (1.0f / 16777216.0f));
  return -log1pf(-((float)((1u << 24) - 1u - k) + 0.5f) * (1.0f / 16777216.0f));
}
// (max, sum exp(x - max)) of a union of two parts
__device__ __forceinline__ void lse_merge(float& m, float& s, float om, float os) {
  const float M = fmaxf(m, om);
  if (M == -INFINITY) return;
  s = s * expf(m - M) + os * expf(om - M);
  m = M;
}
__device__ __forceinline__ void sample_reduce_step(float& best, int& bi, float& bx, float& m, float& s, int o) {
  argmax_shfl(best, bi, o, &bx);
  const float om = __shfl_xor_sync(0xffffffffu, m, o), os = __shfl_xor_sync(0xffffffffu, s, o);
  lse_merge(m, s, om, os);
}

// One CTA per row, one pass over its V logits: training-mode dropout (site SITE_LOGITS), / tau, + Gumbel noise (site SITE_SAMPLE of the
// `noise` pair), both at element (t * B + row) * V + v with one Philox call per 4 elements; arg-max of the noisy value (lowest index
// wins ties) and, in the same pass, the running max / sum-exp of z' / tau for log softmax(z' / tau)[chosen].  live[t] counts the rows
// still unfinished after step t; once it is 0 the remaining steps change nothing.
__global__ void __launch_bounds__(SAMPLE_THREADS) sample_select_kernel(
    const float* __restrict__ logits, long long ld, int V, int B, int t, float tau, long long eos, float p_drop,
    const unsigned long long* __restrict__ rng, const unsigned long long* __restrict__ noise, long long* __restrict__ ids_t,
    float* __restrict__ logp_t, long long* __restrict__ tok, int* __restrict__ finished, int* __restrict__ lengths,
    int* __restrict__ live) {
  if (t > 0 && live[t - 1] == 0) return;                     // frozen: every row has finished
  const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (finished[row]) {                                       // ids / logp of this step stay 0 (cleared by the driver)
    if (tid == 0) tok[row] = 0;
    return;
  }
  __shared__ float sb[SAMPLE_THREADS / 32], sx[SAMPLE_THREADS / 32], sm[SAMPLE_THREADS / 32], ss[SAMPLE_THREADS / 32];
  __shared__ int si[SAMPLE_THREADS / 32];
  const float* z = logits + (long long)row * ld;
  const long long base = ((long long)t * B + row) * V;
  const long long q0 = base >> 2, nq = ((base + V - 1) >> 2) - q0 + 1;
  const bool drop = p_drop > 0.f;
  const Philox dph(drop ? rng[0] : 0ull), nph(noise[0]);
  const unsigned long long dstream = drop ? (rng[1] << 8) | SITE_LOGITS : 0ull, nstream = (noise[1] << 8) | SITE_SAMPLE;
  const float keep = 1.f / (1.f - p_drop);
  float best = -INFINITY, bx = 0.f, m = -INFINITY, s = 0.f;
  int bi = 0x7fffffff;
  for (long long q = tid; q < nq; q += SAMPLE_THREADS) {
    const unsigned long long ctr = (unsigned long long)(q0 + q);
    const uint4 n4 = nph(ctr, nstream);
    const uint4 d4 = drop ? dph(ctr, dstream) : make_uint4(0u, 0u, 0u, 0u);
    const uint32_t nw[4] = {n4.x, n4.y, n4.z, n4.w}, dw[4] = {d4.x, d4.y, d4.z, d4.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long v = 4 * (q0 + q) + j - base;
      if (v < 0 || v >= V) continue;
      float x = z[v];
      if (drop) x *= ((float)(dw[j] >> 8) * (1.0f / 16777216.0f) >= p_drop) ? keep : 0.f;
      x = x / tau;
      const float y = x - logf(neg_log_uniform(nw[j]));
      if (y > best) { best = y; bi = (int)v; bx = x; }      // v grows within a thread: strict > keeps the lowest index
      if (x > m) { s = s * expf(m - x) + 1.f; m = x; } else { s += expf(x - m); }
    }
  }
  for (int o = 16; o > 0; o >>= 1) sample_reduce_step(best, bi, bx, m, s, o);
  if (lane == 0) { sb[warp] = best; si[warp] = bi; sx[warp] = bx; sm[warp] = m; ss[warp] = s; }
  __syncthreads();
  if (warp) return;
  const bool ok = lane < SAMPLE_THREADS / 32;
  best = ok ? sb[lane] : -INFINITY; bi = ok ? si[lane] : 0x7fffffff; bx = ok ? sx[lane] : 0.f;
  m = ok ? sm[lane] : -INFINITY; s = ok ? ss[lane] : 0.f;
  for (int o = 16; o > 0; o >>= 1) sample_reduce_step(best, bi, bx, m, s, o);
  if (lane == 0) {
    ids_t[row] = bi;
    logp_t[row] = bx - (m + logf(s));
    tok[row] = bi;
    if (bi == eos || bi == 0) { finished[row] = 1; lengths[row] = t + 1; }
    else atomicAdd(live + t, 1);
  }
}
__global__ void sample_init_kernel(long long* tok, int* finished, int* lengths, int n, int max_steps) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { tok[i] = 1; finished[i] = 0; lengths[i] = max_steps; }    // <SOS>; a row that never finishes has max_steps tokens
}

// ---- the decode loop ------------------------------------------------------------------------------------------------------------
enum class DecodeMode { GREEDY, BEAM, SAMPLE };

// Workspace of a decode call: the sequence plan at L = 1 (X and c hold the two state blocks a step reads and writes), then the fed-back
// tokens, the per-step counts of non-<PAD> tokens (of unfinished rows when sampling) and the h rows nobody reads; beam search adds its
// scores, <EOS> positions and sequences (two of each: step t reads t & 1, writes (t + 1) & 1) and the source beams, sampling the
// rows' finished flags.
template <typename T>
struct DecodeWs {
  Ws<T> w; long long* tok; int* nonpad; float* h_scratch;
  float* cum[2]; int* eos[2]; int* seq[2]; int* src;       // beam search
  int* finished;                                            // sampling
  size_t bytes;
};
template <typename T>
static DecodeWs<T> plan_decode(const recnet_decoder_desc& d, void* base, DecodeMode mode, int max_steps) {
  DecodeWs<T> g{};
  recnet_decoder_desc d1 = d; d1.L = 1;
  g.w = plan<T>(d1, base);
  Bump m(base); m.off = g.w.bytes;
  g.tok = m.take<long long>(d.B);
  g.nonpad = m.take<int>(max_steps);
  g.h_scratch = m.take<float>((size_t)d.B * d.H);
  if (mode != DecodeMode::GREEDY) m.off += 256;            // 256 bytes of slack after the greedy buffers, as after the sequence plan
  if (mode == DecodeMode::BEAM) {
    for (int i = 0; i < 2; ++i) {
      g.cum[i] = m.take<float>((size_t)d.B);
      g.eos[i] = m.take<int>((size_t)d.B);
      g.seq[i] = m.take<int>((size_t)d.B * max_steps);
    }
    g.src = m.take<int>((size_t)d.B);
  } else if (mode == DecodeMode::SAMPLE) {
    g.finished = m.take<int>((size_t)d.B);
  }
  g.bytes = m.off + 256;
  return g;
}

// The argument checks of the decode entry points and their workspace queries, all before anything is launched.  Greedy checks max_steps
// before the descriptor, beam search and sampling after it.  d = nullptr leaves out every check that reads the descriptor: the greedy
// and beam workspace queries answer for any descriptor.  A decode call ignores the descriptor's L.
static inline int check_decode(const DecDesc* d, DecodeMode mode, int K, int max_steps, float tau, const unsigned long long* noise,
                               const unsigned long long* rng) {
  const bool steps_ok = max_steps >= 1 && max_steps <= 64;
  if (mode == DecodeMode::GREEDY && !steps_ok) return RECNET_ERR_BAD_SHAPE;
  if (d) {
    DecDesc d1 = *d; d1.L = 1;
    RN_TRY(check(d1));
  }
  if (!steps_ok) return RECNET_ERR_BAD_SHAPE;
  if (mode == DecodeMode::BEAM && (K < 1 || K > BEAM_MAX_K || (d && (d->B % K || K > d->V)))) return RECNET_ERR_BAD_SHAPE;
  if (mode == DecodeMode::SAMPLE && (!(tau > 0.f) || !noise || (d && d->train && !rng))) return RECNET_ERR_BAD_SHAPE;
  return 0;
}

// zero initial state of the decode loops: both blocks of X and c, and of every X_x / c_x in a stack
template <typename T>
static int zero_decode_state(const DecDesc& d, Ws<T>& w, cudaStream_t st) {
  const int B = d.B, H = d.H;
  RN_CUDA_OK(cudaMemsetAsync(w.X, 0, (size_t)2 * B * w.KX * sizeof(T), st));
  RN_CUDA_OK(cudaMemsetAsync(w.c, 0, (size_t)2 * B * H * sizeof(float), st));
  for (int l = 1; l < w.NL; ++l) {
    RN_CUDA_OK(cudaMemsetAsync(w.X_x[l - 1], 0, (size_t)2 * B * 2 * H * sizeof(T), st));
    RN_CUDA_OK(cudaMemsetAsync(w.c_x[l - 1], 0, (size_t)2 * B * H * sizeof(float), st));
  }
  return 0;
}

// One decode call on the general step path, the whole loop on the device with no host sync; the arguments passed check_decode.
//   GREEDY: ids_out [max_steps, B]; n_steps_out = the first step (1-based) after which every fed-back token was <PAD> (eval.py:30),
//           else max_steps.
//   BEAM:   d0.B = K * B0 rows, feats [K * B0, T, E] = the B0 samples tiled K times; ids_out [B0, max_steps] = the top-1 sequences
//           (-1 beyond n_steps), n_steps_out as for greedy.
//   SAMPLE: ids_out / logp_out [max_steps, B], lengths_out [B] = sampled tokens of the row, the finishing one included; n_steps_out =
//           the step at which the last row finished + 1 (max_steps if a row never finishes).  In train mode (d0.train) every dropout
//           mask is drawn from the pair rng; noise = the Gumbel pair.
// Greedy and beam search decode in eval mode.  Sampling always runs here: greedy_pf hoists the embedding projection and could not drop
// the embedding.
template <typename T>
static int decode(const DecDesc& d0, const recnet_decoder_tensors& p, const float* feats, DecodeMode mode, int K, int max_steps,
                  float tau, long long eos, const unsigned long long* rng, const unsigned long long* noise, void* ws, long long ws_bytes,
                  long long* ids_out, float* logp_out, int* lengths_out, int* n_steps_out, cudaStream_t st) {
  DecDesc d = d0; d.L = 1;
  if (mode != DecodeMode::SAMPLE) d.train = 0;
  DecodeWs<T> g = plan_decode<T>(d0, ws, mode, max_steps);
  if ((long long)g.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  Ws<T>& w = g.w;
  const bool beam = mode == DecodeMode::BEAM;
  const int B = d.B, B0 = B / K, H = d.H, E = d.E, A = d.A, V = d.V, Tn = d.T, NL = w.NL;
  const float p_emb = d.train ? d.p_emb_drop : 0.f, p_out = d.train ? d.p_out_drop : 0.f, p_lay = d.train ? d.p_layer_drop : 0.f;
  RN_TRY(prepare<T>(d, p, feats, w, st));
  RN_TRY(gemm_full<T>(w.feats, E, 0, w.U, E, 0, w.Uv, A, nullptr, B * Tn, A, E, 0, w.splitk, st));
  RN_TRY(zero_decode_state<T>(d, w, st));
  RN_CUDA_OK(cudaMemsetAsync(g.nonpad, 0, (size_t)max_steps * sizeof(int), st));
  if (mode == DecodeMode::SAMPLE) {
    RN_CUDA_OK(cudaMemsetAsync(ids_out, 0, (size_t)max_steps * B * sizeof(long long), st));
    RN_CUDA_OK(cudaMemsetAsync(logp_out, 0, (size_t)max_steps * B * sizeof(float), st));
    sample_init_kernel<<<rn_cdiv(B, 128), 128, 0, st>>>(g.tok, g.finished, lengths_out, B, max_steps);
  } else {
    fill_tokens_kernel<<<rn_cdiv(B, 128), 128, 0, st>>>(g.tok, B, 1 /* <SOS> */);
  }
  RN_LAUNCH_OK();
  if (beam) {
    beam_init_kernel<<<rn_cdiv(B, 128), 128, 0, st>>>(g.cum[0], g.eos[0], B);
    RN_LAUNCH_OK();
  }
  long long ldq;
  const T* Htop = top_h(d, w, &ldq);
  BeamStateRows<T> rows{};                 // beam search: h (own recurrent slot) and c of every layer, block 1 -> block 0
  rows.n = NL;
  for (int l = 0; l < NL; ++l) {
    T* h = l == 0 ? w.X + E : w.X_x[l - 1] + H;
    float* c = l == 0 ? w.c : w.c_x[l - 1];
    rows.ld[l] = l == 0 ? w.KX : 2 * H;
    rows.h_dst[l] = h; rows.h_src[l] = h + (size_t)B * rows.ld[l];
    rows.c_dst[l] = c; rows.c_src[l] = c + (size_t)B * H;
  }
  for (int t = 0; t < max_steps; ++t) {
    // Greedy and sampling ping-pong the two blocks of every X / c buffer: step t reads block t & 1 and writes block (t + 1) & 1.  Beam
    // search reads block 0 and writes block 1, and its gather moves the selected beams' state back into block 0.  The top layer's h
    // (attention query, vocabulary projection) sits at the same place in either block (top_h).
    const int rd = beam ? 0 : t & 1, wr = beam ? 1 : (t + 1) & 1;
    T* x_t = w.X + (size_t)rd * B * w.KX;
    T* x_n = w.X + (size_t)wr * B * w.KX;
    float* c_p = w.c + (size_t)rd * B * H;
    float* c_n = w.c + (size_t)wr * B * H;
    misc::embed_gather_kernel<T><<<B, 128, 0, st>>>(p.embedding, g.tok, w.Xe, w.EMBp, B, d.EMB, w.EMBp, V, d.embedding_scale, p_emb,
                                                    rng, SITE_EMB, (long long)t * B);
    RN_LAUNCH_OK();
    RN_TRY(gemm_full<T>(w.Xe, w.EMBp, 0, w.Wemb, w.EMBp, 0, w.Gx, w.G * H, p.b_ih, B, w.G * H, w.EMBp, 0, w.splitk, st));
    // GRU keeps its fp32 state h in the c rows (h_prev = c_p, h' -> c_n)
    RN_TRY(step<T>(d, p, w, t, Htop + (size_t)rd * B * ldq, ldq, w.Gx, x_t, x_n, nullptr, nullptr, nullptr, c_p, c_n,
                   d.cell == RECNET_CELL_GRU ? c_n : g.h_scratch, st, NL > 1 ? w.X_x[0] + (size_t)rd * B * 2 * H : nullptr, rng));
    RN_TRY(upper_layers<T>(d, p, w, t, rd, wr, nullptr, p_lay, rng, st));
    RN_TRY(gemm_full<T>(Htop + (size_t)wr * B * ldq, ldq, 0, w.Wout, H, 0, w.logits, w.Vld, p.out_b, B, V, H, 0, w.splitk, st));
    if (mode == DecodeMode::GREEDY) {
      argmax_feedback_kernel<<<B, 256, 0, st>>>(w.logits, w.Vld, V, ids_out + (size_t)t * B, g.tok, g.nonpad + t);
    } else if (mode == DecodeMode::SAMPLE) {
      sample_select_kernel<<<B, SAMPLE_THREADS, 0, st>>>(w.logits, w.Vld, V, B, t, tau, eos, p_out, rng, noise, ids_out + (size_t)t * B,
                                                         logp_out + (size_t)t * B, g.tok, g.finished, lengths_out, g.nonpad);
    } else {
      const int in = t & 1, out = (t + 1) & 1;
      beam_select_kernel<<<B0, BEAM_THREADS, 0, st>>>(w.logits, w.Vld, V, B0, K, t, max_steps, eos, g.cum[in], g.cum[out], g.eos[in],
                                                      g.eos[out], g.seq[in], g.seq[out], g.tok, g.src, g.nonpad);
      RN_LAUNCH_OK();
      beam_gather_layers_kernel<T><<<B, 128, 0, st>>>(rows, H, B0, K, g.src, g.nonpad, t);
    }
    RN_LAUNCH_OK();
  }
  if (beam)
    beam_finalize_kernel<<<1, 256, 0, st>>>(g.nonpad, max_steps, B0, K, g.seq[0], g.seq[1], ids_out, n_steps_out);
  else
    greedy_finalize_kernel<<<1, 1, 0, st>>>(g.nonpad, max_steps, n_steps_out);
  RN_LAUNCH_OK();
  return 0;
}
}  // namespace dec
