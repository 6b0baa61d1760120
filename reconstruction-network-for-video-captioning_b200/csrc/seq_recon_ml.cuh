// Local reconstructor over a STACKED decoder (hiddens (L, NLd, B, H), NLd > 1) -- the reference's quirk A7
// (models/local_reconstructor.py:44-54): the attended input keeps the decoder-layer axis, (NLd, B, H), and nn.LSTM
// treats that axis as TIME, so every outer step t runs NLd pseudo-steps (attention over layer l's states -> LSTM step),
// all NLd attentions sharing ONE query (the state at the start of the outer step); the output projection reads the
// state after pseudo-step 0 (`output[0]`).  One kernel per phase (LSTM cells only).
#pragma once
#include "seq_recon.cuh"

namespace rec {

template <typename T>
__global__ void copy_rows_kernel(const T* __restrict__ src, long long src_row_stride, T* __restrict__ dst, long long n_rows, int cols) {
  const long long total = n_rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols; const int c = (int)(i % cols);
    dst[i] = src[r * src_row_stride + c];
  }
}

template <typename T>
static int local_forward_ml(const LocalDesc& d, const recnet_local_tensors& p, const float* hiddens, const float* feats,
                            const unsigned long long* rng, void* ws, long long ws_bytes, float* mse_out, cudaStream_t st) {
  RN_TRY(check_local(d));
  LocalWs<T> w = plan_local<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, S = d.S, R = d.R, H = d.H, A = d.A, L = d.L, NLd = d.dec_layers;
  const float p_drop = d.train ? d.p_drop : 0.f;
  RN_TRY(misc::cast_pad<T>(p.w_ih, H, w.Wrec, w.KX, 4 * R, H, H, st));
  RN_TRY(misc::cast_pad<T>(p.w_hh, R, w.Wrec + H, w.KX, 4 * R, R, R, st));
  RN_TRY(misc::cast_pad<T>(p.attn_U, H, w.U, H, A, H, H, st));
  RN_TRY(misc::cast_pad<T>(p.attn_W, R, w.Wa, R, A, R, R, st));
  RN_TRY(misc::cast_pad<T>(p.out_w, R, w.Wout, R, R, R, R, st));
  RN_TRY(misc::cast_pad<T>(hiddens, H, w.Hd, H, (long long)L * NLd * B, H, H, st));
  RN_TRY(gemm_full<T>(w.Hd, H, 0, w.U, H, 0, w.Uv, A, nullptr, L * NLd * B, A, H, 0, w.splitk, st));
  RN_CUDA_OK(cudaMemsetAsync(w.X, 0, (size_t)B * w.KX * sizeof(T), st));
  RN_CUDA_OK(cudaMemsetAsync(w.c, 0, (size_t)B * R * sizeof(float), st));
  RN_CUDA_OK(cudaMemsetAsync(w.err, 0, sizeof(int), st));
  int n_whp = 0;
  for (int t = 0; t < S; ++t) {
    for (int l = 0; l < NLd; ++l) {
      const size_t q = (size_t)t * NLd + l;
      T* x_q = w.X + q * B * w.KX;
      T* x_n = x_q + (size_t)B * w.KX;
      if (l == 0) {
        n_whp = 0;
        if (t > 0) {      // ONE query per outer step: the state before the pseudo-steps
          RN_TRY(gemm_partials<T>(x_q + H, w.KX, 0, w.Wa, R, 0, w.WhP, B, A, R, w.pl_wh, st));
          n_whp = w.pl_wh.splits;
        }
      }
      attn::FwdArgs fa{};
      fa.WhP = w.WhP; fa.n_whp = n_whp; fa.whp_stride = (long long)B * A;
      fa.Uv = w.Uv + (size_t)l * B * A; fa.uv_bs = A; fa.uv_ts = (long long)NLd * B * A;          // Uv is (L, NLd, B, A)
      fa.attn_b = p.attn_b; fa.attn_w = p.attn_w;
      fa.V = w.Hd + (size_t)l * B * H; fa.v_bs = H; fa.v_ts = (long long)NLd * B * H;             // layer l of (L, NLd, B, H)
      fa.B = B; fa.Tn = L; fa.A = A; fa.D = H; fa.inv_T = d.softmax ? 1.f : 1.f / L; fa.normalize = d.softmax;   // softmax per layer
      fa.Wh_out = w.Wh + q * B * A; fa.e_out = w.beta + q * B * L; fa.ctx_out = x_q; fa.ctx_ld = w.KX;
      fa.p_drop = p_drop; fa.rng = rng; fa.site = SITE_LOCAL_X; fa.drop_base = (long long)q * B * H;
      RN_TRY((attn::launch_fwd<T, T>(fa, st)));
      RN_TRY(gemm_partials<T>(x_q, w.KX, 0, w.Wrec, w.KX, 0, w.P, B, 4 * R, w.KX, w.pl_gate, st));
      cell::FwdArgs ca{};
      ca.P = w.P; ca.n_p = w.pl_gate.splits; ca.p_stride = (long long)B * 4 * R; ca.p_ld = 4 * R;
      ca.b1 = p.b_ih; ca.b2 = p.b_hh; ca.c_prev = w.c + q * B * R; ca.B = B; ca.H = R;
      ca.gates_out = w.gates + q * B * 4 * R; ca.c_out = w.c + (q + 1) * B * R;
      ca.h_op = x_n + H; ca.hop_ld = w.KX;
      if (l == 0) { ca.h_op2 = w.Hout + (size_t)t * B * R; ca.hop2_ld = R; }                       // `output[0]`
      RN_TRY((cell::launch_fwd<T, T>(ca, st)));
    }
  }
  // query-state rows (state at the start of every outer step) for the attn_W gradient
  for (int t = 0; t < S; ++t) {
    copy_rows_kernel<T><<<rn_cdiv((long long)B * R, 256), 256, 0, st>>>(w.X + (size_t)t * NLd * B * w.KX + H, w.KX, w.Hq + (size_t)t * B * R, B, R);
    RN_LAUNCH_OK();
  }
  RN_TRY(gemm_full<T>(w.Hout, R, 0, w.Wout, R, 0, w.out, R, p.out_b, S * B, R, R, 0, w.splitk, st));
  if (mse_out) {
    loss::mse_local_fwd_kernel<<<MSE_BLOCKS, 256, 0, st>>>(w.out, feats, S, B, R, w.partial);
    RN_LAUNCH_OK();
    loss::sum_kernel<<<1, 1024, 0, st>>>(w.partial, MSE_BLOCKS, mse_out, 1.f / ((float)S * B * R));
    RN_LAUNCH_OK();
  }
  return 0;
}

template <typename T>
static int local_backward_ml(const LocalDesc& d, const recnet_local_tensors& p, const float* hiddens, const float* feats,
                             const unsigned long long* rng, void* ws, long long ws_bytes, const float* g_mse,
                             const recnet_local_tensors& g, float* g_hiddens, cudaStream_t st) {
  RN_TRY(check_local(d));
  LocalWs<T> w = plan_local<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, S = d.S, R = d.R, H = d.H, A = d.A, L = d.L, NLd = d.dec_layers;
  const float p_drop = d.train ? d.p_drop : 0.f;
  const int SB = S * B, Sp = S * NLd;
  loss::mse_local_bwd_kernel<T><<<MSE_BLOCKS, 256, 0, st>>>(w.out, feats, S, B, R, g_mse, 2.f / ((float)S * B * R), w.dOut);
  RN_LAUNCH_OK();
  RN_TRY(gemm_full<T>(w.dOut, R, 0, w.Wout, R, 1, w.dHext, R, nullptr, SB, R, R, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dOut, R, 1, w.Hout, R, 1, g.out_w, R, nullptr, R, R, SB, 0, w.splitk, st));
  RN_TRY(misc::colsum<T>(w.dOut, R, SB, R, g.out_b, 0, w.splitk, st));
  for (int q = Sp - 1; q >= 0; --q) {
    const int t = q / NLd, l = q % NLd;
    const bool last = (q == Sp - 1);
    cell::BwdArgs cb{};
    if (l == 0) { cb.dh_ext = w.dHext + (size_t)t * B * R; cb.dh_ld = R; }                       // out-proj reads pseudo-step (t,0)
    cb.dXp = last ? nullptr : w.dXp; cb.n_p = w.pl_dx.splits; cb.p_stride = (long long)B * w.KX; cb.p_ld = w.KX; cb.col0 = H;
    if (l == NLd - 1 && t < S - 1) {                                                             // query of outer step t+1
      cb.dQp = w.dQp; cb.n_q = w.pl_dq.splits; cb.q_stride = (long long)B * R; cb.q_ld = R;
    }
    cb.dc = w.dc; cb.first = last ? 1 : 0;
    cb.gates = w.gates + (size_t)q * B * 4 * R;
    cb.c_prev = w.c + (size_t)q * B * R; cb.c_new = w.c + (size_t)(q + 1) * B * R;
    cb.B = B; cb.H = R; cb.dG = w.dG + (size_t)q * B * 4 * R; cb.dg_ld = 4 * R;
    RN_TRY((cell::launch_bwd<T, T>(cb, st)));
    RN_TRY(gemm_partials<T>(w.dG + (size_t)q * B * 4 * R, 4 * R, 0, w.Wrec, w.KX, 1, w.dXp, B, w.KX, 4 * R, w.pl_dx, st));
    attn::BwdArgs ab{};
    ab.dXp = w.dXp; ab.n_p = w.pl_dx.splits; ab.p_stride = (long long)B * w.KX; ab.p_ld = w.KX;
    ab.V = w.Hd + (size_t)l * B * H; ab.v_bs = H; ab.v_ts = (long long)NLd * B * H;
    ab.Wh = w.Wh + (size_t)q * B * A; ab.Uv = w.Uv + (size_t)l * B * A; ab.uv_bs = A; ab.uv_ts = (long long)NLd * B * A;
    ab.attn_b = p.attn_b; ab.attn_w = p.attn_w; ab.B = B; ab.Tn = L; ab.A = A; ab.D = H; ab.inv_T = d.softmax ? 1.f : 1.f / L;
    ab.alpha = d.softmax ? w.beta + (size_t)q * B * L : nullptr;
    ab.dWh_out = w.dWh + (size_t)t * B * A; ab.dWh_op = w.dWh_op + (size_t)t * B * A;          // summed over the NLd attentions of step t
    ab.dwh_acc = (l != NLd - 1) ? 1 : 0;
    ab.dUv_acc = w.dUv + (size_t)l * B * A; ab.uv_first = (t == S - 1) ? 1 : 0;
    ab.dw_acc = w.dw_acc; ab.dw_first = last ? 1 : 0;
    ab.dctx_out = w.dx + (size_t)q * B * H;
    ab.p_drop = p_drop; ab.rng = rng; ab.site = SITE_LOCAL_X; ab.drop_base = (long long)q * B * H;
    RN_TRY((attn::launch_bwd<T, T>(ab, st)));
    if (l == 0 && t > 0) RN_TRY(gemm_partials<T>(w.dWh_op + (size_t)t * B * A, A, 0, w.Wa, R, 1, w.dQp, B, R, A, w.pl_dq, st));
  }
  const int SpB = Sp * B;
  RN_TRY(misc::colsum<T>(w.dG, 4 * R, SpB, 4 * R, g.b_ih, 0, w.splitk, st));
  RN_CUDA_OK(cudaMemcpyAsync(g.b_hh, g.b_ih, (size_t)4 * R * sizeof(float), cudaMemcpyDeviceToDevice, st));
  RN_TRY(gemm_full<T>(w.dG, 4 * R, 1, w.X, w.KX, 1, g.w_ih, H, nullptr, 4 * R, H, SpB, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dG, 4 * R, 1, w.X + H, w.KX, 1, g.w_hh, R, nullptr, 4 * R, R, SpB, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dWh_op, A, 1, w.Hq, R, 1, g.attn_W, R, nullptr, A, R, SB, 0, w.splitk, st));
  RN_TRY(misc::cast_pad<T>(w.dUv, A, w.dUv_op, A, (long long)L * NLd * B, A, A, st));
  RN_TRY(gemm_full<T>(w.dUv_op, A, 1, w.Hd, H, 1, g.attn_U, H, nullptr, A, H, L * NLd * B, 0, w.splitk, st));
  RN_TRY(misc::colsum<float>(w.dWh, A, SB, A, g.attn_b, 0, w.splitk, st));
  RN_TRY(misc::colsum<float>(w.dw_acc, A, B, A, g.attn_w, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dUv_op, A, 0, w.U, H, 1, g_hiddens, H, nullptr, L * NLd * B, H, A, 0, w.splitk, st));
  for (int l = 0; l < NLd; ++l)
    RN_TRY(attn::launch_dv(w.beta, w.dx, g_hiddens + (size_t)l * B * H, H, (long long)NLd * B * H, S, B, L, H, d.softmax ? 1.f : 1.f / L, 1, NLd, l, st));
  return 0;
}
}  // namespace rec
