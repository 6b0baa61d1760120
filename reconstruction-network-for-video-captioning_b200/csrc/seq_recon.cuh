// Reconstructor sequence drivers.
//  local  : train.forward_local_reconstructor (train.py:108-131) over LocalReconstructor.forward
//           (models/local_reconstructor.py:37-55): attention over the L decoder states, LSTM(R), Linear(R,R), MSE.
//  global : train.forward_global_reconstructor (train.py:78-105) over GlobalReconstructor.forward
//           (models/global_reconstructor.py:30-46): [h_t ; mean-pool] -> LSTM(R) -> Linear(R,R), MSE of means / L.
// Same restructuring as the decoder: U.hiddens hoisted, [x ; h] K-concatenated gate GEMM per step, output
// projection and all weight gradients batched over time.
// Local over a STACKED decoder (hiddens (L, NLd, B, H), NLd > 1, LSTM cells only) -- the reference's quirk A7
// (models/local_reconstructor.py:44-54): the attended input keeps the decoder-layer axis, (NLd, B, H), and nn.LSTM
// treats that axis as TIME, so every outer step t runs NLd pseudo-steps (attention over layer l's states -> LSTM step),
// all NLd attentions sharing ONE query (the state at the start of the outer step); the output projection reads the
// state after pseudo-step 0 (`output[0]`).
#pragma once
#include "gru_cell.cuh"
#include "runtime.cuh"
#include "seq_recon_persist.cuh"

namespace rec {
using namespace rt;

enum : unsigned { SITE_LOCAL_X = 3, SITE_GLOBAL_MP = 4 };

// ================================================ local =========================================================
template <typename T>
struct LocalWs {
  int KX, G;
  GemmPlan pl_wh, pl_gate, pl_dx, pl_dq;
  GemmPlan pl_gx, pl_gh, pl_dxx, pl_dxh;      // GRU: input / hidden sides kept separate
  T *Wrec, *U, *Wa, *Wout, *Hd;
  float* Uv; T* X; float* WhP; float* Wh; float* beta; float* P; float* P2; T* gates; float* c; float* out; float* partial;
  T* dOut; float* dHext; T* dG; T* dG2; float* dXp; float* dXp2; float* dQp; float* dWh; T* dWh_op; float* dUv; T* dUv_op; float* dw_acc; float* dc;
  float* dx; float* splitk; float* splitk2;        // splitk2: scratch of the side stream (runtime.cuh:Side)
  int* err;
  T* Hout; T* Hq;                 // stacked decoder only: compact rows of h after pseudo-step (t,0) / at the start of outer step t
  float* pXP; float* pWhP; unsigned* psync;      // weight-resident persistent loop (seq_recon_persist.cuh): partial exchange + flags
  size_t bytes;
};
constexpr int MSE_BLOCKS = 592;

// the weight-resident persistent forward loop covers: bf16, LSTM over a 1-layer decoder, shapes whose [W_ih | W_hh] fits the SMs' shared memory
template <typename T>
static inline bool persist_fwd_ok(const recnet_local_desc& d) {
  if (!std::is_same<T, bf16>::value || d.cell != RECNET_CELL_LSTM || d.dec_layers > 1) return false;
  return rp::local_fwd_ok(rp::Shape{d.B, d.S, d.R, d.H, d.A, d.L});
}
template <typename T>
static inline bool persist_bwd_ok(const recnet_local_desc& d) {
  if (!std::is_same<T, bf16>::value || d.cell != RECNET_CELL_LSTM || d.dec_layers > 1) return false;
  static const int on = rn_env_int("RECNET_PERSIST_BWD", 1);
  return on && rp::local_bwd_ok(rp::Shape{d.B, d.S, d.R, d.H, d.A, d.L});
}

template <typename T>
static LocalWs<T> plan_local(const recnet_local_desc& d, void* base) {
  LocalWs<T> w;
  const int NLd = d.dec_layers < 1 ? 1 : d.dec_layers;
  // with a stacked decoder every outer step runs NLd pseudo-steps and the hiddens carry a layer axis: size by S*NLd / L*NLd
  const int B = d.B, S = d.S * NLd, R = d.R, H = d.H, A = d.A, L = d.L * NLd;
  w.KX = H + R;
  w.pl_wh = plan_gemm<T>(B, A, R);
  if (w.pl_wh.splits > 8) {      // the attention kernel sums these partials with one batch of 8 loads per lane
    const int nkb = rn_cdiv(R, 64);
    w.pl_wh.splits = rn_cdiv(nkb, rn_cdiv(nkb, 8));
  }
  w.pl_gate = plan_gemm<T>(B, 4 * R, w.KX);
  w.pl_dx = plan_gemm<T>(B, w.KX, 4 * R);
  w.pl_dq = plan_gemm<T>(B, R, A);
  const bool gru_ = d.cell == RECNET_CELL_GRU;
  w.G = gru_ ? 3 : 4;
  w.pl_gx = plan_gemm<T>(B, 3 * R, H);
  w.pl_gh = plan_gemm<T>(B, 3 * R, R);
  w.pl_dxx = plan_gemm<T>(B, H, 3 * R);
  w.pl_dxh = plan_gemm<T>(B, R, 3 * R);
  Bump m(base);
  w.Wrec = m.take<T>((size_t)4 * R * w.KX);
  w.U = m.take<T>((size_t)A * H);
  w.Wa = m.take<T>((size_t)A * R);
  w.Wout = m.take<T>((size_t)R * R);
  w.Hd = m.take<T>((size_t)L * B * H);
  w.Uv = m.take<float>((size_t)L * B * A);
  w.X = m.take<T>((size_t)(S + 1) * B * w.KX);
  w.WhP = m.take<float>((size_t)(w.pl_wh.splits > rn_cdiv(R, cell::THREADS) ? w.pl_wh.splits : rn_cdiv(R, cell::THREADS)) * B * A);
  w.Wh = m.take<float>((size_t)S * B * A);
  w.beta = m.take<float>((size_t)S * B * L);
  w.P = m.take<float>((size_t)(gru_ ? w.pl_gx.splits : w.pl_gate.splits) * B * 4 * R);
  w.P2 = m.take<float>(gru_ ? (size_t)w.pl_gh.splits * B * 3 * R : 1);
  w.gates = m.take<T>((size_t)S * B * 4 * R);
  w.c = m.take<float>((size_t)(S + 1) * B * R);
  w.out = m.take<float>((size_t)S * B * R);
  w.partial = m.take<float>(MSE_BLOCKS);
  w.dOut = m.take<T>((size_t)S * B * R);
  w.dHext = m.take<float>((size_t)S * B * R);
  w.dG = m.take<T>((size_t)S * B * 4 * R);
  w.dXp = m.take<float>((size_t)(gru_ ? w.pl_dxx.splits : w.pl_dx.splits) * B * w.KX);
  w.dXp2 = m.take<float>(gru_ ? (size_t)w.pl_dxh.splits * B * R : 1);
  w.dG2 = m.take<T>(gru_ ? (size_t)S * B * 3 * R : 1);
  w.dQp = m.take<float>((size_t)w.pl_dq.splits * B * R);
  w.dWh = m.take<float>((size_t)S * B * A);
  w.dWh_op = m.take<T>((size_t)S * B * A);
  w.dUv = m.take<float>((size_t)L * B * A);
  w.dUv_op = m.take<T>((size_t)L * B * A);
  w.dw_acc = m.take<float>((size_t)B * A);
  w.dc = m.take<float>((size_t)B * R);
  w.dx = m.take<float>((size_t)S * B * H);
  w.splitk = m.take<float>(SPLITK_SCRATCH_FLOATS);
  w.splitk2 = m.take<float>(SPLITK_SCRATCH_FLOATS);
  w.err = m.take<int>(64);
  w.Hout = m.take<T>(NLd > 1 ? (size_t)d.S * B * R : 1);
  w.Hq = m.take<T>(NLd > 1 ? (size_t)d.S * B * R : 1);
  const bool pers = persist_fwd_ok<T>(d);
  const rp::Shape shp{d.B, d.S, d.R, d.H, d.A, d.L};
  const bool persb = persist_bwd_ok<T>(d);
  size_t xpn = pers ? rp::xp_floats(shp) : 1;                 // forward K-slice partials and backward gate-slice partials share the buffer
  if (persb && rp::dp_floats(shp) > xpn) xpn = rp::dp_floats(shp);
  w.pXP = m.take<float>(xpn);
  w.pWhP = m.take<float>(pers ? rp::whp_floats(shp) : 1);
  w.psync = m.take<unsigned>(2 * rp::SYNC_WORDS);              // forward flags | backward flags (both zeroed by the forward's staging kernel)
  w.bytes = m.off + 256;
  return w;
}

// Rows of h that the output projection reads and rows of the attention query, S*B each with ld `ld`: the h slots of X over a
// one-layer decoder; over a stacked one the compact copies Hout (`output[0]`) and Hq (state at the start of every outer step).
template <typename T>
struct HRows { const T* out; const T* query; long long ld; };
template <typename T>
static HRows<T> h_rows(const recnet_local_desc& d, const LocalWs<T>& w) {
  if (d.dec_layers > 1) return {w.Hout, w.Hq, d.R};
  return {w.X + (size_t)d.B * w.KX + d.H, w.X + d.H, w.KX};
}

template <typename T>
__global__ void copy_rows_kernel(const T* __restrict__ src, long long src_row_stride, T* __restrict__ dst, long long n_rows, int cols) {
  const long long total = n_rows * cols;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cols; const int c = (int)(i % cols);
    dst[i] = src[r * src_row_stride + c];
  }
}

static inline int check_local(const recnet_local_desc& d) {
  if (d.B < 1 || d.S < 1 || d.L < 1 || d.L > attn::MAX_T) return RECNET_ERR_BAD_SHAPE;
  if (d.cell != RECNET_CELL_LSTM && d.cell != RECNET_CELL_GRU) return RECNET_ERR_UNSUPPORTED;
  if (d.dec_layers > 1 && d.cell != RECNET_CELL_LSTM) return RECNET_ERR_UNSUPPORTED;
  const int al = d.precision == RECNET_PREC_BF16 ? 8 : 4;
  if (d.R % al || d.H % al || d.A % 4) return RECNET_ERR_ALIGNMENT;
  return 0;
}

template <typename T>
static int local_forward(const LocalDesc& d, const recnet_local_tensors& p, const float* hiddens, const float* feats,
                         const unsigned long long* rng, void* ws, long long ws_bytes, float* mse_out, cudaStream_t st) {
  RN_TRY(check_local(d));
  LocalWs<T> w = plan_local<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, S = d.S, R = d.R, H = d.H, A = d.A, L = d.L, NLd = d.dec_layers < 1 ? 1 : d.dec_layers;
  const float p_drop = d.train ? d.p_drop : 0.f;
  const bool is_gru = d.cell == RECNET_CELL_GRU;
  const int GR = w.G * R;
  // operand copies of the weights / decoder states + cleared initial state: ONE multi-tensor staging kernel (misc.cuh:Stager)
  misc::Stager<T> sg;
  sg.add(p.w_ih, H, w.Wrec, w.KX, GR, H, H);
  sg.add(p.w_hh, R, w.Wrec + H, w.KX, GR, R, R);
  sg.add(p.attn_U, H, w.U, H, A, H, H);
  sg.add(p.attn_W, R, w.Wa, R, A, R, R);
  sg.add(p.out_w, R, w.Wout, R, R, R, R);
  sg.add(hiddens, H, w.Hd, H, (long long)L * NLd * B, H, H);
  sg.zero(w.X, (size_t)B * w.KX * sizeof(T));
  sg.zero(w.c, (size_t)B * R * sizeof(float));
  sg.zero(w.err, 64 * sizeof(int));
  const bool persist = persist_fwd_ok<T>(d);
  if (persist || persist_bwd_ok<T>(d)) sg.zero(w.psync, 2 * rp::SYNC_WORDS * sizeof(unsigned));
  RN_TRY(sg.launch(st));
  RN_TRY(gemm_full<T>(w.Hd, H, 0, w.U, H, 0, w.Uv, A, nullptr, L * NLd * B, A, H, 0, w.splitk, st));     // U.hiddens, once
  if constexpr (std::is_same<T, bf16>::value) {
    if (persist) {
      // ONE cooperative launch for all S steps, [W_ih | W_hh] resident in shared memory (seq_recon_persist.cuh); same stash layout
      rp::FwdParams fp{};
      fp.B = B; fp.S = S; fp.R = R; fp.H = H; fp.A = A; fp.L = L; fp.inv_L = d.softmax ? 1.f : 1.f / L; fp.p_drop = p_drop;
      fp.X = w.X; fp.Hd = w.Hd; fp.Uv = w.Uv; fp.Wa = w.Wa; fp.attn_b = p.attn_b; fp.attn_w = p.attn_w; fp.b_ih = p.b_ih; fp.b_hh = p.b_hh;
      fp.Wh = w.Wh; fp.beta = w.beta; fp.gates = w.gates; fp.c = w.c; fp.XP = w.pXP; fp.WhP = w.pWhP; fp.sync = w.psync; fp.err = w.err;
      fp.rng = rng; fp.site = SITE_LOCAL_X;
      RN_TRY(rp::launch_local_fwd(fp, w.Wrec, d.softmax, st));
      RN_TRY(gemm_full<T>(w.X + (size_t)B * w.KX + H, w.KX, 0, w.Wout, R, 0, w.out, R, p.out_b, S * B, R, R, 0, w.splitk, st));
      if (mse_out) {
        loss::mse_local_fwd_kernel<<<MSE_BLOCKS, 256, 0, st>>>(w.out, feats, S, B, R, w.partial);
        RN_LAUNCH_OK();
        loss::sum_kernel<<<1, 1024, 0, st>>>(w.partial, MSE_BLOCKS, mse_out, 1.f / ((float)S * B * R));
        RN_LAUNCH_OK();
      }
      return 0;
    }
  }
  int n_whp = 0;
  for (int q = 0; q < S * NLd; ++q) {      // pseudo-step q = (outer step t, decoder layer l)
    const int t = q / NLd, l = q - t * NLd;
    const size_t r = (size_t)q * B;
    T* x_t = w.X + r * w.KX;
    T* x_n = x_t + (size_t)B * w.KX;
    // attention query W.h_{t-1}: its own small GEMM, partials summed by the attention kernel; ONE per outer step
    if (l == 0) {
      n_whp = 0;
      if (t > 0) {
        RN_TRY(gemm_partials<T>(x_t + H, w.KX, 0, w.Wa, R, 0, w.WhP, B, A, R, w.pl_wh, st));
        n_whp = w.pl_wh.splits;
      }
    }
    attn::FwdArgs fa{};
    fa.WhP = w.WhP; fa.n_whp = n_whp; fa.whp_stride = (long long)B * A;
    fa.Uv = w.Uv + (size_t)l * B * A; fa.uv_bs = A; fa.uv_ts = (long long)NLd * B * A;          // Uv is [L,NLd,B,A]
    fa.attn_b = p.attn_b; fa.attn_w = p.attn_w;
    fa.V = w.Hd + (size_t)l * B * H; fa.v_bs = H; fa.v_ts = (long long)NLd * B * H;             // values = layer l of [L,NLd,B,H]
    fa.B = B; fa.Tn = L; fa.A = A; fa.D = H; fa.inv_T = d.softmax ? 1.f : 1.f / L; fa.normalize = d.softmax;
    fa.Wh_out = w.Wh + r * A; fa.e_out = w.beta + r * L;
    fa.ctx_out = x_t; fa.ctx_ld = w.KX;
    fa.p_drop = p_drop; fa.rng = rng; fa.site = SITE_LOCAL_X; fa.drop_base = (long long)r * H;
    RN_TRY((attn::launch_fwd<T, T>(fa, st)));
    if (is_gru) {
      RN_TRY(gemm_partials<T>(x_t, w.KX, 0, w.Wrec, w.KX, 0, w.P, B, 3 * R, H, w.pl_gx, st));
      if (q > 0) RN_TRY(gemm_partials<T>(x_t + H, w.KX, 0, w.Wrec + H, w.KX, 0, w.P2, B, 3 * R, R, w.pl_gh, st));
      gru::FwdArgs ga{};
      ga.Px = w.P; ga.n_px = w.pl_gx.splits; ga.px_stride = (long long)B * 3 * R; ga.px_ld = 3 * R;
      ga.Ph = q > 0 ? w.P2 : nullptr; ga.n_ph = q > 0 ? w.pl_gh.splits : 0; ga.ph_stride = (long long)B * 3 * R; ga.ph_ld = 3 * R;
      ga.Gx = nullptr; ga.b_ih = p.b_ih; ga.b_hh = p.b_hh;
      ga.h_prev = w.c + r * R; ga.hp_ld = R; ga.B = B; ga.H = R;            // fp32 state h lives in the c rows
      ga.stash = w.gates + r * 4 * R; ga.h_out = w.c + (size_t)(q + 1) * B * R; ga.h_ld = R;
      ga.h_op = x_n + H; ga.hop_ld = w.KX;
      RN_TRY((gru::launch_fwd<T, T>(ga, st)));
      continue;
    }
    RN_TRY(gemm_partials<T>(x_t, w.KX, 0, w.Wrec, w.KX, 0, w.P, B, 4 * R, w.KX, w.pl_gate, st));
    cell::FwdArgs ca{};
    ca.P = w.P; ca.n_p = w.pl_gate.splits; ca.p_stride = (long long)B * 4 * R; ca.p_ld = 4 * R;
    ca.Gx = nullptr; ca.b1 = p.b_ih; ca.b2 = p.b_hh; ca.c_prev = w.c + r * R; ca.B = B; ca.H = R;
    ca.gates_out = w.gates + r * 4 * R; ca.c_out = w.c + (size_t)(q + 1) * B * R; ca.h_out = nullptr;
    ca.h_op = x_n + H; ca.hop_ld = w.KX; ca.h_op2 = nullptr;
    if (NLd > 1 && l == 0) { ca.h_op2 = w.Hout + (size_t)t * B * R; ca.hop2_ld = R; }        // `output[0]`
    RN_TRY((cell::launch_fwd<T, T>(ca, st)));
  }
  // stacked: query-state rows (state at the start of every outer step) for the attn_W gradient
  for (int t = 0; t < S && NLd > 1; ++t) {
    copy_rows_kernel<T><<<rn_cdiv((long long)B * R, 256), 256, 0, st>>>(w.X + (size_t)t * NLd * B * w.KX + H, w.KX, w.Hq + (size_t)t * B * R, B, R);
    RN_LAUNCH_OK();
  }
  const HRows<T> hr = h_rows(d, w);
  RN_TRY(gemm_full<T>(hr.out, hr.ld, 0, w.Wout, R, 0, w.out, R, p.out_b, S * B, R, R, 0, w.splitk, st));
  if (mse_out) {
    loss::mse_local_fwd_kernel<<<MSE_BLOCKS, 256, 0, st>>>(w.out, feats, S, B, R, w.partial);
    RN_LAUNCH_OK();
    loss::sum_kernel<<<1, 1024, 0, st>>>(w.partial, MSE_BLOCKS, mse_out, 1.f / ((float)S * B * R));
    RN_LAUNCH_OK();
  }
  return 0;
}

template <typename T>
static int local_backward_weights(const recnet_local_desc& d, const LocalWs<T>& w, const recnet_local_tensors& g, cudaStream_t st);

// phases: bit 0 = BPTT loop + gradient wrt the decoder states (everything the decoder's backward waits for), bit 1 = the batched
// parameter gradients over the stashed operands.  recnet_local_bwd runs both; a trainer may run bit 1 on a second stream underneath
// the decoder's backward loop (recnet_local_bwd_phase, functional.deferred_weight_grads).
template <typename T>
static int local_backward(const LocalDesc& d, const recnet_local_tensors& p, const float* hiddens, const float* feats,
                          const unsigned long long* rng, void* ws, long long ws_bytes, const float* g_mse,
                          const recnet_local_tensors& g, float* g_hiddens, cudaStream_t st, int phases = 3) {
  RN_TRY(check_local(d));
  LocalWs<T> w = plan_local<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  if (!(phases & 1)) return (phases & 2) ? local_backward_weights<T>(d, w, g, st) : 0;
  const int B = d.B, S = d.S, R = d.R, H = d.H, A = d.A, L = d.L, NLd = d.dec_layers < 1 ? 1 : d.dec_layers;
  const float p_drop = d.train ? d.p_drop : 0.f;
  const int SB = S * B;
  loss::mse_local_bwd_kernel<T><<<MSE_BLOCKS, 256, 0, st>>>(w.out, feats, S, B, R, g_mse, 2.f / ((float)S * B * R), w.dOut);
  RN_LAUNCH_OK();
  RN_TRY(gemm_full<T>(w.dOut, R, 0, w.Wout, R, 1, w.dHext, R, nullptr, SB, R, R, 0, w.splitk, st));
  const bool is_gru = d.cell == RECNET_CELL_GRU;
  const int GR = w.G * R;
  bool persist = false;
  if constexpr (std::is_same<T, bf16>::value) {
    persist = persist_bwd_ok<T>(d);
    if (persist) {
      // ONE cooperative launch for the whole BPTT loop, [W_ih | W_hh] resident in shared memory (seq_recon_persist.cuh)
      rp::BwdParams bp{};
      bp.B = B; bp.S = S; bp.R = R; bp.H = H; bp.A = A; bp.L = L; bp.inv_L = d.softmax ? 1.f : 1.f / L; bp.p_drop = p_drop;
      bp.Hd = w.Hd; bp.Uv = w.Uv; bp.Wa = w.Wa; bp.attn_b = p.attn_b; bp.attn_w = p.attn_w; bp.Wh = w.Wh; bp.gates = w.gates; bp.c = w.c;
      bp.dHext = w.dHext; bp.dG = w.dG; bp.dx = w.dx; bp.dWh = w.dWh; bp.dWh_op = w.dWh_op; bp.dUv = w.dUv; bp.dw_acc = w.dw_acc;
      bp.DP = w.pXP; bp.sync = w.psync + rp::SYNC_WORDS; bp.err = w.err; bp.rng = rng; bp.site = SITE_LOCAL_X;
      bp.alpha = d.softmax ? w.beta : nullptr;
      RN_TRY(rp::launch_local_bwd(bp, w.Wrec, st));
    }
  }
  for (int q = S * NLd - 1; q >= 0 && !persist; --q) {      // pseudo-step q = (outer step t, decoder layer l)
    const int t = q / NLd, l = q - t * NLd;
    const bool last = (q == S * NLd - 1);
    const size_t r = (size_t)q * B;
    if (is_gru) {
      float* dXx = w.dXp;
      float* dXh = w.dXp2;
      gru::BwdArgs gb{};
      gb.dh_ext = w.dHext + r * R; gb.dh_ld = R;
      gb.dHp = last ? nullptr : dXh; gb.n_p = w.pl_dxh.splits; gb.p_stride = (long long)B * R; gb.p_ld = R;
      gb.dQp = last ? nullptr : w.dQp; gb.n_q = w.pl_dq.splits; gb.q_stride = (long long)B * R; gb.q_ld = R;
      gb.carry = w.dc; gb.first = last ? 1 : 0;
      gb.stash = w.gates + r * 4 * R; gb.h_prev = w.c + r * R; gb.hp_ld = R;
      gb.B = B; gb.H = R; gb.dGi = w.dG + r * 3 * R; gb.dGh = w.dG2 + r * 3 * R; gb.dg_ld = 3 * R;
      RN_TRY((gru::launch_bwd<T, T>(gb, st)));
      RN_TRY(gemm_partials<T>(w.dG + r * 3 * R, 3 * R, 0, w.Wrec, w.KX, 1, dXx, B, H, 3 * R, w.pl_dxx, st));
      if (t > 0) RN_TRY(gemm_partials<T>(w.dG2 + r * 3 * R, 3 * R, 0, w.Wrec + H, w.KX, 1, dXh, B, R, 3 * R, w.pl_dxh, st));
      attn::BwdArgs ab{};
      ab.dXp = dXx; ab.n_p = w.pl_dxx.splits; ab.p_stride = (long long)B * H; ab.p_ld = H;
      ab.V = w.Hd; ab.v_bs = H; ab.v_ts = (long long)B * H;
      ab.Wh = w.Wh + r * A; ab.Uv = w.Uv; ab.uv_bs = A; ab.uv_ts = (long long)B * A;
      ab.attn_b = p.attn_b; ab.attn_w = p.attn_w; ab.B = B; ab.Tn = L; ab.A = A; ab.D = H; ab.inv_T = d.softmax ? 1.f : 1.f / L;
      ab.dWh_out = w.dWh + r * A; ab.dWh_op = w.dWh_op + r * A; ab.dUv_acc = w.dUv;
      ab.uv_first = last ? 1 : 0; ab.dw_first = last ? 1 : 0; ab.dw_acc = w.dw_acc;
      ab.dctx_out = w.dx + r * H; ab.de_out = nullptr; ab.alpha = d.softmax ? w.beta + r * L : nullptr;
      ab.p_drop = p_drop; ab.rng = rng; ab.site = SITE_LOCAL_X; ab.drop_base = (long long)r * H;
      RN_TRY((attn::launch_bwd<T, T>(ab, st)));
      if (t > 0) RN_TRY(gemm_partials<T>(w.dWh_op + r * A, A, 0, w.Wa, R, 1, w.dQp, B, R, A, w.pl_dq, st));
      continue;
    }
    cell::BwdArgs cb{};
    if (l == 0) { cb.dh_ext = w.dHext + (size_t)t * B * R; cb.dh_ld = R; }                       // out-proj reads pseudo-step (t,0)
    cb.dXp = last ? nullptr : w.dXp; cb.n_p = w.pl_dx.splits; cb.p_stride = (long long)B * w.KX; cb.p_ld = w.KX; cb.col0 = H;
    if (l == NLd - 1) {                                                                          // query of outer step t+1
      cb.dQp = last ? nullptr : w.dQp; cb.n_q = w.pl_dq.splits; cb.q_stride = (long long)B * R; cb.q_ld = R;
    }
    cb.dc = w.dc; cb.first = last ? 1 : 0;
    cb.gates = w.gates + r * 4 * R;
    cb.c_prev = w.c + r * R; cb.c_new = w.c + (size_t)(q + 1) * B * R;
    cb.B = B; cb.H = R; cb.dG = w.dG + r * 4 * R; cb.dg_ld = 4 * R;
    RN_TRY((cell::launch_bwd<T, T>(cb, st)));
    RN_TRY(gemm_partials<T>(w.dG + r * 4 * R, 4 * R, 0, w.Wrec, w.KX, 1, w.dXp, B, w.KX, 4 * R, w.pl_dx, st));
    attn::BwdArgs ab{};
    ab.dXp = w.dXp; ab.n_p = w.pl_dx.splits; ab.p_stride = (long long)B * w.KX; ab.p_ld = w.KX;
    ab.V = w.Hd + (size_t)l * B * H; ab.v_bs = H; ab.v_ts = (long long)NLd * B * H;
    ab.Wh = w.Wh + r * A; ab.Uv = w.Uv + (size_t)l * B * A; ab.uv_bs = A; ab.uv_ts = (long long)NLd * B * A;
    ab.attn_b = p.attn_b; ab.attn_w = p.attn_w; ab.B = B; ab.Tn = L; ab.A = A; ab.D = H; ab.inv_T = d.softmax ? 1.f : 1.f / L;
    ab.dWh_out = w.dWh + (size_t)t * B * A; ab.dWh_op = w.dWh_op + (size_t)t * B * A;          // summed over the NLd attentions of step t
    ab.dwh_acc = (l != NLd - 1) ? 1 : 0;
    ab.dUv_acc = w.dUv + (size_t)l * B * A; ab.uv_first = (t == S - 1) ? 1 : 0;
    ab.dw_first = last ? 1 : 0; ab.dw_acc = w.dw_acc;
    ab.dctx_out = w.dx + r * H; ab.de_out = nullptr; ab.alpha = d.softmax ? w.beta + r * L : nullptr;
    ab.p_drop = p_drop; ab.rng = rng; ab.site = SITE_LOCAL_X; ab.drop_base = (long long)r * H;
    RN_TRY((attn::launch_bwd<T, T>(ab, st)));
    if (l == 0 && t > 0) RN_TRY(gemm_partials<T>(w.dWh_op + (size_t)t * B * A, A, 0, w.Wa, R, 1, w.dQp, B, R, A, w.pl_dq, st));
  }
  // gradient wrt the decoder states: through U (keys) and through the weighted mean / softmax-weighted sum (values), layer by layer
  RN_TRY(misc::cast_pad<T>(w.dUv, A, w.dUv_op, A, (long long)L * NLd * B, A, A, st));
  RN_TRY(gemm_full<T>(w.dUv_op, A, 0, w.U, H, 1, g_hiddens, H, nullptr, L * NLd * B, H, A, 0, w.splitk2, st));
  for (int l = 0; l < NLd; ++l)
    RN_TRY(attn::launch_dv(w.beta, w.dx, g_hiddens + (size_t)l * B * H, H, (long long)NLd * B * H, S, B, L, H, d.softmax ? 1.f : 1.f / L,
                           1, NLd, l, st));
  if (phases & 2) RN_TRY(local_backward_weights<T>(d, w, g, st));
  return 0;
}

// ---- batched parameter gradients over the stashed operands, two streams (runtime.cuh:Side): the big recurrent / input weight
// gradients on `st`; the output projection and the 128-row attention gradients on the side stream
template <typename T>
static int local_backward_weights(const recnet_local_desc& d, const LocalWs<T>& w, const recnet_local_tensors& g, cudaStream_t st) {
  const int B = d.B, S = d.S, R = d.R, H = d.H, A = d.A, L = d.L, NLd = d.dec_layers < 1 ? 1 : d.dec_layers;
  const int SB = S * B, SpB = S * NLd * B;          // outer steps / pseudo-steps (with a stacked decoder: NLd per outer step)
  const bool is_gru = d.cell == RECNET_CELL_GRU;
  const int GR = w.G * R;
  const HRows<T> hr = h_rows(d, w);
  const T* dGh = is_gru ? w.dG2 : w.dG;
  // Column sums first: on a trainer's background lane they stay within the lane's CTA budget (misc.cuh) and the first ~60 us still run next
  // to the decoder's CE backward rather than its loop.
  cudaStream_t s2 = st;
  const bool lane = rn_background_ctas() > 0;   // on the lane: one capped GEMM at a time (the foreground loop's 512-thread, 128-register
  if (!lane) RN_TRY(side().fork(st, &s2));        // CTAs need SMs that are completely empty)
  RN_TRY(misc::colsum<T>(w.dG, GR, SpB, GR, g.b_ih, 0, w.splitk, st, is_gru ? nullptr : g.b_hh));    // LSTM: b_hh gets the same gradient
  if (is_gru) RN_TRY(misc::colsum<T>(dGh, GR, SpB, GR, g.b_hh, 0, w.splitk, st));
  RN_TRY(misc::colsum<T>(w.dOut, R, SB, R, g.out_b, 0, w.splitk2, s2));
  RN_TRY(misc::colsum<float>(w.dWh, A, SB, A, g.attn_b, 0, w.splitk2, s2));
  RN_TRY(misc::colsum<float>(w.dw_acc, A, B, A, g.attn_w, 0, w.splitk2, s2));
  RN_TRY(gemm_full<T>(w.dOut, R, 1, hr.out, hr.ld, 1, g.out_w, R, nullptr, R, R, SB, 0, w.splitk2, s2));
  RN_TRY(gemm_full<T>(w.dWh_op, A, 1, hr.query, hr.ld, 1, g.attn_W, R, nullptr, A, R, SB, 0, w.splitk2, s2));
  RN_TRY(gemm_full<T>(w.dUv_op, A, 1, w.Hd, H, 1, g.attn_U, H, nullptr, A, H, L * NLd * B, 0, w.splitk2, s2));
  RN_TRY(gemm_full<T>(w.dG, GR, 1, w.X, w.KX, 1, g.w_ih, H, nullptr, GR, H, SpB, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(dGh, GR, 1, w.X + H, w.KX, 1, g.w_hh, R, nullptr, GR, R, SpB, 0, w.splitk, st));
  if (!lane) RN_TRY(side().join(st, s2));
  return 0;
}

// ================================================ global ========================================================
template <typename T>
struct GlobalWs {
  int G;
  GemmPlan pl_gate, pl_dx;
  T *Wih, *Whh, *Wout; float* mp; T* Xg; float* Gx; T* X; float* P; T* gates; float* c; float* out; float* diff; float* partial;
  T* dOut; float* dHext; T* dG; T* dG2; float* dXp; float* dc; float* dXg; float* dmp; float* splitk;
  int* err;
  float* pXP; unsigned* psync;                    // weight-resident persistent loops (seq_recon_persist.cuh)
  size_t bytes;
};
constexpr int GMSE_THREADS = 256;

template <typename T>
static inline bool persist_global_ok(const recnet_global_desc& d, bool bwd) {
  if (!std::is_same<T, bf16>::value || d.cell != RECNET_CELL_LSTM) return false;
  static const int on = rn_env_int("RECNET_PERSIST_GLOBAL", 1);
  if (!on) return false;
  return bwd ? rp::global_bwd_ok(d.B, d.L, d.R) : rp::global_fwd_ok(d.B, d.L, d.R);
}

template <typename T>
static GlobalWs<T> plan_global(const recnet_global_desc& d, void* base) {
  GlobalWs<T> w;
  const int B = d.B, L = d.L, R = d.R, H = d.H;
  const bool gru_ = d.cell == RECNET_CELL_GRU;
  w.G = gru_ ? 3 : 4;
  w.pl_gate = plan_gemm<T>(B, w.G * R, R);
  w.pl_dx = plan_gemm<T>(B, R, w.G * R);
  Bump m(base);
  w.Wih = m.take<T>((size_t)4 * R * 2 * H);
  w.Whh = m.take<T>((size_t)4 * R * R);
  w.Wout = m.take<T>((size_t)R * R);
  w.mp = m.take<float>((size_t)B * H);
  w.Xg = m.take<T>((size_t)L * B * 2 * H);
  w.Gx = m.take<float>((size_t)L * B * 4 * R);
  w.X = m.take<T>((size_t)(L + 1) * B * R);
  w.P = m.take<float>((size_t)w.pl_gate.splits * B * 4 * R);
  w.gates = m.take<T>((size_t)L * B * 4 * R);
  w.c = m.take<float>((size_t)(L + 1) * B * R);
  w.out = m.take<float>((size_t)L * B * R);
  w.diff = m.take<float>((size_t)B * R);
  w.partial = m.take<float>((size_t)rn_cdiv((long long)B * R, GMSE_THREADS));
  w.dOut = m.take<T>((size_t)L * B * R);
  w.dHext = m.take<float>((size_t)L * B * R);
  w.dG = m.take<T>((size_t)L * B * 4 * R);
  w.dXp = m.take<float>((size_t)w.pl_dx.splits * B * R);
  w.dc = m.take<float>((size_t)B * R);
  w.dG2 = m.take<T>(gru_ ? (size_t)L * B * 3 * R : 1);
  w.dXg = m.take<float>((size_t)L * B * 2 * H);
  w.dmp = m.take<float>((size_t)B * H);
  w.splitk = m.take<float>(SPLITK_SCRATCH_FLOATS);
  w.err = m.take<int>(64);
  {
    size_t n = 4;
    if (persist_global_ok<T>(d, false)) n = (size_t)(R / rp::UNITS) * rp::pick_ks(R, 0) * B * rp::NCOL;
    if (persist_global_ok<T>(d, true)) { const size_t n2 = (size_t)(R / 128) * rp::pick_ns(R, 0) * B * 128; n = n2 > n ? n2 : n; }
    w.pXP = m.take<float>(n);
    w.psync = m.take<unsigned>(2 * rp::SYNC_WORDS);
  }
  w.bytes = m.off + 256;
  return w;
}
static inline int check_global(const recnet_global_desc& d) {
  if (d.B < 1 || d.L < 1 || d.T < 1) return RECNET_ERR_BAD_SHAPE;
  if (d.cell != RECNET_CELL_LSTM && d.cell != RECNET_CELL_GRU) return RECNET_ERR_UNSUPPORTED;
  const int al = d.precision == RECNET_PREC_BF16 ? 8 : 4;
  if (d.R % al || d.H % al) return RECNET_ERR_ALIGNMENT;
  return 0;
}

template <typename T>
static int global_forward(const recnet_global_desc& d, const recnet_global_tensors& p, const float* hiddens, const float* feats,
                          const unsigned long long* rng, void* ws, long long ws_bytes, float* loss_out, cudaStream_t st) {
  RN_TRY(check_global(d));
  GlobalWs<T> w = plan_global<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, L = d.L, R = d.R, H = d.H;
  const float p_drop = d.train ? d.p_drop : 0.f;
  const bool is_gru = d.cell == RECNET_CELL_GRU;
  const int GR = w.G * R;
  RN_TRY(misc::cast_pad<T>(p.w_ih, 2 * H, w.Wih, 2 * H, GR, 2 * H, 2 * H, st));
  RN_TRY(misc::cast_pad<T>(p.w_hh, R, w.Whh, R, GR, R, R, st));
  RN_TRY(misc::cast_pad<T>(p.out_w, R, w.Wout, R, R, R, R, st));
  // mean over time (and the single decoder layer), then / L * caption_max_len  (global_reconstructor.py:33-37)
  const long long n = (long long)B * H;
  const int NLd = d.dec_layers < 1 ? 1 : d.dec_layers;      // hiddens is (L, NLd, B, H); mean over time AND layers (global_reconstructor.py:33-36)
  misc::pool_time_kernel<<<rn_cdiv(n, 256), 256, 0, st>>>(hiddens, L * NLd, n, d.caption_max_len / ((float)L * NLd * L), w.mp);
  RN_LAUNCH_OK();
  misc::global_x_kernel<T><<<NUM_SMS * 4, 256, 0, st>>>(hiddens, w.mp, w.Xg, L, B, H, NLd, p_drop, rng, SITE_GLOBAL_MP);
  RN_LAUNCH_OK();
  RN_TRY(gemm_full<T>(w.Xg, 2 * H, 0, w.Wih, 2 * H, 0, w.Gx, GR, p.b_ih, L * B, GR, 2 * H, 0, w.splitk, st));
  RN_CUDA_OK(cudaMemsetAsync(w.X, 0, (size_t)B * R * sizeof(T), st));
  RN_CUDA_OK(cudaMemsetAsync(w.c, 0, (size_t)B * R * sizeof(float), st));
  RN_CUDA_OK(cudaMemsetAsync(w.err, 0, sizeof(int), st));
  bool persist = false;
  if constexpr (std::is_same<T, bf16>::value) {
    persist = persist_global_ok<T>(d, false);
    if (persist || persist_global_ok<T>(d, true)) RN_CUDA_OK(cudaMemsetAsync(w.psync, 0, 2 * rp::SYNC_WORDS * sizeof(unsigned), st));
    if (persist) {
      // ONE cooperative launch for all L steps, W_hh resident in shared memory (seq_recon_persist.cuh, global mode)
      rp::FwdParams fp{};
      fp.B = B; fp.S = L; fp.R = R; fp.H = 0; fp.A = 0; fp.L = 1; fp.inv_L = 1.f; fp.p_drop = 0.f;
      fp.X = w.X; fp.b_ih = p.b_ih; fp.b_hh = p.b_hh; fp.gates = w.gates; fp.c = w.c; fp.XP = w.pXP; fp.sync = w.psync; fp.err = w.err;
      fp.global_mode = 1; fp.Gx = w.Gx;
      RN_TRY(rp::launch_local_fwd(fp, w.Whh, false, st));
    }
  }
  for (int t = 0; t < L && !persist; ++t) {
    const size_t r = (size_t)t * B;
    T* x_t = w.X + r * R;
    int n_p = 0;
    if (t > 0) {
      RN_TRY(gemm_partials<T>(x_t, R, 0, w.Whh, R, 0, w.P, B, GR, R, w.pl_gate, st));
      n_p = w.pl_gate.splits;
    }
    if (is_gru) {
      gru::FwdArgs ga{};
      ga.Px = nullptr; ga.n_px = 0;
      ga.Ph = n_p ? w.P : nullptr; ga.n_ph = n_p; ga.ph_stride = (long long)B * 3 * R; ga.ph_ld = 3 * R;
      ga.Gx = w.Gx + r * 3 * R; ga.gx_ld = 3 * R; ga.b_ih = nullptr; ga.b_hh = p.b_hh;
      ga.h_prev = w.c + r * R; ga.hp_ld = R; ga.B = B; ga.H = R;
      ga.stash = w.gates + r * 4 * R; ga.h_out = w.c + (size_t)(t + 1) * B * R; ga.h_ld = R;
      ga.h_op = x_t + (size_t)B * R; ga.hop_ld = R;
      RN_TRY((gru::launch_fwd<T, T>(ga, st)));
      continue;
    }
    cell::FwdArgs ca{};
    ca.P = w.P; ca.n_p = n_p; ca.p_stride = (long long)B * 4 * R; ca.p_ld = 4 * R;
    ca.Gx = w.Gx + r * 4 * R; ca.gx_ld = 4 * R; ca.b1 = nullptr; ca.b2 = p.b_hh;
    ca.c_prev = w.c + r * R; ca.B = B; ca.H = R;
    ca.gates_out = w.gates + r * 4 * R; ca.c_out = w.c + (size_t)(t + 1) * B * R; ca.h_out = nullptr;
    ca.h_op = x_t + (size_t)B * R; ca.hop_ld = R; ca.h_op2 = nullptr;
    RN_TRY((cell::launch_fwd<T, T>(ca, st)));
  }
  RN_TRY(gemm_full<T>(w.X + (size_t)B * R, R, 0, w.Wout, R, 0, w.out, R, p.out_b, L * B, R, R, 0, w.splitk, st));
  if (loss_out) {
    const int nb = rn_cdiv((long long)B * R, GMSE_THREADS);
    loss::mse_global_diff_kernel<<<nb, GMSE_THREADS, 0, st>>>(w.out, L, feats, d.T, B, R, w.diff, w.partial);
    RN_LAUNCH_OK();
    loss::sum_kernel<<<1, 1024, 0, st>>>(w.partial, nb, loss_out, 1.f / ((float)B * R) / (float)L);
    RN_LAUNCH_OK();
  }
  return 0;
}

template <typename T>
static int global_backward(const recnet_global_desc& d, const recnet_global_tensors& p, const float* hiddens, const float* feats,
                           const unsigned long long* rng, void* ws, long long ws_bytes, const float* g_loss,
                           const recnet_global_tensors& g, float* g_hiddens, cudaStream_t st) {
  RN_TRY(check_global(d));
  GlobalWs<T> w = plan_global<T>(d, ws);
  if ((long long)w.bytes > ws_bytes) return RECNET_ERR_WORKSPACE;
  const int B = d.B, L = d.L, R = d.R, H = d.H;
  const float p_drop = d.train ? d.p_drop : 0.f;
  const int LB = L * B;
  // d loss / d out[t,b,r] = g * 2*diff/(B*R) * (1/L from the mean over t) * (1/L from train.py:100)
  loss::mse_global_bwd_kernel<T><<<NUM_SMS * 4, 256, 0, st>>>(w.diff, L, B, R, g_loss, 2.f / ((float)B * R) / ((float)L * L), w.dOut);
  RN_LAUNCH_OK();
  RN_TRY(gemm_full<T>(w.dOut, R, 0, w.Wout, R, 1, w.dHext, R, nullptr, LB, R, R, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dOut, R, 1, w.X + (size_t)B * R, R, 1, g.out_w, R, nullptr, R, R, LB, 0, w.splitk, st));
  RN_TRY(misc::colsum<T>(w.dOut, R, LB, R, g.out_b, 0, w.splitk, st));
  const bool is_gru = d.cell == RECNET_CELL_GRU;
  const int GR = w.G * R;
  bool persist = false;
  if constexpr (std::is_same<T, bf16>::value) {
    persist = persist_global_ok<T>(d, true);
    if (persist) {
      rp::BwdParams bp{};
      bp.B = B; bp.S = L; bp.R = R; bp.H = 0; bp.A = 0; bp.L = 1; bp.inv_L = 1.f; bp.p_drop = 0.f;
      bp.gates = w.gates; bp.c = w.c; bp.dHext = w.dHext; bp.dG = w.dG; bp.DP = w.pXP; bp.sync = w.psync + rp::SYNC_WORDS; bp.err = w.err;
      bp.global_mode = 1;
      RN_TRY(rp::launch_local_bwd(bp, w.Whh, st));
    }
  }
  for (int t = L - 1; t >= 0 && !persist; --t) {
    const bool last = (t == L - 1);
    const size_t r = (size_t)t * B;
    if (is_gru) {
      gru::BwdArgs gb{};
      gb.dh_ext = w.dHext + r * R; gb.dh_ld = R;
      gb.dHp = last ? nullptr : w.dXp; gb.n_p = w.pl_dx.splits; gb.p_stride = (long long)B * R; gb.p_ld = R;
      gb.dQp = nullptr; gb.carry = w.dc; gb.first = last ? 1 : 0;
      gb.stash = w.gates + r * 4 * R; gb.h_prev = w.c + r * R; gb.hp_ld = R;
      gb.B = B; gb.H = R; gb.dGi = w.dG + r * 3 * R; gb.dGh = w.dG2 + r * 3 * R; gb.dg_ld = 3 * R;
      RN_TRY((gru::launch_bwd<T, T>(gb, st)));
      if (t > 0) RN_TRY(gemm_partials<T>(w.dG2 + r * 3 * R, 3 * R, 0, w.Whh, R, 1, w.dXp, B, R, 3 * R, w.pl_dx, st));
      continue;
    }
    cell::BwdArgs cb{};
    cb.dh_ext = w.dHext + r * R; cb.dh_ld = R;
    cb.dXp = last ? nullptr : w.dXp; cb.n_p = w.pl_dx.splits; cb.p_stride = (long long)B * R; cb.p_ld = R; cb.col0 = 0;
    cb.dQp = nullptr; cb.dc = w.dc; cb.first = last ? 1 : 0;
    cb.gates = w.gates + r * 4 * R;
    cb.c_prev = w.c + r * R; cb.c_new = w.c + (size_t)(t + 1) * B * R;
    cb.B = B; cb.H = R; cb.dG = w.dG + r * 4 * R; cb.dg_ld = 4 * R;
    RN_TRY((cell::launch_bwd<T, T>(cb, st)));
    if (t > 0) RN_TRY(gemm_partials<T>(w.dG + r * 4 * R, 4 * R, 0, w.Whh, R, 1, w.dXp, B, R, 4 * R, w.pl_dx, st));
  }
  const T* dGh = is_gru ? w.dG2 : w.dG;
  RN_TRY(misc::colsum<T>(w.dG, GR, LB, GR, g.b_ih, 0, w.splitk, st));
  if (is_gru) { RN_TRY(misc::colsum<T>(dGh, GR, LB, GR, g.b_hh, 0, w.splitk, st)); }
  else RN_CUDA_OK(cudaMemcpyAsync(g.b_hh, g.b_ih, (size_t)GR * sizeof(float), cudaMemcpyDeviceToDevice, st));
  RN_TRY(gemm_full<T>(dGh, GR, 1, w.X, R, 1, g.w_hh, R, nullptr, GR, R, LB, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dG, GR, 1, w.Xg, 2 * H, 1, g.w_ih, 2 * H, nullptr, GR, 2 * H, LB, 0, w.splitk, st));
  RN_TRY(gemm_full<T>(w.dG, GR, 0, w.Wih, 2 * H, 1, w.dXg, 2 * H, nullptr, LB, 2 * H, GR, 0, w.splitk, st));
  const long long n = (long long)B * H;
  const int NLd = d.dec_layers < 1 ? 1 : d.dec_layers;
  misc::global_x_bwd_kernel<<<rn_cdiv(n, 256), 256, 0, st>>>(w.dXg, g_hiddens, w.dmp, L, B, H, NLd, 0, p_drop, rng, SITE_GLOBAL_MP);
  RN_LAUNCH_OK();
  misc::pool_time_bwd_kernel<<<rn_cdiv(n, 256), 256, 0, st>>>(w.dmp, L * NLd, n, d.caption_max_len / ((float)L * NLd * L), g_hiddens, 1);
  RN_LAUNCH_OK();
  return 0;
}
}  // namespace rec
