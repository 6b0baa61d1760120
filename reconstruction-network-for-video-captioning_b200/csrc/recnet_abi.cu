// extern "C" entry points of librecnet_b200.so (declared in include/recnet_b200.h).
#include "runtime.cuh"
#include "seq_decoder.cuh"
#include "seq_decoder_pf.cuh"
#include "seq_recon.cuh"
#include "optim.cuh"
#include "allreduce.cuh"
#include "cider.cuh"

#define ST(s) reinterpret_cast<cudaStream_t>(s)

// f(float{}) or f(bf16{}) by precision -- the generic lambda takes `using T = decltype(t)` -- and `bad` for any other precision.
template <typename R, typename F>
static R by_prec(int precision, R bad, F&& f) {
  if (precision == RECNET_PREC_FP32) return f(float{});
  if (precision == RECNET_PREC_BF16) return f(bf16{});
  return bad;
}

// Every entry point that takes a descriptor checks it here: a null descriptor is RECNET_ERR_BAD_SHAPE, an unknown precision
// RECNET_ERR_UNSUPPORTED (the pointer accessors return nullptr for both).
template <typename Pub>
static int check_desc(const Pub* d) {
  if (!d) return RECNET_ERR_BAD_SHAPE;
  return by_prec<int>(d->precision, RECNET_ERR_UNSUPPORTED, [](auto) { return 0; });
}
// The decoder and local descriptors also carry RECNET_ATTN_SOFTMAX in their `cell` field; it is split off here, once.
template <typename Pub, typename Int>
static int split_desc(const Pub* d, Int* out) {
  RN_TRY(check_desc(d));
  static_cast<Pub&>(*out) = *d;
  const int32_t flags = d->cell & ~RECNET_CELL_MASK;
  if (flags & ~RECNET_ATTN_SOFTMAX) return RECNET_ERR_UNSUPPORTED;
  out->cell = d->cell & RECNET_CELL_MASK;
  out->softmax = flags != 0;
  return 0;
}

// The workspace layout of the decoder's training drivers: the projected-feature plan, or the general plan (single-layer and stacked).
struct DecLayout { int64_t bytes; float* logits; int64_t ld; int* err; };
template <typename T>
static DecLayout dec_layout(const DecDesc& dd, void* base) {
  if (dec::dec_path(dd) == dec::DecPath::PF) {
    const auto w = dec::plan_pf<T>(dd, base);
    return {(int64_t)w.bytes, w.logits, w.Vld, w.err};
  }
  const auto w = dec::plan<T>(dd, base);
  return {(int64_t)w.bytes, w.logits, w.Vld, w.err};
}

extern "C" {

int recnet_abi_version(void) { return 1; }

long long recnet_launch_count(void) { return prof_state().launches; }

int recnet_profile_enable(int on, int max_records) {
  ProfState& p = prof_state();
  if (on) {
    if (max_records > p.cap) {
      ProfRecord* r = new ProfRecord[max_records]();
      for (int i = 0; i < p.cap; ++i) r[i] = p.rec[i];
      delete[] p.rec;
      p.rec = r; p.cap = max_records;
    }
    p.n = 0;
  }
  p.enabled = on;
  return 0;
}

// out: [n][5] floats = (class, M, N, K, milliseconds); returns the number of records written (after a device sync)
int recnet_profile_collect(float* out, int max_records) {
  ProfState& p = prof_state();
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return -(int)e;
  const int n = p.n < max_records ? p.n : max_records;
  for (int i = 0; i < n; ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, p.rec[i].e0, p.rec[i].e1);
    out[5 * i + 0] = (float)p.rec[i].cls; out[5 * i + 1] = (float)p.rec[i].M; out[5 * i + 2] = (float)p.rec[i].N;
    out[5 * i + 3] = (float)p.rec[i].K; out[5 * i + 4] = ms;
  }
  p.n = 0;
  return n;
}

// developer / test probe: the inverted-dropout scales (0 or 1/(1-p)) the kernels apply to elements 0..n-1 of dropout `site`
// for the (seed, offset) pair in rng -- the same device function the forward and backward kernels call
__global__ void debug_dropout_mask_kernel(const unsigned long long* rng, unsigned int site, long long n, float p, float* out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = dropout_scale(rng, site, (uint64_t)i, p);
}
int recnet_debug_dropout_mask(const uint64_t* rng, uint32_t site, int64_t n, float p, float* out, void* stream) {
  if (n <= 0) return 0;
  if (!rng || !out) return RECNET_ERR_BAD_SHAPE;
  const int blocks = (int)((n + 255) / 256 > 148 * 16 ? 148 * 16 : (n + 255) / 256);
  debug_dropout_mask_kernel<<<blocks, 256, 0, ST(stream)>>>(reinterpret_cast<const unsigned long long*>(rng), site, (long long)n, p, out);
  RN_LAUNCH_OK();
  return 0;
}
int recnet_debug_set_timeline(void* buf) {
  unsigned long long* p = reinterpret_cast<unsigned long long*>(buf);
  unsigned int zero = 0;
  RN_CUDA_OK(cudaMemcpyToSymbol(g_timeline_n, &zero, sizeof(zero)));
  RN_CUDA_OK(cudaMemcpyToSymbol(g_timeline, &p, sizeof(p)));
  return 0;
}

int recnet_query_device(int device, int* sm_count, int* cc_major, int* cc_minor) {
  cudaDeviceProp prop;
  RN_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  if (prop.major != 10) return RECNET_ERR_UNSUPPORTED_ARCH;
  return 0;
}

int recnet_gemm(int precision, const void* A, int64_t lda, int transA, const void* B, int64_t ldb, int transB, float* C,
                int64_t ldc, void* c_op, int64_t ldc_op, const float* bias, int M, int N, int K, int splits,
                int64_t split_stride, int accumulate, int bn_hint, void* stream) {
  return by_prec<int>(precision, RECNET_ERR_UNSUPPORTED, [&](auto t) -> int {
    using T = decltype(t);
    if constexpr (std::is_same<T, float>::value) {
      if (c_op) return RECNET_ERR_UNSUPPORTED;
      return sg::launch(reinterpret_cast<const float*>(A), lda, transA, reinterpret_cast<const float*>(B), ldb, transB, C, ldc,
                        bias, M, N, K, splits, split_stride, accumulate, ST(stream));
    } else {
      return tc::launch(reinterpret_cast<const bf16*>(A), lda, transA, reinterpret_cast<const bf16*>(B), ldb, transB, C, ldc,
                        reinterpret_cast<bf16*>(c_op), ldc_op, bias, M, N, K, splits, split_stride, accumulate, bn_hint,
                        ST(stream));
    }
  });
}

int recnet_plan_persistent_loops(const recnet_local_desc* d, int32_t* out) {
  // out[0..5]  forward : covered?, K-splits, unit groups, resident k-blocks per CTA, activation ring stages, CTAs
  // out[6..11] backward: covered?, gate-row splits, column groups, resident k-blocks per CTA, ring stages, CTAs
  if (!d || !out) return RECNET_ERR_BAD_SHAPE;
  for (int i = 0; i < 12; ++i) out[i] = 0;
  LocalDesc dd;
  RN_TRY(split_desc(d, &dd));            // both attention variants have persistent loops
  if (dd.precision != RECNET_PREC_BF16) return 0;
  const rp::Shape s{dd.B, dd.S, dd.R, dd.H, dd.A, dd.L};
  if (rec::persist_fwd_ok<bf16>(dd)) {
    const int ks = rp::pick_ks(s.R, s.H), res = rp::max_res_kb_fwd(s.R, s.H, ks);
    out[0] = 1; out[1] = ks; out[2] = s.R / rp::UNITS; out[3] = res; out[4] = rp::pick_stages_fwd(s.B, ks, res); out[5] = out[2] * ks;
  }
  if (rec::persist_bwd_ok<bf16>(dd)) {
    const int ns = rp::pick_ns(s.R, s.H), res = (4 * s.R / rp::BK + ns - 1) / ns;
    out[6] = 1; out[7] = ns; out[8] = (s.R + s.H) / 128; out[9] = res; out[10] = rp::pick_stages_bwd(s.B, res); out[11] = out[8] * ns;
  }
  return 0;
}
int recnet_plan_batched_gemm(int precision, int M, int N, int K, int32_t* bn_out, int32_t* splits_out) {
  if (M <= 0 || N <= 0 || K <= 0 || !bn_out || !splits_out) return RECNET_ERR_BAD_SHAPE;
  rt::GemmPlan p = precision == RECNET_PREC_BF16 ? rt::plan_gemm_full<bf16>(M, N, K) : rt::plan_gemm_full<float>(M, N, K);
  *bn_out = p.bn;
  *splits_out = p.splits;
  return 0;
}
int recnet_splitk_reduce(const float* partial, int splits, int64_t split_stride, int64_t ldp, float* out, int64_t ldo, int M,
                         int N, int accumulate, void* stream) {
  return rt::splitk_reduce(partial, splits, split_stride, ldp, out, ldo, M, N, nullptr, accumulate, ST(stream));
}

int recnet_attn_fwd(int precision, const float* wh_partials, int n_wh, int64_t wh_stride, const float* uv, int64_t uv_bs,
                    int64_t uv_ts, const float* attn_b, const float* attn_w, const void* v, int64_t v_bs, int64_t v_ts, int B,
                    int Tn, int A, int D, int normalize, float* wh_out, float* e_out, void* ctx_out, int64_t ctx_ld,
                    float p_drop, const uint64_t* rng, uint32_t site, int64_t drop_base, void* stream) {
  attn::FwdArgs a{};
  a.WhP = wh_partials; a.n_whp = n_wh; a.whp_stride = wh_stride; a.Uv = uv; a.uv_bs = uv_bs; a.uv_ts = uv_ts;
  a.attn_b = attn_b; a.attn_w = attn_w; a.V = v; a.v_bs = v_bs; a.v_ts = v_ts; a.B = B; a.Tn = Tn; a.A = A; a.D = D;
  a.inv_T = 1.f / Tn; a.normalize = normalize; a.Wh_out = wh_out; a.e_out = e_out; a.ctx_out = ctx_out; a.ctx_ld = ctx_ld;
  a.p_drop = p_drop; a.rng = reinterpret_cast<const unsigned long long*>(rng); a.site = site; a.drop_base = drop_base;
  return by_prec<int>(precision, RECNET_ERR_UNSUPPORTED, [&](auto t) { using T = decltype(t); return attn::launch_fwd<T, T>(a, ST(stream)); });
}

// the backward of both attention variants: the reference's mean (alpha = nullptr, context scaled by 1/Tn) and the softmax (alpha, scale 1)
static int attn_bwd(int precision, const float* dctx_partials, int n_p, int64_t p_stride, int64_t p_ld, const void* v, int64_t v_bs,
                    int64_t v_ts, const float* alpha, float inv_T, const float* wh, const float* uv, int64_t uv_bs, int64_t uv_ts,
                    const float* attn_b, const float* attn_w, int B, int Tn, int A, int D, float* dwh_out, void* dwh_op, float* duv_acc,
                    float* dw_acc, int first, float* dctx_out, float p_drop, const uint64_t* rng, uint32_t site, int64_t drop_base,
                    void* stream) {
  attn::BwdArgs a{};
  a.dXp = dctx_partials; a.n_p = n_p; a.p_stride = p_stride; a.p_ld = p_ld; a.V = v; a.v_bs = v_bs; a.v_ts = v_ts;
  a.Wh = wh; a.Uv = uv; a.uv_bs = uv_bs; a.uv_ts = uv_ts; a.attn_b = attn_b; a.attn_w = attn_w; a.B = B; a.Tn = Tn; a.A = A;
  a.D = D; a.inv_T = inv_T; a.dWh_out = dwh_out; a.dWh_op = dwh_op; a.dUv_acc = duv_acc; a.uv_first = first; a.dw_first = first; a.dw_acc = dw_acc;
  a.dctx_out = dctx_out; a.de_out = nullptr; a.alpha = alpha; a.p_drop = p_drop; a.rng = reinterpret_cast<const unsigned long long*>(rng);
  a.site = site; a.drop_base = drop_base;
  return by_prec<int>(precision, RECNET_ERR_UNSUPPORTED, [&](auto t) { using T = decltype(t); return attn::launch_bwd<T, T>(a, ST(stream)); });
}
int recnet_attn_bwd(int precision, const float* dctx_partials, int n_p, int64_t p_stride, int64_t p_ld, const void* v,
                    int64_t v_bs, int64_t v_ts, const float* wh, const float* uv, int64_t uv_bs, int64_t uv_ts,
                    const float* attn_b, const float* attn_w, int B, int Tn, int A, int D, float* dwh_out, void* dwh_op,
                    float* duv_acc, float* dw_acc, int first, float* dctx_out, float p_drop, const uint64_t* rng,
                    uint32_t site, int64_t drop_base, void* stream) {
  return attn_bwd(precision, dctx_partials, n_p, p_stride, p_ld, v, v_bs, v_ts, nullptr, 1.f / Tn, wh, uv, uv_bs, uv_ts, attn_b, attn_w,
                  B, Tn, A, D, dwh_out, dwh_op, duv_acc, dw_acc, first, dctx_out, p_drop, rng, site, drop_base, stream);
}

int recnet_attn_bwd_softmax(int precision, const float* dctx_partials, int n_p, int64_t p_stride, int64_t p_ld, const void* v,
                            int64_t v_bs, int64_t v_ts, const float* alpha, const float* wh, const float* uv, int64_t uv_bs,
                            int64_t uv_ts, const float* attn_b, const float* attn_w, int B, int Tn, int A, int D, float* dwh_out,
                            void* dwh_op, float* duv_acc, float* dw_acc, int first, float* dctx_out, float p_drop,
                            const uint64_t* rng, uint32_t site, int64_t drop_base, void* stream) {
  if (!alpha) return RECNET_ERR_BAD_SHAPE;
  return attn_bwd(precision, dctx_partials, n_p, p_stride, p_ld, v, v_bs, v_ts, alpha, 1.f, wh, uv, uv_bs, uv_ts, attn_b, attn_w,
                  B, Tn, A, D, dwh_out, dwh_op, duv_acc, dw_acc, first, dctx_out, p_drop, rng, site, drop_base, stream);
}

int recnet_lstm_cell_fwd(int precision, const float* partials, int n_p, int64_t p_stride, int64_t p_ld, const float* gx,
                         int64_t gx_ld, const float* b1, const float* b2, const float* c_prev, int B, int H, void* gates_out,
                         float* c_out, float* h_out, int64_t h_ld, void* h_op, int64_t hop_ld, void* h_op2, int64_t hop2_ld,
                         void* stream) {
  cell::FwdArgs a{};
  a.P = partials; a.n_p = n_p; a.p_stride = p_stride; a.p_ld = p_ld; a.Gx = gx; a.gx_ld = gx_ld; a.b1 = b1; a.b2 = b2;
  a.c_prev = c_prev; a.B = B; a.H = H; a.gates_out = gates_out; a.c_out = c_out; a.h_out = h_out; a.h_ld = h_ld;
  a.h_op = h_op; a.hop_ld = hop_ld; a.h_op2 = h_op2; a.hop2_ld = hop2_ld;
  return by_prec<int>(precision, RECNET_ERR_UNSUPPORTED, [&](auto t) { using T = decltype(t); return cell::launch_fwd<T, T>(a, ST(stream)); });
}

int recnet_lstm_cell_bwd(int precision, const float* dh_ext, int64_t dh_ld, const float* dh_scale, const float* dh_ext2,
                         int64_t dh2_ld, const float* dxp, int n_p, int64_t p_stride, int64_t p_ld, int col0, const float* dqp,
                         int n_q, int64_t q_stride, int64_t q_ld, float* dc, int first, const void* gates, const float* c_prev,
                         const float* c_new, int B, int H, void* dg_out, int64_t dg_ld, void* stream) {
  cell::BwdArgs a{};
  a.dh_ext = dh_ext; a.dh_ld = dh_ld; a.dh_scale = dh_scale; a.dh_ext2 = dh_ext2; a.dh2_ld = dh2_ld; a.dXp = dxp; a.n_p = n_p;
  a.p_stride = p_stride; a.p_ld = p_ld; a.col0 = col0; a.dQp = dqp; a.n_q = n_q; a.q_stride = q_stride; a.q_ld = q_ld; a.dc = dc; a.first = first; a.gates = gates;
  a.c_prev = c_prev; a.c_new = c_new; a.B = B; a.H = H; a.dG = dg_out; a.dg_ld = dg_ld;
  return by_prec<int>(precision, RECNET_ERR_UNSUPPORTED, [&](auto t) { using T = decltype(t); return cell::launch_bwd<T, T>(a, ST(stream)); });
}

int recnet_gru_cell_fwd(int precision, const float* px, int n_px, int64_t px_stride, int64_t px_ld, const float* ph, int n_ph,
                        int64_t ph_stride, int64_t ph_ld, const float* gx, int64_t gx_ld, const float* b_ih, const float* b_hh,
                        const float* h_prev, int64_t hp_ld, int B, int H, void* stash, float* h_out, int64_t h_ld, void* h_op,
                        int64_t hop_ld, void* stream) {
  gru::FwdArgs a{};
  a.Px = px; a.n_px = n_px; a.px_stride = px_stride; a.px_ld = px_ld; a.Ph = ph; a.n_ph = n_ph; a.ph_stride = ph_stride; a.ph_ld = ph_ld;
  a.Gx = gx; a.gx_ld = gx_ld; a.b_ih = b_ih; a.b_hh = b_hh; a.h_prev = h_prev; a.hp_ld = hp_ld; a.B = B; a.H = H; a.stash = stash;
  a.h_out = h_out; a.h_ld = h_ld; a.h_op = h_op; a.hop_ld = hop_ld;
  return by_prec<int>(precision, RECNET_ERR_UNSUPPORTED, [&](auto t) { using T = decltype(t); return gru::launch_fwd<T, T>(a, ST(stream)); });
}

int recnet_gru_cell_bwd(int precision, const float* dh_ext, int64_t dh_ld, const float* dh_ext2, int64_t dh2_ld, const float* dhp,
                        int n_p, int64_t p_stride, int64_t p_ld, const float* dqp, int n_q, int64_t q_stride, int64_t q_ld,
                        float* carry, int first, const void* stash, const float* h_prev, int64_t hp_ld, int B, int H, void* dgi,
                        void* dgh, int64_t dg_ld, void* stream) {
  gru::BwdArgs a{};
  a.dh_ext = dh_ext; a.dh_ld = dh_ld; a.dh_ext2 = dh_ext2; a.dh2_ld = dh2_ld; a.dHp = dhp; a.n_p = n_p; a.p_stride = p_stride; a.p_ld = p_ld;
  a.dQp = dqp; a.n_q = n_q; a.q_stride = q_stride; a.q_ld = q_ld; a.carry = carry; a.first = first; a.stash = stash; a.h_prev = h_prev;
  a.hp_ld = hp_ld; a.B = B; a.H = H; a.dGi = dgi; a.dGh = dgh; a.dg_ld = dg_ld;
  return by_prec<int>(precision, RECNET_ERR_UNSUPPORTED, [&](auto t) { using T = decltype(t); return gru::launch_bwd<T, T>(a, ST(stream)); });
}

// ---- decoder ---------------------------------------------------------------------------------------------------
int64_t recnet_decoder_workspace_bytes(const recnet_decoder_desc* d) {
  DecDesc dd;
  RN_TRY(split_desc(d, &dd));
  return by_prec<int64_t>(dd.precision, RECNET_ERR_UNSUPPORTED, [&](auto t) { return dec_layout<decltype(t)>(dd, nullptr).bytes; });
}
int recnet_decoder_fwd(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats, const int64_t* tokens_in,
                       const int64_t* targets, const float* ce_weight, const uint64_t* rng, void* workspace,
                       int64_t workspace_bytes, float* hiddens, float* ce_out, void* stream) {
  return recnet_decoder_fwd_phase(d, w, feats, tokens_in, targets, ce_weight, rng, workspace, workspace_bytes, hiddens, ce_out, 3, stream);
}
int recnet_decoder_fwd_phase(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats, const int64_t* tokens_in,
                             const int64_t* targets, const float* ce_weight, const uint64_t* rng, void* workspace,
                             int64_t workspace_bytes, float* hiddens, float* ce_out, int phases, void* stream) {
  DecDesc dd;
  RN_TRY(split_desc(d, &dd));
  if (phases < 1 || phases > 3) return RECNET_ERR_BAD_SHAPE;
  const dec::DecPath path = dec::dec_path(dd);
  if (path != dec::DecPath::PF && !(phases & 1)) return 0;          // not split on these paths: everything belongs to bit 0
  const long long* ti = reinterpret_cast<const long long*>(tokens_in);
  const long long* tg = reinterpret_cast<const long long*>(targets);
  const unsigned long long* r = reinterpret_cast<const unsigned long long*>(rng);
  return by_prec<int>(dd.precision, RECNET_ERR_UNSUPPORTED, [&](auto t) {
    using T = decltype(t);
    switch (path) {
      case dec::DecPath::PF:
        return dec::forward_pf<T>(dd, *w, feats, ti, tg, ce_weight, r, workspace, workspace_bytes, hiddens, ce_out, ST(stream), phases);
      default:
        return dec::forward<T>(dd, *w, feats, ti, tg, ce_weight, r, workspace, workspace_bytes, hiddens, ce_out, ST(stream));
    }
  });
}
int recnet_decoder_bwd(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats, const int64_t* tokens_in,
                       const int64_t* targets, const float* ce_weight, const uint64_t* rng, void* workspace,
                       int64_t workspace_bytes, const float* g_ce, const float* g_hiddens, const float* hiddens,
                       const recnet_decoder_tensors* grads, void* stream) {
  return recnet_decoder_bwd_phase(d, w, feats, tokens_in, targets, ce_weight, rng, workspace, workspace_bytes, g_ce, g_hiddens, hiddens,
                                  grads, 15, stream);
}
int recnet_decoder_bwd_phase(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats, const int64_t* tokens_in,
                             const int64_t* targets, const float* ce_weight, const uint64_t* rng, void* workspace,
                             int64_t workspace_bytes, const float* g_ce, const float* g_hiddens, const float* hiddens,
                             const recnet_decoder_tensors* grads, int phases, void* stream) {
  DecDesc dd;
  RN_TRY(split_desc(d, &dd));
  if (phases < 1 || phases > 15) return RECNET_ERR_BAD_SHAPE;
  const dec::DecPath path = dec::dec_path(dd);
  if (path != dec::DecPath::PF && !(phases & 1)) return 0;          // not split on these paths: everything belongs to bit 0
  const long long* ti = reinterpret_cast<const long long*>(tokens_in);
  const long long* tg = reinterpret_cast<const long long*>(targets);
  const unsigned long long* r = reinterpret_cast<const unsigned long long*>(rng);
  return by_prec<int>(dd.precision, RECNET_ERR_UNSUPPORTED, [&](auto t) {
    using T = decltype(t);
    switch (path) {
      case dec::DecPath::PF:
        return dec::backward_pf<T>(dd, *w, feats, ti, tg, ce_weight, r, workspace, workspace_bytes, g_ce, g_hiddens, *grads, ST(stream),
                                   phases);
      default:
        return dec::backward<T>(dd, *w, feats, ti, tg, ce_weight, r, workspace, workspace_bytes, g_ce, g_hiddens, hiddens, *grads,
                                ST(stream));
    }
  });
}
int recnet_decoder_bwd_is_split(const recnet_decoder_desc* d) {
  DecDesc dd;
  if (split_desc(d, &dd)) return 0;
  return dec::dec_path(dd) == dec::DecPath::PF ? 1 : 0;
}
float* recnet_decoder_logits(const recnet_decoder_desc* d, void* workspace, int64_t* ld) {
  DecDesc dd;
  if (split_desc(d, &dd)) return nullptr;
  return by_prec<float*>(dd.precision, nullptr, [&](auto t) {
    const DecLayout w = dec_layout<decltype(t)>(dd, workspace);
    if (ld) *ld = w.ld;
    return w.logits;
  });
}
int64_t recnet_greedy_workspace_bytes(const recnet_decoder_desc* d) {
  DecDesc dd;
  RN_TRY(split_desc(d, &dd));
  return by_prec<int64_t>(dd.precision, RECNET_ERR_UNSUPPORTED, [&](auto t) {
    using T = decltype(t);
    const int64_t a = (int64_t)dec::plan_greedy<T>(dd, nullptr, 64).bytes;
    if constexpr (std::is_same<T, bf16>::value) {      // room for either bf16 driver: recnet_decoder_greedy picks one per call
      const int64_t b = dec::greedy_pf_ok(dd) ? (int64_t)dec::plan_greedy_pf<bf16>(dd, nullptr, 64).bytes : 0;
      return a > b ? a : b;
    }
    return a;
  });
}
int recnet_decoder_greedy(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats, int max_steps,
                          void* workspace, int64_t workspace_bytes, int64_t* ids_out, int32_t* n_steps_out, void* stream) {
  DecDesc dd;
  RN_TRY(split_desc(d, &dd));
  if (max_steps < 1 || max_steps > 64) return RECNET_ERR_BAD_SHAPE;
  long long* ids = reinterpret_cast<long long*>(ids_out);
  return by_prec<int>(dd.precision, RECNET_ERR_UNSUPPORTED, [&](auto t) {
    using T = decltype(t);
    if constexpr (std::is_same<T, bf16>::value) {
      DecDesc d1 = dd; d1.L = 1; d1.train = 0;
      // softmax decoders keep dec::greedy: moving them onto greedy_pf changes their launches and needs its own measurement
      if (dec::greedy_pf_ok(d1) && !dd.softmax)      // projected-feature kernels, 4 launches per step
        return dec::greedy_pf(dd, *w, feats, max_steps, workspace, workspace_bytes, ids, n_steps_out, ST(stream));
    }
    return dec::greedy<T>(dd, *w, feats, max_steps, workspace, workspace_bytes, ids, n_steps_out, ST(stream));
  });
}

// byte offset of the loop kernel's int32 error flag inside the workspace (0 = ok, 2 = mbarrier timeout, 3 = grid-barrier timeout)
int64_t recnet_decoder_error_offset(const recnet_decoder_desc* d) {
  DecDesc dd;
  RN_TRY(split_desc(d, &dd));
  uint8_t* base = reinterpret_cast<uint8_t*>(4096);
  return by_prec<int64_t>(dd.precision, RECNET_ERR_UNSUPPORTED,
                          [&](auto t) { return reinterpret_cast<uint8_t*>(dec_layout<decltype(t)>(dd, base).err) - base; });
}
int64_t recnet_local_error_offset(const recnet_local_desc* d) {
  LocalDesc dd;
  RN_TRY(split_desc(d, &dd));
  uint8_t* base = reinterpret_cast<uint8_t*>(4096);
  return by_prec<int64_t>(dd.precision, RECNET_ERR_UNSUPPORTED,
                          [&](auto t) { return reinterpret_cast<uint8_t*>(rec::plan_local<decltype(t)>(dd, base).err) - base; });
}
int64_t recnet_global_error_offset(const recnet_global_desc* d) {
  RN_TRY(check_desc(d));
  uint8_t* base = reinterpret_cast<uint8_t*>(4096);
  return by_prec<int64_t>(d->precision, RECNET_ERR_UNSUPPORTED,
                          [&](auto t) { return reinterpret_cast<uint8_t*>(rec::plan_global<decltype(t)>(*d, base).err) - base; });
}

int64_t recnet_beam_workspace_bytes(const recnet_decoder_desc* d, int beam_width, int max_steps) {
  DecDesc dd;
  RN_TRY(split_desc(d, &dd));
  if (beam_width < 1 || beam_width > dec::BEAM_MAX_K || max_steps < 1 || max_steps > 64) return RECNET_ERR_BAD_SHAPE;
  return by_prec<int64_t>(dd.precision, RECNET_ERR_UNSUPPORTED,
                          [&](auto t) { return (int64_t)dec::plan_beam<decltype(t)>(dd, nullptr, beam_width, max_steps).bytes; });
}
int recnet_decoder_beam(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats_tiled, int beam_width, int max_steps,
                        int64_t eos_id, void* workspace, int64_t workspace_bytes, int64_t* seq_out, int32_t* n_steps_out, void* stream) {
  DecDesc dd;
  RN_TRY(split_desc(d, &dd));
  return by_prec<int>(dd.precision, RECNET_ERR_UNSUPPORTED, [&](auto t) {
    return dec::beam<decltype(t)>(dd, *w, feats_tiled, beam_width, max_steps, (long long)eos_id, workspace, workspace_bytes,
                                  reinterpret_cast<long long*>(seq_out), n_steps_out, ST(stream));
  });
}

int64_t recnet_sample_workspace_bytes(const recnet_decoder_desc* d, int max_steps) {
  DecDesc dd;
  RN_TRY(split_desc(d, &dd));
  DecDesc d1 = dd; d1.L = 1;
  RN_TRY(dec::check(d1));
  if (max_steps < 1 || max_steps > 64) return RECNET_ERR_BAD_SHAPE;
  return by_prec<int64_t>(dd.precision, RECNET_ERR_UNSUPPORTED,
                          [&](auto t) { return (int64_t)dec::plan_sample<decltype(t)>(dd, nullptr, max_steps).bytes; });
}
int recnet_decoder_sample(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats, int max_steps,
                          float temperature, int64_t eos_id, const unsigned long long* rng, const unsigned long long* noise,
                          void* workspace, int64_t workspace_bytes, int64_t* ids_out, float* logp_out, int32_t* lengths_out,
                          int32_t* n_steps_out, void* stream) {
  DecDesc dd;
  RN_TRY(split_desc(d, &dd));
  return by_prec<int>(dd.precision, RECNET_ERR_UNSUPPORTED, [&](auto t) {
    return dec::sample<decltype(t)>(dd, *w, feats, max_steps, temperature, (long long)eos_id, rng, noise, workspace, workspace_bytes,
                                    reinterpret_cast<long long*>(ids_out), logp_out, lengths_out, n_steps_out, ST(stream));
  });
}

// ---- local reconstructor ---------------------------------------------------------------------------------------
int64_t recnet_local_workspace_bytes(const recnet_local_desc* d) {
  LocalDesc dd;
  RN_TRY(split_desc(d, &dd));
  return by_prec<int64_t>(dd.precision, RECNET_ERR_UNSUPPORTED,
                          [&](auto t) { return (int64_t)rec::plan_local<decltype(t)>(dd, nullptr).bytes; });
}
int recnet_local_fwd(const recnet_local_desc* d, const recnet_local_tensors* w, const float* hiddens, const float* feats,
                     const uint64_t* rng, void* workspace, int64_t workspace_bytes, float* mse_out, void* stream) {
  LocalDesc dd;
  RN_TRY(split_desc(d, &dd));
  const unsigned long long* r = reinterpret_cast<const unsigned long long*>(rng);
  return by_prec<int>(dd.precision, RECNET_ERR_UNSUPPORTED, [&](auto t) {
    using T = decltype(t);
    return rec::local_forward<T>(dd, *w, hiddens, feats, r, workspace, workspace_bytes, mse_out, ST(stream));
  });
}
int recnet_local_bwd(const recnet_local_desc* d, const recnet_local_tensors* w, const float* hiddens, const float* feats,
                     const uint64_t* rng, void* workspace, int64_t workspace_bytes, const float* g_mse,
                     const recnet_local_tensors* grads, float* g_hiddens, void* stream) {
  return recnet_local_bwd_phase(d, w, hiddens, feats, rng, workspace, workspace_bytes, g_mse, grads, g_hiddens, 3, stream);
}
int recnet_local_bwd_phase(const recnet_local_desc* d, const recnet_local_tensors* w, const float* hiddens, const float* feats,
                           const uint64_t* rng, void* workspace, int64_t workspace_bytes, const float* g_mse,
                           const recnet_local_tensors* grads, float* g_hiddens, int phases, void* stream) {
  LocalDesc dd;
  RN_TRY(split_desc(d, &dd));
  if (phases < 1 || phases > 3) return RECNET_ERR_BAD_SHAPE;
  if (dd.dec_layers > 1) {                              // stacked decoders: not split -- everything belongs to phase bit 0
    if (!(phases & 1)) return 0;
    phases = 3;
  }
  const unsigned long long* r = reinterpret_cast<const unsigned long long*>(rng);
  return by_prec<int>(dd.precision, RECNET_ERR_UNSUPPORTED, [&](auto t) {
    using T = decltype(t);
    return rec::local_backward<T>(dd, *w, hiddens, feats, r, workspace, workspace_bytes, g_mse, *grads, g_hiddens, ST(stream), phases);
  });
}
int recnet_set_background_ctas(int n) {
  if (n < 0 || n > 4096) return RECNET_ERR_BAD_SHAPE;
  rn_background_ctas() = n;
  return 0;
}
float* recnet_local_outputs(const recnet_local_desc* d, void* workspace) {
  LocalDesc dd;
  if (split_desc(d, &dd)) return nullptr;
  return by_prec<float*>(dd.precision, nullptr, [&](auto t) { return rec::plan_local<decltype(t)>(dd, workspace).out; });
}

// ---- global reconstructor --------------------------------------------------------------------------------------
int64_t recnet_global_workspace_bytes(const recnet_global_desc* d) {
  RN_TRY(check_desc(d));
  return by_prec<int64_t>(d->precision, RECNET_ERR_UNSUPPORTED,
                          [&](auto t) { return (int64_t)rec::plan_global<decltype(t)>(*d, nullptr).bytes; });
}
int recnet_global_fwd(const recnet_global_desc* d, const recnet_global_tensors* w, const float* hiddens, const float* feats,
                      const uint64_t* rng, void* workspace, int64_t workspace_bytes, float* loss_out, void* stream) {
  RN_TRY(check_desc(d));
  const unsigned long long* r = reinterpret_cast<const unsigned long long*>(rng);
  return by_prec<int>(d->precision, RECNET_ERR_UNSUPPORTED, [&](auto t) {
    return rec::global_forward<decltype(t)>(*d, *w, hiddens, feats, r, workspace, workspace_bytes, loss_out, ST(stream));
  });
}
int recnet_global_bwd(const recnet_global_desc* d, const recnet_global_tensors* w, const float* hiddens, const float* feats,
                      const uint64_t* rng, void* workspace, int64_t workspace_bytes, const float* g_loss,
                      const recnet_global_tensors* grads, float* g_hiddens, void* stream) {
  RN_TRY(check_desc(d));
  const unsigned long long* r = reinterpret_cast<const unsigned long long*>(rng);
  return by_prec<int>(d->precision, RECNET_ERR_UNSUPPORTED, [&](auto t) {
    return rec::global_backward<decltype(t)>(*d, *w, hiddens, feats, r, workspace, workspace_bytes, g_loss, *grads, g_hiddens, ST(stream));
  });
}
float* recnet_global_outputs(const recnet_global_desc* d, void* workspace) {
  if (check_desc(d)) return nullptr;
  return by_prec<float*>(d->precision, nullptr, [&](auto t) { return rec::plan_global<decltype(t)>(*d, workspace).out; });
}

// ---- regulariser -----------------------------------------------------------------------------------------------
int recnet_param_norms_fwd(const int64_t* ptrs, const int64_t* sizes, int n, const int32_t* blk_tensor, const int32_t* blk_chunk,
                           int n_blocks, float* partial, float* sumsq, float* reg_out, const float* base, const float* lambda_dev,
                           float* fused_out, void* stream) {
  cudaStream_t st = ST(stream);
  misc::mt_sumsq_kernel<<<n_blocks, 256, 0, st>>>(reinterpret_cast<const long long*>(ptrs), reinterpret_cast<const long long*>(sizes),
                                                  blk_tensor, blk_chunk, partial);
  RN_LAUNCH_OK();
  misc::mt_norm_finalize_kernel<<<1, 512, 0, st>>>(partial, blk_tensor, n_blocks, sumsq, n, reg_out, base, lambda_dev, fused_out);
  RN_LAUNCH_OK();
  return 0;
}
// the two halves of recnet_param_norms_fwd: the squared-norm partials depend on the parameters only, so a trainer can compute them ahead of
// the forward pass (on another stream) and finalise -- including the loss assembly -- once the loss is there
int recnet_param_norms_partial(const int64_t* ptrs, const int64_t* sizes, const int32_t* blk_tensor, const int32_t* blk_chunk, int n_blocks,
                               float* partial, void* stream) {
  misc::mt_sumsq_kernel<<<n_blocks, 256, 0, ST(stream)>>>(reinterpret_cast<const long long*>(ptrs), reinterpret_cast<const long long*>(sizes),
                                                          blk_tensor, blk_chunk, partial);
  RN_LAUNCH_OK();
  return 0;
}
int recnet_param_norms_finalize(const float* partial, const int32_t* blk_tensor, int n_blocks, int n, float* sumsq, float* reg_out,
                                const float* base, const float* lambda_dev, float* fused_out, void* stream) {
  misc::mt_norm_finalize_kernel<<<1, 512, 0, ST(stream)>>>(partial, blk_tensor, n_blocks, sumsq, n, reg_out, base, lambda_dev, fused_out);
  RN_LAUNCH_OK();
  return 0;
}
int recnet_param_norms_bwd(const int64_t* ptrs, const int64_t* grad_ptrs, const int64_t* sizes, int n, const int32_t* blk_tensor,
                           const int32_t* blk_chunk, int n_blocks, const float* sumsq, const float* g, float lambda,
                           const float* lambda_dev, int accumulate, void* stream) {
  (void)n;
  misc::mt_reg_grad_kernel<<<n_blocks, 256, 0, ST(stream)>>>(reinterpret_cast<const long long*>(ptrs),
                                                             reinterpret_cast<const long long*>(grad_ptrs),
                                                             reinterpret_cast<const long long*>(sizes), blk_tensor, blk_chunk, sumsq, g,
                                                             lambda, accumulate, lambda_dev);
  RN_LAUNCH_OK();
  return 0;
}

// ---- teacher-forcing inputs (train.py:25,44-45,54-60,68) ----------------------------------------------------------
int recnet_cider_d(const recnet_cider_corpus* c, const int64_t* ids, int64_t ld_step, int64_t ld_row, int steps, int n_rows,
                   const int32_t* video_of_row, int64_t eos_id, float* scores_out, void* stream) {
  if (!c || c->n_videos < 1 || steps < 1 || steps > cider::kMaxSteps || n_rows <= 0) return RECNET_ERR_BAD_SHAPE;
  if (c->vocab > 65536) return RECNET_ERR_UNSUPPORTED;
  return cider::launch(*c, reinterpret_cast<const long long*>(ids), (long long)ld_step, (long long)ld_row, steps, n_rows, video_of_row,
                       (long long)eos_id, scores_out, ST(stream));
}

int recnet_teacher_forcing_prep(const int64_t* targets, int L, int B, int64_t pad, int64_t sos, int64_t* tokens_in, float* ce_weight,
                                void* stream) {
  if (L < 1 || B < 1 || !targets || !tokens_in || !ce_weight) return RECNET_ERR_BAD_SHAPE;
  misc::tf_prep_kernel<<<1, 1024, (size_t)(L + 1) * sizeof(float), ST(stream)>>>(reinterpret_cast<const long long*>(targets), L, B,
                                                                                  (long long)pad, (long long)sos,
                                                                                  reinterpret_cast<long long*>(tokens_in), ce_weight);
  RN_LAUNCH_OK();
  return 0;
}

// ---- fused gradient clip + Adam (train.py:269-273) ---------------------------------------------------------------
int recnet_adam_step(const int64_t* param_ptrs, const int64_t* grad_ptrs, const int64_t* exp_avg_ptrs, const int64_t* exp_avg_sq_ptrs,
                     const int64_t* max_exp_avg_sq_ptrs, const int64_t* sizes, int n, const int32_t* blk_tensor,
                     const int32_t* blk_chunk, int n_blocks, double lr, double beta1, double beta2, double eps, double weight_decay,
                     double max_grad_norm, float* partial, float* state, int write_clipped_grads, void* stream) {
  typedef const long long* LP;
  return optim::adam_step(reinterpret_cast<LP>(param_ptrs), reinterpret_cast<LP>(grad_ptrs), reinterpret_cast<LP>(exp_avg_ptrs),
                          reinterpret_cast<LP>(exp_avg_sq_ptrs), reinterpret_cast<LP>(max_exp_avg_sq_ptrs), reinterpret_cast<LP>(sizes), n,
                          blk_tensor, blk_chunk, n_blocks, lr, beta1, beta2, eps, weight_decay, max_grad_norm, partial, state,
                          write_clipped_grads, ST(stream));
}
int recnet_allreduce_avg(float* local, float* multicast, const int64_t* peer_ptrs, uint32_t* flags, const int64_t* peer_flag_ptrs,
                         uint32_t* epochs, int32_t* err, int64_t offset_floats, int64_t n_floats, int rank, int world, int ctas, void* stream) {
  if ((offset_floats & 3) || (n_floats & 3)) return RECNET_ERR_ALIGNMENT;
  ar::Args a;
  a.local = local; a.mc = multicast; a.peers = reinterpret_cast<const long long*>(peer_ptrs); a.flags = flags;
  a.peer_flags = reinterpret_cast<const long long*>(peer_flag_ptrs); a.epochs = epochs; a.err = err;
  a.off4 = offset_floats / 4; a.n4 = n_floats / 4; a.rank = rank; a.world = world; a.scale = 1.f / (float)world;
  return ar::launch(a, ctas, ST(stream));
}
}  // extern "C"
