/*
 * recnet_b200 -- C ABI of the B200-native (sm_100a) RecNet hot path.
 *
 * The reference (hobincar/reconstruction-network-for-video-captioning) has no FFI / plugin layer: its
 * boundary for this path is the Python nn.Module surface (SURVEY.md section 8b).  This header is the
 * C-ABI a binding for that surface calls; the Python mirror lives in
 * reconstruction-network-for-video-captioning_b200/ and loads librecnet_b200.so with ctypes.
 * Every entry point says which reference code it replaces (file:line in /root/reference).
 *
 * Conventions
 *   - plain pointers and sizes only; all tensor pointers are DEVICE pointers owned by the caller
 *     (PyTorch's caching allocator); nothing is allocated or freed here; kernels run on `stream`
 *     (a cudaStream_t passed as void*) and the call returns without synchronising.
 *   - return value: 0 = ok, > 0 = cudaError_t of a failed CUDA call, < 0 = recnet_status below.
 *   - re-entrant: no global mutable state besides lazily-resolved driver entry points and
 *     per-kernel shared-memory attributes; safe to call from the autograd engine's thread.
 *   - precision: RECNET_PREC_FP32 = fp32 storage + fp32 FFMA GEMMs (parity build, 1e-3 vs oracle);
 *     RECNET_PREC_BF16 = bf16 GEMM operands on tcgen05 tensor cores with fp32 TMEM accumulation,
 *     fp32 cell state / reductions (2e-2 vs oracle).  There is no CPU path.
 */
#ifndef RECNET_B200_H_
#define RECNET_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  RECNET_OK = 0,
  RECNET_ERR_BAD_SHAPE = -1,
  RECNET_ERR_ALIGNMENT = -2,
  RECNET_ERR_UNSUPPORTED_ARCH = -3,
  RECNET_ERR_UNSUPPORTED = -4,
  RECNET_ERR_WORKSPACE = -5,
  RECNET_ERR_DRIVER = -6
} recnet_status;

typedef enum { RECNET_PREC_FP32 = 0, RECNET_PREC_BF16 = 1 } recnet_precision;
#define RECNET_MAX_LAYERS 4
typedef enum { RECNET_CELL_LSTM = 0, RECNET_CELL_GRU = 1 } recnet_cell;   /* models/decoder.py:32-35: anything but "LSTM" is GRU */
/* Flag OR'd into the `cell` field of recnet_decoder_desc / recnet_local_desc (the low byte holds the recnet_cell value):
 * the paper's softmax attention, alpha = softmax over frames (decoder) / decoder steps (local reconstructor) of the scores e,
 * context = sum alpha * v (no 1/T).  Without it (the default) the attention is the reference's: context = mean(e * v).
 * Any other bit above the low byte makes the call return RECNET_ERR_UNSUPPORTED. */
#define RECNET_ATTN_SOFTMAX 0x100
#define RECNET_CELL_MASK 0xff

/* Library / device checks.  recnet_query_device fails with RECNET_ERR_UNSUPPORTED_ARCH unless the
 * device is compute capability 10.x (sm_100a cubins only; no PTX fallback, no other arch). */
int recnet_abi_version(void);
int recnet_query_device(int device, int* sm_count, int* cc_major, int* cc_minor);

/* Launch accounting and per-launch device timing (used by bench.py for `gpu_launches` and the roofline leg).
 * recnet_launch_count: kernels launched by this library so far in this process.
 * recnet_profile_enable(1, n): record a CUDA-event pair around up to n kernel launches (eager mode only, not under
 * graph capture); recnet_profile_collect synchronises and writes n x 5 floats (class, M, N, K, ms); classes:
 * 1 tcgen05 GEMM, 2 fp32 sgemm, 3 attention fwd, 4 attention bwd, 5 cell fwd, 6 cell bwd, 7 CE, 8 split-K reduce. */
long long recnet_launch_count(void);
int recnet_profile_enable(int on, int max_records);
int recnet_profile_collect(float* out, int max_records);

/* ------------------------------------------------------------------------------------------------
 * Operator level (one kernel family each).  Used by the per-step nn.Module.forward mirrors and by
 * the per-kernel parity tests.
 * ---------------------------------------------------------------------------------------------- */

/* C[m,n] (+)= sum_k A(m,k) B(n,k) (+ bias[n]).   Replaces every nn.Linear / cuBLAS call on the path
 * (models/decoder.py:51,54,68; models/local_reconstructor.py:39,42,54; models/global_reconstructor.py:45)
 * and the two GEMMs inside each nn.LSTM step (decoder.py:66 etc).
 *   transA = 0: A is [M,K] row-major, lda; 1: A is [K,M] row-major.   transB = 0: B is [N,K] row-major
 *   (nn.Linear weight layout); 1: B is [K,N] row-major.  Element type of A/B: float (FP32) or bf16 (BF16).
 *   C fp32 [M,N] ldc (nullable if c_op given); c_op: optional second output in the operand type (bf16 only).
 *   splits > 1: slice s of K writes its partial to C + s*split_stride (consumers sum the partials).
 *   bn_hint: 0 = auto, or 64/128/256 = tcgen05 tile width (BF16 only). */
int recnet_gemm(int precision, const void* A, int64_t lda, int transA, const void* B, int64_t ldb, int transB,
                float* C, int64_t ldc, void* c_op, int64_t ldc_op, const float* bias, int M, int N, int K,
                int splits, int64_t split_stride, int accumulate, int bn_hint, void* stream);

/* out[m*ldo + n] (+)= sum_s partial[s*split_stride + m*ldp + n] */
/* Host-only: the tile / split-K plan the batched GEMMs of the sequence calls use for an [M x N x K] product (bf16: bn = 64 / 128 / 256 for the
 * one-tile-per-CTA kernel, 1000 + width for the persistent kernel with single CTAs, 2000 + width with CTA pairs; splits = split-K slices).
 * No device work: lets tests pin the planner's decisions (profiles/r2_h_gemm_sweep.md). */
int recnet_plan_batched_gemm(int precision, int M, int N, int K, int32_t* bn_out, int32_t* splits_out);
int recnet_splitk_reduce(const float* partial, int splits, int64_t split_stride, int64_t ldp, float* out, int64_t ldo,
                         int M, int N, int accumulate, void* stream);

/* Fused additive attention, forward (models/decoder.py:50-62, models/local_reconstructor.py:38-50 minus the
 * U-projection, which is hoisted):  e = w.tanh(Wh + Uv + b);  ctx = mean_tau(e * V)   [no softmax: SURVEY 0.1].
 *   wh_partials [n_wh][B,A] fp32 (split-K partials of h W^T, summed here); uv[b*uv_bs + tau*uv_ts + a] fp32;
 *   v[b*v_bs + tau*v_ts + d] in `precision` storage; ctx_out[b*ctx_ld + d] in `precision` storage.
 *   wh_out [B,A], e_out [B,Tn] fp32: saved for backward (nullable).  normalize=1 -> the paper's attention:
 *   alpha = softmax_tau(e), ctx = sum_tau alpha * V, and e_out holds alpha (its backward: recnet_attn_bwd_softmax).
 *   p_drop/rng/site/drop_base: train-mode dropout on ctx (local reconstructor). */
int recnet_attn_fwd(int precision, const float* wh_partials, int n_wh, int64_t wh_stride, const float* uv,
                    int64_t uv_bs, int64_t uv_ts, const float* attn_b, const float* attn_w, const void* v,
                    int64_t v_bs, int64_t v_ts, int B, int Tn, int A, int D, int normalize, float* wh_out,
                    float* e_out, void* ctx_out, int64_t ctx_ld, float p_drop, const uint64_t* rng, uint32_t site,
                    int64_t drop_base, void* stream);

/* Fused additive attention, backward (autograd of the same lines).  dctx arrives as n_p split-K partials
 * [n_p][B,p_ld] (columns [0,D)).  Outputs: dwh_out [B,A] fp32 and dwh_op [B,A] in operand storage (nullable;
 * A-operand of the dWh @ attn_W GEMM); duv_acc (same strides as uv) and dw_acc [B,A] are accumulated across
 * timesteps (first=1 overwrites); dctx_out [B,D] optional (summed, dropout-masked). */
int recnet_attn_bwd(int precision, const float* dctx_partials, int n_p, int64_t p_stride, int64_t p_ld, const void* v,
                    int64_t v_bs, int64_t v_ts, const float* wh, const float* uv, int64_t uv_bs, int64_t uv_ts,
                    const float* attn_b, const float* attn_w, int B, int Tn, int A, int D, float* dwh_out,
                    void* dwh_op, float* duv_acc, float* dw_acc, int first, float* dctx_out, float p_drop,
                    const uint64_t* rng, uint32_t site, int64_t drop_base, void* stream);
/* Backward of recnet_attn_fwd(normalize=1), same arguments as recnet_attn_bwd plus alpha [B,Tn] fp32 = the e_out that forward
 * wrote: d alpha = dctx . V, d e = alpha (d alpha - sum_tau alpha d alpha), then the same score backward. */
int recnet_attn_bwd_softmax(int precision, const float* dctx_partials, int n_p, int64_t p_stride, int64_t p_ld, const void* v,
                            int64_t v_bs, int64_t v_ts, const float* alpha, const float* wh, const float* uv, int64_t uv_bs,
                            int64_t uv_ts, const float* attn_b, const float* attn_w, int B, int Tn, int A, int D, float* dwh_out,
                            void* dwh_op, float* duv_acc, float* dw_acc, int first, float* dctx_out, float p_drop,
                            const uint64_t* rng, uint32_t site, int64_t drop_base, void* stream);

/* Fused LSTM gate activation + cell update (the pointwise half of nn.LSTM, decoder.py:66; gate order i,f,g,o).
 *   pre = sum_s partials[s] + gx + b1 + b2.  gates_out [B,4H] (stash, `precision` storage), c_out/h_out fp32,
 *   h_op / h_op2: h' in operand storage written into next step's [x;h] rows (nullable). */
int recnet_lstm_cell_fwd(int precision, const float* partials, int n_p, int64_t p_stride, int64_t p_ld, const float* gx,
                         int64_t gx_ld, const float* b1, const float* b2, const float* c_prev, int B, int H,
                         void* gates_out, float* c_out, float* h_out, int64_t h_ld, void* h_op, int64_t hop_ld,
                         void* h_op2, int64_t hop2_ld, void* stream);

/* Backward of the same step.  dh = dh_scale*dh_ext + dh_ext2 + sum_s dxp[s][:, col0:col0+H] + sum_s dqp[s]
 * (dxp: split-K partials of d[x;h]; dqp [n_q][B,q_ld]: split-K partials of dWh @ attn_W, the attention-query
 * path).  dc is in/out ([B,H]; first=1 -> treated as 0).  dg_out [B,4H] in operand storage. */
int recnet_lstm_cell_bwd(int precision, const float* dh_ext, int64_t dh_ld, const float* dh_scale, const float* dh_ext2,
                         int64_t dh2_ld, const float* dxp, int n_p, int64_t p_stride, int64_t p_ld, int col0,
                         const float* dqp, int n_q, int64_t q_stride, int64_t q_ld, float* dc, int first, const void* gates,
                         const float* c_prev, const float* c_new, int B, int H, void* dg_out, int64_t dg_ld,
                         void* stream);

/* Fused GRU gate activation + state update (the pointwise half of nn.GRU, models/decoder.py:32-40,66; gate order r,z,n).
 *   gi = sum_s px[s] + gx + b_ih ; gh = sum_s ph[s] + b_hh ; r,z = sigmoid(gi + gh) ; n = tanh(gi_n + r * gh_n) ;
 *   h' = (1 - z) n + z h.  stash [B,4H] (r, z, n, gh_n) in `precision` storage for BPTT. */
int recnet_gru_cell_fwd(int precision, const float* px, int n_px, int64_t px_stride, int64_t px_ld, const float* ph,
                        int n_ph, int64_t ph_stride, int64_t ph_ld, const float* gx, int64_t gx_ld, const float* b_ih,
                        const float* b_hh, const float* h_prev, int64_t hp_ld, int B, int H, void* stash, float* h_out,
                        int64_t h_ld, void* h_op, int64_t hop_ld, void* stream);
/* Backward: dh' = dh_ext + dh_ext2 + carry + sum dhp + sum dqp ; writes dgi / dgh [B,3H] (operand storage) and the new
 * carry = z * dh' (direct path into h_{t-1}); first=1 treats the incoming carry as 0. */
int recnet_gru_cell_bwd(int precision, const float* dh_ext, int64_t dh_ld, const float* dh_ext2, int64_t dh2_ld,
                        const float* dhp, int n_p, int64_t p_stride, int64_t p_ld, const float* dqp, int n_q,
                        int64_t q_stride, int64_t q_ld, float* carry, int first, const void* stash, const float* h_prev,
                        int64_t hp_ld, int B, int H, void* dgi, void* dgh, int64_t dg_ld, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Sequence level: whole teacher-forced loops, forward and BPTT, one host call each.
 * ---------------------------------------------------------------------------------------------- */

/* Decoder (reference Decoder module + train.forward_decoder loop, models/decoder.py:45-70, train.py:17-75). */
typedef struct {
  int32_t B, T, E, H, A, EMB, V, L;     /* L = decoded steps (<= caption_max_len + 1, train.py:41,66) */
  int32_t precision;                    /* recnet_precision */
  int32_t train;                        /* 1 = apply dropout (embedding, logits) */
  float embedding_scale, p_emb_drop, p_out_drop;
  int32_t cell;                         /* recnet_cell: LSTM (i,f,g,o; state h,c) or GRU (r,z,n; state h); | RECNET_ATTN_SOFTMAX */
  int32_t n_layers;                     /* stacked decoder layers (decoder.py:36-40), 0/1 = one; > 1: LSTM only */
  float p_layer_drop;                   /* nn.LSTM(dropout=) between layers, train mode only */
} recnet_decoder_desc;

typedef struct {                        /* fp32 master weights, reference state_dict layout (SURVEY 8b) */
  float *embedding, *attn_W, *attn_U, *attn_b, *attn_w, *w_ih, *w_hh, *b_ih, *b_hh, *out_w, *out_b;
  /* layers 1 .. n_layers-1 (index l-1): rnn.weight_ih_l{l} [4H,H], rnn.weight_hh_l{l} [4H,H], biases [4H]; NULL when absent */
  float *w_ih_x[RECNET_MAX_LAYERS - 1], *w_hh_x[RECNET_MAX_LAYERS - 1], *b_ih_x[RECNET_MAX_LAYERS - 1], *b_hh_x[RECNET_MAX_LAYERS - 1];
} recnet_decoder_tensors;

/* bytes of caller-provided workspace that must stay alive from fwd to bwd */
int64_t recnet_decoder_workspace_bytes(const recnet_decoder_desc* d);

/* tokens_in [L,B] int64 (SOS then targets[t-1], train.py:25,44-45); targets [L,B] int64; ce_weight [L,B] fp32 =
 * mask/(n_t * sum n_t) (train.py:54-60,68).  Outputs: hiddens [L,NL,B,H] fp32 (train.py:61-64,73), ce_out[1] =
 * sum_t CE_t / sum_t n_t, logits_out [L*B, ld = round_up(V,4)] lives inside the workspace
 * (recnet_decoder_logits returns it). */
int recnet_decoder_fwd(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats,
                       const int64_t* tokens_in, const int64_t* targets, const float* ce_weight, const uint64_t* rng,
                       void* workspace, int64_t workspace_bytes, float* hiddens, float* ce_out, void* stream);
/* g_ce: device scalar dLoss/dCE (nullable = 1); g_hiddens [L,B,H] fp32 (nullable); hiddens: the forward's fp32 output
 * (read by the GRU backward, which keeps no separate cell state). grads: every field written (overwritten, not accumulated). */
int recnet_decoder_bwd(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats,
                       const int64_t* tokens_in, const int64_t* targets, const float* ce_weight, const uint64_t* rng,
                       void* workspace, int64_t workspace_bytes, const float* g_ce, const float* g_hiddens,
                       const float* hiddens, const recnet_decoder_tensors* grads, void* stream);
/* recnet_decoder_fwd in parts, same arguments (split where recnet_decoder_bwd_is_split says so; otherwise bit 0 runs everything):
 *   1 = staging, hoisted projections, the time loop (-> hiddens)      2 = vocabulary projection, attention contexts, CE (-> ce_out; needs 1)
 * Nothing of part 2 feeds the reconstructor: a trainer may run it on another stream next to the reconstructor's staging. */
int recnet_decoder_fwd_phase(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats, const int64_t* tokens_in,
                             const int64_t* targets, const float* ce_weight, const uint64_t* rng, void* workspace,
                             int64_t workspace_bytes, float* hiddens, float* ce_out, int phases, void* stream);
/* recnet_decoder_bwd in parts, same arguments (single-layer decoders on the projected-feature path; recnet_decoder_bwd_is_split says
 * whether the split applies -- otherwise bit 0 runs everything and the other bits nothing):
 *   1 = CE backward + gradient wrt the states through the vocabulary projection     2 = the BPTT loop (needs 1)
 *   4 = the vocabulary projection's weight gradient (needs 1 only)                 8 = all other parameter gradients (need 2)
 * phases = 4 alone may run on another stream while 2 runs (own scratch); 15 is recnet_decoder_bwd. */
int recnet_decoder_bwd_phase(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats, const int64_t* tokens_in,
                             const int64_t* targets, const float* ce_weight, const uint64_t* rng, void* workspace,
                             int64_t workspace_bytes, const float* g_ce, const float* g_hiddens, const float* hiddens,
                             const recnet_decoder_tensors* grads, int phases, void* stream);
int recnet_decoder_bwd_is_split(const recnet_decoder_desc* d);
float* recnet_decoder_logits(const recnet_decoder_desc* d, void* workspace, int64_t* ld);

/* Greedy decoding (eval.greedy_search, eval.py:19-33): argmax feedback on device, zero host syncs.
 * ids_out [max_steps,B] int64; n_steps_out[1] int32 (device) = steps until every fed-back token is <PAD>.  The loop runs all max_steps
 * steps (rows after n_steps_out[0] continue the argmax feedback).  LSTM decoders with 1-4 layers, single-layer GRU; a stacked GRU or
 * n_layers > RECNET_MAX_LAYERS is RECNET_ERR_UNSUPPORTED. */
int64_t recnet_greedy_workspace_bytes(const recnet_decoder_desc* d);
int recnet_decoder_greedy(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats,
                          int max_steps, void* workspace, int64_t workspace_bytes, int64_t* ids_out,
                          int32_t* n_steps_out, void* stream);

/* Beam search (eval.beam_search, eval.py:36-120) as a device loop with zero host syncs: d->B = beam_width * B0 rows, row k * B0 + b =
 * beam k of sample b; feats_tiled [beam_width * B0, T, E] = the B0 samples repeated beam_width times.  Scores log(sigmoid(logit)),
 * running score divided by len^0.7 at every step (len = position of the last <EOS> + 1, else t + 1), top-k over beams x vocabulary, stop
 * when every fed-back token is <PAD> -- the reference's rules.  seq_out [B0, max_steps] int64 = the top-1 sequence of every sample
 * (-1 beyond n_steps_out[0]); beam_width <= 8; LSTM decoders with 1-4 layers, single-layer GRU (others: RECNET_ERR_UNSUPPORTED). */
int64_t recnet_beam_workspace_bytes(const recnet_decoder_desc* d, int beam_width, int max_steps);
int recnet_decoder_beam(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats_tiled, int beam_width, int max_steps,
                        int64_t eos_id, void* workspace, int64_t workspace_bytes, int64_t* seq_out, int32_t* n_steps_out, void* stream);

/* Sampling (Gumbel-max) as a device loop with zero host syncs: every row draws its token of step t from softmax(z'/temperature), z' =
 * the logits after their dropout (site 2) when d->train is set, with Gumbel noise from Philox site 5 of the `noise` (seed, offset) pair
 * at element (t*B + row)*V + v.  In train mode every dropout mask is drawn from `rng` (the module's pair, device memory) at the element
 * the sequence forward uses for row t*B + row, so recnet_decoder_fwd over tokens_in = [<SOS>; ids[:-1]], targets = ids with the same
 * pair computes the logits the sampler drew from.  A row finishes once it emits eos_id or <PAD>, then emits <PAD> with log-prob 0.
 * Outputs (device): ids_out [max_steps,B] int64, logp_out [max_steps,B] = log softmax(z'/temperature)[id], lengths_out [B] = tokens up
 * to and including the finishing one (max_steps if none), n_steps_out[1] = the step at which the last row finished + 1.  rng and noise are
 * device pointers.  Coverage of recnet_decoder_greedy (others: RECNET_ERR_UNSUPPORTED); temperature <= 0 or max_steps outside 1..64:
 * RECNET_ERR_BAD_SHAPE. */
int64_t recnet_sample_workspace_bytes(const recnet_decoder_desc* d, int max_steps);
int recnet_decoder_sample(const recnet_decoder_desc* d, const recnet_decoder_tensors* w, const float* feats, int max_steps,
                          float temperature, int64_t eos_id, const unsigned long long* rng, const unsigned long long* noise,
                          void* workspace, int64_t workspace_bytes, int64_t* ids_out, float* logp_out, int32_t* lengths_out,
                          int32_t* n_steps_out, void* stream);

/* Local reconstructor (models/local_reconstructor.py:37-55 + train.forward_local_reconstructor, train.py:108-131). */
typedef struct {
  int32_t B, S, R, H, A, L;             /* S = encoder_output_len steps, R = hidden (= feature dim), H = decoder hidden */
  int32_t precision, train;
  float p_drop;
  int32_t cell;                         /* recnet_cell of the reconstructor RNN; | RECNET_ATTN_SOFTMAX (one softmax over L per decoder layer) */
  int32_t dec_layers;                   /* decoder layers NLd: hiddens is (L, NLd, B, H) and every outer step runs NLd pseudo-steps */
} recnet_local_desc;
typedef struct {
  float *attn_W, *attn_U, *attn_b, *attn_w, *w_ih, *w_hh, *b_ih, *b_hh, *out_w, *out_b;
} recnet_local_tensors;
int64_t recnet_local_workspace_bytes(const recnet_local_desc* d);
/* hiddens [L,B,H] fp32 (decoder states), feats [B,S,R] fp32; mse_out[1] = MSELoss(outputs^T, feats). */
int recnet_local_fwd(const recnet_local_desc* d, const recnet_local_tensors* w, const float* hiddens, const float* feats,
                     const uint64_t* rng, void* workspace, int64_t workspace_bytes, float* mse_out, void* stream);
int recnet_local_bwd(const recnet_local_desc* d, const recnet_local_tensors* w, const float* hiddens, const float* feats,
                     const uint64_t* rng, void* workspace, int64_t workspace_bytes, const float* g_mse,
                     const recnet_local_tensors* grads, float* g_hiddens, void* stream);
/* recnet_local_bwd in two parts, same arguments: phases bit 0 = the BPTT loop and g_hiddens (what the decoder's backward waits for),
 * bit 1 = the batched parameter gradients (read only the workspace; write only `grads`).  A trainer may issue bit 1 on a second
 * stream underneath the decoder's backward loop; the workspace must stay alive until that stream is joined.  phases = 3 is
 * recnet_local_bwd.  recnet_set_background_ctas(n): upper bound on the CTAs of the persistent batched GEMMs launched from now on
 * by this process (0 = none) -- set it around such background work so that it never occupies the SMs the foreground loop needs. */
int recnet_local_bwd_phase(const recnet_local_desc* d, const recnet_local_tensors* w, const float* hiddens, const float* feats,
                           const uint64_t* rng, void* workspace, int64_t workspace_bytes, const float* g_mse,
                           const recnet_local_tensors* grads, float* g_hiddens, int phases, void* stream);
int recnet_set_background_ctas(int n);
/* Host-only: how the weight-resident persistent loops (csrc/seq_recon_persist.cuh) would lay a local-reconstructor call out, 12 ints:
 * forward {covered, K-splits, unit groups, resident k-blocks per CTA, ring stages, CTAs}, backward {covered, gate-row splits, column groups,
 * resident k-blocks per CTA, ring stages, CTAs}; covered = 0 means the call takes the kernel-per-phase path. */
int recnet_plan_persistent_loops(const recnet_local_desc* d, int32_t* out);
float* recnet_local_outputs(const recnet_local_desc* d, void* workspace);   /* [S,B,R] fp32 */

/* Global reconstructor (models/global_reconstructor.py:30-46 + train.forward_global_reconstructor, train.py:78-105). */
typedef struct {
  int32_t B, L, R, H, T;                /* T = frames of feats (mean target), L = decoder steps */
  int32_t precision, train;
  float p_drop, caption_max_len;
  int32_t cell;                         /* recnet_cell of the reconstructor RNN */
  int32_t dec_layers;                   /* decoder layers NLd: hiddens is (L, NLd, B, H); 0/1 = one */
} recnet_global_desc;
typedef struct {
  float *w_ih, *w_hh, *b_ih, *b_hh, *out_w, *out_b;
} recnet_global_tensors;
int64_t recnet_global_workspace_bytes(const recnet_global_desc* d);
/* loss_out[1] = MSELoss(mean_t outputs, mean_tau feats) / L  (train.py:96-100) */
int recnet_global_fwd(const recnet_global_desc* d, const recnet_global_tensors* w, const float* hiddens, const float* feats,
                      const uint64_t* rng, void* workspace, int64_t workspace_bytes, float* loss_out, void* stream);
int recnet_global_bwd(const recnet_global_desc* d, const recnet_global_tensors* w, const float* hiddens, const float* feats,
                      const uint64_t* rng, void* workspace, int64_t workspace_bytes, const float* g_loss,
                      const recnet_global_tensors* grads, float* g_hiddens, void* stream);
float* recnet_global_outputs(const recnet_global_desc* d, void* workspace);  /* [L,B,R] fp32 */

/* The weight-resident time loops of the bf16 build (local reconstructor, LSTM, MSVD-class shapes) run as ONE persistent
 * cooperative kernel per loop (csrc/seq_recon_persist.cuh): [W_ih | W_hh] stays in the shared memory of 144 CTAs for all steps
 * and the CTAs meet at three flag waits per step.  Every spin has a timeout; on a protocol failure the kernel raises an int32
 * flag inside the workspace instead of hanging the GPU.  These return the flag's byte offset in the workspace
 * (0 = ok, 2 = mbarrier timeout, 3 = flag-wait timeout). */
int64_t recnet_decoder_error_offset(const recnet_decoder_desc* d);
int64_t recnet_local_error_offset(const recnet_local_desc* d);
int64_t recnet_global_error_offset(const recnet_global_desc* d);

/* developer probe: %globaltimer stamps of block 0 at the phase boundaries of the persistent loops -> buf (device u64[4096]); NULL = off */
int recnet_debug_set_timeline(void* buf);

/* test probe: out[i] = the inverted-dropout scale (0 or 1/(1-p)) the kernels apply to element i of dropout site `site`
 * (1 embedding [L,B,EMB], 2 logits [L,B,V], 3 local-reconstructor input [S,B,H], 4 global-reconstructor mean-pool [L,B,H]; reference
 * models/decoder.py:48,69, models/local_reconstructor.py:50, models/global_reconstructor.py:38) for rng = {seed, offset} on the device.
 * Lets a checker feed the SAME masks to the oracle / the reference (tests/test_gpu_dropout_parity.py). */
int recnet_debug_dropout_mask(const uint64_t* rng, uint32_t site, int64_t n, float p, float* out, void* stream);

/* L2-norm regulariser over a parameter list (train.py:69,101,127): reg = sum_p ||p||_2.
 * ptrs/sizes: device int64 tables of n tensors; blk_tensor/blk_chunk: device int32 tables mapping block ->
 * (tensor, 16384-element chunk); partial [n_blocks] fp32 scratch (two-stage, fixed-order => bitwise reproducible);
 * sumsq [n] fp32 kept for the backward.
 * fused_out != NULL: also writes the assembled loss of train.py:70,102,128, fused_out[0] = base[0] + lambda_dev[0] * reg
 * (base / lambda_dev: device scalars, NULL = 0 / 1) -- saves the elementwise mul + add nodes of every module. */
int recnet_param_norms_fwd(const int64_t* ptrs, const int64_t* sizes, int n, const int32_t* blk_tensor,
                           const int32_t* blk_chunk, int n_blocks, float* partial, float* sumsq, float* reg_out,
                           const float* base, const float* lambda_dev, float* fused_out, void* stream);
/* grad_p (+)= lambda * lambda_dev[0] * g[0] * p / ||p||     (g, lambda_dev: device scalars, NULL = 1) */
/* recnet_param_norms_fwd in two halves: `partial` (n_blocks floats) depends on the parameters only. */
int recnet_param_norms_partial(const int64_t* ptrs, const int64_t* sizes, const int32_t* blk_tensor, const int32_t* blk_chunk, int n_blocks,
                               float* partial, void* stream);
int recnet_param_norms_finalize(const float* partial, const int32_t* blk_tensor, int n_blocks, int n, float* sumsq, float* reg_out,
                                const float* base, const float* lambda_dev, float* fused_out, void* stream);
int recnet_param_norms_bwd(const int64_t* ptrs, const int64_t* grad_ptrs, const int64_t* sizes, int n,
                           const int32_t* blk_tensor, const int32_t* blk_chunk, int n_blocks, const float* sumsq,
                           const float* g, float lambda, const float* lambda_dev, int accumulate, void* stream);

/* Teacher-forcing inputs of train.forward_decoder in one launch (train.py:25,44-45,54-60,68): targets (>= L rows of B int64,
 * row-major) -> tokens_in [L,B] = (<SOS> row, targets[0..L-2]) and ce_weight [L,B] = [target > pad] / (max(n_t,1) * sum_t n_t). */
int recnet_teacher_forcing_prep(const int64_t* targets, int L, int B, int64_t pad, int64_t sos, int64_t* tokens_in,
                                float* ce_weight, void* stream);

/* Fused gradient-norm clip + Adam step over a parameter list -- replaces torch.nn.utils.clip_grad_norm_ (reference
 * train.py:269-270) followed by torch.optim.Adam.step (train.py:271-273; optimisers built at train.py:149-150,186-187:
 * L2 weight decay, optional amsgrad).  Tables as for recnet_param_norms_*: device int64 address tables of the n
 * parameters, their gradients and the optimiser state tensors (exp_avg, exp_avg_sq, max_exp_avg_sq or NULL = no
 * amsgrad), sizes[n], and the block -> (tensor, 16384-element chunk) map.
 * max_grad_norm > 0: total L2 norm over ALL n gradients, grads scaled by min(1, max_norm / (norm + 1e-6)) on the fly
 * (written back to the gradient tensors only if write_clipped_grads); partial [n_blocks] fp32 scratch.
 * state: device float[8], zero-initialised by the caller: [0] step count (advanced by one per call, on the device,
 * so a captured CUDA graph keeps counting), [1] last total grad norm, [2] last clip coefficient, [3..7] internal. */
int recnet_adam_step(const int64_t* param_ptrs, const int64_t* grad_ptrs, const int64_t* exp_avg_ptrs,
                     const int64_t* exp_avg_sq_ptrs, const int64_t* max_exp_avg_sq_ptrs, const int64_t* sizes, int n,
                     const int32_t* blk_tensor, const int32_t* blk_chunk, int n_blocks, double lr, double beta1, double beta2,
                     double eps, double weight_decay, double max_grad_norm, float* partial, float* state,
                     int write_clipped_grads, void* stream);

/* Data-parallel gradient all-reduce (average) over NVLink / NVSwitch as ONE kernel of this library (SURVEY.md 8e; the reference has
 * no distributed code; replaces an ncclAllReduce between backward, train.py:268, and clip + Adam, train.py:269-273).
 * The gradients of all ranks live in SYMMETRIC memory: `local` = this rank's buffer, `multicast` = the NVSwitch multicast alias of all
 * ranks' buffers (NULL -> two-shot over the peer pointers in the device table peer_ptrs[world]), flags / peer_flag_ptrs = a zeroed
 * symmetric block of 2 * 64 * 16 uint32 per rank and the device table of every rank's block, epochs = 64 zeroed local uint32,
 * err = local int32 (4 = a peer did not arrive within ~2 s).  Reduces floats [offset, offset + n) in place on every rank
 * (two-shot: rank r sums slice r across ranks with multimem.ld_reduce and broadcasts it with multimem.st).  offset, n: multiples of 4.
 * Every rank must launch it in the same order; `ctas` (<= 64) CTAs of 512 threads. */
int recnet_allreduce_avg(float* local, float* multicast, const int64_t* peer_ptrs, uint32_t* flags, const int64_t* peer_flag_ptrs,
                         uint32_t* epochs, int32_t* err, int64_t offset_floats, int64_t n_floats, int rank, int world, int ctas, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RECNET_B200_H_ */
