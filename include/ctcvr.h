/*
 * ctcvr.h — C-ABI of libctcvr.so: the B200 (sm_100a) transducer hot path of CentaureaHO/CTC-VR.
 *
 * The reference has NO plugin / FFI layer for this path: the boundary is a set of Python call
 * sites into third-party wheels (SURVEY.md §8b).  Each entry point below names the reference
 * call site it replaces (paths relative to the reference tree; `site-packages/` = installed
 * torchaudio / torch).  The reference-side binding is a ctypes stub: see INTEGRATION.md and
 * ctc-vr_b200/_lib.py.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named h_*.
 *   - the caller owns every buffer (PyTorch allocates); kernels are enqueued on `stream`
 *     (a cudaStream_t passed as void*); no entry point synchronises, allocates device memory
 *     or reads device data on the host.
 *   - return 0 on success, non-zero on error; `ctcvr_last_error()` gives the message; the Python
 *     shim raises RuntimeError (rnnt_train.py:139 relies on `except RuntimeError`).
 *   - all tensors are dense row-major ("contiguous"); T = max encoder frames, U1 = max target
 *     length + 1, D = joint dim, V = vocabulary size; lengths are int32.
 *   - precision: CTCVR_F32 = fp32 SIMT path (1e-4 parity path), CTCVR_BF16 = tcgen05 path
 *     (bf16 operands - enc_proj / pred_proj are rounded to bf16 too - fp32 accumulate / softmax /
 *     lattice).  enc_proj / pred_proj must be 16-byte aligned in the bf16 path.
 *     CTCVR_BF16X3 = the tcgen05 path at fp32 accuracy: every fp32 operand x is split into
 *     hi = bf16(x), lo = bf16(x - hi) and each product is hi*hi + hi*lo + lo*hi (three MMAs into one
 *     fp32 accumulator); tanh, G = d cost / d logits and the reductions stay fp32.  Loss and gradients
 *     within 1e-4 of the reference, like CTCVR_F32; same shape limits and alignment as CTCVR_BF16.
 *   - joint activation: `precision` of the fused joint entry points (and their _ws_bytes queries) carries one
 *     CTCVR_ACT_* value OR'ed into it: z = tanh / relu / gelu(enc_proj + pred_proj) (joint.py `activation`).  0 is
 *     tanh, so CTCVR_F32 / CTCVR_BF16 / CTCVR_BF16X3 alone keep their meaning; any other bit is an error return.  fp32
 *     and bf16x3 form act and act' in fp32; bf16 forms h as a packed bf16 add (relu: packed max with 0; gelu: erff in
 *     fp32 from the bf16 h).  The post-join linear of joint.py folds into enc_proj / pred_proj (it is linear):
 *     post(e + p) = (W_post e + b_post) + W_post p.  The _bf16in entry points and ctcvr_joint_logits are tanh only.
 */
#ifndef CTCVR_H_
#define CTCVR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTCVR_F32 0
#define CTCVR_BF16 1
#define CTCVR_BF16X3 2
/* joint activation z = act(enc_proj + pred_proj), OR'ed into `precision` of ctcvr_joint_rnnt_fwd / _bwd and their
 * _ws_bytes queries (0 = tanh, so the plain precision values keep their meaning) and set in
 * ctcvr_decoder_weights.activation */
#define CTCVR_ACT_TANH 0x000
#define CTCVR_ACT_RELU 0x100 /* nn.ReLU: derivative h > 0 (0 at h = 0, as torch) */
#define CTCVR_ACT_GELU 0x200 /* nn.GELU(), exact erf form: h Phi(h), derivative Phi(h) + h phi(h) */

const char* ctcvr_last_error(void);
int ctcvr_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py's gpu_launches) */
unsigned long long ctcvr_launch_count(void);
/* debug: non-zero if a tcgen05 kernel hit its bounded mbarrier wait (synchronises; clears the flag) */
unsigned int ctcvr_debug_tc_error(void);
/* debug: device buffer of 4*2048 int64 receiving a per-role timeline of CTA 0 of the next tcgen05 forward (NULL = off) */
void ctcvr_debug_set_prof(void* device_buf);
/* debug (A/B timing): bit 0 = single-CTA forward kernel (default 1; 0 runs the parked CTA-pair forward), bit 1 =
 * single-CTA backward kernel where the CTA-pair kernel is the default, bits 2.. = experiment switches of the peer
 * exchange kernel (tools/peer_time.py).  Production value: 1. */
void ctcvr_debug_set_mode(int mode);

/* ---- A1: TransducerJoint.forward dense logits — model/component/joint.py:57-68
 * logits[b,t,u,:] = W_out · tanh(enc_proj[b,t,:] + pred_proj[b,u,:]) + b_out.
 * enc_proj/pred_proj are the outputs of enc_ffn/pred_ffn (joint.py:54-55). */
int ctcvr_joint_logits(const float* enc_proj, const float* pred_proj, const float* w_out,
                       const float* b_out, float* logits, int B, int T, int U1, int D, int V,
                       void* stream);

/* ---- A1+A2 fused forward — model/component/joint.py:57-68 followed by the log-softmax /
 * log-prob gather of torchaudio.functional.rnnt_loss as called at
 * model/component/transducer.py:180-187 and model/online_rnnt_model.py:247-255.
 * Emits only lse, lp_blank, lp_label [B,T,U1]; logits never reach HBM.
 * targets [B,U1-1] int32.  Cells with t>=t_len[b] or u>u_len[b] are not written. */
size_t ctcvr_joint_rnnt_fwd_ws_bytes(int B, int T, int U1, int D, int V, int precision);
int ctcvr_joint_rnnt_fwd(const float* enc_proj, const float* pred_proj, const float* w_out,
                         const float* b_out, const int32_t* targets, const int32_t* t_len,
                         const int32_t* u_len, float* lse, float* lp_blank, float* lp_label,
                         int B, int T, int U1, int D, int V, int blank, int precision,
                         void* ws, size_t ws_bytes, void* stream);

/* ---- A2 lattice — the alpha/beta recursion and costs of torchaudio rnnt_loss
 * (site-packages/torchaudio/functional/functional.py:1725; SURVEY.md §8 A2).
 * alpha, beta [B,T,U1]; costs [B] = -beta(0,0). */
int ctcvr_rnnt_lattice(const float* lp_blank, const float* lp_label, const int32_t* t_len,
                       const int32_t* u_len, float* alpha, float* beta, float* costs,
                       int B, int T, int U1, void* stream);

/* ---- A1+A2 fused backward — replaces RnntLoss.backward (functional.py:1730-1734) + the
 * autograd backward of joint.py:57-68.  Recomputes logits tiles; grad_costs [B] is dL/dcost_b
 * (1/B for reduction='mean').  Outputs are OVERWRITTEN: d_enc_proj [B,T,D], d_pred_proj
 * [B,U1,D], d_w_out [V,D], d_b_out [V]. */
size_t ctcvr_joint_rnnt_bwd_ws_bytes(int B, int T, int U1, int D, int V, int precision);
int ctcvr_joint_rnnt_bwd(const float* enc_proj, const float* pred_proj, const float* w_out,
                         const float* b_out, const int32_t* targets, const int32_t* t_len,
                         const int32_t* u_len, const float* lse, const float* lp_blank,
                         const float* lp_label, const float* alpha,
                         const float* beta, const float* costs, const float* grad_costs,
                         float clamp, float* d_enc_proj, float* d_pred_proj, float* d_w_out,
                         float* d_b_out, int B, int T, int U1, int D, int V, int blank,
                         int precision, void* ws, size_t ws_bytes, void* stream);

/* ---- bf16-input variants of the fused forward / backward (precision = CTCVR_BF16 implied): enc_proj / pred_proj
 * are bf16 tensors (what the reference's joint.enc_ffn / pred_ffn produce under torch.autocast), used in place -
 * no fp32 round trip - and the backward returns d_enc_proj / d_pred_proj as bf16 tensors of the same shapes (autograd
 * hands gradients back in the dtype of the inputs); d_w_out / d_b_out stay fp32.  ctcvr_joint_tc_supported() tells whether the shape fits the tensor-core tiling
 * (D % 128 == 0, D <= 512, V <= 512, U1 <= 128); other shapes must use the fp32-input entry points.
 * Workspace sizes are those of the fp32-input entry points with precision = CTCVR_BF16. */
int ctcvr_joint_tc_supported(int U1, int D, int V);
int ctcvr_joint_rnnt_fwd_bf16in(const void* enc_proj_bf16, const void* pred_proj_bf16, const float* w_out,
                                const float* b_out, const int32_t* targets, const int32_t* t_len,
                                const int32_t* u_len, float* lse, float* lp_blank, float* lp_label, int B,
                                int T, int U1, int D, int V, int blank, void* ws, size_t ws_bytes, void* stream);
int ctcvr_joint_rnnt_bwd_bf16in(const void* enc_proj_bf16, const void* pred_proj_bf16, const float* w_out,
                                const float* b_out, const int32_t* targets, const int32_t* t_len,
                                const int32_t* u_len, const float* lse, const float* lp_blank,
                                const float* lp_label, const float* alpha, const float* beta,
                                const float* costs, const float* grad_costs, float clamp, void* d_enc_proj_bf16,
                                void* d_pred_proj_bf16, float* d_w_out, float* d_b_out, int B, int T, int U1, int D,
                                int V, int blank, void* ws, size_t ws_bytes, void* stream);

/* ---- section 8(f)3: glue of Transducer._compute_rnnt_loss / forward (model/component/transducer.py:8-19,113,168,
 * 174-178,122-128).  ctcvr_rnnt_prologue: ys_in [B,U+1] int64 = [blank, text]; targets [B,U] int32 = text with
 * ignore_id -> 0; t_len / u_len [B] int32 from the int64 encoder lengths and the int32 (or int64) text lengths - one
 * launch.  ctcvr_loss_combine: out2[0] = transducer_weight * mean(costs) + ctc_weight * loss_ctc[0] (loss_ctc may be
 * NULL), out2[1] = mean(costs). */
int ctcvr_rnnt_prologue(const int64_t* text, const void* text_lens, int text_lens_are_int64, const int64_t* enc_lens,
                        int B, int U, int blank, int ignore_id, int64_t* ys_in, int32_t* targets, int32_t* t_len,
                        int32_t* u_len, void* stream);
int ctcvr_loss_combine(const float* costs, int B, const float* loss_ctc, float transducer_weight, float ctc_weight,
                       float* out2, void* stream);

/* ---- section 8(f)2: the predictor's LSTM over a whole label sequence (model/component/predictor.py:43-63,
 * `out, (m, c) = self.rnn(embed, states)`; one call per layer).  fp32, torch's gate order (i, f, g, o).
 * xg [B,U1,4H] = x_t W_ih^T + b_ih + b_hh for every step (one plain GEMM on the caller's side); w_hh [4H,H];
 * h0 / c0 [B,H] (NULL = zeros).  Forward writes out [B,U1,H] = h_t, hn / cn [B,H], and - for a later backward -
 * cs [B,U1,H] = c_t and act [B,U1,4H] = the activated gates (both may be NULL).  Backward takes d_out [B,U1,H] =
 * dL/dh_t (NULL = zeros), d_hn / d_cn [B,H] (NULL = zeros) and writes dgates [B,U1,4H] = dL/d(pre-activation gates)
 * - from which dW_ih, dW_hh, the bias gradients and dx are three plain GEMMs and a column sum - and d_h0 / d_c0 [B,H].
 * One persistent cooperative launch per call: needs H <= 8 x SM count (ctcvr_lstm_seq_supported); a CTA that waits
 * longer than 2 s for a step flag gives up and the NEXT call returns an error.  ws: ctcvr_lstm_seq_ws_bytes. */
int ctcvr_lstm_seq_supported(int B, int H);
size_t ctcvr_lstm_seq_ws_bytes(int B, int H);
int ctcvr_lstm_seq_fwd(const float* xg, const float* w_hh, const float* h0, const float* c0, float* out, float* cs,
                       float* act, float* hn, float* cn, int B, int U1, int H, void* ws, size_t ws_bytes, void* stream);
int ctcvr_lstm_seq_bwd(const float* act, const float* cs, const float* c0, const float* w_hh, const float* d_out,
                       const float* d_hn, const float* d_cn, float* dgates, float* d_h0, float* d_c0, int B, int U1,
                       int H, void* ws, size_t ws_bytes, void* stream);

/* Operand split for the plain fp32 products around the LSTM recurrence (x W_ih^T and the three gradient products): in
 * [rows, cols] fp32 -> the three TF32 terms stacked along the reduction dimension, so that A B ~= A_hi B_hi + A_hi B_lo +
 * A_lo B_hi is ONE tensor-core GEMM with fp32-level error (~2^-20).  stack_cols = 1: out [rows, 3*cols] (p0 | p1 | p2);
 * stack_cols = 0: out [3*rows, cols] (p0 over p1 over p2).  pattern 0 = (hi, hi, lo), 1 = (hi, lo, hi): one operand of
 * a product takes 0, the other 1. */
int ctcvr_split_tf32(const float* in, float* out, long rows, long cols, int stack_cols, int pattern, void* stream);

/* ---- section 8(f)4: calculate_cer (rnnt_eval.py:11-56) for N (hypothesis, reference) pairs: hyp [N,Lh], ref [N,Lr]
 * int32 padded, lengths [N]; out_sdin [N,4] int32 = substitutions, deletions, insertions, reference length, with the
 * reference's backtrace tie-breaking (match, substitution, deletion, insertion).  ws: ctcvr_cer_ws_bytes. */
size_t ctcvr_cer_ws_bytes(int N, int Lh, int Lr);
int ctcvr_cer_batch(const int32_t* hyp, const int32_t* hyp_len, int Lh, const int32_t* ref, const int32_t* ref_len, int Lr,
                    int N, void* ws, size_t ws_bytes, int32_t* out_sdin, void* stream);

/* ---- section 8(e): data-parallel gradient exchange over NVLink peer memory (replaces the all-reduce the reference
 * gets from torch DistributedDataParallel around the train step, rnnt_train.py:60-75).  One rank = one process = one
 * GPU of a node.  ctcvr_peer_create allocates the rank's staging buffer (room for max_floats payload floats, the
 * same value on every rank) and
 * returns its 64-byte CUDA IPC handle; the host exchanges the handles (any transport), ctcvr_peer_connect maps the
 * peers' buffers (handles: world x 64 bytes; or local_ptrs[world] = buffers of ranks living in THIS process, then
 * handles may be NULL).  ctcvr_peer_allreduce launches ONE kernel on `stream` that sums nseg fp32 tensors
 * (seg_ptrs[i], seg_floats[i] floats, <= 24 per call) over all ranks in place, in rank order 0..world-1, so every rank
 * ends with bit-identical sums; it can be captured in a CUDA graph.  Every rank must pass the same segment sizes and
 * the same `ctas` (<= 128, 0 = 128).  A rank that waits longer than the timeout (default 10 s) for a peer gives up and the
 * NEXT call returns an error.  world == 1: no launch. */
int ctcvr_peer_create(int rank, int world, size_t max_floats, void** out_ctx, void* out_handle64);
int ctcvr_peer_connect(void* ctx, const void* handles, void* const* local_ptrs);
void* ctcvr_peer_local_buffer(void* ctx);
int ctcvr_peer_set_timeout_ms(void* ctx, long ms);
int ctcvr_peer_allreduce(void* ctx, void* const* seg_ptrs, const long* seg_floats, int nseg, int ctas, void* stream);
int ctcvr_peer_destroy(void* ctx);

/* ---- A2 on dense logits — torch.ops.torchaudio.rnnt_loss_forward
 * (site-packages/torchaudio/functional/functional.py:1725,1737-1744), fused_log_softmax=True.
 * logits [B,T,U1,V] fp32; costs [B]; grads [B,T,U1,V] (may be NULL) = d cost_b / d logits,
 * exact zeros at padded cells, clamped to +-clamp when clamp > 0.
 * ws: 5*B*T*U1 floats (ctcvr_rnnt_loss_dense_ws_bytes). */
size_t ctcvr_rnnt_loss_dense_ws_bytes(int B, int T, int U1);
int ctcvr_rnnt_loss_dense(const float* logits, const int32_t* targets, const int32_t* t_len,
                          const int32_t* u_len, float* costs, float* grads, int B, int T,
                          int U1, int V, int blank, float clamp, void* ws, size_t ws_bytes,
                          void* stream);

/* ---- A4 CTC head tail — F.log_softmax + nn.CTCLoss(blank, zero_infinity=True) as used at
 * model/rnnt_model.py:55-58, model/online_rnnt_model.py:29-30, model/model.py:289-293.
 * ctcvr_log_softmax: y[r,:] = log_softmax(x[r,:]) over rows x V.
 * ctcvr_ctc_loss: log_probs [B,T,V]; targets [B,Umax] int64 (as the reference passes them);
 * nll [B] (inf -> 0 when zero_infinity); grad_logits [B,T,V] (may be NULL) = d nll_b/d logits
 * scaled by grad_scale[b]; ws: ctcvr_ctc_loss_ws_bytes.  Umax <= 511.  in_lens are clamped to
 * [0, T] and tgt_lens to [0, Umax]: a negative length behaves exactly like 0.  A label outside
 * [0, V) behaves exactly like blank, in the cost and the gradient, whichever kernel runs. */
int ctcvr_log_softmax(const float* x, float* y, long rows, int V, void* stream);
size_t ctcvr_ctc_loss_ws_bytes(int B, int T, int Umax);
int ctcvr_ctc_loss(const float* log_probs, const int64_t* targets, const int32_t* in_lens,
                   const int32_t* tgt_lens, const float* grad_scale, float* nll,
                   float* grad_logits, int B, int T, int V, int Umax, int blank,
                   int zero_infinity, void* ws, size_t ws_bytes, void* stream);

/* ---- A10 CTC greedy — model/rnnt_model.py:188-210, model/online_rnnt_model.py:647-671,
 * wenet/transformer/search.py:107-122: per-frame argmax, collapse repeats, drop blank.
 * scores [B,T,V] (logits or log-probs); out_tokens [B,T] int32; out_lens [B] int32. */
int ctcvr_ctc_greedy(const float* scores, const int32_t* lens, int32_t* out_tokens,
                     int32_t* out_lens, int B, int T, int V, int blank, void* stream);

/* ---- Forced alignment: the best (Viterbi) path of a known transcript, batched, one CTA per utterance
 * (csrc/align.cu).  Lengths are clamped to the tensor extents (a negative length acts as 0) and a CTC label outside
 * [0, V) acts as blank, as in the loss entry points.  An utterance without a path of finite log-probability (T_b = 0;
 * CTC: T_b < U_b + repeated neighbours; or every path crossing a -inf log-prob) gets score -inf and -1 in every frame,
 * label and span entry; no error is raised.  ws: the _ws_bytes query (0 when the shapes take the shared-memory form;
 * ws may then be NULL).
 *
 * ctcvr_rnnt_viterbi: lp_blank / lp_label [B,T,U1] as ctcvr_joint_rnnt_fwd writes them.  delta(0,0) = 0,
 * delta(t,u) = max(delta(t-1,u) + lp_blank(t-1,u), delta(t,u-1) + lp_label(t,u-1)); scores [B] = delta(T_b-1,U_b) +
 * lp_blank(T_b-1,U_b).  frames [B,U1-1] int32 = the frame at which label u is emitted (non-decreasing; -1 beyond U_b),
 * token_logprobs [B,U1-1] = lp_label at that cell (0 beyond U_b).  An exact tie takes the blank predecessor (t-1,u):
 * the label is emitted at the earlier frame.
 * ctcvr_ctc_viterbi: log_probs [B,T,V], targets [B,Umax] int64 (padded, as ctcvr_ctc_loss takes them), Umax <= 511.
 * labels [B,T] int32 = per frame the blank or the label of the best path's state (-1 for t >= T_b), frame_logprobs
 * [B,T] = its log-prob (0 for t >= T_b), scores [B], spans [B,Umax,2] int32 = first frame and last frame + 1 of each
 * target token (torchaudio.functional.merge_tokens' convention; -1 beyond U_b).  State s-2 is a predecessor of s only
 * when label(s) != blank and label(s) != label(s-2); an exact tie takes the smaller jump, and between the two end
 * states the final blank. */
size_t ctcvr_rnnt_viterbi_ws_bytes(int B, int T, int U1);
int ctcvr_rnnt_viterbi(const float* lp_blank, const float* lp_label, const int32_t* t_len, const int32_t* u_len,
                       int32_t* frames, float* token_logprobs, float* scores, int B, int T, int U1, void* ws,
                       size_t ws_bytes, void* stream);
size_t ctcvr_ctc_viterbi_ws_bytes(int B, int T, int Umax);
int ctcvr_ctc_viterbi(const float* log_probs, const int64_t* targets, const int32_t* in_lens, const int32_t* tgt_lens,
                      int32_t* labels, float* frame_logprobs, float* scores, int32_t* spans, int B, int T, int V,
                      int Umax, int blank, void* ws, size_t ws_bytes, void* stream);

/* Predictor + joint weights for the on-device decoders, in the layouts the kernels stream
 * (all fp32, device).  Source parameters: model/component/predictor.py:27-38 /
 * wenet/transducer/predictor.py:60-89 (embed, rnn.weight_ih_l*, rnn.weight_hh_l*, rnn.bias_*,
 * projection) and model/component/joint.py:38-46 (pred_ffn, ffn_out).  The host shim
 * (ctc-vr_b200/decode.py::prepare_decoder_weights) derives them once per weight version:
 * "_t" = transposed so that consecutive threads (output rows) read consecutive addresses. */
typedef struct {
  const float* gate_tok;   /* [V,4H]     embed . W_ih_l0^T + b_ih_l0 + b_hh_l0 (gate order i,f,g,o) */
  const float* w_hh_t;     /* [L][H,4H]  W_hh_l^T */
  const float* w_ih_t;     /* [L-1][H,4H] W_ih_l^T for layers >= 1 (NULL when L == 1) */
  const float* b_gate;     /* [L-1][4H]  b_ih_l + b_hh_l for layers >= 1 (NULL when L == 1) */
  const float* proj_t;     /* [H,P]      projection.weight^T */
  const float* proj_b;     /* [P] */
  const float* pred_ffn_t; /* [P,D]      joint.pred_ffn.weight^T */
  const float* pred_ffn_b; /* [D] */
  const float* out_t;      /* [D,V]      joint.ffn_out.weight^T */
  const float* out_b;      /* [V] */
  int V, H, L, P, D;
  int activation;          /* joint activation: CTCVR_ACT_TANH (0) / CTCVR_ACT_RELU / CTCVR_ACT_GELU.  A post-join
                              linear is folded in by the caller: pred_ffn_t <- pred_ffn_t W_post^T, pred_ffn_b <-
                              W_post pred_ffn_b, and enc_proj = post_ffn(enc_ffn(encoder_out)) */
} ctcvr_decoder_weights;

/* ---- A5/A6/A6' greedy — model/component/transducer.py:22-70 (n_steps=64, fresh state),
 * model/online_rnnt_model.py:166-222 (n_steps=10, state carried across chunks),
 * wenet/transducer/search/greedy_search.py:6-54.
 * enc_proj [N,T,D] = enc_ffn(encoder_out); lens [N]; h,c [L,N,H] in/out; last_token [N]
 * in/out; out_tokens [N,max_out] int32; out_lens [N]. No host sync per step. */
size_t ctcvr_rnnt_greedy_ws_bytes(const ctcvr_decoder_weights* w, int N);
int ctcvr_rnnt_greedy(const ctcvr_decoder_weights* w, const float* enc_proj,
                      const int32_t* lens, float* h, float* c, int32_t* last_token,
                      int32_t* out_tokens, int32_t* out_lens, int N, int T, int max_out,
                      int blank, int n_steps, void* ws, size_t ws_bytes, void* stream);

/* ---- A7 online beam — model/online_rnnt_model.py:389-522.  One stream (batch 1), beam state
 * carried across chunks in `beam_state` (opaque, ctcvr_rnnt_beam_state_bytes).  After the
 * call: out_n hyps, out_tokens [beam,max_out], out_lens [beam], out_scores [beam] fp64, and
 * out_h/out_c [beam,L,H] predictor states, ordered as the reference's list. */
size_t ctcvr_rnnt_beam_state_bytes(const ctcvr_decoder_weights* w, int beam, int n_steps, int max_out);
int ctcvr_rnnt_beam_reset(void* beam_state, const ctcvr_decoder_weights* w, int beam, int n_steps,
                          int max_out, void* stream);
int ctcvr_rnnt_beam_chunk(const ctcvr_decoder_weights* w, const float* enc_proj, int T,
                          void* beam_state, int beam, int n_steps, int max_out, int blank,
                          int32_t* out_n, int32_t* out_tokens, int32_t* out_lens,
                          double* out_scores, float* out_h, float* out_c, void* stream);

/* A7 for S independent streams in ONE launch (one CTA per stream; the reference decodes one stream at a time,
 * online_rnnt_model.py:277-278 - the per-stream arithmetic is unchanged, so every stream's hypotheses equal the
 * single-stream call's).  beam_states: S consecutive states of ctcvr_rnnt_beam_state_bytes each; enc_proj [S,T,D];
 * chunk_lens [S] frames of each stream's chunk (<= T; NULL = T for all); outputs carry a leading S dimension:
 * out_n [S], out_tokens [S,beam,max_out], out_lens / out_scores [S,beam], out_h / out_c [S,beam,L,H]. */
int ctcvr_rnnt_beam_reset_batch(void* beam_states, const ctcvr_decoder_weights* w, int S, int beam, int n_steps,
                                int max_out, void* stream);
int ctcvr_rnnt_beam_chunk_batch(const ctcvr_decoder_weights* w, const float* enc_proj, const int32_t* chunk_lens,
                                int S, int T, void* beam_states, int beam, int n_steps, int max_out, int blank,
                                int32_t* out_n, int32_t* out_tokens, int32_t* out_lens, double* out_scores,
                                float* out_h, float* out_c, void* stream);

/* ---- A8 wenet transducer prefix beam with CTC shallow fusion —
 * wenet/transducer/search/prefix_beam_search.py:42-148.  enc_proj [T,D]; ctc_logp [T,V] (log-probs);
 * out_tokens [beam][T+1] (every hypothesis starts with the blank, as in the reference), out_lens [beam],
 * out_scores [beam] fp64, out_n [1], best first.  beam <= 16. */
size_t ctcvr_rnnt_prefix_beam_ws_bytes(const ctcvr_decoder_weights* w, int beam, int T);
int ctcvr_rnnt_prefix_beam(const ctcvr_decoder_weights* w, const float* enc_proj,
                           const float* ctc_logp, int T, int beam, int blank, float ctc_weight,
                           float transducer_weight, int32_t* out_n, int32_t* out_tokens,
                           int32_t* out_lens, double* out_scores, void* ws, size_t ws_bytes,
                           void* stream);

/* A8 for S utterances in ONE launch (one CTA per utterance): enc_proj [S,T,D], ctc_logp [S,T,V], lens [S] frames per
 * utterance (<= T; NULL = T), out_n [S], out_tokens [S,beam,T+1], out_lens / out_scores [S,beam];
 * ws: S x ctcvr_rnnt_prefix_beam_ws_bytes(w, beam, T). */
int ctcvr_rnnt_prefix_beam_batch(const ctcvr_decoder_weights* w, const float* enc_proj, const float* ctc_logp,
                                 const int32_t* lens, int S, int T, int beam, int blank, float ctc_weight,
                                 float transducer_weight, int32_t* out_n, int32_t* out_tokens, int32_t* out_lens,
                                 double* out_scores, void* ws, size_t ws_bytes, void* stream);

/* ---- A9 CTC prefix beam search — wenet/transformer/search.py:125-247 (context_graph=None).
 * ctc_probs [B,T,V] log-probs; per utterance up to `beam` hyps: out_tokens [B,beam,T],
 * out_lens [B,beam], out_scores [B,beam] fp64 (log_add(s,ns)), out_times [B,beam,T],
 * out_n [B]. */
size_t ctcvr_ctc_prefix_beam_ws_bytes(int B, int T, int V, int beam);
int ctcvr_ctc_prefix_beam(const float* ctc_probs, const int32_t* lens, int B, int T, int V,
                          int beam, int blank, int32_t* out_n, int32_t* out_tokens,
                          int32_t* out_lens, double* out_scores, int32_t* out_times,
                          void* ws, size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CTCVR_H_ */
