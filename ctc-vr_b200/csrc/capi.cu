// extern "C" boundary of libctcvr.so (declared in include/ctcvr.h).  Argument validation lives here;
// every error becomes a non-zero return + ctcvr_last_error(), which the Python shim raises as
// RuntimeError (the reference's train loop relies on `except RuntimeError`, rnnt_train.py:139).
#include <stdarg.h>

#include "common.cuh"

namespace ctcvr {

static thread_local char g_err[1024] = "";
static unsigned long long g_launches = 0;
void count_launch() { __atomic_fetch_add(&g_launches, 1ULL, __ATOMIC_RELAXED); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// implemented in the other translation units
int joint_logits_f32(const float*, const float*, const float*, const float*, float*, int, int, int, int, int, cudaStream_t);
int joint_fwd_f32(const float*, const float*, const float*, const float*, const int32_t*, const int32_t*,
                  const int32_t*, float*, float*, float*, int, int, int, int, int, int, int, cudaStream_t);
size_t joint_bwd_f32_ws_bytes(int, int, int, int, int);
int joint_bwd_f32(const float*, const float*, const float*, const float*, const int32_t*, const int32_t*,
                  const int32_t*, const float*, const float*, const float*, const float*, const float*, float, float*,
                  float*, float*, float*, int, int, int, int, int, int, int, void*, size_t, cudaStream_t);
size_t joint_fwd_tc_ws_bytes(int, int, int, int, int, int);
int joint_fwd_tc(const void*, const void*, int, int, int, const float*, const float*, const int32_t*, const int32_t*,
                 const int32_t*, float*, float*, float*, int, int, int, int, int, int, void*, size_t, cudaStream_t);
bool joint_tc_bwd_supported(int, int, int);
size_t joint_bwd_tc_ws_bytes(int, int, int, int, int, int);
int joint_bwd_tc(const void*, const void*, int, int, int, const float*, const float*, const int32_t*, const int32_t*,
                 const int32_t*, const float*, const float*, const float*, const float*, const float*, const float*,
                 const float*, float, float*,
                 float*, float*, float*, int, int, int, int, int, int, void*, size_t, cudaStream_t);
int rnnt_lattice(const float*, const float*, const int32_t*, const int32_t*, float*, float*, float*, int, int, int,
                 cudaStream_t);
int rnnt_loss_dense(const float*, const int32_t*, const int32_t*, const int32_t*, float*, float*, int, int, int, int,
                    int, float, void*, size_t, cudaStream_t);
int log_softmax(const float*, float*, long, int, cudaStream_t);
size_t ctc_loss_ws_bytes(int, int, int);
int ctc_loss(const float*, const int64_t*, const int32_t*, const int32_t*, const float*, float*, float*, int, int, int,
             int, int, int, void*, size_t, cudaStream_t);
int ctc_greedy(const float*, const int32_t*, int32_t*, int32_t*, int, int, int, int, cudaStream_t);
size_t rnnt_viterbi_ws_bytes(int, int, int);
int rnnt_viterbi(const float*, const float*, const int32_t*, const int32_t*, int32_t*, float*, float*, int, int, int, void*,
                 size_t, cudaStream_t);
size_t ctc_viterbi_ws_bytes(int, int, int);
int ctc_viterbi(const float*, const int64_t*, const int32_t*, const int32_t*, int32_t*, float*, float*, int32_t*, int, int,
                int, int, int, void*, size_t, cudaStream_t);
int rnnt_greedy(const ctcvr_decoder_weights&, const float*, const int32_t*, float*, float*, int32_t*, int32_t*,
                int32_t*, int, int, int, int, int, cudaStream_t);
size_t rnnt_beam_state_bytes(const ctcvr_decoder_weights&, int, int, int);
int rnnt_beam_reset(void*, const ctcvr_decoder_weights&, int, int, int, int, cudaStream_t);
int rnnt_beam_chunk(const ctcvr_decoder_weights&, const float*, const int32_t*, int, int, void*, int, int, int, int, int32_t*,
                    int32_t*, int32_t*, double*, float*, float*, cudaStream_t);
size_t rnnt_prefix_beam_ws_bytes(const ctcvr_decoder_weights&, int, int);
int rnnt_prefix_beam(const ctcvr_decoder_weights&, const float*, const float*, const int32_t*, int, int, int, int, float,
                     float, int32_t*, int32_t*, int32_t*, double*, void*, size_t, cudaStream_t);
size_t ctc_prefix_beam_ws_bytes(int, int, int, int);
int ctc_prefix_beam(const float*, const int32_t*, int, int, int, int, int, int32_t*, int32_t*, int32_t*, double*,
                    int32_t*, void*, size_t, cudaStream_t);

int rnnt_prologue(const int64_t*, const void*, int, const int64_t*, int, int, int, int, int64_t*, int32_t*, int32_t*,
                  int32_t*, cudaStream_t);
int loss_combine(const float*, int, const float*, float, float, float*, cudaStream_t);
size_t cer_ws_bytes(int, int, int);
int cer_batch(const int32_t*, const int32_t*, int, const int32_t*, const int32_t*, int, int, void*, size_t, int32_t*,
              cudaStream_t);

int lstm_seq_supported(int, int);
size_t lstm_seq_ws_bytes(int, int);
int lstm_seq_fwd(const float*, const float*, const float*, const float*, float*, float*, float*, float*, float*, int, int, int,
                 void*, size_t, cudaStream_t);
int lstm_seq_bwd(const float*, const float*, const float*, const float*, const float*, const float*, const float*, float*,
                 float*, float*, int, int, int, void*, size_t, cudaStream_t);

int split_tf32(const float*, float*, long, long, int, int, cudaStream_t);

int peer_create(int, int, size_t, void**, void*);
int peer_connect(void*, const void*, void* const*);
void* peer_local_buffer(void*);
int peer_set_timeout_ms(void*, long);
int peer_allreduce(void*, void* const*, const long*, int, int, cudaStream_t);
int peer_destroy(void*);
void peer_set_prof(void*);
void peer_set_mode(int);

unsigned int tc_error_flag();
void tc_set_prof(void*);
void tc_set_mode(int);

static int check_dims(const char* op, int B, int T, int U1, int D, int V) {
  CTCVR_REQUIRE(B > 0 && T > 0 && U1 > 0 && D > 0 && V > 0, "%s: bad dims B=%d T=%d U1=%d D=%d V=%d", op, B, T, U1, D, V);
  return 0;
}

// `precision` of the fused joint entry points: CTCVR_F32 / CTCVR_BF16 / CTCVR_BF16X3 in the low byte, OR'ed with one
// CTCVR_ACT_* value.  Splits it into (precision, activation); false for any other bit.
static bool split_precision(int precision, int* prec, int* act) {
  *prec = precision & 0xff;
  *act = (precision & ~0xff) >> 8;
  return (*prec == CTCVR_F32 || *prec == CTCVR_BF16 || *prec == CTCVR_BF16X3) &&
         (*act == ACT_TANH || *act == ACT_RELU || *act == ACT_GELU);
}
#define CTCVR_SPLIT_PRECISION(op, precision, prec, act)                                                          \
  CTCVR_REQUIRE(split_precision(precision, &prec, &act),                                                          \
                "%s: unknown precision 0x%x (low byte: CTCVR_F32 / CTCVR_BF16 / CTCVR_BF16X3, OR'ed with one of "  \
                "CTCVR_ACT_TANH / CTCVR_ACT_RELU / CTCVR_ACT_GELU)", op, (unsigned)(precision))

static int check_weights(const char* op, const ctcvr_decoder_weights* w) {
  CTCVR_REQUIRE(w != nullptr, "%s: weights is NULL", op);
  CTCVR_REQUIRE(w->V > 0 && w->H > 0 && w->L > 0 && w->P > 0 && w->D > 0, "%s: bad weight dims", op);
  CTCVR_REQUIRE(w->gate_tok && w->w_hh_t && w->proj_t && w->proj_b && w->pred_ffn_t && w->pred_ffn_b && w->out_t &&
                    w->out_b && (w->L == 1 || (w->w_ih_t && w->b_gate)),
                "%s: NULL weight pointer", op);
  CTCVR_REQUIRE(w->activation == CTCVR_ACT_TANH || w->activation == CTCVR_ACT_RELU || w->activation == CTCVR_ACT_GELU,
                "%s: unknown activation 0x%x (CTCVR_ACT_TANH / CTCVR_ACT_RELU / CTCVR_ACT_GELU)", op,
                (unsigned)w->activation);
  return 0;
}

}  // namespace ctcvr

using namespace ctcvr;
#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" {

const char* ctcvr_last_error(void) { return g_err; }
int ctcvr_version(void) { return 100; }
unsigned int ctcvr_debug_tc_error(void) { return tc_error_flag(); }
void ctcvr_debug_set_prof(void* buf) { tc_set_prof(buf); peer_set_prof(buf); }
void ctcvr_debug_set_mode(int mode) { tc_set_mode(mode & 3); peer_set_mode(mode >> 2); }
unsigned long long ctcvr_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

int ctcvr_joint_logits(const float* enc_proj, const float* pred_proj, const float* w_out, const float* b_out,
                       float* logits, int B, int T, int U1, int D, int V, void* stream) {
  if (int rc = check_dims("joint_logits", B, T, U1, D, V)) return rc;
  CTCVR_REQUIRE(enc_proj && pred_proj && w_out && b_out && logits, "joint_logits: NULL pointer");
  return joint_logits_f32(enc_proj, pred_proj, w_out, b_out, logits, B, T, U1, D, V, ST(stream));
}

size_t ctcvr_joint_rnnt_fwd_ws_bytes(int B, int T, int U1, int D, int V, int precision) {
  precision &= 0xff;                        // the activation bits do not change the workspace
  if (precision == CTCVR_BF16 || precision == CTCVR_BF16X3)
    return joint_fwd_tc_ws_bytes(B, T, U1, D, V, precision == CTCVR_BF16X3);
  return 256;
}

int ctcvr_joint_rnnt_fwd(const float* enc_proj, const float* pred_proj, const float* w_out, const float* b_out,
                         const int32_t* targets, const int32_t* t_len, const int32_t* u_len, float* lse,
                         float* lp_blank, float* lp_label, int B, int T, int U1, int D, int V, int blank,
                         int precision, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_dims("joint_rnnt_fwd", B, T, U1, D, V)) return rc;
  CTCVR_REQUIRE(enc_proj && pred_proj && w_out && b_out && t_len && u_len && lse && lp_blank && lp_label &&
                    (targets || U1 == 1), "joint_rnnt_fwd: NULL pointer");
  CTCVR_REQUIRE(blank >= 0 && blank < V, "joint_rnnt_fwd: blank %d must be within [0, %d)", blank, V);
  int prec = 0, act = 0;
  CTCVR_SPLIT_PRECISION("joint_rnnt_fwd", precision, prec, act);
  precision = prec;
  if (precision == CTCVR_BF16 || precision == CTCVR_BF16X3)
    return joint_fwd_tc(enc_proj, pred_proj, 0, precision == CTCVR_BF16X3, act, w_out, b_out, targets, t_len, u_len, lse, lp_blank, lp_label, B, T, U1, D,
                        V, blank, ws, ws_bytes, ST(stream));
  return joint_fwd_f32(enc_proj, pred_proj, w_out, b_out, targets, t_len, u_len, lse, lp_blank, lp_label, B, T, U1, D,
                       V, blank, act, ST(stream));
}

int ctcvr_rnnt_lattice(const float* lp_blank, const float* lp_label, const int32_t* t_len, const int32_t* u_len,
                       float* alpha, float* beta, float* costs, int B, int T, int U1, void* stream) {
  CTCVR_REQUIRE(B > 0 && T > 0 && U1 > 0, "rnnt_lattice: bad dims");
  CTCVR_REQUIRE(lp_blank && lp_label && t_len && u_len && alpha && beta && costs, "rnnt_lattice: NULL pointer");
  return rnnt_lattice(lp_blank, lp_label, t_len, u_len, alpha, beta, costs, B, T, U1, ST(stream));
}

size_t ctcvr_joint_rnnt_bwd_ws_bytes(int B, int T, int U1, int D, int V, int precision) {
  precision &= 0xff;                        // the activation bits do not change the workspace
  if (precision == CTCVR_BF16 || precision == CTCVR_BF16X3)
    return joint_bwd_tc_ws_bytes(B, T, U1, D, V, precision == CTCVR_BF16X3);
  return joint_bwd_f32_ws_bytes(B, T, U1, D, V);
}

int ctcvr_joint_rnnt_bwd(const float* enc_proj, const float* pred_proj, const float* w_out, const float* b_out,
                         const int32_t* targets, const int32_t* t_len, const int32_t* u_len, const float* lse,
                         const float* lp_blank, const float* lp_label,
                         const float* alpha, const float* beta, const float* costs, const float* grad_costs,
                         float clamp, float* d_enc_proj, float* d_pred_proj, float* d_w_out, float* d_b_out, int B,
                         int T, int U1, int D, int V, int blank, int precision, void* ws, size_t ws_bytes,
                         void* stream) {
  if (int rc = check_dims("joint_rnnt_bwd", B, T, U1, D, V)) return rc;
  CTCVR_REQUIRE(enc_proj && pred_proj && w_out && b_out && t_len && u_len && lse && lp_blank && lp_label && alpha &&
                    beta && costs && grad_costs && d_enc_proj && d_pred_proj && d_w_out && d_b_out && ws,
                "joint_rnnt_bwd: NULL pointer");
  CTCVR_REQUIRE(blank >= 0 && blank < V, "joint_rnnt_bwd: blank %d must be within [0, %d)", blank, V);
  int prec = 0, act = 0;
  CTCVR_SPLIT_PRECISION("joint_rnnt_bwd", precision, prec, act);
  precision = prec;
  if (precision == CTCVR_BF16 || precision == CTCVR_BF16X3)
    return joint_bwd_tc(enc_proj, pred_proj, 0, precision == CTCVR_BF16X3, act, w_out, b_out, targets, t_len, u_len, lse, lp_blank, lp_label, alpha, beta, costs, grad_costs,
                        clamp, d_enc_proj, d_pred_proj, d_w_out, d_b_out, B, T, U1, D, V, blank, ws, ws_bytes,
                        ST(stream));
  return joint_bwd_f32(enc_proj, pred_proj, w_out, b_out, targets, t_len, u_len, lse, alpha, beta, costs, grad_costs,
                       clamp, d_enc_proj, d_pred_proj, d_w_out, d_b_out, B, T, U1, D, V, blank, act, ws, ws_bytes,
                       ST(stream));
}

int ctcvr_joint_tc_supported(int U1, int D, int V) { return joint_tc_bwd_supported(U1, D, V) ? 1 : 0; }

int ctcvr_joint_rnnt_fwd_bf16in(const void* enc_proj_bf16, const void* pred_proj_bf16, const float* w_out,
                                const float* b_out, const int32_t* targets, const int32_t* t_len, const int32_t* u_len,
                                float* lse, float* lp_blank, float* lp_label, int B, int T, int U1, int D, int V,
                                int blank, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_dims("joint_rnnt_fwd_bf16in", B, T, U1, D, V)) return rc;
  CTCVR_REQUIRE(enc_proj_bf16 && pred_proj_bf16 && w_out && b_out && t_len && u_len && lse && lp_blank && lp_label &&
                    (targets || U1 == 1), "joint_rnnt_fwd_bf16in: NULL pointer");
  CTCVR_REQUIRE(blank >= 0 && blank < V, "joint_rnnt_fwd_bf16in: blank %d must be within [0, %d)", blank, V);
  return joint_fwd_tc(enc_proj_bf16, pred_proj_bf16, 1, 0, ACT_TANH, w_out, b_out, targets, t_len, u_len, lse, lp_blank, lp_label, B,
                      T, U1, D, V, blank, ws, ws_bytes, ST(stream));
}

int ctcvr_joint_rnnt_bwd_bf16in(const void* enc_proj_bf16, const void* pred_proj_bf16, const float* w_out,
                                const float* b_out, const int32_t* targets, const int32_t* t_len, const int32_t* u_len,
                                const float* lse, const float* lp_blank, const float* lp_label, const float* alpha,
                                const float* beta, const float* costs,
                                const float* grad_costs, float clamp, void* d_enc_proj_bf16, void* d_pred_proj_bf16,
                                float* d_w_out, float* d_b_out, int B, int T, int U1, int D, int V, int blank, void* ws,
                                size_t ws_bytes, void* stream) {
  if (int rc = check_dims("joint_rnnt_bwd_bf16in", B, T, U1, D, V)) return rc;
  CTCVR_REQUIRE(enc_proj_bf16 && pred_proj_bf16 && w_out && b_out && t_len && u_len && lse && lp_blank && lp_label &&
                    alpha && beta && costs && grad_costs && d_enc_proj_bf16 && d_pred_proj_bf16 && d_w_out && d_b_out && ws, "joint_rnnt_bwd_bf16in: NULL pointer");
  CTCVR_REQUIRE(blank >= 0 && blank < V, "joint_rnnt_bwd_bf16in: blank %d must be within [0, %d)", blank, V);
  return joint_bwd_tc(enc_proj_bf16, pred_proj_bf16, 1, 0, ACT_TANH, w_out, b_out, targets, t_len, u_len, lse, lp_blank, lp_label, alpha, beta, costs,
                      grad_costs, clamp, reinterpret_cast<float*>(d_enc_proj_bf16), reinterpret_cast<float*>(d_pred_proj_bf16),
                      d_w_out, d_b_out, B, T, U1, D, V, blank, ws, ws_bytes, ST(stream));
}

int ctcvr_rnnt_prologue(const int64_t* text, const void* text_lens, int text_lens_are_int64, const int64_t* enc_lens,
                        int B, int U, int blank, int ignore_id, int64_t* ys_in, int32_t* targets, int32_t* t_len,
                        int32_t* u_len, void* stream) {
  CTCVR_REQUIRE(B > 0 && U >= 0, "rnnt_prologue: bad dims");
  CTCVR_REQUIRE(text_lens && enc_lens && ys_in && t_len && u_len && (U == 0 || (text && targets)), "rnnt_prologue: NULL pointer");
  return rnnt_prologue(text, text_lens, text_lens_are_int64, enc_lens, B, U, blank, ignore_id, ys_in, targets, t_len, u_len,
                       ST(stream));
}

int ctcvr_loss_combine(const float* costs, int B, const float* loss_ctc, float transducer_weight, float ctc_weight,
                       float* out2, void* stream) {
  CTCVR_REQUIRE(costs && out2 && B > 0, "loss_combine: bad arguments");
  return loss_combine(costs, B, loss_ctc, transducer_weight, ctc_weight, out2, ST(stream));
}

size_t ctcvr_cer_ws_bytes(int N, int Lh, int Lr) { return cer_ws_bytes(N, Lh, Lr); }

int ctcvr_cer_batch(const int32_t* hyp, const int32_t* hyp_len, int Lh, const int32_t* ref, const int32_t* ref_len, int Lr,
                    int N, void* ws, size_t ws_bytes, int32_t* out_sdin, void* stream) {
  CTCVR_REQUIRE(N > 0 && Lh >= 0 && Lr >= 0, "cer_batch: bad dims");
  CTCVR_REQUIRE(hyp_len && ref_len && out_sdin && ws && (Lh == 0 || hyp) && (Lr == 0 || ref), "cer_batch: NULL pointer");
  return cer_batch(hyp, hyp_len, Lh, ref, ref_len, Lr, N, ws, ws_bytes, out_sdin, ST(stream));
}

int ctcvr_lstm_seq_supported(int B, int H) { return lstm_seq_supported(B, H); }
size_t ctcvr_lstm_seq_ws_bytes(int B, int H) { return (B > 0 && H > 0) ? lstm_seq_ws_bytes(B, H) : 0; }

int ctcvr_lstm_seq_fwd(const float* xg, const float* w_hh, const float* h0, const float* c0, float* out, float* cs,
                       float* act, float* hn, float* cn, int B, int U1, int H, void* ws, size_t ws_bytes, void* stream) {
  CTCVR_REQUIRE(B > 0 && U1 > 0 && H > 0, "lstm_seq_fwd: bad dims");
  CTCVR_REQUIRE(xg && w_hh && out && hn && cn && ws, "lstm_seq_fwd: NULL pointer");
  return lstm_seq_fwd(xg, w_hh, h0, c0, out, cs, act, hn, cn, B, U1, H, ws, ws_bytes, ST(stream));
}

int ctcvr_lstm_seq_bwd(const float* act, const float* cs, const float* c0, const float* w_hh, const float* d_out,
                       const float* d_hn, const float* d_cn, float* dgates, float* d_h0, float* d_c0, int B, int U1,
                       int H, void* ws, size_t ws_bytes, void* stream) {
  CTCVR_REQUIRE(B > 0 && U1 > 0 && H > 0, "lstm_seq_bwd: bad dims");
  CTCVR_REQUIRE(act && cs && w_hh && dgates && d_h0 && d_c0 && ws, "lstm_seq_bwd: NULL pointer");
  return lstm_seq_bwd(act, cs, c0, w_hh, d_out, d_hn, d_cn, dgates, d_h0, d_c0, B, U1, H, ws, ws_bytes, ST(stream));
}

int ctcvr_split_tf32(const float* in, float* out, long rows, long cols, int stack_cols, int pattern, void* stream) {
  CTCVR_REQUIRE(in && out && rows > 0 && cols > 0 && (pattern == 0 || pattern == 1), "split_tf32: bad arguments");
  return split_tf32(in, out, rows, cols, stack_cols, pattern, ST(stream));
}

int ctcvr_peer_create(int rank, int world, size_t max_floats, void** out_ctx, void* out_handle64) {
  return peer_create(rank, world, max_floats, out_ctx, out_handle64);
}
int ctcvr_peer_connect(void* ctx, const void* handles, void* const* local_ptrs) { return peer_connect(ctx, handles, local_ptrs); }
void* ctcvr_peer_local_buffer(void* ctx) { return peer_local_buffer(ctx); }
int ctcvr_peer_set_timeout_ms(void* ctx, long ms) { return peer_set_timeout_ms(ctx, ms); }
int ctcvr_peer_allreduce(void* ctx, void* const* seg_ptrs, const long* seg_floats, int nseg, int ctas, void* stream) {
  return peer_allreduce(ctx, seg_ptrs, seg_floats, nseg, ctas, ST(stream));
}
int ctcvr_peer_destroy(void* ctx) { return peer_destroy(ctx); }

size_t ctcvr_rnnt_loss_dense_ws_bytes(int B, int T, int U1) { return (size_t)5 * B * T * U1 * sizeof(float); }

int ctcvr_rnnt_loss_dense(const float* logits, const int32_t* targets, const int32_t* t_len, const int32_t* u_len,
                          float* costs, float* grads, int B, int T, int U1, int V, int blank, float clamp, void* ws,
                          size_t ws_bytes, void* stream) {
  CTCVR_REQUIRE(B > 0 && T > 0 && U1 > 0 && V > 0, "rnnt_loss_dense: bad dims");
  CTCVR_REQUIRE(logits && t_len && u_len && costs && ws && (targets || U1 == 1), "rnnt_loss_dense: NULL pointer");
  CTCVR_REQUIRE(blank >= 0 && blank < V, "rnnt_loss_dense: blank must be within [0, logits.shape[-1])");
  return rnnt_loss_dense(logits, targets, t_len, u_len, costs, grads, B, T, U1, V, blank, clamp, ws, ws_bytes,
                         ST(stream));
}

int ctcvr_log_softmax(const float* x, float* y, long rows, int V, void* stream) {
  CTCVR_REQUIRE(rows >= 0 && V > 0 && x && y, "log_softmax: bad arguments");
  return log_softmax(x, y, rows, V, ST(stream));
}

size_t ctcvr_ctc_loss_ws_bytes(int B, int T, int Umax) { return ctc_loss_ws_bytes(B, T, Umax); }

int ctcvr_ctc_loss(const float* log_probs, const int64_t* targets, const int32_t* in_lens, const int32_t* tgt_lens,
                   const float* grad_scale, float* nll, float* grad_logits, int B, int T, int V, int Umax, int blank,
                   int zero_infinity, void* ws, size_t ws_bytes, void* stream) {
  CTCVR_REQUIRE(B > 0 && T > 0 && V > 0 && Umax >= 0, "ctc_loss: bad dims");
  CTCVR_REQUIRE(log_probs && in_lens && tgt_lens && nll && ws && (targets || Umax == 0), "ctc_loss: NULL pointer");
  CTCVR_REQUIRE(blank >= 0 && blank < V, "ctc_loss: blank must be in label range");
  return ctc_loss(log_probs, targets, in_lens, tgt_lens, grad_scale, nll, grad_logits, B, T, V, Umax, blank,
                  zero_infinity, ws, ws_bytes, ST(stream));
}

int ctcvr_ctc_greedy(const float* scores, const int32_t* lens, int32_t* out_tokens, int32_t* out_lens, int B, int T,
                     int V, int blank, void* stream) {
  CTCVR_REQUIRE(B >= 0 && T > 0 && V > 0 && scores && lens && out_tokens && out_lens, "ctc_greedy: bad arguments");
  return ctc_greedy(scores, lens, out_tokens, out_lens, B, T, V, blank, ST(stream));
}

size_t ctcvr_rnnt_viterbi_ws_bytes(int B, int T, int U1) {
  return (B > 0 && T > 0 && U1 > 0) ? rnnt_viterbi_ws_bytes(B, T, U1) : 0;
}

int ctcvr_rnnt_viterbi(const float* lp_blank, const float* lp_label, const int32_t* t_len, const int32_t* u_len,
                       int32_t* frames, float* token_logprobs, float* scores, int B, int T, int U1, void* ws,
                       size_t ws_bytes, void* stream) {
  CTCVR_REQUIRE(B > 0 && T > 0 && U1 > 0, "rnnt_viterbi: bad dims B=%d T=%d U1=%d", B, T, U1);
  CTCVR_REQUIRE(lp_blank && lp_label && t_len && u_len && scores && (U1 == 1 || (frames && token_logprobs)),
                "rnnt_viterbi: NULL pointer");
  return rnnt_viterbi(lp_blank, lp_label, t_len, u_len, frames, token_logprobs, scores, B, T, U1, ws, ws_bytes,
                      ST(stream));
}

size_t ctcvr_ctc_viterbi_ws_bytes(int B, int T, int Umax) {
  return (B > 0 && T > 0 && Umax >= 0) ? ctc_viterbi_ws_bytes(B, T, Umax) : 0;
}

int ctcvr_ctc_viterbi(const float* log_probs, const int64_t* targets, const int32_t* in_lens, const int32_t* tgt_lens,
                      int32_t* labels, float* frame_logprobs, float* scores, int32_t* spans, int B, int T, int V,
                      int Umax, int blank, void* ws, size_t ws_bytes, void* stream) {
  CTCVR_REQUIRE(B > 0 && T > 0 && V > 0 && Umax >= 0, "ctc_viterbi: bad dims B=%d T=%d V=%d Umax=%d", B, T, V, Umax);
  CTCVR_REQUIRE(log_probs && in_lens && tgt_lens && labels && frame_logprobs && scores && (Umax == 0 || (targets && spans)),
                "ctc_viterbi: NULL pointer");
  CTCVR_REQUIRE(blank >= 0 && blank < V, "ctc_viterbi: blank %d must be within [0, %d)", blank, V);
  return ctc_viterbi(log_probs, targets, in_lens, tgt_lens, labels, frame_logprobs, scores, spans, B, T, V, Umax, blank,
                     ws, ws_bytes, ST(stream));
}

size_t ctcvr_rnnt_greedy_ws_bytes(const ctcvr_decoder_weights* w, int N) { (void)w; (void)N; return 256; }

int ctcvr_rnnt_greedy(const ctcvr_decoder_weights* w, const float* enc_proj, const int32_t* lens, float* h, float* c,
                      int32_t* last_token, int32_t* out_tokens, int32_t* out_lens, int N, int T, int max_out,
                      int blank, int n_steps, void* ws, size_t ws_bytes, void* stream) {
  (void)ws; (void)ws_bytes;
  if (int rc = check_weights("rnnt_greedy", w)) return rc;
  CTCVR_REQUIRE(N >= 0 && T > 0 && max_out > 0 && n_steps > 0, "rnnt_greedy: bad dims");
  CTCVR_REQUIRE(enc_proj && lens && h && c && last_token && out_tokens && out_lens, "rnnt_greedy: NULL pointer");
  CTCVR_REQUIRE(blank >= 0 && blank < w->V, "rnnt_greedy: blank out of range");
  return rnnt_greedy(*w, enc_proj, lens, h, c, last_token, out_tokens, out_lens, N, T, max_out, blank, n_steps,
                     ST(stream));
}

size_t ctcvr_rnnt_beam_state_bytes(const ctcvr_decoder_weights* w, int beam, int n_steps, int max_out) {
  return w ? rnnt_beam_state_bytes(*w, beam, n_steps, max_out) : 0;
}

int ctcvr_rnnt_beam_reset(void* beam_state, const ctcvr_decoder_weights* w, int beam, int n_steps, int max_out,
                          void* stream) {
  if (int rc = check_weights("rnnt_beam_reset", w)) return rc;
  CTCVR_REQUIRE(beam_state && beam > 0 && n_steps > 0 && max_out > 0, "rnnt_beam_reset: bad arguments");
  return rnnt_beam_reset(beam_state, *w, 1, beam, n_steps, max_out, ST(stream));
}

int ctcvr_rnnt_beam_reset_batch(void* beam_states, const ctcvr_decoder_weights* w, int S, int beam, int n_steps,
                                int max_out, void* stream) {
  if (int rc = check_weights("rnnt_beam_reset_batch", w)) return rc;
  CTCVR_REQUIRE(beam_states && S > 0 && beam > 0 && n_steps > 0 && max_out > 0, "rnnt_beam_reset_batch: bad arguments");
  return rnnt_beam_reset(beam_states, *w, S, beam, n_steps, max_out, ST(stream));
}

int ctcvr_rnnt_beam_chunk(const ctcvr_decoder_weights* w, const float* enc_proj, int T, void* beam_state, int beam,
                          int n_steps, int max_out, int blank, int32_t* out_n, int32_t* out_tokens, int32_t* out_lens,
                          double* out_scores, float* out_h, float* out_c, void* stream) {
  if (int rc = check_weights("rnnt_beam_chunk", w)) return rc;
  CTCVR_REQUIRE((enc_proj || T == 0) && beam_state && out_n && out_tokens && out_lens && out_scores, "rnnt_beam_chunk: NULL pointer");
  CTCVR_REQUIRE(T >= 0 && beam > 0 && n_steps > 0 && max_out > 0, "rnnt_beam_chunk: bad dims");
  CTCVR_REQUIRE(blank >= 0 && blank < w->V, "rnnt_beam_chunk: blank out of range");
  return rnnt_beam_chunk(*w, enc_proj, nullptr, 1, T, beam_state, beam, n_steps, max_out, blank, out_n, out_tokens, out_lens,
                         out_scores, out_h, out_c, ST(stream));
}

int ctcvr_rnnt_beam_chunk_batch(const ctcvr_decoder_weights* w, const float* enc_proj, const int32_t* chunk_lens, int S,
                                int T, void* beam_states, int beam, int n_steps, int max_out, int blank, int32_t* out_n,
                                int32_t* out_tokens, int32_t* out_lens, double* out_scores, float* out_h, float* out_c,
                                void* stream) {
  if (int rc = check_weights("rnnt_beam_chunk_batch", w)) return rc;
  CTCVR_REQUIRE((enc_proj || T == 0) && beam_states && out_n && out_tokens && out_lens && out_scores && out_h && out_c,
                "rnnt_beam_chunk_batch: NULL pointer");
  CTCVR_REQUIRE(S > 0 && T >= 0 && beam > 0 && n_steps > 0 && max_out > 0, "rnnt_beam_chunk_batch: bad dims");
  CTCVR_REQUIRE(blank >= 0 && blank < w->V, "rnnt_beam_chunk_batch: blank out of range");
  return rnnt_beam_chunk(*w, enc_proj, chunk_lens, S, T, beam_states, beam, n_steps, max_out, blank, out_n, out_tokens,
                         out_lens, out_scores, out_h, out_c, ST(stream));
}

size_t ctcvr_rnnt_prefix_beam_ws_bytes(const ctcvr_decoder_weights* w, int beam, int T) {
  return w ? rnnt_prefix_beam_ws_bytes(*w, beam, T) : 0;
}

int ctcvr_rnnt_prefix_beam(const ctcvr_decoder_weights* w, const float* enc_proj, const float* ctc_logp, int T,
                           int beam, int blank, float ctc_weight, float transducer_weight, int32_t* out_n,
                           int32_t* out_tokens, int32_t* out_lens, double* out_scores, void* ws, size_t ws_bytes,
                           void* stream) {
  if (int rc = check_weights("rnnt_prefix_beam", w)) return rc;
  CTCVR_REQUIRE(enc_proj && ctc_logp && out_n && out_tokens && out_lens && out_scores && ws, "rnnt_prefix_beam: NULL pointer");
  CTCVR_REQUIRE(T > 0 && beam > 0, "rnnt_prefix_beam: bad dims");
  return rnnt_prefix_beam(*w, enc_proj, ctc_logp, nullptr, 1, T, beam, blank, ctc_weight, transducer_weight, out_n, out_tokens,
                          out_lens, out_scores, ws, ws_bytes, ST(stream));
}

int ctcvr_rnnt_prefix_beam_batch(const ctcvr_decoder_weights* w, const float* enc_proj, const float* ctc_logp,
                                 const int32_t* lens, int S, int T, int beam, int blank, float ctc_weight,
                                 float transducer_weight, int32_t* out_n, int32_t* out_tokens, int32_t* out_lens,
                                 double* out_scores, void* ws, size_t ws_bytes, void* stream) {
  if (int rc = check_weights("rnnt_prefix_beam_batch", w)) return rc;
  CTCVR_REQUIRE(enc_proj && ctc_logp && out_n && out_tokens && out_lens && out_scores && ws, "rnnt_prefix_beam_batch: NULL pointer");
  CTCVR_REQUIRE(S > 0 && T > 0 && beam > 0, "rnnt_prefix_beam_batch: bad dims");
  return rnnt_prefix_beam(*w, enc_proj, ctc_logp, lens, S, T, beam, blank, ctc_weight, transducer_weight, out_n, out_tokens,
                          out_lens, out_scores, ws, ws_bytes, ST(stream));
}

size_t ctcvr_ctc_prefix_beam_ws_bytes(int B, int T, int V, int beam) { return ctc_prefix_beam_ws_bytes(B, T, V, beam); }

int ctcvr_ctc_prefix_beam(const float* ctc_probs, const int32_t* lens, int B, int T, int V, int beam, int blank,
                          int32_t* out_n, int32_t* out_tokens, int32_t* out_lens, double* out_scores,
                          int32_t* out_times, void* ws, size_t ws_bytes, void* stream) {
  CTCVR_REQUIRE(ctc_probs && lens && out_n && out_tokens && out_lens && out_scores && out_times && ws,
                "ctc_prefix_beam: NULL pointer");
  CTCVR_REQUIRE(B > 0 && T > 0 && V > 0 && beam > 0 && beam <= V, "ctc_prefix_beam: bad dims (beam must be <= V)");
  return ctc_prefix_beam(ctc_probs, lens, B, T, V, beam, blank, out_n, out_tokens, out_lens, out_scores, out_times,
                         ws, ws_bytes, ST(stream));
}

}  // extern "C"
