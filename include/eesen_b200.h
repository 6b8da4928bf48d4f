/* include/eesen_b200.h -- C ABI of the B200-native Eesen CTC-training hot path.
 *
 * The drop-in boundary (DESIGN.md section 2).  Plain pointers and sizes only; no C++ or
 * torch types.  Every entry point returns 0 on success or a non-zero code (the CUDA/NCCL
 * error value, or EESEN_B200_E*); eesen_b200_last_error() returns the message.  The C++
 * host mirror (eesen_b200/host, namespace eesen: Net / Layer / BiLstmParallel / Ctc, same
 * method names and argument meaning as the reference) turns a non-zero code into a
 * std::runtime_error, matching the reference convention that any CUDA failure throws
 * (reference src/gpucompute/cuda-common.h:37-44 CU_SAFE_CALL -> KALDI_ERR).
 *
 * There is NO CPU fallback: without a CUDA device eesen_b200_create() fails.
 *
 * Conventions at the seam (reference src/netbin/train-ctc-parallel.cc:186-193):
 *   packed minibatch, time-major interleaved: row r = t*S + s (frame t of utterance s),
 *   zero padded to T frames; fp32 row-major; leading dimensions (ld*) are in floats and
 *   must be multiples of 4 (16-byte rows) -- the reference's cudaMallocPitch strides satisfy
 *   this; blank = class 0, labels are 1-based, padded label cells are ignored.
 *   All device pointers must be 16-byte aligned.  Calls are stream-ordered on the context's
 *   stream and asynchronous unless stated; one context per process/GPU, not thread-safe
 *   (same contract as the reference's singleton CuDevice, src/gpucompute/cuda-device.h:47,128).
 */
#ifndef EESEN_B200_H_
#define EESEN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EESEN_B200_EINVAL 100001   /* bad argument */
#define EESEN_B200_ENOGPU 100002   /* no CUDA device / kernel image unusable on this device */
#define EESEN_B200_ENCCL 100003    /* NCCL unavailable or failed */
#define EESEN_B200_EIO 100004      /* model / archive I/O error */
#define EESEN_B200_ESHAPE 100005   /* shape / capacity not supported (recurrent kernels, decoder token stores) */

/* Arithmetic of the tensor-core contractions (storage is always fp32):
 *   0 = 3xTF32 split (fp32-faithful, default)   1 = TF32   2 = BF16 (dense GEMMs only) */
#define EESEN_B200_PREC_FP32X3 0
#define EESEN_B200_PREC_TF32 1
#define EESEN_B200_PREC_BF16 2

typedef struct eesen_b200_ctx eesen_b200_ctx;
typedef struct eesen_b200_net eesen_b200_net;

/* ---------------------------------------------------------------- context (replaces CuDevice,
 * reference src/gpucompute/cuda-device.{h,cc}: SelectGpuId :64-168, allocator :473-816) */
int eesen_b200_create(eesen_b200_ctx **ctx, int device /* -1: LOCAL_RANK or 0 */);
void eesen_b200_destroy(eesen_b200_ctx *ctx);
const char *eesen_b200_last_error(const eesen_b200_ctx *ctx /* may be NULL: last create() error */);
int eesen_b200_set_precision(eesen_b200_ctx *ctx, int gemm_precision, int recurrent_precision);
int eesen_b200_synchronize(eesen_b200_ctx *ctx);
void *eesen_b200_stream(eesen_b200_ctx *ctx); /* cudaStream_t */
int eesen_b200_sm_count(const eesen_b200_ctx *ctx);
/* number of kernels this library launched on the context so far (bench.py "gpu_launches") */
long eesen_b200_launch_count(const eesen_b200_ctx *ctx);

/* Per-category device timing with CUDA events on the context's stream (for bench.py's roofline).
 * Categories: 0 gemm (main stream), 1 lstm_forward, 2 lstm_backward, 3 softmax/argmax, 4 ctc, 5 sgd, 6 all-reduce, 7 misc,
 * 8 gemm on the side stream (weight gradients, streamed chunks, conversions: they overlap the recurrent kernels).
 * Synchronises, returns the milliseconds / launch counts accumulated since the last reset in
 * ms[9] / counts[9] (either may be NULL); enable = 1/0 switches recording and resets, -1 only reads. */
#define EESEN_B200_NUM_PROFILE_CATEGORIES 9
int eesen_b200_profile(eesen_b200_ctx *ctx, int enable, double *ms, long *counts);

/* Debug builds only (make TIMING=1): clock64 deltas per phase of the recurrent kernels, [2][16]
 * (forward, backward); returns 1 when compiled in, else 0. */
int eesen_b200_debug_lstm_timing(eesen_b200_ctx *ctx, long long *out32, int reset);

/* Which recurrent kernels a layer of `cells` cells per direction, `ndir` directions and `num_utts` parallel
 * utterances runs on (pass 0 = forward, 1 = backward): 1 = tcgen05 kernels (lstm_tc_{fwd,bwd}_kernel),
 * 0 = warp-level kernels (lstm_{fwd,bwd}_kernel), -1 = no plan for this shape.  For bench.py's labels. */
int eesen_b200_lstm_engine(eesen_b200_ctx *ctx, int num_utts, int cells, int ndir, int pass);

/* ---------------------------------------------------------------- level 1: device operators */

/* NaN/Inf scan of a device array: *flags = bit 0 (a NaN) | bit 1 (an Inf).  Replaces the host-side sum test of
 * Net::Check / CheckNanInf (reference src/net/net.cc:461-468, src/net/utils-functions.h:118-122), which copies
 * every parameter to the host.  Synchronises the stream (it returns a host value). */
int eesen_b200_check_finite(eesen_b200_ctx *ctx, const float *d_x, int64_t n, int *flags);

/* C = alpha*op(A)*op(B) + beta*C.  Replaces CuMatrixBase::AddMatMat -> cublasSgemm
 * (reference src/gpucompute/cuda-matrix.cc:603-639).  transA/transB: 0 = as stored, 1 = transposed;
 * (1,1) is not provided (unused by the path). */
int eesen_b200_gemm(eesen_b200_ctx *ctx, int transA, int transB, int M, int N, int K, float alpha,
                    const float *A, int lda, const float *B, int ldb, float beta, float *C, int ldc);

/* Parameters of one BiLSTM layer, both directions ([0] = forward cells, [1] = backward cells), in
 * the reference's shapes (src/net/bilstm-layer.h:187-210): wx[4C x I], wm[4C x C], bias[4C],
 * peepholes pi/pf/po[C]; gate row blocks in the order g, i, f, o.
 * ldwx / ldwm: row strides (in floats) of the wx / wm matrices, 0 = dense (I resp. C).  The reference's
 * CuMatrix weights are cudaMallocPitch'ed (src/gpucompute/cuda-matrix.cc:46-79), so wei_gifo_x_fw_.Data()
 * binds with ldwx = wei_gifo_x_fw_.Stride() without repacking.  Strides that are not a multiple of 4 floats
 * (or bases not 16-byte aligned) cannot be addressed by TMA: such products run on the warp-level GEMM. */
typedef struct {
  const float *wx[2], *wm[2], *bias[2], *pi[2], *pf[2], *po[2];
  int ldwx, ldwm;
} eesen_b200_bilstm_params;
typedef struct {
  float *wx[2], *wm[2], *bias[2], *pi[2], *pf[2], *po[2];
  int ldwx, ldwm;
} eesen_b200_bilstm_grads;

/* BiLstmParallel::PropagateFnc (reference src/net/bilstm-parallel-layer.h:379-420).
 *   x     [T*S x I] (ldx)          in
 *   gates [T*S x 8C] (ld = 8C)     out: post-activation g,i,f,o; forward cells cols [0,4C), backward [4C,8C)
 *   cell  [T*S x 2C] (ld = 2C)     out: cell state c (fw | bw)
 *   out   [T*S x 2C] (ldo)         out: m = o*tanh(c) (fw | bw) -- the layer output
 * gates/cell are what the reference keeps in propagate_buf_{fw,bw}_ (h = tanh(c) is recomputed). */
int eesen_b200_bilstm_forward(eesen_b200_ctx *ctx, int T, int S, int I, int C, const int *d_len,
                              const float *x, int ldx, const eesen_b200_bilstm_params *p, float *gates,
                              float *cell, float *out, int ldo);

/* BiLstmParallel::BackpropagateFnc (reference :881-913, :422-602).  dgates [T*S x 8C] is scratch/out
 * (the DGIFO blocks of backpropagate_buf_); dx may be NULL (first layer).  grads receives the RAW
 * gradient sums over all rows (no momentum: corr = grad + momentum*corr is applied by
 * eesen_b200_sgd_update after the data-parallel all-reduce).
 * Stream order: dgates and dx are complete in the order of eesen_b200_stream when the call returns its work to it; the
 * weight gradients (grads->wx, ->wm) are produced on the library's side stream, overlapped with whatever the caller
 * queues next, and are complete for eesen_b200_sgd_update / eesen_b200_allreduce_sum* / eesen_b200_synchronize (each
 * joins the side stream) -- a caller reading them with its own kernels synchronizes first. */
int eesen_b200_bilstm_backward(eesen_b200_ctx *ctx, int T, int S, int I, int C, const float *x, int ldx,
                               const eesen_b200_bilstm_params *p, const float *gates, const float *cell,
                               const float *out, int ldo, const float *dout, int ldd, float *dgates,
                               float *dx, int lddx, const eesen_b200_bilstm_grads *grads);

/* The dropout variants of BiLstmParallel (reference src/net/bilstm-parallel-layer.h:46-94 masks, :209-377
 * forward, :604-879 backward; options src/net/bilstm-layer.h:62-135).
 *   drop   1 = no-mem-loss dropout (c = r*(g*i) + c_prev*f), 2 = RNNdrop (c = r*(g*i + c_prev*f)); 0 = the plain calls
 *   rmask  scaled recurrent mask (0 | 1/(1-p)), forward cells in cols [0,C), backward cells in [C,2C), ld = ldr;
 *          [T*S x 2C] (row t*S+s) when per_step != 0 (RecurrentTimeStepDropout), else [S x 2C]
 * Forward (non-recurrent) dropout is a product of the layer OUTPUT and of out_diff with a [T*S x 2C] mask
 * (:409-416, :891-895): eesen_b200_mul_elements; the un-masked m must be kept for the Wm gradient (pass it as
 * `out` to the backward call).  eesen_b200_dropout_mask draws a mask on the device (the reference draws on the
 * CPU from a random_device-seeded generator and uploads it; parity is per given mask): one draw per element, or
 * per column repeated in every row when per_col != 0 (the reference's "sequence" masks, SetRandUniformCol
 * src/cpucompute/matrix.cc:952-965); deterministic in (seed, stream). */
int eesen_b200_bilstm_forward_dropout(eesen_b200_ctx *ctx, int T, int S, int I, int C, const int *d_len,
                                      const float *x, int ldx, const eesen_b200_bilstm_params *p, float *gates,
                                      float *cell, float *out, int ldo, int drop, const float *rmask, int ldr,
                                      int per_step);
int eesen_b200_bilstm_backward_dropout(eesen_b200_ctx *ctx, int T, int S, int I, int C, const float *x, int ldx,
                                       const eesen_b200_bilstm_params *p, const float *gates, const float *cell,
                                       const float *out, int ldo, const float *dout, int ldd, float *dgates,
                                       float *dx, int lddx, const eesen_b200_bilstm_grads *grads, int drop,
                                       const float *rmask, int ldr, int per_step);
int eesen_b200_mul_elements(eesen_b200_ctx *ctx, int N, int cols, const float *a, int lda, const float *b, int ldb,
                            float *out, int ldo);
int eesen_b200_dropout_mask(eesen_b200_ctx *ctx, int rows, int cols, float *d_mask, int ld, float p, int per_col,
                            unsigned long long seed, unsigned long long stream);

/* LstmParallel::PropagateFnc / BackpropagateFnc (reference src/net/lstm-parallel-layer.h:47-113,
 * :115-213): the uni-directional layer = the forward cells of the layer above, nothing masked (the
 * length check is commented out in the reference, :107-110).  Same structs, index [0] only:
 *   gates [T*S x 4C] (ld 4C), cell [T*S x C] (ld C), out/dout [T*S x C], dgates [T*S x 4C]. */
int eesen_b200_lstm_forward(eesen_b200_ctx *ctx, int T, int S, int I, int C, const float *x, int ldx,
                            const eesen_b200_bilstm_params *p, float *gates, float *cell, float *out, int ldo);
int eesen_b200_lstm_backward(eesen_b200_ctx *ctx, int T, int S, int I, int C, const float *x, int ldx,
                             const eesen_b200_bilstm_params *p, const float *gates, const float *cell,
                             const float *out, int ldo, const float *dout, int ldd, float *dgates,
                             float *dx, int lddx, const eesen_b200_bilstm_grads *grads);

/* AffineTransform::PropagateFnc / BackpropagateFnc / gradient part of Update
 * (reference src/net/affine-trans-layer.h:161-166, 168-172, 182-183).  W[K x D], b[K]. */
int eesen_b200_affine_forward(eesen_b200_ctx *ctx, int N, int D, int K, const float *x, int ldx,
                              const float *W, const float *b, float *y, int ldy);
int eesen_b200_affine_backward(eesen_b200_ctx *ctx, int N, int D, int K, const float *x, int ldx,
                               const float *diff, int lddiff, const float *W, float *dx, int lddx,
                               float *dW, float *db);

/* Softmax::PropagateFnc (reference src/net/softmax-layer.h:44-47); argmax may be NULL, else
 * receives FindRowMaxId (src/gpucompute/cuda-matrix.cc:1038-1095) of each row.  Columns
 * [K, ldp) of probs are zeroed. */
int eesen_b200_softmax(eesen_b200_ctx *ctx, int N, int K, const float *logits, int ld, float *probs,
                       int ldp, int *d_argmax);
int eesen_b200_row_argmax(eesen_b200_ctx *ctx, int N, int K, const float *x, int ld, int *d_argmax);
/* Output side of the forward-only path (reference src/netbin/net-output-extract.cc:100-110), in
 * place on y [N x K] (ld): CuMatrixBase::ApplyLog (src/gpucompute/cuda-matrix.cc ApplyLog ->
 * cuda-kernels.cu:221-227) if apply_log != 0, then ClassPrior::SubtractOnLogpost
 * (src/net/class-prior.cc:78-90: y -= prior_scale * log_prior[col]) if d_log_prior != NULL. */
int eesen_b200_loglik(eesen_b200_ctx *ctx, int N, int K, float *y, int ld, int apply_log,
                      const float *d_log_prior, float prior_scale);

/* Ctc::EvalParallel compute (reference src/net/ctc-loss.cc:101-168).
 *   probs    [T*S x K] (ldp) softmax outputs           d_len[S] valid frames
 *   d_labels [S x max_lab] int32, row s holds d_lab_len[s] labels (1-based), rest ignored
 *   pzx[S]   out: log p(z|x) per utterance             diff [T*S x K] (ldd) out: d(-log p)/d(logits) */
int eesen_b200_ctc_eval(eesen_b200_ctx *ctx, int T, int S, int K, int max_lab, const int *d_len,
                        const int *d_labels, const int *d_lab_len, const float *probs, int ldp,
                        float *pzx, float *diff, int ldd);

/* CE::EvalParallel compute (reference src/net/ce-loss.cc:94-169), frame-level cross-entropy.
 *   probs     [T*S x K] (ldp) softmax outputs           d_len[S] valid frames: row t*S+s is valid iff t < d_len[s]
 *   ldp, ldd must be multiples of 4 and probs, diff 16-byte aligned (rows are moved as float4): EESEN_B200_EINVAL
 *   otherwise
 *   d_targets [T*S] int32, packed like the rows; the class of each valid row, in [0, K) (padded rows ignored)
 *   diff      [T*S x K] (ldd) out: y - onehot(target) on valid rows (d(CE)/d(logits)), exactly 0 on padded rows;
 *             columns [K, ldd) untouched
 *   d_stats   double[3] (device), overwritten: [0] sum over valid rows of -log y[target] (the target column only,
 *             so a posterior of 0 elsewhere leaves it finite), [1] valid rows whose first row maximum is the
 *             target (FindRowMaxId tie rule), [2] valid rows.  A valid row with a target outside [0, K) makes [0]
 *             NaN; nothing outside the row is read.  The statistics are the same bits on every run. */
int eesen_b200_ce_eval(eesen_b200_ctx *ctx, int T, int S, int K, const int *d_len, const float *probs, int ldp,
                       const int *d_targets, float *diff, int ldd, double *d_stats);

/* Momentum + clip + SGD over a contiguous arena (reference src/net/bilstm-layer.h:846-883,
 * affine-trans-layer.h:182-195):  corr = grad + momentum*corr; clamp(corr, +-max_grad); w -= lr*corr.
 * segments (host memory) partition [0, n): lr = learn_rate*learn_rate_coef, max_grad <= 0 disables clipping. */
typedef struct {
  int64_t offset, count;
  float lr, max_grad;
} eesen_b200_sgd_segment;
int eesen_b200_sgd_update(eesen_b200_ctx *ctx, float *w, float *corr, const float *grad, int64_t n,
                          float momentum, const eesen_b200_sgd_segment *segments, int nseg);

/* ---------------------------------------------------------------- data parallelism (new; replaces the
 * file-system model averaging of reference src/net/communicator.h:39-119 with one gradient all-reduce) */
int eesen_b200_nccl_unique_id(char id[128]);
int eesen_b200_nccl_init(eesen_b200_ctx *ctx, int rank, int nranks, const char id[128]);
int eesen_b200_allreduce_sum(eesen_b200_ctx *ctx, float *buf, int64_t n);
/* Same reduction, issued on the library's low-priority side stream behind everything queued so far, so that it
 * overlaps with the back-propagation of the layers below (per-layer gradient buckets; reference update order
 * src/net/net.cc:98-105).  Consumers of the buffer (eesen_b200_sgd_update, eesen_b200_synchronize, ...) join the
 * side stream themselves. */
int eesen_b200_allreduce_sum_overlapped(eesen_b200_ctx *ctx, float *d_buf, int64_t n);
int eesen_b200_world(const eesen_b200_ctx *ctx, int *rank, int *nranks);

/* ---------------------------------------------------------------- level 2: the Net/Ctc host mirror
 * (what src/netbin/train-ctc-parallel.cc:112-119,195-207,244 calls) */
int eesen_b200_net_read(eesen_b200_ctx *ctx, const char *model_path, eesen_b200_net **net); /* Net::Read */
int eesen_b200_net_write(eesen_b200_net *net, const char *path, int binary);               /* Net::Write */
void eesen_b200_net_free(eesen_b200_net *net);
int eesen_b200_net_set_train_options(eesen_b200_net *net, float learn_rate, float momentum); /* SetTrainOptions */
/* Net::SetUpdateAlgorithm (reference src/net/net.cc:481-496; driver option --opt-algorithm,
 * src/netbin/train-ctc-parallel.cc:77-78,114) plus the two adaptive options of NetTrainOptions
 * (src/net/train-opts.h:33-50).  algorithm: "SGD" | "Adagrad" | "RMSProp".  The update rules are
 * trainable-layer.h:65-114 applied by bilstm-layer.h:885-955 / affine-trans-layer.h:196-219.
 * NOTE the reference fixes rmsprop_one_minus_rho at 0.1 whatever --rms-prop-rho says (it is computed
 * inside Register(), before the command line is parsed: train-opts.h:50); pass one_minus_rho < 0 to get
 * that behaviour, or the value you want. */
int eesen_b200_net_set_optimizer(eesen_b200_net *net, const char *algorithm, float adagrad_epsilon,
                                 float rmsprop_rho, float rmsprop_one_minus_rho);
/* Dropout of the BiLstmParallel layers.  Net::ChangeDropoutParameters (reference src/net/net.cc:414-434, tool
 * src/netbin/net-change-model.cc) with the reference's consistency checks (src/net/bilstm-layer.h:74-112); the
 * options are stored in the model file.  Masks are drawn on the device; eesen_b200_net_set_dropout_seed fixes the
 * generator (default: a fresh random seed per Net, like the reference's random_device-seeded generator).
 * eesen_b200_net_set_dropout_masks injects explicit scaled masks (0 | 1/(1-p), HOST pointers) for layer `layer`
 * (0-based): fmask [T*S x 2C] or NULL, rmask [rmask_rows x 2C] or NULL with rmask_rows = T*S (step) or S
 * (sequence); they stay in force until called again with NULLs.  This is how the parity tests replay the masks the
 * reference drew.  Steps run with train == 0 are in test mode: no dropout (reference driver: SetTestMode). */
int eesen_b200_net_change_dropout(eesen_b200_net *net, float forward_dropout, int fw_step, int fw_sequence, int rnndrop,
                                  int no_mem_loss, float recurrent_dropout, int rec_step, int rec_sequence,
                                  int twiddle_forward);
int eesen_b200_net_set_dropout_seed(eesen_b200_net *net, unsigned long long seed);
int eesen_b200_net_set_dropout_masks(eesen_b200_net *net, int layer, const float *fmask, int fmask_rows,
                                     const float *rmask, int rmask_rows);
int eesen_b200_net_dims(const eesen_b200_net *net, int *in_dim, int *out_dim, int *num_layers, int64_t *num_params);

/* One minibatch exactly as the reference driver does it (train-ctc-parallel.cc:195-207):
 * SetSeqLengths, Propagate (H2D copy of the packed features included), Ctc::EvalParallel,
 * Ctc::ErrorRateMSeq, and -- if train != 0 -- Backpropagate with the gradient all-reduce (when NCCL
 * is initialised) and the parameter update.  HOST inputs; blocks until the statistics are back.
 *   feats [T*S x I] packed, frames[S], labels: concatenated, lab_len[S]
 *   stats out: [0] sum_s log p(z|x)  [1] token errors  [2] reference tokens  [3] valid frames */
int eesen_b200_net_train_step(eesen_b200_net *net, const float *feats, int T, int S, const int *frames,
                              const int *labels, const int *lab_len, int train, double stats[4]);
/* Same step with inputs ALREADY RESIDENT on the device (d_feats [T*S x I], ld = I); asynchronous:
 * statistics stay on the device until eesen_b200_net_read_stats. */
int eesen_b200_net_train_step_device(eesen_b200_net *net, const float *d_feats, int T, int S,
                                     const int *frames, const int *labels, const int *lab_len, int train);
/* The same step with frame-level cross-entropy instead of CTC (reference src/netbin/train-ce-parallel.cc:167-177):
 * SetSeqLengths, Propagate, CE::EvalParallel and -- if train != 0 -- Backpropagate with the all-reduce and the
 * update.  HOST inputs; blocks until the statistics are back.
 *   feats [T*S x I] packed, frames[S], targets: concatenated per utterance, frames[s] class ids each, in [0, K)
 *   stats out: [0] sum of -log y[target] over valid frames  [1] correctly classified frames  [2] valid frames
 *              [3] padded rows (T*S, the reference's frame count) */
int eesen_b200_net_train_step_ce(eesen_b200_net *net, const float *feats, int T, int S, const int *frames,
                                 const int *targets, int train, double stats[4]);
/* Same step with inputs ALREADY RESIDENT on the device: d_feats [T*S x I] (ld = I), d_targets [T*S] packed like the
 * rows (padded rows ignored, the caller guarantees [0, K)); frames[S] on the host.  Asynchronous: statistics stay on
 * the device until eesen_b200_net_read_stats.  Targets are NOT checked here: a valid row with a target outside [0, K)
 * gets no -1 in its gradient and makes stats[0] NaN, so a caller that has not validated its targets checks that. */
int eesen_b200_net_train_step_ce_device(eesen_b200_net *net, const float *d_feats, int T, int S, const int *frames,
                                        const int *d_targets, int train);
/* Statistics of the last step, whichever loss it used (layouts above). */
int eesen_b200_net_read_stats(eesen_b200_net *net, double stats[4]);
/* The loss of the last step: 0 = CTC (or no step yet), 1 = frame-level cross-entropy. */
int eesen_b200_net_last_loss(const eesen_b200_net *net);

/* ---------------------------------------------------------------- forward-only path (SURVEY.md 8f N2)
 * One packed batch through what reference src/netbin/net-output-extract.cc:83-118 does per
 * utterance: Net::Feedforward (src/net/net.cc:110-137), CuMatrixBase::ApplyLog if apply_log != 0,
 * ClassPrior::SubtractOnLogpost (src/net/class-prior.cc:78-90) if log_priors != NULL.
 *   feats [T*S x I] packed time-major (row t*S+s), frames[S]; HOST buffers.  frames == NULL (S must
 *   be 1): no SetSeqLengths call at all, the reference tool's own call pattern -- accepted by <BiLstm>
 *   layers (one sequence of T rows, src/net/bilstm-layer.h:548), an error for <BiLstmParallel>
 *   log_priors [K] host (from eesen_b200_class_log_priors) or NULL, prior_scale = --prior-scale
 *   out [T*S x K] host, same packing; rows of padding frames hold no meaning
 * Works for <BiLstmParallel> and <BiLstm> models alike (the reference converts on the fly,
 * src/net/layer.cc:164-170). */
int eesen_b200_net_feedforward(eesen_b200_net *net, const float *feats, int T, int S, const int *frames,
                               int apply_log, const float *log_priors, float prior_scale, float *out);
/* Host arithmetic of ClassPrior::ClassPrior (src/net/class-prior.cc:28-76): frame counts -> log priors
 * (classes with count < prior_cutoff get +FLT_MAX/2 so that their likelihood vanishes; class 0 is
 * scaled by blank_scale before normalisation).  No device work. */
int eesen_b200_class_log_priors(const double *counts, int K, float prior_cutoff, float blank_scale, float *log_priors);
/* Net::WriteNonParal (src/net/net.cc:337-353; tool src/netbin/format-to-nonparallel.cc) */
int eesen_b200_net_write_nonparallel(eesen_b200_net *net, const char *path, int binary);

/* Introspection for the parity tests (host copies, synchronous).  which:
 *   0..L    Net::propagate_buf_[which]     (layer inputs/outputs, L = num_layers)
 *   100     obj_diff (CTC or CE gradient wrt logits, from the last step)      101  per-utterance pzx [S]
 *   102     in_diff  (gradient wrt the network input)
 *   200     parameters   201 momentum buffers (corr)   202 raw gradients of the last step (after all-reduce)
 *   203     Adagrad/RMSProp accumulators (zeros while none exist)
 *   300+l   forward dropout mask used by layer l in the last step   400+l  its recurrent dropout mask
 * rows/cols describe the logical matrix; data may be NULL to query the shape only. */
int eesen_b200_net_get(eesen_b200_net *net, int which, float *data, int64_t capacity, int *rows, int *cols);
int eesen_b200_net_set_params(eesen_b200_net *net, const float *flat, int64_t n);

/* ---------------------------------------------------------------- decoding (SURVEY.md 8f row N3, first slice)
 * One-best WFST token passing for a batch of utterances: the search core of `latgen-faster`
 * (reference src/decoderbin/latgen-faster.cc:96-126 -> LatticeFasterDecoder::Decode
 * src/decoder/lattice-faster-decoder.cc:77-97, ProcessEmitting :660-752, ProcessNonemitting :756-816, GetCutoff :594-658,
 * ComputeFinalCosts :531-577; acoustic scores as DecodableMatrixScaled src/decoder/decodable-matrix.h:54-56).
 * Output: the words (non-zero output labels) of the best path and its cost; lattices are not produced.
 * The graph is handed over WITHOUT OpenFst: CSR over states, the arcs of a state stored emitting arcs first
 * (ilabel = 1-based CTC token id), then epsilon-input arcs; all arrays on the HOST, copied once. */
typedef struct eesen_b200_graph eesen_b200_graph;
int eesen_b200_graph_create(eesen_b200_ctx *ctx, int num_states, int num_arcs, int start, const int *row /*[ns+1]*/,
                            const int *eps /*[ns]*/, const int *ilabel, const int *olabel, const float *weight,
                            const int *nextstate, const float *final_cost /*[ns], +inf = not final*/,
                            eesen_b200_graph **out);
void eesen_b200_graph_free(eesen_b200_graph *g);
/* d_loglikes: device, packed time-major [T*S x K] (row t*S + s, ld floats per row) -- what eesen_b200_net_feedforward
 * produces with apply_log; frames[S] (host): frames per utterance.  beam, max_active, min_active as the options of
 * latgen-faster (GetCutoff, lattice-faster-decoder.cc:594-658: the k-th best cost is selected exactly, as nth_element
 * does); 2147483647 / 0 = beam pruning only.
 * frame_cap: most tokens one frame of one utterance may hold; tok_cap: most tokens one utterance may hold in total.
 * out_labels [S x max_out], out_len [S] (-1: no surviving token), out_cost [S]: host arrays.
 * stats (may be NULL): [0] closure rounds, [1] device milliseconds. */
int eesen_b200_decode_best_path(eesen_b200_ctx *ctx, const eesen_b200_graph *g, int S, int T, const int *frames,
                                const float *d_loglikes, int ld, int K, float acoustic_scale, float beam,
                                int max_active, int min_active, int frame_cap, int tok_cap, int *out_labels,
                                int max_out, int *out_len, float *out_cost, double *stats);

#ifdef __cplusplus
}
#endif
#endif /* EESEN_B200_H_ */
