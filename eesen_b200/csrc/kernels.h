// eesen_b200/csrc/kernels.h -- internal (C++) launch interface of the sm_100a kernels.
// The public boundary is the C ABI in include/eesen_b200.h; these are what it dispatches to.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace eb {

// gemm.cu
cudaError_t gemm(cudaStream_t st, int num_sms, int transA, int transB, int M, int N, int K, float alpha,
                 const float *A, int lda, long strideA, const float *B, int ldb, long strideB, float beta,
                 float *C, int ldc, long strideC, const float *bias, long strideBias, int batch,
                 int precision, float *ws, size_t ws_bytes);
size_t gemm_workspace_bytes(int M, int N, int K, int batch, int num_sms);

// gemm_tc.cu -- tcgen05 / TMEM / TMA path (fp32x3 and tf32 arithmetic); one matrix per call
bool gemm_tc_supported(int transA, int transB, int M, int N, int K, const float *A, int lda, const float *B, int ldb,
                       int precision);
size_t gemm_tc_workspace_bytes(int M, int N, int K, int num_sms);
cudaError_t gemm_tc(cudaStream_t st, int num_sms, int transA, int transB, int M, int N, int K, float alpha,
                    const float *A, int lda, const float *B, int ldb, float beta, float *C, int ldc,
                    const float *bias, int precision, float *ws, size_t ws_bytes);

// bf16 arithmetic (precision 2, BASELINE config 4): tcgen05 kind::f16 on bf16 copies of the operands
size_t gemm_tc16_operand_bytes(long rows, int cols);
cudaError_t convert_bf16(cudaStream_t st, int num_sms, const float *src, long rows, int cols, long lds, void *dst);
cudaError_t gemm_tc16(cudaStream_t st, int num_sms, int transA, int transB, int M, int N, int K, float alpha,
                      const void *A16, const void *B16, float beta, float *C, int ldc, const float *bias, float *ws,
                      size_t ws_bytes);

// fp32-faithful arithmetic on the 16-bit tensor pipe ("fp16x3"): operands as two fp16 planes of the power-of-two
// scaled matrix (22 mantissa bits), three kind::f16 MMAs per k-slice
struct F16View {
  const void *hi, *lo;   // planes of the matrix as stored (row-major), both with leading dimension ld (halfs)
  int ld;
  const int *kexp;       // device: the scale exponent the conversion chose
};
size_t f16x2_plane_bytes(long rows, int cols);
// known_max != NULL: the bits of max |src| are already there (device) -- no scan of the matrix
cudaError_t convert_f16x2(cudaStream_t st, int num_sms, const float *src, long rows, int cols, long lds, void *hi, void *lo,
                          unsigned *scratch_max, int *kexp, const unsigned *known_max = nullptr);
cudaError_t gemm_tc16x3(cudaStream_t st, int num_sms, int transA, int transB, int M, int N, int K, float alpha,
                        const F16View &A, const F16View &B, float beta, float *C, int ldc, const float *bias, float *ws,
                        size_t ws_bytes);

// lstm.cu -- persistent recurrent kernels (both directions in one cooperative launch)
struct LstmDirParams {
  const float *wm;  // [4C x C] recurrent weights, row blocks g,i,f,o
  int ldwm;         // row stride of wm in floats (>= C)
  const float *pi, *pf, *po;  // [C] peepholes
};
struct LstmFwdArgs {
  int T, S, C;
  int s_begin, s_count;  // utterances [s_begin, s_begin+s_count) are processed by this launch
  const int *len;        // [S] valid frames per utterance (device)
  float *G; int ldg;     // [T*S x 8C]: in = x*Wx^T + b (dir block d at col d*4C), out = post-activation g,i,f,o
  float *cell; int ldc;  // [T*S x 2C] cell state c (dir d at col d*C)
  float *out; int ldo;   // [T*S x 2C] m = o*tanh(c): the layer output (dir d at col d*C)
  LstmDirParams p[2];
  void *xbuf;            // [2 parity][2 dir][groups][8*NUT][C] tagged 8-byte exchange words (zeroed per launch)
  int precision;         // 0 = 3xTF32, 1 = TF32
  // recurrent dropout (bilstm-parallel-layer.h:209-377): 0 none, 1 no-mem-loss (mask on g*i), 2 RNNdrop (mask on c)
  int drop = 0;
  const float *rmask = nullptr;  // scaled mask (0 | 1/(1-p)); dir d at col d*C; row t*S+s if per_step else s
  int ldr = 0, rmask_per_step = 0;
  // Streamed input product (tcgen05 engine): G arrives in chunks of `gchunk` positions of each direction's OWN time
  // order (chunk ci = rows t in [ci*gchunk, ..) for dir 0, mirrored from the end for dir 1); chunk ci may be read once
  // gflag[ci] == gepoch, chunks < gready were complete before the launch.  gflag == nullptr: everything is there.
  const unsigned *gflag = nullptr;
  unsigned gepoch = 0;
  int gchunk = 0, gready = 0;
  // (tcgen05 engine) fp16 planes of the layer output for the dense products that read it next (the input product of the
  // layer above, the weight gradients): hi = fp16(2^13 * m), lo = fp16(2^13 * m - hi) -- |m| < 1, so the scale is fixed
  // and the kernel can write them next to m itself; [T*S x ldh] halfs each, dir d at col d*C.  NULL: not wanted.
  void *out_hi = nullptr, *out_lo = nullptr;
  int ldh = 0;
};
struct LstmBwdArgs {
  int T, S, C;
  int s_begin, s_count;
  const float *G; int ldg;      // saved post-activation gates
  const float *cell; int ldc;   // saved cell states
  const float *dout; int ldd;   // [T*S x 2C] gradient wrt the layer output
  float *DG; int lddg;          // [T*S x 8C] out: d(pre-activations) g,i,f,o per direction
  LstmDirParams p[2];
  float *pbuf;                  // [2 parity][2 dir][groups][slices][8*NUT][C] tagged partial d_m words
  float *gsum;                  // [2 dir][groups][7][C] per-group sums: db_g,db_i,db_f,db_o,dpi,dpf,dpo
  int precision;
  int drop = 0;                 // as LstmFwdArgs (:604-879)
  const float *rmask = nullptr;
  int ldr = 0, rmask_per_step = 0;
  unsigned *dgmax = nullptr;    // (tcgen05 engine) atomicMax of the bits of max |DG| over the launch, or NULL
};
struct LstmPlan {
  int engine;            // 0: warp-level mma.sync kernels (lstm.cu), 1: tcgen05 kernels (lstm_tc.cu)
  int nut, nct, ksplit;  // utterance tiles / cell tiles per CTA, K-split warps (fwd)
  int groups, slices;    // grid = (slices, groups, ndir)
  int ndir;              // 2: BiLstmParallel (fw + bw cells), 1: LstmParallel (fw cells only)
  int threads;
  size_t smem_fwd, smem_bwd;
  size_t pbuf_floats, gsum_floats, xbuf_bytes;
  int cluster;           // (engine 1) 1: the CTAs of a (dir, group) form a thread-block cluster and exchange through DSMEM
  int valid;
};
// pass: 0 = forward, 1 = backward (the engines are chosen per pass, lstm.cu:engine_for_pass)
LstmPlan lstm_plan(int S, int C, int num_sms, size_t max_smem, int ndir = 2, int pass = 0);
cudaError_t lstm_forward(cudaStream_t st, const LstmPlan &plan, const LstmFwdArgs &a);
cudaError_t lstm_backward(cudaStream_t st, const LstmPlan &plan, const LstmBwdArgs &a);
// bias/peephole gradient from the per-group sums: dst[7 blocks] = sum_groups gsum
cudaError_t lstm_reduce_gsum(cudaStream_t st, const LstmPlan &plan, int C, const float *gsum, int nchunks,
                             float *db /*[4C]*/, float *dpi, float *dpf, float *dpo, int dir);

int lstm_debug_timing(long long *out32, int reset);  // 1 if built with -DEB_LSTM_TIMING

// lstm_tc.cu -- the same recurrences with the per-step product on tcgen05 (fp16 hi/lo' split, TMEM accumulator);
// lstm_plan() returns such a plan (engine = 1) when the shape allows, EESEN_B200_LSTM_ENGINE=legacy forces lstm.cu
LstmPlan lstm_tc_plan(int S, int C, int num_sms, size_t max_smem, int ndir);
cudaError_t lstm_tc_forward(cudaStream_t st, const LstmPlan &plan, const LstmFwdArgs &a);
cudaError_t lstm_tc_backward(cudaStream_t st, const LstmPlan &plan, const LstmBwdArgs &a);
cudaError_t lstm_set_flag(cudaStream_t st, unsigned *flag, unsigned value);   // stream-ordered 4-byte store
int lstm_tc_debug_timing(long long *out32, int reset);

// ctc.cu
cudaError_t softmax_rows(cudaStream_t st, int N, int K, const float *logits, int ld, float *probs, int ldp,
                         int *argmax);
cudaError_t row_argmax(cudaStream_t st, int N, int K, const float *x, int ld, int *argmax);
// in place: y = log(y) (if apply_log) - prior_scale * log_prior[col] (if log_prior)
cudaError_t loglik_rows(cudaStream_t st, int num_sms, int N, int K, float *y, int ld, int apply_log,
                        const float *log_prior, float prior_scale);
size_t ctc_workspace_floats(int T, int S, int max_lab);
cudaError_t ctc_eval(cudaStream_t st, int T, int S, int K, int max_lab, const int *len, const int *labels,
                     const int *lab_len, const float *probs, int ldp, float *pzx, float *diff, int ldd,
                     float *ws);

// ce.cu -- frame-level cross-entropy: diff = (y - onehot(target)) on rows t < len[s], 0 on the others;
// stats[3] (device, overwritten) = sum of -log y[target], correct argmax count, valid rows
size_t ce_workspace_bytes(int T, int S, int num_sms);
cudaError_t ce_eval(cudaStream_t st, int num_sms, int T, int S, int K, const int *len, const float *probs, int ldp,
                    const int *targets, float *diff, int ldd, double *stats, void *ws);

// decode.cu -- one-best WFST token passing for a batch of utterances (reference src/decoder/lattice-faster-decoder.cc)
struct DecodeGraph {      // device pointers; CSR over states, emitting arcs of a state first, then its epsilon arcs
  int num_states, num_arcs, start;
  const int *row;         // [num_states + 1]
  const int *eps;         // [num_states]     first epsilon-input arc of the state
  const int *ilabel, *olabel, *nextstate, *arc_from;   // [num_arcs]
  const float *weight;    // [num_arcs] graph cost
  const float *final_cost;   // [num_states], +inf = not final
};
size_t decode_workspace_bytes(int S, int num_states, int frame_cap, int wl_cap, int tok_cap);
cudaError_t decode_best_path(cudaStream_t st, int num_sms, const DecodeGraph &g, int S, int T, const int *h_frames,
                             const float *d_loglikes, int ld, float scale, float beam, int max_active, int min_active,
                             void *ws, int frame_cap, int wl_cap, int tok_cap, int *d_out_labels, int max_out,
                             int *d_out_len, float *d_out_cost, int *err_bits, long *closure_rounds);

// optim.cu
struct SgdSegment {
  long offset, count;
  float lr;        // learn_rate * learn_rate_coef
  float max_grad;  // <= 0: no clipping
};
cudaError_t sgd_momentum_clip(cudaStream_t st, int num_sms, float *w, float *corr, const float *grad,
                              float momentum, const SgdSegment *d_segs, int nseg, long total);
// mode 0 SGD, 1 Adagrad, 2 RMSProp (accu: the adaptive accumulator arena, same layout as w)
cudaError_t optimizer_update(cudaStream_t st, int num_sms, int mode, float *w, float *corr, float *accu,
                             const float *grad, float momentum, float eps, float rho, float one_minus_rho,
                             const SgdSegment *d_segs, int nseg, long total);
// *d_flags = bit 0 (NaN present) | bit 1 (Inf present) over x[0, n)
cudaError_t check_finite(cudaStream_t st, int num_sms, const float *x, long n, int *d_flags);
cudaError_t mul_elements(cudaStream_t st, int num_sms, int N, int cols, const float *a, int lda, const float *b, int ldb,
                         float *out, int ldo);
// scaled Bernoulli mask 0 | 1/(1-p) from a counter-based generator (per_col: one draw per column for all rows)
cudaError_t dropout_mask(cudaStream_t st, int num_sms, int rows, int cols, float *mask, int ld, float p, int per_col,
                         unsigned long long seed, unsigned long long stream);
cudaError_t col_sum(cudaStream_t st, int num_sms, int N, int K, const float *x, int ld, float *out, float *ws);
size_t col_sum_ws_floats(int K, int num_sms);

}  // namespace eb
