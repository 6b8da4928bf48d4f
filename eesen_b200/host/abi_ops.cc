// eesen_b200/host/abi_ops.cc -- level-1 C ABI: context + device operators (include/eesen_b200.h).
#include <dlfcn.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/eesen_b200.h"
#include "context.h"

static std::string g_create_error;

#define CTX_CHECK(call, what)                 \
  do {                                        \
    int rc__ = ctx->check((call), what);      \
    if (rc__) return rc__;                    \
  } while (0)

// n kernels launched by f() on the stream of on_side, timed under profile category cat (kUntimed: not timed)
enum { kUntimed = -1 };
template <class F>
static int launch(eesen_b200_ctx *ctx, int cat, int n, const char *what, F &&f, bool on_side = false) {
  ctx->launches += n;
  const int pe = cat == kUntimed ? -1 : ctx->prof_begin(cat, on_side);
  const cudaError_t e = f();
  ctx->prof_end(pe);
  return ctx->check(e, what);
}

extern "C" {

int eesen_b200_create(eesen_b200_ctx **out, int device) {
  if (!out) return EESEN_B200_EINVAL;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    g_create_error = std::string("no CUDA device available (") + cudaGetErrorString(e) +
                     "); eesen_b200 has no CPU fallback";
    return EESEN_B200_ENOGPU;
  }
  if (device < 0) {
    const char *lr = getenv("LOCAL_RANK");
    device = lr ? atoi(lr) % ndev : 0;
  }
  if (device >= ndev) {
    g_create_error = "device index out of range";
    return EESEN_B200_EINVAL;
  }
  e = cudaSetDevice(device);
  if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); return (int)e; }
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); return (int)e; }
  if (prop.major != 10) {
    g_create_error = "eesen_b200 kernels are built for sm_100a only; found sm_" + std::to_string(prop.major) +
                     std::to_string(prop.minor);
    return EESEN_B200_ENOGPU;
  }
  eesen_b200_ctx *ctx = new eesen_b200_ctx();
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  ctx->max_smem = prop.sharedMemPerBlockOptin;
  {
    const char *eng = getenv("EESEN_B200_GEMM_ENGINE");
    ctx->gemm_engine = (eng && std::string(eng) == "legacy") ? 1 : 0;
  }
  {
    const char *ov = getenv("EESEN_B200_OVERLAP");
    ctx->overlap = (ov && ov[0] == '0') ? 0 : 1;
    const char *fx = getenv("EESEN_B200_GEMM_FP32X3");
    ctx->f16x3 = (fx && std::string(fx) == "tf32") ? 0 : 1;
  }
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);   // lo = numerically greatest = lowest priority
  e = cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi);
  if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); delete ctx; return (int)e; }
  e = cudaStreamCreateWithPriority(&ctx->side, cudaStreamNonBlocking, prio_lo);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming);
  if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); delete ctx; return (int)e; }
  *out = ctx;
  return 0;
}

void eesen_b200_destroy(eesen_b200_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  ctx->join_side();
  cudaStreamSynchronize(ctx->stream);
  for (const auto &e : ctx->f16_slots)
    if (e.planes.p) cudaFree(e.planes.p);
  for (const auto &e : ctx->act)
    if (e.planes.p) cudaFree(e.planes.p);
  eesen_b200_ctx::Buf *bufs[] = {&ctx->f16_meta, &ctx->f16_tmp[0], &ctx->f16_tmp[1], &ctx->f16_tmp[2], &ctx->f16_tmp[3], &ctx->decode_ws, &ctx->gemm_ws_side, &ctx->bf16_a_side, &ctx->bf16_b_side,&ctx->gemm_ws, &ctx->lstm_pbuf, &ctx->lstm_gsum, &ctx->lstm_flags,
                                 &ctx->ctc_ws, &ctx->ce_ws, &ctx->colsum_ws, &ctx->seg_buf, &ctx->flag_buf, &ctx->bf16_a, &ctx->bf16_b, &ctx->lstm_gflags};
  for (auto *b : bufs)
    if (b->p) cudaFree(b->p);
  if (ctx->nccl_comm && ctx->nccl_lib) {
    typedef int (*destroy_t)(void *);
    destroy_t f = (destroy_t)dlsym(ctx->nccl_lib, "ncclCommDestroy");
    if (f) f(ctx->nccl_comm);
  }
  cudaStreamDestroy(ctx->stream);
  if (ctx->side) cudaStreamDestroy(ctx->side);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
  if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  delete ctx;
}

const char *eesen_b200_last_error(const eesen_b200_ctx *ctx) {
  return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

int eesen_b200_set_precision(eesen_b200_ctx *ctx, int gemm_precision, int recurrent_precision) {
  if (!ctx || gemm_precision < 0 || gemm_precision > 2 || recurrent_precision < 0 || recurrent_precision > 1)
    return EESEN_B200_EINVAL;
  ctx->gemm_prec = gemm_precision;
  ctx->rec_prec = recurrent_precision;
  return 0;
}

int eesen_b200_synchronize(eesen_b200_ctx *ctx) {
  ctx->join_side();
  CTX_CHECK(cudaStreamSynchronize(ctx->stream), "cudaStreamSynchronize");
  return 0;
}
void *eesen_b200_stream(eesen_b200_ctx *ctx) { return (void *)ctx->stream; }
int eesen_b200_sm_count(const eesen_b200_ctx *ctx) { return ctx->num_sms; }
long eesen_b200_launch_count(const eesen_b200_ctx *ctx) { return ctx->launches; }

// ---- fp16x3 operand planes --------------------------------------------------------------------------------------
// record idx of f16_meta (eesen_b200_ctx::kMeta*): {max scratch, kexp}
static int f16_meta(eesen_b200_ctx *ctx, int idx, unsigned **mx, int **kexp) {
  void *m = nullptr;
  int rc = ctx->reserve(ctx->f16_meta, 4096, &m);
  if (rc) return rc;
  *mx = (unsigned *)m + 2 * idx;
  *kexp = (int *)m + 2 * idx + 1;
  return 0;
}

// hi / lo planes [rows x ldd] in `planes`, both 256-byte aligned
static int reserve_planes(eesen_b200_ctx *ctx, eesen_b200_ctx::Buf &planes, long rows, int cols, int ldd, eb::F16View *view) {
  const size_t pb = eb::f16x2_plane_bytes(rows, cols);
  void *pl = nullptr;
  int rc = ctx->reserve(planes, 2 * pb + 256, &pl);
  if (rc) return rc;
  view->hi = pl; view->lo = (char *)pl + ((pb + 255) & ~(size_t)255); view->ld = ldd;
  return 0;
}

// convert src [rows x cols] (ld) into planes on the stream of on_side; the scan scratch and the scale exponent go to
// f16_meta record `meta`.  timed: as a product of that stream (else it is timed inside the product it feeds).
static int convert_planes(eesen_b200_ctx *ctx, eesen_b200_ctx::Buf &planes, int meta, const float *src, long rows, int cols,
                          int ld, bool on_side, const unsigned *known_max, bool timed, eb::F16View *view) {
  unsigned *mx; int *kx;
  int rc;
  if ((rc = reserve_planes(ctx, planes, rows, cols, (cols + 7) & ~7, view))) return rc;
  if ((rc = f16_meta(ctx, meta, &mx, &kx))) return rc;
  view->kexp = kx;
  return launch(ctx, timed ? (int)eesen_b200_ctx::kGemm : kUntimed, known_max ? 1 : 2, "convert_f16x2", [&] {
    return eb::convert_f16x2(on_side ? ctx->side : ctx->stream, ctx->num_sms, src, rows, cols, ld, (void *)view->hi,
                             (void *)view->lo, mx, kx, known_max);
  }, on_side);
}

// the per-pass entry of `base`: its own slot, else the next one round robin
static int act_slot(eesen_b200_ctx *ctx, const float *base) {
  int slot = -1;
  for (int i = 0; i < eesen_b200_ctx::kActSlots; i++)
    if (ctx->act[i].base == base) slot = i;
  if (slot < 0) { slot = ctx->act_next; ctx->act_next = (ctx->act_next + 1) % eesen_b200_ctx::kActSlots; }
  return slot;
}

// a [r x c] block at P with leading dimension ld: inside a registered matrix (or a layer output whose planes the
// recurrent forward kernel wrote during this forward pass)?
static bool f16_lookup(eesen_b200_ctx *ctx, const float *P, long r, int c, int ld, eb::F16View *out) {
  for (int i = 0; i < ctx->f16_used; i++)
    if (ctx->f16_slots[i].find(P, r, c, ld, out)) return true;
  for (int i = 0; i < eesen_b200_ctx::kActSlots; i++)
    if (ctx->act[i].gen == ctx->act_gen && ctx->act[i].find(P, r, c, ld, out)) return true;
  return false;
}

// convert the whole matrix [rows x cols] (ld) and remember it: later products find sub-blocks by address
// persist (only while a Net drives a training forward pass, ctx->act_enable): the planes go to a per-pass entry and stay
// valid until the next forward pass -- the input weights Wx, which the dX product of the backward pass reads again
static int f16_register(eesen_b200_ctx *ctx, const float *base, long rows, int cols, int ld, bool on_side = false,
                        const unsigned *known_max = nullptr, bool persist = false) {
  if (!ctx->f16x3 || ctx->gemm_prec != 0 || ctx->gemm_engine != 0 || !base || rows <= 0 || cols <= 0) return 0;
  { eb::F16View have; if (f16_lookup(ctx, base, rows, cols, ld, &have)) return 0; }   // (e.g. planes the forward kernel wrote)
  const bool act = persist && ctx->act_enable;
  if (!act && ctx->f16_used >= eesen_b200_ctx::kF16Slots) return 0;   // (falls back to per-call conversion)
  const int slot = act ? act_slot(ctx, base) : ctx->f16_used;
  eesen_b200_ctx::PlaneEntry &e = act ? ctx->act[slot] : ctx->f16_slots[slot];
  const int meta = act ? eesen_b200_ctx::kMetaAct + slot : eesen_b200_ctx::kMetaCall + slot;
  int rc = convert_planes(ctx, e.planes, meta, base, rows, cols, ld, on_side, known_max, true, &e.view);
  if (rc) return rc;
  e.base = base; e.rows = rows; e.cols = cols; e.ld = ld; e.gen = act ? ctx->act_gen : 0;
  if (!act) ctx->f16_used++;
  return 0;
}

// planes for the layer output `out` [rows x cols] (ld) that the tcgen05 forward kernel is about to write (fixed scale 2^13)
static int act_planes_for(eesen_b200_ctx *ctx, const float *out, long rows, int cols, int ld, eb::LstmFwdArgs *a) {
  if (!ctx->act_enable || !ctx->f16x3 || ctx->gemm_prec != 0 || ctx->gemm_engine != 0 || (cols & 7)) return 0;
  eesen_b200_ctx::PlaneEntry &e = ctx->act[act_slot(ctx, out)];
  int rc = reserve_planes(ctx, e.planes, rows, cols, cols, &e.view);
  if (rc) return rc;
  if (!ctx->act_kexp) {
    unsigned *mx; int *kx;
    if ((rc = f16_meta(ctx, eesen_b200_ctx::kMetaK13, &mx, &kx))) return rc;
    static const int k13 = 13;
    if ((rc = ctx->check(cudaMemcpyAsync(kx, &k13, sizeof(int), cudaMemcpyHostToDevice, ctx->stream), "cudaMemcpyAsync"))) return rc;
    ctx->act_kexp = kx;
  }
  e.base = out; e.rows = rows; e.cols = cols; e.ld = ld; e.gen = ctx->act_gen; e.view.kexp = ctx->act_kexp;
  a->out_hi = (void *)e.view.hi; a->out_lo = (void *)e.view.lo; a->ldh = e.view.ld;
  return 0;
}

// view of an operand: registered, or converted on the spot into the stream's temporary planes (which = 0 A, 1 B)
static int f16_operand(eesen_b200_ctx *ctx, bool on_side, int which, const float *P, long r, int c, int ld, eb::F16View *out) {
  if (f16_lookup(ctx, P, r, c, ld, out)) return 0;
  const int t = (on_side ? 2 : 0) + which;
  return convert_planes(ctx, ctx->f16_tmp[t], eesen_b200_ctx::kMetaTmp + t, P, r, c, ld, on_side, nullptr, false, out);
}

static int do_gemm(eesen_b200_ctx *ctx, int ta, int tb, int M, int N, int K, float alpha, const float *A, int lda,
                   long sA, const float *B, int ldb, long sB, float beta, float *C, int ldc, long sC,
                   const float *bias, long sBias, int batch, bool on_side = false) {
  void *ws = nullptr;
  int rc;
  cudaStream_t st = on_side ? ctx->side : ctx->stream;
  eesen_b200_ctx::Buf &gemm_ws = on_side ? ctx->gemm_ws_side : ctx->gemm_ws;
  eesen_b200_ctx::Buf &bf16_a = on_side ? ctx->bf16_a_side : ctx->bf16_a, &bf16_b = on_side ? ctx->bf16_b_side : ctx->bf16_b;
  // tensor-core engine: tcgen05/TMEM/TMA (gemm_tc.cu) for every arithmetic mode -- fp16x3: fp32-faithful arithmetic on
  // the 16-bit tensor pipe, two fp16 planes per operand (registered whole-matrix conversions where the caller made them,
  // else converted here), three kind::f16 MMAs per k-slice; bf16: kind::f16 on bf16 copies of the operands (BASELINE
  // config 4); kind::tf32 for EESEN_B200_GEMM_FP32X3=tf32 and tf32.  The warp-level mma.sync kernel (gemm.cu) is kept
  // for EESEN_B200_GEMM_ENGINE=legacy (A/B measurements) and matrices TMA cannot address.
  enum { kLegacy, kF16x3, kBf16, kTf32 } eng = kLegacy;
  const bool tc16 = !(ta && tb) && M > 0 && N > 0 && K > 0;
  if (ctx->gemm_engine == 0) {
    if (ctx->gemm_prec == 0 && ctx->f16x3 && tc16 && eb::gemm_tc_supported(ta, tb, M, N, K, A, 4, B, 4, 0))
      eng = kF16x3;
    else if (ctx->gemm_prec == 2 && tc16 && eb::gemm_tc_supported(ta, tb, M, N, K, A, 4, B, 4, 0))
      eng = kBf16;
    else if (eb::gemm_tc_supported(ta, tb, M, N, K, A, lda, B, ldb, ctx->gemm_prec) &&
             (batch == 1 || ((sA & 3) == 0 && (sB & 3) == 0)))
      eng = kTf32;
  }
  if (eng == kLegacy) {
    if (K >= 4096 && (rc = ctx->reserve(gemm_ws, eb::gemm_workspace_bytes(M, N, K, batch, ctx->num_sms), &ws))) return rc;
    return launch(ctx, eesen_b200_ctx::kGemm, 1, "gemm", [&] {
      return eb::gemm(st, ctx->num_sms, ta, tb, M, N, K, alpha, A, lda, sA, B, ldb, sB, beta, C, ldc, sC, bias, sBias,
                      batch, ctx->gemm_prec, (float *)ws, ws ? gemm_ws.bytes : 0);
    }, on_side);
  }
  const size_t need_tc = eb::gemm_tc_workspace_bytes(M, N, K, ctx->num_sms);
  if (need_tc && (rc = ctx->reserve(gemm_ws, need_tc, &ws))) return rc;
  const size_t ws_bytes = ws ? gemm_ws.bytes : 0;
  // operands as stored: A [M x K] or [K x M], B [N x K] or [K x N]
  const long ar = ta ? K : M, br = tb ? N : K;
  const int ac = ta ? M : K, bc = tb ? K : N;
  void *a16 = nullptr, *b16 = nullptr;
  if (eng == kBf16) {
    if ((rc = ctx->reserve(bf16_a, eb::gemm_tc16_operand_bytes(ar, ac), &a16))) return rc;
    if ((rc = ctx->reserve(bf16_b, eb::gemm_tc16_operand_bytes(br, bc), &b16))) return rc;
  }
  for (int b = 0; b < batch; b++) {
    const float *Ab = A + b * sA, *Bb = B + b * sB, *bb = bias ? bias + b * sBias : nullptr;
    float *Cb = C + b * sC;
    int pe = ctx->prof_begin(eesen_b200_ctx::kGemm, on_side);
    cudaError_t e = cudaSuccess;
    const char *what = "gemm_tc";
    if (eng == kF16x3) {
      eb::F16View va, vb;
      if ((rc = f16_operand(ctx, on_side, 0, Ab, ar, ac, lda, &va))) return rc;
      if ((rc = f16_operand(ctx, on_side, 1, Bb, br, bc, ldb, &vb))) return rc;
      e = eb::gemm_tc16x3(st, ctx->num_sms, ta, tb, M, N, K, alpha, va, vb, beta, Cb, ldc, bb, (float *)ws, ws_bytes);
      what = "gemm_tc16x3";
    } else if (eng == kBf16) {
      if (b == 0 || sA != 0) { e = eb::convert_bf16(st, ctx->num_sms, Ab, ar, ac, lda, a16); ctx->launches += 1; }
      if (e == cudaSuccess && (b == 0 || sB != 0)) { e = eb::convert_bf16(st, ctx->num_sms, Bb, br, bc, ldb, b16); ctx->launches += 1; }
      if (e == cudaSuccess) e = eb::gemm_tc16(st, ctx->num_sms, ta, tb, M, N, K, alpha, a16, b16, beta, Cb, ldc, bb, (float *)ws, ws_bytes);
      what = "gemm_tc16";
    } else {
      e = eb::gemm_tc(st, ctx->num_sms, ta, tb, M, N, K, alpha, Ab, lda, Bb, ldb, beta, Cb, ldc, bb, ctx->gemm_prec,
                      (float *)ws, ws_bytes);
    }
    ctx->prof_end(pe);
    ctx->launches += 1;
    if ((rc = ctx->check(e, what))) return rc;
  }
  return 0;
}

int eesen_b200_gemm(eesen_b200_ctx *ctx, int transA, int transB, int M, int N, int K, float alpha, const float *A,
                    int lda, const float *B, int ldb, float beta, float *C, int ldc) {
  if (!ctx || !A || !B || !C) return EESEN_B200_EINVAL;
  return do_gemm(ctx, transA, transB, M, N, K, alpha, A, lda, 0, B, ldb, 0, beta, C, ldc, 0, nullptr, 0, 1);
}

// Picks the resident-weight plan.  The recurrence is independent per utterance, so a minibatch that
// does not fit one co-resident grid (e.g. 128 utterances at C=320) is processed in utterance chunks
// of the largest size that does: chunk = S, else the largest multiple of 8 in {64, 32, 16, 8}.
static int lstm_prepare(eesen_b200_ctx *ctx, int ndir, int pass, int S, int C, eb::LstmPlan *plan, int *chunk, float **pbuf,
                        float **gsum, void **xbuf) {
  const int cands[5] = {S, 64, 32, 16, 8};
  plan->valid = 0;
  for (int i = 0; i < 5 && !plan->valid; i++) {
    if (cands[i] > S || cands[i] <= 0) continue;
    *plan = eb::lstm_plan(cands[i], C, ctx->num_sms, ctx->max_smem, ndir, pass);
    *chunk = cands[i];
  }
  if (!plan->valid)
    return ctx->fail(EESEN_B200_ESHAPE, "no resident-weight LSTM configuration fits C=" + std::to_string(C) +
                                            " on this device (cells per direction must be a multiple of 8, <= ~640)");
  int rc;
  const int nchunks = (S + *chunk - 1) / *chunk;
  if ((rc = ctx->reserve(ctx->lstm_pbuf, plan->pbuf_floats * sizeof(float), (void **)pbuf))) return rc;
  if ((rc = ctx->reserve(ctx->lstm_gsum, plan->gsum_floats * sizeof(float) * nchunks, (void **)gsum))) return rc;
  if ((rc = ctx->reserve(ctx->lstm_flags, plan->xbuf_bytes, xbuf))) return rc;
  return 0;
}

// the recurrent weights and peepholes of each direction for the kernels (ndir = 1: direction 0 in both), and the row
// stride of Wx (0 in the params = dense)
static int lstm_dir_params(eesen_b200_ctx *ctx, int ndir, int I, int C, const eesen_b200_bilstm_params *p,
                           eb::LstmDirParams dp[2], int *ldwx) {
  const int ldwm = p->ldwm > 0 ? p->ldwm : C;
  *ldwx = p->ldwx > 0 ? p->ldwx : I;
  if (*ldwx < I || ldwm < C) return ctx->fail(EESEN_B200_EINVAL, "ldwx / ldwm smaller than the matrix width");
  for (int d = 0; d < 2; d++) {
    const int q = d < ndir ? d : 0;
    dp[d].wm = p->wm[q]; dp[d].ldwm = ldwm; dp[d].pi = p->pi[q]; dp[d].pf = p->pf[q]; dp[d].po = p->po[q];
  }
  return 0;
}

// ndir = 2: BiLstmParallel (gates [N x 8C], cell/out [N x 2C]); ndir = 1: LstmParallel, the forward cells
// alone (gates [N x 4C], cell/out [N x C], index 0 of the parameter arrays) -- lstm-parallel-layer.h:47-113
// is the forward-cell pass of bilstm-parallel-layer.h:97-150 line for line.
static int lstm_forward_impl(eesen_b200_ctx *ctx, int ndir, int T, int S, int I, int C, const int *d_len,
                             const float *x, int ldx, const eesen_b200_bilstm_params *p, float *gates, float *cell,
                             float *out, int ldo, int drop = 0, const float *rmask = nullptr, int ldr = 0,
                             int per_step = 0) {
  if (drop < 0 || drop > 2 || (drop != 0 && (!rmask || ldr < ndir * C))) return EESEN_B200_EINVAL;
  if (!ctx || !p || !x || !gates || !cell || !out || T <= 0 || S <= 0) return EESEN_B200_EINVAL;
  eb::LstmPlan plan;
  float *pbuf, *gsum;
  void *xbuf;
  int chunk = S;
  int rc = lstm_prepare(ctx, ndir, 0, S, C, &plan, &chunk, &pbuf, &gsum, &xbuf);
  if (rc) return rc;
  // input-side gate pre-activations for both directions: G[:, d*4C..] = x * Wx_d^T + b_d
  // (bilstm-parallel-layer.h:109-110,163-164).  Batched over the direction when the two weight
  // blocks are equally strided (they are in the Net arena), else two launches.
  long sW = ndir == 2 ? p->wx[1] - p->wx[0] : 0, sB = ndir == 2 ? p->bias[1] - p->bias[0] : 0;
  const int N = T * S, ldg = ndir * 4 * C;
  eb::LstmFwdArgs a;
  int ldwx;
  if ((rc = lstm_dir_params(ctx, ndir, I, C, p, a.p, &ldwx))) return rc;
  // fp16x3: the layer input feeds the products of both directions -- one conversion
  ctx->join_side();
  ctx->f16_clear();
  if ((rc = f16_register(ctx, x, N, I, ldx))) return rc;
  for (int d = 0; d < ndir; d++)
    if ((rc = f16_register(ctx, p->wx[d], 4 * C, I, ldwx, false, nullptr, true))) return rc;
  // Streamed: with the tcgen05 engine (80 of 148 SMs, latency-bound) the product is cut along time into chunks in the
  // order the two directions consume G -- direction 0 from t = 0 upwards, direction 1 from t = T-1 downwards.  The
  // first kReady chunks run here, the others on the side stream next to the recurrent kernel, which checks
  // gflag[chunk] before the first read of a chunk.
  const int kReady = 1;   // (measured per C2 step: 14.86 ms at 1, 15.13 at 2, 15.45 at 3)
  int gchunk = 0, nchunks_g = 0;
  unsigned *gflags = nullptr;
  if (plan.engine == 1 && chunk == S && ctx->overlap && T >= 256) {
    gchunk = std::max(32, (T + 9) / 10);
    nchunks_g = (T + gchunk - 1) / gchunk;
    if (nchunks_g <= kReady || nchunks_g > 64) nchunks_g = 0;
  }
  if (nchunks_g) {
    void *gf = nullptr;
    const bool fresh = ctx->lstm_gflags.bytes == 0;
    if ((rc = ctx->reserve(ctx->lstm_gflags, 64 * sizeof(unsigned), &gf))) return rc;
    gflags = (unsigned *)gf;
    if (fresh && (rc = ctx->check(cudaMemsetAsync(gf, 0, 64 * sizeof(unsigned), ctx->stream), "cudaMemsetAsync"))) return rc;
    ctx->gepoch += 1;
    if (ctx->gepoch == 0u) ctx->gepoch = 1;     // 0 = "never set"
    ctx->fork_side();                           // the side stream waits for the operand conversions above
    for (int ci = 0; ci < nchunks_g; ci++) {
      const bool on_side = ci >= kReady;
      const int t0 = ci * gchunk, nt = std::min(gchunk, T - t0);
      for (int d = 0; d < ndir; d++) {
        const long r0 = (long)(d == 0 ? t0 : T - t0 - nt) * S;
        rc = do_gemm(ctx, 0, 1, nt * S, 4 * C, I, 1.f, x + r0 * ldx, ldx, 0, p->wx[d], ldwx, 0, 0.f,
                     gates + r0 * ldg + (size_t)d * 4 * C, ldg, 0, p->bias[d], 0, 1, on_side);
        if (rc) return rc;
      }
      if (on_side && (rc = launch(ctx, kUntimed, 1, "lstm_set_flag",
                                  [&] { return eb::lstm_set_flag(ctx->side, gflags + ci, ctx->gepoch); })))
        return rc;
    }
  } else if (ndir == 2 && sW > 0 && (sW & 3) == 0 && sB > 0) {
    rc = do_gemm(ctx, 0, 1, N, 4 * C, I, 1.f, x, ldx, 0, p->wx[0], ldwx, sW, 0.f, gates, ldg, 4 * C, p->bias[0], sB, 2);
    if (rc) return rc;
  } else {
    for (int d = 0; d < ndir; d++) {
      rc = do_gemm(ctx, 0, 1, N, 4 * C, I, 1.f, x, ldx, 0, p->wx[d], ldwx, 0, 0.f, gates + (size_t)d * 4 * C, ldg, 0,
                   p->bias[d], 0, 1);
      if (rc) return rc;
    }
  }
  a.T = T; a.S = S; a.C = C; a.len = d_len;
  a.G = gates; a.ldg = ldg;
  a.cell = cell; a.ldc = ndir * C;
  a.out = out; a.ldo = ldo;
  a.xbuf = xbuf;
  a.precision = ctx->rec_prec;
  a.drop = drop; a.rmask = rmask; a.ldr = ldr; a.rmask_per_step = per_step;
  if (plan.engine == 1 && (rc = act_planes_for(ctx, out, N, ndir * C, ldo, &a))) return rc;
  if (nchunks_g) { a.gflag = gflags; a.gepoch = ctx->gepoch; a.gchunk = gchunk; a.gready = kReady; }
  for (int s0 = 0; s0 < S; s0 += chunk) {
    a.s_begin = s0;
    a.s_count = std::min(chunk, S - s0);
    if ((rc = launch(ctx, eesen_b200_ctx::kLstmFwd, 1, "lstm_forward", [&] { return eb::lstm_forward(ctx->stream, plan, a); })))
      return rc;
  }
  return 0;
}

int eesen_b200_bilstm_forward(eesen_b200_ctx *ctx, int T, int S, int I, int C, const int *d_len, const float *x,
                              int ldx, const eesen_b200_bilstm_params *p, float *gates, float *cell, float *out,
                              int ldo) {
  if (!d_len) return EESEN_B200_EINVAL;
  return lstm_forward_impl(ctx, 2, T, S, I, C, d_len, x, ldx, p, gates, cell, out, ldo);
}

int eesen_b200_bilstm_forward_dropout(eesen_b200_ctx *ctx, int T, int S, int I, int C, const int *d_len, const float *x,
                                      int ldx, const eesen_b200_bilstm_params *p, float *gates, float *cell,
                                      float *out, int ldo, int drop, const float *rmask, int ldr, int per_step) {
  if (!d_len) return EESEN_B200_EINVAL;
  return lstm_forward_impl(ctx, 2, T, S, I, C, d_len, x, ldx, p, gates, cell, out, ldo, drop, rmask, ldr, per_step);
}

int eesen_b200_bilstm_backward_dropout(eesen_b200_ctx *ctx, int T, int S, int I, int C, const float *x, int ldx,
                                       const eesen_b200_bilstm_params *p, const float *gates, const float *cell,
                                       const float *out, int ldo, const float *dout, int ldd, float *dgates, float *dx,
                                       int lddx, const eesen_b200_bilstm_grads *gr, int drop, const float *rmask,
                                       int ldr, int per_step);

int eesen_b200_mul_elements(eesen_b200_ctx *ctx, int N, int cols, const float *a, int lda, const float *b, int ldb,
                            float *out, int ldo) {
  if (!ctx || !a || !b || !out || N < 0 || cols < 1) return EESEN_B200_EINVAL;
  return launch(ctx, eesen_b200_ctx::kMisc, 1, "mul_elements",
                [&] { return eb::mul_elements(ctx->stream, ctx->num_sms, N, cols, a, lda, b, ldb, out, ldo); });
}

int eesen_b200_dropout_mask(eesen_b200_ctx *ctx, int rows, int cols, float *d_mask, int ld, float p, int per_col,
                            unsigned long long seed, unsigned long long stream) {
  if (!ctx || !d_mask || rows < 0 || cols < 1 || ld < cols || !(p >= 0.f && p < 1.f)) return EESEN_B200_EINVAL;
  return launch(ctx, eesen_b200_ctx::kMisc, 1, "dropout_mask",
                [&] { return eb::dropout_mask(ctx->stream, ctx->num_sms, rows, cols, d_mask, ld, p, per_col, seed, stream); });
}

int eesen_b200_lstm_forward(eesen_b200_ctx *ctx, int T, int S, int I, int C, const float *x, int ldx,
                            const eesen_b200_bilstm_params *p, float *gates, float *cell, float *out, int ldo) {
  return lstm_forward_impl(ctx, 1, T, S, I, C, NULL, x, ldx, p, gates, cell, out, ldo);
}

static int lstm_backward_impl(eesen_b200_ctx *ctx, int ndir, int T, int S, int I, int C, const float *x, int ldx,
                              const eesen_b200_bilstm_params *p, const float *gates, const float *cell,
                              const float *out, int ldo, const float *dout, int ldd, float *dgates, float *dx,
                              int lddx, const eesen_b200_bilstm_grads *gr, int drop = 0, const float *rmask = nullptr,
                              int ldr = 0, int per_step = 0) {
  if (drop < 0 || drop > 2 || (drop != 0 && (!rmask || ldr < ndir * C))) return EESEN_B200_EINVAL;
  if (!ctx || !p || !gr || !x || !gates || !cell || !out || !dout || !dgates || T <= 0 || S <= 0) return EESEN_B200_EINVAL;
  eb::LstmPlan plan;
  float *pbuf, *gsum;
  void *xbuf;
  int chunk = S;
  int rc = lstm_prepare(ctx, ndir, 1, S, C, &plan, &chunk, &pbuf, &gsum, &xbuf);
  if (rc) return rc;
  const int nchunks = (S + chunk - 1) / chunk;
  const int ldg = ndir * 4 * C;
  eb::LstmBwdArgs a;
  int ldwx;
  if ((rc = lstm_dir_params(ctx, ndir, I, C, p, a.p, &ldwx))) return rc;
  const int gldwx = gr->ldwx > 0 ? gr->ldwx : I, gldwm = gr->ldwm > 0 ? gr->ldwm : C;
  if (gldwx < I || gldwm < C) return ctx->fail(EESEN_B200_EINVAL, "ldwx / ldwm smaller than the matrix width");
  a.T = T; a.S = S; a.C = C;
  a.G = gates; a.ldg = ldg;
  a.cell = cell; a.ldc = ndir * C;
  a.dout = dout; a.ldd = ldd;
  a.DG = dgates; a.lddg = ldg;
  a.pbuf = pbuf; a.gsum = gsum;
  a.precision = ctx->rec_prec;
  a.drop = drop; a.rmask = rmask; a.ldr = ldr; a.rmask_per_step = per_step;
  // fp16x3: the layer input and m feed the weight-gradient products; they are forward activations, so their planes are
  // made on the side stream (behind the weight-gradient products of the layer above, which still read the previous
  // planes) WHILE the recurrent kernel below runs.  d(gates) and Wx follow on `stream` behind the kernel.
  const int N = T * S;
  const bool sd = ctx->overlap != 0;
  ctx->f16_clear();
  // max |DG| comes out of the tcgen05 kernel itself (a.dgmax): the conversion of DG below needs no scan of its own
  unsigned *dgmax = nullptr;
  if (plan.engine == 1 && ctx->f16x3 && ctx->gemm_prec == 0 && ctx->gemm_engine == 0) {
    int *unused_k;
    if ((rc = f16_meta(ctx, eesen_b200_ctx::kMetaDgmax, &dgmax, &unused_k))) return rc;
    if ((rc = ctx->check(cudaMemsetAsync(dgmax, 0, sizeof(unsigned), ctx->stream), "cudaMemsetAsync"))) return rc;
    a.dgmax = dgmax;
  }
  if (sd) {
    ctx->fork_side();
    if ((rc = f16_register(ctx, x, N, I, ldx, true))) return rc;
    if (T > 1 && (rc = f16_register(ctx, out, N, ndir * C, ldo, true))) return rc;
  }
  for (int ci = 0; ci < nchunks; ci++) {
    a.s_begin = ci * chunk;
    a.s_count = std::min(chunk, S - a.s_begin);
    a.gsum = gsum + (size_t)ci * plan.gsum_floats;
    if ((rc = launch(ctx, eesen_b200_ctx::kLstmBwd, 1, "lstm_backward", [&] { return eb::lstm_backward(ctx->stream, plan, a); })))
      return rc;
  }
  for (int d = 0; d < ndir; d++)
    if ((rc = launch(ctx, eesen_b200_ctx::kMisc, 1, "lstm_reduce_gsum", [&] {
           return eb::lstm_reduce_gsum(ctx->stream, plan, C, gsum, nchunks, gr->bias[d], gr->pi[d], gr->pf[d], gr->po[d], d);
         })))
      return rc;
  // fp16x3: d(gates), the layer input, m and Wx each feed several of the products below -- one conversion each.
  // The planes of the previous layer call may still be read by its weight-gradient products on the side stream:
  // they have had the whole recurrent kernel above to finish, now they are waited for.
  ctx->join_side();
  if (!sd) {
    if ((rc = f16_register(ctx, x, N, I, ldx))) return rc;
    if (T > 1 && (rc = f16_register(ctx, out, N, ndir * C, ldo))) return rc;
  }
  if ((rc = f16_register(ctx, dgates, N, ndir * 4 * C, ldg, false, dgmax))) return rc;
  if (dx) {
    for (int d = 0; d < ndir; d++)
      if ((rc = f16_register(ctx, p->wx[d], 4 * C, I, ldwx))) return rc;
    // dx = DG_fw * Wx_fw + DG_bw * Wx_bw   (:502 beta=0, :593 beta=1)
    for (int d = 0; d < ndir; d++)
      if ((rc = do_gemm(ctx, 0, 0, N, I, 4 * C, 1.f, dgates + (size_t)d * 4 * C, ldg, 0, p->wx[d], ldwx, 0,
                        d == 0 ? 0.f : 1.f, dx, lddx, 0, nullptr, 0, 1)))
        return rc;
  }
  // The weight-gradient products below are consumed only by the all-reduce / update at the end of the step: they go
  // to the side stream (forked here, after the recurrent kernel and the bias / peephole sums) and overlap with the
  // dX product above and with the recurrent backward of the layer below.
  if (sd) ctx->fork_side();
  long sGW = ndir == 2 ? gr->wx[1] - gr->wx[0] : 0, sGM = ndir == 2 ? gr->wm[1] - gr->wm[0] : 0;
  bool batched = ndir == 2 && sGW > 0 && (sGW & 3) == 0 && sGM > 0 && (sGM & 3) == 0;
  // Wx grad = DG^T * x   (:505 / :596), both directions batched
  if (batched) {
    rc = do_gemm(ctx, 1, 0, 4 * C, I, N, 1.f, dgates, ldg, 4 * C, x, ldx, 0, 0.f, gr->wx[0], gldwx, sGW, nullptr, 0, 2, sd);
    if (rc) return rc;
  } else {
    for (int d = 0; d < ndir; d++) {
      rc = do_gemm(ctx, 1, 0, 4 * C, I, N, 1.f, dgates + (size_t)d * 4 * C, ldg, 0, x, ldx, 0, 0.f, gr->wx[d], gldwx, 0,
                   nullptr, 0, 1, sd);
      if (rc) return rc;
    }
  }
  // Wm grad = DG^T * m_prev: fw pairs DG rows [S, N) with out rows [0, N-S) (:506);
  //                          bw pairs DG rows [0, N-S) with out rows [S, N) (:597)
  if (T > 1) {
    const int Nm = N - S;
    // (no layer below -- dx == NULL: nothing waits on `stream`, so the forward cells' product runs there, next to the
    // backward cells' on the side stream; it shortens the tail of the step in front of the optimiser)
    rc = do_gemm(ctx, 1, 0, 4 * C, C, Nm, 1.f, dgates + (size_t)S * ldg, ldg, 0, out, ldo, 0, 0.f, gr->wm[0], gldwm, 0,
                 nullptr, 0, 1, sd && (dx != nullptr || ndir == 1));
    if (rc) return rc;
    if (ndir == 2) {
      rc = do_gemm(ctx, 1, 0, 4 * C, C, Nm, 1.f, dgates + 4 * C, ldg, 0, out + (size_t)S * ldo + C, ldo, 0, 0.f,
                   gr->wm[1], gldwm, 0, nullptr, 0, 1, sd);
      if (rc) return rc;
    }
  } else {
    for (int d = 0; d < ndir; d++)
      CTX_CHECK(cudaMemset2DAsync(gr->wm[d], sizeof(float) * gldwm, 0, sizeof(float) * C, 4 * C, sd ? ctx->side : ctx->stream), "memset");
  }
  return 0;
}

int eesen_b200_bilstm_backward(eesen_b200_ctx *ctx, int T, int S, int I, int C, const float *x, int ldx,
                               const eesen_b200_bilstm_params *p, const float *gates, const float *cell,
                               const float *out, int ldo, const float *dout, int ldd, float *dgates, float *dx,
                               int lddx, const eesen_b200_bilstm_grads *gr) {
  return lstm_backward_impl(ctx, 2, T, S, I, C, x, ldx, p, gates, cell, out, ldo, dout, ldd, dgates, dx, lddx, gr);
}

int eesen_b200_bilstm_backward_dropout(eesen_b200_ctx *ctx, int T, int S, int I, int C, const float *x, int ldx,
                                       const eesen_b200_bilstm_params *p, const float *gates, const float *cell,
                                       const float *out, int ldo, const float *dout, int ldd, float *dgates, float *dx,
                                       int lddx, const eesen_b200_bilstm_grads *gr, int drop, const float *rmask,
                                       int ldr, int per_step) {
  return lstm_backward_impl(ctx, 2, T, S, I, C, x, ldx, p, gates, cell, out, ldo, dout, ldd, dgates, dx, lddx, gr, drop,
                            rmask, ldr, per_step);
}

int eesen_b200_lstm_backward(eesen_b200_ctx *ctx, int T, int S, int I, int C, const float *x, int ldx,
                             const eesen_b200_bilstm_params *p, const float *gates, const float *cell,
                             const float *out, int ldo, const float *dout, int ldd, float *dgates, float *dx,
                             int lddx, const eesen_b200_bilstm_grads *gr) {
  return lstm_backward_impl(ctx, 1, T, S, I, C, x, ldx, p, gates, cell, out, ldo, dout, ldd, dgates, dx, lddx, gr);
}

int eesen_b200_affine_forward(eesen_b200_ctx *ctx, int N, int D, int K, const float *x, int ldx, const float *W,
                              const float *b, float *y, int ldy) {
  if (!ctx || !x || !W || !b || !y) return EESEN_B200_EINVAL;
  return do_gemm(ctx, 0, 1, N, K, D, 1.f, x, ldx, 0, W, D, 0, 0.f, y, ldy, 0, b, 0, 1);
}

int eesen_b200_affine_backward(eesen_b200_ctx *ctx, int N, int D, int K, const float *x, int ldx, const float *diff,
                               int lddiff, const float *W, float *dx, int lddx, float *dW, float *db) {
  if (!ctx || !x || !diff || !W) return EESEN_B200_EINVAL;
  int rc;
  if (dx && (rc = do_gemm(ctx, 0, 0, N, D, K, 1.f, diff, lddiff, 0, W, D, 0, 0.f, dx, lddx, 0, nullptr, 0, 1))) return rc;
  if (dW && (rc = do_gemm(ctx, 1, 0, K, D, N, 1.f, diff, lddiff, 0, x, ldx, 0, 0.f, dW, D, 0, nullptr, 0, 1))) return rc;
  if (db) {
    void *ws = nullptr;
    if ((rc = ctx->reserve(ctx->colsum_ws, eb::col_sum_ws_floats(K, ctx->num_sms) * sizeof(float), &ws))) return rc;
    if ((rc = launch(ctx, eesen_b200_ctx::kMisc, 2, "col_sum",
                     [&] { return eb::col_sum(ctx->stream, ctx->num_sms, N, K, diff, lddiff, db, (float *)ws); })))
      return rc;
  }
  return 0;
}

int eesen_b200_softmax(eesen_b200_ctx *ctx, int N, int K, const float *logits, int ld, float *probs, int ldp,
                       int *d_argmax) {
  if (!ctx || !logits || !probs) return EESEN_B200_EINVAL;
  return launch(ctx, eesen_b200_ctx::kSoftmax, 1, "softmax_rows",
                [&] { return eb::softmax_rows(ctx->stream, N, K, logits, ld, probs, ldp, d_argmax); });
}

int eesen_b200_row_argmax(eesen_b200_ctx *ctx, int N, int K, const float *x, int ld, int *d_argmax) {
  if (!ctx || !x || !d_argmax) return EESEN_B200_EINVAL;
  return launch(ctx, eesen_b200_ctx::kSoftmax, 1, "row_argmax",
                [&] { return eb::row_argmax(ctx->stream, N, K, x, ld, d_argmax); });
}

int eesen_b200_loglik(eesen_b200_ctx *ctx, int N, int K, float *y, int ld, int apply_log, const float *d_log_prior,
                      float prior_scale) {
  if (!ctx || !y || N < 0 || K < 1 || ld < K) return EESEN_B200_EINVAL;
  if (!apply_log && !d_log_prior) return 0;
  return launch(ctx, eesen_b200_ctx::kSoftmax, 1, "loglik_rows", [&] {
    return eb::loglik_rows(ctx->stream, ctx->num_sms, N, K, y, ld, apply_log, d_log_prior, prior_scale);
  });
}

int eesen_b200_ctc_eval(eesen_b200_ctx *ctx, int T, int S, int K, int max_lab, const int *d_len, const int *d_labels,
                        const int *d_lab_len, const float *probs, int ldp, float *pzx, float *diff, int ldd) {
  if (!ctx || !d_len || !d_labels || !d_lab_len || !probs || !pzx || !diff || max_lab < 1) return EESEN_B200_EINVAL;
  if (2 * max_lab + 1 > 1024) return ctx->fail(EESEN_B200_ESHAPE, "more than 511 labels per utterance");
  void *ws = nullptr;
  int rc = ctx->reserve(ctx->ctc_ws, eb::ctc_workspace_floats(T, S, max_lab) * sizeof(float), &ws);
  if (rc) return rc;
  return launch(ctx, eesen_b200_ctx::kCtc, 1, "ctc_eval", [&] {
    return eb::ctc_eval(ctx->stream, T, S, K, max_lab, d_len, d_labels, d_lab_len, probs, ldp, pzx, diff, ldd, (float *)ws);
  });
}

int eesen_b200_ce_eval(eesen_b200_ctx *ctx, int T, int S, int K, const int *d_len, const float *probs, int ldp,
                       const int *d_targets, float *diff, int ldd, double *d_stats) {
  if (!ctx || !d_len || !probs || !d_targets || !diff || !d_stats || T < 0 || S < 0 || K < 1 || ldp < K || ldd < K ||
      (ldp & 3) || (ldd & 3) || (((uintptr_t)probs | (uintptr_t)diff) & 15))   // ce_kernel moves rows as float4
    return EESEN_B200_EINVAL;
  void *ws = nullptr;
  int rc = ctx->reserve(ctx->ce_ws, eb::ce_workspace_bytes(T, S, ctx->num_sms), &ws);
  if (rc) return rc;
  return launch(ctx, eesen_b200_ctx::kSoftmax, 2, "ce_eval", [&] {
    return eb::ce_eval(ctx->stream, ctx->num_sms, T, S, K, d_len, probs, ldp, d_targets, diff, ldd, d_stats, ws);
  });
}

int eesen_b200_check_finite(eesen_b200_ctx *ctx, const float *d_x, int64_t n, int *flags) {
  if (!ctx || !flags || (n > 0 && !d_x) || n < 0) return EESEN_B200_EINVAL;
  ctx->join_side();
  void *d = nullptr;
  int rc = ctx->reserve(ctx->flag_buf, 64, &d);
  if (rc) return rc;
  if ((rc = launch(ctx, eesen_b200_ctx::kMisc, 1, "check_finite",
                   [&] { return eb::check_finite(ctx->stream, ctx->num_sms, d_x, (long)n, (int *)d); })))
    return rc;
  CTX_CHECK(cudaMemcpyAsync(flags, d, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream), "memcpy(flags)");
  CTX_CHECK(cudaStreamSynchronize(ctx->stream), "sync(flags)");
  return 0;
}

int eesen_b200_sgd_update(eesen_b200_ctx *ctx, float *w, float *corr, const float *grad, int64_t n, float momentum,
                          const eesen_b200_sgd_segment *segments, int nseg) {
  if (!ctx || !w || !corr || !grad || !segments || nseg < 1) return EESEN_B200_EINVAL;
  ctx->join_side();
  std::vector<eb::SgdSegment> h(nseg);
  for (int i = 0; i < nseg; i++) {
    h[i].offset = segments[i].offset; h[i].count = segments[i].count;
    h[i].lr = segments[i].lr; h[i].max_grad = segments[i].max_grad;
  }
  void *d;
  int rc = ctx->reserve(ctx->seg_buf, sizeof(eb::SgdSegment) * nseg, &d);
  if (rc) return rc;
  // synchronous small copy: the host vector dies at return
  CTX_CHECK(cudaMemcpyAsync(d, h.data(), sizeof(eb::SgdSegment) * nseg, cudaMemcpyHostToDevice, ctx->stream), "memcpy(segments)");
  CTX_CHECK(cudaStreamSynchronize(ctx->stream), "sync(segments)");
  return launch(ctx, kUntimed, 1, "sgd_momentum_clip", [&] {
    return eb::sgd_momentum_clip(ctx->stream, ctx->num_sms, w, corr, grad, momentum, (eb::SgdSegment *)d, nseg, (long)n);
  });
}

// ------------------------------------------------------------------------------------ NCCL (dlopen)
typedef struct { char internal[128]; } nccl_uid;
static void *nccl_open() {
  static void *lib = nullptr;
  if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  return lib;
}

int eesen_b200_nccl_unique_id(char id[128]) {
  void *lib = nccl_open();
  if (!lib) return EESEN_B200_ENCCL;
  typedef int (*fn_t)(nccl_uid *);
  fn_t f = (fn_t)dlsym(lib, "ncclGetUniqueId");
  if (!f) return EESEN_B200_ENCCL;
  nccl_uid u;
  int r = f(&u);
  if (r != 0) return EESEN_B200_ENCCL;
  memcpy(id, u.internal, 128);
  return 0;
}

int eesen_b200_nccl_init(eesen_b200_ctx *ctx, int rank, int nranks, const char id[128]) {
  if (!ctx || nranks < 1 || rank < 0 || rank >= nranks) return EESEN_B200_EINVAL;
  ctx->rank = rank;
  ctx->nranks = nranks;
  if (nranks == 1) return 0;
  void *lib = nccl_open();
  if (!lib) return ctx->fail(EESEN_B200_ENCCL, std::string("cannot load libnccl: ") + dlerror());
  ctx->nccl_lib = lib;
  typedef int (*init_t)(void **, int, nccl_uid, int);
  init_t f = (init_t)dlsym(lib, "ncclCommInitRank");
  if (!f) return ctx->fail(EESEN_B200_ENCCL, "ncclCommInitRank not found");
  nccl_uid u;
  memcpy(u.internal, id, 128);
  cudaSetDevice(ctx->device);
  int r = f(&ctx->nccl_comm, nranks, u, rank);
  if (r != 0) return ctx->fail(EESEN_B200_ENCCL, "ncclCommInitRank failed with code " + std::to_string(r));
  return 0;
}

static int allreduce_impl(eesen_b200_ctx *ctx, float *buf, int64_t n, bool on_side) {
  if (!ctx || !buf) return EESEN_B200_EINVAL;
  if (ctx->nranks == 1) return 0;
  if (!ctx->nccl_comm) return ctx->fail(EESEN_B200_ENCCL, "NCCL communicator not initialised");
  // ncclAllReduce(sendbuff, recvbuff, count, ncclFloat32 = 7, ncclSum = 0, comm, stream)
  typedef int (*ar_t)(const void *, void *, size_t, int, int, void *, cudaStream_t);
  static ar_t f = nullptr;
  if (!f) f = (ar_t)dlsym(ctx->nccl_lib, "ncclAllReduce");
  if (!f) return ctx->fail(EESEN_B200_ENCCL, "ncclAllReduce not found");
  int pe = ctx->prof_begin(eesen_b200_ctx::kAllReduce, on_side);
  int r = f(buf, buf, (size_t)n, 7, 0, ctx->nccl_comm, on_side ? ctx->side : ctx->stream);
  ctx->prof_end(pe);
  if (r != 0) return ctx->fail(EESEN_B200_ENCCL, "ncclAllReduce failed with code " + std::to_string(r));
  return 0;
}

int eesen_b200_allreduce_sum(eesen_b200_ctx *ctx, float *buf, int64_t n) {
  if (ctx) ctx->join_side();
  return allreduce_impl(ctx, buf, n, false);
}

// Bucketed variant for the layer loop of Net::Backpropagate (reference update order, src/net/net.cc:98-105): the
// gradient block of a layer is reduced on the side stream as soon as it is final -- behind that layer's
// weight-gradient products, in front of the next layer's -- while `stream` keeps back-propagating.  Everything
// queued on `stream` so far (bias / peephole sums, affine gradients) is waited for first.
int eesen_b200_allreduce_sum_overlapped(eesen_b200_ctx *ctx, float *buf, int64_t n) {
  if (!ctx) return EESEN_B200_EINVAL;
  if (ctx->nranks == 1) return 0;
  if (!ctx->overlap) return allreduce_impl(ctx, buf, n, false);
  ctx->fork_side();
  return allreduce_impl(ctx, buf, n, true);
}

int eesen_b200_profile(eesen_b200_ctx *ctx, int enable, double *ms, long *counts) {
  if (!ctx) return EESEN_B200_EINVAL;
  ctx->prof_collect();
  if (ms)
    for (int i = 0; i < eesen_b200_ctx::kNumCat; i++) ms[i] = ctx->prof_ms[i];
  if (counts)
    for (int i = 0; i < eesen_b200_ctx::kNumCat; i++) counts[i] = ctx->prof_count[i];
  if (enable >= 0) {
    ctx->prof_on = enable != 0;
    for (int i = 0; i < eesen_b200_ctx::kNumCat; i++) { ctx->prof_ms[i] = 0; ctx->prof_count[i] = 0; }
  }
  return 0;
}

int eesen_b200_lstm_engine(eesen_b200_ctx *ctx, int num_utts, int cells, int ndir, int pass) {
  if (!ctx) return -1;
  const eb::LstmPlan pl = eb::lstm_plan(num_utts, cells, ctx->num_sms, ctx->max_smem, ndir, pass);
  return pl.valid ? pl.engine : -1;
}

int eesen_b200_debug_lstm_timing(eesen_b200_ctx *ctx, long long *out32, int reset) {
  if (ctx) cudaStreamSynchronize(ctx->stream);
  return eb::lstm_debug_timing(out32, reset);
}

int eesen_b200_world(const eesen_b200_ctx *ctx, int *rank, int *nranks) {
  if (!ctx) return EESEN_B200_EINVAL;
  if (rank) *rank = ctx->rank;
  if (nranks) *nranks = ctx->nranks;
  return 0;
}

}  // extern "C"
