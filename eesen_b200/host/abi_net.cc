// eesen_b200/host/abi_net.cc -- level-2 C ABI: the Net/Ctc host mirror behind opaque handles
// (include/eesen_b200.h).  C++ exceptions (KALDI_ERR) are translated to error codes here.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/eesen_b200.h"
#include "context.h"
#include "net.h"

using namespace eesen;

struct eesen_b200_net {
  eesen_b200_ctx *ctx;
  Net net;
  Ctc ctc;
  CE ce;
  bool last_ce = false;       // the loss of the last step (eesen_b200_net_read_stats)
  CuMatrix<BaseFloat> feats, net_out, obj_diff, in_diff;
  float *h_pinned = nullptr;  // pinned staging for the packed features
  size_t h_cap = 0;
  std::vector<int> frames;
  std::vector<std::vector<int32> > labels;
  int S = 0;
  bool want_in_diff = false;
  float *d_prior = nullptr;   // log priors of the forward-only path
  size_t prior_dim = 0;
  std::vector<int32> targets;  // packed [T*S] frame targets of the host CE step
  explicit eesen_b200_net(eesen_b200_ctx *c) : ctx(c), net(c), ctc(c), ce(c) {}
  ~eesen_b200_net() {
    if (h_pinned) cudaFreeHost(h_pinned);
    if (d_prior) cudaFree(d_prior);
  }
};

#define GUARD(ctxp, body)                                      \
  try {                                                        \
    body;                                                      \
    return 0;                                                  \
  } catch (const std::exception &e) {                          \
    if (ctxp) (ctxp)->err = e.what();                          \
    return EESEN_B200_EIO;                                     \
  }

static void unpack_labels(eesen_b200_net *n, int S, const int *frames, const int *labels, const int *lab_len) {
  n->S = S;
  n->frames.assign(frames, frames + S);
  n->labels.resize(S);
  size_t off = 0;
  for (int s = 0; s < S; s++) {
    n->labels[s].assign(labels + off, labels + off + lab_len[s]);
    off += lab_len[s];
  }
}

// A caller that already holds the minibatch in page-locked memory (cudaHostAlloc / cudaHostRegister) is copied from
// directly; pageable memory goes through the pinned staging buffer first.  Either way ONE asynchronous H2D copy; the
// steps return only after the statistics are back, so the caller's buffer is free again on return.
static const float *stage_feats(eesen_b200_net *n, const float *feats, size_t elems) {
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, feats) == cudaSuccess && attr.type == cudaMemoryTypeHost) return feats;
  cudaGetLastError();   // a pageable pointer may leave cudaErrorInvalidValue behind on older drivers
  if (elems > n->h_cap) {
    if (n->h_pinned) cudaFreeHost(n->h_pinned);
    n->h_pinned = nullptr; n->h_cap = 0;
    if (cudaMallocHost((void **)&n->h_pinned, sizeof(float) * elems) != cudaSuccess) KALDI_ERR << "cudaMallocHost failed";
    n->h_cap = elems;
  }
  memcpy(n->h_pinned, feats, sizeof(float) * elems);
  return n->h_pinned;
}

static void run_step(eesen_b200_net *n, const CuMatrixBase<BaseFloat> &in, int train) {
  if (train) n->net.SetTrainMode(); else n->net.SetTestMode();           // train-ctc-parallel.cc:116-120
  n->net.SetSeqLengths(n->frames);                                      // train-ctc-parallel.cc:195
  n->net.Propagate(in, &n->net_out);                                    // :198
  n->ctc.EvalParallelAsync(n->frames, n->net_out, n->labels, &n->obj_diff);   // :199
  n->ctc.ErrorRateMSeqAsync(n->frames, n->net_out, n->labels);          // :202
  if (train) n->net.Backpropagate(n->obj_diff, n->want_in_diff ? &n->in_diff : NULL);   // :207
  n->last_ce = false;
}

// train-ce-parallel.cc:167-177; d_targets == NULL: the host targets in n->targets (validated by CE::EvalParallel)
static void run_step_ce(eesen_b200_net *n, const CuMatrixBase<BaseFloat> &in, const int *d_targets, int train) {
  if (train) n->net.SetTrainMode(); else n->net.SetTestMode();
  n->net.SetSeqLengths(n->frames);
  n->net.Propagate(in, &n->net_out);
  if (d_targets) n->ce.EvalParallelAsync(n->frames, n->net_out, d_targets, &n->obj_diff);
  else n->ce.EvalParallel(n->frames, n->net_out, n->targets, &n->obj_diff);
  if (train) n->net.Backpropagate(n->obj_diff, n->want_in_diff ? &n->in_diff : NULL);
  n->last_ce = true;
}

extern "C" {

int eesen_b200_net_read(eesen_b200_ctx *ctx, const char *model_path, eesen_b200_net **out) {
  if (!ctx || !model_path || !out) return EESEN_B200_EINVAL;
  *out = nullptr;
  eesen_b200_net *n = nullptr;
  try {
    n = new eesen_b200_net(ctx);
    n->net.Read(model_path);
    *out = n;
    return 0;
  } catch (const std::exception &e) {
    ctx->err = e.what();
    delete n;
    return EESEN_B200_EIO;
  }
}

int eesen_b200_net_write(eesen_b200_net *n, const char *path, int binary) {
  if (!n || !path) return EESEN_B200_EINVAL;
  GUARD(n->ctx, n->net.Write(path, binary != 0));
}

void eesen_b200_net_free(eesen_b200_net *n) { delete n; }

int eesen_b200_net_set_train_options(eesen_b200_net *n, float learn_rate, float momentum) {
  if (!n) return EESEN_B200_EINVAL;
  NetTrainOptions o = n->net.GetTrainOptions();
  o.learn_rate = learn_rate;
  o.momentum = momentum;
  GUARD(n->ctx, { n->net.SetTrainOptions(o); n->net.SetTrainMode(); });
}

int eesen_b200_net_set_optimizer(eesen_b200_net *n, const char *algorithm, float adagrad_epsilon, float rmsprop_rho,
                                 float rmsprop_one_minus_rho) {
  if (!n || !algorithm) return EESEN_B200_EINVAL;
  NetTrainOptions o = n->net.GetTrainOptions();
  o.adagrad_epsilon = adagrad_epsilon;
  o.rmsprop_rho = rmsprop_rho;
  o.rmsprop_one_minus_rho = rmsprop_one_minus_rho < 0.f ? 0.1f : rmsprop_one_minus_rho;
  GUARD(n->ctx, { n->net.SetUpdateAlgorithm(algorithm); n->net.SetTrainOptions(o); });
}

int eesen_b200_net_write_nonparallel(eesen_b200_net *n, const char *path, int binary) {
  if (!n || !path) return EESEN_B200_EINVAL;
  GUARD(n->ctx, n->net.WriteNonParal(path, binary != 0));
}

int eesen_b200_class_log_priors(const double *counts, int K, float prior_cutoff, float blank_scale, float *log_priors) {
  if (!counts || !log_priors || K < 1) return EESEN_B200_EINVAL;
  try {
    std::vector<double> c(counts, counts + K);
    std::vector<float> lp;
    ClassPrior::LogPriors(c, prior_cutoff, blank_scale, &lp);
    memcpy(log_priors, lp.data(), sizeof(float) * K);
    return 0;
  } catch (const std::exception &) {
    return EESEN_B200_EIO;
  }
}

int eesen_b200_net_feedforward(eesen_b200_net *n, const float *feats, int T, int S, const int *frames, int apply_log,
                               const float *log_priors, float prior_scale, float *out) {
  if (!n || !feats || !out || T <= 0 || S <= 0 || (!frames && S != 1)) return EESEN_B200_EINVAL;
  try {
    const int I = n->net.InputDim(), K = n->net.OutputDim();
    size_t elems = (size_t)T * S * std::max(I, K);
    if (elems > n->h_cap) {
      if (n->h_pinned) cudaFreeHost(n->h_pinned);
      n->h_pinned = nullptr; n->h_cap = 0;
      if (cudaMallocHost((void **)&n->h_pinned, sizeof(float) * elems) != cudaSuccess) KALDI_ERR << "cudaMallocHost failed";
      n->h_cap = elems;
    }
    memcpy(n->h_pinned, feats, sizeof(float) * (size_t)T * S * I);
    if (frames) n->frames.assign(frames, frames + S);
    else n->frames.clear();   // no SetSeqLengths, the reference tool's own call pattern: <BiLstm> layers only
    n->feats.Resize(T * S, I, kUndefined);
    n->feats.CopyFromHost(n->h_pinned, I);
    n->net.SetTestMode();   // net-output-extract.cc:75-76: no dropout in the forward-only path
    n->net.SetSeqLengths(n->frames);
    n->net.Feedforward(n->feats, &n->net_out);
    if (log_priors) {
      if ((int)n->prior_dim != K) {
        if (n->d_prior) cudaFree(n->d_prior);
        n->d_prior = nullptr;
        if (cudaMalloc((void **)&n->d_prior, sizeof(float) * K) != cudaSuccess) KALDI_ERR << "cudaMalloc failed";
        n->prior_dim = K;
      }
      if (cudaMemcpyAsync(n->d_prior, log_priors, sizeof(float) * K, cudaMemcpyHostToDevice, n->ctx->stream) != cudaSuccess)
        KALDI_ERR << "prior upload failed";
    }
    // ApplyLog + SubtractOnLogpost fused into one pass over [T*S x K]
    CheckAbi(n->ctx, eesen_b200_loglik(n->ctx, T * S, K, n->net_out.Data(), n->net_out.Stride(), apply_log,
                                       log_priors ? n->d_prior : NULL, prior_scale), "eesen_b200_loglik");
    n->net_out.CopyToHost(n->h_pinned, K);
    if (cudaStreamSynchronize(n->ctx->stream) != cudaSuccess) KALDI_ERR << "stream sync failed";
    memcpy(out, n->h_pinned, sizeof(float) * (size_t)T * S * K);
    return 0;
  } catch (const std::exception &e) {
    n->ctx->err = e.what();
    return EESEN_B200_EIO;
  }
}

int eesen_b200_net_change_dropout(eesen_b200_net *n, float forward_dropout, int fw_step, int fw_sequence, int rnndrop,
                                  int no_mem_loss, float recurrent_dropout, int rec_step, int rec_sequence,
                                  int twiddle_forward) {
  if (!n) return EESEN_B200_EINVAL;
  GUARD(n->ctx, n->net.ChangeDropoutParameters(forward_dropout, fw_step != 0, fw_sequence != 0, rnndrop != 0,
                                               no_mem_loss != 0, recurrent_dropout, rec_step != 0, rec_sequence != 0,
                                               twiddle_forward != 0));
}

int eesen_b200_net_set_dropout_seed(eesen_b200_net *n, unsigned long long seed) {
  if (!n) return EESEN_B200_EINVAL;
  GUARD(n->ctx, n->net.SetDropoutSeed(seed));
}

int eesen_b200_net_set_dropout_masks(eesen_b200_net *n, int layer, const float *fmask, int fmask_rows, const float *rmask,
                                     int rmask_rows) {
  if (!n || layer < 0 || layer >= n->net.NumLayers()) return EESEN_B200_EINVAL;
  BiLstmParallel *bl = dynamic_cast<BiLstmParallel *>(n->net.GetLayer(layer));
  if (!bl) return EESEN_B200_EINVAL;
  GUARD(n->ctx, bl->InjectDropoutMasks(fmask, fmask_rows, rmask, rmask_rows));
}

int eesen_b200_net_dims(const eesen_b200_net *n, int *in_dim, int *out_dim, int *num_layers, int64_t *num_params) {
  if (!n) return EESEN_B200_EINVAL;
  if (in_dim) *in_dim = n->net.InputDim();
  if (out_dim) *out_dim = n->net.OutputDim();
  if (num_layers) *num_layers = n->net.NumLayers();
  if (num_params) *num_params = n->net.NumParams();
  return 0;
}

int eesen_b200_net_train_step(eesen_b200_net *n, const float *feats, int T, int S, const int *frames,
                              const int *labels, const int *lab_len, int train, double stats[4]) {
  if (!n || !feats || !frames || !labels || !lab_len || T <= 0 || S <= 0) return EESEN_B200_EINVAL;
  try {
    static const bool trace = getenv("EESEN_B200_TRACE") != nullptr;
    auto t0 = std::chrono::steady_clock::now();
    unpack_labels(n, S, frames, labels, lab_len);
    const int I = n->net.InputDim();
    size_t elems = (size_t)T * S * I;
    const float *src = stage_feats(n, feats, elems);
    auto t1 = std::chrono::steady_clock::now();
    n->feats.Resize(T * S, I, kUndefined);
    n->feats.CopyFromHost(src, I);
    run_step(n, n->feats, train);
    auto t2 = std::chrono::steady_clock::now();
    double st[4];
    n->ctc.Finish(st);
    auto t3 = std::chrono::steady_clock::now();
    if (trace) {
      auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return (long)std::chrono::duration_cast<std::chrono::microseconds>(b - a).count();
      };
      fprintf(stderr, "[eesen_b200 trace] stage-to-pinned %ld us, enqueue %ld us, wait+stats %ld us\n", us(t0, t1),
              us(t1, t2), us(t2, t3));
    }
    if (stats) memcpy(stats, st, sizeof(st));
    return 0;
  } catch (const std::exception &e) {
    n->ctx->err = e.what();
    return EESEN_B200_EIO;
  }
}

int eesen_b200_net_train_step_device(eesen_b200_net *n, const float *d_feats, int T, int S, const int *frames,
                                     const int *labels, const int *lab_len, int train) {
  if (!n || !d_feats || !frames || !labels || !lab_len || T <= 0 || S <= 0) return EESEN_B200_EINVAL;
  try {
    unpack_labels(n, S, frames, labels, lab_len);
    const int I = n->net.InputDim();
    CuSubMatrix<BaseFloat> in(const_cast<float *>(d_feats), T * S, I, I);
    run_step(n, in, train);
    return 0;
  } catch (const std::exception &e) {
    n->ctx->err = e.what();
    return EESEN_B200_EIO;
  }
}

int eesen_b200_net_train_step_ce(eesen_b200_net *n, const float *feats, int T, int S, const int *frames,
                                 const int *targets, int train, double stats[4]) {
  if (!n || !feats || !frames || !targets || T <= 0 || S <= 0) return EESEN_B200_EINVAL;
  for (int s = 0; s < S; s++)
    if (frames[s] < 0 || frames[s] > T) return n->ctx->fail(EESEN_B200_EINVAL, "frames[s] outside [0, T]");
  try {
    n->S = S;
    n->frames.assign(frames, frames + S);
    n->targets.assign((size_t)T * S, 0);
    size_t off = 0;
    for (int s = 0; s < S; s++)
      for (int t = 0; t < frames[s]; t++) n->targets[(size_t)t * S + s] = targets[off++];
    const int I = n->net.InputDim();
    const float *src = stage_feats(n, feats, (size_t)T * S * I);
    n->feats.Resize(T * S, I, kUndefined);
    n->feats.CopyFromHost(src, I);
    run_step_ce(n, n->feats, nullptr, train);
    n->ce.Finish(stats);
    return 0;
  } catch (const std::exception &e) {
    n->ctx->err = e.what();
    return EESEN_B200_EIO;
  }
}

int eesen_b200_net_train_step_ce_device(eesen_b200_net *n, const float *d_feats, int T, int S, const int *frames,
                                        const int *d_targets, int train) {
  if (!n || !d_feats || !frames || !d_targets || T <= 0 || S <= 0) return EESEN_B200_EINVAL;
  try {
    n->S = S;
    n->frames.assign(frames, frames + S);
    const int I = n->net.InputDim();
    CuSubMatrix<BaseFloat> in(const_cast<float *>(d_feats), T * S, I, I);
    run_step_ce(n, in, d_targets, train);
    return 0;
  } catch (const std::exception &e) {
    n->ctx->err = e.what();
    return EESEN_B200_EIO;
  }
}

int eesen_b200_net_last_loss(const eesen_b200_net *n) { return n && n->last_ce ? 1 : 0; }

int eesen_b200_net_read_stats(eesen_b200_net *n, double stats[4]) {
  if (!n || !stats) return EESEN_B200_EINVAL;
  GUARD(n->ctx, { if (n->last_ce) n->ce.Finish(stats); else n->ctc.Finish(stats); });
}

static int copy_out(const CuMatrixBase<BaseFloat> &m, float *data, int64_t cap, int *rows, int *cols) {
  if (rows) *rows = m.NumRows();
  if (cols) *cols = m.NumCols();
  if (!data) return 0;
  if ((int64_t)m.NumRows() * m.NumCols() > cap) return EESEN_B200_EINVAL;
  m.CopyToHost(data, m.NumCols());
  return 0;
}

int eesen_b200_net_get(eesen_b200_net *n, int which, float *data, int64_t capacity, int *rows, int *cols) {
  if (!n) return EESEN_B200_EINVAL;
  try {
    const int L = n->net.NumLayers();
    if (which >= 0 && which <= L) return copy_out(n->net.PropagateBuffer()[which], data, capacity, rows, cols);
    if (which == 100) return copy_out(n->obj_diff, data, capacity, rows, cols);
    if (which == 101) {
      n->ctc.Finish(NULL);
      const std::vector<float> &p = n->ctc.LastPzx();
      if (rows) *rows = 1;
      if (cols) *cols = (int)p.size();
      if (data) {
        if ((int64_t)p.size() > capacity) return EESEN_B200_EINVAL;
        memcpy(data, p.data(), sizeof(float) * p.size());
      }
      return 0;
    }
    if (which == 102) {
      n->want_in_diff = true;  // takes effect from the next step
      return copy_out(n->in_diff, data, capacity, rows, cols);
    }
    if (which >= 300 && which < 500) {
      const int layer = which >= 400 ? which - 400 : which - 300;
      if (layer >= L) return EESEN_B200_EINVAL;
      BiLstmParallel *bl = dynamic_cast<BiLstmParallel *>(n->net.GetLayer(layer));
      if (!bl) return EESEN_B200_EINVAL;
      return copy_out(which >= 400 ? bl->RecurrentMask() : bl->ForwardMask(), data, capacity, rows, cols);
    }
    if (which == 203 && !n->net.Accu()) {
      if (rows) *rows = 1;
      if (cols) *cols = (int)n->net.NumParams();
      if (data) {
        if (n->net.NumParams() > capacity) return EESEN_B200_EINVAL;
        memset(data, 0, sizeof(float) * n->net.NumParams());
      }
      return 0;
    }
    if (which >= 200 && which <= 203) {
      if (rows) *rows = 1;
      if (cols) *cols = (int)n->net.NumParams();
      if (data) {
        if (n->net.NumParams() > capacity) return EESEN_B200_EINVAL;
        std::vector<float> h;
        n->net.GetArena(which == 200 ? n->net.Params() : which == 201 ? n->net.Corr() : which == 202 ? n->net.Grads()
                                                                                                      : n->net.Accu(), &h);
        memcpy(data, h.data(), sizeof(float) * h.size());
      }
      return 0;
    }
    return EESEN_B200_EINVAL;
  } catch (const std::exception &e) {
    n->ctx->err = e.what();
    return EESEN_B200_EIO;
  }
}

int eesen_b200_net_set_params(eesen_b200_net *n, const float *flat, int64_t cnt) {
  if (!n || !flat) return EESEN_B200_EINVAL;
  GUARD(n->ctx, n->net.SetParams(flat, cnt));
}

}  // extern "C"
