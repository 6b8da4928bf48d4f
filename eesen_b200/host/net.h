// eesen_b200/host/net.h -- host mirror of the reference's Net / Layer / Ctc API for the hot path.
//
// Same class and method names, argument meaning and error behaviour as the reference
// (src/net/net.h:37-176, layer.h:43-217, trainable-layer.h:44-62, bilstm-parallel-layer.h:31-44,
//  affine-trans-layer.h, softmax-layer.h, ctc-loss.h:29-86, gpucompute/cuda-matrix.h) so that
// src/netbin/train-ctc-parallel.cc reads unchanged against it (see train-ctc-parallel.cc here).
// All compute goes through the C ABI (include/eesen_b200.h); errors surface as std::runtime_error
// via KALDI_ERR.  Differences that are deliberate and documented in DESIGN.md:
//   * parameters, raw gradients and momentum buffers of ALL layers live in three contiguous device
//     arenas owned by Net (model-file order) so that one NCCL all-reduce and one fused update cover
//     the whole model; the update runs once at the end of Net::Backpropagate instead of layer by
//     layer (net.cc:98-105) -- equivalent because each layer's back-propagation reads only its own
//     weights;
//   * CuMatrix rows are 16-byte aligned (stride = cols rounded up to 4) instead of cudaMallocPitch.
#ifndef EESEN_B200_HOST_NET_H_
#define EESEN_B200_HOST_NET_H_

#include <memory>
#include <string>
#include <vector>

#include "../../include/eesen_b200.h"
#include "base.h"

namespace eesen {

void CheckAbi(eesen_b200_ctx *ctx, int rc, const char *what);  // non-zero -> KALDI_ERR (throws)

// Device matrix (reference CuMatrix/CuSubMatrix, gpucompute/cuda-matrix.h:40-447), fp32 only.
template <typename Real>
class CuMatrixBase {
 public:
  int32 NumRows() const { return num_rows_; }
  int32 NumCols() const { return num_cols_; }
  int32 Stride() const { return stride_; }
  const Real *Data() const { return data_; }
  Real *Data() { return data_; }
  void SetZero();
  void CopyFromMat(const CuMatrixBase<Real> &src);
  void CopyFromHost(const Real *src, int32 ld);
  void CopyToHost(Real *dst, int32 ld) const;
  void ApplyLog();                                                   // cuda-matrix.h ApplyLog
  void AddVecToRows(Real alpha, const Real *d_vec, int32 dim);       // cuda-matrix.h AddVecToRows (device vector)

 protected:
  CuMatrixBase() {}
  Real *data_ = nullptr;
  int32 num_rows_ = 0, num_cols_ = 0, stride_ = 0;
};

enum MatrixResizeType { kSetZero, kUndefined };

template <typename Real>
class CuMatrix : public CuMatrixBase<Real> {
 public:
  CuMatrix() {}
  CuMatrix(int32 rows, int32 cols, MatrixResizeType t = kSetZero) { Resize(rows, cols, t); }
  explicit CuMatrix(const HostMatrix &m);  // H2D copy, as CuMatrix<BaseFloat>(feat_mat_host)
  CuMatrix(const CuMatrix<Real> &o);
  CuMatrix<Real> &operator=(const CuMatrixBase<Real> &o);
  CuMatrix<Real> &operator=(const CuMatrix<Real> &o);
  ~CuMatrix();
  void Resize(int32 rows, int32 cols, MatrixResizeType t = kSetZero);

 private:
  size_t capacity_ = 0;  // floats
};

// Non-owning view (reference CuSubMatrix)
template <typename Real>
class CuSubMatrix : public CuMatrixBase<Real> {
 public:
  CuSubMatrix(Real *data, int32 rows, int32 cols, int32 stride) {
    this->data_ = data; this->num_rows_ = rows; this->num_cols_ = cols; this->stride_ = stride;
  }
};

// train-opts.h:29-51
struct NetTrainOptions {
  BaseFloat learn_rate = 0.008f, momentum = 0.0f, adagrad_epsilon = 1e-6f, rmsprop_rho = 0.9f,
            rmsprop_one_minus_rho = 0.1f;
};

class Net;

class Layer {
 public:
  enum LayerType { l_Unknown, l_BiLstm_Parallel, l_BiLstm, l_Lstm_Parallel, l_Lstm, l_Affine_Transform, l_Softmax };
  Layer(int32 in, int32 out) : input_dim_(in), output_dim_(out) {}
  virtual ~Layer() {}
  virtual LayerType GetType() const = 0;
  virtual bool IsTrainable() const { return false; }
  int32 InputDim() const { return input_dim_; }
  int32 OutputDim() const { return output_dim_; }
  virtual void SetSeqLengths(std::vector<int> &) {}
  virtual void SetTrainMode() {}   // layer.h:93-94
  virtual void SetTestMode() {}
  // layer.h:184-217
  void Propagate(const CuMatrixBase<BaseFloat> &in, CuMatrix<BaseFloat> *out);
  void Backpropagate(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                     const CuMatrixBase<BaseFloat> &out_diff, CuMatrix<BaseFloat> *in_diff);
  static Layer *Read(std::istream &is, bool binary);            // layer.cc:138-176
  void Write(std::ostream &os, bool binary) const;              // layer.cc:209-222
  void WriteNonParal(std::ostream &os, bool binary) const;      // layer.cc:224-237
  virtual LayerType GetTypeNonParal() const { return GetType(); }
  static bool IsLstmType(LayerType t) {   // layer.h:177-182
    return t == l_BiLstm_Parallel || t == l_BiLstm || t == l_Lstm_Parallel || t == l_Lstm;
  }
  static const char *TypeToMarker(LayerType t);
  static LayerType MarkerToType(const std::string &s);
  virtual std::string Info() const { return ""; }

 protected:
  friend class Net;
  virtual void PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out) = 0;
  virtual void BackpropagateFnc(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                                const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff) = 0;
  virtual void ReadData(std::istream &, bool) {}
  virtual void WriteData(std::ostream &, bool) const {}
  int32 input_dim_, output_dim_;
  eesen_b200_ctx *ctx_ = nullptr;
  bool need_in_diff_ = true;  // false for the first layer when Backpropagate(.., NULL)
};

class TrainableLayer : public Layer {
 public:
  TrainableLayer(int32 in, int32 out) : Layer(in, out) {}
  bool IsTrainable() const { return true; }
  virtual int64 NumParams() const = 0;
  BaseFloat learn_rate_coef_ = 1.0f, max_grad_ = 0.0f;

 protected:
  friend class Net;
  // host staging of the parameters between ReadData and Net::BindArena / for WriteData
  std::vector<float> host_params_;
  // Adagrad/RMSProp accumulators (<BiLstmAccus>/<AffineAccus>), same tensor order as host_params_;
  // has_accu_ mirrors the reference's adaBuffersInitialized (bilstm-layer.h:375-395,458-475)
  std::vector<float> host_accu_;
  bool has_accu_ = false;
  float *w_ = nullptr, *g_ = nullptr;  // this layer's block of the Net arenas (device)
  virtual void Bind(float *w, float *g) { w_ = w; g_ = g; }
};

// bilstm-layer.h + bilstm-parallel-layer.h (vanilla, no dropout)
class BiLstmParallel : public TrainableLayer {
 public:
  BiLstmParallel(int32 in, int32 out) : TrainableLayer(in, out), cell_dim_(out / 2) {}
  LayerType GetType() const { return l_BiLstm_Parallel; }
  LayerType GetTypeNonParal() const { return l_BiLstm; }
  void SetSeqLengths(std::vector<int> &sequence_lengths);
  int64 NumParams() const;
  std::string Info() const;
  void SetTrainMode() { in_train_ = true; }    // bilstm-layer.h:49-55: impacts dropout only
  void SetTestMode() { in_train_ = false; }
  // bilstm-layer.h:62-135 (same consistency checks, same errors)
  void ChangeDropoutParameters(BaseFloat forward_dropout, bool fw_step, bool fw_sequence, bool rnndrop, bool no_mem_loss,
                               BaseFloat recurrent_dropout, bool rec_step, bool rec_sequence, bool twiddle_forward);
  // Masks.  By default they are drawn on the device from (seed, layer stream, draw counter); tests inject the
  // masks the reference drew.  Injected masks stay in force until cleared (NULL / empty).
  void SetDropoutSeed(uint64_t seed, uint64_t stream) { drop_seed_ = seed; drop_stream_ = stream; drop_draws_ = 0; }
  void InjectDropoutMasks(const float *fmask, int32 frows, const float *rmask, int32 rrows);
  const CuMatrix<BaseFloat> &ForwardMask() const { return fmask_; }
  const CuMatrix<BaseFloat> &RecurrentMask() const { return rmask_; }

 protected:
  void PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out);
  void BackpropagateFnc(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                        const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff);
  void ReadData(std::istream &is, bool binary);
  void WriteData(std::ostream &os, bool binary) const;
  void Params(eesen_b200_bilstm_params *p, eesen_b200_bilstm_grads *g) const;
  void ReadDirections(std::istream &is, bool binary, std::vector<float> *flat) const;
  void WriteDirections(std::ostream &os, bool binary, const std::vector<float> &flat) const;
  int32 cell_dim_;
  std::vector<int> sequence_lengths_;
  int *d_len_ = nullptr;
  int32 d_len_cap_ = 0;
  CuMatrix<BaseFloat> gates_, cell_, dgates_;  // propagate_buf_{fw,bw}_ / backpropagate_buf_{fw,bw}_
  // dropout options (bilstm-layer.h:1040-1056); flags_: ForwardTimeStepDropout, ForwardSequenceDropout,
  // RecurrentTimeStepDropout, RecurrentSequenceDropout, RNNDrop, NoMemLossDropout, TwiddleForward
  BaseFloat forward_dropout_ = 0.f, recurrent_dropout_ = 0.f;
  bool flags_[7] = {false, false, false, false, false, false, false};
  bool in_train_ = true;
  bool apply_fwd_ = false, apply_rec_ = false;       // decided by the last Propagate (:389-390)
  CuMatrix<BaseFloat> fmask_, rmask_, m_, dout_;    // masks, un-masked output m, masked out_diff
  std::vector<float> inj_fmask_, inj_rmask_;
  int32 inj_frows_ = 0, inj_rrows_ = 0;
  uint64_t drop_seed_ = 0x5eed5eedULL, drop_stream_ = 0, drop_draws_ = 0;
  void PrepareMask(CuMatrix<BaseFloat> *mask, int32 rows, BaseFloat p, bool per_col, const std::vector<float> &inj,
                   int32 inj_rows);

 public:
  ~BiLstmParallel();
};

// <BiLstm> (bilstm-layer.h:547-700): the marker format-to-nonparallel writes for decoding.  Same
// parameters and arithmetic; without SetSeqLengths the whole input is ONE sequence (what the
// reference's BiLstm::PropagateFnc does), with SetSeqLengths it runs packed like the parallel layer
// (valid frames do not depend on the packing, SURVEY.md section 7 hard part 2).
class BiLstm : public BiLstmParallel {
 public:
  BiLstm(int32 in, int32 out) : BiLstmParallel(in, out) {}
  LayerType GetType() const { return l_BiLstm; }

 protected:
  void PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out);
  void BackpropagateFnc(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                        const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff);
};

// lstm-layer.h + lstm-parallel-layer.h: the uni-directional layer (<CellDim> = output dim = cells).
// nonparallel_ = true is the <Lstm> marker; like <BiLstm> it treats the input as ONE sequence when no
// lengths were set (lstm-layer.h PropagateFnc) -- lengths only give the packing (S), nothing is masked.
class LstmParallel : public TrainableLayer {
 public:
  LstmParallel(int32 in, int32 out, bool nonparallel = false)
      : TrainableLayer(in, out), cell_dim_(out), nonparallel_(nonparallel) {}
  LayerType GetType() const { return nonparallel_ ? l_Lstm : l_Lstm_Parallel; }
  LayerType GetTypeNonParal() const { return l_Lstm; }
  void SetSeqLengths(std::vector<int> &sequence_lengths) { num_streams_ = (int32)sequence_lengths.size(); }
  int64 NumParams() const { int64 C = cell_dim_, I = input_dim_; return 4 * C * I + 4 * C * C + 4 * C + 3 * C; }
  std::string Info() const;

 protected:
  void PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out);
  void BackpropagateFnc(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                        const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff);
  void ReadData(std::istream &is, bool binary);
  void WriteData(std::ostream &os, bool binary) const;
  void Params(eesen_b200_bilstm_params *p, eesen_b200_bilstm_grads *g) const;
  int32 Streams(int32 rows) const;
  int32 cell_dim_;
  bool nonparallel_;
  int32 num_streams_ = 0;
  CuMatrix<BaseFloat> gates_, cell_, dgates_;
};

class AffineTransform : public TrainableLayer {
 public:
  AffineTransform(int32 in, int32 out) : TrainableLayer(in, out) {}
  LayerType GetType() const { return l_Affine_Transform; }
  int64 NumParams() const { return (int64)output_dim_ * input_dim_ + output_dim_; }

 protected:
  void PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out);
  void BackpropagateFnc(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                        const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff);
  void ReadData(std::istream &is, bool binary);
  void WriteData(std::ostream &os, bool binary) const;
};

class Softmax : public Layer {
 public:
  Softmax(int32 in, int32 out) : Layer(in, out) {}
  LayerType GetType() const { return l_Softmax; }

 protected:
  void PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out);
  void BackpropagateFnc(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                        const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff);
};

class Net {
 public:
  explicit Net(eesen_b200_ctx *ctx) : ctx_(ctx) {}
  ~Net();
  void Read(const std::string &file);                    // net.cc:248-297
  void Read(std::istream &is, bool binary);
  void Write(const std::string &file, bool binary);      // net.cc:319-334
  void Write(std::ostream &os, bool binary);
  void WriteNonParal(const std::string &file, bool binary);   // net.cc:337-353
  // forward only, two ping-pong buffers that are released afterwards (net.cc:110-137)
  void Feedforward(const CuMatrixBase<BaseFloat> &in, CuMatrix<BaseFloat> *out);
  void Propagate(const CuMatrixBase<BaseFloat> &in, CuMatrix<BaseFloat> *out);       // net.cc:67-86
  void Backpropagate(const CuMatrixBase<BaseFloat> &out_diff, CuMatrix<BaseFloat> *in_diff);  // net.cc:88-108
  // Data-parallel step that tolerates ranks running out of data: a rank without a minibatch passes
  // out_diff == NULL, contributes a zero gradient and still takes part in the all-reduce and the
  // (identical) update.  Returns how many ranks had a minibatch this step (0: everybody is done).
  // Replaces the done-file handshake of the reference (src/net/communicator.h:57-71,107-113).
  int32 BackpropagateShared(const CuMatrixBase<BaseFloat> *out_diff);
  void SetSeqLengths(std::vector<int> &sequence_lengths);                            // net.h:157-161
  void Check() const;                                    // net.cc:448-468 (dims + NaN/Inf in the parameters)
  void SetTrainOptions(const NetTrainOptions &opts);
  const NetTrainOptions &GetTrainOptions() const { return opts_; }
  void SetUpdateAlgorithm(const std::string &opt);       // SGD | Adagrad | RMSProp (net.cc:481-496)
  int UpdateAlgorithm() const { return update_algorithm_; }
  void SetTrainMode();    // net.cc:396-412: also tells the layers (dropout is a train-mode thing)
  void SetTestMode();
  void ChangeDropoutParameters(BaseFloat forward_dropout, bool fw_step, bool fw_sequence, bool rnndrop, bool no_mem_loss,
                               BaseFloat recurrent_dropout, bool rec_step, bool rec_sequence, bool twiddle_forward);   // net.cc:414-434
  void SetDropoutSeed(uint64_t seed);
  Layer *GetLayer(int32 i) { return layers_[i]; }
  int32 InputDim() const;
  int32 OutputDim() const;
  int32 NumLayers() const { return (int32)layers_.size(); }
  int64 NumParams() const { return num_params_; }
  std::string Info() const;
  std::string InfoGradient() const;
  const std::vector<CuMatrix<BaseFloat> > &PropagateBuffer() const { return propagate_buf_; }
  const std::vector<CuMatrix<BaseFloat> > &BackpropagateBuffer() const { return backpropagate_buf_; }
  // arenas (device), model-file order
  float *Params() { return w_; }
  float *Grads() { return g_; }
  float *Corr() { return corr_; }
  float *Accu() { return accu_; }   // NULL until an accumulator was read or an adaptive update ran
  void GetParams(std::vector<float> *host) const;
  void GetArena(const float *arena, std::vector<float> *host) const;  // packs one arena in model-file order
  void SetParams(const float *host, int64 n);
  int64 ArenaSize() const { return arena_size_; }
  eesen_b200_ctx *Context() { return ctx_; }

 private:
  void BindArena();
  void RefreshHostCopies();
  void UploadSegments();
  void BackpropagateLayers(const CuMatrixBase<BaseFloat> *out_diff, CuMatrix<BaseFloat> *in_diff);
  void Update();
  eesen_b200_ctx *ctx_;
  std::vector<Layer *> layers_;
  std::vector<CuMatrix<BaseFloat> > propagate_buf_, backpropagate_buf_;
  NetTrainOptions opts_;
  bool in_train_ = true;
  int64 num_params_ = 0, arena_size_ = 0;
  std::vector<int64> layer_offset_;  // arena offset of each layer's block (-1: not trainable)
  float *w_ = nullptr, *g_ = nullptr, *corr_ = nullptr;
  float *accu_ = nullptr;
  void EnsureAccu(bool mark_all_layers);
  int update_algorithm_ = 0;  // 0 sgd_update, 1 adagrad_update, 2 rmsprop_update (trainable-layer.h:34-38)
  void *d_segs_ = nullptr;
  int nseg_ = 0;
  bool segs_dirty_ = true;
};

// class-prior.h:29-73, class-prior.cc:28-90
struct ClassPriorOptions {
  std::string class_frame_counts;
  BaseFloat prior_scale = 1.0f, prior_cutoff = 1e-10f, blank_scale = 1.0f;
};
class ClassPrior {
 public:
  ClassPrior(eesen_b200_ctx *ctx, const ClassPriorOptions &opts);
  ~ClassPrior();
  void SubtractOnLogpost(CuMatrixBase<BaseFloat> *llk);
  // the host arithmetic of the constructor: counts -> log priors (+FLT_MAX/2 where count < cutoff)
  static void LogPriors(const std::vector<double> &counts, BaseFloat prior_cutoff, BaseFloat blank_scale,
                        std::vector<float> *log_priors);
  int32 Dim() const { return dim_; }
  const float *DeviceLogPriors() const { return d_log_priors_; }
  BaseFloat PriorScale() const { return prior_scale_; }

 private:
  eesen_b200_ctx *ctx_;
  BaseFloat prior_scale_;
  float *d_log_priors_ = nullptr;
  int32 dim_ = 0;
};

// ctc-loss.h:29-86
class Ctc {
 public:
  explicit Ctc(eesen_b200_ctx *ctx);
  ~Ctc();
  void EvalParallel(const std::vector<int32> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                    std::vector<std::vector<int32> > &label, CuMatrix<BaseFloat> *diff);
  void ErrorRateMSeq(const std::vector<int> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                     std::vector<std::vector<int> > &label, std::string &out);
  void SetReportStep(int32 report_step) { report_step_ = report_step; }
  std::string Report();
  float NumErrorTokens() { Finish(NULL); return error_num_; }
  int32 NumRefTokens() { Finish(NULL); return ref_num_; }
  // asynchronous halves used by the device-resident step (statistics are folded in by Finish())
  void EvalParallelAsync(const std::vector<int32> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                         std::vector<std::vector<int32> > &label, CuMatrix<BaseFloat> *diff);
  void ErrorRateMSeqAsync(const std::vector<int> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                          std::vector<std::vector<int> > &label);
  void Finish(double stats[4]);  // waits, folds pzx / argmax into the registries
  const std::vector<float> &LastPzx() const { return pzx_host_; }
  const float *DevicePzx() const { return d_pzx_; }

 private:
  void Upload(const std::vector<int32> &frame_num_utt, std::vector<std::vector<int32> > &label, int32 num_classes);
  eesen_b200_ctx *ctx_;
  int32 frames_ = 0, sequences_num_ = 0, ref_num_ = 0;
  float error_num_ = 0;
  int32 frames_progress_ = 0, ref_num_progress_ = 0;
  float error_num_progress_ = 0;
  int32 sequences_progress_ = 0;
  double obj_progress_ = 0;
  int32 report_step_ = 100;
  // device staging
  int *d_len_ = nullptr, *d_lab_ = nullptr, *d_lablen_ = nullptr, *d_argmax_ = nullptr;
  float *d_pzx_ = nullptr;
  size_t cap_len_ = 0, cap_lab_ = 0, cap_arg_ = 0;
  int *h_argmax_ = nullptr;  // pinned
  float *h_pzx_ = nullptr;   // pinned
  size_t cap_harg_ = 0, cap_hpzx_ = 0;
  std::vector<float> pzx_host_;
  // pending async state
  bool pending_eval_ = false, pending_err_ = false;
  std::vector<int32> p_frames_;
  std::vector<std::vector<int32> > p_labels_;
  int32 p_S_ = 0, p_rows_ = 0;
  int32 max_lab_ = 1;
};

// ce-loss.h:32-86, the parallel half.  The rows valid in the mask are t < frame_num_utt[s] (no float mask); the
// statistics of each call stay on the device and are folded, in call order, at the next Finish() -- with the
// reference's progress lines -- so that a training loop never waits for the device per minibatch.
// Deliberate differences (DESIGN.md section 5): 64-bit counters, Report() prints the real quotient, the
// objective reads the target column only.
class CE {
 public:
  explicit CE(eesen_b200_ctx *ctx);
  ~CE();
  // target: [T*S] packed like the rows of net_out; entries of padded rows are ignored, the others must lie in [0, K)
  void EvalParallel(const std::vector<int32> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                    const std::vector<int32> &target, CuMatrix<BaseFloat> *diff);
  // the same with the packed targets already on the device (validated by the caller)
  void EvalParallelAsync(const std::vector<int32> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                         const int32 *d_target, CuMatrix<BaseFloat> *diff);
  void SetReportStep(int32 report_step) { report_step_ = report_step; }
  std::string Report();
  // waits, folds every pending call; stats (may be NULL) of the last call: obj, correct, valid frames, padded rows
  void Finish(double stats[4]);

 private:
  eesen_b200_ctx *ctx_;
  int64 frames_ = 0, sequences_num_ = 0, correct_ = 0;
  double obj_ = 0;
  int64 frames_progress_ = 0, sequences_progress_ = 0, correct_progress_ = 0;
  double obj_progress_ = 0;
  int32 report_step_ = 100;
  int *d_len_ = nullptr;         // [S] lengths, then [T*S] targets (host-target calls)
  size_t cap_len_ = 0;
  double *d_stats_ = nullptr;    // [kSlots][3] one slot per pending call
  double *h_stats_ = nullptr;    // pinned mirror
  static const int kSlots = 64;
  struct Pending { int32 S, rows; };
  std::vector<Pending> pending_;
  double last_[4] = {0, 0, 0, 0};
};

}  // namespace eesen
#endif
