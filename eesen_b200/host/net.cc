// eesen_b200/host/net.cc -- see net.h.
#include "net.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <fstream>
#include <random>

#include "context.h"

namespace eesen {

static eesen_b200_ctx *g_ctx = nullptr;  // the process-wide device context (reference: CuDevice singleton)
static cudaStream_t Stream() { return g_ctx ? g_ctx->stream : (cudaStream_t)0; }
// host-visible results need BOTH streams drained (the weight-gradient products run on the side stream)
static cudaError_t SyncStream() {
  if (g_ctx) g_ctx->join_side();
  return cudaStreamSynchronize(Stream());
}

#define CU_CHECK(call)                                                                  \
  do {                                                                                  \
    cudaError_t e__ = (call);                                                           \
    if (e__ != cudaSuccess) KALDI_ERR << "CUDA error: " << cudaGetErrorString(e__) << " in " #call; \
  } while (0)

void CheckAbi(eesen_b200_ctx *ctx, int rc, const char *what) {
  if (rc != 0) KALDI_ERR << what << " failed (code " << rc << "): " << eesen_b200_last_error(ctx);
}

// ------------------------------------------------------------------------------------ CuMatrix
template <typename Real>
void CuMatrixBase<Real>::SetZero() {
  if (num_rows_ == 0) return;
  CU_CHECK(cudaMemsetAsync(data_, 0, sizeof(Real) * (size_t)num_rows_ * stride_, Stream()));
}
template <typename Real>
void CuMatrixBase<Real>::CopyFromMat(const CuMatrixBase<Real> &src) {
  KALDI_ASSERT(src.NumRows() == num_rows_ && src.NumCols() == num_cols_);
  if (num_rows_ == 0) return;
  if (stride_ == src.Stride()) {   // same pitch on both sides (padding columns included): one flat copy
    CU_CHECK(cudaMemcpyAsync(data_, src.Data(), sizeof(Real) * (size_t)num_rows_ * stride_,
                             cudaMemcpyDeviceToDevice, Stream()));
    return;
  }
  CU_CHECK(cudaMemcpy2DAsync(data_, sizeof(Real) * stride_, src.Data(), sizeof(Real) * src.Stride(),
                             sizeof(Real) * num_cols_, num_rows_, cudaMemcpyDeviceToDevice, Stream()));
}
template <typename Real>
void CuMatrixBase<Real>::CopyFromHost(const Real *src, int32 ld) {
  if (num_rows_ == 0) return;
  if (stride_ == num_cols_ && ld == num_cols_) {
    CU_CHECK(cudaMemcpyAsync(data_, src, sizeof(Real) * (size_t)num_rows_ * num_cols_, cudaMemcpyHostToDevice, Stream()));
    return;
  }
  CU_CHECK(cudaMemcpy2DAsync(data_, sizeof(Real) * stride_, src, sizeof(Real) * ld, sizeof(Real) * num_cols_,
                             num_rows_, cudaMemcpyHostToDevice, Stream()));
}
template <typename Real>
void CuMatrixBase<Real>::CopyToHost(Real *dst, int32 ld) const {
  if (num_rows_ == 0) return;
  if (stride_ == num_cols_ && ld == num_cols_) {
    CU_CHECK(cudaMemcpyAsync(dst, data_, sizeof(Real) * (size_t)num_rows_ * num_cols_, cudaMemcpyDeviceToHost, Stream()));
    CU_CHECK(SyncStream());
    return;
  }
  CU_CHECK(cudaMemcpy2DAsync(dst, sizeof(Real) * ld, data_, sizeof(Real) * stride_, sizeof(Real) * num_cols_,
                             num_rows_, cudaMemcpyDeviceToHost, Stream()));
  CU_CHECK(SyncStream());
}

template <typename Real>
void CuMatrix<Real>::Resize(int32 rows, int32 cols, MatrixResizeType t) {
  int32 stride = (cols + 3) & ~3;
  size_t need = (size_t)rows * stride;
  if (need > capacity_) {
    if (this->data_) {
      CU_CHECK(SyncStream());
      CU_CHECK(cudaFree(this->data_));
      this->data_ = nullptr;
    }
    CU_CHECK(cudaMalloc((void **)&this->data_, sizeof(Real) * need));
    capacity_ = need;
  }
  this->num_rows_ = rows; this->num_cols_ = cols; this->stride_ = stride;
  if (t == kSetZero) this->SetZero();
}
template <typename Real>
CuMatrix<Real>::CuMatrix(const HostMatrix &m) {
  Resize(m.rows, m.cols, kUndefined);
  this->CopyFromHost(m.data.data(), m.cols);
}
template <typename Real>
CuMatrix<Real>::CuMatrix(const CuMatrix<Real> &o) : CuMatrixBase<Real>() {
  Resize(o.NumRows(), o.NumCols(), kUndefined);
  this->CopyFromMat(o);
}
template <typename Real>
CuMatrix<Real> &CuMatrix<Real>::operator=(const CuMatrixBase<Real> &o) {
  if (&o == this) return *this;
  Resize(o.NumRows(), o.NumCols(), kUndefined);
  this->CopyFromMat(o);
  return *this;
}
template <typename Real>
CuMatrix<Real> &CuMatrix<Real>::operator=(const CuMatrix<Real> &o) {
  return *this = static_cast<const CuMatrixBase<Real> &>(o);
}
template <typename Real>
CuMatrix<Real>::~CuMatrix() {
  if (this->data_) cudaFree(this->data_);
}
template <typename Real>
void CuMatrixBase<Real>::ApplyLog() {
  CheckAbi(g_ctx, eesen_b200_loglik(g_ctx, num_rows_, num_cols_, data_, stride_, 1, NULL, 0.f), "eesen_b200_loglik");
}
template <typename Real>
void CuMatrixBase<Real>::AddVecToRows(Real alpha, const Real *d_vec, int32 dim) {
  KALDI_ASSERT(dim == num_cols_);
  // y += alpha * vec  ==  y -= (-alpha) * vec
  CheckAbi(g_ctx, eesen_b200_loglik(g_ctx, num_rows_, num_cols_, data_, stride_, 0, d_vec, -alpha), "eesen_b200_loglik");
}
template class CuMatrixBase<float>;
template class CuMatrix<float>;

// ------------------------------------------------------------------------------------ Layer
const char *Layer::TypeToMarker(LayerType t) {
  switch (t) {
    case l_BiLstm_Parallel: return "<BiLstmParallel>";
    case l_BiLstm: return "<BiLstm>";
    case l_Lstm_Parallel: return "<LstmParallel>";
    case l_Lstm: return "<Lstm>";
    case l_Affine_Transform: return "<AffineTransform>";
    case l_Softmax: return "<Softmax>";
    default: return "<Unknown>";
  }
}
Layer::LayerType Layer::MarkerToType(const std::string &s) {
  if (s == "<BiLstmParallel>") return l_BiLstm_Parallel;
  if (s == "<BiLstm>") return l_BiLstm;
  if (s == "<LstmParallel>") return l_Lstm_Parallel;
  if (s == "<Lstm>") return l_Lstm;
  if (s == "<AffineTransform>") return l_Affine_Transform;
  if (s == "<Softmax>") return l_Softmax;
  KALDI_ERR << "Unknown or unsupported layer marker on the B200 CTC path: " << s
            << " (supported: <BiLstmParallel> <BiLstm> <LstmParallel> <Lstm> <AffineTransform> <Softmax>)";
  return l_Unknown;
}

void Layer::Propagate(const CuMatrixBase<BaseFloat> &in, CuMatrix<BaseFloat> *out) {
  if (input_dim_ != in.NumCols())
    KALDI_ERR << "Non-matching dims! " << TypeToMarker(GetType()) << " input-dim : " << input_dim_
              << " data : " << in.NumCols();
  out->Resize(in.NumRows(), output_dim_, kUndefined);  // every kernel overwrites its full output
  PropagateFnc(in, out);
}

void Layer::Backpropagate(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                          const CuMatrixBase<BaseFloat> &out_diff, CuMatrix<BaseFloat> *in_diff) {
  if (output_dim_ != out_diff.NumCols())
    KALDI_ERR << "Non-matching output dims, component:" << output_dim_ << " data:" << out_diff.NumCols();
  in_diff->Resize(out_diff.NumRows(), input_dim_, kUndefined);
  KALDI_ASSERT(in.NumRows() == out.NumRows() && in.NumRows() == out_diff.NumRows());
  BackpropagateFnc(in, out, out_diff, in_diff);
}

Layer *Layer::Read(std::istream &is, bool binary) {
  int32 dim_out, dim_in;
  std::string token;
  int first_char = Peek(is, binary);
  if (first_char == EOF) return NULL;
  ReadToken(is, binary, &token);
  if (token == "</Nnet>") return NULL;
  if (token == "<Nnet>") ReadToken(is, binary, &token);
  LayerType type = MarkerToType(token);
  ExpectToken(is, binary, "<InputDim>");
  ReadBasicType(is, binary, &dim_in);
  ExpectToken(is, binary, IsLstmType(type) ? "<CellDim>" : "<OutputDim>");
  ReadBasicType(is, binary, &dim_out);
  Layer *layer = NULL;
  switch (type) {
    case l_BiLstm_Parallel: layer = new BiLstmParallel(dim_in, dim_out); break;
    case l_BiLstm: layer = new BiLstm(dim_in, dim_out); break;
    case l_Lstm_Parallel: layer = new LstmParallel(dim_in, dim_out, false); break;
    case l_Lstm: layer = new LstmParallel(dim_in, dim_out, true); break;
    case l_Affine_Transform: layer = new AffineTransform(dim_in, dim_out); break;
    case l_Softmax: layer = new Softmax(dim_in, dim_out); break;
    default: KALDI_ERR << "Missing type: " << token;
  }
  layer->ReadData(is, binary);
  return layer;
}

static void WriteLayerAs(const Layer &l, Layer::LayerType t, std::ostream &os, bool binary) {
  WriteToken(os, binary, Layer::TypeToMarker(t));
  WriteToken(os, binary, "<InputDim>");
  WriteBasicType(os, binary, l.InputDim());
  WriteToken(os, binary, Layer::IsLstmType(t) ? "<CellDim>" : "<OutputDim>");
  WriteBasicType(os, binary, l.OutputDim());
  if (!binary) os << "\n";
}
void Layer::Write(std::ostream &os, bool binary) const {
  WriteLayerAs(*this, GetType(), os, binary);
  WriteData(os, binary);
}
void Layer::WriteNonParal(std::ostream &os, bool binary) const {
  WriteLayerAs(*this, GetTypeNonParal(), os, binary);
  WriteData(os, binary);
}

// ------------------------------------------------------------------------------------ BiLstmParallel
static const char *kBiLstmFlagTokens[7] = {"<ForwardTimeStepDropout>", "<ForwardSequenceDropout>",
                                           "<RecurrentTimeStepDropout>", "<RecurrentSequenceDropout>",
                                           "<RNNDrop>", "<NoMemLossDropout>", "<TwiddleForward>"};

int64 BiLstmParallel::NumParams() const {
  int64 C = cell_dim_, I = input_dim_;
  return 2 * (4 * C * I + 4 * C * C + 4 * C + 3 * C);
}

BiLstmParallel::~BiLstmParallel() {
  if (d_len_) cudaFree(d_len_);
}

void BiLstmParallel::ReadData(std::istream &is, bool binary) {
  // optional tokens, in the order of bilstm-layer.h:317-375
  while ('<' == Peek(is, binary)) {
    std::string tok;
    ReadToken(is, binary, &tok);
    if (tok == "<LearnRateCoef>") ReadBasicType(is, binary, &learn_rate_coef_);
    else if (tok == "<MaxGrad>") ReadBasicType(is, binary, &max_grad_);
    else if (tok == "<ForwardDropoutFactor>") ReadBasicType(is, binary, &forward_dropout_);
    else if (tok == "<RecurrentDropoutFactor>") ReadBasicType(is, binary, &recurrent_dropout_);
    else if (tok == "<BiLstmAccus>") {   // bilstm-layer.h:375-395: 12 accumulators, then the weights
      ReadDirections(is, binary, &host_accu_);
      has_accu_ = true;
      break;
    } else {
      int f = -1;
      for (int i = 0; i < 7; i++)
        if (tok == kBiLstmFlagTokens[i]) f = i;
      if (f < 0) KALDI_ERR << "Unknown token " << tok << " in <BiLstmParallel>";
      ReadBasicType(is, binary, &flags_[f]);
    }
  }
  if (flags_[4] && flags_[5]) KALDI_ERR << "Only one of RNNDrop, NoMemLossDropout can be true. Pick one.";
  const int64 C = cell_dim_, I = input_dim_;
  if (C % 8 != 0 || I % 4 != 0)
    KALDI_ERR << "BiLstmParallel on B200 needs cells/direction % 8 == 0 and input dim % 4 == 0, got C=" << C
              << " I=" << I;
  ReadDirections(is, binary, &host_params_);
}

// wx, wm, bias, phole i/f/o for fw then bw (bilstm-layer.h:395-424; the accumulators use the same order :381-393)
void BiLstmParallel::ReadDirections(std::istream &is, bool binary, std::vector<float> *flat) const {
  const int64 C = cell_dim_, I = input_dim_;
  flat->clear();
  flat->reserve(NumParams());
  for (int d = 0; d < 2; d++) {
    HostMatrix wx, wm;
    HostVector b, pi, pf, po;
    wx.Read(is, binary); wm.Read(is, binary);
    b.Read(is, binary); pi.Read(is, binary); pf.Read(is, binary); po.Read(is, binary);
    KALDI_ASSERT(wx.rows == 4 * C && wx.cols == I && wm.rows == 4 * C && wm.cols == C);
    KALDI_ASSERT((int64)b.data.size() == 4 * C && (int64)pi.data.size() == C && (int64)pf.data.size() == C &&
                 (int64)po.data.size() == C);
    flat->insert(flat->end(), wx.data.begin(), wx.data.end());
    flat->insert(flat->end(), wm.data.begin(), wm.data.end());
    flat->insert(flat->end(), b.data.begin(), b.data.end());
    flat->insert(flat->end(), pi.data.begin(), pi.data.end());
    flat->insert(flat->end(), pf.data.begin(), pf.data.end());
    flat->insert(flat->end(), po.data.begin(), po.data.end());
  }
}

void BiLstmParallel::WriteDirections(std::ostream &os, bool binary, const std::vector<float> &flat) const {
  const int64 C = cell_dim_, I = input_dim_;
  const float *p = flat.data();
  for (int d = 0; d < 2; d++) {
    HostMatrix wx, wm;
    wx.rows = 4 * C; wx.cols = I; wx.data.assign(p, p + 4 * C * I); p += 4 * C * I;
    wm.rows = 4 * C; wm.cols = C; wm.data.assign(p, p + 4 * C * C); p += 4 * C * C;
    HostVector b, pi, pf, po;
    b.data.assign(p, p + 4 * C); p += 4 * C;
    pi.data.assign(p, p + C); p += C;
    pf.data.assign(p, p + C); p += C;
    po.data.assign(p, p + C); p += C;
    wx.Write(os, binary); wm.Write(os, binary);
    b.Write(os, binary); pi.Write(os, binary); pf.Write(os, binary); po.Write(os, binary);
  }
}

void BiLstmParallel::WriteData(std::ostream &os, bool binary) const {
  // bilstm-layer.h:429-493
  WriteToken(os, binary, "<LearnRateCoef>"); WriteBasicType(os, binary, learn_rate_coef_);
  WriteToken(os, binary, "<MaxGrad>"); WriteBasicType(os, binary, max_grad_);
  WriteToken(os, binary, "<ForwardDropoutFactor>"); WriteBasicType(os, binary, forward_dropout_);
  for (int i = 0; i < 6; i++) { WriteToken(os, binary, kBiLstmFlagTokens[i]); WriteBasicType(os, binary, flags_[i]); }
  WriteToken(os, binary, "<RecurrentDropoutFactor>"); WriteBasicType(os, binary, recurrent_dropout_);
  WriteToken(os, binary, kBiLstmFlagTokens[6]); WriteBasicType(os, binary, flags_[6]);
  if (has_accu_) {   // bilstm-layer.h:458-475
    WriteToken(os, binary, "<BiLstmAccus>");
    WriteDirections(os, binary, host_accu_);
  }
  WriteDirections(os, binary, host_params_);
}

void BiLstmParallel::Params(eesen_b200_bilstm_params *p, eesen_b200_bilstm_grads *g) const {
  const int64 C = cell_dim_, I = input_dim_;
  if (p) { p->ldwx = 0; p->ldwm = 0; }   // the arena holds the matrices densely
  if (g) { g->ldwx = 0; g->ldwm = 0; }
  const int64 dir_stride = 4 * C * I + 4 * C * C + 4 * C + 3 * C;
  for (int d = 0; d < 2; d++) {
    int64 o = d * dir_stride;
    if (p) {
      p->wx[d] = w_ + o; p->wm[d] = w_ + o + 4 * C * I; p->bias[d] = w_ + o + 4 * C * I + 4 * C * C;
      p->pi[d] = p->bias[d] + 4 * C; p->pf[d] = p->pi[d] + C; p->po[d] = p->pf[d] + C;
    }
    if (g) {
      g->wx[d] = g_ + o; g->wm[d] = g_ + o + 4 * C * I; g->bias[d] = g_ + o + 4 * C * I + 4 * C * C;
      g->pi[d] = g->bias[d] + 4 * C; g->pf[d] = g->pi[d] + C; g->po[d] = g->pf[d] + C;
    }
  }
}

void BiLstmParallel::SetSeqLengths(std::vector<int> &sequence_lengths) {
  sequence_lengths_ = sequence_lengths;
  int32 S = sequence_lengths.size();
  if (S == 0) return;
  if (S > d_len_cap_) {
    if (d_len_) { CU_CHECK(SyncStream()); CU_CHECK(cudaFree(d_len_)); }
    CU_CHECK(cudaMalloc((void **)&d_len_, sizeof(int) * S));
    d_len_cap_ = S;
  }
  CU_CHECK(cudaMemcpyAsync(d_len_, sequence_lengths_.data(), sizeof(int) * S, cudaMemcpyHostToDevice, Stream()));
}

void BiLstmParallel::ChangeDropoutParameters(BaseFloat forward_dropout, bool fw_step, bool fw_sequence, bool rnndrop,
                                             bool no_mem_loss, BaseFloat recurrent_dropout, bool rec_step,
                                             bool rec_sequence, bool twiddle_forward) {
  // bilstm-layer.h:74-112
  if (forward_dropout > 0.0 && !(fw_sequence || fw_step))
    KALDI_ERR << "ForwardDropoutFactor > 0 but ForwardTimeStepDropout and ForwardSequenceDropout are both false, One must be true.";
  if (fw_sequence && fw_step)
    KALDI_ERR << "Both ForwardTimeStepDropout and ForwardSequenceDropout are true, Only one can be true.";
  if (forward_dropout == 0.0 && (fw_sequence || fw_step))
    KALDI_ERR << "ForwardDropoutFactor = 0 but ForwardTimeStepDropout and/or ForwardSequenceDropout is true, both must be false.";
  if (rec_sequence && rec_step)
    KALDI_ERR << "RecurrentSequenceDropout and RecurrentTimeStepDropout cannot be true at the same time. Pick one.";
  if (rnndrop && no_mem_loss) KALDI_ERR << "Only one of RNNDrop, NoMemLossDropout can be true. Pick one.";
  if (recurrent_dropout == 0.0 && (no_mem_loss || rnndrop))
    KALDI_ERR << "RecurrentDropoutFactor must be nonzero if RNNDrop or NoMemLossDropout is true";
  if (!(rec_step || rec_sequence) && (rnndrop || no_mem_loss))
    KALDI_ERR << " Either RecurrentSequenceDropout or RecurrentTimeStepDropout must be true if RNNDrop or NoMemLossDropout is true";
  if (forward_dropout >= 1.0 || recurrent_dropout >= 1.0 || forward_dropout < 0.0 || recurrent_dropout < 0.0)
    KALDI_ERR << "dropout factors must lie in [0, 1)";
  forward_dropout_ = forward_dropout; flags_[0] = fw_step; flags_[1] = fw_sequence; flags_[6] = twiddle_forward;
  recurrent_dropout_ = recurrent_dropout; flags_[2] = rec_step; flags_[3] = rec_sequence;
  flags_[4] = rnndrop; flags_[5] = no_mem_loss;
}

void BiLstmParallel::InjectDropoutMasks(const float *fmask, int32 frows, const float *rmask, int32 rrows) {
  const size_t w = (size_t)2 * cell_dim_;
  if (fmask && frows > 0) { inj_fmask_.assign(fmask, fmask + (size_t)frows * w); inj_frows_ = frows; }
  else { inj_fmask_.clear(); inj_frows_ = 0; }
  if (rmask && rrows > 0) { inj_rmask_.assign(rmask, rmask + (size_t)rrows * w); inj_rrows_ = rrows; }
  else { inj_rmask_.clear(); inj_rrows_ = 0; }
}

// scaled mask [rows x 2C]: the injected one (tests: the masks the reference drew) or a fresh device draw
void BiLstmParallel::PrepareMask(CuMatrix<BaseFloat> *mask, int32 rows, BaseFloat p, bool per_col,
                                 const std::vector<float> &inj, int32 inj_rows) {
  const int32 w = 2 * cell_dim_;
  mask->Resize(rows, w, kUndefined);
  if (!inj.empty()) {
    if (inj_rows != rows) KALDI_ERR << "injected dropout mask has " << inj_rows << " rows, this minibatch needs " << rows;
    mask->CopyFromHost(inj.data(), w);
    CU_CHECK(SyncStream());   // inj may be replaced by the caller right after
    return;
  }
  CheckAbi(ctx_, eesen_b200_dropout_mask(ctx_, rows, w, mask->Data(), mask->Stride(), p, per_col ? 1 : 0, drop_seed_,
                                         (drop_stream_ << 32) + drop_draws_++), "eesen_b200_dropout_mask");
}

void BiLstmParallel::PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out) {
  int32 S = sequence_lengths_.size();
  KALDI_ASSERT(S > 0 && in.NumRows() % S == 0);
  int32 T = in.NumRows() / S, C = cell_dim_;
  const int32 N = in.NumRows();
  gates_.Resize(N, 8 * C, kUndefined);
  cell_.Resize(N, 2 * C, kUndefined);
  eesen_b200_bilstm_params p;
  Params(&p, NULL);
  // which dropout applies to this pass (bilstm-parallel-layer.h:385-390); TwiddleForward picks one of the two
  // at random per minibatch
  const bool has_rec = flags_[4] || flags_[5];
  bool twiddle_fwd = false;
  if (flags_[6]) {
    uint64_t z = drop_seed_ + 0x9e3779b97f4a7c15ULL * (++drop_draws_) + (drop_stream_ << 32);
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL; z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL; z ^= z >> 31;
    twiddle_fwd = (z >> 63) != 0;   // BernoulliDist(0.5)
  }
  apply_rec_ = in_train_ && has_rec && recurrent_dropout_ > 0.f && (!flags_[6] || !twiddle_fwd);
  apply_fwd_ = in_train_ && forward_dropout_ > 0.f && (!flags_[6] || twiddle_fwd);
  if (GetType() == l_BiLstm && (apply_rec_ || apply_fwd_)) KALDI_ERR << "Dropout not implemented on BiLstm";   // bilstm-layer.h:555-556
  float *m_dst = out->Data();
  int32 m_ld = out->Stride();
  if (apply_fwd_) { m_.Resize(N, 2 * C, kUndefined); m_dst = m_.Data(); m_ld = m_.Stride(); }
  if (apply_rec_) {
    PrepareMask(&rmask_, flags_[2] ? N : S, recurrent_dropout_, flags_[3], inj_rmask_, inj_rrows_);
    CheckAbi(ctx_, eesen_b200_bilstm_forward_dropout(ctx_, T, S, input_dim_, C, d_len_, in.Data(), in.Stride(), &p,
                                                     gates_.Data(), cell_.Data(), m_dst, m_ld, flags_[4] ? 2 : 1,
                                                     rmask_.Data(), rmask_.Stride(), flags_[2] ? 1 : 0),
             "eesen_b200_bilstm_forward_dropout");
  } else {
    CheckAbi(ctx_, eesen_b200_bilstm_forward(ctx_, T, S, input_dim_, C, d_len_, in.Data(), in.Stride(), &p,
                                             gates_.Data(), cell_.Data(), m_dst, m_ld),
             "eesen_b200_bilstm_forward");
  }
  if (apply_fwd_) {   // :409-416: the mask hits the layer OUTPUT only; the recurrence saw the un-masked m
    PrepareMask(&fmask_, N, forward_dropout_, flags_[1], inj_fmask_, inj_frows_);
    CheckAbi(ctx_, eesen_b200_mul_elements(ctx_, N, 2 * C, m_.Data(), m_.Stride(), fmask_.Data(), fmask_.Stride(),
                                           out->Data(), out->Stride()), "eesen_b200_mul_elements");
  }
}

void BiLstm::PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out) {
  if (!sequence_lengths_.empty()) { BiLstmParallel::PropagateFnc(in, out); return; }
  std::vector<int> one(1, in.NumRows());   // bilstm-layer.h:548: T = in.NumRows(), a single sequence
  SetSeqLengths(one);
  BiLstmParallel::PropagateFnc(in, out);
  sequence_lengths_.clear();
}
void BiLstm::BackpropagateFnc(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                              const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff) {
  if (!sequence_lengths_.empty()) { BiLstmParallel::BackpropagateFnc(in, out, out_diff, in_diff); return; }
  std::vector<int> one(1, in.NumRows());
  SetSeqLengths(one);
  BiLstmParallel::BackpropagateFnc(in, out, out_diff, in_diff);
  sequence_lengths_.clear();
}

void BiLstmParallel::BackpropagateFnc(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                                      const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff) {
  int32 S = sequence_lengths_.size();
  KALDI_ASSERT(S > 0 && in.NumRows() % S == 0);
  int32 T = in.NumRows() / S, C = cell_dim_;
  const int32 N = in.NumRows();
  dgates_.Resize(N, 8 * C, kUndefined);
  eesen_b200_bilstm_params p;
  eesen_b200_bilstm_grads g;
  Params(&p, &g);
  const float *dout = out_diff.Data(), *m = out.Data();
  int32 ldd = out_diff.Stride(), ldm = out.Stride();
  if (apply_fwd_) {   // :891-895 out_diff_drop = out_diff (.) mask; the Wm gradient pairs DGIFO with the UN-masked m
    dout_.Resize(N, 2 * C, kUndefined);
    CheckAbi(ctx_, eesen_b200_mul_elements(ctx_, N, 2 * C, out_diff.Data(), out_diff.Stride(), fmask_.Data(),
                                           fmask_.Stride(), dout_.Data(), dout_.Stride()), "eesen_b200_mul_elements");
    dout = dout_.Data(); ldd = dout_.Stride();
    m = m_.Data(); ldm = m_.Stride();
  }
  if (apply_rec_) {
    CheckAbi(ctx_, eesen_b200_bilstm_backward_dropout(ctx_, T, S, input_dim_, C, in.Data(), in.Stride(), &p, gates_.Data(),
                                                      cell_.Data(), m, ldm, dout, ldd, dgates_.Data(),
                                                      need_in_diff_ ? in_diff->Data() : NULL, in_diff->Stride(), &g,
                                                      flags_[4] ? 2 : 1, rmask_.Data(), rmask_.Stride(), flags_[2] ? 1 : 0),
             "eesen_b200_bilstm_backward_dropout");
  } else {
    CheckAbi(ctx_, eesen_b200_bilstm_backward(ctx_, T, S, input_dim_, C, in.Data(), in.Stride(), &p, gates_.Data(),
                                              cell_.Data(), m, ldm, dout, ldd, dgates_.Data(),
                                              need_in_diff_ ? in_diff->Data() : NULL, in_diff->Stride(), &g),
             "eesen_b200_bilstm_backward");
  }
}

std::string BiLstmParallel::Info() const {
  std::ostringstream os;
  os << "<BiLstmParallel> input " << input_dim_ << " cells/direction " << cell_dim_;
  return os.str();
}

// ------------------------------------------------------------------------------------ LstmParallel
static void ReadLstmTensors(std::istream &is, bool binary, int64 C, int64 I, std::vector<float> *flat) {
  HostMatrix wx, wm;
  HostVector b, pi, pf, po;
  wx.Read(is, binary); wm.Read(is, binary);
  b.Read(is, binary); pi.Read(is, binary); pf.Read(is, binary); po.Read(is, binary);
  KALDI_ASSERT(wx.rows == 4 * C && wx.cols == I && wm.rows == 4 * C && wm.cols == C);
  KALDI_ASSERT((int64)b.data.size() == 4 * C && (int64)pi.data.size() == C && (int64)pf.data.size() == C &&
               (int64)po.data.size() == C);
  flat->clear();
  flat->insert(flat->end(), wx.data.begin(), wx.data.end());
  flat->insert(flat->end(), wm.data.begin(), wm.data.end());
  flat->insert(flat->end(), b.data.begin(), b.data.end());
  flat->insert(flat->end(), pi.data.begin(), pi.data.end());
  flat->insert(flat->end(), pf.data.begin(), pf.data.end());
  flat->insert(flat->end(), po.data.begin(), po.data.end());
}
static void WriteLstmTensors(std::ostream &os, bool binary, int64 C, int64 I, const std::vector<float> &flat) {
  const float *p = flat.data();
  HostMatrix wx, wm;
  wx.rows = 4 * C; wx.cols = I; wx.data.assign(p, p + 4 * C * I); p += 4 * C * I;
  wm.rows = 4 * C; wm.cols = C; wm.data.assign(p, p + 4 * C * C); p += 4 * C * C;
  HostVector b, pi, pf, po;
  b.data.assign(p, p + 4 * C); p += 4 * C;
  pi.data.assign(p, p + C); p += C;
  pf.data.assign(p, p + C); p += C;
  po.data.assign(p, p + C); p += C;
  wx.Write(os, binary); wm.Write(os, binary);
  b.Write(os, binary); pi.Write(os, binary); pf.Write(os, binary); po.Write(os, binary);
}

void LstmParallel::ReadData(std::istream &is, bool binary) {   // lstm-layer.h:103-145
  while ('<' == Peek(is, binary)) {
    std::string tok;
    ReadToken(is, binary, &tok);
    if (tok == "<LearnRateCoef>") ReadBasicType(is, binary, &learn_rate_coef_);
    else if (tok == "<MaxGrad>") ReadBasicType(is, binary, &max_grad_);
    else if (tok == "<LstmAccus>") {
      ReadLstmTensors(is, binary, cell_dim_, input_dim_, &host_accu_);
      has_accu_ = true;
      break;
    } else KALDI_ERR << "Unknown token " << tok << " in <LstmParallel>";
  }
  if (cell_dim_ % 8 != 0 || input_dim_ % 4 != 0)
    KALDI_ERR << "LstmParallel on B200 needs cells % 8 == 0 and input dim % 4 == 0, got C=" << cell_dim_
              << " I=" << input_dim_;
  ReadLstmTensors(is, binary, cell_dim_, input_dim_, &host_params_);
}

void LstmParallel::WriteData(std::ostream &os, bool binary) const {   // lstm-layer.h:147-172
  WriteToken(os, binary, "<LearnRateCoef>"); WriteBasicType(os, binary, learn_rate_coef_);
  WriteToken(os, binary, "<MaxGrad>"); WriteBasicType(os, binary, max_grad_);
  if (has_accu_) {
    // DELIBERATE deviation from a reference bug: lstm-layer.h:153-163 writes the WEIGHTS (wei_gifo_x_ ...
    // phole_o_c_) a second time under <LstmAccus>, and ReadData (:119-131) then loads them as the
    // Adagrad/RMSProp accumulators -- after one reload sqrt(accu + eps) of a negative weight is NaN.  The real
    // accumulators have the same shapes, so the reference reads this file exactly like its own.
    KALDI_ASSERT((int64)host_accu_.size() == NumParams());
    WriteToken(os, binary, "<LstmAccus>");
    WriteLstmTensors(os, binary, cell_dim_, input_dim_, host_accu_);
  }
  WriteLstmTensors(os, binary, cell_dim_, input_dim_, host_params_);
}

void LstmParallel::Params(eesen_b200_bilstm_params *p, eesen_b200_bilstm_grads *g) const {
  const int64 C = cell_dim_, I = input_dim_;
  if (p) { p->ldwx = 0; p->ldwm = 0; }
  if (g) { g->ldwx = 0; g->ldwm = 0; }
  for (int d = 0; d < 2; d++) {   // index 1 mirrors index 0 (unused by the uni-directional entry points)
    if (p) {
      const float *b = w_;
      p->wx[d] = b; b += 4 * C * I;
      p->wm[d] = b; b += 4 * C * C;
      p->bias[d] = b; b += 4 * C;
      p->pi[d] = b; b += C;
      p->pf[d] = b; b += C;
      p->po[d] = b;
    }
    if (g) {
      float *b = g_;
      g->wx[d] = b; b += 4 * C * I;
      g->wm[d] = b; b += 4 * C * C;
      g->bias[d] = b; b += 4 * C;
      g->pi[d] = b; b += C;
      g->pf[d] = b; b += C;
      g->po[d] = b;
    }
  }
}

int32 LstmParallel::Streams(int32 rows) const {
  int32 S = num_streams_;
  if (S == 0 && nonparallel_) S = 1;   // <Lstm>: the whole input is one sequence
  KALDI_ASSERT(S > 0 && rows % S == 0);
  return S;
}

void LstmParallel::PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out) {
  const int32 S = Streams(in.NumRows()), T = in.NumRows() / S, C = cell_dim_;
  gates_.Resize(in.NumRows(), 4 * C, kUndefined);
  cell_.Resize(in.NumRows(), C, kUndefined);
  eesen_b200_bilstm_params p;
  Params(&p, NULL);
  CheckAbi(ctx_, eesen_b200_lstm_forward(ctx_, T, S, input_dim_, C, in.Data(), in.Stride(), &p, gates_.Data(),
                                         cell_.Data(), out->Data(), out->Stride()), "eesen_b200_lstm_forward");
}

void LstmParallel::BackpropagateFnc(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &out,
                                    const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff) {
  const int32 S = Streams(in.NumRows()), T = in.NumRows() / S, C = cell_dim_;
  dgates_.Resize(in.NumRows(), 4 * C, kUndefined);
  eesen_b200_bilstm_params p;
  eesen_b200_bilstm_grads g;
  Params(&p, &g);
  CheckAbi(ctx_, eesen_b200_lstm_backward(ctx_, T, S, input_dim_, C, in.Data(), in.Stride(), &p, gates_.Data(),
                                          cell_.Data(), out.Data(), out.Stride(), out_diff.Data(), out_diff.Stride(),
                                          dgates_.Data(), need_in_diff_ ? in_diff->Data() : NULL, in_diff->Stride(),
                                          &g), "eesen_b200_lstm_backward");
}

std::string LstmParallel::Info() const {
  std::ostringstream os;
  os << "<LstmParallel> input " << input_dim_ << " cells " << cell_dim_;
  return os.str();
}

// ------------------------------------------------------------------------------------ Affine / Softmax
void AffineTransform::ReadData(std::istream &is, bool binary) {
  while ('<' == Peek(is, binary)) {
    std::string tok;
    ReadToken(is, binary, &tok);
    if (tok == "<LearnRateCoef>") ReadBasicType(is, binary, &learn_rate_coef_);
    else if (tok == "<MaxGrad>") ReadBasicType(is, binary, &max_grad_);
    else if (tok == "<AffineAccus>") {   // affine-trans-layer.h:98-106
      HostMatrix aw;
      HostVector ab;
      aw.Read(is, binary);
      ab.Read(is, binary);
      KALDI_ASSERT(aw.rows == output_dim_ && aw.cols == input_dim_ && (int32)ab.data.size() == output_dim_);
      host_accu_ = aw.data;
      host_accu_.insert(host_accu_.end(), ab.data.begin(), ab.data.end());
      has_accu_ = true;
      break;
    } else KALDI_ERR << "Unknown token " << tok << " in <AffineTransform>";
  }
  if (input_dim_ % 4 != 0) KALDI_ERR << "AffineTransform on B200 needs input dim % 4 == 0, got " << input_dim_;
  HostMatrix w;
  HostVector b;
  w.Read(is, binary);
  b.Read(is, binary);
  KALDI_ASSERT(w.rows == output_dim_ && w.cols == input_dim_ && (int32)b.data.size() == output_dim_);
  host_params_ = w.data;
  host_params_.insert(host_params_.end(), b.data.begin(), b.data.end());
}

void AffineTransform::WriteData(std::ostream &os, bool binary) const {
  WriteToken(os, binary, "<LearnRateCoef>"); WriteBasicType(os, binary, learn_rate_coef_);
  WriteToken(os, binary, "<MaxGrad>"); WriteBasicType(os, binary, max_grad_);
  const size_t nw = (size_t)output_dim_ * input_dim_;
  if (has_accu_) {   // affine-trans-layer.h:123-129
    WriteToken(os, binary, "<AffineAccus>");
    HostMatrix aw;
    aw.rows = output_dim_; aw.cols = input_dim_;
    aw.data.assign(host_accu_.begin(), host_accu_.begin() + nw);
    HostVector ab;
    ab.data.assign(host_accu_.begin() + nw, host_accu_.end());
    aw.Write(os, binary);
    ab.Write(os, binary);
  }
  HostMatrix w;
  w.rows = output_dim_; w.cols = input_dim_;
  w.data.assign(host_params_.begin(), host_params_.begin() + nw);
  HostVector b;
  b.data.assign(host_params_.begin() + nw, host_params_.end());
  w.Write(os, binary);
  b.Write(os, binary);
}

void AffineTransform::PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out) {
  CheckAbi(ctx_, eesen_b200_affine_forward(ctx_, in.NumRows(), input_dim_, output_dim_, in.Data(), in.Stride(), w_,
                                           w_ + (size_t)output_dim_ * input_dim_, out->Data(), out->Stride()),
           "eesen_b200_affine_forward");
}

void AffineTransform::BackpropagateFnc(const CuMatrixBase<BaseFloat> &in, const CuMatrixBase<BaseFloat> &,
                                       const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff) {
  // in_diff = out_diff * W (affine-trans-layer.h:171) and the gradient part of Update (:182-183)
  CheckAbi(ctx_, eesen_b200_affine_backward(ctx_, in.NumRows(), input_dim_, output_dim_, in.Data(), in.Stride(),
                                            out_diff.Data(), out_diff.Stride(), w_,
                                            need_in_diff_ ? in_diff->Data() : NULL, in_diff->Stride(), g_,
                                            g_ + (size_t)output_dim_ * input_dim_),
           "eesen_b200_affine_backward");
}

void Softmax::PropagateFnc(const CuMatrixBase<BaseFloat> &in, CuMatrixBase<BaseFloat> *out) {
  CheckAbi(ctx_, eesen_b200_softmax(ctx_, in.NumRows(), input_dim_, in.Data(), in.Stride(), out->Data(),
                                    out->Stride(), NULL), "eesen_b200_softmax");
}
void Softmax::BackpropagateFnc(const CuMatrixBase<BaseFloat> &, const CuMatrixBase<BaseFloat> &,
                               const CuMatrixBase<BaseFloat> &out_diff, CuMatrixBase<BaseFloat> *in_diff) {
  in_diff->CopyFromMat(out_diff);  // softmax-layer.h:49-57: the CTC diff is already wrt the activations
}

// ------------------------------------------------------------------------------------ ClassPrior
void ClassPrior::LogPriors(const std::vector<double> &counts, BaseFloat prior_cutoff, BaseFloat blank_scale,
                           std::vector<float> *log_priors) {
  // class-prior.cc:44-76
  std::vector<double> p(counts);
  const size_t n = p.size();
  std::vector<float> mask(n, 0.f);
  int32 num_cutoff = 0;
  for (size_t i = 0; i < n; i++)
    if (p[i] < prior_cutoff) { p[i] = prior_cutoff; mask[i] = FLT_MAX / 2; num_cutoff++; }
  if (num_cutoff > 0)
    KALDI_WARN << num_cutoff << " out of " << n << " classes have counts lower than " << prior_cutoff;
  if (blank_scale != 1.0f && n > 0) p[0] *= blank_scale;
  double sum = 0.0;
  for (size_t i = 0; i < n; i++) sum += p[i];
  log_priors->resize(n);
  for (size_t i = 0; i < n; i++) {
    double lp = std::log(p[i] * (1.0 / sum));
    (*log_priors)[i] = (float)lp + mask[i];
  }
}

ClassPrior::ClassPrior(eesen_b200_ctx *ctx, const ClassPriorOptions &opts) : ctx_(ctx), prior_scale_(opts.prior_scale) {
  if (opts.class_frame_counts == "") return;
  KALDI_LOG << "Computing class-priors from : " << opts.class_frame_counts;
  std::ifstream is(opts.class_frame_counts.c_str());
  if (!is.is_open()) KALDI_ERR << "Failed to open " << opts.class_frame_counts;
  std::vector<double> counts;   // text vector "[ c0 c1 ... ]" (Vector<double>::Read, class-prior.cc:37-42)
  std::string tok;
  if (!(is >> tok) || tok != "[") KALDI_ERR << "Expected '[' at the start of " << opts.class_frame_counts;
  while (is >> tok && tok != "]") counts.push_back(atof(tok.c_str()));
  if (tok != "]") KALDI_ERR << "Missing ']' in " << opts.class_frame_counts;
  std::vector<float> lp;
  LogPriors(counts, opts.prior_cutoff, opts.blank_scale, &lp);
  dim_ = (int32)lp.size();
  if (dim_ == 0) return;
  CU_CHECK(cudaMalloc((void **)&d_log_priors_, sizeof(float) * dim_));
  CU_CHECK(cudaMemcpy(d_log_priors_, lp.data(), sizeof(float) * dim_, cudaMemcpyHostToDevice));
}

ClassPrior::~ClassPrior() {
  if (d_log_priors_) cudaFree(d_log_priors_);
}

void ClassPrior::SubtractOnLogpost(CuMatrixBase<BaseFloat> *llk) {   // class-prior.cc:78-90
  if (dim_ == 0) KALDI_ERR << "--class-frame-counts is empty: Cannot initialize priors without the counts.";
  if (dim_ != llk->NumCols())
    KALDI_ERR << "Dimensionality mismatch, class_frame_counts " << dim_ << " class_output_llk " << llk->NumCols();
  g_ctx = ctx_;
  llk->AddVecToRows(-prior_scale_, d_log_priors_, dim_);
}

// ------------------------------------------------------------------------------------ Net
Net::~Net() {
  for (size_t i = 0; i < layers_.size(); i++) delete layers_[i];
  if (w_) cudaFree(w_);
  if (g_) cudaFree(g_);
  if (corr_) cudaFree(corr_);
  if (accu_) cudaFree(accu_);
  if (d_segs_) cudaFree(d_segs_);
}

void Net::Read(const std::string &file) {
  g_ctx = ctx_;
  std::ifstream is(file.c_str(), std::ios::in | std::ios::binary);
  if (!is.is_open()) KALDI_ERR << "Failed to open model file " << file;
  bool binary;
  if (!InitKaldiInputStream(is, &binary)) KALDI_ERR << "Bad header in " << file;
  Read(is, binary);
  if (NumLayers() == 0) KALDI_WARN << "The network '" << file << "' is empty.";
}

void Net::Read(std::istream &is, bool binary) {
  g_ctx = ctx_;
  Layer *layer;
  while (NULL != (layer = Layer::Read(is, binary))) {
    if (NumLayers() > 0 && layers_.back()->OutputDim() != layer->InputDim())
      KALDI_ERR << "Dimensionality mismatch! Previous layer output:" << layers_.back()->OutputDim()
                << " Current layer input:" << layer->InputDim();
    layer->ctx_ = ctx_;
    layers_.push_back(layer);
  }
  propagate_buf_.resize(NumLayers() + 1);
  backpropagate_buf_.resize(NumLayers() + 1);
  opts_.learn_rate = 0.0;  // net.cc:274,294
  BindArena();
  // the reference's masks come from a std::random_device-seeded generator (kaldi-math.h:107-131): a fresh seed per
  // process unless the caller fixes one (Net::SetDropoutSeed)
  SetDropoutSeed(((uint64_t)std::random_device{}() << 32) ^ (uint64_t)std::random_device{}());
  Check();   // net.cc:276,296
}

// Net::Check (reference net.cc:448-468): buffer counts, layer dimensions, and no NaN/Inf in the parameters.
// The reference gathers every parameter on the host and tests the sum; here one kernel scans the parameter
// arena in place and returns two bits.
void Net::Check() const {
  KALDI_ASSERT((int32)propagate_buf_.size() == NumLayers() + 1);
  KALDI_ASSERT((int32)backpropagate_buf_.size() == NumLayers() + 1);
  for (size_t i = 0; i + 1 < layers_.size(); i++) {
    KALDI_ASSERT(layers_[i] != NULL);
    KALDI_ASSERT(layers_[i]->OutputDim() == layers_[i + 1]->InputDim());
  }
  if (arena_size_ == 0) return;
  int flags = 0;
  CheckAbi(ctx_, eesen_b200_check_finite(ctx_, w_, arena_size_, &flags), "eesen_b200_check_finite");
  if (flags & 2) KALDI_ERR << "'inf' in network parameters";
  if (flags & 1) KALDI_ERR << "'nan' in network parameters";
}

// Lay all trainable layers out in three contiguous arenas (params / raw grads / momentum), each
// layer block starting on a 16-byte boundary.
void Net::BindArena() {
  int64 total = 0;
  num_params_ = 0;
  std::vector<int64> offs;
  for (size_t i = 0; i < layers_.size(); i++) {
    if (!layers_[i]->IsTrainable()) { offs.push_back(-1); continue; }
    TrainableLayer *tl = dynamic_cast<TrainableLayer *>(layers_[i]);
    total = (total + 3) & ~(int64)3;
    offs.push_back(total);
    total += tl->NumParams();
    num_params_ += tl->NumParams();
  }
  arena_size_ = (total + 3) & ~(int64)3;
  if (arena_size_ == 0) return;
  CU_CHECK(cudaMalloc((void **)&w_, sizeof(float) * arena_size_));
  CU_CHECK(cudaMalloc((void **)&g_, sizeof(float) * (arena_size_ + 4)));   // +4: vote slot of BackpropagateShared
  CU_CHECK(cudaMalloc((void **)&corr_, sizeof(float) * arena_size_));
  CU_CHECK(cudaMemsetAsync(w_, 0, sizeof(float) * arena_size_, Stream()));
  CU_CHECK(cudaMemsetAsync(g_, 0, sizeof(float) * arena_size_, Stream()));
  CU_CHECK(cudaMemsetAsync(corr_, 0, sizeof(float) * arena_size_, Stream()));   // *_corr_.SetZero() bilstm-layer.h:401-406
  layer_offset_ = offs;
  for (size_t i = 0; i < layers_.size(); i++) {
    if (offs[i] < 0) continue;
    TrainableLayer *tl = dynamic_cast<TrainableLayer *>(layers_[i]);
    KALDI_ASSERT((int64)tl->host_params_.size() == tl->NumParams());
    CU_CHECK(cudaMemcpyAsync(w_ + offs[i], tl->host_params_.data(), sizeof(float) * tl->NumParams(),
                             cudaMemcpyHostToDevice, Stream()));
    tl->Bind(w_ + offs[i], g_ + offs[i]);
  }
  CU_CHECK(SyncStream());
  segs_dirty_ = true;
  bool any_accu = false;
  for (size_t i = 0; i < layers_.size(); i++)
    if (offs[i] >= 0 && dynamic_cast<TrainableLayer *>(layers_[i])->has_accu_) any_accu = true;
  if (any_accu) EnsureAccu(false);
}

// The accumulator arena of the adaptive rules: allocated when a model file carries accumulators or
// at the first Adagrad/RMSProp update (InitAdaBuffers, bilstm-layer.h:275-315: zero-initialised).
void Net::EnsureAccu(bool mark_all_layers) {
  if (!accu_ && arena_size_ > 0) {
    CU_CHECK(cudaMalloc((void **)&accu_, sizeof(float) * arena_size_));
    CU_CHECK(cudaMemsetAsync(accu_, 0, sizeof(float) * arena_size_, Stream()));
    for (size_t i = 0; i < layers_.size(); i++) {
      if (layer_offset_[i] < 0) continue;
      TrainableLayer *tl = dynamic_cast<TrainableLayer *>(layers_[i]);
      if (!tl->has_accu_) continue;
      KALDI_ASSERT((int64)tl->host_accu_.size() == tl->NumParams());
      CU_CHECK(cudaMemcpyAsync(accu_ + layer_offset_[i], tl->host_accu_.data(), sizeof(float) * tl->NumParams(),
                               cudaMemcpyHostToDevice, Stream()));
    }
    CU_CHECK(SyncStream());
  }
  if (mark_all_layers)
    for (size_t i = 0; i < layers_.size(); i++)
      if (layer_offset_[i] >= 0) dynamic_cast<TrainableLayer *>(layers_[i])->has_accu_ = true;
}

void Net::GetParams(std::vector<float> *host) const { GetArena(w_, host); }

void Net::GetArena(const float *arena, std::vector<float> *host) const {
  host->resize(num_params_);
  int64 o = 0;
  CU_CHECK(SyncStream());
  for (size_t i = 0; i < layers_.size(); i++) {
    if (layer_offset_[i] < 0) continue;
    TrainableLayer *tl = dynamic_cast<TrainableLayer *>(layers_[i]);
    CU_CHECK(cudaMemcpy(host->data() + o, arena + layer_offset_[i], sizeof(float) * tl->NumParams(),
                        cudaMemcpyDeviceToHost));
    o += tl->NumParams();
  }
}

void Net::SetParams(const float *host, int64 n) {
  KALDI_ASSERT(n == num_params_);
  int64 o = 0;
  CU_CHECK(SyncStream());
  for (size_t i = 0; i < layers_.size(); i++) {
    if (layer_offset_[i] < 0) continue;
    TrainableLayer *tl = dynamic_cast<TrainableLayer *>(layers_[i]);
    CU_CHECK(cudaMemcpy(w_ + layer_offset_[i], host + o, sizeof(float) * tl->NumParams(), cudaMemcpyHostToDevice));
    o += tl->NumParams();
  }
}

void Net::Write(const std::string &file, bool binary) {
  std::ofstream os(file.c_str(), std::ios::out | std::ios::binary);
  if (!os.is_open()) KALDI_ERR << "Failed to open " << file << " for writing";
  if (binary) { os.put('\0'); os.put('B'); }
  Write(os, binary);
  os.close();
  if (os.fail()) KALDI_ERR << "Failed to write " << file;
}

void Net::Write(std::ostream &os, bool binary) {
  Check();   // net.cc:326,345
  RefreshHostCopies();
  WriteToken(os, binary, "<Nnet>");
  if (!binary) os << std::endl;
  for (int32 i = 0; i < NumLayers(); i++) layers_[i]->Write(os, binary);
  WriteToken(os, binary, "</Nnet>");
  if (!binary) os << std::endl;
}

// refresh the host copies of parameters / accumulators from the device arenas
void Net::RefreshHostCopies() {
  CU_CHECK(SyncStream());
  for (size_t i = 0; i < layers_.size(); i++) {
    if (layer_offset_[i] < 0) continue;
    TrainableLayer *tl = dynamic_cast<TrainableLayer *>(layers_[i]);
    tl->host_params_.resize(tl->NumParams());
    CU_CHECK(cudaMemcpy(tl->host_params_.data(), w_ + layer_offset_[i], sizeof(float) * tl->NumParams(),
                        cudaMemcpyDeviceToHost));
    if (tl->has_accu_ && accu_) {
      tl->host_accu_.resize(tl->NumParams());
      CU_CHECK(cudaMemcpy(tl->host_accu_.data(), accu_ + layer_offset_[i], sizeof(float) * tl->NumParams(),
                          cudaMemcpyDeviceToHost));
    }
  }
}

void Net::WriteNonParal(const std::string &file, bool binary) {
  std::ofstream os(file.c_str(), std::ios::out | std::ios::binary);
  if (!os.is_open()) KALDI_ERR << "Failed to open " << file << " for writing";
  if (binary) { os.put('\0'); os.put('B'); }
  RefreshHostCopies();
  WriteToken(os, binary, "<Nnet>");
  if (!binary) os << std::endl;
  for (int32 i = 0; i < NumLayers(); i++) layers_[i]->WriteNonParal(os, binary);
  WriteToken(os, binary, "</Nnet>");
  if (!binary) os << std::endl;
  os.close();
  if (os.fail()) KALDI_ERR << "Failed to write " << file;
}

void Net::Feedforward(const CuMatrixBase<BaseFloat> &in, CuMatrix<BaseFloat> *out) {
  KALDI_ASSERT(NULL != out);
  g_ctx = ctx_;
  if (NumLayers() == 0) { (*out) = in; return; }
  if (NumLayers() == 1) { layers_[0]->Propagate(in, out); return; }
  KALDI_ASSERT(propagate_buf_.size() >= 2);
  int32 L = 0;
  layers_[L]->Propagate(in, &propagate_buf_[L % 2]);
  for (L++; L <= NumLayers() - 2; L++) layers_[L]->Propagate(propagate_buf_[(L - 1) % 2], &propagate_buf_[L % 2]);
  layers_[L]->Propagate(propagate_buf_[(L - 1) % 2], out);
  // the reference releases the two buffers here (net.cc:134-136); ours stay allocated for the next
  // utterance batch (stream-ordered reuse, no cudaFree/cudaMalloc per call) but hold no result
}

void Net::SetTrainMode() {
  in_train_ = true;
  for (size_t i = 0; i < layers_.size(); i++) layers_[i]->SetTrainMode();
}
void Net::SetTestMode() {
  in_train_ = false;
  for (size_t i = 0; i < layers_.size(); i++) layers_[i]->SetTestMode();
}
void Net::ChangeDropoutParameters(BaseFloat forward_dropout, bool fw_step, bool fw_sequence, bool rnndrop,
                                  bool no_mem_loss, BaseFloat recurrent_dropout, bool rec_step, bool rec_sequence,
                                  bool twiddle_forward) {
  for (size_t i = 0; i < layers_.size(); i++) {
    BiLstmParallel *bl = dynamic_cast<BiLstmParallel *>(layers_[i]);
    if (!bl) continue;
    KALDI_LOG << "Changing dropout params for layer " << i;
    bl->ChangeDropoutParameters(forward_dropout, fw_step, fw_sequence, rnndrop, no_mem_loss, recurrent_dropout,
                                rec_step, rec_sequence, twiddle_forward);
  }
}
void Net::SetDropoutSeed(uint64_t seed) {
  for (size_t i = 0; i < layers_.size(); i++) {
    BiLstmParallel *bl = dynamic_cast<BiLstmParallel *>(layers_[i]);
    if (bl) bl->SetDropoutSeed(seed, (uint64_t)i + 1);
  }
}

int32 Net::InputDim() const { return layers_.empty() ? 0 : layers_.front()->InputDim(); }
int32 Net::OutputDim() const { return layers_.empty() ? 0 : layers_.back()->OutputDim(); }

void Net::SetSeqLengths(std::vector<int> &sequence_lengths) {
  for (size_t i = 0; i < layers_.size(); i++) layers_[i]->SetSeqLengths(sequence_lengths);
}

void Net::SetTrainOptions(const NetTrainOptions &opts) {
  opts_ = opts;
  segs_dirty_ = true;
}

void Net::SetUpdateAlgorithm(const std::string &opt) {   // net.cc:481-496
  if (opt == "SGD") update_algorithm_ = 0;
  else if (opt == "Adagrad") update_algorithm_ = 1;
  else if (opt == "RMSProp") update_algorithm_ = 2;
  else KALDI_ERR << "This optimization algorithm is unsupported: " << opt;
  segs_dirty_ = true;
}

void Net::UploadSegments() {
  std::vector<eb::SgdSegment> segs;
  for (size_t i = 0; i < layers_.size(); i++) {
    if (layer_offset_[i] < 0) continue;
    TrainableLayer *tl = dynamic_cast<TrainableLayer *>(layers_[i]);
    eb::SgdSegment s;
    s.offset = layer_offset_[i];
    s.count = 0;  // fixed below: up to the next segment start
    // learn_rate_coef_ scales the SGD step only; the adaptive branch uses opts_.learn_rate as is
    // (bilstm-layer.h:865-869 vs :885-955, affine-trans-layer.h:191-219)
    s.lr = update_algorithm_ == 0 ? opts_.learn_rate * tl->learn_rate_coef_ : opts_.learn_rate;
    s.max_grad = tl->max_grad_;
    segs.push_back(s);
  }
  for (size_t k = 0; k < segs.size(); k++)
    segs[k].count = (k + 1 < segs.size() ? segs[k + 1].offset : arena_size_) - segs[k].offset;
  nseg_ = segs.size();
  if (!d_segs_) CU_CHECK(cudaMalloc(&d_segs_, sizeof(eb::SgdSegment) * std::max<size_t>(1, layers_.size())));
  CU_CHECK(cudaMemcpy(d_segs_, segs.data(), sizeof(eb::SgdSegment) * nseg_, cudaMemcpyHostToDevice));
  segs_dirty_ = false;
}

void Net::Propagate(const CuMatrixBase<BaseFloat> &in, CuMatrix<BaseFloat> *out) {
  KALDI_ASSERT(NULL != out);
  g_ctx = ctx_;
  if (NumLayers() == 0) { (*out) = in; return; }
  propagate_buf_[0].Resize(in.NumRows(), in.NumCols(), kUndefined);
  propagate_buf_[0].CopyFromMat(in);
  // in training mode the recurrent forward kernels also write the fp16 planes of their outputs (context.h:ActPlanes):
  // one generation per forward pass
  ctx_->act_gen += 1;
  ctx_->act_enable = in_train_ ? 1 : 0;
  for (int32 i = 0; i < NumLayers(); i++) layers_[i]->Propagate(propagate_buf_[i], &propagate_buf_[i + 1]);
  ctx_->act_enable = 0;
  (*out) = propagate_buf_[NumLayers()];
}

// Data-parallel runs reduce the gradient block of a layer as soon as that layer has back-propagated (top-down, the
// reference's update order net.cc:98-105): one NCCL all-reduce per trainable layer on the side stream, overlapped with
// the layers below.  `zero` = this rank has no minibatch (BackpropagateShared): it contributes zeros in the same
// sequence of collectives.
void Net::BackpropagateLayers(const CuMatrixBase<BaseFloat> *out_diff, CuMatrix<BaseFloat> *in_diff) {
  if (out_diff && !in_train_) KALDI_ERR << "Can't backpropagate in test mode";
  int rank, nranks;
  eesen_b200_world(ctx_, &rank, &nranks);
  const CuMatrixBase<BaseFloat> *diff = out_diff;
  for (int32 i = NumLayers() - 1; i >= 0; i--) {
    if (out_diff) {
      layers_[i]->need_in_diff_ = (i > 0) || (in_diff != NULL);
      layers_[i]->Backpropagate(propagate_buf_[i], propagate_buf_[i + 1], *diff, &backpropagate_buf_[i]);
      diff = &backpropagate_buf_[i];
    }
    if (nranks > 1 && layer_offset_[i] >= 0) {
      int64 end = arena_size_;
      for (int32 k = i + 1; k < NumLayers(); k++)
        if (layer_offset_[k] >= 0) { end = layer_offset_[k]; break; }
      CheckAbi(ctx_, eesen_b200_allreduce_sum_overlapped(ctx_, g_ + layer_offset_[i], end - layer_offset_[i]),
               "eesen_b200_allreduce_sum_overlapped");
    }
  }
}

// ... then the identical momentum / clip / SGD update on every rank
void Net::Update() {
  if (segs_dirty_) UploadSegments();
  ctx_->join_side();   // every gradient product and every per-layer all-reduce has to be in
  if (nseg_ > 0) {
    int pe = ctx_->prof_begin(eesen_b200_ctx::kSgd);
    if (update_algorithm_ != 0) EnsureAccu(true);
    cudaError_t e = eb::optimizer_update(ctx_->stream, ctx_->num_sms, update_algorithm_, w_, corr_, accu_, g_,
                                         opts_.momentum, opts_.adagrad_epsilon, opts_.rmsprop_rho,
                                         opts_.rmsprop_one_minus_rho, (const eb::SgdSegment *)d_segs_, nseg_,
                                         arena_size_);
    ctx_->prof_end(pe);
    ctx_->launches += 1;
    if (e != cudaSuccess) KALDI_ERR << "optimizer_update: " << cudaGetErrorString(e);
  }
}

void Net::Backpropagate(const CuMatrixBase<BaseFloat> &out_diff, CuMatrix<BaseFloat> *in_diff) {
  g_ctx = ctx_;
  if (NumLayers() == 0) { if (in_diff) (*in_diff) = out_diff; return; }
  BackpropagateLayers(&out_diff, in_diff);
  Update();
  if (NULL != in_diff) (*in_diff) = backpropagate_buf_[0];
}

int32 Net::BackpropagateShared(const CuMatrixBase<BaseFloat> *out_diff) {
  g_ctx = ctx_;
  if (NumLayers() == 0 || arena_size_ == 0) return out_diff ? 1 : 0;
  if (!out_diff) CU_CHECK(cudaMemsetAsync(g_, 0, sizeof(float) * arena_size_, Stream()));
  BackpropagateLayers(out_diff, NULL);   // per-layer all-reduces (an idle rank contributes zeros)
  // the 4 spare floats behind the arena carry the "I had a minibatch" vote through one more (tiny) all-reduce
  const float vote[4] = {out_diff ? 1.0f : 0.0f, 0.f, 0.f, 0.f};
  CU_CHECK(cudaMemcpyAsync(g_ + arena_size_, vote, sizeof(vote), cudaMemcpyHostToDevice, Stream()));
  CheckAbi(ctx_, eesen_b200_allreduce_sum(ctx_, g_ + arena_size_, 4), "eesen_b200_allreduce_sum");
  float active = 0.f;
  CU_CHECK(cudaMemcpyAsync(&active, g_ + arena_size_, sizeof(float), cudaMemcpyDeviceToHost, Stream()));
  CU_CHECK(SyncStream());
  const int32 n_active = (int32)(active + 0.5f);
  if (n_active > 0) Update();   // a step in which NO rank had data is not a training step: no momentum-only update
  return n_active;
}

static std::string Moments(const std::vector<float> &v, int64 b, int64 n) {
  double s = 0, s2 = 0, mn = 1e30, mx = -1e30;
  for (int64 i = b; i < b + n; i++) { s += v[i]; s2 += (double)v[i] * v[i]; mn = std::min<double>(mn, v[i]); mx = std::max<double>(mx, v[i]); }
  double mean = s / n, var = s2 / n - mean * mean;
  std::ostringstream os;
  os << " ( min " << mn << ", max " << mx << ", mean " << mean << ", variance " << var << " ) ";
  return os.str();
}

std::string Net::Info() const {
  std::ostringstream os;
  os << "num-layers " << NumLayers() << "\ninput-dim " << InputDim() << "\noutput-dim " << OutputDim()
     << "\nnumber-of-parameters " << num_params_ / 1e6 << " millions\n";
  std::vector<float> p;
  GetArena(w_, &p);
  int64 o = 0;
  for (size_t i = 0; i < layers_.size(); i++) {
    os << "layer " << i + 1 << " : " << Layer::TypeToMarker(layers_[i]->GetType()) << ", input-dim "
       << layers_[i]->InputDim() << ", output-dim " << layers_[i]->OutputDim();
    if (layer_offset_[i] >= 0) {
      TrainableLayer *tl = dynamic_cast<TrainableLayer *>(layers_[i]);
      os << ", params" << Moments(p, o, tl->NumParams());
      o += tl->NumParams();
    }
    os << "\n";
  }
  return os.str();
}

std::string Net::InfoGradient() const {
  std::ostringstream os;
  std::vector<float> c;
  GetArena(corr_, &c);
  int64 o = 0;
  os << "### Gradient stats :\n";
  for (size_t i = 0; i < layers_.size(); i++) {
    if (layer_offset_[i] < 0) continue;
    TrainableLayer *tl = dynamic_cast<TrainableLayer *>(layers_[i]);
    os << "Layer " << i + 1 << " : " << Layer::TypeToMarker(layers_[i]->GetType()) << ", corr_"
       << Moments(c, o, tl->NumParams()) << "\n";
    o += tl->NumParams();
  }
  return os.str();
}

// ------------------------------------------------------------------------------------ Ctc
template <typename Tp>
static void GrowDevice(Tp **p, size_t *cap, size_t need) {
  if (need <= *cap) return;
  if (*p) { CU_CHECK(SyncStream()); CU_CHECK(cudaFree(*p)); }
  size_t want = need + need / 4 + 16;
  CU_CHECK(cudaMalloc((void **)p, sizeof(Tp) * want));
  *cap = want;
}
template <typename Tp>
static void GrowPinned(Tp **p, size_t *cap, size_t need) {
  if (need <= *cap) return;
  if (*p) { CU_CHECK(SyncStream()); CU_CHECK(cudaFreeHost(*p)); }
  size_t want = need + need / 4 + 16;
  CU_CHECK(cudaMallocHost((void **)p, sizeof(Tp) * want));
  *cap = want;
}

Ctc::Ctc(eesen_b200_ctx *ctx) : ctx_(ctx) { g_ctx = ctx; }

Ctc::~Ctc() {
  if (d_len_) cudaFree(d_len_);
  if (d_argmax_) cudaFree(d_argmax_);
  if (h_argmax_) cudaFreeHost(h_argmax_);
  if (h_pzx_) cudaFreeHost(h_pzx_);
}

// label staging: [S x max_lab] padded matrix + lengths (the reference uploads the expanded
// S x (2*max+1) matrix on every one of its 2T kernel launches, cuda-matrix.cc:882-883,948-950)
void Ctc::Upload(const std::vector<int32> &frame_num_utt, std::vector<std::vector<int32> > &label, int32 num_classes) {
  int32 S = frame_num_utt.size();
  KALDI_ASSERT((int32)label.size() >= S);
  max_lab_ = 1;
  for (int32 s = 0; s < S; s++) {
    max_lab_ = std::max<int32>(max_lab_, label[s].size());
    // the reference never validates the ids (ctc-loss.cc:122-128): a label >= K reads past the posterior row
    for (size_t l = 0; l < label[s].size(); l++)
      if (label[s][l] < 0 || label[s][l] >= num_classes)
        KALDI_ERR << "utterance " << s << " of the minibatch: label " << label[s][l] << " outside [0, " << num_classes
                  << ") (the network has " << num_classes << " outputs, blank = 0)";
  }
  // one buffer: [len S][lablen S][pzx S as float][labels S*max_lab]
  size_t ints = (size_t)3 * S + (size_t)S * max_lab_;
  GrowDevice(&d_len_, &cap_len_, ints);
  std::vector<int32> h(ints, 0);
  for (int32 s = 0; s < S; s++) {
    h[s] = frame_num_utt[s];
    h[S + s] = label[s].size();
    for (size_t l = 0; l < label[s].size(); l++) h[3 * S + (size_t)s * max_lab_ + l] = label[s][l];
  }
  CU_CHECK(cudaMemcpyAsync(d_len_, h.data(), sizeof(int32) * ints, cudaMemcpyHostToDevice, Stream()));
  d_lablen_ = d_len_ + S;
  d_pzx_ = reinterpret_cast<float *>(d_len_ + 2 * S);
  d_lab_ = nullptr;  // labels live inside the same buffer
}

void Ctc::EvalParallelAsync(const std::vector<int32> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                            std::vector<std::vector<int32> > &label, CuMatrix<BaseFloat> *diff) {
  g_ctx = ctx_;
  if (pending_eval_) Finish(NULL);
  diff->Resize(net_out.NumRows(), net_out.NumCols(), kUndefined);
  int32 S = frame_num_utt.size();
  int32 num_frames = net_out.NumRows();
  KALDI_ASSERT(S > 0 && num_frames % S == 0);
  int32 T = num_frames / S;
  Upload(frame_num_utt, label, net_out.NumCols());
  CheckAbi(ctx_, eesen_b200_ctc_eval(ctx_, T, S, net_out.NumCols(), max_lab_, d_len_, d_len_ + 3 * S, d_lablen_,
                                     net_out.Data(), net_out.Stride(), d_pzx_, diff->Data(), diff->Stride()),
           "eesen_b200_ctc_eval");
  GrowPinned(&h_pzx_, &cap_hpzx_, (size_t)S);
  CU_CHECK(cudaMemcpyAsync(h_pzx_, d_pzx_, sizeof(float) * S, cudaMemcpyDeviceToHost, Stream()));
  p_frames_ = frame_num_utt;
  p_S_ = S;
  pending_eval_ = true;
}

void Ctc::ErrorRateMSeqAsync(const std::vector<int> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                             std::vector<std::vector<int> > &label) {
  g_ctx = ctx_;
  if (pending_err_) Finish(NULL);
  int32 rows = net_out.NumRows();
  GrowDevice(&d_argmax_, &cap_arg_, (size_t)rows);
  GrowPinned(&h_argmax_, &cap_harg_, (size_t)rows);
  CheckAbi(ctx_, eesen_b200_row_argmax(ctx_, rows, net_out.NumCols(), net_out.Data(), net_out.Stride(), d_argmax_),
           "eesen_b200_row_argmax");
  CU_CHECK(cudaMemcpyAsync(h_argmax_, d_argmax_, sizeof(int) * rows, cudaMemcpyDeviceToHost, Stream()));
  p_frames_ = frame_num_utt;
  p_labels_ = label;
  p_S_ = frame_num_utt.size();
  p_rows_ = rows;
  pending_err_ = true;
}

// util/edit-distance-inl.h:28-75
static int32 LevenshteinEditDistance(const std::vector<int32> &a, const std::vector<int32> &b) {
  std::vector<int32> prev(b.size() + 1), cur(b.size() + 1);
  for (size_t j = 0; j <= b.size(); j++) prev[j] = j;
  for (size_t i = 1; i <= a.size(); i++) {
    cur[0] = i;
    for (size_t j = 1; j <= b.size(); j++)
      cur[j] = std::min(std::min(prev[j] + 1, cur[j - 1] + 1), prev[j - 1] + (a[i - 1] != b[j - 1] ? 1 : 0));
    prev.swap(cur);
  }
  return prev[b.size()];
}

void Ctc::Finish(double stats[4]) {
  if (!pending_eval_ && !pending_err_) { if (stats) stats[0] = stats[1] = stats[2] = stats[3] = 0; return; }
  CU_CHECK(SyncStream());
  double obj = 0, err_batch = 0, ref_batch = 0, frames_batch = 0;
  if (pending_eval_) {
    pzx_host_.assign(h_pzx_, h_pzx_ + p_S_);
    for (int32 s = 0; s < p_S_; s++) obj += pzx_host_[s];
    obj_progress_ += obj;                      // ctc-loss.cc:171-177
    sequences_progress_ += p_S_;
    sequences_num_ += p_S_;
    for (int32 s = 0; s < p_S_; s++) { frames_progress_ += p_frames_[s]; frames_ += p_frames_[s]; frames_batch += p_frames_[s]; }
  }
  if (pending_err_) {
    // ctc-loss.cc:250-282: per sequence, collapse repeats, drop blanks, edit distance
    int32 S = p_S_;
    for (int32 s = 0; s < S; s++) {
      int32 nf = p_frames_[s];
      std::vector<int32> hyp;
      int32 prev = -1;
      for (int32 f = 0; f < nf; f++) {
        int32 c = h_argmax_[(size_t)f * S + s];
        if (c != prev && c != 0) hyp.push_back(c);
        prev = c;
      }
      int32 e = LevenshteinEditDistance(p_labels_[s], hyp);
      err_batch += e;
      ref_batch += p_labels_[s].size();
    }
    error_num_ += err_batch; ref_num_ += ref_batch;
    error_num_progress_ += err_batch; ref_num_progress_ += ref_batch;
  }
  if (pending_eval_ && sequences_progress_ >= report_step_) {   // ctc-loss.cc:180-192
    KALDI_VLOG(1) << "After " << sequences_num_ << " sequences (" << frames_ / (100.0 * 3600) << "Hr): "
                  << "Obj(log[Pzx]) = " << obj_progress_ / sequences_progress_
                  << "   TokenAcc = " << 100.0 * (1.0 - error_num_progress_ / ref_num_progress_) << "%";
    sequences_progress_ = 0; frames_progress_ = 0; obj_progress_ = 0.0;
    error_num_progress_ = 0; ref_num_progress_ = 0;
  }
  pending_eval_ = pending_err_ = false;
  if (stats) { stats[0] = obj; stats[1] = err_batch; stats[2] = ref_batch; stats[3] = frames_batch; }
}

void Ctc::EvalParallel(const std::vector<int32> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                       std::vector<std::vector<int32> > &label, CuMatrix<BaseFloat> *diff) {
  EvalParallelAsync(frame_num_utt, net_out, label, diff);
  // statistics are folded lazily (Finish) so that ErrorRateMSeq can share the single host sync;
  // a caller that never calls ErrorRateMSeq/Report still gets them at the next Eval/Report.
}

void Ctc::ErrorRateMSeq(const std::vector<int> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                        std::vector<std::vector<int> > &label, std::string &out) {
  ErrorRateMSeqAsync(frame_num_utt, net_out, label);
  if (out.length()) {
    Finish(NULL);
    // ctc-loss.cc:283-291: hypothesis with frame index and probability, appended to `out`
    std::ofstream output(out.c_str(), std::ofstream::out | std::ofstream::app);
    std::vector<float> host((size_t)net_out.NumRows() * net_out.NumCols());
    net_out.CopyToHost(host.data(), net_out.NumCols());
    int32 S = frame_num_utt.size();
    for (int32 s = 0; s < S; s++) {
      output << "utt";
      int32 prev = -1;
      for (int32 f = 0; f < frame_num_utt[s]; f++) {
        int32 c = h_argmax_[(size_t)f * S + s];
        if (c != prev && c != 0)
          output << " | " << c << " " << f << " " << host[((size_t)f * S + s) * net_out.NumCols() + c];
        prev = c;
      }
      output << "\n";
    }
  }
}

std::string Ctc::Report() {
  Finish(NULL);
  std::ostringstream oss;
  oss << "\nTOKEN_ACCURACY >> " << 100.0 * (1.0 - error_num_ / ref_num_) << "% <<";
  return oss.str();
}

CE::CE(eesen_b200_ctx *ctx) : ctx_(ctx) { g_ctx = ctx; }

CE::~CE() {
  if (d_len_) cudaFree(d_len_);
  if (d_stats_) cudaFree(d_stats_);
  if (h_stats_) cudaFreeHost(h_stats_);
}

void CE::EvalParallel(const std::vector<int32> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                      const std::vector<int32> &target, CuMatrix<BaseFloat> *diff) {
  g_ctx = ctx_;
  const int32 S = frame_num_utt.size(), rows = net_out.NumRows(), K = net_out.NumCols();
  KALDI_ASSERT(S > 0 && rows % S == 0 && (int32)target.size() == rows);
  for (int32 r = 0; r < rows; r++)   // ce-loss.cc:104-111 (the reference checks only the upper bound)
    if (r / S < frame_num_utt[r % S] && (target[r] < 0 || target[r] >= K))
      KALDI_ERR << "Class id out of network output dimension. Net outputs: " << K << ", class ID : " << target[r];
  if (!pending_.empty()) Finish(NULL);   // the target buffer below is about to be overwritten
  size_t ints = (size_t)S + rows;
  GrowDevice(&d_len_, &cap_len_, ints);
  CU_CHECK(cudaMemcpyAsync(d_len_ + S, target.data(), sizeof(int32) * rows, cudaMemcpyHostToDevice, Stream()));
  EvalParallelAsync(frame_num_utt, net_out, d_len_ + S, diff);
}

void CE::EvalParallelAsync(const std::vector<int32> &frame_num_utt, const CuMatrixBase<BaseFloat> &net_out,
                           const int32 *d_target, CuMatrix<BaseFloat> *diff) {
  g_ctx = ctx_;
  const int32 S = frame_num_utt.size(), rows = net_out.NumRows();
  KALDI_ASSERT(S > 0 && rows % S == 0);
  if ((int)pending_.size() == kSlots) Finish(NULL);
  if (!d_stats_) {
    CU_CHECK(cudaMalloc((void **)&d_stats_, sizeof(double) * 3 * kSlots));
    CU_CHECK(cudaMallocHost((void **)&h_stats_, sizeof(double) * 3 * kSlots));
  }
  GrowDevice(&d_len_, &cap_len_, (size_t)S + (d_target == d_len_ + S ? rows : 0));
  // pageable source: the copy is staged before cudaMemcpyAsync returns, so frame_num_utt may change afterwards
  CU_CHECK(cudaMemcpyAsync(d_len_, frame_num_utt.data(), sizeof(int32) * S, cudaMemcpyHostToDevice, Stream()));
  diff->Resize(rows, net_out.NumCols(), kUndefined);
  CheckAbi(ctx_, eesen_b200_ce_eval(ctx_, rows / S, S, net_out.NumCols(), d_len_, net_out.Data(), net_out.Stride(),
                                    d_target, diff->Data(), diff->Stride(), d_stats_ + 3 * pending_.size()),
           "eesen_b200_ce_eval");
  pending_.push_back(Pending{S, rows});
}

void CE::Finish(double stats[4]) {
  if (!pending_.empty()) {
    const size_t n = pending_.size();
    CU_CHECK(cudaMemcpyAsync(h_stats_, d_stats_, sizeof(double) * 3 * n, cudaMemcpyDeviceToHost, Stream()));
    CU_CHECK(SyncStream());
    for (size_t i = 0; i < n; i++) {
      const double obj = h_stats_[3 * i], correct = h_stats_[3 * i + 1], valid = h_stats_[3 * i + 2];
      const int64 S = pending_[i].S, rows = pending_[i].rows;
      obj_ += obj; obj_progress_ += obj;                              // ce-loss.cc:144-150
      correct_ += (int64)correct; correct_progress_ += (int64)correct;
      sequences_progress_ += S; sequences_num_ += S;
      frames_progress_ += rows; frames_ += rows;                      // padded rows, as the reference counts them
      if (sequences_progress_ > report_step_) {                       // ce-loss.cc:152-167
        KALDI_LOG << "After " << sequences_num_ << " sequences (" << frames_ / (100.0 * 3600) << "Hr): "
                  << "CE-Obj = " << obj_progress_ / sequences_progress_
                  << "Frame-level CE-Obj = " << obj_progress_ / frames_progress_
                  << "   FrameAcc = " << 100.0 * (double(correct_progress_) / frames_progress_) << "%"
                  << " obj_progress_=  " << obj_progress_
                  << " sequences_progress_=  " << sequences_progress_
                  << " frames_progress_=  " << frames_progress_;
        sequences_progress_ = 0; frames_progress_ = 0; obj_progress_ = 0.0; correct_progress_ = 0;
      }
      last_[0] = obj; last_[1] = correct; last_[2] = valid; last_[3] = (double)rows;
    }
    pending_.clear();
  }
  if (stats) memcpy(stats, last_, sizeof(last_));
}

std::string CE::Report() {
  Finish(NULL);
  std::ostringstream oss;
  oss << "\nFRAME_ACCURACY >> " << 100.0 * (double(correct_) / frames_) << "% <<";   // ce-loss.cc:171-175, real quotient
  return oss.str();
}

}  // namespace eesen
