// eesen_b200/host/context.h -- per-process device context: replaces the reference's singleton
// CuDevice (src/gpucompute/cuda-device.{h,cc}) with {device, one compute stream, grow-only
// workspace arenas, optional NCCL communicator}.  No per-call device synchronisation
// (the reference syncs after every kernel, cuda-common.h:37-44).
#ifndef EESEN_B200_HOST_CONTEXT_H_
#define EESEN_B200_HOST_CONTEXT_H_

#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "../csrc/kernels.h"

struct eesen_b200_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  int num_sms = 0;
  size_t max_smem = 0;
  int gemm_prec = 0, rec_prec = 0;
  int gemm_engine = 0;  // 0 = tcgen05 (gemm_tc.cu), 1 = warp-level mma.sync (gemm.cu)
  std::string err;
  long launches = 0;

  struct Buf {
    void *p = nullptr;
    size_t bytes = 0;
  };
  Buf gemm_ws, lstm_pbuf, lstm_gsum, lstm_flags, ctc_ws, colsum_ws, seg_buf, flag_buf, bf16_a, bf16_b, lstm_gflags;
  Buf gemm_ws_side, bf16_a_side, bf16_b_side;   // the side stream's own scratch
  Buf decode_ws;
  Buf ce_ws;   // per-CTA partial sums of the cross-entropy statistics

  // fp16x3 arithmetic (gemm_prec 0 on the 16-bit tensor pipe): converted operand planes of whole matrices that feed
  // several products; do_gemm finds sub-blocks of them by address.
  struct PlaneEntry {
    const float *base = nullptr;
    long rows = 0;
    int cols = 0, ld = 0;
    unsigned gen = 0;    // (act) the forward pass that made the planes
    Buf planes;          // hi plane, then lo plane
    eb::F16View view;
    // the [r x c] block at P with leading dimension ld_, if it lies in this matrix on an 8-column boundary
    bool find(const float *P, long r, int c, int ld_, eb::F16View *out) const {
      if (!base || ld_ != ld || P < base) return false;
      const long off = (long)(P - base), ro = off / ld, co = off % ld;
      if (ro + r > rows || co + c > cols || (co & 7)) return false;
      *out = view;
      out->hi = (const char *)view.hi + ((size_t)ro * view.ld + co) * 2;
      out->lo = (const char *)view.lo + ((size_t)ro * view.ld + co) * 2;
      return true;
    }
  };
  // Per layer call: d(gates), the layer input, m, Wx are converted ONCE and registered here; they live until the next
  // f16_clear().
  enum { kF16Slots = 6 };
  PlaneEntry f16_slots[kF16Slots];
  int f16_used = 0;
  void f16_clear() { f16_used = 0; }
  Buf f16_tmp[4];        // ad-hoc operands: [0] A / [1] B on `stream`, [2] A / [3] B on the side stream
  int f16x3 = 1;         // EESEN_B200_GEMM_FP32X3=tf32 : keep the kind::tf32 3-term split (A/B measurements)
  // Per forward pass: planes of layer outputs written by the recurrent forward kernel itself (LstmFwdArgs::out_hi), and
  // of the input weights Wx, outlive f16_clear() -- the next layer's input product, and the products of the backward
  // pass, find them by address and convert nothing.  Only while a Net drives the step (act_enable, set by
  // Net::Propagate in training mode; act_gen: one generation per forward pass, older entries are dead), so that callers
  // of the level-1 operators who reuse buffers never meet planes of other data.
  enum { kActSlots = 32 };
  PlaneEntry act[kActSlots];
  int act_next = 0, act_enable = 0;
  unsigned act_gen = 1;
  int *act_kexp = nullptr;   // device: the constant 13
  // f16_meta: 4096 bytes of 8-byte device records {unsigned max scratch, int kexp}, indexed from these bases: per-call
  // entries, the four temporary operands (as f16_tmp), max |d(gates)| of the recurrent backward kernel, act_kexp,
  // per-pass entries
  enum { kMetaCall = 0, kMetaTmp = kF16Slots, kMetaDgmax = kMetaTmp + 4, kMetaK13 = kMetaTmp + 5, kMetaAct = kMetaTmp + 8 };
  Buf f16_meta;

  // Side stream (lower priority): work nothing on the critical path waits for -- the weight-gradient products of
  // layer l and the all-reduce of its gradient block run here while `stream` carries dX and the recurrent backward
  // of layer l-1 (the tcgen05 recurrent kernels occupy 80 of the 148 SMs).  fork_side(): side waits for everything
  // queued on `stream` so far; join_side(): `stream` waits for everything queued on side.  Every consumer of the
  // gradient arena (all-reduce, optimiser, host reads, eesen_b200_synchronize) joins first.
  cudaStream_t side = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  bool side_pending = false;
  int overlap = 1;   // EESEN_B200_OVERLAP=0: everything on `stream` (A/B measurements)
  // Streamed input product of the recurrent forward pass: x*Wx^T is cut into chunks of time steps in the order the
  // two directions consume them; the first chunk runs on `stream`, the rest on the side stream WHILE the recurrent
  // kernel runs (it checks a per-chunk flag before it reads a chunk).
  unsigned gepoch = 0;
  void fork_side() {
    cudaEventRecord(ev_fork, stream);
    cudaStreamWaitEvent(side, ev_fork, 0);
    side_pending = true;
  }
  void join_side() {
    if (!side_pending) return;
    cudaEventRecord(ev_join, side);
    cudaStreamWaitEvent(stream, ev_join, 0);
    side_pending = false;
  }

  // optional per-category kernel timing with CUDA events on `stream` (bench.py roofline)
  enum { kGemm = 0, kLstmFwd, kLstmBwd, kSoftmax, kCtc, kSgd, kAllReduce, kMisc, kGemmSide, kNumCat };   // kGemmSide: dense products / conversions of the side stream
  struct ProfEv { cudaEvent_t a, b; int cat; cudaStream_t st; };
  bool prof_on = false;
  std::vector<ProfEv> prof_events;
  std::vector<ProfEv> prof_pool;
  double prof_ms[kNumCat] = {0};
  long prof_count[kNumCat] = {0};
  int prof_begin(int cat, bool on_side = false) {
    if (!prof_on) return -1;
    ProfEv e;
    if (!prof_pool.empty()) { e = prof_pool.back(); prof_pool.pop_back(); }
    else { cudaEventCreate(&e.a); cudaEventCreate(&e.b); }
    e.cat = (cat == kGemm && on_side) ? (int)kGemmSide : cat;
    e.st = on_side ? side : stream;
    cudaEventRecord(e.a, e.st);
    prof_events.push_back(e);
    return (int)prof_events.size() - 1;
  }
  void prof_end(int idx) {
    if (idx >= 0) cudaEventRecord(prof_events[idx].b, prof_events[idx].st);
  }
  void prof_collect() {
    join_side();
    cudaStreamSynchronize(stream);
    // EESEN_B200_TRACE_FILE=<path>: one line per launch since the last collect -- stream (0 main, 1 side), category,
    // start and duration in ms relative to the first launch: the timeline of a step without a profiler attached
    FILE *tf = nullptr;
    if (const char *tp = getenv("EESEN_B200_TRACE_FILE")) tf = fopen(tp, "a");
    if (tf) fprintf(tf, "# collect: %zu launches\n", prof_events.size());
    for (auto &e : prof_events) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, e.a, e.b) == cudaSuccess) { prof_ms[e.cat] += ms; prof_count[e.cat] += 1; }
      if (tf) {
        float t0 = 0.f;
        cudaEventElapsedTime(&t0, prof_events[0].a, e.a);
        fprintf(tf, "%d %d %.4f %.4f\n", e.st == side ? 1 : 0, e.cat, t0, ms);
      }
      prof_pool.push_back(e);
    }
    if (tf) fclose(tf);
    prof_events.clear();
  }

  // NCCL (dlopen'ed on demand)
  void *nccl_lib = nullptr;
  void *nccl_comm = nullptr;
  int rank = 0, nranks = 1;

  int fail(int code, const std::string &msg) {
    err = msg;
    return code;
  }
  int check(cudaError_t e, const char *what) {
    if (e == cudaSuccess) return 0;
    err = std::string(what) + ": " + cudaGetErrorString(e);
    return (int)e;
  }
  // grow-only scratch; stream-ordered reuse is safe because everything runs on `stream`
  int reserve(Buf &b, size_t bytes, void **out) {
    if (bytes > b.bytes) {
      if (b.p) {
        cudaError_t e = cudaStreamSynchronize(stream);
        if (e == cudaSuccess && side) e = cudaStreamSynchronize(side);
        if (e != cudaSuccess) return check(e, "cudaStreamSynchronize");
        cudaFree(b.p);
        b.p = nullptr;
        b.bytes = 0;
      }
      size_t want = bytes + bytes / 8 + 256;
      cudaError_t e = cudaMalloc(&b.p, want);
      if (e != cudaSuccess) return check(e, "cudaMalloc(workspace)");
      b.bytes = want;
    }
    *out = b.p;
    return 0;
  }
};

#endif
