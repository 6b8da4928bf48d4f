// eesen_b200/csrc/ce.cu -- frame-level cross-entropy on softmax posteriors, one fused pass.
//
// Replaces CE::EvalParallel (reference src/net/ce-loss.cc:94-169) for one packed minibatch
// (row r = t*S + s, valid iff t < len[s]):
//   diff = (y - onehot(target)) * mask        target matrix upload, AddMat, mask upload, MulRowsVec
//   correct += [FindRowMaxId(y) == target]    FindRowMaxId + D2H of the ids + host loop
//   obj -= log y[target]                      ApplyLog, MulElements, MulRowsVec, Sum
// with two launches.  ce_kernel: one warp per row, 16-byte loads and stores; per-CTA partial sums go to a
// workspace and ce_finish_kernel adds them up in a fixed order, so the statistics are the same bits from run to
// run.  The objective reads the target column only: a posterior that underflows to 0 elsewhere in the row
// cannot turn it into NaN (log 0 * 0 in the reference).
#include "common.cuh"
#include "kernels.h"

namespace eb {

namespace {

constexpr int kCeWarps = 8;   // rows in flight per CTA
constexpr int kCeUnroll = 4;  // float4 loads in flight per lane

__global__ void __launch_bounds__(kCeWarps * 32)
ce_kernel(int T, int S, int K, const int *__restrict__ len, const float *__restrict__ probs, int ldp,
          const int *__restrict__ targets, float *__restrict__ diff, int ldd, double *__restrict__ part_obj,
          unsigned long long *__restrict__ part_cnt) {
  __shared__ double obj_sm[kCeWarps];
  __shared__ unsigned long long cnt_sm[kCeWarps][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long N = (long)T * S;
  const int nvec = K >> 2;   // whole float4 columns; the K % 4 tail is done with scalar accesses
  double obj = 0.0;
  unsigned long long correct = 0, valid = 0;
  for (long row = (long)blockIdx.x * kCeWarps + warp; row < N; row += (long)gridDim.x * kCeWarps) {
    const int t = (int)(row / S), s = (int)(row - (long)t * S);
    float *drow = diff + row * ldd;
    if (t >= len[s]) {   // padded row: exactly 0, nothing read
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int c = lane; c < nvec; c += 32) reinterpret_cast<float4 *>(drow)[c] = z;
      for (int k = 4 * nvec + lane; k < K; k += 32) drow[k] = 0.f;
      continue;
    }
    const int tgt = targets[row];
    const bool in_range = (unsigned)tgt < (unsigned)K;
    const float *yrow = probs + row * ldp;
    // first index of the row maximum (the tie rule of row_argmax_kernel / FindRowMaxId): each lane scans its
    // columns in increasing order with a strict >, the shuffle tree prefers the lower index on equal values
    float mx = -INFINITY;
    int mi = 0x7fffffff;
    for (int c0 = lane; c0 < nvec; c0 += 32 * kCeUnroll) {
      float4 v[kCeUnroll];
#pragma unroll
      for (int u = 0; u < kCeUnroll; u++) {
        const int c = c0 + 32 * u;
        if (c < nvec) v[u] = __ldg(reinterpret_cast<const float4 *>(yrow) + c);
      }
#pragma unroll
      for (int u = 0; u < kCeUnroll; u++) {
        const int c = c0 + 32 * u;
        if (c < nvec) {
          const int k = 4 * c;
          if (v[u].x > mx) { mx = v[u].x; mi = k; }
          if (v[u].y > mx) { mx = v[u].y; mi = k + 1; }
          if (v[u].z > mx) { mx = v[u].z; mi = k + 2; }
          if (v[u].w > mx) { mx = v[u].w; mi = k + 3; }
          float4 d = v[u];   // y - 1 on the target column, y elsewhere: AddMat(-1, onehot) bit for bit
          if (tgt == k) d.x -= 1.f;
          if (tgt == k + 1) d.y -= 1.f;
          if (tgt == k + 2) d.z -= 1.f;
          if (tgt == k + 3) d.w -= 1.f;
          reinterpret_cast<float4 *>(drow)[c] = d;
        }
      }
    }
    for (int k = 4 * nvec + lane; k < K; k += 32) {
      const float y = yrow[k];
      if (y > mx) { mx = y; mi = k; }
      drow[k] = tgt == k ? y - 1.f : y;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float ov = __shfl_xor_sync(0xffffffffu, mx, o);
      int oi = __shfl_xor_sync(0xffffffffu, mi, o);
      if (ov > mx || (ov == mx && oi < mi)) { mx = ov; mi = oi; }
    }
    if (lane == 0) {
      // accurate logf (the reference's ApplyLog is log() in fp32); a target outside [0, K) is never read
      obj -= in_range ? (double)logf(yrow[tgt]) : (double)NAN;
      correct += (mi == tgt);
      valid += 1;
    }
  }
  if (lane == 0) { obj_sm[warp] = obj; cnt_sm[warp][0] = correct; cnt_sm[warp][1] = valid; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double o = 0.0;
    unsigned long long c = 0, v = 0;
    for (int w = 0; w < kCeWarps; w++) { o += obj_sm[w]; c += cnt_sm[w][0]; v += cnt_sm[w][1]; }
    part_obj[blockIdx.x] = o;
    part_cnt[2 * blockIdx.x] = c;
    part_cnt[2 * blockIdx.x + 1] = v;
  }
}

// one warp: lane-strided sums, then a fixed shuffle tree -- the same order on every run
__global__ void ce_finish_kernel(int nparts, const double *__restrict__ part_obj,
                                 const unsigned long long *__restrict__ part_cnt, double *__restrict__ stats) {
  const int lane = threadIdx.x;
  double o = 0.0;
  unsigned long long c = 0, v = 0;
  for (int i = lane; i < nparts; i += 32) { o += part_obj[i]; c += part_cnt[2 * i]; v += part_cnt[2 * i + 1]; }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    o += __shfl_xor_sync(0xffffffffu, o, off);
    c += __shfl_xor_sync(0xffffffffu, c, off);
    v += __shfl_xor_sync(0xffffffffu, v, off);
  }
  if (lane == 0) { stats[0] = o; stats[1] = (double)c; stats[2] = (double)v; }
}

int ce_grid(long N, int num_sms) {
  long want = (N + kCeWarps - 1) / kCeWarps;
  long cap = 8L * num_sms;   // 8 CTAs of 8 warps per SM keep enough 16-byte loads in flight to stream HBM
  return (int)(want < 1 ? 1 : (want < cap ? want : cap));
}

}  // namespace

size_t ce_workspace_bytes(int T, int S, int num_sms) {
  return (size_t)ce_grid((long)T * S, num_sms) * (sizeof(double) + 2 * sizeof(unsigned long long));
}

cudaError_t ce_eval(cudaStream_t st, int num_sms, int T, int S, int K, const int *len, const float *probs, int ldp,
                    const int *targets, float *diff, int ldd, double *stats, void *ws) {
  if (T <= 0 || S <= 0) return cudaMemsetAsync(stats, 0, 3 * sizeof(double), st);
  const int grid = ce_grid((long)T * S, num_sms);
  double *part_obj = static_cast<double *>(ws);
  unsigned long long *part_cnt = reinterpret_cast<unsigned long long *>(part_obj + grid);
  ce_kernel<<<grid, kCeWarps * 32, 0, st>>>(T, S, K, len, probs, ldp, targets, diff, ldd, part_obj, part_cnt);
  ce_finish_kernel<<<1, 32, 0, st>>>(grid, part_obj, part_cnt, stats);
  return cudaGetLastError();
}

}  // namespace eb
