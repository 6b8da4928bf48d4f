// eesen_b200/csrc/lstm_tc.cu -- persistent recurrent kernels on the 5th-generation tensor cores.
//
// Same contract as lstm.cu (reference BiLstmParallel::PropagateFncVanillaPass{Forward,Backward}
// bilstm-parallel-layer.h:112-149,166-205 and BackpropagateFncVanillaPass* :450-499,541-590 plus the
// bias / peephole reductions :507-510,598-601): ONE launch per layer and pass runs all T
// steps of both directions.  What changes is the per-step product m_{t-1} * Wm^T (forward) and
// d(gates) * Wm (backward): it runs as tcgen05.mma kind::f16 with the accumulator in TMEM instead
// of 60 warp-level mma.sync per warp and step.
//
// Decomposition: CTA(dir, group, slice) owns 32 cells (= 128 gate rows = one M=128 tile) of one direction
// for a group of 16 utterances.  Its rows of Wm stay resident in TENSOR MEMORY for the whole sequence ("TS" form MMAs;
// the tiles that do not fit at 384 / 512 cells stay in shared memory) as fp16 pairs
//   W = W_hi + 2^-11 * W_lo'        W_hi = fp16(W),  W_lo' = fp16((W - W_hi) * 2^11)
// and the per-step activations are split the same way, stacked along N in a K-major SWIZZLE_128B tile:
//   B = [ x_hi (16 utterances) ; x_lo' (16 utterances) ]          (32 x K, K-major)
// Two MMAs per 16-wide k-slice:  X += W_hi * B  (N = 32: hi*hi | hi*lo'),  Y += W_lo' * B[0:16]  (N = 16:
// lo'*hi); result = X[:, u] + 2^-11 * (X[:, 16+u] + Y[:, u]) -- the dropped lo'*lo' term is 2^-22 relative,
// the same fidelity class as the 3xTF32 split of lstm.cu (both operands carry 22 mantissa bits; fp16 x fp16
// products are exact in the fp32 accumulator).  Forward: |m| < 1, so fp16 never overflows.  Backward:
// d(gates) has no fixed range, so every utterance column is scaled by its own power of two (exact) to
// [2^13, 2^14) before the split and scaled back in the epilogue.  (One instruction cannot mix fp16 and bf16
// operands on sm_100a -- measured, tests/micro/umma_probe.cu -- hence the scaling instead of a bf16 split.)
//
// Exchange between the CTAs of one (dir, group), two implementations behind the template parameter CL:
//   CL = 1 (default up to 384 cells): the CTAs form ONE thread-block cluster and push m_t / the partial d_m straight into
//          each other's shared memory -- st.async with complete_tx on the destination's mbarrier, receive tiles
//          double-buffered by step parity; no polling, no grid-wide co-residency (see the kernels' comments);
//   CL = 0 (512 cells, or when the clusters of a pass are not all co-resident): "LL" style tagged words through L2 as
//          in lstm.cu, but 4 bytes wide -- the step tag is ONE bit that replaces the least significant bit of the
//          payload (of lo' forward: 2^-21 relative; of the fp32 partial d_m backward: 2^-24 relative); a buffer is
//          reused every second step with the bit flipped ((step >> 1) & 1), buffers start as 0xFF bytes; cooperative launch.
// 256 threads: every warp evaluates the gates (two (cell, utterance) pairs per thread) and owns a part of the TMEM ->
// register epilogue (lane quadrant = warp % 4); warp 0 additionally allocates TMEM and issues the MMAs from one elected
// lane (and, in the backward kernel, leaves its share of the epilogue to warp 4).
#include <cuda_fp16.h>

#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "kernels.h"
#include "tc_common.cuh"

namespace eb {

#ifdef EB_LSTM_TIMING
// debug build only (make TIMING=1): per-phase clock64 deltas of thread 0 of CTA (0,0,0), accumulated in REGISTERS
// and written once at the end (a global read-modify-write per tick would stall the MMA-issuing warp on an L2 round
// trip five times per step)
__device__ long long g_lstm_tc_timing[2][16];
#define TC_T0() long long tk_ = clock64()
#define TC_ACC_DECL() long long tacc_[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}
#define TC_TICK(kernel, i)                                                          \
  do {                                                                              \
    if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) {        \
      long long n_ = clock64();                                                     \
      tacc_[i] += n_ - tk_;                                                         \
      tk_ = n_;                                                                     \
    }                                                                               \
  } while (0)
#define TC_COUNT(i) tacc_[i] += 1
// second observer (thread 128 = warp 4 of CTA (0,0,0)): cycles from the moment thread 0 starts issuing the MMAs of a step
// (TC_MARK) to the moment this thread sees the commit of tile bi (TC_SEEN), accumulated in slots 12 + bi
#define TC_MARK_DECL() __shared__ long long tc_mark_; long long tseen_[4] = {0, 0, 0, 0}
#define TC_MARK() do { if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) *(volatile long long *)&tc_mark_ = clock64(); } while (0)
#define TC_SEEN(bi) do { if (tid == 128 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) tseen_[bi] += clock64() - *(volatile long long *)&tc_mark_; } while (0)
#define TC_SEEN_FLUSH(kernel) do { if (tid == 128 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) for (int i_ = 0; i_ < 4; i_++) g_lstm_tc_timing[kernel][12 + i_] += tseen_[i_]; } while (0)
// the same observer's own epilogue phases (backward kernel; slots 12..15 of the FORWARD table, which that kernel leaves
// alone): 0 commit wait, 1 TMEM loads, 2 arithmetic, 3 pushes
#define TC_OBS_DECL() long long tobs_[4] = {0, 0, 0, 0}, tol_ = 0
#define TC_OBS_START() do { if (tid == 128) tol_ = clock64(); } while (0)
#define TC_OBS(i) do { if (tid == 128) { long long n_ = clock64(); tobs_[i] += n_ - tol_; tol_ = n_; } } while (0)
#define TC_OBS_FLUSH() do { if (tid == 128 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) for (int i_ = 0; i_ < 4; i_++) g_lstm_tc_timing[0][12 + i_] += tobs_[i_]; } while (0)
#define TC_FLUSH(kernel)                                                            \
  do {                                                                              \
    if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0)          \
      for (int i_ = 0; i_ < 12; i_++) g_lstm_tc_timing[kernel][i_] += tacc_[i_];     \
  } while (0)
#else
#define TC_T0()
#define TC_ACC_DECL()
#define TC_TICK(kernel, i)
#define TC_COUNT(i)
#define TC_FLUSH(kernel)
#define TC_MARK_DECL()
#define TC_MARK()
#define TC_SEEN(bi)
#define TC_SEEN_FLUSH(kernel)
#define TC_OBS_DECL()
#define TC_OBS_START()
#define TC_OBS(i)
#define TC_OBS_FLUSH()
#endif

namespace {

constexpr int TCL_CS = 32;        // cells per slice (x 4 gates = the 128 rows of one UMMA tile)
constexpr int TCL_UG = 16;        // utterances per group
constexpr int TCL_WORKERS = 256;  // worker threads (8 warps)
constexpr int TCL_THREADS = TCL_WORKERS;   // 8 warps = 2 per SM sub-partition (a 9th warp would cap every thread at 168 registers)
constexpr float kLoScale = 2048.f, kLoUnscale = 1.f / 2048.f;

// byte offset of element (row r, k) of a K-major SWIZZLE_128B tile of 16-bit elements with `rows` rows:
// 64-wide k-blocks of rows*128 bytes, 8-row atoms of 1024 bytes, 16-byte chunks XOR-swizzled by (row & 7)
__device__ __forceinline__ uint32_t sw128_off(int rows, int r, int k) {
  const int kb = k >> 6, kk = k & 63;
  return (uint32_t)(kb * rows * 128 + (r >> 3) * 1024 + (r & 7) * 128 + ((((kk >> 3) ^ (r & 7)) << 4)) + ((kk & 7) << 1));
}

__device__ __forceinline__ void split_f16(float x, uint32_t &hi, uint32_t &lo) {
  const __half h = __float2half_rn(x);
  hi = (uint32_t)__half_as_ushort(h);
  lo = (uint32_t)__half_as_ushort(__float2half_rn((x - __half2float(h)) * kLoScale));
}

// instruction descriptor, kind::f16: D = F32, A = B = F16, both K-major
__device__ __forceinline__ uint32_t idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// 4-byte exchange words, relaxed at gpu scope (served by L2, never by a stale L1 line)
__device__ __forceinline__ void st_word(uint32_t *p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.b32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint4 ld_word4(const uint4 *p) {
  uint4 q;
  asm volatile("ld.relaxed.gpu.global.v4.b32 {%0, %1, %2, %3}, [%4];\n"
               : "=r"(q.x), "=r"(q.y), "=r"(q.z), "=r"(q.w) : "l"(p) : "memory");
  return q;
}

// A operand resident in TMEM ("TS" form): lane = row, two fp16 per 32-bit column, 8 columns per 16-wide k-slice
// (layout and speed measured in tests/micro/umma_probe.cu: the 40 MMAs of one step complete in ~830 cycles with the
// weights in TMEM against ~2700 with both operands in shared memory, where the 160 KB weight stream is the limit)
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n.reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&w)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};\n" ::"r"(taddr), "r"(w[0]), "r"(w[1]),
               "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
               : "memory");
}
// NLO = number of leading k-slices whose W_lo' sits in TMEM; the remaining ones (C = 512: TMEM is full) are read from
// the shared-memory tile dWloS ("SS" form).
// (Measured, tests/micro/umma_probe.cu + profiles/r02_d_chains.txt: these small MMAs are ISSUE-bound, ~22-27 cycles per
// instruction whatever N (16..64) and whether or not consecutive ones hit the same accumulator -- splitting K over four
// independent accumulator chains, or interleaving the tiles of the backward step, changed nothing and was removed.)
template <int KB, int NLO>
__device__ __forceinline__ void issue_fwd_mmas_ts(uint32_t tWhi, uint32_t tWlo, uint64_t dWloS, uint64_t dB, uint32_t tmem,
                                                  uint32_t idN, uint32_t idH) {
#pragma unroll
  for (int kb = 0; kb < KB; kb++) {
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
      const uint64_t bd = dB + (uint64_t)((kb * 4096 + ks * 32) >> 4);
      umma_f16_ts(tmem, tWhi + (kb * 4 + ks) * 8, bd, idN, (kb | ks) != 0);
      if (kb * 4 + ks < NLO)
        umma_f16_ts(tmem + 32, tWlo + (kb * 4 + ks) * 8, bd, idH, (kb | ks) != 0);
      else
        umma_f16(tmem + 32, dWloS + (uint64_t)((((kb * 4 + ks - NLO) >> 2) * 16384 + ks * 32) >> 4), bd, idH, (kb | ks) != 0);
    }
  }
}

// One recurrent step's MMAs from the elected lane: fully unrolled, descriptors = 64-bit base + constant
// (SASS: back-to-back UTCHMMA with one UIADD3.64 in between; a loop with run-time offsets costs ~45 clk per MMA).
template <int KB>
__device__ __forceinline__ void issue_fwd_mmas(uint64_t dWhi, uint64_t dWlo, uint64_t dB, uint32_t tmem, uint32_t idN,
                                               uint32_t idH) {
#pragma unroll
  for (int kb = 0; kb < KB; kb++) {
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
      const uint64_t bd = dB + (uint64_t)((kb * 4096 + ks * 32) >> 4);
      umma_f16(tmem, dWhi + (uint64_t)((kb * 16384 + ks * 32) >> 4), bd, idN, (kb | ks) != 0);
      umma_f16(tmem + 32, dWlo + (uint64_t)((kb * 16384 + ks * 32) >> 4), bd, idH, (kb | ks) != 0);
    }
  }
}
__device__ __forceinline__ void issue_bwd_tile_ts(uint32_t tAhi, uint32_t tAlo, uint64_t dB, uint32_t tmem) {
  const uint32_t idN = idesc_f16(128, 32), idH = idesc_f16(128, 16);
#pragma unroll
  for (int ks = 0; ks < 8; ks++) {
    const int kb = ks >> 2, k4 = ks & 3;
    const uint64_t bd = dB + (uint64_t)((kb * 4096 + k4 * 32) >> 4);
    umma_f16_ts(tmem, tAhi + ks * 8, bd, idN, ks != 0);
    umma_f16_ts(tmem + 32, tAlo + ks * 8, bd, idH, ks != 0);
  }
}
// "stacked" tile for the last 64 rows when C % 128 == 64: ONE M = 128 operand in TMEM whose lanes 0-63 hold the hi
// halves of the 64 rows and lanes 64-127 their lo' halves, so that a single N = 32 MMA per k-slice yields hi*hi | hi*lo'
// (lanes 0-63) and lo'*hi (lanes 64-127, columns 0-15; columns 16-31 there are the dropped lo'*lo' term)
__device__ __forceinline__ void issue_bwd_tile_stacked(uint32_t tA, uint64_t dB, uint32_t tmem) {
  const uint32_t idN = idesc_f16(128, 32);
#pragma unroll
  for (int ks = 0; ks < 8; ks++) {
    const int kb = ks >> 2, k4 = ks & 3;
    umma_f16_ts(tmem, tA + ks * 8, dB + (uint64_t)((kb * 4096 + k4 * 32) >> 4), idN, ks != 0);
  }
}
__device__ __forceinline__ void issue_bwd_tile(uint64_t dAhi, uint64_t dAlo, uint64_t dB, uint32_t tmem) {
  const uint32_t idN = idesc_f16(128, 32), idH = idesc_f16(128, 16);
#pragma unroll
  for (int ks = 0; ks < 8; ks++) {
    const int kb = ks >> 2, k4 = ks & 3;
    const uint64_t bd = dB + (uint64_t)((kb * 4096 + k4 * 32) >> 4);
    umma_f16(tmem, dAhi + (uint64_t)((kb * 16384 + k4 * 32) >> 4), bd, idN, ks != 0);
    umma_f16(tmem + 32, dAlo + (uint64_t)((kb * 16384 + k4 * 32) >> 4), bd, idH, ks != 0);
  }
}

// spin until *p == v (acquire at gpu scope: what the stream that stored v wrote before is visible afterwards).
// Bounded: a producer that never comes (a host-side sequencing bug) ends in a trap after ~4 s, not in a hung device.
__device__ __forceinline__ void wait_flag(const unsigned *p, unsigned v) {
  unsigned x;
  const long long t0 = clock64();
  for (;;) {
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];\n" : "=r"(x) : "l"(p) : "memory");
    if (x == v) break;
    if (clock64() - t0 > (1ll << 33)) __trap();
  }
}
// mbarrier wait on bytes that peers of the cluster push (st.async complete_tx); bounded like wait_flag
__device__ __forceinline__ void mbar_wait_peers(uint64_t *bar, uint32_t parity) {
  uint32_t done;
  long long t0 = 0;
  for (;;) {
    asm volatile(
        "{\n.reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (done) break;
    if (t0 == 0) t0 = clock64();
    else if (clock64() - t0 > (1ll << 33)) __trap();
  }
}
__global__ void set_flag_kernel(unsigned *flag, unsigned value) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;\n" ::"l"(flag), "r"(value) : "memory");
}

__device__ __forceinline__ void named_bar_workers() { asm volatile("bar.sync 1, 256;\n" ::: "memory"); }

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }


// ------------------------------------------------------------------------------------ forward
// WIDE = 1: 384 < C <= 512 (4 exchange chunks per thread; at C = 512 the last 8 k-slices of W_lo' in shared memory)
// CL = 1: the `slices` CTAs of one (dir, group) are ONE thread-block cluster and exchange m_t through distributed shared
// memory instead of L2: every warp pushes the hi / lo' halves of its 2 utterances x 32 cells as 16-byte st.async stores
// straight into the (double-buffered) B tile of all CTAs of the cluster, complete_tx on the destination's mbarrier; the
// MMA-issuing warp sleeps on that mbarrier -- no polling, no staging pass, no grid-wide co-residency requirement.
// Measured ping-pong (tests/micro/cluster_exchange2.cu, 8 clusters of 10 CTAs): 1.63 k cycles per step against 2.80 k
// (mean; slowest CTA 4.0 k) for the tagged words through L2.
template <int DROP, int WIDE, int CL>
__global__ void __launch_bounds__(TCL_THREADS, 1)
lstm_tc_fwd_kernel(LstmFwdArgs a, int groups, int ndir) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment by pointer arithmetic ON the __shared__ array: a round trip through uintptr_t loses the address
  // space and every access below would compile to generic LD.E / ST.E instead of LDS / STS
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int C = a.C, S = a.S, T = a.T;
  const int KB = C >> 6;                                  // 64-wide k-blocks (C % 64 == 0)
  uint8_t *Bt = smem;                                     // [CL ? 2 : 1][KB][32 rows][128 B]: rows 0-15 hi, 16-31 lo'
  const uint32_t bt_bytes = (uint32_t)KB * 4096u;
  float *stg = reinterpret_cast<float *>(Bt + (size_t)(CL ? 2 : 1) * bt_bytes);   // [4 gates][16 utts][32 cells]
  uint8_t *pub = reinterpret_cast<uint8_t *>(stg) + 8192;  // (CL) [8 warps][hi | lo'][2 utts][32 cells] fp16: 256 B per warp
  // TMEM columns: [0,32) X accumulator, [32,48) Y accumulator, [64, 64 + C/2) W_hi, [64 + C/2, ..) W_lo' of the first
  // nlo k-slices (all of them up to C = 448; 24 of 32 at C = 512, the other 8 in the shared-memory tile WloS)
  constexpr uint32_t kColW = 64;
  const int nks = C >> 4;
  const int nlo = (WIDE && nks > 28) ? 24 : nks;
  uint8_t *WloS = Bt + (size_t)KB * 4096 + 8192;                     // [k-blocks from slice nlo on][128 rows][128 B]
  __shared__ uint64_t b_full, mma_done, xfull[2];
  const uint32_t slices = gridDim.x, xbytes = slices * 2048u;        // (CL) bytes a CTA receives per step
  __shared__ uint32_t tmem_base_sm;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slice = blockIdx.x, group = blockIdx.y, dir = blockIdx.z;
  const LstmDirParams P = a.p[dir];
  uint32_t *xbuf = reinterpret_cast<uint32_t *>(a.xbuf);  // [2 parity][ndir][groups][16][C] 4-byte tagged words
  const int s0 = a.s_begin, s1 = a.s_begin + a.s_count;

  for (int idx = tid; idx < (CL ? 2 : 1) * KB * 1024; idx += TCL_THREADS) reinterpret_cast<uint32_t *>(Bt)[idx] = 0u;
  if (tid == 0) {
    mbar_init(&b_full, TCL_WORKERS);
    mbar_init(&mma_done, 1);
    mbar_init(&xfull[0], 1);
    mbar_init(&xfull[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    if (CL) {   // m_0 lands in tile 0, m_1 in tile 1; each tile is re-armed when its MMAs have been issued
      mbar_expect_tx(&xfull[0], xbytes);
      mbar_expect_tx(&xfull[1], xbytes);
    }
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&tmem_base_sm)), "n"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem_base = tmem_base_sm;
  if (CL) cluster_sync_all();   // every CTA of the cluster has its barriers armed and its tiles zeroed before anyone pushes

  // ---- resident weights, in TMEM for the whole sequence: lane = gate*32 + local cell, the row's K = C values split
  // into fp16 hi / lo' and packed two per column.  Warps w and w+4 own the same lane quadrant: they take alternate
  // 16-wide k-slices.
  {
    const int r = (warp & 3) * 32 + lane;
    const float *wrow = P.wm + ((size_t)(r >> 5) * C + slice * TCL_CS + (r & 31)) * P.ldwm;
    const uint32_t tl = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + kColW;
    for (int ks = warp >> 2; ks < C / 16; ks += 2) {
      float w[16];
#pragma unroll
      for (int j = 0; j < 16; j++) w[j] = __ldg(wrow + ks * 16 + j);
      uint32_t wh[8], wl[8];
#pragma unroll
      for (int j = 0; j < 8; j++) {
        uint32_t h0, l0, h1, l1;
        split_f16(w[2 * j], h0, l0);
        split_f16(w[2 * j + 1], h1, l1);
        wh[j] = h0 | (h1 << 16);
        wl[j] = l0 | (l1 << 16);
      }
      tmem_st8(tl + ks * 8, wh);
      if (ks < nlo) {
        tmem_st8(tl + (C >> 1) + ks * 8, wl);
      } else {
        const int k0 = (ks - nlo) * 16;
        *reinterpret_cast<uint4 *>(WloS + sw128_off(128, r, k0)) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
        *reinterpret_cast<uint4 *>(WloS + sw128_off(128, r, k0 + 8)) = make_uint4(wl[4], wl[5], wl[6], wl[7]);
      }
    }
    asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // (WloS: generic-proxy writes -> UMMA reads)
  }
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");

  {
    // ===== workers =====
    const int cl = lane, up = warp;                        // gate phase: local cell, utterance pair
    const int cell = slice * TCL_CS + cl;
    int uidx[2], lenu[2];
    bool valid[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      uidx[e] = s0 + group * TCL_UG + 2 * up + e;
      valid[e] = uidx[e] < s1;
      lenu[e] = (a.len && valid[e]) ? a.len[uidx[e]] : 0;   // NULL: uni-directional (no masking)
    }
    const float ppi = P.pi[cell], ppf = P.pf[cell], ppo = P.po[cell];
    float cprev[2] = {0.f, 0.f};
    float pre[4][2];
    float rmk[2] = {1.f, 1.f};
    auto load_pre = [&](int t) {
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const float *row = a.G + ((size_t)t * S + (valid[e] ? uidx[e] : 0)) * a.ldg + (size_t)dir * 4 * C + cell;
#pragma unroll
        for (int q = 0; q < 4; q++) pre[q][e] = valid[e] ? __ldcs(row + (size_t)q * C) : 0.f;
        if (DROP != 0)
          rmk[e] = valid[e] ? __ldg(a.rmask + (size_t)(a.rmask_per_step ? (size_t)t * S + uidx[e] : (size_t)uidx[e]) * a.ldr +
                                    (size_t)dir * C + cell)
                            : 0.f;
      }
    };
    load_pre(dir == 0 ? 0 : T - 1);
    int ghave = a.gready - 1;                              // last chunk of G known to be complete
    const int c8n = C >> 3;                                // 8-cell chunks per utterance row
    const int quad = warp & 3, uh = warp >> 2;             // epilogue: TMEM lane quadrant (= gate), utterance half
    const uint64_t dBt0 = umma_desc(smem_u32(Bt), 16, 1024, 2);
    // exchange chunks of this thread (fixed for the whole sequence; L2 path)
    constexpr int MAXT = WIDE ? 4 : 3;                     // 16 * (C/8) / 256 <= 3 for C <= 384, 4 for C <= 512
    uint4 xq[MAXT][2];
    size_t xoff[MAXT];
    bool live[MAXT];
#pragma unroll
    for (int i = 0; i < MAXT; i++) {
      const int v = tid + i * TCL_WORKERS;
      const int u = v / c8n, c8 = v - u * c8n;
      live[i] = v < TCL_UG * c8n && s0 + group * TCL_UG + u < s1;
      xoff[i] = ((size_t)u * C + c8 * 8) / 4;
      xq[i][0] = make_uint4(0u, 0u, 0u, 0u); xq[i][1] = xq[i][0];
    }

    TC_ACC_DECL();
    for (int step = 0; step < T; step++) {
      const int t = dir == 0 ? step : T - 1 - step;
      float acc[4][2];
#pragma unroll
      for (int q = 0; q < 4; q++) { acc[q][0] = 0.f; acc[q][1] = 0.f; }
      TC_T0();
      if (step > 0) {
        if (!CL) {
        // ---- stage m_{t-1} of the group: spin on the tagged words, write the hi / lo' rows of the B tile
        const uint4 *xr = reinterpret_cast<const uint4 *>(
            xbuf + ((size_t)(((step - 1) & 1) * ndir + dir) * groups + group) * TCL_UG * C);
        const uint32_t want = (uint32_t)(((step - 1) >> 1) & 1) << 16;   // tag bit of the data produced at step-1
        // every thread owns up to 3 chunks (utterance u, 8 cells).  Their first loads went out at the end of the
        // previous step, right behind the publish and in front of the saved-state stores (the words need a round trip
        // through L2 anyway); whatever has not arrived by now is polled again
#pragma unroll
        for (int i = 0; i < MAXT; i++) {
          const int v = tid + i * TCL_WORKERS;
          if (v >= TCL_UG * c8n) continue;
          const int u = v / c8n, c8 = v - u * c8n;
          uint4 hi4 = make_uint4(0u, 0u, 0u, 0u), lo4 = hi4;
          if (live[i]) {
            while (((((xq[i][0].x ^ want) | (xq[i][0].y ^ want) | (xq[i][0].z ^ want) | (xq[i][0].w ^ want) |
                      (xq[i][1].x ^ want) | (xq[i][1].y ^ want) | (xq[i][1].z ^ want) | (xq[i][1].w ^ want)) & 0x10000u)) != 0u) {
              xq[i][0] = ld_word4(xr + xoff[i]); xq[i][1] = ld_word4(xr + xoff[i] + 1);
              TC_COUNT(5);   // (debug build: re-polls of thread 0)
            }
            hi4 = make_uint4(__byte_perm(xq[i][0].x, xq[i][0].y, 0x5410), __byte_perm(xq[i][0].z, xq[i][0].w, 0x5410),
                             __byte_perm(xq[i][1].x, xq[i][1].y, 0x5410), __byte_perm(xq[i][1].z, xq[i][1].w, 0x5410));
            // the tag bit (LSB of every lo' half) is cleared again: a zero stays an exact zero
            lo4 = make_uint4(__byte_perm(xq[i][0].x, xq[i][0].y, 0x7632) & 0xfffefffeu, __byte_perm(xq[i][0].z, xq[i][0].w, 0x7632) & 0xfffefffeu,
                             __byte_perm(xq[i][1].x, xq[i][1].y, 0x7632) & 0xfffefffeu, __byte_perm(xq[i][1].z, xq[i][1].w, 0x7632) & 0xfffefffeu);
          }
          const int k0 = c8 * 8;
          *reinterpret_cast<uint4 *>(Bt + sw128_off(32, u, k0)) = hi4;
          *reinterpret_cast<uint4 *>(Bt + sw128_off(32, 16 + u, k0)) = lo4;
        }
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // generic-proxy writes -> async proxy (UMMA)
        mbar_arrive(&b_full);
        }
        TC_TICK(0, 0);
        if (warp == 0) {
          // ===== MMA issue: 2 instructions per 16-wide k-slice, one commit =====
          if (CL) {
            // m_{t-1} of the whole group has landed in tile (step-1)&1 when the bytes armed on its mbarrier are complete
            mbar_wait_peers(&xfull[(step - 1) & 1], (uint32_t)(((step - 1) >> 1) & 1));
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // remote generic-proxy stores -> UMMA reads
            if (lane == 0) mbar_expect_tx(&xfull[(step - 1) & 1], xbytes);      // armed again for m_{t+1}
          } else {
            mbar_wait(&b_full, (uint32_t)((step - 1) & 1));
          }
          asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
          if (elect_one()) {
            const uint64_t dBt = dBt0 + (uint64_t)(CL ? ((uint32_t)((step - 1) & 1) * (bt_bytes >> 4)) : 0u);
            const uint32_t idN = idesc_f16(128, 32), idH = idesc_f16(128, 16);
            const uint32_t tWhi = tmem_base + kColW, tWlo = tmem_base + kColW + (uint32_t)(C >> 1);
            const uint64_t dWloS = umma_desc(smem_u32(WloS), 16, 1024, 2);
            if (WIDE) {
              if (KB == 7) issue_fwd_mmas_ts<7, 28>(tWhi, tWlo, dWloS, dBt, tmem_base, idN, idH);
              else issue_fwd_mmas_ts<8, 24>(tWhi, tWlo, dWloS, dBt, tmem_base, idN, idH);
            } else {
              switch (KB) {
                case 1: issue_fwd_mmas_ts<1, 4>(tWhi, tWlo, dWloS, dBt, tmem_base, idN, idH); break;
                case 2: issue_fwd_mmas_ts<2, 8>(tWhi, tWlo, dWloS, dBt, tmem_base, idN, idH); break;
                case 3: issue_fwd_mmas_ts<3, 12>(tWhi, tWlo, dWloS, dBt, tmem_base, idN, idH); break;
                case 4: issue_fwd_mmas_ts<4, 16>(tWhi, tWlo, dWloS, dBt, tmem_base, idN, idH); break;
                case 5: issue_fwd_mmas_ts<5, 20>(tWhi, tWlo, dWloS, dBt, tmem_base, idN, idH); break;
                default: issue_fwd_mmas_ts<6, 24>(tWhi, tWlo, dWloS, dBt, tmem_base, idN, idH); break;
              }
            }
            umma_commit(&mma_done);
          }
          __syncwarp();
        }
        // ---- the product runs on the tensor pipe; wait for its commit
        mbar_wait(&mma_done, (uint32_t)((step - 1) & 1));
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        TC_TICK(0, 1);
        {
          uint32_t x0[8], x1[8], y0[8];
          const uint32_t tl = tmem_base + ((uint32_t)(quad * 32) << 16);
          tmem_ld8(tl + 8 * uh, x0);
          tmem_ld8(tl + 16 + 8 * uh, x1);
          tmem_ld8(tl + 32 + 8 * uh, y0);
          tmem_ld_wait();
          asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
          float *dst = stg + ((size_t)(quad * TCL_UG + 8 * uh)) * 32 + lane;
#pragma unroll
          for (int j = 0; j < 8; j++)
            dst[j * 32] = u2f(x0[j]) + (u2f(x1[j]) + u2f(y0[j])) * kLoUnscale;
        }
        named_bar_workers();
#pragma unroll
        for (int q = 0; q < 4; q++) {
          acc[q][0] = stg[(q * TCL_UG + 2 * up) * 32 + cl];
          acc[q][1] = stg[(q * TCL_UG + 2 * up + 1) * 32 + cl];
        }
        TC_TICK(0, 2);
      }

      // ---- gates, cell update (bilstm-parallel-layer.h:127-147), padding mask of the backward cells (:201-204)
      float sg[2], si[2], sf[2], so[2], sc[2], sm[2];
#pragma unroll
      for (int e = 0; e < 2; e++) {
        float yg = pre[0][e] + acc[0][e];
        float yi = pre[1][e] + acc[1][e] + cprev[e] * ppi;
        float yf = pre[2][e] + acc[2][e] + cprev[e] * ppf;
        float gi = sigmoidf_(yi), gf = sigmoidf_(yf), gg = tanhf_(yg);
        float c;
        if (DROP == 0) c = gg * gi + cprev[e] * gf;
        else if (DROP == 1) c = rmk[e] * (gg * gi) + cprev[e] * gf;
        else c = rmk[e] * (gg * gi + cprev[e] * gf);
        float h = tanhf_(c);
        float go = sigmoidf_(pre[3][e] + acc[3][e] + c * ppo);
        float m = h * go;
        const bool keep = valid[e] && !(dir == 1 && t >= lenu[e]);
        sg[e] = keep ? gg : 0.f; si[e] = keep ? gi : 0.f; sf[e] = keep ? gf : 0.f; so[e] = keep ? go : 0.f;
        sc[e] = keep ? c : 0.f; sm[e] = keep ? m : 0.f;
        cprev[e] = sc[e];
      }
      // fp16 planes of m for the dense products that read the layer output (LstmFwdArgs::out_hi): fixed scale 2^13
      auto store_planes = [&](int e, int tt) {
        if (a.out_hi) {
          const float xs = sm[e] * 8192.f;
          const __half h = __float2half_rn(xs);
          const size_t o = ((size_t)tt * S + uidx[e]) * a.ldh + (size_t)dir * C + cell;
          reinterpret_cast<__half *>(a.out_hi)[o] = h;
          reinterpret_cast<__half *>(a.out_lo)[o] = __float2half_rn(xs - __half2float(h));
        }
      };
      // only m is on the inter-CTA critical path: publish it first
      if (CL) {
        if (step + 1 < T) {
          // the warp's [hi | lo'][2 utts][32 cells] halves -> 16 chunks of 16 bytes in its own staging area, then lane
          // (chunk, half of the destinations) pushes its chunk into tile `step & 1` of every CTA of the cluster
          uint16_t *pw = reinterpret_cast<uint16_t *>(pub + warp * 256);
#pragma unroll
          for (int e = 0; e < 2; e++) {
            uint32_t h, l;
            split_f16(sm[e], h, l);          // (sm = 0 for padded / absent utterances: the rows are zeros)
            pw[e * 32 + cl] = (uint16_t)h;
            pw[(2 + e) * 32 + cl] = (uint16_t)l;
          }
          __syncwarp();
          const int ch = lane & 15;                        // chunk = (kind, e, 8-cell group)
          const uint4 v = *reinterpret_cast<const uint4 *>(pub + warp * 256 + ch * 16);
          const int row = (ch >> 3) * 16 + 2 * up + ((ch >> 2) & 1);
          const uint32_t la = smem_u32(Bt) + (uint32_t)(step & 1) * bt_bytes + sw128_off(32, row, slice * TCL_CS + (ch & 3) * 8);
          const uint32_t lb = smem_u32(&xfull[step & 1]);
          for (uint32_t d = (uint32_t)(lane >> 4); d < slices; d += 2) st_async16(mapa_u32(la, d), v, mapa_u32(lb, d));
          __syncwarp();   // (the staging area is rewritten at the next step)
        }
#pragma unroll
        for (int e = 0; e < 2; e++)
          if (valid[e]) { __stcs(a.out + ((size_t)t * S + uidx[e]) * a.ldo + (size_t)dir * C + cell, sm[e]); store_planes(e, t); }
      } else {
#pragma unroll
      for (int e = 0; e < 2; e++) {
        if (valid[e]) {
          if (step + 1 < T) {
            uint32_t h, l;
            split_f16(sm[e], h, l);
            st_word(xbuf + (((size_t)((step & 1) * ndir + dir) * groups + group) * TCL_UG) * C + (size_t)(2 * up + e) * C + cell,
                    h | ((l & 0xfffeu) << 16) | ((uint32_t)((step >> 1) & 1) << 16));   // tag = LSB of lo'
          }
          __stcs(a.out + ((size_t)t * S + uidx[e]) * a.ldo + (size_t)dir * C + cell, sm[e]);
          store_planes(e, t);
        }
      }
      }
      auto first_poll = [&]() {   // first poll of the words the group is publishing right now (consumed at the next step)
        const uint4 *xn = reinterpret_cast<const uint4 *>(xbuf + ((size_t)((step & 1) * ndir + dir) * groups + group) * TCL_UG * C);
#pragma unroll
        for (int i = 0; i < MAXT; i++)
          if (live[i]) { xq[i][0] = ld_word4(xn + xoff[i]); xq[i][1] = ld_word4(xn + xoff[i] + 1); }
      };
      if (!CL && step + 1 < T) first_poll();
      TC_TICK(0, 3);
#pragma unroll
      for (int e = 0; e < 2; e++) {
        if (valid[e]) {
          float *grow = a.G + ((size_t)t * S + uidx[e]) * a.ldg + (size_t)dir * 4 * C + cell;
          __stcs(grow, sg[e]); __stcs(grow + (size_t)C, si[e]);
          __stcs(grow + (size_t)2 * C, sf[e]); __stcs(grow + (size_t)3 * C, so[e]);
          __stcs(a.cell + ((size_t)t * S + uidx[e]) * a.ldc + (size_t)dir * C + cell, sc[e]);
        }
      }
      if (step + 1 < T) {
        if (a.gflag) {   // streamed input product: the next position may lie in a chunk that is still being computed
          const int need = (step + 1) / a.gchunk;
          if (need > ghave) { wait_flag(a.gflag + need, a.gepoch); ghave = need; }
        }
        load_pre(dir == 0 ? t + 1 : t - 1);
      }
      TC_TICK(0, 4);
    }
    TC_FLUSH(0);
  }

  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  if (CL) cluster_sync_all();   // no CTA leaves while a peer could still address its shared memory
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(512) : "memory");
  }
}

// ------------------------------------------------------------------------------------ backward
// Partial d_m of ALL C cells from this CTA's 128 gate rows:  P[j, u] = sum_r Wm[r, j] * D[u, r]
// A = Wm^T tiles [j rows x 128 k] (hi, lo'): M tiles of 128 rows, the first two resident in TMEM, a third full one
// (C = 384) in shared memory; the 64 rows left when C % 128 == 64 form a "stacked" TMEM tile (hi in lanes 0-63, lo' in
// lanes 64-127);  B = D (scaled per utterance, hi rows 0-15 | lo' rows 16-31) [32 x 128 k].
// WIDE = 1: 384 < C <= 512 (up to 4 M tiles: 192 accumulator columns, two tiles in shared memory; 16 producers)
// CL = 1: the `slices` CTAs of one (dir, group) are one thread-block cluster (see lstm_tc_fwd_kernel); the partial d_m
// rows a CTA computed for the cells of CTA d go straight into d's receive buffer R[parity][producer][32 cells][16 utts]
// (row stride 80 bytes) as two 16-byte st.async stores per thread and tile -- the 32 accumulator rows of a warp's TMEM lane
// quadrant are exactly the 32 cells of ONE destination -- and the owner adds the `slices` blocks in producer order.
template <int DROP, int WIDE, int CL>
__global__ void __launch_bounds__(TCL_THREADS, 1)
lstm_tc_bwd_kernel(LstmBwdArgs a, int groups, int slices, int ndir) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment by pointer arithmetic ON the __shared__ array: a round trip through uintptr_t loses the address
  // space and every access below would compile to generic LD.E / ST.E instead of LDS / STS
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int C = a.C, S = a.S, T = a.T;
  const int n128 = C >> 7, rem64 = (C & 127) ? 1 : 0, MT = n128 + rem64;
  const int NTS = n128 < 2 ? n128 : 2;                    // full tiles resident in TMEM
  uint8_t *Bt = smem;                                     // [2 k-blocks][32 rows][128 B]
  // [2 step parities][16] inverse column scales.  Two sets: a warp may write the scales of step s+1 while another warp of
  // the CTA has not yet read those of step s in its epilogue -- with the cluster exchange a warp's gather depends only on
  // the two warps of every CTA that own its cells' accumulator rows, not on all warps of its own CTA (found by
  // compute-sanitizer timing on C = 256 / 384, where no stacked-tile barrier hides it; two sets suffice: step s+2's scales
  // are written behind b_full of step s+1, which every thread reaches after its epilogue of step s)
  float *scl = reinterpret_cast<float *>(Bt + 8192);
  float *gsm = scl + 32;                                  // [2 halves][16 utts][32 cells] gathered partial d_m
  float *ysm = gsm + 2 * TCL_UG * 32;                     // [16 utts][64 rows] lo'*hi part of the stacked tile
  float *red = ysm + TCL_UG * 64;                         // [7][16 utts][32 cells] bias / peephole sums at the end
  uint8_t *Ahi = smem + 32768;                            // full tiles beyond the TMEM-resident ones: [2 k-blocks][128][128 B] each
  uint8_t *Alo = Ahi + (size_t)(n128 - NTS) * 32768;
  constexpr int kRRow = 20, kRBlk = 32 * kRRow;           // (CL) floats per cell row (16 utts + pad: 80 B) / per producer block
  // (CL) [2 parity][slices][32 cells][kRRow], behind 32 KB of unused padding: kept so that tc_bwd_smem, and with it which
  // plans fit (occupancy, cluster eligibility), stays as measured
  float *R = reinterpret_cast<float *>(Alo + (size_t)(n128 - NTS) * 32768 + 32768);
  const uint32_t rbytes = (uint32_t)slices * 2048u;       // (CL) payload bytes a CTA receives per step
  __shared__ uint64_t b_full, mma_done[4], rfull[2];   // one commit barrier per M tile (at most 4 tiles)
  __shared__ uint32_t tmem_base_sm;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slice = blockIdx.x, group = blockIdx.y, dir = blockIdx.z;
  const LstmDirParams P = a.p[dir];
  uint32_t *pbuf = reinterpret_cast<uint32_t *>(a.pbuf);  // [2 parity][ndir][groups][slices][16][C] partial d_m, tag in the LSB
  const int s0 = a.s_begin, s1 = a.s_begin + a.s_count;

  // A[j, k = gate*32 + c] = Wm[gate*C + slice*32 + c][j]   (j fastest: coalesced reads of the Wm rows, 8 in flight)
  for (int mt = NTS; mt < n128; mt++) {
    for (int base = 0; base < 128 * 128; base += 8 * TCL_THREADS) {
      float w[8];
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int idx = base + i * TCL_THREADS + tid;
        const int kk = idx >> 7, j = mt * 128 + (idx & 127);
        w[i] = __ldg(P.wm + ((size_t)(kk >> 5) * C + slice * TCL_CS + (kk & 31)) * P.ldwm + j);
      }
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int idx = base + i * TCL_THREADS + tid;
        const int kk = idx >> 7;
        uint32_t h, l;
        split_f16(w[i], h, l);
        const uint32_t off = (uint32_t)(mt - NTS) * 32768 + sw128_off(128, idx & 127, kk);
        *reinterpret_cast<uint16_t *>(Ahi + off) = (uint16_t)h;
        *reinterpret_cast<uint16_t *>(Alo + off) = (uint16_t)l;
      }
    }
  }
  for (int idx = tid; idx < 2048; idx += TCL_THREADS) reinterpret_cast<uint32_t *>(Bt)[idx] = 0u;
  if (tid == 0) {
    mbar_init(&b_full, TCL_WORKERS);
    for (int i = 0; i < 4; i++) mbar_init(&mma_done[i], 1);
    mbar_init(&rfull[0], 1);
    mbar_init(&rfull[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    if (CL) {   // the partials of step 0 land in buffer 0, of step 1 in buffer 1; re-armed after every gather
      mbar_expect_tx(&rfull[0], rbytes);
      mbar_expect_tx(&rfull[1], rbytes);
    }
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&tmem_base_sm)), "n"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem_base = tmem_base_sm;
  if (CL) cluster_sync_all();   // barriers of every CTA of the cluster armed before anyone pushes

  // ---- the first two full M tiles of Wm^T also go to TMEM (columns [160, 160 + 128 * NTS): per tile 64 columns hi,
  // 64 columns lo'; lane = output cell within the tile, 8 columns per 16-wide k-slice of this CTA's 128 gate rows):
  // their MMAs read the weights from TMEM ("TS" form) instead of streaming 128 KB through shared memory per step.
  // A third FULL tile (C = 384) keeps both operands in shared memory.
  constexpr uint32_t kColA = WIDE ? 192 : 160;   // behind the accumulators: 48 columns per full tile, 32 for the stacked one
  for (int mt = 0; mt < NTS; mt++) {
    const int j = mt * 128 + (warp & 3) * 32 + lane;
    const uint32_t tl = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + kColA + (uint32_t)mt * 128;
    for (int ks = warp >> 2; ks < 8; ks += 2) {
      float w[16];
#pragma unroll
      for (int i = 0; i < 16; i++) {
        const int kk = ks * 16 + i;
        w[i] = __ldg(P.wm + ((size_t)(kk >> 5) * C + slice * TCL_CS + (kk & 31)) * P.ldwm + j);
      }
      uint32_t wh[8], wl[8];
#pragma unroll
      for (int i = 0; i < 8; i++) {
        uint32_t h0, l0, h1, l1;
        split_f16(w[2 * i], h0, l0);
        split_f16(w[2 * i + 1], h1, l1);
        wh[i] = h0 | (h1 << 16);
        wl[i] = l0 | (l1 << 16);
      }
      tmem_st8(tl + ks * 8, wh);
      tmem_st8(tl + 64 + ks * 8, wl);
    }
  }
  // the stacked tile of the last 64 rows (columns [160 + 128 * NTS, + 64)): lane quadrants 0-1 hold hi, 2-3 lo'
  const uint32_t colS = kColA + (uint32_t)NTS * 128;
  if (rem64) {
    const int j = n128 * 128 + (warp & 1) * 32 + lane;
    const bool lo_half = (warp & 2) != 0;
    const uint32_t tl = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + colS;
    for (int ks = warp >> 2; ks < 8; ks += 2) {
      float w[16];
#pragma unroll
      for (int i = 0; i < 16; i++) {
        const int kk = ks * 16 + i;
        w[i] = __ldg(P.wm + ((size_t)(kk >> 5) * C + slice * TCL_CS + (kk & 31)) * P.ldwm + j);
      }
      uint32_t wv[8];
#pragma unroll
      for (int i = 0; i < 8; i++) {
        uint32_t h0, l0, h1, l1;
        split_f16(w[2 * i], h0, l0);
        split_f16(w[2 * i + 1], h1, l1);
        wv[i] = lo_half ? (l0 | (l1 << 16)) : (h0 | (h1 << 16));
      }
      tmem_st8(tl + ks * 8, wv);
    }
  }
  asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");

  {
    // ===== workers: two (cell, utterance) items per thread =====
    const int cl = lane, up = warp;
    const int cell = slice * TCL_CS + cl;
    int uidx[2];
    bool ok[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      uidx[e] = s0 + group * TCL_UG + 2 * up + e;
      ok[e] = uidx[e] < s1;
    }
    const float ppi = P.pi[cell], ppf = P.pf[cell], ppo = P.po[cell];
    float dc_next[2] = {0.f, 0.f}, f_next[2] = {0.f, 0.f}, di_next[2] = {0.f, 0.f}, df_next[2] = {0.f, 0.f};
    float dcm_next[2] = {0.f, 0.f};
    float sb[4][2], spi[2] = {0.f, 0.f}, spf[2] = {0.f, 0.f}, spo[2] = {0.f, 0.f};
#pragma unroll
    for (int q = 0; q < 4; q++) { sb[q][0] = 0.f; sb[q][1] = 0.f; }
    float vg[2], vi[2], vf[2], vo[2], vc[2], vcp[2], vd[2], vr[2] = {1.f, 1.f};
    float runmax = 0.f;
    const int tstep = dir == 0 ? -1 : 1;   // time order of the forward pass: c_prev lives at t + tstep
    auto prefetch = [&](int t) {
#pragma unroll
      for (int e = 0; e < 2; e++) {
        if (!ok[e]) { vg[e] = vi[e] = vf[e] = vo[e] = vc[e] = vcp[e] = vd[e] = 0.f; continue; }
        const int u = uidx[e];
        const float *grow = a.G + ((size_t)t * S + u) * a.ldg + (size_t)dir * 4 * C + cell;
        vg[e] = __ldcs(grow); vi[e] = __ldcs(grow + (size_t)C); vf[e] = __ldcs(grow + (size_t)2 * C); vo[e] = __ldcs(grow + (size_t)3 * C);
        vc[e] = __ldcs(a.cell + ((size_t)t * S + u) * a.ldc + (size_t)dir * C + cell);
        const int tp = t + tstep;
        vcp[e] = (tp >= 0 && tp < T) ? __ldcs(a.cell + ((size_t)tp * S + u) * a.ldc + (size_t)dir * C + cell) : 0.f;
        vd[e] = __ldcs(a.dout + ((size_t)t * S + u) * a.ldd + (size_t)dir * C + cell);
        if (DROP != 0)
          vr[e] = __ldg(a.rmask + (size_t)(a.rmask_per_step ? (size_t)t * S + u : (size_t)u) * a.ldr + (size_t)dir * C + cell);
      }
    };
    prefetch(dir == 0 ? T - 1 : 0);
    const size_t pstride_slice = (size_t)TCL_UG * C;
    const int quad = warp & 3, uh = warp >> 2;
    const uint64_t dAhi = umma_desc(smem_u32(Ahi), 16, 1024, 2), dAlo = umma_desc(smem_u32(Alo), 16, 1024, 2),
                   dBt = umma_desc(smem_u32(Bt), 16, 1024, 2);
    // accumulator columns: full tile mt at mt * 48, the stacked tile behind them (a 64-column stride, X on a 32-column
    // boundary, measured no faster)
    auto acc_col = [&](int mt) -> uint32_t { return (uint32_t)mt * 48u; };
    const uint32_t accS = (uint32_t)n128 * 48u;

    TC_ACC_DECL();
    TC_MARK_DECL();
    TC_OBS_DECL();
    for (int step = 0; step < T; step++) {
      const int t = dir == 0 ? T - 1 - step : step;
      TC_T0();
      float dm[2] = {vd[0], vd[1]};
      if (CL && step > 0) {
        // ---- d_m of this thread's items: the `slices` blocks that landed in buffer (step-1)&1, added in producer order
        const int par = (step - 1) & 1;
        mbar_wait_peers(&rfull[par], (uint32_t)(((step - 1) >> 1) & 1));
        const float *rb = R + (size_t)par * slices * kRBlk + cl * kRRow + 2 * up;
        float s0_ = 0.f, s1_ = 0.f;
        for (int p = 0; p < slices; p++) {
          const float2 v = *reinterpret_cast<const float2 *>(rb + (size_t)p * kRBlk);
          s0_ += v.x; s1_ += v.y;
        }
        if (ok[0]) dm[0] += s0_;
        if (ok[1]) dm[1] += s1_;
        // armed again for the partials of step + 1 (they cannot arrive before this CTA has published step's partials,
        // which it does behind the b_full barrier all its threads reach after this gather)
        if (tid == 0) mbar_expect_tx(&rfull[par], rbytes);
      }
      if (!CL && step > 0) {
        // ---- d_m of this thread's items: the `slices` tagged partials, summed in fixed order (:470 / :561)
        // Cooperative and wide: the CTA needs, from each of the `slices` producers, a [16 utterances x 32 cells] block of
        // partials (128 contiguous bytes per utterance row).  Thread (half, u, c4) fetches 4 cells of utterance u from
        // one half of the producers with 16-byte loads (<= 6 requests per thread instead of 2 x slices scalar ones),
        // sums them in producer order, and the two halves meet in shared memory -- a fixed order: deterministic.
        const uint32_t want = (uint32_t)(((step - 1) >> 1) & 1);
        const int c4 = tid & 7, gu = (tid >> 3) & 15, half = tid >> 7;
        const int hs = (slices + 1) >> 1, sl0 = half * hs, sl1 = half ? slices : hs;
        const bool uv = s0 + group * TCL_UG + gu < s1;
        const uint4 *pv = reinterpret_cast<const uint4 *>(
            pbuf + ((size_t)((((step - 1) & 1) * ndir + dir) * groups + group) * slices) * pstride_slice + (size_t)gu * C +
            slice * TCL_CS + c4 * 4);
        constexpr int NQ = WIDE ? 8 : 6;   // producers per half
        uint4 q[NQ];
#pragma unroll
        for (int i = 0; i < NQ; i++)
          if (uv && sl0 + i < sl1) q[i] = ld_word4(pv + (size_t)(sl0 + i) * (pstride_slice / 4));
        float4 acc4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < NQ; i++) {
          if (uv && sl0 + i < sl1) {
            while ((((q[i].x ^ want) | (q[i].y ^ want) | (q[i].z ^ want) | (q[i].w ^ want)) & 1u) != 0u) {
              q[i] = ld_word4(pv + (size_t)(sl0 + i) * (pstride_slice / 4));
              TC_COUNT(5);   // (debug build: re-polls of thread 0)
            }
            acc4.x += __uint_as_float(q[i].x & 0xfffffffeu); acc4.y += __uint_as_float(q[i].y & 0xfffffffeu);   // tag bit cleared
            acc4.z += __uint_as_float(q[i].z & 0xfffffffeu); acc4.w += __uint_as_float(q[i].w & 0xfffffffeu);
          }
        }
        *reinterpret_cast<float4 *>(gsm + ((size_t)(half * TCL_UG + gu) * 32 + c4 * 4)) = acc4;
        named_bar_workers();
#pragma unroll
        for (int e = 0; e < 2; e++)
          if (ok[e]) dm[e] += gsm[(size_t)(2 * up + e) * 32 + cl] + gsm[(size_t)(TCL_UG + 2 * up + e) * 32 + cl];   // :470 / :561
      }
      TC_TICK(1, 0);
      float dgt[4][2], mxe[2];
#pragma unroll
      for (int e = 0; e < 2; e++) {
        float dg = 0.f, di = 0.f, df = 0.f, dO = 0.f;
        if (ok[e]) {
          float h = tanhf_(vc[e]);
          float dh = dm[e] * vo[e] * (1.f - h * h);                               // :473-474
          dO = dm[e] * h * vo[e] * (1.f - vo[e]);                                 // :477-478
          float dc, dcm;
          if (DROP == 0) {
            dc = dh + dc_next[e] * f_next[e] + di_next[e] * ppi + df_next[e] * ppf + dO * ppo;   // :481-485
            dcm = dc;
          } else {
            dc = dh + di_next[e] * ppi + df_next[e] * ppf + dO * ppo + (DROP == 2 ? dcm_next[e] : dc_next[e]) * f_next[e];
            dcm = dc * vr[e];
          }
          df = (DROP == 2 ? dcm : dc) * vcp[e] * vf[e] * (1.f - vf[e]);           // :488-489 / :715-719
          di = dcm * vg[e] * vi[e] * (1.f - vi[e]);                               // :492-493 / :723
          dg = dcm * vi[e] * (1.f - vg[e] * vg[e]);                               // :496-497 / :727
          dc_next[e] = dc; dcm_next[e] = dcm; f_next[e] = vf[e]; di_next[e] = di; df_next[e] = df;
          float *drow = a.DG + ((size_t)t * S + uidx[e]) * a.lddg + (size_t)dir * 4 * C + cell;
          drow[0] = dg; drow[(size_t)C] = di; drow[(size_t)2 * C] = df; drow[(size_t)3 * C] = dO;
          sb[0][e] += dg; sb[1][e] += di; sb[2][e] += df; sb[3][e] += dO;         // :507 / :598
          spi[e] += di * vcp[e]; spf[e] += df * vcp[e]; spo[e] += dO * vc[e];     // :508-510 / :599-601
        }
        dgt[0][e] = dg; dgt[1][e] = di; dgt[2][e] = df; dgt[3][e] = dO;
        mxe[e] = fmaxf(fmaxf(fabsf(dg), fabsf(di)), fmaxf(fabsf(df), fabsf(dO)));
        runmax = fmaxf(runmax, mxe[e]);   // max |d(gates)| of everything this thread writes (-> a.dgmax)
      }
      if (step + 1 == T) break;   // the last step's recurrent contribution is never consumed
      // ---- D operand: every utterance column scaled by its own power of two into [2^13, 2^14), fp16 hi / lo'
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const float mx = mxe[e];
        const unsigned mb = __reduce_max_sync(0xffffffffu, __float_as_uint(mx));   // non-negative floats order like their bits
        int ex = (int)(mb >> 23) - 127;                    // floor(log2(max)); -127 for zero / subnormal columns
        int kexp = 13 - ex;
        kexp = kexp > 120 ? 120 : (kexp < -120 ? -120 : kexp);
        if (mb == 0u || mb >= 0x7f800000u) kexp = 0;       // all-zero column, or inf/nan (propagates as it is)
        const float sc = __uint_as_float((uint32_t)(kexp + 127) << 23);
        if (lane == 0) scl[(step & 1) * 16 + 2 * up + e] = __uint_as_float((uint32_t)(127 - kexp) << 23);
        const int u = 2 * up + e;
#pragma unroll
        for (int q = 0; q < 4; q++) {
          uint32_t h, l;
          split_f16(dgt[q][e] * sc, h, l);
          *reinterpret_cast<uint16_t *>(Bt + sw128_off(32, u, q * 32 + cl)) = (uint16_t)h;
          *reinterpret_cast<uint16_t *>(Bt + sw128_off(32, 16 + u, q * 32 + cl)) = (uint16_t)l;
        }
      }
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
      mbar_arrive(&b_full);
      TC_TICK(1, 1);
      if (warp == 0) {
        // ===== MMA issue (the last step's partial is never consumed: T-1 products) =====
        mbar_wait(&b_full, (uint32_t)(step & 1));
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        TC_TICK(1, 10);   // (debug build: waiting for the other warps' part of the B tile)
        TC_MARK();
        if (elect_one()) {
          // one commit per M tile: the epilogue (TMEM -> partial words) of a tile runs while the tensor pipe is
          // still working on the next one.  The stacked tile goes first: its epilogue has one more hand-over.
          int nb = 0;
          if (rem64) {
            issue_bwd_tile_stacked(tmem_base + colS, dBt, tmem_base + accS);
            umma_commit(&mma_done[nb++]);
          }
          for (int mt = 0; mt < n128; mt++) {
            const uint64_t toff = (uint64_t)(((mt - NTS) * 32768) >> 4);
            if (mt < NTS) issue_bwd_tile_ts(tmem_base + kColA + mt * 128, tmem_base + kColA + mt * 128 + 64, dBt, tmem_base + acc_col(mt));
            else issue_bwd_tile(dAhi + toff, dAlo + toff, dBt, tmem_base + acc_col(mt));
            umma_commit(&mma_done[nb++]);
          }
        }
        __syncwarp();
      }
      // (Measured and dropped, profiles/r02_ac_ab.txt: letting the other warps sleep until warp 0 has issued the whole
      // product.  In isolation the elected thread issues the 40 MMAs in 0.64 k cycles alone and in 1.8 k next to four
      // warps of global loads (tests/micro/umma_probe.cu, profiles/r02_ab_umma_noise.txt), but inside the kernel the
      // wait costs 0.9 ms per C2 step: the overlap of prefetch and epilogue with the product is worth more.)
      TC_TICK(1, 2);
      // the saved state of the next position (measured: issuing these loads in front of the MMA issue instead costs
      // 0.2 ms per C2 step -- it delays the product; behind it their latency hides under the tensor pipe's work)
      prefetch(t + tstep);
      TC_TICK(1, 4);
      {
        uint32_t *pw = pbuf + ((size_t)((((step & 1) * ndir + dir) * groups + group) * slices + slice)) * pstride_slice;
        const uint32_t tagw = (uint32_t)((step >> 1) & 1);
        // Warp 0 issues the MMAs and is the last to get to the epilogue; every consumer of the cluster waits for ITS
        // pushes (ncu stall samples, profiles/r02_p_lstm_tc_hotspots.txt: 27 % of all warp time in the wait for the peers'
        // partials).  So warp 0 takes no part in the epilogue: warp 4, which owns the same TMEM lane quadrant, handles
        // both utterance halves while warp 0 is still issuing (profiles/r02_v_ab.txt).
        const bool w0 = warp == 0;
        const int nhalves = warp == 4 ? 2 : 1;
        const int nbar2 = 224;   // threads on the stacked tile's hand-over barrier
        // (CL) the 8 utterance values of accumulator row `row` of the 32-row block that belongs to CTA d of the cluster:
        // two 16-byte stores into d's receive buffer (step & 1), block `slice` (= this producer), complete_tx on d's barrier
        auto push8 = [&](uint32_t d, int row, int uhh, const float (&pv)[8]) {
          const uint32_t la = smem_u32(R) + (uint32_t)((((step & 1) * slices + slice) * kRBlk + row * kRRow + 8 * uhh) * 4);
          const uint32_t ra = mapa_u32(la, d), rbar = mapa_u32(smem_u32(&rfull[step & 1]), d);
          st_async16(ra, make_uint4(__float_as_uint(pv[0]), __float_as_uint(pv[1]), __float_as_uint(pv[2]), __float_as_uint(pv[3])), rbar);
          st_async16(ra + 16, make_uint4(__float_as_uint(pv[4]), __float_as_uint(pv[5]), __float_as_uint(pv[6]), __float_as_uint(pv[7])), rbar);
        };
        // (measured, profiles/r02_w_ab.txt: holding the epilogue back until the last tile has committed costs 0.3 ms per
        // C2 step, moving the prefetch loads behind the epilogue 0.8 ms: the overlap below is what pays)
        for (int bi = 0; bi < MT; bi++) {
          if (w0 && bi + 1 < MT) continue;   // warp 0 only makes sure the last tile is done (the B tile is rewritten next step)
          TC_OBS_START();
          mbar_wait(&mma_done[bi], (uint32_t)(step & 1));
          asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
          TC_TICK(1, 6);   // (debug build: time spent waiting for the tiles' commits)
          TC_SEEN(bi);
          TC_OBS(0);
          if (w0) continue;
          // (the column scales were written by the other warps before they arrived on b_full: they are read only behind a
          // commit, which is behind b_full; two sets by step parity, see the declaration of scl)
          if (rem64 && bi == 0) {
            // stacked tile: lanes 0-63 (quadrants 0-1) carry hi*hi | hi*lo', lanes 64-127 the lo'*hi term of the same
            // rows -- it crosses to the other warps through shared memory
            const uint32_t tl = tmem_base + ((uint32_t)(quad * 32) << 16) + accS;
            const int r = (quad & 1) * 32 + lane;
            if (quad >= 2) {
              uint32_t y0[8];
              tmem_ld8(tl + 8 * uh, y0);
              tmem_ld_wait();
#pragma unroll
              for (int jj = 0; jj < 8; jj++) ysm[(8 * uh + jj) * 64 + r] = u2f(y0[jj]);
              asm volatile("bar.arrive 2, %0;\n" ::"r"(nbar2) : "memory");
            } else {
              for (int hh = 0; hh < nhalves; hh++) {
                const int uhh = nhalves == 2 ? 1 - hh : uh;
                uint32_t x0[8], x1[8];
                tmem_ld8(tl + 8 * uhh, x0);
                tmem_ld8(tl + 16 + 8 * uhh, x1);
                tmem_ld_wait();
                if (hh == 0) asm volatile("bar.sync 2, %0;\n" ::"r"(nbar2) : "memory");
                TC_OBS(1);
                const int j = n128 * 128 + r;
                float pv[8];
#pragma unroll
                for (int jj = 0; jj < 8; jj++)
                  pv[jj] = (u2f(x0[jj]) + (u2f(x1[jj]) + ysm[(8 * uhh + jj) * 64 + r]) * kLoUnscale) * scl[(step & 1) * 16 + 8 * uhh + jj];
                TC_OBS(2);
                if (CL) {
                  push8((uint32_t)(n128 * 4 + (quad & 1)), lane, uhh, pv);
                  TC_OBS(3);
                } else {
#pragma unroll
                  for (int jj = 0; jj < 8; jj++)
                    st_word(pw + (size_t)(8 * uhh + jj) * C + j, (__float_as_uint(pv[jj]) & 0xfffffffeu) | tagw);   // tag = LSB
                }
              }
            }
            TC_TICK(1, 3);
            continue;
          }
          const int mt = bi - rem64;
          const uint32_t tl = tmem_base + ((uint32_t)(quad * 32) << 16) + acc_col(mt);
          for (int hh = 0; hh < nhalves; hh++) {
            const int uhh = nhalves == 2 ? 1 - hh : uh;
            uint32_t x0[8], x1[8], y0[8];
            tmem_ld8(tl + 8 * uhh, x0);
            tmem_ld8(tl + 16 + 8 * uhh, x1);
            tmem_ld8(tl + 32 + 8 * uhh, y0);
            tmem_ld_wait();
            TC_OBS(1);
            const int j = mt * 128 + quad * 32 + lane;   // lane = row
            float pv[8];
#pragma unroll
            for (int jj = 0; jj < 8; jj++)
              pv[jj] = (u2f(x0[jj]) + (u2f(x1[jj]) + u2f(y0[jj])) * kLoUnscale) * scl[(step & 1) * 16 + 8 * uhh + jj];
            TC_OBS(2);
            if (CL) {
              push8((uint32_t)(mt * 4 + quad), lane, uhh, pv);
              TC_OBS(3);
            } else {
#pragma unroll
              for (int jj = 0; jj < 8; jj++)
                st_word(pw + (size_t)(8 * uhh + jj) * C + j, (__float_as_uint(pv[jj]) & 0xfffffffeu) | tagw);   // tag = LSB
            }
          }
          TC_TICK(1, 3);
        }
        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
      }
      TC_TICK(1, 3);
    }

    TC_FLUSH(1);
    TC_SEEN_FLUSH(1);
    TC_OBS_FLUSH();
    // max |d(gates)| over the launch: the scale of the fp16 planes the dense products read DG through (gemm_tc.cu) --
    // saves them a pass over the 393 MB matrix (NaN / inf order above every finite value as bit patterns: they reach the
    // conversion as they would have through its own scan)
    if (a.dgmax) {
      const unsigned mbits = __reduce_max_sync(0xffffffffu, __float_as_uint(runmax));
      if (lane == 0 && mbits) atomicMax(a.dgmax, mbits);
    }
    // ---- bias / peephole gradient partial sums of this (dir, group): reduce over the CTA's 16 utterances
    named_bar_workers();
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int u = 2 * up + e;
      float v[7] = {sb[0][e], sb[1][e], sb[2][e], sb[3][e], spi[e], spf[e], spo[e]};
#pragma unroll
      for (int q = 0; q < 7; q++) red[(q * TCL_UG + u) * 32 + cl] = v[q];
    }
    named_bar_workers();
    if (tid < 7 * 32) {
      const int q = tid >> 5, c_ = tid & 31;
      float s_ = 0.f;
      for (int uu = 0; uu < TCL_UG; uu++) s_ += red[(q * TCL_UG + uu) * 32 + c_];
      a.gsum[(((size_t)dir * groups + group) * 7 + q) * C + slice * TCL_CS + c_] = s_;
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  if (CL) cluster_sync_all();   // no CTA leaves while a peer could still address its shared memory
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(512) : "memory");
  }
}

// the forward kernel needs only the B tile and the gate staging in shared memory (the weights live in TMEM); it still
// asks for most of the SM's shared memory so that no GEMM CTA of the side stream is placed next to it -- such a CTA
// would sit in tcgen05.alloc until this kernel releases its 512 TMEM columns
size_t tc_fwd_smem(int C) {
  // (cluster exchange, C <= 384: two B tiles + the warps' 2 KB publish staging)
  const size_t need = (size_t)(C <= 384 ? 2 : 1) * (C / 64) * 4096 + 4 * TCL_UG * 32 * sizeof(float) + 2048 + (C > 448 ? 32768 : 0) + 1024;
  return need > 180 * 1024 ? need : (size_t)180 * 1024;
}
// backward: B tile + small scratch in the first 32 KB, then the full M tiles that do not fit TMEM (C = 384: one), then
// (cluster exchange, C <= 384) the receive buffers [2][slices][32 cells][80 B];
// like the forward kernel it asks for most of the SM so that no TMEM-allocating GEMM CTA lands beside it
size_t tc_bwd_smem(int C) {
  const int n128 = C >> 7, nts = n128 < 2 ? n128 : 2;
  const size_t need = 32768 + (size_t)(n128 - nts) * 65536 + 32768 + 1024 +   // (+ 32 KB unused, see lstm_tc_bwd_kernel)
                      (C <= 384 ? (size_t)2 * (C / TCL_CS) * 32 * 80 : 0);
  return need > 180 * 1024 ? need : (size_t)180 * 1024;
}

const void *tc_fwd_fn(int drop, bool wide, bool cl) {
  if (wide) return drop == 0 ? (const void *)lstm_tc_fwd_kernel<0, 1, 0> : drop == 1 ? (const void *)lstm_tc_fwd_kernel<1, 1, 0> : (const void *)lstm_tc_fwd_kernel<2, 1, 0>;
  if (cl) return drop == 0 ? (const void *)lstm_tc_fwd_kernel<0, 0, 1> : drop == 1 ? (const void *)lstm_tc_fwd_kernel<1, 0, 1> : (const void *)lstm_tc_fwd_kernel<2, 0, 1>;
  return drop == 0 ? (const void *)lstm_tc_fwd_kernel<0, 0, 0> : drop == 1 ? (const void *)lstm_tc_fwd_kernel<1, 0, 0> : (const void *)lstm_tc_fwd_kernel<2, 0, 0>;
}
const void *tc_bwd_fn(int drop, bool wide, bool cl) {
  if (wide) return drop == 0 ? (const void *)lstm_tc_bwd_kernel<0, 1, 0> : drop == 1 ? (const void *)lstm_tc_bwd_kernel<1, 1, 0> : (const void *)lstm_tc_bwd_kernel<2, 1, 0>;
  if (cl) return drop == 0 ? (const void *)lstm_tc_bwd_kernel<0, 0, 1> : drop == 1 ? (const void *)lstm_tc_bwd_kernel<1, 0, 1> : (const void *)lstm_tc_bwd_kernel<2, 0, 1>;
  return drop == 0 ? (const void *)lstm_tc_bwd_kernel<0, 0, 0> : drop == 1 ? (const void *)lstm_tc_bwd_kernel<1, 0, 0> : (const void *)lstm_tc_bwd_kernel<2, 0, 0>;
}

// launch configuration of the cluster variant: one cluster = the `slices` CTAs of one (dir, group)
struct ClusterLaunch {
  cudaLaunchConfig_t cfg;
  cudaLaunchAttribute at[1];
  ClusterLaunch(const LstmPlan &pl, size_t smem, cudaStream_t st) {
    cfg = cudaLaunchConfig_t{};
    cfg.gridDim = dim3(pl.slices, pl.groups, pl.ndir);
    cfg.blockDim = dim3(pl.threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = pl.slices; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
  }
};
cudaError_t tc_prepare_fn(const void *fn, size_t smem, int slices, bool cl) {
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e == cudaSuccess && cl && slices > 8) e = cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  return e;
}

// 1 when every (dir, group) cluster of `slices` CTAs of both passes can be resident at the same time (else the clusters
// would run in waves and the tagged-word exchange through L2 is the better plan).  EESEN_B200_LSTM_EXCHANGE=l2 forces
// the L2 exchange (A/B measurements).
int tc_cluster_ok(const LstmPlan &pl, int C) {
  const char *ex = getenv("EESEN_B200_LSTM_EXCHANGE");
  if (ex && strcmp(ex, "l2") == 0) return 0;
  if (C > 384 || pl.slices > 16 || pl.slices < 1) return 0;
  static int cache[2][17][17];   // [ndir - 1][groups][slices]: 0 unknown, 1 no, 2 yes
  if (pl.groups > 16) return 0;
  int &c = cache[pl.ndir - 1][pl.groups][pl.slices];
  if (c == 0) {
    bool ok = true;
    for (int pass = 0; pass < 2 && ok; pass++) {
      const void *fn = pass == 0 ? tc_fwd_fn(0, false, true) : tc_bwd_fn(0, false, true);
      const size_t smem = pass == 0 ? pl.smem_fwd : pl.smem_bwd;
      if (tc_prepare_fn(fn, smem, pl.slices, true) != cudaSuccess) { cudaGetLastError(); ok = false; break; }
      ClusterLaunch cl(pl, smem, 0);
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, fn, &cl.cfg) != cudaSuccess) { cudaGetLastError(); ok = false; break; }
      ok = n >= pl.ndir * pl.groups;
    }
    c = ok ? 2 : 1;
  }
  return c == 2;
}

}  // namespace

cudaError_t lstm_set_flag(cudaStream_t st, unsigned *flag, unsigned value) {
  set_flag_kernel<<<1, 1, 0, st>>>(flag, value);
  return cudaGetLastError();
}

int lstm_tc_debug_timing(long long *out32, int reset) {
#ifdef EB_LSTM_TIMING
  if (out32) cudaMemcpyFromSymbol(out32, g_lstm_tc_timing, sizeof(long long) * 32);
  if (reset) {
    long long z[32] = {0};
    cudaMemcpyToSymbol(g_lstm_tc_timing, z, sizeof(z));
  }
  return 1;
#else
  (void)out32; (void)reset;
  return 0;
#endif
}

// Plan of the tensor-core engine (engine = 1): valid when the cells of a direction tile into 64-wide k-blocks,
// the resident tiles fit shared memory and one co-resident grid holds every (dir, group, slice).
LstmPlan lstm_tc_plan(int S, int C, int num_sms, size_t max_smem, int ndir) {
  LstmPlan pl;
  memset(&pl, 0, sizeof(pl));
  pl.ndir = ndir;
  if (C % 64 != 0 || C < 64 || S <= 0 || ndir < 1 || ndir > 2) return pl;
  const int groups = (S + TCL_UG - 1) / TCL_UG, slices = C / TCL_CS;
  const size_t sf = tc_fwd_smem(C), sb = tc_bwd_smem(C);
  if ((long)ndir * groups * slices > num_sms || sf > max_smem || sb > max_smem || slices > 16) return pl;
  pl.engine = 1;
  pl.nut = 2; pl.nct = 4; pl.ksplit = 1;
  pl.groups = groups; pl.slices = slices;
  pl.threads = TCL_THREADS;
  pl.smem_fwd = sf; pl.smem_bwd = sb;
  pl.pbuf_floats = (size_t)2 * ndir * groups * slices * TCL_UG * C;       // 4-byte words, tag in the LSB
  pl.xbuf_bytes = (size_t)2 * ndir * groups * TCL_UG * C * 4;
  pl.gsum_floats = (size_t)2 * groups * 7 * C;
  pl.cluster = tc_cluster_ok(pl, C);
  pl.valid = 1;
  return pl;
}

cudaError_t lstm_tc_forward(cudaStream_t st, const LstmPlan &pl, const LstmFwdArgs &a) {
  if (!pl.valid || pl.engine != 1) return cudaErrorInvalidConfiguration;
  if (a.drop < 0 || a.drop > 2 || (a.drop != 0 && !a.rmask)) return cudaErrorInvalidValue;
  const bool wide = a.C > 384, cl = pl.cluster && !wide;
  const void *fn = tc_fwd_fn(a.drop, wide, cl);
  cudaError_t e = tc_prepare_fn(fn, pl.smem_fwd, pl.slices, cl);
  if (e != cudaSuccess) return e;
  int groups = pl.groups, ndir = pl.ndir;
  LstmFwdArgs args = a;
  void *kargs[] = {&args, &groups, &ndir};
  if (cl) {   // clusters are self-contained: no tagged-word buffer, no grid-wide co-residency
    ClusterLaunch c(pl, pl.smem_fwd, st);
    return cudaLaunchKernelExC(&c.cfg, fn, kargs);
  }
  e = cudaMemsetAsync(a.xbuf, 0xff, pl.xbuf_bytes, st);   // tag bit 1 = "not the data of steps 0 / 1"
  if (e != cudaSuccess) return e;
  dim3 grid(pl.slices, pl.groups, pl.ndir), block(pl.threads);
  return cudaLaunchCooperativeKernel(fn, grid, block, kargs, pl.smem_fwd, st);
}

cudaError_t lstm_tc_backward(cudaStream_t st, const LstmPlan &pl, const LstmBwdArgs &a) {
  if (!pl.valid || pl.engine != 1) return cudaErrorInvalidConfiguration;
  if (a.drop < 0 || a.drop > 2 || (a.drop != 0 && !a.rmask)) return cudaErrorInvalidValue;
  const bool wide = a.C > 384, cl = pl.cluster && !wide;
  const void *fn = tc_bwd_fn(a.drop, wide, cl);
  cudaError_t e = tc_prepare_fn(fn, pl.smem_bwd, pl.slices, cl);
  if (e != cudaSuccess) return e;
  int groups = pl.groups, slices = pl.slices, ndir = pl.ndir;
  LstmBwdArgs args = a;
  void *kargs[] = {&args, &groups, &slices, &ndir};
  if (cl) {
    ClusterLaunch c(pl, pl.smem_bwd, st);
    return cudaLaunchKernelExC(&c.cfg, fn, kargs);
  }
  e = cudaMemsetAsync(a.pbuf, 0xff, pl.pbuf_floats * sizeof(float), st);
  if (e != cudaSuccess) return e;
  dim3 grid(pl.slices, pl.groups, pl.ndir), block(pl.threads);
  return cudaLaunchCooperativeKernel(fn, grid, block, kargs, pl.smem_bwd, st);
}

}  // namespace eb
