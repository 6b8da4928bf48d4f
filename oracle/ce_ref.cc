// oracle/ce_ref.cc -- TEST INFRASTRUCTURE ONLY.
//
// A small driver (our own code) that links against the UNMODIFIED reference objects compiled in place
// (oracle/ce_ref.mk, the CPU objects of oracle/Makefile) and runs the reference's own CE::EvalParallel
// (src/net/ce-loss.cc:94-169) on given posteriors, exactly as src/netbin/train-ce-parallel.cc:140-168 calls it:
// the float frame mask 1 on rows t < frames[s], the packed targets (0 on padded rows), S sequences.
//   ref_ce_cpu <posteriors.npy f32 [T*S x K]> <targets.npy i32 [T*S]> <frames.npy i32 [S]> <outdir>
// writes <outdir>/ce_diff.npy and prints one JSON line {"obj", "correct", "frames", "sequences"} read from the
// CE object's own counters (the "#define private public" shim on the reference header only).
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <limits>
#include <list>
#include <map>
#include <set>
#include <sstream>
#include <stdexcept>
#include <typeinfo>
#include <utility>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

// standard headers first: the shim below must reach the reference header only
#define private public
#include "net/ce-loss.h"
#undef private
#include "base/kaldi-common.h"

using namespace eesen;

// minimal .npy (version 1.0, C order) reader: returns the shape, fills raw bytes
static std::vector<size_t> read_npy(const char *path, const char *descr, std::vector<char> *raw, size_t item) {
  FILE *f = fopen(path, "rb");
  if (!f) { fprintf(stderr, "cannot open %s\n", path); exit(2); }
  char pre[10];
  if (fread(pre, 1, 10, f) != 10 || memcmp(pre, "\x93NUMPY", 6) != 0) { fprintf(stderr, "bad npy %s\n", path); exit(2); }
  size_t hl = (unsigned char)pre[8] | ((unsigned char)pre[9] << 8);
  std::string hdr(hl, ' ');
  if (fread(&hdr[0], 1, hl, f) != hl) exit(2);
  if (hdr.find(descr) == std::string::npos || hdr.find("'fortran_order': False") == std::string::npos) {
    fprintf(stderr, "%s: want %s, C order\n", path, descr);
    exit(2);
  }
  std::vector<size_t> shape;
  size_t p = hdr.find('(') + 1, n = 1;
  while (p < hdr.size() && hdr[p] != ')') {
    if (isdigit((unsigned char)hdr[p])) {
      size_t v = strtoull(hdr.c_str() + p, nullptr, 10);
      shape.push_back(v);
      n *= v;
      while (isdigit((unsigned char)hdr[p])) p++;
    } else {
      p++;
    }
  }
  raw->resize(n * item);
  if (fread(raw->data(), item, n, f) != n) { fprintf(stderr, "short npy %s\n", path); exit(2); }
  fclose(f);
  return shape;
}

static void write_npy_f32(const std::string &path, const float *data, size_t rows, size_t cols) {
  char shape[96];
  snprintf(shape, sizeof(shape), "{'descr': '<f4', 'fortran_order': False, 'shape': (%zu, %zu), }", rows, cols);
  std::string h = shape;
  while ((10 + h.size() + 1) % 64) h += ' ';
  h += '\n';
  FILE *f = fopen(path.c_str(), "wb");
  if (!f) { fprintf(stderr, "cannot write %s\n", path.c_str()); exit(2); }
  fwrite("\x93NUMPY\x01\x00", 1, 8, f);
  unsigned short hl = (unsigned short)h.size();
  fwrite(&hl, 2, 1, f);
  fwrite(h.data(), 1, h.size(), f);
  fwrite(data, 4, rows * cols, f);
  fclose(f);
}

int main(int argc, char **argv) {
  if (argc != 5) {
    fprintf(stderr, "usage: %s <posteriors.npy> <targets.npy> <frames.npy> <outdir>\n", argv[0]);
    return 1;
  }
  try {
    std::vector<char> yr, tr, fr;
    std::vector<size_t> ys = read_npy(argv[1], "'<f4'", &yr, 4);
    std::vector<size_t> ts = read_npy(argv[2], "'<i4'", &tr, 4);
    std::vector<size_t> fs = read_npy(argv[3], "'<i4'", &fr, 4);
    if (ys.size() != 2 || ts.size() != 1 || fs.size() != 1 || ts[0] != ys[0] || ys[0] % fs[0]) {
      fprintf(stderr, "shape mismatch\n");
      return 2;
    }
    const int32 rows = ys[0], K = ys[1], S = fs[0];
    const float *y = reinterpret_cast<const float *>(yr.data());
    const int32 *tg = reinterpret_cast<const int32 *>(tr.data());
    const int32 *frames = reinterpret_cast<const int32 *>(fr.data());
    Matrix<BaseFloat> host(rows, K, kUndefined);
    for (int32 r = 0; r < rows; r++)
      for (int32 k = 0; k < K; k++) host(r, k) = y[(size_t)r * K + k];
    // train-ce-parallel.cc:140-151: mask 1 and the target on valid rows, 0 on padded rows
    Vector<BaseFloat> mask(rows, kSetZero);
    std::vector<int32> target(rows, 0);
    for (int32 r = 0; r < rows; r++)
      if (r / S < frames[r % S]) { mask(r) = 1.0; target[r] = tg[r]; }
    CE ce;
    ce.SetReportStep(2000000000);   // no progress line: the counters are read directly below
    CuMatrix<BaseFloat> net_out(host), diff;
    ce.EvalParallel(net_out, target, &diff, mask, S);
    Matrix<BaseFloat> dh(diff);
    std::vector<float> flat((size_t)rows * K);
    for (int32 r = 0; r < rows; r++)
      for (int32 k = 0; k < K; k++) flat[(size_t)r * K + k] = dh(r, k);
    write_npy_f32(std::string(argv[4]) + "/ce_diff.npy", flat.data(), rows, K);
    printf("{\"obj\": %.17g, \"correct\": %d, \"frames\": %d, \"sequences\": %d}\n", ce.obj_, (int)ce.correct_,
           (int)ce.frames_, (int)ce.sequences_num_);
    return 0;
  } catch (const std::exception &e) {
    fprintf(stderr, "%s\n", e.what());
    return -1;
  }
}
