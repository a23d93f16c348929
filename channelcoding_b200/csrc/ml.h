// ml.h -- host interface of the maximum-likelihood (Viterbi) decoder of high-rate binary BCH codes (ml.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "codes.hpp"

namespace ccgpu {

constexpr unsigned kMlMaxN = 127, kMlMinK = 4, kMlMaxK = 12;

// the column syndromes of the k-row H: sigma[c] = sum_r H[r][c] 2^r.  They travel to the kernel by value, so the
// decoder needs no device memory of its own.  k stays 0 for codes the kernel does not take.
struct MlCode {
  int n = 0, k = 0;
  uint16_t sigma[kMlMaxN] = {};
};

// fills *m when spec is a binary BCH code with n <= 127, 4 <= k <= 12 and no zero column (else leaves m->k = 0).
// spec.H must still be the k-row H it was created with.
void ml_prepare(const CodeSpec &spec, MlCode *m);
// y: frames x n channel values (device); bits: frames x n.  0 ok, -1 CUDA error, -3 unsupported code
int ml_launch(const MlCode &m, const float *y, uint64_t frames, uint8_t *bits, int sm_count, cudaStream_t stream);
// frames [frame0, frame0 + frames) of the Philox stream of ccgpu_awgn_point at `sigma`, decoded on chip; the
// counters (ccgpu_counters layout, 8 x uint64 on the device) are accumulated into
int ml_awgn_launch(const MlCode &m, float sigma, uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames,
                   unsigned long long *counters, int sm_count, cudaStream_t stream);

}  // namespace ccgpu
