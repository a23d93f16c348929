// osd.h -- host interface of the ordered-statistics decoder of binary BCH codes (osd.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "codes.hpp"

namespace ccgpu {

constexpr uint32_t kOsdMaxOrder = 3;  // at most three flipped information positions per candidate
constexpr unsigned kOsdMaxN = 127, kOsdMaxK = 64;

// the k-row H of a binary BCH code packed for the kernel: row r is rows[2 r] (columns 0..63) | rows[2 r + 1]
// (columns 64..127), bit c <-> column c.  rows stays null for codes the kernel does not take.
struct OsdDevice {
  int n = 0, k = 0;
  unsigned long long *rows = nullptr;
};

// packs and uploads H when spec is a binary BCH code with n <= 127 and k <= 64 (else leaves d->rows null); 0 ok,
// -1 CUDA error.  spec.H must still be the k-row H it was created with.
int osd_upload(const CodeSpec &spec, OsdDevice *d);
void osd_free(OsdDevice *d);
// y: frames x n channel values (device); bits: frames x n, weight (nullable): frames bytes.
// 0 ok, -1 CUDA error, -3 unsupported code or order > 3
int osd_launch(const OsdDevice &d, uint32_t order, const float *y, uint64_t frames, uint8_t *bits, uint8_t *weight,
               int sm_count, cudaStream_t stream);
// frames [frame0, frame0 + frames) of the Philox stream of ccgpu_awgn_point at `sigma`, decoded on chip; the
// counters (ccgpu_counters layout, 8 x uint64 on the device) are accumulated into
int osd_awgn_launch(const OsdDevice &d, uint32_t order, float sigma, uint64_t seed, uint32_t point, uint64_t frame0,
                    uint64_t frames, unsigned long long *counters, int sm_count, cudaStream_t stream);

}  // namespace ccgpu
