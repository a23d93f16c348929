// abp.h -- host interface of the adaptive belief-propagation decoder of binary BCH codes (abp.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "osd.h"

namespace ccgpu {

constexpr uint32_t kAbpMaxIter = 255;  // iter is a byte

// The kernel runs on the packed k-row H of the ordered-statistics decoder (OsdDevice, osd.h): same codes, same upload.
// y: frames x n channel values (device); bits: frames x n; L (nullable): frames x n; iter, failed: frames bytes.
// 0 ok, -1 CUDA error, -3 unsupported code or max_iter > 255
int abp_launch(const OsdDevice &d, uint32_t max_iter, float gamma, const float *y, uint64_t frames, uint8_t *bits,
               float *L, uint8_t *iter, uint8_t *failed, int sm_count, cudaStream_t stream);
// frames [frame0, frame0 + frames) of the Philox stream of ccgpu_awgn_point at `sigma`, decoded on chip; the
// counters (ccgpu_counters layout, 8 x uint64 on the device) are accumulated into
int abp_awgn_launch(const OsdDevice &d, uint32_t max_iter, float gamma, float sigma, uint64_t seed, uint32_t point,
                    uint64_t frame0, uint64_t frames, unsigned long long *counters, int sm_count, cudaStream_t stream);

}  // namespace ccgpu
