// chase.h -- host interface of the Chase-II soft-decision decoder of binary BCH codes (chase.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "gf_decode.h"

namespace ccgpu {

constexpr uint32_t kChaseMaxP = 8;  // at most 2^8 test patterns per frame

// y: frames x n channel values (device); bits: frames x n, failed / chosen (nullable): frames bytes.
// 0 ok, -1 CUDA error, -3 unsupported code (not binary BCH, t > 31, 2t > 64) or p > min(8, n)
int chase_launch(const GfDevice &d, uint32_t p, const float *y, uint64_t frames, uint8_t *bits, uint8_t *failed,
                 uint8_t *chosen, int sm_count, cudaStream_t stream);
// frames [frame0, frame0 + frames) of the Philox stream of ccgpu_awgn_point at `sigma`, decoded on chip; the
// counters (ccgpu_counters layout, 8 x uint64 on the device) are accumulated into
int chase_awgn_launch(const GfDevice &d, uint32_t p, float sigma, uint64_t seed, uint32_t point, uint64_t frame0,
                      uint64_t frames, unsigned long long *counters, int sm_count, cudaStream_t stream);

}  // namespace ccgpu
