// gmd.h -- host interface of the GMD soft-decision decoder of Reed-Solomon codes (gmd.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "gf_decode.h"

namespace ccgpu {

constexpr uint32_t kGmdMaxRoots = 32;  // 2t <= 32: one syndrome per lane

// y: frames x (n q) channel values of the binary image (device); words: frames x n symbols, failed / chosen
// (nullable): frames bytes.  0 ok, -1 CUDA error, -3 unsupported code (not RS, 2t > 32, step != 1) or max_erasures
// odd or > 2t
int gmd_launch(const GfDevice &d, uint32_t max_erasures, const float *y, uint64_t frames, uint8_t *words,
               uint8_t *failed, uint8_t *chosen, int sm_count, cudaStream_t stream);
// frames [frame0, frame0 + frames) of the Philox stream of ccgpu_awgn_point (n q values a frame) at `sigma`, decoded
// on chip; the counters (ccgpu_counters layout, 8 x uint64 on the device) are accumulated into
int gmd_awgn_launch(const GfDevice &d, uint32_t max_erasures, float sigma, uint64_t seed, uint32_t point, uint64_t frame0,
                    uint64_t frames, unsigned long long *counters, int sm_count, cudaStream_t stream);

}  // namespace ccgpu
