// api.cu -- the extern "C" boundary of libccgpu.so (include/ccgpu.h) and the host-side launch logic.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/ccgpu.h"
#include "channel.cuh"
#include "chase.h"
#include "codes.hpp"
#include "gf_decode.h"
#include "abp.h"
#include "gmd.h"
#include "ml.h"
#include "ms_csr.h"
#include "ms_params.h"
#include "osd.h"

using namespace ccgpu;

// host-buffer calls are pipelined over this many staging slots (stream + device buffer each)
constexpr int kSlots = 3;

// ------------------------------------------------------------------------------------------------
struct ccgpu_ctx {
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  std::mutex mu;
  std::mutex err_mu;   // guards err: entry-point checks fail before `mu` is taken, and pool threads share a context
  std::string err;
  std::atomic<uint64_t> launches{0};
  // overrides (ccgpu_set_option; the environment variables CCGPU_QUICK / CCGPU_WORK_BATCH give the initial values and
  // are read ONCE, at ccgpu_create)
  int opt_quick = -1;        // -1: the host's estimate decides (api.cu ccgpu_awgn_point), 0 / 1: force
  int opt_work_batch = 0;    // 0: default
  int opt_lane = -1;         // lane-per-frame kernel for the small codes (ms_cyclic_lane.cuh): -1 / 1 use it, 0 do not
  // device staging for host-pointer calls (grown on demand)
  void *d_stage = nullptr;
  size_t d_stage_bytes = 0;
  unsigned long long *d_counters = nullptr;
  unsigned long long *d_work = nullptr;  // queue heads of the dynamically scheduled kernels: [0] main, [1..2] slots
  ccgpu_counters *h_counters = nullptr;  // pinned
  // host-buffer calls are cut into chunks that rotate over kSlots slots (stream + staging
  // buffer each), so the H2D copy of chunk i+1 and the D2H copy of chunk i-1 overlap the decode
  // of chunk i
  cudaStream_t slot_stream[kSlots] = {};
  cudaEvent_t main_ready = nullptr;
  void *slot_buf[kSlots] = {};
  size_t slot_bytes = 0;
};

struct ccgpu_code {
  ccgpu_ctx *ctx = nullptr;
  CodeSpec spec;
  HShape shape;
  // min-sum kernel selection per vertical-node flavour (VN_PLAIN, VN_SC, VN_2D)
  const MsCyclicEntry *cyc[VN_COUNT] = {};
  int grid_max[VN_COUNT] = {};
  size_t smem[VN_COUNT] = {};
  // lane-per-frame kernels of the small codes (VN_PLAIN, VN_2D, VN_SPA), preferred for HBM / Philox sources
  const MsCyclicEntry *lane[VN_COUNT] = {};
  int lane_grid_max[VN_COUNT] = {};
  bool all_columns_covered = false;
  unsigned max_col_weight = 0;
  MsCsrDevice csr;     // general-H kernel tables (device)
  GfDevice gf;         // algebraic decoder tables (device)
  OsdDevice osd;       // packed k-row H of the ordered-statistics decoder (device; binary BCH, n <= 127, k <= 64)
  MlCode ml;           // column syndromes of the k-row H for the Viterbi decoder (host; binary BCH, n <= 127, k <= 12)
};

namespace {

int fail(ccgpu_ctx *ctx, int code, const std::string &msg) {
  if (ctx) {
    std::lock_guard<std::mutex> g(ctx->err_mu);
    ctx->err = msg;
  }
  return code;
}
int cuda_fail(ccgpu_ctx *ctx, cudaError_t e, const char *what) {
  return fail(ctx, CCGPU_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(call)                                                    \
  do {                                                              \
    cudaError_t e_ = (call);                                        \
    if (e_ != cudaSuccess) return cuda_fail(ctx, e_, #call);        \
  } while (0)

bool is_device_ptr(const void *p) {
  if (!p) return false;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}
// whether every non-null pointer of `ptrs` is device memory (dev) or every one is host memory (!dev)
bool same_residency(bool dev, std::initializer_list<const void *> ptrs) {
  for (const void *p : ptrs)
    if (p && is_device_ptr(p) != dev) return false;
  return true;
}

int check_code(ccgpu_ctx *ctx, const ccgpu_code *code) {
  return code->ctx == ctx ? CCGPU_OK : fail(ctx, CCGPU_ERR_INVALID, "code was not created on this context");
}

// grid of a grid-stride kernel with one thread (or warp) per item and `per_cta` items per CTA, at most `per_sm` CTAs
// per SM
unsigned grid_for(const ccgpu_ctx *ctx, uint64_t items, unsigned per_cta, unsigned per_sm = 16) {
  return static_cast<unsigned>(
      std::max<uint64_t>(1, std::min<uint64_t>((items + per_cta - 1) / per_cta, uint64_t(ctx->sm_count) * per_sm)));
}

size_t align256(size_t v) { return (v + 255) & ~size_t(255); }
// Cuts typed pieces, each 256-byte aligned, out of a device buffer in order.  On a null base it hands out null
// pointers and only adds up the size: the size a buffer is allocated with comes from the code that cuts it.
struct Arena {
  char *base = nullptr;
  size_t used = 0;
  template <class T> T *take(size_t count, bool present = true) {
    if (!present) return nullptr;
    T *p = base ? reinterpret_cast<T *>(base + used) : nullptr;
    used += align256(count * sizeof(T));
    return p;
  }
};

int ensure_slots(ccgpu_ctx *ctx, size_t bytes) {
  for (int s = 0; s < kSlots; ++s)
    if (!ctx->slot_stream[s]) CU(cudaStreamCreateWithFlags(&ctx->slot_stream[s], cudaStreamNonBlocking));
  if (!ctx->main_ready) CU(cudaEventCreateWithFlags(&ctx->main_ready, cudaEventDisableTiming));
  if (bytes <= ctx->slot_bytes) return CCGPU_OK;
  for (int s = 0; s < kSlots; ++s) {
    if (ctx->slot_buf[s]) cudaFree(ctx->slot_buf[s]);
    ctx->slot_buf[s] = nullptr;
  }
  ctx->slot_bytes = 0;
  for (int s = 0; s < kSlots; ++s) CU(cudaMalloc(&ctx->slot_buf[s], bytes));
  ctx->slot_bytes = bytes;
  return CCGPU_OK;
}

// grows the stage arena to fit the layout that cut(Arena &) cuts, then cuts it there
template <class Cut>
int cut_stage(ccgpu_ctx *ctx, Cut &&cut) {
  Arena size;
  cut(size);
  if (size.used > ctx->d_stage_bytes) {
    if (ctx->d_stage) cudaFree(ctx->d_stage);
    ctx->d_stage = nullptr;
    ctx->d_stage_bytes = 0;
    const size_t want = std::max(size.used, size_t(1) << 20);
    CU(cudaMalloc(&ctx->d_stage, want));
    ctx->d_stage_bytes = want;
  }
  Arena a{static_cast<char *>(ctx->d_stage)};
  cut(a);
  return CCGPU_OK;
}

// one per-frame field of a call whose buffers are in host memory
struct HostField {
  size_t bytes;      // per frame
  const void *host;  // nullptr: the caller left this field out
  bool out;          // copied back after the launch (else copied in before it)
};

// Decodes `frames` frames from and into host buffers.  Chunks rotate over the kSlots staging slots, so that the
// copy-in of one chunk, the decode of the next and the copy-out of a third overlap.  launch(dev, nf, stream, slot)
// runs nf frames on `stream` over the slot's device copies dev[i] of the fields (nullptr where a field is absent).
template <size_t N, class Launch>
int host_pipeline(ccgpu_ctx *ctx, uint64_t frames, const HostField (&fields)[N], Launch &&launch) {
  size_t per_frame = 0;
  for (const HostField &f : fields) per_frame += f.host ? f.bytes : 0;
  const uint64_t chunk = std::max<uint64_t>(1024, std::min<uint64_t>((frames + 15) / 16, (size_t(32) << 20) / per_frame));
  void *dev[N];
  auto cut = [&](void *base) {
    Arena a{static_cast<char *>(base)};
    for (size_t i = 0; i < N; ++i) dev[i] = a.take<char>(chunk * fields[i].bytes, fields[i].host != nullptr);
    return a.used;
  };
  int rc = ensure_slots(ctx, cut(nullptr));
  if (rc) return rc;
  CU(cudaEventRecord(ctx->main_ready, ctx->stream));
  for (int s = 0; s < kSlots; ++s) CU(cudaStreamWaitEvent(ctx->slot_stream[s], ctx->main_ready, 0));
  int slot = 0;
  for (uint64_t f0 = 0; f0 < frames; f0 += chunk, slot = (slot + 1) % kSlots) {
    const uint64_t nf = std::min(chunk, frames - f0);
    cudaStream_t st = ctx->slot_stream[slot];
    cut(ctx->slot_buf[slot]);
    for (size_t i = 0; i < N; ++i)
      if (fields[i].host && !fields[i].out)
        CU(cudaMemcpyAsync(dev[i], static_cast<const char *>(fields[i].host) + f0 * fields[i].bytes, nf * fields[i].bytes,
                           cudaMemcpyHostToDevice, st));
    rc = launch(dev, nf, st, slot);
    if (rc) return rc;
    for (size_t i = 0; i < N; ++i)
      if (fields[i].host && fields[i].out)
        CU(cudaMemcpyAsync(static_cast<char *>(const_cast<void *>(fields[i].host)) + f0 * fields[i].bytes, dev[i],
                           nf * fields[i].bytes, cudaMemcpyDeviceToHost, st));
  }
  for (int s = 0; s < kSlots; ++s) CU(cudaStreamSynchronize(ctx->slot_stream[s]));
  return CCGPU_OK;
}

// Runs body(counters) on the device counters (ccgpu_counters layout) to accumulate into: `out` itself when it is
// device memory, else the context's scratch counters, zeroed before and copied into *out after.
template <class Body>
int with_counters(ccgpu_ctx *ctx, ccgpu_counters *out, Body &&body) {
  if (is_device_ptr(out)) return body(reinterpret_cast<unsigned long long *>(out));
  CU(cudaMemsetAsync(ctx->d_counters, 0, sizeof(ccgpu_counters), ctx->stream));
  const int rc = body(ctx->d_counters);
  if (rc) return rc;
  CU(cudaMemcpyAsync(ctx->h_counters, ctx->d_counters, sizeof(ccgpu_counters), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  *out = *ctx->h_counters;
  return CCGPU_OK;
}

// K1: one thread = one Philox block = four consecutive symbols of one frame.  The tile of
// tile_frames frames is assembled in shared memory and leaves the SM as coalesced 16-byte streaming stores.
// Tiles are handed out by a grid-stride loop over a grid of exactly the resident CTAs; the block -> (frame, block)
// split uses a host-computed reciprocal (no integer division), the Philox round keys come from the constant bank.
constexpr int kAwgnThreads = 256;
struct AwgnParams {
  float *y;
  uint64_t frame0, frames;
  uint32_t n, nblk, nblk_magic, tile_frames, point;
  float sigma;
  PhiloxKeys keys;
};
__global__ void __launch_bounds__(kAwgnThreads) awgn_llr_kernel(const __grid_constant__ AwgnParams p) {
  extern __shared__ float tile[];
  const uint32_t n = p.n, nblk = p.nblk;
  const uint64_t tiles = (p.frames + p.tile_frames - 1) / p.tile_frames;
  for (uint64_t t = blockIdx.x; t < tiles; t += gridDim.x) {
    const uint64_t f0 = t * p.tile_frames;
    const uint32_t nf = static_cast<uint32_t>(min(static_cast<uint64_t>(p.tile_frames), p.frames - f0));
    for (uint32_t b = threadIdx.x; b < nf * nblk; b += blockDim.x) {
      const uint32_t f = nblk == 1 ? b : __umulhi(b, p.nblk_magic);  // = b / nblk, exact for b * nblk < 2^32
      const uint32_t blk = b - f * nblk;
      const float4 v = awgn_block(p.keys, p.point, p.frame0 + f0 + f, blk, p.sigma);
      float *dst = tile + f * n + 4 * blk;
      // branch-free: a separate path for the last block of a frame (n is not a multiple of four) made every warp run
      // both paths, since every warp holds a last block
      const uint32_t left = n - 4 * blk;  // >= 1
      dst[0] = v.x;
      if (left > 1) dst[1] = v.y;
      if (left > 2) dst[2] = v.z;
      if (left > 3) dst[3] = v.w;
    }
    __syncthreads();
    const uint64_t base = f0 * n;              // multiple of 4 floats because tile_frames % 4 == 0
    const uint32_t total = nf * n;
    float4 *out4 = reinterpret_cast<float4 *>(p.y + base);
    const float4 *in4 = reinterpret_cast<const float4 *>(tile);
    for (uint32_t i = threadIdx.x; i < total / 4; i += blockDim.x) __stcs(out4 + i, in4[i]);
    for (uint32_t i = (total & ~3u) + threadIdx.x; i < total; i += blockDim.x) p.y[base + i] = tile[i];
    __syncthreads();
  }
}

// K1 launch: frames x n channel values into a 16-byte aligned device buffer
int launch_awgn(ccgpu_ctx *ctx, float *d_y, uint32_t n, float sigma, uint64_t seed, uint32_t point, uint64_t frame0,
                uint64_t frames) {
  if (frames == 0) return CCGPU_OK;
  if (reinterpret_cast<uintptr_t>(d_y) % 16 != 0) return fail(ctx, CCGPU_ERR_INVALID, "y must be 16-byte aligned");
  // tile: a multiple of 4 frames (keeps every tile base 16-byte aligned), about 16 KB: eight CTAs = 64 warps per SM
  AwgnParams ap;
  ap.y = d_y;
  ap.frame0 = frame0;
  ap.frames = frames;
  ap.n = n;
  ap.nblk = (n + 3) >> 2;
  ap.nblk_magic = static_cast<uint32_t>(((uint64_t(1) << 32) + ap.nblk - 1) / ap.nblk);  // ceil(2^32 / nblk)
  ap.tile_frames = std::max<uint32_t>(4, (4096 / n) & ~3u);
  ap.point = point;
  ap.sigma = sigma;
  ap.keys = philox_round_keys(seed);
  const size_t smem = size_t(ap.tile_frames) * n * sizeof(float);
  const uint64_t tiles = (frames + ap.tile_frames - 1) / ap.tile_frames;
  CU(cudaFuncSetAttribute(awgn_llr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  int resident = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, awgn_llr_kernel, kAwgnThreads, smem));
  const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(tiles, uint64_t(ctx->sm_count) * std::max(1, resident)));
  awgn_llr_kernel<<<grid, kAwgnThreads, smem, ctx->stream>>>(ap);
  CU(cudaGetLastError());
  ctx->launches++;
  return CCGPU_OK;
}

// ---- multiple-bases decoding (extension, BASELINE config 3): the code is cyclic, so decoding the received word
// rotated by s positions on H is decoding the word itself on H rotated by -s: B rotations = B parity-check
// matrices ("bases") from one compiled kernel.  Candidates are rotated back and the best one is kept.
__global__ void __launch_bounds__(256) mbbp_roll_kernel(const float *__restrict__ y, float *__restrict__ out,
                                                        const uint32_t *__restrict__ shifts, uint32_t n, uint32_t nb,
                                                        uint64_t frames) {
  const uint64_t total = frames * nb * n;
  for (uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
    const uint64_t fb = i / n;
    const uint32_t c = static_cast<uint32_t>(i - fb * n);
    const uint64_t f = fb / nb;
    const uint32_t b = static_cast<uint32_t>(fb - f * nb);
    uint32_t src = c + shifts[b];
    if (src >= n) src -= n;
    out[i] = y[f * n + src];  // y_b[c] = y[(c + s_b) mod n]
  }
}
// one thread per frame: correlation sum_c y[c] (1 - 2 x[c]) of every candidate (float32, c ascending in the
// un-rotated domain), the best converged candidate wins (ties: lowest base), if none converged the frame fails and
// the best failed candidate is reported
__global__ void __launch_bounds__(128) mbbp_select_kernel(const float *__restrict__ y, const uint8_t *__restrict__ bits_b,
                                                          const uint8_t *__restrict__ iter_b,
                                                          const uint8_t *__restrict__ failed_b,
                                                          const uint32_t *__restrict__ shifts, uint32_t n, uint32_t nb,
                                                          uint32_t max_iter, uint64_t frames, uint8_t *__restrict__ chosen,
                                                          uint8_t *__restrict__ iter_out, uint8_t *__restrict__ failed_out,
                                                          unsigned long long *counters) {
  unsigned long long executed = 0;
  for (uint64_t f = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; f < frames;
       f += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
    int best = -1;
    bool best_ok = false;
    float best_m = 0.0f;
    for (uint32_t b = 0; b < nb; ++b) {
      const bool ok = failed_b[f * nb + b] == 0;
      executed += ok ? iter_b[f * nb + b] + 1u : max_iter;
      const uint8_t *x = bits_b + (f * nb + b) * n;
      const uint32_t s = shifts[b];
      float m = 0.0f;
      uint32_t src = n - s;  // candidate bit of un-rotated column c is x[(c - s) mod n]
      if (src >= n) src -= n;
      for (uint32_t c = 0; c < n; ++c) {
        const float v = y[f * n + c];
        m = __fadd_rn(m, x[src] ? -v : v);
        if (++src == n) src = 0;
      }
      const bool better = best < 0 || (ok && !best_ok) || (ok == best_ok && m > best_m);
      if (better) {
        best = static_cast<int>(b);
        best_ok = ok;
        best_m = m;
      }
    }
    chosen[f] = static_cast<uint8_t>(best);
    failed_out[f] = best_ok ? 0 : 1;
    if (iter_out) iter_out[f] = iter_b[f * nb + best];
  }
  if (counters != nullptr) {
    for (int o = 16; o > 0; o >>= 1) executed += __shfl_xor_sync(0xffffffffu, executed, o);
    if ((threadIdx.x & 31) == 0 && executed) atomicAdd(counters + C_ITER, executed);
  }
}
__global__ void __launch_bounds__(256) mbbp_unroll_kernel(const uint8_t *__restrict__ bits_b, const float *__restrict__ L_b,
                                                          const uint8_t *__restrict__ chosen,
                                                          const uint32_t *__restrict__ shifts, uint32_t n, uint32_t nb,
                                                          uint64_t frames, uint8_t *__restrict__ bits, float *__restrict__ L) {
  const uint64_t total = frames * n;
  for (uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
    const uint64_t f = i / n;
    const uint32_t c = static_cast<uint32_t>(i - f * n);
    const uint32_t b = chosen[f];
    uint32_t src = c + n - shifts[b];
    if (src >= n) src -= n;
    const uint64_t at = (f * nb + b) * n + src;
    bits[i] = bits_b[at];
    if (L) L[i] = L_b[at];
  }
}

// ---- binary BCH with erasures the way the reference's PGZ decoder does it (codes/bch.h:97-149): the erased positions
// are filled with zeros, then with ones, both words are decoded errors-only, the success with fewer corrected
// positions wins (ties: the zero fill, it is tried first)
__global__ void __launch_bounds__(256) pgz_fill_kernel(const uint8_t *__restrict__ words, const uint8_t *__restrict__ epos,
                                                       const uint8_t *__restrict__ ecnt, uint32_t me, uint32_t n,
                                                       uint64_t count, uint8_t *__restrict__ out) {
  const uint64_t total = count * n;
  for (uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
    const uint64_t w = i / n;
    const uint32_t c = static_cast<uint32_t>(i - w * n);
    bool erased = false;
    const uint32_t e = min(static_cast<uint32_t>(ecnt[w]), me);
    for (uint32_t k = 0; k < e; ++k) erased |= epos[w * me + k] == c;
    const uint8_t v = words[i];
    out[(2 * w) * n + c] = erased ? 0 : v;
    out[(2 * w + 1) * n + c] = erased ? 1 : v;
  }
}
__global__ void __launch_bounds__(256) pgz_select_kernel(const uint8_t *__restrict__ words, const uint8_t *__restrict__ cand,
                                                         const uint8_t *__restrict__ cand_ne,
                                                         const uint8_t *__restrict__ cand_fail,
                                                         const uint8_t *__restrict__ ecnt, uint32_t t, uint32_t n,
                                                         uint64_t count, uint8_t *__restrict__ corrected,
                                                         uint8_t *__restrict__ n_errors, uint8_t *__restrict__ failed) {
  const uint64_t total = count * n;
  for (uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
    const uint64_t w = i / n;
    const uint32_t c = static_cast<uint32_t>(i - w * n);
    const bool ok0 = cand_fail[2 * w] == 0, ok1 = cand_fail[2 * w + 1] == 0;
    const bool too_many = ecnt[w] > 2 * t;  // bch.h:104-106
    const bool fail = too_many || (!ok0 && !ok1);
    const int pick = (ok0 && (!ok1 || cand_ne[2 * w] <= cand_ne[2 * w + 1])) ? 0 : 1;
    corrected[i] = fail ? words[i] : cand[(2 * w + pick) * n + c];
    if (c == 0) {
      failed[w] = fail ? 1 : 0;
      if (n_errors) n_errors[w] = fail ? 0 : cand_ne[2 * w + pick];
    }
  }
}

// the "uncoded" decoder of the reference (codes/uncoded.h:36-46: hard decision, nothing else) inside one Eb/N0
// point: one warp per frame, lane <-> Philox block, negative channel values counted on the fly
__global__ void __launch_bounds__(256) awgn_uncoded_kernel(uint32_t n, float sigma, PhiloxKeys keys, uint32_t point,
                                                           uint64_t frame0, uint64_t frames, unsigned long long *counters) {
  const int lane = threadIdx.x & 31;
  const uint32_t nblk = (n + 3) >> 2;
  const uint64_t warps = static_cast<uint64_t>(gridDim.x) * (blockDim.x >> 5);
  unsigned long long c_frames = 0, c_ferr = 0, c_berr = 0;
  for (uint64_t f = blockIdx.x * static_cast<uint64_t>(blockDim.x >> 5) + (threadIdx.x >> 5); f < frames; f += warps) {
    unsigned neg = 0;
    for (uint32_t blk = lane; blk < nblk; blk += 32) {
      const float4 v = awgn_block(keys, point, frame0 + f, blk, sigma);
      const float vv[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
      for (int e = 0; e < 4; ++e) neg += (4 * blk + e < n && vv[e] < 0.0f) ? 1u : 0u;
    }
    for (int o = 16; o > 0; o >>= 1) neg += __shfl_xor_sync(0xffffffffu, neg, o);
    c_frames += 1;
    c_berr += neg;
    c_ferr += neg ? 1 : 0;
  }
  if (lane == 0) {
    if (c_frames) atomicAdd(counters + C_FRAMES, c_frames);
    if (c_ferr) atomicAdd(counters + C_FRAME_ERR, c_ferr);
    if (c_berr) atomicAdd(counters + C_BIT_ERR, c_berr);
  }
}

bool columns_covered(const CodeSpec &s) {
  for (unsigned c = 0; c < s.n; ++c) {
    bool any = false;
    for (unsigned r = 0; r < s.rows && !any; ++r) any = s.H[size_t(r) * s.n + c] != 0;
    if (!any) return false;
  }
  return true;
}
unsigned max_column_weight(const CodeSpec &s) {
  unsigned best = 0;
  for (unsigned c = 0; c < s.n; ++c) {
    unsigned w = 0;
    for (unsigned r = 0; r < s.rows; ++r) w += s.H[size_t(r) * s.n + c] != 0;
    best = std::max(best, w);
  }
  return best;
}

// channel + hard decision (codes/codes.h:43-52: bit = y < 0): one thread = one Philox block = four symbols
__global__ void __launch_bounds__(kAwgnThreads) awgn_hard_kernel(uint8_t *__restrict__ words, uint32_t n, float sigma,
                                                                uint64_t seed, uint32_t point, uint64_t frame0,
                                                                uint64_t frames) {
  const uint32_t nblk = (n + 3) >> 2;
  const uint64_t total = frames * nblk;
  for (uint64_t i = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
    const uint64_t f = i / nblk;
    const uint32_t blk = static_cast<uint32_t>(i - f * nblk);
    const float4 v = awgn_block(seed, point, frame0 + f, blk, sigma);
    const float vv[4] = { v.x, v.y, v.z, v.w };
    uint8_t *dst = words + f * n + 4 * blk;
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (4 * blk + e < n) dst[e] = vv[e] < 0.0f ? 1 : 0;
  }
}

// word-error test of simulation.c++:126-135 over decoded words (all-zero codeword sent): one warp per word
__global__ void __launch_bounds__(256) count_words_kernel(const uint8_t *__restrict__ words, const uint8_t *__restrict__ failed,
                                                          uint32_t n, uint64_t count, unsigned long long *counters) {
  const int lane = threadIdx.x & 31;
  const uint64_t warps = static_cast<uint64_t>(gridDim.x) * (blockDim.x >> 5);
  unsigned long long c_frames = 0, c_ferr = 0, c_berr = 0, c_fail = 0, c_und = 0;
  for (uint64_t w = blockIdx.x * static_cast<uint64_t>(blockDim.x >> 5) + (threadIdx.x >> 5); w < count; w += warps) {
    unsigned nz = 0;
    for (uint32_t i = lane; i < n; i += 32) nz += words[w * n + i] != 0;
    for (int o = 16; o > 0; o >>= 1) nz += __shfl_xor_sync(0xffffffffu, nz, o);
    if (lane == 0) {
      const bool f = failed[w] != 0;
      c_frames += 1;
      c_fail += f;
      c_berr += nz;
      c_ferr += (f || nz) ? 1 : 0;
      c_und += (!f && nz) ? 1 : 0;
    }
  }
  if (lane == 0) {
    if (c_frames) atomicAdd(counters + C_FRAMES, c_frames);
    if (c_ferr) atomicAdd(counters + C_FRAME_ERR, c_ferr);
    if (c_berr) atomicAdd(counters + C_BIT_ERR, c_berr);
    if (c_fail) atomicAdd(counters + C_FAIL, c_fail);
    if (c_und) atomicAdd(counters + C_UNDETECTED, c_und);
  }
}

// pick the cyclic kernel instantiations (one per vertical-node flavour) compiled for exactly this
// H: same n, same tap offsets, and either the same number of rows without wrap-around or a
// redundant (run-time rows, wrap-around) shape.  Nothing fits -> CSR kernel.
void select_cyclic(ccgpu_code *c) {
  for (int vn = 0; vn < VN_COUNT; ++vn) c->cyc[vn] = c->lane[vn] = nullptr;
  if (c->shape.kind > 1 || c->shape.taps.empty()) return;
  const int n = static_cast<int>(c->spec.n), k = static_cast<int>(c->spec.rows);
  const int w = static_cast<int>(c->shape.taps.size());
  for (int i = 0, m = ms_cyclic_count(); i < m; ++i) {
    const MsCyclicEntry *e = ms_cyclic_at(i);
    if (e->n != n || e->w != w || !std::equal(c->shape.taps.begin(), c->shape.taps.end(), e->taps)) continue;
    const bool exact = e->k == k && !e->wrap && c->shape.kind == 0;
    if (e->cta == 2) {
      if (exact) c->lane[e->vn] = e;
      continue;
    }
    const bool redundant = e->k == 0 && e->wrap && k <= (e->cta ? e->threads : 32) * e->rpl;
    if (!exact && !redundant) continue;
    if (c->cyc[e->vn] && !exact) {
      // an exact shape wins over a redundant one.  Between two redundant shapes the CTA form beats a warp kernel with
      // three or more rows per lane (255 registers, spills) when its column sum needs no block barrier per tap: the
      // fixed-point kernel (no order to keep) and the float kernel in gather form (dyn_smem > 0, ms_cyclic_cta.cuh)
      const MsCyclicEntry *old = c->cyc[e->vn];
      const bool prefer_cta = (e->vn == VN_FIX || e->dyn_smem > 0) && e->cta && !old->cta && old->wrap && old->rpl >= 3;
      if (!prefer_cta) continue;
    }
    c->cyc[e->vn] = e;
  }
  for (int vn = 0; vn < VN_COUNT; ++vn) {
    if (!c->cyc[vn]) continue;
    c->smem[vn] = c->cyc[vn]->cta ? size_t(c->cyc[vn]->dyn_smem) : size_t(kMsThreads / 32) * 2 * 32 * c->cyc[vn]->np * sizeof(float);
    // opt in whenever static + dynamic shared memory may pass 48 KB (the CTA kernels keep y / S / staging rows static)
    if (c->smem[vn] > 32 * 1024)
      cudaFuncSetAttribute(reinterpret_cast<const void *>(c->cyc[vn]->fn), cudaFuncAttributeMaxDynamicSharedMemorySize,
                           static_cast<int>(c->smem[vn]));
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, reinterpret_cast<const void *>(c->cyc[vn]->fn),
                                                  c->cyc[vn]->threads, c->smem[vn]);
    c->grid_max[vn] = std::max(1, occ) * c->ctx->sm_count;
  }
  for (int vn = 0; vn < VN_COUNT; ++vn) {
    if (!c->lane[vn]) continue;
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, reinterpret_cast<const void *>(c->lane[vn]->fn), c->lane[vn]->threads,
                                                  size_t(c->lane[vn]->dyn_smem));
    c->lane_grid_max[vn] = std::max(1, occ) * c->ctx->sm_count;
  }
}

// everything derived from H: shape, coverage, column weight and, on a context, the kernel choice and the CSR tables
int refresh_H(ccgpu_code *c) {
  c->shape = analyse_H(c->spec.H.data(), c->spec.rows, c->spec.n);
  c->all_columns_covered = columns_covered(c->spec);
  c->max_col_weight = max_column_weight(c->spec);
  if (!c->ctx) return CCGPU_OK;  // host-only description: no device tables, no decoding
  select_cyclic(c);
  ms_csr_free(&c->csr);
  if (ms_csr_upload(c->spec.H.data(), c->spec.rows, c->spec.n, &c->csr) != 0)
    return fail(c->ctx, CCGPU_ERR_CUDA, "ms_csr_upload failed");
  return CCGPU_OK;
}

int finish_code(ccgpu_ctx *ctx, ccgpu_code *c) {
  c->ctx = ctx;
  const int rc = refresh_H(c);
  if (rc || !ctx || c->spec.family == 2) return rc;
  if (gf_upload(c->spec, &c->gf) != 0) return fail(ctx, CCGPU_ERR_CUDA, "gf_upload failed");
  if (osd_upload(c->spec, &c->osd) != 0) return fail(ctx, CCGPU_ERR_CUDA, "osd_upload failed");
  ml_prepare(c->spec, &c->ml);
  return CCGPU_OK;
}

int check_params(ccgpu_ctx *ctx, const ccgpu_ms_params *p) {
  if (!p) return fail(ctx, CCGPU_ERR_INVALID, "params is null");
  if (p->variant < CCGPU_MS || p->variant > CCGPU_OMS_Q) return fail(ctx, CCGPU_ERR_INVALID, "unknown variant");
  if (p->stop_rule < 0 || p->stop_rule > CCGPU_STOP_NONE) return fail(ctx, CCGPU_ERR_INVALID, "unknown stop rule");
  if (p->max_iter < 1 || p->max_iter > 255) return fail(ctx, CCGPU_ERR_INVALID, "max_iter must be in 1..255");
  if ((p->variant == CCGPU_OMS || p->variant == CCGPU_OMS_Q) && !(p->beta >= 0.0)) return fail(ctx, CCGPU_ERR_INVALID, "OMS needs beta >= 0");
  return CCGPU_OK;
}

bool is_fixed(int variant) { return variant >= CCGPU_MS_Q && variant <= CCGPU_OMS_Q; }

// the quantiser of the fixed-point variants with its defaults filled in (include/ccgpu.h)
struct QuantSpec {
  float scale;
  int ymax, mmax, A, B;
};
QuantSpec quant_spec(const ccgpu_ms_params *p) {
  QuantSpec q;
  q.scale = static_cast<float>(p->q_scale > 0.0 ? p->q_scale : 8.0);
  q.ymax = static_cast<int>(p->q_y_max ? p->q_y_max : 31u);
  q.mmax = static_cast<int>(p->q_msg_max ? p->q_msg_max : 31u);
  q.A = p->variant == CCGPU_NMS_Q ? static_cast<int>(std::lrint(p->alpha * 1024.0)) : 1024;
  q.B = p->variant == CCGPU_OMS_Q ? static_cast<int>(std::lrint(p->beta * static_cast<double>(q.scale))) : 0;
  return q;
}
// fn_h of the fixed-point variants on the host (the bound of the device kernel is stated with it)
int fixed_fn_h(const QuantSpec &q, int m) {
  const long long t = static_cast<long long>(q.A) * m, fl = t >> 10, rem = t & 1023;
  const long long v = fl + ((rem > 512 || (rem == 512 && (fl & 1))) ? 1 : 0);
  return static_cast<int>(std::max<long long>(v - q.B, 0));
}
// the two-frames-per-lane kernel carries its integers in fp16 halves: everything must stay within +-2048
int check_params_q(ccgpu_ctx *ctx, const ccgpu_code *c, const ccgpu_ms_params *p) {
  if (!is_fixed(p->variant)) return CCGPU_OK;
  if (p->variant == CCGPU_NMS_Q && !(p->alpha >= 0.0 && p->alpha <= 1.0))
    return fail(ctx, CCGPU_ERR_UNSUPPORTED, "fixed-point NMS needs 0 <= alpha <= 1");
  if (!(p->q_scale >= 0.0) || p->q_scale > 1e6) return fail(ctx, CCGPU_ERR_INVALID, "q_scale out of range");
  const QuantSpec q = quant_spec(p);
  if (q.mmax > 1023 || q.B > 1024 || q.ymax > 2047) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "fixed-point: q_msg_max <= 1023, q_y_max <= 2047, offset <= 1024 steps");
  const long long bound = static_cast<long long>(c->max_col_weight) * fixed_fn_h(q, q.mmax) + q.ymax;
  if (bound > 2048) {
    char msg[200];
    std::snprintf(msg, sizeof msg, "fixed-point: column weight %u x fn_h(q_msg_max) %d + q_y_max %d = %lld exceeds the 2048 the "
                  "packed kernel represents exactly; lower q_msg_max / q_y_max", c->max_col_weight, fixed_fn_h(q, q.mmax), q.ymax, bound);
    return fail(ctx, CCGPU_ERR_UNSUPPORTED, msg);
  }
  return CCGPU_OK;
}

// fills the decoder part of a parameter block
void fill_decoder(MsParams &mp, const ccgpu_code *c, const ccgpu_ms_params *p) {
  mp.n = static_cast<int>(c->spec.n);
  mp.k = static_cast<int>(c->spec.rows);
  mp.variant = p->variant;
  mp.stop_rule = p->stop_rule;
  mp.max_iter = static_cast<int>(p->max_iter);
  mp.alpha_f = static_cast<float>(p->alpha);  // double -> float where the reference's functor call does
  mp.beta_f = static_cast<float>(p->beta);
  mp.beta_d = p->beta;
  // the reference's stop test passes iff every row's integer overlap with b is 0 mod 256; when every
  // column is covered by some row and all row weights are < 256 that is exactly "b is all-zero"
  mp.stop_simple = (p->stop_rule == CCGPU_STOP_REF_ZERO_OVERLAP && c->all_columns_covered && c->shape.max_row_weight < 256) ? 1 : 0;
  if (is_fixed(p->variant)) {
    const QuantSpec q = quant_spec(p);
    mp.q_scale = q.scale;
    mp.q_ymax = q.ymax;
    mp.q_mmax = q.mmax;
    mp.q_alpha = q.A;
    mp.q_beta = q.B;
    auto splat = [](float v) { return 0x10001u * static_cast<uint32_t>(__half_as_ushort(__float2half_rn(v))); };  // exact values
    mp.q_h2_mmax = splat(static_cast<float>(q.mmax));
    mp.q_h2_alpha = splat(static_cast<float>(q.A) / 1024.0f);
    mp.q_h2_1024 = splat(1024.0f);
    mp.q_h2_1024b = splat(static_cast<float>(1024 + q.B));
  }
}

// launch the min-sum decoder for one batch described by mp (source/outputs already filled)
int launch_ms(ccgpu_ctx *ctx, const ccgpu_code *c, const ccgpu_ms_params *p, MsParams mp, int slot = -1) {
  if (mp.frames == 0) return CCGPU_OK;
  cudaStream_t stream = slot < 0 ? ctx->stream : ctx->slot_stream[slot];
  unsigned long long *work = ctx->d_work + (slot + 1);
  const int vn = (p->variant == CCGPU_SCMS1 || p->variant == CCGPU_SCMS2) ? VN_SC
                 : p->variant == CCGPU_NMS2D                             ? VN_2D
                 : p->variant == CCGPU_SPA                               ? VN_SPA
                 : is_fixed(p->variant)                                  ? VN_FIX
                                                                         : VN_PLAIN;
  if (vn == VN_FIX) {
    if (!c->cyc[VN_FIX]) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "fixed-point min-sum runs on the shape-specialised cyclic kernels only");
    const int rc = check_params_q(ctx, c, p);
    if (rc) return rc;
  }
  const MsCyclicEntry *e;
  uint64_t per_cta;
  int grid_max;
  size_t smem;
  // small codes: one lane per frame (ms_cyclic_lane.cuh) for frames from HBM or the Philox channel; the exhaustive
  // bit-flip source and the self-correcting flavour stay on the warp kernel
  if (ctx->opt_lane != 0 && c->lane[vn] && mp.src != SRC_BITFLIP) {
    e = c->lane[vn];
    per_cta = e->threads;
    grid_max = c->lane_grid_max[vn];
    smem = size_t(e->dyn_smem);
  } else {
    // the QUICK instantiation retires all-positive frames without iterating (ms_cyclic.cuh); it pays when such frames
    // are frequent, i.e. in Monte-Carlo points at high Eb/N0 (the hint is set by ccgpu_awgn_point; CCGPU_QUICK=0/1
    // overrides it for every path, which is how the parity tests drive both instantiations over the same inputs)
    // the fixed-point kernels test for all-positive frames at run time when the hint is set; with several frames per
    // warp all of them must be all-positive at once, which is rare: measured slower there (profiles/r2_notes.md)
    if (vn == VN_FIX && c->cyc[VN_FIX] && !c->cyc[VN_FIX]->cta && c->cyc[VN_FIX]->fpw != 1) mp.quick_hint = 0;
    // the float CTA kernel screens groups of frames at any Eb/N0 (ms_cyclic_cta.cuh, grouped mode): no cost where no
    // frame is all-positive, measured in profiles/r2_notes.md
    if (c->cyc[vn] && c->cyc[vn]->cta && mp.src == SRC_PHILOX) mp.quick_hint = 1;
    if (ctx->opt_quick >= 0) mp.quick_hint = ctx->opt_quick;
    const int vq = (mp.quick_hint && vn != VN_SPA && vn != VN_FIX && mp.L == nullptr && p->stop_rule != CCGPU_STOP_NONE && c->cyc[vn + VN_QUICK] &&
                    c->cyc[vn] && !c->cyc[vn]->cta && c->cyc[vn + VN_QUICK]->k == c->cyc[vn]->k && c->cyc[vn + VN_QUICK]->fpw == 1)
                       ? vn + VN_QUICK
                       : vn;
    e = c->cyc[vq];
    if (!e) {
      const int rc = ms_csr_launch(c->csr, mp, ctx->sm_count, stream);
      if (rc == -3) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "parity-check matrix too large for the CSR kernel");
      if (rc != 0) return cuda_fail(ctx, cudaGetLastError(), "ms_csr_launch");
      ctx->launches++;
      return CCGPU_OK;
    }
    per_cta = (e->cta ? 1 : uint64_t(kMsThreads / 32) * e->fpw) * e->slots;
    grid_max = c->grid_max[vq];
    smem = c->smem[vq];
  }
  const unsigned grid = static_cast<unsigned>(std::min<uint64_t>((mp.frames + per_cta - 1) / per_cta, grid_max));
  CU(cudaMemsetAsync(work, 0, sizeof(unsigned long long), stream));
  mp.work = work;
  // guided self-scheduling of the frame queue: a warp takes up to 32 frame indices per atomic while more than
  // 4 x 32 frames per warp are left, fewer towards the end (work_shift = log2(4 x warps))
  const uint64_t warps = uint64_t(grid) * (e->threads / 32);
  unsigned shift = 0;
  while ((uint64_t(1) << shift) < 4 * warps) ++shift;
  mp.work_batch = ctx->opt_work_batch > 0 ? static_cast<unsigned>(ctx->opt_work_batch) : 32;
  mp.work_shift = shift;
  void *args[] = { &mp };
  CU(cudaLaunchKernel(reinterpret_cast<const void *>(e->fn), dim3(grid), dim3(e->threads), args, smem, stream));
  ctx->launches++;
  return CCGPU_OK;
}


// work buffers of multiple-bases decoding: every candidate of `frames` frames, and the rotations
struct MbbpWork {
  float *rolled, *L_b;  // L_b only when the caller wants L
  uint8_t *bits_b, *iter_b, *failed_b;
  uint32_t *shifts;
};
MbbpWork cut_mbbp_work(Arena &a, size_t n, uint32_t nb, uint64_t frames, bool want_L) {
  return { a.take<float>(nb * frames * n), a.take<float>(nb * frames * n, want_L), a.take<uint8_t>(nb * frames * n),
           a.take<uint8_t>(nb * frames),   a.take<uint8_t>(nb * frames),           a.take<uint32_t>(nb) };
}
// the stage arena of one chunk of multiple-bases decoding: channel values and outputs (iter and chosen also stand in
// for the ones a device caller leaves out), then the work buffers
struct MbbpStage {
  float *y, *L;  // L only when the caller wants L
  uint8_t *bits, *iter, *failed, *chosen;
  MbbpWork work;
};
MbbpStage cut_mbbp_stage(Arena &a, size_t n, uint32_t nb, uint64_t frames, bool want_L) {
  return { a.take<float>(frames * n), a.take<float>(frames * n, want_L), a.take<uint8_t>(frames * n),
           a.take<uint8_t>(frames),   a.take<uint8_t>(frames),           a.take<uint8_t>(frames),
           cut_mbbp_work(a, n, nb, frames, want_L) };
}

// multiple-bases decoding of `frames` frames whose channel values are in device memory (d_y), in the work buffers
// `w` cut for at least `frames` frames; outputs are device pointers (L / iter nullable, L only if w has L_b); when
// `counters` is given the Monte-Carlo statistics of the all-zero codeword are accumulated as well.
int mbbp_run(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, const uint32_t *shifts, uint32_t nb,
             const float *d_y, uint64_t frames, const MbbpWork &w, uint8_t *d_bits, float *d_L, uint8_t *d_iter,
             uint8_t *d_failed, uint8_t *d_chosen, unsigned long long *counters) {
  const size_t n = code->spec.n;
  CU(cudaMemcpyAsync(w.shifts, shifts, nb * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  mbbp_roll_kernel<<<grid_for(ctx, nb * frames * n, 256), 256, 0, ctx->stream>>>(d_y, w.rolled, w.shifts,
                                                                                static_cast<uint32_t>(n), nb, frames);
  CU(cudaGetLastError());
  MsParams mp{};
  fill_decoder(mp, code, params);
  mp.src = SRC_HBM;
  mp.frames = nb * frames;
  mp.y = w.rolled;
  mp.bits = w.bits_b;
  mp.L = w.L_b;
  mp.iter = w.iter_b;
  mp.failed = w.failed_b;
  const int rc = launch_ms(ctx, code, params, mp);
  if (rc) return rc;
  mbbp_select_kernel<<<grid_for(ctx, frames, 128), 128, 0, ctx->stream>>>(d_y, w.bits_b, w.iter_b, w.failed_b, w.shifts,
                                                                         static_cast<uint32_t>(n), nb, params->max_iter,
                                                                         frames, d_chosen, d_iter, d_failed, counters);
  CU(cudaGetLastError());
  mbbp_unroll_kernel<<<grid_for(ctx, frames * n, 256), 256, 0, ctx->stream>>>(w.bits_b, w.L_b, d_chosen, w.shifts,
                                                                              static_cast<uint32_t>(n), nb, frames, d_bits,
                                                                              d_L);
  CU(cudaGetLastError());
  ctx->launches += 3;
  if (counters) {
    count_words_kernel<<<grid_for(ctx, frames, 8, 8), 256, 0, ctx->stream>>>(d_bits, d_failed, static_cast<uint32_t>(n),
                                                                             frames, counters);
    CU(cudaGetLastError());
    ctx->launches++;
  }
  return CCGPU_OK;
}
int check_bases(ccgpu_ctx *ctx, const ccgpu_code *code, const uint32_t *shifts, uint32_t nb) {
  if (!shifts || nb == 0 || nb > 64) return fail(ctx, CCGPU_ERR_INVALID, "1..64 bases");
  if (code->spec.family != 0) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "multiple-bases decoding needs a cyclic (BCH) code");
  for (uint32_t b = 0; b < nb; ++b)
    if (shifts[b] >= code->spec.n) return fail(ctx, CCGPU_ERR_INVALID, "rotation must be below n");
  return CCGPU_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
extern "C" {

int ccgpu_abi_version(void) { return CCGPU_ABI_VERSION; }

int ccgpu_create(int device, ccgpu_ctx **out) {
  if (!out) return CCGPU_ERR_INVALID;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
    cudaGetLastError();
    return CCGPU_ERR_NO_DEVICE;
  }
  ccgpu_ctx *ctx = new (std::nothrow) ccgpu_ctx();
  if (!ctx) return CCGPU_ERR_CUDA;
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess ||
      cudaMalloc(&ctx->d_counters, sizeof(ccgpu_counters)) != cudaSuccess ||
      cudaMalloc(&ctx->d_work, (kSlots + 1) * sizeof(unsigned long long)) != cudaSuccess ||
      cudaMallocHost(&ctx->h_counters, sizeof(ccgpu_counters)) != cudaSuccess) {
    cudaGetLastError();
    delete ctx;
    return CCGPU_ERR_CUDA;
  }
  if (const char *env = std::getenv("CCGPU_QUICK")) ctx->opt_quick = std::atoi(env) != 0;
  if (const char *env = std::getenv("CCGPU_WORK_BATCH")) ctx->opt_work_batch = std::max(1, std::atoi(env));
  *out = ctx;
  return CCGPU_OK;
}

void ccgpu_destroy(ccgpu_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->d_stage) cudaFree(ctx->d_stage);
  if (ctx->d_counters) cudaFree(ctx->d_counters);
  if (ctx->d_work) cudaFree(ctx->d_work);
  for (int s = 0; s < kSlots; ++s) {
    if (ctx->slot_stream[s]) {
      cudaStreamSynchronize(ctx->slot_stream[s]);
      cudaStreamDestroy(ctx->slot_stream[s]);
    }
    if (ctx->slot_buf[s]) cudaFree(ctx->slot_buf[s]);
  }
  if (ctx->main_ready) cudaEventDestroy(ctx->main_ready);
  if (ctx->h_counters) cudaFreeHost(ctx->h_counters);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char *ccgpu_last_error(const ccgpu_ctx *ctx) {
  // a copy per calling thread: the context's string may be rewritten by another pool thread at any time
  thread_local std::string copy;
  if (!ctx) return "no context";
  {
    std::lock_guard<std::mutex> g(const_cast<ccgpu_ctx *>(ctx)->err_mu);
    copy = ctx->err;
  }
  return copy.c_str();
}

int ccgpu_set_option(ccgpu_ctx *ctx, const char *name, int64_t value) {
  if (!ctx || !name) return CCGPU_ERR_INVALID;
  std::lock_guard<std::mutex> g(ctx->mu);
  const std::string n(name);
  if (n == "quick") ctx->opt_quick = value < 0 ? -1 : (value ? 1 : 0);
  else if (n == "lane") ctx->opt_lane = value < 0 ? -1 : (value ? 1 : 0);
  else if (n == "work_batch") ctx->opt_work_batch = value > 0 ? static_cast<int>(std::min<int64_t>(value, 1024)) : 0;
  else return fail(ctx, CCGPU_ERR_INVALID, "unknown option " + n);
  return CCGPU_OK;
}

const char *ccgpu_build_info(void) {
#define CCGPU_STR_(x) #x
#define CCGPU_STR(x) CCGPU_STR_(x)
  return "nvcc " CCGPU_STR(__CUDACC_VER_MAJOR__) "." CCGPU_STR(__CUDACC_VER_MINOR__) "." CCGPU_STR(__CUDACC_VER_BUILD__)
         " sm_100a abi " CCGPU_STR(CCGPU_ABI_VERSION);
}

int ccgpu_set_stream(ccgpu_ctx *ctx, void *cuda_stream) {
  if (!ctx) return CCGPU_ERR_INVALID;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (ctx->own_stream && ctx->stream) {
    cudaStreamSynchronize(ctx->stream);
    cudaStreamDestroy(ctx->stream);
  }
  ctx->stream = static_cast<cudaStream_t>(cuda_stream);
  ctx->own_stream = false;
  return CCGPU_OK;
}
void *ccgpu_get_stream(ccgpu_ctx *ctx) { return ctx ? static_cast<void *>(ctx->stream) : nullptr; }

int ccgpu_sync(ccgpu_ctx *ctx) {
  if (!ctx) return CCGPU_ERR_INVALID;
  CU(cudaStreamSynchronize(ctx->stream));
  return CCGPU_OK;
}
uint64_t ccgpu_kernel_launches(const ccgpu_ctx *ctx) { return ctx ? ctx->launches.load() : 0; }

// ---- codes -------------------------------------------------------------------------------------
static int make_code(ccgpu_ctx *ctx, CodeSpec &&spec, ccgpu_code **out) {
  ccgpu_code *c = new ccgpu_code();
  c->spec = std::move(spec);
  if (ctx) cudaSetDevice(ctx->device);
  const int rc = finish_code(ctx, c);
  if (rc != CCGPU_OK) {
    ccgpu_code_destroy(c);
    return rc;
  }
  *out = c;
  return CCGPU_OK;
}

int ccgpu_bch_create(ccgpu_ctx *ctx, uint32_t q, int cap_kind, uint32_t cap_value, ccgpu_code **out) {
  if (!out) return CCGPU_ERR_INVALID;
  std::unique_lock<std::mutex> g;
  if (ctx) g = std::unique_lock<std::mutex>(ctx->mu);
  try {
    return make_code(ctx, make_bch(q, cap_kind, cap_value), out);
  } catch (const std::exception &e) {
    return fail(ctx, CCGPU_ERR_INVALID, e.what());
  }
}

int ccgpu_rs_create(ccgpu_ctx *ctx, uint32_t q, uint32_t t, uint32_t mu, uint32_t step, ccgpu_code **out) {
  if (!out) return CCGPU_ERR_INVALID;
  std::unique_lock<std::mutex> g;
  if (ctx) g = std::unique_lock<std::mutex>(ctx->mu);
  try {
    return make_code(ctx, make_rs(q, t, mu, step), out);
  } catch (const std::exception &e) {
    return fail(ctx, CCGPU_ERR_INVALID, e.what());
  }
}

int ccgpu_code_from_dense(ccgpu_ctx *ctx, const uint8_t *H, uint32_t rows, uint32_t cols, double rate, ccgpu_code **out) {
  if (!out || !H || rows == 0 || cols == 0) return CCGPU_ERR_INVALID;
  std::unique_lock<std::mutex> g;
  if (ctx) g = std::unique_lock<std::mutex>(ctx->mu);
  try {  // the ABI never throws: allocation failures come back as an error code
    CodeSpec s;
    s.family = 2;
    s.n = cols;
    s.rows = rows;
    s.k = rows;
    s.l = cols > rows ? cols - rows : 0;
    s.rate = rate;
    s.H.assign(H, H + size_t(rows) * cols);
    for (auto &v : s.H) v = v ? 1 : 0;
    return make_code(ctx, std::move(s), out);
  } catch (const std::exception &e) {
    return ctx ? fail(ctx, CCGPU_ERR_INVALID, e.what()) : CCGPU_ERR_INVALID;
  }
}

int ccgpu_code_set_rows(ccgpu_code *code, uint32_t rows) {
  if (!code) return CCGPU_ERR_INVALID;
  ccgpu_ctx *ctx = code->ctx;
  std::unique_lock<std::mutex> g;
  if (ctx) g = std::unique_lock<std::mutex>(ctx->mu);
  try {
    if (rows < code->spec.k) return fail(ctx, CCGPU_ERR_INVALID, "rows must be >= k");
    code->spec.set_rows(rows);
  } catch (const std::exception &e) {
    return fail(ctx, CCGPU_ERR_INVALID, e.what());
  }
  if (ctx) {  // the kernels of earlier calls may still read the CSR tables
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
  }
  return refresh_H(code);
}

void ccgpu_code_destroy(ccgpu_code *code) {
  if (!code) return;
  if (code->ctx) {
    cudaSetDevice(code->ctx->device);
    cudaStreamSynchronize(code->ctx->stream);
  }
  ms_csr_free(&code->csr);
  gf_free(&code->gf);
  osd_free(&code->osd);
  delete code;
}

int ccgpu_code_get_info(const ccgpu_code *code, ccgpu_code_info *out) {
  if (!code || !out) return CCGPU_ERR_INVALID;
  std::memset(out, 0, sizeof(*out));
  const CodeSpec &s = code->spec;
  out->family = s.family;
  out->q = s.q;
  out->n = s.n;
  out->l = s.l;
  out->k = s.k;
  out->dmin = s.dmin;
  out->t = s.t;
  out->h_rows = s.rows;
  out->row_weight = code->shape.max_row_weight;
  out->edges = code->shape.edges;
  out->h_kind = code->shape.kind;
  out->kernel = !code->ctx ? 0 : (code->cyc[0] ? 1 : 2);
  out->rate = s.rate;
  return CCGPU_OK;
}

int ccgpu_code_to_string(const ccgpu_code *code, const char *tag, char *buf, size_t cap) {
  if (!code || !buf || cap == 0) return CCGPU_ERR_INVALID;
  try {
    std::snprintf(buf, cap, "%s", code->spec.to_string(tag ? tag : "").c_str());
  } catch (const std::exception &) {
    return CCGPU_ERR_INVALID;
  }
  return CCGPU_OK;
}

int ccgpu_code_H(const ccgpu_code *code, uint8_t *out) {
  if (!code || !out) return CCGPU_ERR_INVALID;
  std::memcpy(out, code->spec.H.data(), code->spec.H.size());
  return CCGPU_OK;
}

int ccgpu_code_H_alt(const ccgpu_code *code, int as_reference, uint8_t *out, uint32_t *rows) {
  if (!code || !rows || code->spec.family == 2) return CCGPU_ERR_INVALID;
  try {
    unsigned r = 0;
    const std::vector<uint8_t> M = code->spec.h_alt(as_reference != 0, &r);
    *rows = r;
    if (out) std::memcpy(out, M.data(), M.size());
  } catch (const std::exception &) {
    return CCGPU_ERR_INVALID;
  }
  return CCGPU_OK;
}

int ccgpu_code_poly(const ccgpu_code *code, int which, uint16_t *out, size_t cap) {
  if (!code || !out) return CCGPU_ERR_INVALID;
  const Poly &p = which ? code->spec.h : code->spec.g;
  if (p.size() > cap) return CCGPU_ERR_INVALID;
  std::copy(p.begin(), p.end(), out);
  return static_cast<int>(p.size());
}

int ccgpu_gf_tables(uint32_t q, uint32_t poly, uint16_t *exp_out, uint16_t *log_out) {
  if (!exp_out || !log_out) return CCGPU_ERR_INVALID;
  try {
    Field F(q, poly);
    std::copy(F.exp.begin(), F.exp.end(), exp_out);
    std::copy(F.log.begin(), F.log.end(), log_out);
  } catch (const std::exception &) {
    return CCGPU_ERR_INVALID;
  }
  return CCGPU_OK;
}

int ccgpu_encode(const ccgpu_code *code, const uint8_t *msgs, uint64_t count, uint8_t *words) {
  if (!code || !msgs || !words || code->spec.family == 2) return CCGPU_ERR_INVALID;
  try {
    for (uint64_t i = 0; i < count; ++i) code->spec.encode(msgs + i * code->spec.l, words + i * code->spec.n);
  } catch (const std::exception &e) {
    return fail(code->ctx, CCGPU_ERR_INVALID, e.what());
  }
  return CCGPU_OK;
}

double ccgpu_sigma(double rate, double ebno_db) {
  // simulation.c++:83-85 evaluates 1.0f / sqrt(2 R 10^(EbN0/10)) in double
  return 1.0f / std::sqrt(2 * rate * std::pow(10, ebno_db / 10.0));
}

static double biawgn_capacity(double snr) {  // bit/use at Es/N0 = snr (linear); LLR ~ N(4 snr, 8 snr)
  const double mean = 4.0 * snr, sd = std::sqrt(8.0 * snr);
  const int steps = 4000;
  const double lo = mean - 10 * sd, hi = mean + 10 * sd, dx = (hi - lo) / steps;
  double acc = 0;
  for (int i = 0; i <= steps; ++i) {
    const double x = lo + i * dx;
    const double pdf = std::exp(-0.5 * (x - mean) * (x - mean) / (sd * sd)) / (sd * std::sqrt(2 * M_PI));
    const double f = (x > 30 ? std::exp(-x) : std::log1p(std::exp(-x))) / std::log(2.0);
    acc += (i == 0 || i == steps ? 0.5 : 1.0) * pdf * f * dx;
  }
  return 1.0 - acc;
}

// The reference's table of the Shannon limit Eb/N0 [dB] of the binary-input AWGN channel (simulation.c++:21-52): 131
// (rate, limit) pairs, rates 0.01 .. 0.80 in steps of 0.01, then an irregular grid up to 0.999.  The sweep start of
// every decoder -- hence the points of every log file -- derives from these very numbers, so they are reproduced as
// data, not recomputed (a numerically computed limit is 2.419 dB at rate 0.8387 where the table's rounded-up entry is
// 2.503 dB: BCH(31,26) then starts at 3.0 instead of 3.5 dB).
static const double kShannonRates[131] = {
  0.01,  0.02,  0.03,  0.04,  0.05,  0.06,  0.07,  0.08,  0.09,  0.10,  0.11,  0.12,  0.13,  0.14,  0.15,  0.16,  0.17,
  0.18,  0.19,  0.20,  0.21,  0.22,  0.23,  0.24,  0.25,  0.26,  0.27,  0.28,  0.29,  0.30,  0.31,  0.32,  0.33,  0.34,
  0.35,  0.36,  0.37,  0.38,  0.39,  0.40,  0.41,  0.42,  0.43,  0.44,  0.45,  0.46,  0.47,  0.48,  0.49,  0.50,  0.51,
  0.52,  0.53,  0.54,  0.55,  0.56,  0.57,  0.58,  0.59,  0.60,  0.61,  0.62,  0.63,  0.64,  0.65,  0.66,  0.67,  0.68,
  0.69,  0.70,  0.71,  0.72,  0.73,  0.74,  0.75,  0.76,  0.77,  0.78,  0.79,  0.800, 0.807, 0.817, 0.827, 0.837, 0.846,
  0.855, 0.864, 0.872, 0.880, 0.887, 0.894, 0.900, 0.907, 0.913, 0.918, 0.924, 0.929, 0.934, 0.938, 0.943, 0.947, 0.951,
  0.954, 0.958, 0.961, 0.964, 0.967, 0.970, 0.972, 0.974, 0.976, 0.978, 0.980, 0.982, 0.983, 0.984, 0.985, 0.986, 0.987,
  0.988, 0.989, 0.990, 0.991, 0.992, 0.993, 0.994, 0.995, 0.996, 0.997, 0.998, 0.999 };
static const double kShannonLimits[131] = {
  -1.548, -1.531, -1.500, -1.470, -1.440, -1.409, -1.378, -1.347, -1.316, -1.285, -1.254, -1.222, -1.190, -1.158, -1.126,
  -1.094, -1.061, -1.028, -0.995, -0.963, -0.928, -0.896, -0.861, -0.827, -0.793, -0.757, -0.724, -0.687, -0.651, -0.616,
  -0.579, -0.544, -0.507, -0.469, -0.432, -0.394, -0.355, -0.314, -0.276, -0.236, -0.198, -0.156, -0.118, -0.074, -0.032,
  0.010,  0.055,  0.097,  0.144,  0.188,  0.233,  0.279,  0.326,  0.374,  0.424,  0.474,  0.526,  0.574,  0.628,  0.682,
  0.734,  0.791,  0.844,  0.904,  0.960,  1.021,  1.084,  1.143,  1.208,  1.275,  1.343,  1.412,  1.483,  1.554,  1.628,
  1.708,  1.784,  1.867,  1.952,  2.045,  2.108,  2.204,  2.302,  2.402,  2.503,  2.600,  2.712,  2.812,  2.913,  3.009,
  3.114,  3.205,  3.312,  3.414,  3.500,  3.612,  3.709,  3.815,  3.906,  4.014,  4.115,  4.218,  4.304,  4.425,  4.521,
  4.618,  4.725,  4.841,  4.922,  5.004,  5.104,  5.196,  5.307,  5.418,  5.484,  5.549,  5.615,  5.681,  5.756,  5.842,
  5.927,  6.023,  6.119,  6.234,  6.360,  6.495,  6.651,  6.837,  7.072,  7.378,  7.864 };

// ebno(rate) of simulation.c++:56-70: rate <= 0.8 indexes the table with size_t(rate * 100) (that is the entry of the
// next tabulated rate, the table starts at 0.01), rate >= 0.999 takes the last entry, anything between the first
// tabulated rate >= rate from index 80 on.  Rates outside (0, 1] have no entry in the reference (it would throw /
// read out of range): the first / last entry is returned.
double ccgpu_shannon_limit_db(double rate) {
  if (!(rate > 0.0)) return kShannonLimits[0];
  if (rate <= 0.800) return kShannonLimits[static_cast<size_t>(rate * 100)];
  if (rate >= 0.999) return kShannonLimits[130];
  size_t i = 80;
  while (i < 130 && !(kShannonRates[i] >= rate)) ++i;
  return kShannonLimits[i];
}

// the same limit computed from the channel capacity (numerical integral + bisection); not used by the sweep, kept as
// a cross-check of the table (tests/test_host_abi.py) and for callers who want the exact figure of an arbitrary rate
double ccgpu_shannon_limit_db_numeric(double rate) {
  if (!(rate > 0.0)) return -1.59;
  const double r = std::min(rate, 0.9995);
  double lo = -3.0, hi = 12.0;
  for (int i = 0; i < 60; ++i) {
    const double mid = 0.5 * (lo + hi);
    if (biawgn_capacity(r * std::pow(10.0, mid / 10.0)) < r) lo = mid;
    else hi = mid;
  }
  return 0.5 * (lo + hi);
}

double ccgpu_sweep_start_ebno(double rate, double step) {
  const double lim = std::max(0.0, ccgpu_shannon_limit_db(rate));
  const size_t tmp = static_cast<size_t>(lim / step);
  return (tmp + (1.0 / step)) * step;
}

uint64_t ccgpu_sweep_samples(double previous_wer, uint64_t cap) {
  if (!(previous_wer > 0.0)) return cap;
  return static_cast<uint64_t>(std::min(static_cast<double>(cap), 5e3 / previous_wer));
}

// ---- decoding ----------------------------------------------------------------------------------
// one implementation behind ccgpu_decode_llr (the reference's layout: one byte per decided bit, iter, failed) and
// ccgpu_decode_llr_packed (compact layout: ceil(n/32) words of decided bits + one status byte per frame)
static int decode_llr_impl(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, const float *y,
                           uint64_t frames, uint8_t *bits, float *L, uint8_t *iter, uint8_t *failed, uint32_t *packed,
                           uint8_t *status) {
  std::lock_guard<std::mutex> g(ctx->mu);
  int rc = check_params(ctx, params);
  if (rc) return rc;
  if (frames == 0) return CCGPU_OK;
  CU(cudaSetDevice(ctx->device));
  const size_t n = code->spec.n, npw = (n + 31) / 32;
  MsParams mp{};
  fill_decoder(mp, code, params);
  mp.src = SRC_HBM;
  mp.frames = frames;
  if (is_device_ptr(y)) {
    if (!same_residency(true, {bits, failed, L, iter, packed, status}))
      return fail(ctx, CCGPU_ERR_INVALID, "y is a device pointer: every output must be one too");
    mp.y = y;
    mp.bits = bits;
    mp.L = L;
    mp.iter = iter;
    mp.failed = failed;
    mp.packed = packed;
    mp.status = status;
    return launch_ms(ctx, code, params, mp);
  }
  const HostField fields[] = { { n * sizeof(float), y, false },       { n * sizeof(float), L, true },
                               { npw * sizeof(uint32_t), packed, true }, { n, bits, true },
                               { 1, iter, true },                      { 1, failed, true },
                               { 1, status, true } };
  return host_pipeline(ctx, frames, fields, [&](void *const *d, uint64_t nf, cudaStream_t, int slot) {
    mp.y = static_cast<const float *>(d[0]);
    mp.L = static_cast<float *>(d[1]);
    mp.packed = static_cast<uint32_t *>(d[2]);
    mp.bits = static_cast<uint8_t *>(d[3]);
    mp.iter = static_cast<uint8_t *>(d[4]);
    mp.failed = static_cast<uint8_t *>(d[5]);
    mp.status = static_cast<uint8_t *>(d[6]);
    mp.frames = nf;
    return launch_ms(ctx, code, params, mp, slot);
  });
}

int ccgpu_decode_llr(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, const float *y,
                     uint64_t frames, uint8_t *bits, float *L, uint8_t *iter, uint8_t *failed) {
  if (!ctx || !code || !y || !bits || !failed) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  if (int rc = check_code(ctx, code)) return rc;
  return decode_llr_impl(ctx, code, params, y, frames, bits, L, iter, failed, nullptr, nullptr);
}

int ccgpu_decode_llr_packed(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, const float *y,
                            uint64_t frames, uint32_t *packed, uint8_t *status) {
  if (!ctx || !code || !y || !packed || !status) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  if (int rc = check_code(ctx, code)) return rc;
  return decode_llr_impl(ctx, code, params, y, frames, nullptr, nullptr, nullptr, nullptr, packed, status);
}

int ccgpu_awgn_llr(ccgpu_ctx *ctx, uint32_t n, double sigma, uint64_t seed, uint32_t point, uint64_t frame0,
                   uint64_t frames, float *y) {
  if (!ctx || !y || n == 0) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> g(ctx->mu);
  if (frames == 0) return CCGPU_OK;
  CU(cudaSetDevice(ctx->device));
  const bool dev = is_device_ptr(y);
  float *d_y = y;
  if (!dev) {
    const int rc = cut_stage(ctx, [&](Arena &a) { d_y = a.take<float>(frames * n); });
    if (rc) return rc;
  }
  const int rc = launch_awgn(ctx, d_y, n, static_cast<float>(sigma), seed, point, frame0, frames);
  if (rc) return rc;
  if (!dev) {
    CU(cudaMemcpyAsync(y, d_y, frames * n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  return CCGPU_OK;
}

int ccgpu_awgn_point(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, double ebno_db,
                     uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!ctx || !code || !out) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  if (int rc = check_code(ctx, code)) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  int rc = check_params(ctx, params);
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  MsParams mp{};
  fill_decoder(mp, code, params);
  mp.src = SRC_PHILOX;
  mp.sigma = static_cast<float>(ccgpu_sigma(code->spec.rate, ebno_db));  // simulation.c++:113-115
  // the min-sum family is scale invariant and takes the raw channel values like the reference; the
  // sum-product extension needs log-likelihood ratios 2 y / sigma^2
  mp.llr_scale = params->variant == CCGPU_SPA ? 2.0f / (mp.sigma * mp.sigma) : 1.0f;
  mp.seed = seed;
  mp.keys = philox_round_keys(seed);
  {  // share of frames whose n channel values are all positive: (1 - Q(1 / sigma))^n
    const double q = 0.5 * std::erfc(1.0 / (static_cast<double>(mp.sigma) * std::sqrt(2.0)));
    // measured on BCH(63,36): the QUICK kernel is 3.5 % slower at 4 dB (5 % such frames), 7 % faster at 6 dB (35 %),
    // 27 % faster at 7 dB (59 %), 50 % faster at 8 dB (78 %); shapes with several frames per warp do not gain
    mp.quick_hint = std::pow(1.0 - q, static_cast<double>(code->spec.n)) >= 0.25 ? 1 : 0;
    if (is_fixed(params->variant)) {
      // fixed point: "positive" is decided after quantisation (y * scale rounds to >= 1); the two-slot kernel skips an
      // iteration only when BOTH slots hold such frames: measured to pay from about half of the frames on
      const QuantSpec qs = quant_spec(params);
      const double qq = 0.5 * std::erfc((1.0 - 0.5 / qs.scale) / (static_cast<double>(mp.sigma) * std::sqrt(2.0)));
      mp.quick_hint = std::pow(1.0 - qq, static_cast<double>(code->spec.n)) >= 0.5 ? 1 : 0;
    }
  }
  mp.point = point;
  mp.frame0 = frame0;
  mp.frames = frames;
  return with_counters(ctx, out, [&](unsigned long long *counters) {
    mp.counters = counters;
    return launch_ms(ctx, code, params, mp);
  });
}

int ccgpu_decode_llr_mbbp(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, const uint32_t *shifts,
                          uint32_t n_bases, const float *y, uint64_t frames, uint8_t *bits, float *L, uint8_t *iter,
                          uint8_t *failed, uint8_t *chosen) {
  if (!ctx || !code || !y || !bits || !failed) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  if (int rc = check_code(ctx, code)) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  int rc = check_params(ctx, params);
  if (rc) return rc;
  rc = check_bases(ctx, code, shifts, n_bases);
  if (rc) return rc;
  if (frames == 0) return CCGPU_OK;
  CU(cudaSetDevice(ctx->device));
  const size_t n = code->spec.n;
  const bool dev = is_device_ptr(y);
  if (dev && !same_residency(true, {bits, failed, L, iter, chosen}))
    return fail(ctx, CCGPU_ERR_INVALID, "y is a device pointer: every output must be one too");
  // chunks bound the work arena (all candidates of a chunk are decoded in one launch)
  Arena one;
  cut_mbbp_work(one, n, n_bases, 1, L != nullptr);
  const size_t per_frame = one.used + n * (sizeof(float) * 2 + 1) + 3;
  const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>(frames, (size_t(512) << 20) / per_frame));
  MbbpStage s;
  rc = cut_stage(ctx, [&](Arena &a) { s = cut_mbbp_stage(a, n, n_bases, chunk, L != nullptr); });
  if (rc) return rc;
  for (uint64_t f0 = 0; f0 < frames; f0 += chunk) {
    const uint64_t nf = std::min(chunk, frames - f0);
    if (dev) {
      rc = mbbp_run(ctx, code, params, shifts, n_bases, y + f0 * n, nf, s.work, bits + f0 * n, L ? L + f0 * n : nullptr,
                    iter ? iter + f0 : s.iter, failed + f0, chosen ? chosen + f0 : s.chosen, nullptr);
      if (rc) return rc;
    } else {
      CU(cudaMemcpyAsync(s.y, y + f0 * n, nf * n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
      rc = mbbp_run(ctx, code, params, shifts, n_bases, s.y, nf, s.work, s.bits, s.L, s.iter, s.failed, s.chosen, nullptr);
      if (rc) return rc;
      CU(cudaMemcpyAsync(bits + f0 * n, s.bits, nf * n, cudaMemcpyDeviceToHost, ctx->stream));
      if (L) CU(cudaMemcpyAsync(L + f0 * n, s.L, nf * n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
      if (iter) CU(cudaMemcpyAsync(iter + f0, s.iter, nf, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaMemcpyAsync(failed + f0, s.failed, nf, cudaMemcpyDeviceToHost, ctx->stream));
      if (chosen) CU(cudaMemcpyAsync(chosen + f0, s.chosen, nf, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaStreamSynchronize(ctx->stream));  // the staging buffers are reused by the next chunk
    }
  }
  return CCGPU_OK;
}

int ccgpu_awgn_point_mbbp(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, const uint32_t *shifts,
                          uint32_t n_bases, double ebno_db, uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames,
                          ccgpu_counters *out) {
  if (!ctx || !code || !out) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  if (int rc = check_code(ctx, code)) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  int rc = check_params(ctx, params);
  if (rc) return rc;
  rc = check_bases(ctx, code, shifts, n_bases);
  if (rc) return rc;
  CU(cudaSetDevice(ctx->device));
  if (params->variant == CCGPU_SPA) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "multiple-bases points take the min-sum variants");
  const size_t n = code->spec.n;
  Arena one;
  cut_mbbp_work(one, n, n_bases, 1, false);
  const size_t per_frame = one.used + n * (sizeof(float) + 1) + 3;
  const uint64_t chunk = std::max<uint64_t>(4, std::min<uint64_t>(std::max<uint64_t>(frames, 4), (size_t(512) << 20) / per_frame) & ~uint64_t(3));
  const float sigma = static_cast<float>(ccgpu_sigma(code->spec.rate, ebno_db));
  return with_counters(ctx, out, [&](unsigned long long *counters) -> int {
    MbbpStage s;
    rc = cut_stage(ctx, [&](Arena &a) { s = cut_mbbp_stage(a, n, n_bases, chunk, false); });
    if (rc) return rc;
    for (uint64_t f0 = 0; f0 < frames; f0 += chunk) {
      const uint64_t nf = std::min(chunk, frames - f0);
      rc = launch_awgn(ctx, s.y, static_cast<uint32_t>(n), sigma, seed, point, frame0 + f0, nf);
      if (rc) return rc;
      rc = mbbp_run(ctx, code, params, shifts, n_bases, s.y, nf, s.work, s.bits, nullptr, s.iter, s.failed, s.chosen, counters);
      if (rc) return rc;
    }
    return CCGPU_OK;
  });
}

int ccgpu_awgn_point_uncoded(ccgpu_ctx *ctx, uint32_t n, double rate, double ebno_db, uint64_t seed, uint32_t point,
                             uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!ctx || !out || n == 0) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  if (!(rate > 0.0)) return fail(ctx, CCGPU_ERR_INVALID, "rate must be positive");
  std::lock_guard<std::mutex> g(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  return with_counters(ctx, out, [&](unsigned long long *counters) -> int {
    if (frames) {
      awgn_uncoded_kernel<<<grid_for(ctx, frames, 8, 8), 256, 0, ctx->stream>>>(
          n, static_cast<float>(ccgpu_sigma(rate, ebno_db)), philox_round_keys(seed), point, frame0, frames, counters);
      CU(cudaGetLastError());
      ctx->launches++;
    }
    return CCGPU_OK;
  });
}

int ccgpu_bitflip_point(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, uint32_t weight,
                        uint64_t first, uint64_t count, ccgpu_counters *out) {
  if (!ctx || !code || !out) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  if (int rc = check_code(ctx, code)) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  int rc = check_params(ctx, params);
  if (rc) return rc;
  const unsigned n = code->spec.n;
  if (weight > n) return fail(ctx, CCGPU_ERR_INVALID, "weight > n");
  long double total = 1;
  for (unsigned i = 1; i <= weight; ++i) total = total * (n - weight + i) / i;
  if (total > 1.8e19L) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "C(n, weight) does not fit 64 bits");
  const uint64_t patterns = static_cast<uint64_t>(total + 0.5L);
  if (first > patterns) return fail(ctx, CCGPU_ERR_INVALID, "first > C(n, weight)");
  if (count == 0 || count > patterns - first) count = patterns - first;
  CU(cudaSetDevice(ctx->device));
  MsParams mp{};
  fill_decoder(mp, code, params);
  mp.src = SRC_BITFLIP;
  mp.flip_weight = weight;
  mp.frame0 = first;
  mp.frames = count;
  return with_counters(ctx, out, [&](unsigned long long *counters) {
    mp.counters = counters;
    return launch_ms(ctx, code, params, mp);
  });
}

static int gf_rc(ccgpu_ctx *ctx, int rc) {
  if (rc == -3) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "code not supported by the algebraic kernel (t <= 31, 2t <= 64, step = 1)");
  if (rc != 0) return cuda_fail(ctx, cudaGetLastError(), "gf_launch");
  ctx->launches++;
  return CCGPU_OK;
}

int ccgpu_gf_decode_erasures(ccgpu_ctx *ctx, const ccgpu_code *code, const uint8_t *words, uint64_t count,
                             const uint8_t *erasure_pos, const uint8_t *erasure_cnt, uint32_t max_erasures,
                             uint8_t *corrected, uint8_t *n_errors, uint8_t *failed) {
  if (!ctx || !code || !words || !corrected || !failed) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  if (int rc = check_code(ctx, code)) return rc;
  if (code->spec.family == 2) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "algebraic decoding needs a BCH/RS code");
  if ((erasure_pos == nullptr) != (erasure_cnt == nullptr)) return fail(ctx, CCGPU_ERR_INVALID, "erasure_pos and erasure_cnt go together");
  if (erasure_pos && (max_erasures == 0 || max_erasures > 30)) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "max_erasures must be in 1..30");
  std::lock_guard<std::mutex> g(ctx->mu);
  if (count == 0) return CCGPU_OK;
  CU(cudaSetDevice(ctx->device));
  const size_t n = code->spec.n;
  const int me = erasure_pos ? static_cast<int>(max_erasures) : 0;
  if (is_device_ptr(words)) {
    if (!same_residency(true, {corrected, failed, n_errors, erasure_pos, erasure_cnt}))
      return fail(ctx, CCGPU_ERR_INVALID, "words is a device pointer: every other buffer must be one too");
    return gf_rc(ctx, gf_launch(code->gf, words, count, erasure_pos, erasure_cnt, me, corrected, n_errors, failed,
                                ctx->sm_count, ctx->stream));
  }
  const HostField fields[] = { { n, words, false },  { size_t(me), erasure_pos, false }, { 1, erasure_cnt, false },
                               { n, corrected, true }, { 1, n_errors, true },             { 1, failed, true } };
  return host_pipeline(ctx, count, fields, [&](void *const *d, uint64_t nw, cudaStream_t st, int) {
    return gf_rc(ctx, gf_launch(code->gf, static_cast<const uint8_t *>(d[0]), nw, static_cast<const uint8_t *>(d[1]),
                                static_cast<const uint8_t *>(d[2]), me, static_cast<uint8_t *>(d[3]),
                                static_cast<uint8_t *>(d[4]), static_cast<uint8_t *>(d[5]), ctx->sm_count, st));
  });
}

int ccgpu_gf_decode_erasures_pgz(ccgpu_ctx *ctx, const ccgpu_code *code, const uint8_t *words, uint64_t count,
                                 const uint8_t *erasure_pos, const uint8_t *erasure_cnt, uint32_t max_erasures,
                                 uint8_t *corrected, uint8_t *n_errors, uint8_t *failed) {
  if (!ctx || !code || !words || !corrected || !failed || !erasure_pos || !erasure_cnt)
    return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  if (int rc = check_code(ctx, code)) return rc;
  if (code->spec.family != 0) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "the zero/one fill rule is for binary BCH codes");
  if (max_erasures == 0 || max_erasures > 255) return fail(ctx, CCGPU_ERR_INVALID, "max_erasures must be in 1..255");
  std::lock_guard<std::mutex> g(ctx->mu);
  if (count == 0) return CCGPU_OK;
  CU(cudaSetDevice(ctx->device));
  const size_t n = code->spec.n, me = max_erasures;
  const bool dev = is_device_ptr(words);
  if (dev && !same_residency(true, {corrected, failed, n_errors, erasure_pos, erasure_cnt}))
    return fail(ctx, CCGPU_ERR_INVALID, "words is a device pointer: every other buffer must be one too");
  const size_t per_word = 4 * n + 4 + (dev ? 0 : 2 * n + 3 + me);
  const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>(count, (size_t(256) << 20) / per_word));
  // both fills of every word, the decoder's outputs for them, then the staging of host buffers
  uint8_t *d_fill, *d_cand, *d_cne, *d_cfail, *s_in, *s_out, *s_ne, *s_fail, *s_ec, *s_ep;
  int rc = cut_stage(ctx, [&](Arena &a) {
    d_fill = a.take<uint8_t>(2 * chunk * n);
    d_cand = a.take<uint8_t>(2 * chunk * n);
    d_cne = a.take<uint8_t>(2 * chunk);
    d_cfail = a.take<uint8_t>(2 * chunk);
    s_in = a.take<uint8_t>(chunk * n, !dev);
    s_out = a.take<uint8_t>(chunk * n, !dev);
    s_ne = a.take<uint8_t>(chunk, !dev);
    s_fail = a.take<uint8_t>(chunk, !dev);
    s_ec = a.take<uint8_t>(chunk, !dev);
    s_ep = a.take<uint8_t>(chunk * me, !dev);
  });
  if (rc) return rc;
  for (uint64_t w0 = 0; w0 < count; w0 += chunk) {
    const uint64_t nw = std::min(chunk, count - w0);
    const uint8_t *in = words + w0 * n, *ep = erasure_pos + w0 * me, *ec = erasure_cnt + w0;
    uint8_t *out = corrected + w0 * n, *ne = n_errors ? n_errors + w0 : nullptr, *fl = failed + w0;
    if (!dev) {
      CU(cudaMemcpyAsync(s_in, in, nw * n, cudaMemcpyHostToDevice, ctx->stream));
      CU(cudaMemcpyAsync(s_ep, ep, nw * me, cudaMemcpyHostToDevice, ctx->stream));
      CU(cudaMemcpyAsync(s_ec, ec, nw, cudaMemcpyHostToDevice, ctx->stream));
      in = s_in, ep = s_ep, ec = s_ec, out = s_out, ne = s_ne, fl = s_fail;
    }
    const unsigned grid = grid_for(ctx, nw * n, 256);
    pgz_fill_kernel<<<grid, 256, 0, ctx->stream>>>(in, ep, ec, static_cast<uint32_t>(me), static_cast<uint32_t>(n), nw, d_fill);
    CU(cudaGetLastError());
    rc = gf_rc(ctx, gf_launch(code->gf, d_fill, 2 * nw, nullptr, nullptr, 0, d_cand, d_cne, d_cfail, ctx->sm_count, ctx->stream));
    if (rc) return rc;
    pgz_select_kernel<<<grid, 256, 0, ctx->stream>>>(in, d_cand, d_cne, d_cfail, ec, code->spec.t, static_cast<uint32_t>(n), nw, out,
                                                     ne, fl);
    CU(cudaGetLastError());
    ctx->launches += 2;
    if (!dev) {
      CU(cudaMemcpyAsync(corrected + w0 * n, s_out, nw * n, cudaMemcpyDeviceToHost, ctx->stream));
      if (n_errors) CU(cudaMemcpyAsync(n_errors + w0, s_ne, nw, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaMemcpyAsync(failed + w0, s_fail, nw, cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaStreamSynchronize(ctx->stream));
    }
  }
  return CCGPU_OK;
}

int ccgpu_gf_decode(ccgpu_ctx *ctx, const ccgpu_code *code, const uint8_t *words, uint64_t count,
                    uint8_t *corrected, uint8_t *n_errors, uint8_t *failed) {
  return ccgpu_gf_decode_erasures(ctx, code, words, count, nullptr, nullptr, 0, corrected, n_errors, failed);
}

int ccgpu_awgn_point_hard(ccgpu_ctx *ctx, const ccgpu_code *code, double ebno_db, uint64_t seed, uint32_t point,
                          uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!ctx || !code || !out) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  if (int rc = check_code(ctx, code)) return rc;
  if (code->spec.family != 0) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "hard-decision AWGN points need a binary BCH code");
  std::lock_guard<std::mutex> g(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  const size_t n = code->spec.n;
  const uint64_t chunk = std::min<uint64_t>(std::max<uint64_t>(frames, 1), uint64_t(1) << 22);
  const float sigma = static_cast<float>(ccgpu_sigma(code->spec.rate, ebno_db));
  return with_counters(ctx, out, [&](unsigned long long *counters) -> int {
    uint8_t *d_words, *d_out, *d_ne, *d_fail;
    int rc = cut_stage(ctx, [&](Arena &a) {
      d_words = a.take<uint8_t>(chunk * n);
      d_out = a.take<uint8_t>(chunk * n);
      d_ne = a.take<uint8_t>(chunk);
      d_fail = a.take<uint8_t>(chunk);
    });
    if (rc) return rc;
    for (uint64_t f0 = 0; f0 < frames; f0 += chunk) {
      const uint64_t nf = std::min(chunk, frames - f0);
      awgn_hard_kernel<<<grid_for(ctx, nf * ((n + 3) / 4), kAwgnThreads), kAwgnThreads, 0, ctx->stream>>>(
          d_words, static_cast<uint32_t>(n), sigma, seed, point, frame0 + f0, nf);
      CU(cudaGetLastError());
      rc = gf_rc(ctx, gf_launch(code->gf, d_words, nf, nullptr, nullptr, 0, d_out, d_ne, d_fail, ctx->sm_count, ctx->stream));
      if (rc) return rc;
      count_words_kernel<<<grid_for(ctx, nf, 8, 8), 256, 0, ctx->stream>>>(d_out, d_fail, static_cast<uint32_t>(n), nf,
                                                                           counters);
      CU(cudaGetLastError());
      ctx->launches += 2;
    }
    return CCGPU_OK;
  });
}

// ---- Chase-II (extension): K5 in chase.cu
static int check_chase(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t p) {
  if (int rc = check_code(ctx, code)) return rc;
  if (p > kChaseMaxP) return fail(ctx, CCGPU_ERR_INVALID, "Chase-II takes 0 <= p <= 8 test positions");
  if (code->spec.family != 0) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "Chase-II decoding needs a binary BCH code");
  if (p > code->spec.n) return fail(ctx, CCGPU_ERR_INVALID, "p > n");
  return CCGPU_OK;
}
static int chase_rc(ccgpu_ctx *ctx, int rc) {
  if (rc == -3) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "code not supported by the Chase kernel (t <= 31)");
  if (rc != 0) return cuda_fail(ctx, cudaGetLastError(), "chase_launch");
  ctx->launches++;
  return CCGPU_OK;
}

int ccgpu_decode_llr_chase(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t p, const float *y, uint64_t frames,
                           uint8_t *bits, uint8_t *failed, uint8_t *chosen) {
  if (!ctx || !code || !y || !bits || !failed) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  int rc = check_chase(ctx, code, p);
  if (rc) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (frames == 0) return CCGPU_OK;
  CU(cudaSetDevice(ctx->device));
  const size_t n = code->spec.n;
  const bool dev = is_device_ptr(y);
  if (!same_residency(dev, {bits, failed, chosen}))
    return fail(ctx, CCGPU_ERR_INVALID, "y and the outputs must all be device pointers or all host pointers");
  if (dev) return chase_rc(ctx, chase_launch(code->gf, p, y, frames, bits, failed, chosen, ctx->sm_count, ctx->stream));
  const HostField fields[] = { { n * sizeof(float), y, false }, { n, bits, true }, { 1, failed, true }, { 1, chosen, true } };
  return host_pipeline(ctx, frames, fields, [&](void *const *d, uint64_t nf, cudaStream_t st, int) {
    return chase_rc(ctx, chase_launch(code->gf, p, static_cast<const float *>(d[0]), nf, static_cast<uint8_t *>(d[1]),
                                      static_cast<uint8_t *>(d[2]), static_cast<uint8_t *>(d[3]), ctx->sm_count, st));
  });
}

int ccgpu_awgn_point_chase(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t p, double ebno_db, uint64_t seed,
                           uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!ctx || !code || !out) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  int rc = check_chase(ctx, code, p);
  if (rc) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  const float sigma = static_cast<float>(ccgpu_sigma(code->spec.rate, ebno_db));
  return with_counters(ctx, out, [&](unsigned long long *counters) {
    return chase_rc(ctx, chase_awgn_launch(code->gf, p, sigma, seed, point, frame0, frames, counters, ctx->sm_count, ctx->stream));
  });
}

// ---- ordered-statistics decoding (extension): K6 in osd.cu
static int check_osd(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t order) {
  if (int rc = check_code(ctx, code)) return rc;
  if (order > kOsdMaxOrder) return fail(ctx, CCGPU_ERR_INVALID, "OSD takes 0 <= order <= 3");
  if (code->spec.family != 0) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "OSD decoding needs a binary BCH code");
  if (!code->osd.rows) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "code not supported by the OSD kernel (n <= 127, n - l <= 64)");
  return CCGPU_OK;
}
static int osd_rc(ccgpu_ctx *ctx, int rc) {
  if (rc == -3) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "code not supported by the OSD kernel (n <= 127, n - l <= 64)");
  if (rc != 0) return cuda_fail(ctx, cudaGetLastError(), "osd_launch");
  ctx->launches++;
  return CCGPU_OK;
}

int ccgpu_decode_llr_osd(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t order, const float *y, uint64_t frames,
                         uint8_t *bits, uint8_t *weight) {
  if (!ctx || !code || !y || !bits) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  int rc = check_osd(ctx, code, order);
  if (rc) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (frames == 0) return CCGPU_OK;
  CU(cudaSetDevice(ctx->device));
  const size_t n = code->spec.n;
  const bool dev = is_device_ptr(y);
  if (!same_residency(dev, {bits, weight}))
    return fail(ctx, CCGPU_ERR_INVALID, "y and the outputs must all be device pointers or all host pointers");
  if (dev) return osd_rc(ctx, osd_launch(code->osd, order, y, frames, bits, weight, ctx->sm_count, ctx->stream));
  const HostField fields[] = { { n * sizeof(float), y, false }, { n, bits, true }, { 1, weight, true } };
  return host_pipeline(ctx, frames, fields, [&](void *const *d, uint64_t nf, cudaStream_t st, int) {
    return osd_rc(ctx, osd_launch(code->osd, order, static_cast<const float *>(d[0]), nf, static_cast<uint8_t *>(d[1]),
                                  static_cast<uint8_t *>(d[2]), ctx->sm_count, st));
  });
}

int ccgpu_awgn_point_osd(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t order, double ebno_db, uint64_t seed,
                         uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!ctx || !code || !out) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  int rc = check_osd(ctx, code, order);
  if (rc) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  const float sigma = static_cast<float>(ccgpu_sigma(code->spec.rate, ebno_db));
  return with_counters(ctx, out, [&](unsigned long long *counters) {
    return osd_rc(ctx, osd_awgn_launch(code->osd, order, sigma, seed, point, frame0, frames, counters, ctx->sm_count, ctx->stream));
  });
}

// ---- GMD decoding of Reed-Solomon codes (extension): K7 in gmd.cu
static int check_gmd(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t max_erasures) {
  if (int rc = check_code(ctx, code)) return rc;
  if (code->spec.family != 1)
    return fail(ctx, CCGPU_ERR_UNSUPPORTED, "GMD decoding needs a Reed-Solomon code (binary BCH codes have Chase-II)");
  if (code->spec.roots.size() > kGmdMaxRoots || code->spec.step != 1)
    return fail(ctx, CCGPU_ERR_UNSUPPORTED, "code not supported by the GMD kernel (2t <= 32, step = 1)");
  if ((max_erasures & 1u) || max_erasures > 2 * code->spec.t)
    return fail(ctx, CCGPU_ERR_INVALID, "GMD takes an even max_erasures <= 2t");
  return CCGPU_OK;
}
static int gmd_rc(ccgpu_ctx *ctx, int rc) {
  if (rc == -3) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "code not supported by the GMD kernel (2t <= 32, step = 1)");
  if (rc != 0) return cuda_fail(ctx, cudaGetLastError(), "gmd_launch");
  ctx->launches++;
  return CCGPU_OK;
}

int ccgpu_decode_llr_gmd(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t max_erasures, const float *y, uint64_t frames,
                         uint8_t *words, uint8_t *failed, uint8_t *chosen) {
  if (!ctx || !code || !y || !words || !failed) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  int rc = check_gmd(ctx, code, max_erasures);
  if (rc) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (frames == 0) return CCGPU_OK;
  CU(cudaSetDevice(ctx->device));
  const size_t n = code->spec.n, nq = n * code->spec.q;
  const bool dev = is_device_ptr(y);
  if (!same_residency(dev, {words, failed, chosen}))
    return fail(ctx, CCGPU_ERR_INVALID, "y and the outputs must all be device pointers or all host pointers");
  if (dev) return gmd_rc(ctx, gmd_launch(code->gf, max_erasures, y, frames, words, failed, chosen, ctx->sm_count, ctx->stream));
  const HostField fields[] = { { nq * sizeof(float), y, false }, { n, words, true }, { 1, failed, true }, { 1, chosen, true } };
  return host_pipeline(ctx, frames, fields, [&](void *const *d, uint64_t nf, cudaStream_t st, int) {
    return gmd_rc(ctx, gmd_launch(code->gf, max_erasures, static_cast<const float *>(d[0]), nf, static_cast<uint8_t *>(d[1]),
                                  static_cast<uint8_t *>(d[2]), static_cast<uint8_t *>(d[3]), ctx->sm_count, st));
  });
}

int ccgpu_awgn_point_gmd(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t max_erasures, double ebno_db, uint64_t seed,
                         uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!ctx || !code || !out) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  int rc = check_gmd(ctx, code, max_erasures);
  if (rc) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  const float sigma = static_cast<float>(ccgpu_sigma(code->spec.rate, ebno_db));
  return with_counters(ctx, out, [&](unsigned long long *counters) {
    return gmd_rc(ctx, gmd_awgn_launch(code->gf, max_erasures, sigma, seed, point, frame0, frames, counters, ctx->sm_count,
                                       ctx->stream));
  });
}

// ---- adaptive belief propagation (extension): K8 in abp.cu, on the OSD kernel's packed k-row H
static int check_abp(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t max_iter, double gamma) {
  if (int rc = check_code(ctx, code)) return rc;
  if (max_iter > kAbpMaxIter) return fail(ctx, CCGPU_ERR_INVALID, "ABP takes 0 <= max_iter <= 255");
  if (!(gamma > 0.0 && gamma <= 1.0)) return fail(ctx, CCGPU_ERR_INVALID, "ABP takes a finite gamma with 0 < gamma <= 1");
  if (code->spec.family != 0) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "ABP decoding needs a binary BCH code");
  if (!code->osd.rows) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "code not supported by the ABP kernel (n <= 127, n - l <= 64)");
  return CCGPU_OK;
}
static int abp_rc(ccgpu_ctx *ctx, int rc) {
  if (rc == -3) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "code not supported by the ABP kernel (n <= 127, n - l <= 64)");
  if (rc != 0) return cuda_fail(ctx, cudaGetLastError(), "abp_launch");
  ctx->launches++;
  return CCGPU_OK;
}

int ccgpu_decode_llr_abp(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t max_iter, double gamma, const float *y,
                         uint64_t frames, uint8_t *bits, float *L, uint8_t *iter, uint8_t *failed) {
  if (!ctx || !code || !y || !bits || !iter || !failed) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  int rc = check_abp(ctx, code, max_iter, gamma);
  if (rc) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (frames == 0) return CCGPU_OK;
  CU(cudaSetDevice(ctx->device));
  const size_t n = code->spec.n;
  const float gf = static_cast<float>(gamma);
  const bool dev = is_device_ptr(y);
  if (!same_residency(dev, {bits, L, iter, failed}))
    return fail(ctx, CCGPU_ERR_INVALID, "y and the outputs must all be device pointers or all host pointers");
  if (dev) return abp_rc(ctx, abp_launch(code->osd, max_iter, gf, y, frames, bits, L, iter, failed, ctx->sm_count, ctx->stream));
  const HostField fields[] = { { n * sizeof(float), y, false }, { n, bits, true }, { n * sizeof(float), L, true },
                               { 1, iter, true }, { 1, failed, true } };
  return host_pipeline(ctx, frames, fields, [&](void *const *d, uint64_t nf, cudaStream_t st, int) {
    return abp_rc(ctx, abp_launch(code->osd, max_iter, gf, static_cast<const float *>(d[0]), nf, static_cast<uint8_t *>(d[1]),
                                  static_cast<float *>(d[2]), static_cast<uint8_t *>(d[3]), static_cast<uint8_t *>(d[4]),
                                  ctx->sm_count, st));
  });
}

int ccgpu_awgn_point_abp(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t max_iter, double gamma, double ebno_db,
                         uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!ctx || !code || !out) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  int rc = check_abp(ctx, code, max_iter, gamma);
  if (rc) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  const float sigma = static_cast<float>(ccgpu_sigma(code->spec.rate, ebno_db));
  return with_counters(ctx, out, [&](unsigned long long *counters) {
    return abp_rc(ctx, abp_awgn_launch(code->osd, max_iter, static_cast<float>(gamma), sigma, seed, point, frame0, frames,
                                       counters, ctx->sm_count, ctx->stream));
  });
}

// ---- maximum-likelihood decoding (extension): K9 in ml.cu, on the column syndromes of the k-row H
static int check_ml(ccgpu_ctx *ctx, const ccgpu_code *code) {
  if (int rc = check_code(ctx, code)) return rc;
  if (code->spec.family != 0) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "ML decoding needs a binary BCH code");
  if (!code->ml.k) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "code not supported by the ML kernel (n <= 127, n - l <= 12)");
  return CCGPU_OK;
}
static int ml_rc(ccgpu_ctx *ctx, int rc) {
  if (rc == -3) return fail(ctx, CCGPU_ERR_UNSUPPORTED, "code not supported by the ML kernel (n <= 127, n - l <= 12)");
  if (rc != 0) return cuda_fail(ctx, cudaGetLastError(), "ml_launch");
  ctx->launches++;
  return CCGPU_OK;
}

int ccgpu_decode_llr_ml(ccgpu_ctx *ctx, const ccgpu_code *code, const float *y, uint64_t frames, uint8_t *bits) {
  if (!ctx || !code || !y || !bits) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  int rc = check_ml(ctx, code);
  if (rc) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  if (frames == 0) return CCGPU_OK;
  CU(cudaSetDevice(ctx->device));
  const size_t n = code->spec.n;
  const bool dev = is_device_ptr(y);
  if (!same_residency(dev, {bits}))
    return fail(ctx, CCGPU_ERR_INVALID, "y and the outputs must all be device pointers or all host pointers");
  if (dev) return ml_rc(ctx, ml_launch(code->ml, y, frames, bits, ctx->sm_count, ctx->stream));
  const HostField fields[] = { { n * sizeof(float), y, false }, { n, bits, true } };
  return host_pipeline(ctx, frames, fields, [&](void *const *d, uint64_t nf, cudaStream_t st, int) {
    return ml_rc(ctx, ml_launch(code->ml, static_cast<const float *>(d[0]), nf, static_cast<uint8_t *>(d[1]),
                                ctx->sm_count, st));
  });
}

int ccgpu_awgn_point_ml(ccgpu_ctx *ctx, const ccgpu_code *code, double ebno_db, uint64_t seed, uint32_t point,
                        uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!ctx || !code || !out) return fail(ctx, CCGPU_ERR_INVALID, "null argument");
  int rc = check_ml(ctx, code);
  if (rc) return rc;
  std::lock_guard<std::mutex> g(ctx->mu);
  CU(cudaSetDevice(ctx->device));
  const float sigma = static_cast<float>(ccgpu_sigma(code->spec.rate, ebno_db));
  return with_counters(ctx, out, [&](unsigned long long *counters) {
    return ml_rc(ctx, ml_awgn_launch(code->ml, sigma, seed, point, frame0, frames, counters, ctx->sm_count, ctx->stream));
  });
}

int ccgpu_code_set_recheck(ccgpu_code *code, int enable) {
  if (!code) return CCGPU_ERR_INVALID;
  code->gf.recheck = enable ? 1 : 0;
  return CCGPU_OK;
}

}  // extern "C"
