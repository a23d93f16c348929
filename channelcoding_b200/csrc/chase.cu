// chase.cu -- K5: Chase-II soft-decision decoding of binary primitive BCH codes, one warp per frame.
//
// Per frame (include/ccgpu.h, ccgpu_decode_llr_chase, states the contract):
//   h_c = (y_c < 0); the p least reliable columns u_0 .. u_{p-1} are the p smallest (bits(|y_c|), c);
//   test word m = h with u_j flipped for every set bit j of m, m = 0 .. 2^p - 1;
//   every test word is decoded errors-only exactly as K4 (gf_decode.cu) decodes it, a success x_m is a candidate
//   with metric D_m = sum over the columns where x_m != h of |y_c| (float32, c ascending, from +0.0);
//   the candidate with the smallest (bits(D_m), m) wins; without a candidate the frame fails and h is returned.
//
// Work split inside the warp
//   channel     lane <-> column (HBM) or Philox block (fused path, awgn_block of channel.cuh); the values stay in
//               shared memory for the reliability order and the metric.
//   screening   a frame without a negative value has h = 0, a codeword: pattern 0 wins with D = +0.0.
//   syndromes   of h once, with K4's Horner routine (gf_device.cuh); zero syndromes end the frame the same way.
//   order       p rounds of two REDUX.MIN: the smallest key, then the lowest column holding it.
//   patterns    Gray-code order: each step flips one position u_j, so the syndromes of the test word change by
//               alpha^(root_i * u_j), a per-lane column computed once per frame (one XOR per lane and step).
//   BM          lane <-> locator coefficient as in K4; the discrepancy of every second step is zero for binary
//               words (S_2i = S_i^2), so those steps only shift B -- the locator is the same.
//   roots       lane <-> column; the ballots of the root search are the error columns.
//   metric      lane bit ch of (flips ^ errors) marks column 32 ch + lane; lane 0 sums |y| over the set bits in
//               ascending column order, the warp keeps the running minimum of (bits(D), m).
#include <algorithm>

#include "channel.cuh"
#include "chase.h"
#include "gf_device.cuh"
#include "ms_params.h"

namespace ccgpu {

namespace {

constexpr int kChaseThreads = 256;
constexpr int kChaseWarps = kChaseThreads / 32;
// per warp: y[256] floats, h[256], syndromes[64], locator logs[32], positions[16], syndrome columns[8][64]
constexpr int kChaseWarpBytes = 1024 + 256 + 64 + 32 + 16 + 8 * 64;

struct ChaseParams {
  int q, n, t, nroots, p;
  const uint8_t *tables;
  const float *y;  // HBM source
  unsigned long long frames;
  uint8_t *bits, *failed, *chosen;
  // fused source: frame f is frame frame0 + f of the stream (keys, point)
  float sigma;
  uint32_t point;
  unsigned long long frame0;
  unsigned long long *counters;
  PhiloxKeys keys;
};

template <bool kFused>
__global__ void __launch_bounds__(kChaseThreads) chase_kernel(const __grid_constant__ ChaseParams p) {
  extern __shared__ __align__(16) uint8_t sm[];
  const GfShared tabs = gf_table_layout(sm, p.q, p.nroots);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t *base = tabs.rest + warp * kChaseWarpBytes;
  float *sy = reinterpret_cast<float *>(base);  // [256] channel values
  uint8_t *word = base + 1024;                  // [256] hard decision h, zero padded for the Horner segments
  uint8_t *synd = word + 256;                   // [64]
  uint8_t *llog = synd + 64;                    // [32] logarithms of the locator coefficients (0xff: zero)
  uint8_t *upos = llog + 32;                    // [16] u_0 .. u_{p-1}
  uint8_t *col = upos + 16;                     // [8][64] alpha^(root_i * u_j), row j
  gf_fill_tables(tabs, p.tables, p.q, p.n, p.nroots, 1);
  const Gf F{ tabs.exp, tabs.log };
  const int n = p.n, nroots = p.nroots;
  const int nch = (n + 31) / 32;           // column chunks: lane bit ch <-> column 32 ch + lane
  const int seg4 = ((n + 15) / 16) * 16;   // <= 32 nch
  unsigned long long c_frames = 0, c_ferr = 0, c_berr = 0, c_fail = 0, c_und = 0;

  const unsigned long long nwarps = static_cast<unsigned long long>(gridDim.x) * kChaseWarps;
  for (unsigned long long w = static_cast<unsigned long long>(blockIdx.x) * kChaseWarps + warp; w < p.frames; w += nwarps) {
    if (kFused) {
      for (int blk = lane; blk < (n + 3) / 4; blk += 32) {
        const float4 v = awgn_block(p.keys, p.point, p.frame0 + w, blk, p.sigma);
        const float vv[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (4 * blk + e < n) sy[4 * blk + e] = vv[e];
      }
    } else {
      for (int i = lane; i < n; i += 32) sy[i] = p.y[w * n + i];
    }
    __syncwarp();
    unsigned h = 0;  // lane bit ch: h of column 32 ch + lane (codes.h:43-52: y < 0; 0 for -0.0 and NaN)
    for (int ch = 0; ch < nch; ++ch) {
      const int c = 32 * ch + lane;
      const bool one = c < n && sy[c] < 0.0f;
      h |= static_cast<unsigned>(one) << ch;
      if (c < seg4) word[c] = one ? 1 : 0;
    }
    bool failed = false;
    unsigned chosen = 0, best_diff = 0;  // best_diff: lane bit ch <-> column 32 ch + lane differs from h
    if (__any_sync(kGfAll, h != 0)) {
      __syncwarp();
      if (syndromes(p, F, word, tabs.mtab, tabs.rexp, synd, lane)) {
        // ---------------- the p least reliable columns and their syndrome columns
        unsigned taken = 0;
        for (int j = 0; j < p.p; ++j) {
          unsigned bk = 0xffffffffu, bc = 0xffffffffu;
          for (int ch = 0; ch < nch; ++ch) {
            const int c = 32 * ch + lane;
            if (c < n && !((taken >> ch) & 1u)) {
              const unsigned key = __float_as_uint(sy[c]) & 0x7fffffffu;  // bits of fabsf(y): NaN above +inf
              if (key < bk) bk = key, bc = static_cast<unsigned>(c);   // ascending c: ties keep the lower column
            }
          }
          const unsigned kmin = __reduce_min_sync(kGfAll, bk);
          const unsigned u = __reduce_min_sync(kGfAll, bk == kmin ? bc : 0xffffffffu);
          if ((u & 31u) == static_cast<unsigned>(lane)) taken |= 1u << (u >> 5);
          if (lane == 0) upos[j] = static_cast<uint8_t>(u);
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int r = lane + 32 * half;
            col[j * 64 + r] = static_cast<uint8_t>(r < nroots ? F.exp[(tabs.rexp[r] * u) % n] : 0u);
          }
        }
        __syncwarp();
        // ---------------- 2^p test patterns in Gray-code order
        unsigned s0 = lane < nroots ? synd[lane] : 0u, s1 = lane + 32 < nroots ? synd[lane + 32] : 0u;
        unsigned flips = 0, m = 0;
        unsigned long long best = ~0ull;
        for (int k = 0; k < (1 << p.p); ++k) {
          if (k) {
            const int j = __ffs(k) - 1;
            m ^= 1u << j;
            const unsigned u = upos[j];
            if ((u & 31u) == static_cast<unsigned>(lane)) flips ^= 1u << (u >> 5);
            s0 ^= col[j * 64 + lane];
            s1 ^= col[j * 64 + 32 + lane];
          }
          // errors-only bounded-distance decode of the test word, K4's rules
          unsigned err = 0;
          bool ok = true;
          if (__any_sync(kGfAll, (s0 | s1) != 0)) {
            synd[lane] = static_cast<uint8_t>(s0);
            synd[lane + 32] = static_cast<uint8_t>(s1);
            __syncwarp();
            unsigned lam = lane == 0, B = lam;
            int L = 0;
            for (int r = 0; r < nroots; ++r) {
              const unsigned bs = __shfl_up_sync(kGfAll, B, 1);
              B = lane ? bs : 0u;  // B <- x B
              if (r & 1) continue;
              const unsigned term = (lane <= L && lane <= r) ? F.mul(lam, synd[r - lane]) : 0u;
              const unsigned delta = xor_reduce(term);
              if (delta) {
                const unsigned nl = lam ^ F.mul(delta, B);
                if (2 * L <= r) {
                  B = F.mul(lam, F.exp[n - F.log[delta]]);  // Lambda / delta
                  L = r - L + 1;
                }
                lam = nl;
              }
              if (L > 31) break;
            }
            ok = !(2 * L > nroots || L > 31 || L == 0);
            if (ok) {
              llog[lane] = static_cast<uint8_t>((lane <= L && lam) ? F.log[lam] : 0xff);
              __syncwarp();
              int found = 0;
              for (int ch = 0; ch < nch; ++ch) {
                const int i = 32 * ch + lane;
                unsigned v = 1;  // Lambda(alpha^-i), Lambda_0 = 1
                if (i < n) {
                  const unsigned e = i ? n - i : 0;
                  unsigned acc = 0;
                  for (int kk = 1; kk <= L; ++kk) {
                    acc += e;
                    if (acc >= static_cast<unsigned>(n)) acc -= n;
                    const unsigned lg = llog[kk];
                    if (lg != 0xff) v ^= F.exp[lg + acc];
                  }
                }
                const bool root = i < n && v == 0;
                found += __popc(__ballot_sync(kGfAll, root));
                err |= static_cast<unsigned>(root) << ch;
              }
              ok = found == L;
            }
            __syncwarp();
          }
          if (ok) {
            const unsigned diff = flips ^ err;
            float D = 0.0f;
            for (int ch = 0; ch < nch; ++ch) {
              unsigned mask = __ballot_sync(kGfAll, (diff >> ch) & 1u);
              if (lane == 0) {
                while (mask) {
                  const int b = __ffs(mask) - 1;
                  mask &= mask - 1;
                  D = __fadd_rn(D, fabsf(sy[32 * ch + b]));
                }
              }
            }
            D = __shfl_sync(kGfAll, D, 0);
            const unsigned long long key = (static_cast<unsigned long long>(__float_as_uint(D)) << 32) | m;
            if (key < best) {
              best = key;
              best_diff = diff;
            }
          }
        }
        failed = best == ~0ull;
        chosen = failed ? 0u : static_cast<unsigned>(best & 0xffu);
        if (failed) best_diff = 0;
      }
    }
    const unsigned out = h ^ best_diff;
    if (kFused) {
      const unsigned nz = __reduce_add_sync(kGfAll, __popc(out));
      c_frames += 1;
      c_fail += failed;
      c_berr += nz;
      c_ferr += (failed || nz) ? 1 : 0;
      c_und += (!failed && nz) ? 1 : 0;
    } else {
      for (int ch = 0; ch < nch; ++ch) {
        const int c = 32 * ch + lane;
        if (c < n) p.bits[w * n + c] = static_cast<uint8_t>((out >> ch) & 1u);
      }
      if (lane == 0) {
        if (p.failed) p.failed[w] = failed ? 1 : 0;
        if (p.chosen) p.chosen[w] = static_cast<uint8_t>(chosen);
      }
    }
    __syncwarp();
  }
  if (kFused && lane == 0) {
    if (c_frames) atomicAdd(p.counters + C_FRAMES, c_frames);
    if (c_ferr) atomicAdd(p.counters + C_FRAME_ERR, c_ferr);
    if (c_berr) atomicAdd(p.counters + C_BIT_ERR, c_berr);
    if (c_fail) atomicAdd(p.counters + C_FAIL, c_fail);
    if (c_und) atomicAdd(p.counters + C_UNDETECTED, c_und);
  }
}

template <bool kFused> int launch(const GfDevice &d, const ChaseParams &cp, int sm_count, cudaStream_t stream) {
  if (cp.frames == 0) return 0;
  const size_t smem = gf_table_bytes(d.q, d.nroots) + size_t(kChaseWarps) * kChaseWarpBytes;
  if (cudaFuncSetAttribute(chase_kernel<kFused>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) !=
      cudaSuccess)
    return -1;
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, chase_kernel<kFused>, kChaseThreads, smem);
  const uint64_t want = (cp.frames + kChaseWarps - 1) / kChaseWarps;
  const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(want, uint64_t(std::max(1, occ)) * sm_count));
  chase_kernel<kFused><<<grid, kChaseThreads, smem, stream>>>(cp);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

bool supported(const GfDevice &d, uint32_t p) {
  return d.tables && d.binary && d.t <= 31 && d.nroots <= 64 && d.step == 1 && d.mu == 1 && p <= kChaseMaxP &&
         p <= static_cast<uint32_t>(d.n);
}

ChaseParams params_of(const GfDevice &d, uint32_t p) {
  ChaseParams cp{};
  cp.q = d.q;
  cp.n = d.n;
  cp.t = d.t;
  cp.nroots = d.nroots;
  cp.p = static_cast<int>(p);
  cp.tables = d.tables;
  return cp;
}

}  // namespace

int chase_launch(const GfDevice &d, uint32_t p, const float *y, uint64_t frames, uint8_t *bits, uint8_t *failed,
                 uint8_t *chosen, int sm_count, cudaStream_t stream) {
  if (!supported(d, p)) return -3;
  ChaseParams cp = params_of(d, p);
  cp.y = y;
  cp.frames = frames;
  cp.bits = bits;
  cp.failed = failed;
  cp.chosen = chosen;
  return launch<false>(d, cp, sm_count, stream);
}

int chase_awgn_launch(const GfDevice &d, uint32_t p, float sigma, uint64_t seed, uint32_t point, uint64_t frame0,
                      uint64_t frames, unsigned long long *counters, int sm_count, cudaStream_t stream) {
  if (!supported(d, p)) return -3;
  ChaseParams cp = params_of(d, p);
  cp.frames = frames;
  cp.sigma = sigma;
  cp.point = point;
  cp.frame0 = frame0;
  cp.counters = counters;
  cp.keys = philox_round_keys(seed);
  return launch<true>(d, cp, sm_count, stream);
}

}  // namespace ccgpu
