// gmd.cu -- K7: generalized minimum distance (GMD) decoding of Reed-Solomon codes over GF(2^q) from the channel values
// of their binary image, one warp per frame.
//
// Per frame (include/ccgpu.h, ccgpu_decode_llr_gmd, states the contract):
//   bit j of symbol c is image position c q + j; r_c = sum_j (y_{cq+j} < 0) << j; kappa_c = min_j K(|y_{cq+j}|);
//   the symbols are ranked in ascending (kappa_c, c); trial i = 0 .. F/2 erases the first 2i of them and decodes r
//   with errors and erasures exactly as K4 (gf_decode.cu) does; a success x_i is a candidate with metric D_i = sum of
//   |y_b| over the image bits where x_i differs from r (float32, b ascending, from +0.0); the smallest (K(D_i), i)
//   wins; without a candidate the frame fails and r is returned.
//
// Work split inside the warp
//   channel     lane <-> value (HBM) or Philox block (fused path, awgn_block of channel.cuh); the n q values stay in
//               shared memory for the symbol keys and the metric.
//   symbols     lane <-> symbol (lane slot ch <-> symbol 32 ch + lane): r_c into the Horner buffer, kappa_c in a
//               register.  A frame with r = 0 is a codeword: trial 0 wins with D = +0.0.
//   syndromes   of r once, with K4's Horner routine (gf_device.cuh); zero syndromes end the frame the same way.
//               The erasure sets only grow, r never changes: every trial reuses them.
//   order       F rounds of two REDUX.MIN: the smallest key, then the lowest symbol holding it.
//   trials      lane <-> locator coefficient: the erasure locator Gamma gains the factors (1 + X x) of the two new
//               erasures (one shuffle per factor), Berlekamp-Massey runs from it as in K4 (from r = rho, length rho).
//   roots       lane <-> symbol, ballots give the errata positions in ascending order.  The trial with 2i = 2t has
//               no BM step left: its locator IS Gamma, whose roots are the erasures by construction, so the search
//               is skipped.  That is also the only trial whose locator can have degree 32, i.e. 33 coefficients: the
//               lanes hold coefficients 0 .. 31 and Gamma_32 is never needed (Forney reads Omega_0..31, which has
//               degree < 32, and the odd coefficients of Lambda only).
//   Forney      lane <-> errata index, K4's formula and failure rules; the values go to a per-warp array indexed by
//               position, so the metric walks them in ascending position with one ballot per 32 symbols and lane 0
//               adds |y| over the set bits of each value serially (the contract's summation order).
#include <algorithm>

#include "channel.cuh"
#include "gf_device.cuh"
#include "gmd.h"
#include "ms_params.h"

namespace ccgpu {

namespace {

constexpr int kGmdThreads = 256;
constexpr int kGmdWarps = kGmdThreads / 32;
constexpr int kGmdMaxChunks = 8;  // n <= 255 symbols
// per warp after the channel values: r[256] (zero padded for the Horner segments), errata values by position[256],
// syndromes[64], locator coefficients[32] and their logs[32], evaluator[32], errata positions[32], ranking[32]
constexpr int kGmdFixedBytes = 256 + 256 + 64 + 5 * 32;

struct GmdParams {
  int q, n, nroots, mu, F;
  int y_bytes, warp_bytes;  // per-warp channel buffer (16-byte multiple) and the whole per-warp block
  const uint8_t *tables;
  const float *y;  // HBM source
  unsigned long long frames;
  uint8_t *words, *failed, *chosen;
  // fused source: frame f is frame frame0 + f of the stream (keys, point)
  float sigma;
  uint32_t point;
  unsigned long long frame0;
  unsigned long long *counters;
  PhiloxKeys keys;
};

__device__ __forceinline__ unsigned nan_key(float v) {  // K: bits of v >= 0, every NaN counted as 0x7fc00000
  return isnan(v) ? 0x7fc00000u : __float_as_uint(v);
}

template <bool kFused>
__global__ void __launch_bounds__(kGmdThreads) gmd_kernel(const __grid_constant__ GmdParams p) {
  extern __shared__ __align__(16) uint8_t sm[];
  const GfShared tabs = gf_table_layout(sm, p.q, p.nroots);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t *base = tabs.rest + warp * p.warp_bytes;
  float *sy = reinterpret_cast<float *>(base);  // [n q] channel values
  uint8_t *word = base + p.y_bytes;             // [256] r
  uint8_t *ev = word + 256;                     // [256] errata values of the current trial by position, else 0
  uint8_t *synd = ev + 256;                     // [64]
  uint8_t *lamv = synd + 64;                    // [32] locator coefficients 0 .. 31
  uint8_t *llog = lamv + 32;                    // [32] their logarithms (0xff: zero coefficient)
  uint8_t *omega = llog + 32;                   // [32]
  uint8_t *pos = omega + 32;                    // [32] errata positions, ascending
  uint8_t *upos = pos + 32;                     // [32] the F least reliable symbols, in ranking order
  for (int i = lane; i < 256; i += 32) ev[i] = 0;
  gf_fill_tables(tabs, p.tables, p.q, p.n, p.nroots, p.mu);
  const Gf F{ tabs.exp, tabs.log };
  const int n = p.n, q = p.q, nq = n * q, nroots = p.nroots;
  const int nch = (n + 31) / 32;          // symbol chunks: lane slot ch <-> symbol 32 ch + lane
  const int seg4 = ((n + 15) / 16) * 16;  // <= 32 nch
  const unsigned mu_exp = static_cast<unsigned>(((1 - p.mu) % n + n) % n);
  unsigned long long c_frames = 0, c_ferr = 0, c_berr = 0, c_fail = 0, c_und = 0;

  const unsigned long long nwarps = static_cast<unsigned long long>(gridDim.x) * kGmdWarps;
  for (unsigned long long w = static_cast<unsigned long long>(blockIdx.x) * kGmdWarps + warp; w < p.frames; w += nwarps) {
    if (kFused) {
      for (int blk = lane; blk < (nq + 3) / 4; blk += 32) {
        const float4 v = awgn_block(p.keys, p.point, p.frame0 + w, blk, p.sigma);
        const float vv[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (4 * blk + e < nq) sy[4 * blk + e] = vv[e];
      }
    } else {
      for (int i = lane; i < nq; i += 32) sy[i] = p.y[w * nq + i];
    }
    __syncwarp();
    // ---------------- hard symbols r_c and symbol keys kappa_c
    unsigned kap[kGmdMaxChunks];
    bool nonzero = false;
#pragma unroll
    for (int ch = 0; ch < kGmdMaxChunks; ++ch) {
      const int c = 32 * ch + lane;
      unsigned r = 0, k = 0xffffffffu;  // symbols c >= n keep the key above every real one
      if (ch < nch && c < n) {
        k = 0x7fc00000u;
        for (int j = 0; j < q; ++j) {
          const float v = sy[c * q + j];
          r |= static_cast<unsigned>(v < 0.0f) << j;  // codes.h:43-52: 0 for -0.0 and NaN
          k = min(k, nan_key(fabsf(v)));
        }
      }
      kap[ch] = k;
      nonzero |= r != 0;
      if (ch < nch && c < seg4) word[c] = static_cast<uint8_t>(r);
    }
    bool failed = false;
    unsigned chosen = 0;
    if (__any_sync(kGfAll, nonzero)) {
      __syncwarp();
      if (syndromes(p, F, word, tabs.mtab, tabs.rexp, synd, lane)) {
        // ---------------- the F least reliable symbols
        unsigned taken = 0;
        for (int j = 0; j < p.F; ++j) {
          unsigned bk = 0xffffffffu, bc = 0xffffffffu;
#pragma unroll
          for (int ch = 0; ch < kGmdMaxChunks; ++ch)
            if (ch < nch && !((taken >> ch) & 1u) && kap[ch] < bk) bk = kap[ch], bc = 32 * ch + lane;  // ties: lower c
          const unsigned kmin = __reduce_min_sync(kGfAll, bk);
          const unsigned u = __reduce_min_sync(kGfAll, bk == kmin ? bc : 0xffffffffu);
          if ((u & 31u) == static_cast<unsigned>(lane)) taken |= 1u << (u >> 5);
          if (lane == 0) upos[j] = static_cast<uint8_t>(u);
        }
        __syncwarp();
        // ---------------- trials i = 0 .. F/2
        unsigned gam = lane == 0;  // erasure locator Gamma, coefficient `lane`
        unsigned long long best = ~0ull;
        unsigned bpos = 0, bval = 0;  // lane k of the best trial: its k-th errata position and value (0: none)
        for (int tr = 0; 2 * tr <= p.F; ++tr) {
          const int rho = 2 * tr;
          if (tr) {
            for (int e = rho - 2; e < rho; ++e) {  // Gamma <- Gamma (1 + X_e x), X_e = alpha^position
              const unsigned up = __shfl_up_sync(kGfAll, gam, 1);
              gam ^= F.mul_alpha(lane ? up : 0u, upos[e]);
            }
          }
          // ---------------- Berlekamp-Massey from r = rho (K4)
          unsigned lam = gam, B = gam;
          int L = rho;
          for (int r = rho; r < nroots; ++r) {
            const unsigned bs = __shfl_up_sync(kGfAll, B, 1);
            B = lane ? bs : 0u;  // B <- x B
            const unsigned term = (lane <= L && lane <= r) ? F.mul(lam, synd[r - lane]) : 0u;
            const unsigned delta = xor_reduce(term);
            if (delta) {
              const unsigned nl = lam ^ F.mul(delta, B);
              if (2 * L <= r + rho) {
                B = F.mul(lam, F.exp[n - F.log[delta]]);  // Lambda / delta
                L = r + rho - L + 1;
              }
              lam = nl;
            }
            if (L > 31) break;  // then 2L > 2t + rho: the trial fails below
          }
          bool ok = 2 * L <= nroots + rho && L != 0;
          unsigned pk = 0, val = 0;
          if (ok) {
            lamv[lane] = static_cast<uint8_t>(lane <= L ? lam : 0);
            llog[lane] = static_cast<uint8_t>((lane <= L && lam) ? F.log[lam] : 0xff);
            int found = 0;
            if (rho == nroots) {  // Lambda = Gamma: its roots are the erasures
              if (lane < L) pos[lane] = upos[lane];
              found = L;
            } else {
              __syncwarp();
              for (int i0 = 0; i0 < n; i0 += 32) {  // Lambda(alpha^-i) == 0  <=>  errata at position i
                const int i = i0 + lane;
                unsigned v = 1;  // Lambda_0 = 1
                if (i < n) {
                  const unsigned e = i ? n - i : 0;
                  unsigned acc = 0;
                  for (int k = 1; k <= L; ++k) {
                    acc += e;
                    if (acc >= static_cast<unsigned>(n)) acc -= n;
                    const unsigned lg = llog[k];
                    if (lg != 0xff) v ^= F.exp[lg + acc];
                  }
                }
                const unsigned hit = __ballot_sync(kGfAll, i < n && v == 0);
                if (i < n && v == 0) {
                  const int slot = found + __popc(hit & ((1u << lane) - 1u));
                  if (slot < 32) pos[slot] = static_cast<uint8_t>(i);
                }
                found += __popc(hit);
              }
            }
            __syncwarp();
            ok = found == L;
            if (ok) {
              // ---------------- Forney: Omega = S * Lambda mod x^(2t);  e = X^(1-mu) Omega(1/X) / Lambda'(1/X)
              if (lane < L) {
                unsigned o = 0;
                for (int j = 0; j <= lane; ++j) o ^= F.mul(lamv[j], synd[lane - j]);
                omega[lane] = static_cast<uint8_t>(o);
              }
              __syncwarp();
              bool bad = false;
              if (lane < L) {
                pk = pos[lane];
                const unsigned e = pk ? n - pk : 0;  // 1/X = alpha^-pos
                unsigned num = 0, den = 0, acc = 0;  // acc = exponent of (1/X)^k
                for (int k = 0; k < L; ++k) {
                  num ^= F.mul_alpha(omega[k], acc);
                  if ((k & 1) == 0) den ^= F.mul_alpha(lamv[k + 1], acc);  // Lambda' = sum_{k odd} Lambda_k x^(k-1)
                  acc += e;
                  if (acc >= static_cast<unsigned>(n)) acc -= n;
                }
                const unsigned xe = (pk * mu_exp) % n;  // X^(1-mu)
                if (den != 0 && num != 0) val = F.exp[(F.log[num] + n - F.log[den] + xe) % n];
                // K4's rule: a zero value is a failure unless the position is erased
                if (val == 0) {
                  bool erased = false;
                  for (int e2 = 0; e2 < rho; ++e2) erased |= upos[e2] == pk;
                  bad = !erased;
                }
              }
              ok = !__any_sync(kGfAll, bad);
            }
          }
          if (ok) {
            // ---------------- metric over the changed bits, ascending image position
            if (lane < L) ev[pk] = static_cast<uint8_t>(val);
            __syncwarp();
            float D = 0.0f;
            for (int ch = 0; ch < nch; ++ch) {
              const int c = 32 * ch + lane;
              unsigned mask = __ballot_sync(kGfAll, c < n && ev[c] != 0);
              if (lane == 0) {
                while (mask) {
                  const int s = 32 * ch + __ffs(mask) - 1;
                  mask &= mask - 1;
                  const unsigned v = ev[s];
                  for (int j = 0; j < q; ++j)
                    if ((v >> j) & 1u) D = __fadd_rn(D, fabsf(sy[s * q + j]));
                }
              }
            }
            D = __shfl_sync(kGfAll, D, 0);
            __syncwarp();
            if (lane < L) ev[pk] = 0;
            const unsigned long long key = (static_cast<unsigned long long>(nan_key(D)) << 32) | static_cast<unsigned>(tr);
            if (key < best) {
              best = key;
              bpos = pk;
              bval = lane < L ? val : 0u;
            }
          }
          __syncwarp();
        }
        failed = best == ~0ull;
        chosen = failed ? 0u : static_cast<unsigned>(best & 0xffu);
        if (!failed && bval) word[bpos] ^= static_cast<uint8_t>(bval);
        __syncwarp();
      }
    }
    if (kFused) {
      unsigned nzs = 0, nb = 0;
      for (int c = lane; c < n; c += 32) {
        const unsigned v = word[c];
        nzs += v != 0;
        nb += __popc(v);
      }
      const unsigned nz = __reduce_add_sync(kGfAll, nzs);
      c_frames += 1;
      c_fail += failed;
      c_berr += __reduce_add_sync(kGfAll, nb);
      c_ferr += (failed || nz) ? 1 : 0;
      c_und += (!failed && nz) ? 1 : 0;
    } else {
      for (int c = lane; c < n; c += 32) p.words[w * n + c] = word[c];
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

template <bool kFused> int launch(const GfDevice &d, const GmdParams &gp, int sm_count, cudaStream_t stream) {
  if (gp.frames == 0) return 0;
  const size_t smem = gf_table_bytes(d.q, d.nroots) + size_t(kGmdWarps) * gp.warp_bytes;
  if (cudaFuncSetAttribute(gmd_kernel<kFused>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) !=
      cudaSuccess)
    return -1;
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gmd_kernel<kFused>, kGmdThreads, smem);
  const uint64_t want = (gp.frames + kGmdWarps - 1) / kGmdWarps;
  const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(want, uint64_t(std::max(1, occ)) * sm_count));
  gmd_kernel<kFused><<<grid, kGmdThreads, smem, stream>>>(gp);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

bool supported(const GfDevice &d, uint32_t max_erasures) {
  return d.tables && !d.binary && d.nroots <= static_cast<int>(kGmdMaxRoots) && d.step == 1 && d.n <= 255 &&
         (max_erasures & 1u) == 0 && max_erasures <= static_cast<uint32_t>(d.nroots);
}

GmdParams params_of(const GfDevice &d, uint32_t max_erasures) {
  GmdParams gp{};
  gp.q = d.q;
  gp.n = d.n;
  gp.nroots = d.nroots;
  gp.mu = d.mu;
  gp.F = static_cast<int>(max_erasures);
  gp.y_bytes = (d.n * d.q * static_cast<int>(sizeof(float)) + 15) & ~15;
  gp.warp_bytes = gp.y_bytes + kGmdFixedBytes;
  gp.tables = d.tables;
  return gp;
}

}  // namespace

int gmd_launch(const GfDevice &d, uint32_t max_erasures, const float *y, uint64_t frames, uint8_t *words,
               uint8_t *failed, uint8_t *chosen, int sm_count, cudaStream_t stream) {
  if (!supported(d, max_erasures)) return -3;
  GmdParams gp = params_of(d, max_erasures);
  gp.y = y;
  gp.frames = frames;
  gp.words = words;
  gp.failed = failed;
  gp.chosen = chosen;
  return launch<false>(d, gp, sm_count, stream);
}

int gmd_awgn_launch(const GfDevice &d, uint32_t max_erasures, float sigma, uint64_t seed, uint32_t point, uint64_t frame0,
                    uint64_t frames, unsigned long long *counters, int sm_count, cudaStream_t stream) {
  if (!supported(d, max_erasures)) return -3;
  GmdParams gp = params_of(d, max_erasures);
  gp.frames = frames;
  gp.sigma = sigma;
  gp.point = point;
  gp.frame0 = frame0;
  gp.counters = counters;
  gp.keys = philox_round_keys(seed);
  return launch<true>(d, gp, sm_count, stream);
}

}  // namespace ccgpu
