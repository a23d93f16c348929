// abp.cu -- K8: adaptive belief propagation (ABP, Jiang-Narayanan) of binary primitive BCH codes with the min-sum check
// pass, one warp per frame.
//
// Per frame (include/ccgpu.h, ccgpu_decode_llr_abp, states the contract):
//   L_c = y_c clamped to [-B, B] (NaN -> +0.0, B = 2^20); for j = 0, 1, ..: x = (L < 0); H x = 0 stops with iter = j,
//   j = max_iter stops failed; otherwise the columns are visited in ascending (bits(|L_c|), c), P = p_0, p_1, .. are
//   the columns picked greedily in that order whose H-column is independent of those picked before, A is the matrix
//   with the row space of H and A[:, P] = I (row i <-> p_i), and each column gets S_c = +0.0 + sum over the rows i of A
//   holding c, i ascending, of the min-sum message m_{i,c}; then L_c <- clamp(L_c + gamma S_c).
//
// Work split inside the warp (n <= 127, k <= 64: a column set is two uint64, bit c <-> column c)
//   channel     lane <-> column (HBM) or Philox block (fused path, awgn_block of channel.cuh); L lives in registers,
//               lane bit ch <-> column 32 ch + lane, with a copy in shared memory for the row walks.
//   stop test   lane r holds rows r and r + 32 of H in registers; ballots give x, parity(row & x) per row.
//   order       comparison counting: rank of column j = #{i : (key_i, i) < (key_j, j)}, lane <-> column (as K6).
//   elimination Gauss-Jordan from H in the visiting order (as K6): a ballot finds the unpivoted rows holding column c,
//               the lowest one becomes the pivot row of c and is shuffled to the warp, every other row holding c adds
//               it.  The pivot row of the i-th pick is row i of A: its pick index is recorded.
//   rows        lane <-> row: one walk over the row's columns gives min1, min2, the first column attaining min1 and the
//               parity of the negatives; they and the row are stored at the row's pick index.  Then mu_{i,c} =
//               (c == argmin) ? min2 : min1, which is the minimum over the other columns, ties included.
//   columns     lane <-> column: rows i = 0..k-1 in ascending order, __fadd_rn of each message, then the damped update
//               with __fmul_rn / __fadd_rn (no contraction into FMA: the contract multiplies and adds separately).
#include <algorithm>

#include "abp.h"
#include "channel.cuh"
#include "ms_params.h"

namespace ccgpu {

namespace {

constexpr unsigned kAll = 0xffffffffu;
constexpr int kAbpThreads = 256;
constexpr int kAbpWarps = kAbpThreads / 32;
constexpr float kAbpBound = 1048576.0f;  // B = 2^20
// per warp: L[128] floats, the rows of A[64] as column sets, their statistics[64] as uint4, order[128]
constexpr int kAbpWarpBytes = 512 + 64 * 16 + 64 * 16 + 128;

struct AbpParams {
  int n, k, max_iter;
  float gamma;
  const unsigned long long *rows;
  const float *y;  // HBM source
  unsigned long long frames;
  uint8_t *bits, *iter, *failed;
  float *L;
  // fused source: frame f is frame frame0 + f of the stream (keys, point)
  float sigma;
  uint32_t point;
  unsigned long long frame0;
  unsigned long long *counters;
  PhiloxKeys keys;
};

__device__ __forceinline__ bool has(unsigned long long lo, unsigned long long hi, int c) {
  return (((c < 64) ? lo : hi) >> (c & 63)) & 1ull;
}

// step 1 of the contract: NaN -> +0.0, everything else clamped to [-B, B]
__device__ __forceinline__ float clamp_llr(float v) { return v != v ? 0.0f : fminf(fmaxf(v, -kAbpBound), kAbpBound); }

// min1, min2 (as bits), the first column attaining min1, and the parity of the negatives over the columns of a row
__device__ __forceinline__ uint4 row_stats(unsigned long long r0, unsigned long long r1, const float *sL) {
  float m1 = __int_as_float(0x7f800000), m2 = m1;
  unsigned arg = 0, par = 0;
#pragma unroll
  for (int wd = 0; wd < 2; ++wd) {
    for (unsigned long long rest = wd ? r1 : r0; rest; rest &= rest - 1) {
      const unsigned c = 64 * wd + __ffsll(rest) - 1;
      const float v = sL[c], a = fabsf(v);
      par ^= v < 0.0f ? 1u : 0u;
      if (a < m1) {
        m2 = m1;
        m1 = a;
        arg = c;
      } else if (a < m2) {
        m2 = a;
      }
    }
  }
  if (m2 == __int_as_float(0x7f800000)) m2 = 0.0f;  // a row of weight 1 sends +0.0
  return make_uint4(__float_as_uint(m1), __float_as_uint(m2), arg, par);
}

template <bool kFused>
__global__ void __launch_bounds__(kAbpThreads) abp_kernel(const __grid_constant__ AbpParams p) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t *base = sm + warp * kAbpWarpBytes;
  float *sL = reinterpret_cast<float *>(base);                    // [128] L_c
  ulonglong2 *srow = reinterpret_cast<ulonglong2 *>(base + 512);  // [64] row i of A
  uint4 *sst = reinterpret_cast<uint4 *>(srow + 64);              // [64] min1, min2, argmin, parity of row i
  uint8_t *order = reinterpret_cast<uint8_t *>(sst + 64);         // [128] column of rank i
  const int n = p.n, k = p.k;
  const int nch = (n + 31) / 32;
  const bool ra = lane < k, rb = lane + 32 < k;
  const unsigned long long a0i = ra ? p.rows[2 * lane] : 0ull, a1i = ra ? p.rows[2 * lane + 1] : 0ull;
  const unsigned long long b0i = rb ? p.rows[2 * (lane + 32)] : 0ull, b1i = rb ? p.rows[2 * (lane + 32) + 1] : 0ull;
  unsigned long long c_frames = 0, c_ferr = 0, c_berr = 0, c_iter = 0, c_fail = 0, c_undet = 0;

  const unsigned long long nwarps = static_cast<unsigned long long>(gridDim.x) * kAbpWarps;
  for (unsigned long long w = static_cast<unsigned long long>(blockIdx.x) * kAbpWarps + warp; w < p.frames; w += nwarps) {
    float Lr[4];  // L of columns 32 ch + lane; +0.0 beyond n
    if (kFused) {
      for (int blk = lane; blk < (n + 3) / 4; blk += 32) {
        const float4 v = awgn_block(p.keys, p.point, p.frame0 + w, blk, p.sigma);
        const float vv[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (4 * blk + e < n) sL[4 * blk + e] = vv[e];
      }
      __syncwarp();
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) Lr[ch] = 32 * ch + lane < n ? sL[32 * ch + lane] : 0.0f;
      __syncwarp();
    } else {
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) Lr[ch] = 32 * ch + lane < n ? p.y[w * n + 32 * ch + lane] : 0.0f;
    }
#pragma unroll
    for (int ch = 0; ch < 4; ++ch) {
      Lr[ch] = clamp_llr(Lr[ch]);
      if (32 * ch + lane < n) sL[32 * ch + lane] = Lr[ch];
    }
    __syncwarp();
    unsigned long long h0, h1;
    int j = 0;
    bool failed;
    for (;; ++j) {
      unsigned hw[4];
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) hw[ch] = __ballot_sync(kAll, Lr[ch] < 0.0f);
      h0 = hw[0] | (static_cast<unsigned long long>(hw[1]) << 32);
      h1 = hw[2] | (static_cast<unsigned long long>(hw[3]) << 32);
      const bool odd = ((__popcll(a0i & h0) + __popcll(a1i & h1)) & 1) | ((__popcll(b0i & h0) + __popcll(b1i & h1)) & 1);
      if (!__any_sync(kAll, odd)) {
        failed = false;
        break;
      }
      if (j == p.max_iter) {
        failed = true;
        break;
      }
      // ---------------- visiting order: rank of each column by comparison counting
      {
        unsigned key[4], rank[4] = { 0, 0, 0, 0 };
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) key[ch] = __float_as_uint(fabsf(Lr[ch]));
        for (int i = 0; i < n; ++i) {
          const unsigned ki = __float_as_uint(fabsf(sL[i]));
#pragma unroll
          for (int ch = 0; ch < 4; ++ch)  // (key_i, i) < (key_j, j)  <=>  key_i + (i >= j) <= key_j  (keys < 2^31)
            if (ch < nch) rank[ch] += (ki + (i >= 32 * ch + lane ? 1u : 0u)) <= key[ch] ? 1u : 0u;
        }
#pragma unroll
        for (int ch = 0; ch < 4; ++ch)
          if (ch < nch && 32 * ch + lane < n) order[rank[ch]] = static_cast<uint8_t>(32 * ch + lane);
      }
      __syncwarp();
      // ---------------- Gauss-Jordan elimination of H in the visiting order
      unsigned long long a0 = a0i, a1 = a1i, b0 = b0i, b1 = b1i;
      bool fa = ra, fb = rb;  // row not yet a pivot row
      int ia = 0, ib = 0;     // pick indices of this lane's rows: their row index in A
      int piv = 0;
      for (int i = 0; i < n && piv < k; ++i) {
        const int c = order[i];
        const bool ba = has(a0, a1, c), bb = has(b0, b1, c);
        const unsigned ma = __ballot_sync(kAll, ba && fa), mb = __ballot_sync(kAll, bb && fb);
        if (!(ma | mb)) continue;  // dependent on the picks so far
        const bool second = ma == 0;
        const int src = __ffs(second ? mb : ma) - 1;
        const unsigned long long q0 = __shfl_sync(kAll, second ? b0 : a0, src);
        const unsigned long long q1 = __shfl_sync(kAll, second ? b1 : a1, src);
        const bool mine_a = !second && lane == src, mine_b = second && lane == src;
        if (ba && !mine_a) a0 ^= q0, a1 ^= q1;
        if (bb && !mine_b) b0 ^= q0, b1 ^= q1;
        if (mine_a) fa = false, ia = piv;
        if (mine_b) fb = false, ib = piv;
        ++piv;
      }
      // ---------------- check statistics, lane <-> row, stored in pick order
      if (ra) {
        srow[ia] = make_ulonglong2(a0, a1);
        sst[ia] = row_stats(a0, a1, sL);
      }
      if (rb) {
        srow[ib] = make_ulonglong2(b0, b1);
        sst[ib] = row_stats(b0, b1, sL);
      }
      __syncwarp();
      // ---------------- column sums in ascending row order and the damped update, lane <-> column
      float S[4] = { 0.0f, 0.0f, 0.0f, 0.0f };
      for (int i = 0; i < k; ++i) {
        const ulonglong2 row = srow[i];
        const uint4 st = sst[i];
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int c = 32 * ch + lane;
          if (ch < nch && has(row.x, row.y, c)) {
            const float mu = __uint_as_float(static_cast<unsigned>(c) == st.z ? st.y : st.x);
            const bool s = (st.w != 0) != (Lr[ch] < 0.0f);  // parity of the other columns' negatives
            S[ch] = __fadd_rn(S[ch], s ? -mu : mu);
          }
        }
      }
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const int c = 32 * ch + lane;
        if (ch < nch && c < n) {
          Lr[ch] = fminf(fmaxf(__fadd_rn(Lr[ch], __fmul_rn(p.gamma, S[ch])), -kAbpBound), kAbpBound);
          sL[c] = Lr[ch];
        }
      }
      __syncwarp();
    }
    if (kFused) {
      const unsigned nz = __popcll(h0) + __popcll(h1);
      c_frames += 1;
      c_iter += j;
      c_fail += failed ? 1 : 0;
      c_ferr += (failed || nz) ? 1 : 0;
      c_berr += nz;
      c_undet += (!failed && nz) ? 1 : 0;
    } else {
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const int c = 32 * ch + lane;
        if (c < n) {
          p.bits[w * n + c] = static_cast<uint8_t>(has(h0, h1, c));
          if (p.L) p.L[w * n + c] = Lr[ch];
        }
      }
      if (lane == 0) {
        p.iter[w] = static_cast<uint8_t>(j);
        p.failed[w] = failed ? 1 : 0;
      }
    }
    __syncwarp();
  }
  if (kFused && lane == 0) {
    if (c_frames) atomicAdd(p.counters + C_FRAMES, c_frames);
    if (c_ferr) atomicAdd(p.counters + C_FRAME_ERR, c_ferr);
    if (c_berr) atomicAdd(p.counters + C_BIT_ERR, c_berr);
    if (c_iter) atomicAdd(p.counters + C_ITER, c_iter);
    if (c_fail) atomicAdd(p.counters + C_FAIL, c_fail);
    if (c_undet) atomicAdd(p.counters + C_UNDETECTED, c_undet);
  }
}

template <bool kFused> int launch(const AbpParams &ap, int sm_count, cudaStream_t stream) {
  if (ap.frames == 0) return 0;
  const size_t smem = size_t(kAbpWarps) * kAbpWarpBytes;
  if (cudaFuncSetAttribute(abp_kernel<kFused>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) !=
      cudaSuccess)
    return -1;
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, abp_kernel<kFused>, kAbpThreads, smem);
  const uint64_t want = (ap.frames + kAbpWarps - 1) / kAbpWarps;
  const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(want, uint64_t(std::max(1, occ)) * sm_count));
  abp_kernel<kFused><<<grid, kAbpThreads, smem, stream>>>(ap);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

AbpParams params_of(const OsdDevice &d, uint32_t max_iter, float gamma) {
  AbpParams ap{};
  ap.n = d.n;
  ap.k = d.k;
  ap.max_iter = static_cast<int>(max_iter);
  ap.gamma = gamma;
  ap.rows = d.rows;
  return ap;
}

}  // namespace

int abp_launch(const OsdDevice &d, uint32_t max_iter, float gamma, const float *y, uint64_t frames, uint8_t *bits,
               float *L, uint8_t *iter, uint8_t *failed, int sm_count, cudaStream_t stream) {
  if (!d.rows || max_iter > kAbpMaxIter) return -3;
  AbpParams ap = params_of(d, max_iter, gamma);
  ap.y = y;
  ap.frames = frames;
  ap.bits = bits;
  ap.L = L;
  ap.iter = iter;
  ap.failed = failed;
  return launch<false>(ap, sm_count, stream);
}

int abp_awgn_launch(const OsdDevice &d, uint32_t max_iter, float gamma, float sigma, uint64_t seed, uint32_t point,
                    uint64_t frame0, uint64_t frames, unsigned long long *counters, int sm_count, cudaStream_t stream) {
  if (!d.rows || max_iter > kAbpMaxIter) return -3;
  AbpParams ap = params_of(d, max_iter, gamma);
  ap.frames = frames;
  ap.sigma = sigma;
  ap.point = point;
  ap.frame0 = frame0;
  ap.counters = counters;
  ap.keys = philox_round_keys(seed);
  return launch<true>(ap, sm_count, stream);
}

}  // namespace ccgpu
