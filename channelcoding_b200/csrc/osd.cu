// osd.cu -- K6: ordered-statistics decoding (OSD-i) of binary primitive BCH codes, one warp per frame.
//
// Per frame (include/ccgpu.h, ccgpu_decode_llr_osd, states the contract):
//   h_c = (y_c < 0); the columns are visited in ascending (bits(|y_c|), c); P = the columns picked greedily in that
//   order whose H-column is independent of those picked before (|P| = k), I = the other l columns, i_0 < .. < i_{l-1};
//   candidate e is the codeword x_e with x_e[I] = h[I] ^ 1_{E_e}, E_e the sets of at most `order` positions of I in
//   the order empty, singles, pairs, triples (each lexicographic); D_e = sum over the columns where x_e != h of |y_c|
//   (float32, c ascending, from +0.0); the smallest (K(D_e), e) wins, K = bits with every NaN as 0x7fc00000.
//
// Work split inside the warp (n <= 127, k <= 64: a column set is two uint64, bit c <-> column c)
//   channel     lane <-> column (HBM) or Philox block (fused path, awgn_block of channel.cuh); |y| stays in shared
//               memory for the order and the metric.
//   syndrome    lane r holds rows r and r + 32 of H in registers; parity(row & h) per row.  All zero: h is a codeword,
//               candidate 0 wins with D = +0.0 and the frame ends.
//   order       comparison counting: rank of column j = #{i : (key_i, i) < (key_j, j)}, lane <-> column.
//   elimination Gauss-Jordan in the visiting order: a ballot finds the unpivoted rows holding column c, the lowest one
//               becomes the pivot of c and is shuffled to the warp, every other row holding c adds it.  No such row:
//               c is an information column.  Stops after k pivots.
//   generator   row r of the reduced H has bit p_r (its pivot) and otherwise only information columns, so the
//               codeword with information part u has x[p_r] = parity(row_r & u).  Hence x_0 ^ h is the set of pivots
//               whose row has odd parity with h, and flipping information column c flips g_c = 1_c | {p_r : row_r
//               has c}.  g is built lane <-> information column into shared memory.
//   candidates  lane <-> candidate (e = lane, lane + 32, .. within each weight class); diff = diff0 ^ g_a ^ g_b ^ g_c,
//               summed serially over its set bits in ascending column order, so every lane computes the contract's
//               float sum on its own.  A lane stops a sum once it reaches its own best key: the sum cannot decrease
//               and the lane's later candidates lose ties.  One warp minimum per frame picks the winner.
#include <algorithm>

#include "channel.cuh"
#include "ms_params.h"
#include "osd.h"

namespace ccgpu {

namespace {

constexpr unsigned kAll = 0xffffffffu;
constexpr int kOsdThreads = 256;
constexpr int kOsdWarps = kOsdThreads / 32;
// per warp: |y|[128] floats, g[128] and reduced rows[64] as column sets, order[128], pivot column of row[64]
constexpr int kOsdWarpBytes = 512 + 128 * 16 + 64 * 16 + 128 + 64;

struct OsdParams {
  int n, k, l, order;
  uint32_t count[4];  // C(l, w) candidates of weight w, 0 above the order
  const unsigned long long *rows;
  const float *y;  // HBM source
  unsigned long long frames;
  uint8_t *bits, *weight;
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

// moves the combination (a < b < c of the first w) s places on in the lexicographic order of w-subsets of 0..l-1;
// the caller guarantees the target exists
__device__ __forceinline__ void advance(int w, int l, int &a, int &b, int &c, int s) {
  if (w == 1) {
    a += s;
  } else if (w == 2) {
    b += s;
    while (b >= l) {
      const int over = b - l;
      ++a;
      b = a + 1 + over;
    }
  } else if (w == 3) {
    c += s;
    while (c >= l) {
      const int over = c - l;
      if (++b >= l - 1) {
        ++a;
        b = a + 1;
      }
      c = b + 1 + over;
    }
  }
}

template <bool kFused>
__global__ void __launch_bounds__(kOsdThreads) osd_kernel(const __grid_constant__ OsdParams p) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t *base = sm + warp * kOsdWarpBytes;
  float *sa = reinterpret_cast<float *>(base);                  // [128] |y_c|
  ulonglong2 *gt = reinterpret_cast<ulonglong2 *>(base + 512);  // [128] g of information column i_a, by a
  ulonglong2 *srow = gt + 128;                                  // [64] reduced rows
  uint8_t *order = reinterpret_cast<uint8_t *>(srow + 64);      // [128] column of rank i
  uint8_t *pivcol = order + 128;                                // [64] pivot column of row r
  const int n = p.n, k = p.k, l = p.l;
  const int nch = (n + 31) / 32;  // column chunks: lane bit ch <-> column 32 ch + lane
  const bool ra = lane < k, rb = lane + 32 < k;
  const unsigned long long a0i = ra ? p.rows[2 * lane] : 0ull, a1i = ra ? p.rows[2 * lane + 1] : 0ull;
  const unsigned long long b0i = rb ? p.rows[2 * (lane + 32)] : 0ull, b1i = rb ? p.rows[2 * (lane + 32) + 1] : 0ull;
  unsigned long long c_frames = 0, c_ferr = 0, c_berr = 0;

  const unsigned long long nwarps = static_cast<unsigned long long>(gridDim.x) * kOsdWarps;
  for (unsigned long long w = static_cast<unsigned long long>(blockIdx.x) * kOsdWarps + warp; w < p.frames; w += nwarps) {
    unsigned hw[4];  // hard decision, word ch <-> columns 32 ch .. 32 ch + 31 (codes.h:43-52: y < 0)
    if (kFused) {
      for (int blk = lane; blk < (n + 3) / 4; blk += 32) {
        const float4 v = awgn_block(p.keys, p.point, p.frame0 + w, blk, p.sigma);
        const float vv[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (4 * blk + e < n) sa[4 * blk + e] = vv[e];
      }
      __syncwarp();
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const int c = 32 * ch + lane;
        const float v = c < n ? sa[c] : 0.0f;
        hw[ch] = __ballot_sync(kAll, v < 0.0f);
        if (c < n) sa[c] = fabsf(v);
      }
    } else {
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const int c = 32 * ch + lane;
        const float v = c < n ? p.y[w * n + c] : 0.0f;
        hw[ch] = __ballot_sync(kAll, v < 0.0f);
        if (c < n) sa[c] = fabsf(v);
      }
    }
    const unsigned long long h0 = hw[0] | (static_cast<unsigned long long>(hw[1]) << 32);
    const unsigned long long h1 = hw[2] | (static_cast<unsigned long long>(hw[3]) << 32);
    unsigned long long d0 = 0, d1 = 0;  // winner's x ^ h
    unsigned wweight = 0;
    const bool odd = ((__popcll(a0i & h0) + __popcll(a1i & h1)) & 1) | ((__popcll(b0i & h0) + __popcll(b1i & h1)) & 1);
    __syncwarp();
    if (__any_sync(kAll, odd)) {
      // ---------------- visiting order: rank of each column by comparison counting
      {
        unsigned key[4], rank[4] = { 0, 0, 0, 0 };
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) key[ch] = 32 * ch + lane < n ? __float_as_uint(sa[32 * ch + lane]) : 0u;
        for (int i = 0; i < n; ++i) {
          const unsigned ki = __float_as_uint(sa[i]);
#pragma unroll
          for (int ch = 0; ch < 4; ++ch)  // (key_i, i) < (key_j, j)  <=>  key_i + (i >= j) <= key_j  (keys < 2^31)
            if (ch < nch) rank[ch] += (ki + (i >= 32 * ch + lane ? 1u : 0u)) <= key[ch] ? 1u : 0u;
        }
#pragma unroll
        for (int ch = 0; ch < 4; ++ch)
          if (ch < nch && 32 * ch + lane < n) order[rank[ch]] = static_cast<uint8_t>(32 * ch + lane);
      }
      __syncwarp();
      // ---------------- Gauss-Jordan elimination in the visiting order
      unsigned long long a0 = a0i, a1 = a1i, b0 = b0i, b1 = b1i;
      bool fa = ra, fb = rb;  // row not yet a pivot row
      int pa = 0, pb = 0;     // pivot columns of this lane's rows
      unsigned long long pm0 = 0, pm1 = 0;  // pivot columns
      int piv = 0;
      for (int i = 0; i < n && piv < k; ++i) {
        const int c = order[i];
        const bool ba = has(a0, a1, c), bb = has(b0, b1, c);
        const unsigned ma = __ballot_sync(kAll, ba && fa), mb = __ballot_sync(kAll, bb && fb);
        if (!(ma | mb)) continue;  // dependent on the pivots so far: information column
        const bool second = ma == 0;
        const int src = __ffs(second ? mb : ma) - 1;
        const unsigned long long q0 = __shfl_sync(kAll, second ? b0 : a0, src);
        const unsigned long long q1 = __shfl_sync(kAll, second ? b1 : a1, src);
        const bool mine_a = !second && lane == src, mine_b = second && lane == src;
        if (ba && !mine_a) a0 ^= q0, a1 ^= q1;
        if (bb && !mine_b) b0 ^= q0, b1 ^= q1;
        if (mine_a) fa = false, pa = c;
        if (mine_b) fb = false, pb = c;
        if (c < 64) pm0 |= 1ull << c;
        else pm1 |= 1ull << (c - 64);
        ++piv;
      }
      if (ra) {
        srow[lane] = make_ulonglong2(a0, a1);
        pivcol[lane] = static_cast<uint8_t>(pa);
      }
      if (rb) {
        srow[lane + 32] = make_ulonglong2(b0, b1);
        pivcol[lane + 32] = static_cast<uint8_t>(pb);
      }
      // diff0 = x_0 ^ h: the pivots of the rows with odd parity against h
      {
        const bool oa = ra && (((__popcll(a0 & h0) + __popcll(a1 & h1)) & 1) != 0);
        const bool ob = rb && (((__popcll(b0 & h0) + __popcll(b1 & h1)) & 1) != 0);
        unsigned part[4];
#pragma unroll
        for (int wd = 0; wd < 4; ++wd)
          part[wd] = (oa && (pa >> 5) == wd ? 1u << (pa & 31) : 0u) | (ob && (pb >> 5) == wd ? 1u << (pb & 31) : 0u);
#pragma unroll
        for (int wd = 0; wd < 4; ++wd) part[wd] = __reduce_or_sync(kAll, part[wd]);
        d0 = part[0] | (static_cast<unsigned long long>(part[1]) << 32);
        d1 = part[2] | (static_cast<unsigned long long>(part[3]) << 32);
      }
      __syncwarp();
      // ---------------- g of every information column, lane <-> column
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const int j = 32 * ch + lane;
        if (ch < nch && j < n && !has(pm0, pm1, j)) {
          // a = number of information columns below j
          const unsigned long long below0 = j < 64 ? (1ull << j) - 1 : ~0ull;
          const unsigned long long below1 = j < 64 ? 0ull : (1ull << (j - 64)) - 1;
          const int a = j - __popcll(pm0 & below0) - __popcll(pm1 & below1);
          unsigned long long g0 = j < 64 ? 1ull << j : 0ull, g1 = j < 64 ? 0ull : 1ull << (j - 64);
          for (int r = 0; r < k; ++r) {
            const ulonglong2 row = srow[r];
            if (has(row.x, row.y, j)) {
              const int pc = pivcol[r];
              if (pc < 64) g0 |= 1ull << pc;
              else g1 |= 1ull << (pc - 64);
            }
          }
          gt[a] = make_ulonglong2(g0, g1);
        }
      }
      __syncwarp();
      // ---------------- candidates
      unsigned kbest = 0xffffffffu, ebest = 0xffffffffu, wbest = 0;
      unsigned long long bd0 = 0, bd1 = 0;
      uint32_t ebase = 0;
      for (int wt = 0; wt <= p.order; ++wt) {
        const uint32_t cnt = p.count[wt];
        int ia = 0, ib = 1, ic = 2;
        if (static_cast<uint32_t>(lane) < cnt) advance(wt, l, ia, ib, ic, lane);
        for (uint32_t m = lane; m < cnt; m += 32) {
          unsigned long long x0 = d0, x1 = d1;
          if (wt >= 1) {
            const ulonglong2 g = gt[ia];
            x0 ^= g.x, x1 ^= g.y;
          }
          if (wt >= 2) {
            const ulonglong2 g = gt[ib];
            x0 ^= g.x, x1 ^= g.y;
          }
          if (wt >= 3) {
            const ulonglong2 g = gt[ic];
            x0 ^= g.x, x1 ^= g.y;
          }
          float D = 0.0f;
          unsigned kd = 0;
          bool live = kbest != 0;
          for (unsigned long long rest = x0; rest && live;) {
            D = __fadd_rn(D, sa[__ffsll(rest) - 1]);
            rest &= rest - 1;
            kd = D != D ? 0x7fc00000u : __float_as_uint(D);
            live = kd < kbest;
          }
          for (unsigned long long rest = x1; rest && live;) {
            D = __fadd_rn(D, sa[63 + __ffsll(rest)]);
            rest &= rest - 1;
            kd = D != D ? 0x7fc00000u : __float_as_uint(D);
            live = kd < kbest;
          }
          if (live) {  // kd < kbest: e grows along a lane, so a tie never replaces the lane's best
            kbest = kd;
            ebest = ebase + m;
            wbest = wt;
            bd0 = x0, bd1 = x1;
          }
          if (m + 32 < cnt) advance(wt, l, ia, ib, ic, 32);
        }
        ebase += cnt;
      }
      const unsigned kmin = __reduce_min_sync(kAll, kbest);
      const unsigned emin = __reduce_min_sync(kAll, kbest == kmin ? ebest : 0xffffffffu);
      const int src = __ffs(__ballot_sync(kAll, kbest == kmin && ebest == emin)) - 1;
      d0 = __shfl_sync(kAll, bd0, src);
      d1 = __shfl_sync(kAll, bd1, src);
      wweight = __shfl_sync(kAll, wbest, src);
    }
    const unsigned long long o0 = h0 ^ d0, o1 = h1 ^ d1;
    if (kFused) {
      const unsigned nz = __popcll(o0) + __popcll(o1);
      c_frames += 1;
      c_berr += nz;
      c_ferr += nz ? 1 : 0;
    } else {
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        const int c = 32 * ch + lane;
        if (c < n) p.bits[w * n + c] = static_cast<uint8_t>(has(o0, o1, c));
      }
      if (lane == 0 && p.weight) p.weight[w] = static_cast<uint8_t>(wweight);
    }
    __syncwarp();
  }
  if (kFused && lane == 0) {
    if (c_frames) atomicAdd(p.counters + C_FRAMES, c_frames);
    if (c_ferr) atomicAdd(p.counters + C_FRAME_ERR, c_ferr);
    if (c_berr) atomicAdd(p.counters + C_BIT_ERR, c_berr);
    if (c_ferr) atomicAdd(p.counters + C_UNDETECTED, c_ferr);  // every frame decodes to a codeword
  }
}

template <bool kFused> int launch(const OsdParams &op, int sm_count, cudaStream_t stream) {
  if (op.frames == 0) return 0;
  const size_t smem = size_t(kOsdWarps) * kOsdWarpBytes;
  if (cudaFuncSetAttribute(osd_kernel<kFused>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) !=
      cudaSuccess)
    return -1;
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, osd_kernel<kFused>, kOsdThreads, smem);
  const uint64_t want = (op.frames + kOsdWarps - 1) / kOsdWarps;
  const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(want, uint64_t(std::max(1, occ)) * sm_count));
  osd_kernel<kFused><<<grid, kOsdThreads, smem, stream>>>(op);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

bool supported(const OsdDevice &d, uint32_t order) { return d.rows && order <= kOsdMaxOrder; }

OsdParams params_of(const OsdDevice &d, uint32_t order) {
  OsdParams op{};
  op.n = d.n;
  op.k = d.k;
  op.l = d.n - d.k;
  op.order = static_cast<int>(order);
  uint64_t c = 1;
  for (uint32_t w = 0; w <= order; ++w) {  // C(l, w) = C(l, w - 1) (l - w + 1) / w
    if (w) c = c * static_cast<uint64_t>(std::max(op.l - static_cast<int>(w) + 1, 0)) / w;
    op.count[w] = static_cast<uint32_t>(c);
  }
  op.rows = d.rows;
  return op;
}

}  // namespace

int osd_upload(const CodeSpec &spec, OsdDevice *d) {
  osd_free(d);
  if (spec.family != 0 || spec.n > kOsdMaxN || spec.k > kOsdMaxK || spec.k == 0 || spec.rows != spec.k) return 0;
  std::vector<unsigned long long> packed(2 * size_t(spec.k), 0ull);
  for (unsigned r = 0; r < spec.k; ++r)
    for (unsigned c = 0; c < spec.n; ++c)
      if (spec.H[size_t(r) * spec.n + c]) packed[2 * r + c / 64] |= 1ull << (c % 64);
  if (cudaMalloc(&d->rows, packed.size() * sizeof(unsigned long long)) != cudaSuccess) {
    d->rows = nullptr;
    return -1;
  }
  if (cudaMemcpy(d->rows, packed.data(), packed.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice) !=
      cudaSuccess) {
    osd_free(d);
    return -1;
  }
  d->n = static_cast<int>(spec.n);
  d->k = static_cast<int>(spec.k);
  return 0;
}

void osd_free(OsdDevice *d) {
  if (d->rows) cudaFree(d->rows);
  *d = OsdDevice{};
}

int osd_launch(const OsdDevice &d, uint32_t order, const float *y, uint64_t frames, uint8_t *bits, uint8_t *weight,
               int sm_count, cudaStream_t stream) {
  if (!supported(d, order)) return -3;
  OsdParams op = params_of(d, order);
  op.y = y;
  op.frames = frames;
  op.bits = bits;
  op.weight = weight;
  return launch<false>(op, sm_count, stream);
}

int osd_awgn_launch(const OsdDevice &d, uint32_t order, float sigma, uint64_t seed, uint32_t point, uint64_t frame0,
                    uint64_t frames, unsigned long long *counters, int sm_count, cudaStream_t stream) {
  if (!supported(d, order)) return -3;
  OsdParams op = params_of(d, order);
  op.frames = frames;
  op.sigma = sigma;
  op.point = point;
  op.frame0 = frame0;
  op.counters = counters;
  op.keys = philox_round_keys(seed);
  return launch<true>(op, sm_count, stream);
}

}  // namespace ccgpu
