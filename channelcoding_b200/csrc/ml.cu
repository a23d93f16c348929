// ml.cu -- K9: maximum-likelihood decoding of high-rate binary BCH codes by a Viterbi search over the syndrome trellis
// of the k-row H (2^k states, n sections), one thread group per frame.
//
// Per frame (include/ccgpu.h, ccgpu_decode_llr_ml, states the contract):
//   h_c = (y_c < 0), w_c = fminf(|y_c|, 2^20) (NaN -> +0.0); M_0 = (+0.0, +inf, ..); for each column c every state s
//   keeps the cheaper of the branch x_c = 0 from s and x_c = 1 from s ^ sigma_c, the branch with x_c != h_c costing
//   w_c, ties to x_c = h_c; the traceback from state 0 gives x.  A frame whose h has a zero syndrome returns h.
//
// Work split (NB = 2^(k-1) butterflies per section, G threads per frame, BPT = NB / G butterflies per thread)
//   staging     thread <-> column (HBM) or Philox block (fused path, awgn_block of channel.cuh): w_c with the sign
//               of h_c (h_c = 1 implies w_c > 0) in shared memory.  Every warp then reduces the syndrome of h.
//   forward     the metrics live in shared memory, in place.  Butterfly j of section c pairs s = j with a zero inserted
//               at the lowest set bit of sigma_c and s ^ sigma_c; both new metrics come from the same two old ones, so
//               the pairs are disjoint and the update needs no second buffer.  Only the branch with x_c != h_c adds
//               w_c: M + 0.0 == M for every metric (all are +0.0, positive or +inf).  Two ballots per warp give the
//               decisions of the lower and upper states of 32 butterflies.  One barrier per section.
//   traceback   thread 0 of the group walks the n decisions from state 0 and leaves x as four words in shared memory.
//   G           32 (one warp, k <= 9; lanes j >= NB idle for k < 6), else NB / 8 (one block of 64..256 threads).
#include <algorithm>

#include "channel.cuh"
#include "ml.h"
#include "ms_params.h"

namespace ccgpu {

namespace {

constexpr unsigned kAll = 0xffffffffu;
constexpr float kMlBound = 1048576.0f;  // 2^20

struct MlParams {
  int n;
  const float *y;  // HBM source
  unsigned long long frames;
  uint8_t *bits;
  // fused source: frame f is frame frame0 + f of the stream (keys, point)
  float sigma;
  uint32_t point;
  unsigned long long frame0;
  unsigned long long *counters;
  PhiloxKeys keys;
  uint16_t syn[kMlMaxN];  // column syndromes
};

template <int K> struct MlShape {
  static constexpr int NB = 1 << (K - 1);                       // butterflies per section
  static constexpr int G = NB / 8 > 32 ? NB / 8 : 32;           // threads per frame
  static constexpr int BPT = NB / G > 1 ? NB / G : 1;           // butterflies per thread
  static constexpr int W = NB / 32 > 1 ? NB / 32 : 1;           // decision words per half section
  static constexpr int THREADS = G == 32 ? 256 : G;             // threads per block
  static constexpr int GP = THREADS / G;                        // frames (groups) per block
  // per group: metrics [2^K], decisions [n][2][W], staged w [128], x [4]
  __host__ __device__ static size_t group_bytes(int n) { return 4u * (1u << K) + 8u * W * n + 512u + 16u; }
};

// step 2 of the contract, with the sign of h: NaN -> +0.0, else fminf(|v|, 2^20), negative when v < 0
__device__ __forceinline__ float signed_weight(float v) {
  const float w = v != v ? 0.0f : fminf(fabsf(v), kMlBound);
  return v < 0.0f ? -w : w;
}

template <int K, bool kFused>
__global__ void __launch_bounds__(MlShape<K>::THREADS) ml_kernel(const __grid_constant__ MlParams p) {
  using S = MlShape<K>;
  extern __shared__ __align__(16) uint8_t sm[];
  const int n = p.n;
  const int t = threadIdx.x % S::G, grp = threadIdx.x / S::G, lane = threadIdx.x & 31, wig = t >> 5;
  uint8_t *base = sm + grp * S::group_bytes(n);
  float *M = reinterpret_cast<float *>(base);                       // [2^K]
  unsigned *dec = reinterpret_cast<unsigned *>(M + (1 << K));       // [n][2][W]
  float *yv = reinterpret_cast<float *>(dec + 2 * S::W * n);        // [128]
  unsigned *xw = reinterpret_cast<unsigned *>(yv + 128);            // [4]
  auto sync = [] {
    if (S::G == 32)
      __syncwarp();
    else
      __syncthreads();
  };
  unsigned long long c_frames = 0, c_ferr = 0, c_berr = 0;

  const unsigned long long stride = static_cast<unsigned long long>(gridDim.x) * S::GP;
  for (unsigned long long f = static_cast<unsigned long long>(blockIdx.x) * S::GP + grp; f < p.frames; f += stride) {
    if (kFused) {
      for (int blk = t; blk < (n + 3) / 4; blk += S::G) {
        const float4 v = awgn_block(p.keys, p.point, p.frame0 + f, blk, p.sigma);
        const float vv[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (4 * blk + e < n) yv[4 * blk + e] = signed_weight(vv[e]);
      }
    } else {
      for (int c = t; c < n; c += S::G) yv[c] = signed_weight(p.y[f * n + c]);
    }
    sync();
    // syndrome and weight of h, reduced by every warp of the group
    unsigned syn = 0, hw = 0;
    for (int c = lane; c < n; c += 32)
      if (yv[c] < 0.0f) syn ^= p.syn[c], ++hw;
    syn = __reduce_xor_sync(kAll, syn);
    if (syn != 0) {
      for (int s = t; s < (1 << K); s += S::G) M[s] = s ? __int_as_float(0x7f800000) : 0.0f;
      sync();
      // ---------------- forward pass: one butterfly section per column
      for (int c = 0; c < n; ++c) {
        const unsigned sg = p.syn[c], low = (sg & (0u - sg)) - 1u;  // the bits below the lowest set bit of sigma_c
        const float v = yv[c], w = fabsf(v);
        const bool h = v < 0.0f;
#pragma unroll
        for (int i = 0; i < S::BPT; ++i) {
          const unsigned j = t + S::G * i;
          bool xl = false, xu = false;
          if (S::NB >= 32 || j < unsigned(S::NB)) {
            const unsigned s = ((j & ~low) << 1) | (j & low), s2 = s ^ sg;
            const float a = M[s], b = M[s2];
            const float aw = __fadd_rn(a, w), bw = __fadd_rn(b, w);
            const bool P = a <= bw, Q = b <= aw;  // s keeps its x_c = 0 branch, s2 keeps its x_c = 0 branch
            const float m1 = P ? a : bw, m2 = Q ? b : aw;
            M[s] = h ? m2 : m1;
            M[s2] = h ? m1 : m2;
            xl = h ? Q : !P;
            xu = h ? P : !Q;
          }
          const unsigned lo = __ballot_sync(kAll, xl), hi = __ballot_sync(kAll, xu);
          if (lane == 0) {
            const int word = wig + (S::G / 32) * i;
            dec[(2 * c) * S::W + word] = lo;
            dec[(2 * c + 1) * S::W + word] = hi;
          }
        }
        sync();
      }
      // ---------------- traceback from state 0
      if (t == 0) {
        unsigned s = 0, cur = 0, nz = 0;
        for (int c = n - 1; c >= 0; --c) {
          const unsigned sg = p.syn[c], low = (sg & (0u - sg)) - 1u;
          const unsigned up = (s & (low + 1)) != 0, lower = up ? s ^ sg : s;
          const unsigned j = ((lower >> 1) & ~low) | (lower & low);
          const unsigned x = (dec[(2 * c + up) * S::W + (j >> 5)] >> (j & 31)) & 1u;
          s ^= x ? sg : 0u;
          cur |= x << (c & 31);
          if ((c & 31) == 0) {
            xw[c >> 5] = cur;
            nz += __popc(cur);
            cur = 0;
          }
        }
        hw = nz;
      }
      sync();
    } else {
      hw = __reduce_add_sync(kAll, hw);
    }
    if (kFused) {
      if (t == 0) {  // hw is the weight of the decided word here
        c_frames += 1;
        c_ferr += hw ? 1 : 0;
        c_berr += hw;
      }
    } else {
      for (int c = t; c < n; c += S::G)
        p.bits[f * n + c] = static_cast<uint8_t>(syn ? (xw[c >> 5] >> (c & 31)) & 1u : (yv[c] < 0.0f ? 1u : 0u));
    }
    sync();
  }
  if (kFused && t == 0) {
    if (c_frames) atomicAdd(p.counters + C_FRAMES, c_frames);
    if (c_ferr) {
      atomicAdd(p.counters + C_FRAME_ERR, c_ferr);
      atomicAdd(p.counters + C_UNDETECTED, c_ferr);
    }
    if (c_berr) atomicAdd(p.counters + C_BIT_ERR, c_berr);
  }
}

template <int K, bool kFused> int launch_k(const MlParams &mp, int sm_count, cudaStream_t stream) {
  using S = MlShape<K>;
  const size_t smem = size_t(S::GP) * S::group_bytes(mp.n);
  if (cudaFuncSetAttribute(ml_kernel<K, kFused>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) !=
      cudaSuccess)
    return -1;
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ml_kernel<K, kFused>, S::THREADS, smem);
  const uint64_t want = (mp.frames + S::GP - 1) / S::GP;
  const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(want, uint64_t(std::max(1, occ)) * sm_count));
  ml_kernel<K, kFused><<<grid, S::THREADS, smem, stream>>>(mp);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

template <bool kFused> int launch(int k, const MlParams &mp, int sm_count, cudaStream_t stream) {
  if (mp.frames == 0) return 0;
  switch (k) {
  case 4: return launch_k<4, kFused>(mp, sm_count, stream);
  case 5: return launch_k<5, kFused>(mp, sm_count, stream);
  case 6: return launch_k<6, kFused>(mp, sm_count, stream);
  case 7: return launch_k<7, kFused>(mp, sm_count, stream);
  case 8: return launch_k<8, kFused>(mp, sm_count, stream);
  case 9: return launch_k<9, kFused>(mp, sm_count, stream);
  case 10: return launch_k<10, kFused>(mp, sm_count, stream);
  case 11: return launch_k<11, kFused>(mp, sm_count, stream);
  case 12: return launch_k<12, kFused>(mp, sm_count, stream);
  default: return -3;
  }
}

MlParams params_of(const MlCode &m) {
  MlParams mp{};
  mp.n = m.n;
  std::copy(m.sigma, m.sigma + kMlMaxN, mp.syn);
  return mp;
}

}  // namespace

void ml_prepare(const CodeSpec &spec, MlCode *m) {
  *m = MlCode{};
  if (spec.family != 0 || spec.n > kMlMaxN || spec.k < kMlMinK || spec.k > kMlMaxK || spec.rows != spec.k) return;
  for (unsigned c = 0; c < spec.n; ++c) {
    unsigned s = 0;
    for (unsigned r = 0; r < spec.k; ++r)
      if (spec.H[size_t(r) * spec.n + c]) s |= 1u << r;
    if (s == 0) {  // the butterflies pair s with s ^ sigma_c: a zero column has no partner
      *m = MlCode{};
      return;
    }
    m->sigma[c] = static_cast<uint16_t>(s);
  }
  m->n = static_cast<int>(spec.n);
  m->k = static_cast<int>(spec.k);
}

int ml_launch(const MlCode &m, const float *y, uint64_t frames, uint8_t *bits, int sm_count, cudaStream_t stream) {
  if (!m.k) return -3;
  MlParams mp = params_of(m);
  mp.y = y;
  mp.frames = frames;
  mp.bits = bits;
  return launch<false>(m.k, mp, sm_count, stream);
}

int ml_awgn_launch(const MlCode &m, float sigma, uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames,
                   unsigned long long *counters, int sm_count, cudaStream_t stream) {
  if (!m.k) return -3;
  MlParams mp = params_of(m);
  mp.frames = frames;
  mp.sigma = sigma;
  mp.point = point;
  mp.frame0 = frame0;
  mp.counters = counters;
  mp.keys = philox_round_keys(seed);
  return launch<true>(m.k, mp, sm_count, stream);
}

}  // namespace ccgpu
