// gf_device.cuh -- device pieces shared by the algebraic decoders over GF(2^q), q <= 8: K4 gf_decode_kernel
// (gf_decode.cu) and K5 chase_kernel (chase.cu).  One warp per word; lane <-> syndrome index.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace ccgpu {

constexpr unsigned kGfAll = 0xffffffffu;

struct Gf {
  const uint8_t *exp, *log;
  __device__ __forceinline__ unsigned mul(unsigned a, unsigned b) const { return (a && b) ? exp[log[a] + log[b]] : 0u; }
  __device__ __forceinline__ unsigned mul_alpha(unsigned a, unsigned e) const { return a ? exp[log[a] + e] : 0u; }  // e < n
};

__device__ __forceinline__ unsigned xor_reduce(unsigned v) {
  return __reduce_xor_sync(kGfAll, v);  // REDUX.XOR: one instruction instead of a five-step shuffle butterfly
}

// shared memory in front of the per-warp buffers: per-lane multiplication tables, exp / log, root exponents
struct GfShared {
  uint32_t *mtab;   // [ntab][size][32]: T[x * 32 + lane] = x * alpha^(root_(32 tb + lane))
  uint8_t *exp;     // [2*size]
  uint8_t *log;     // [size]
  uint8_t *rexp;    // [64] root exponents (mu + j) mod n
  uint8_t *rest;    // first byte after the tables (16-byte aligned)
};

__host__ __device__ __forceinline__ size_t gf_table_bytes(int q, int nroots) {
  const size_t size = size_t(1) << q;
  return size_t((nroots + 31) / 32) * size * 32 * sizeof(uint32_t) + 3 * size + 64;
}

// where the tables live in front of the per-warp buffers
__device__ __forceinline__ GfShared gf_table_layout(uint8_t *sm, int q, int nroots) {
  const int size = 1 << q;
  const int ntab = (nroots + 31) / 32;
  GfShared s;
  s.mtab = reinterpret_cast<uint32_t *>(sm);
  s.exp = sm + size_t(ntab) * size * 32 * sizeof(uint32_t);
  s.log = s.exp + 2 * size;
  s.rexp = s.log + size;
  s.rest = s.rexp + 64;
  return s;
}

// fills the tables from `tables` (exp[2*size] then log[size], as gf_upload stores them); every thread of the block
// takes part, the block is synchronised on return.  gf_decode_kernel carries the same prologue written out (see there).
__device__ __forceinline__ void gf_fill_tables(const GfShared &s, const uint8_t *tables, int q, int n, int nroots, int mu) {
  const int size = 1 << q;
  const int ntab = (nroots + 31) / 32;
  for (int i = threadIdx.x; i < 3 * size; i += blockDim.x) s.exp[i] = tables[i];
  if (threadIdx.x < 64) s.rexp[threadIdx.x] = static_cast<uint8_t>(threadIdx.x < nroots ? (mu + threadIdx.x) % n : 0);
  __syncthreads();
  for (int i = threadIdx.x; i < ntab * size * 32; i += blockDim.x) {
    const int tb = i / (size * 32), x = (i / 32) % size, j = tb * 32 + (i & 31);
    unsigned v = 0;
    if (x && j < nroots) v = s.exp[s.log[x] + s.rexp[j]];
    s.mtab[i] = v;
  }
  __syncthreads();
}

// syndromes of `word` (zero padded to a multiple of 4 bytes per segment) into synd[0..nroots); P has q, n, nroots.
//   lane <-> syndrome index.  Multiplying by the constant alpha^(root_j) is ONE shared-memory lookup in a per-lane
//   table T[x][lane] (32-bit entries: lane j always hits bank j, conflict free); the word is cut into four segments
//   whose Horner chains run interleaved (4 independent dependency chains), symbols arrive as 32-bit broadcasts of
//   four packed bytes.  Returns whether any syndrome is non-zero.
template <typename P>
__device__ __forceinline__ bool syndromes(const P &p, const Gf &F, const uint8_t *word, const uint32_t *mtab,
                                          const uint8_t *rexp, uint8_t *synd, int lane) {
  const int seg = ((p.n + 15) / 16) * 4;  // segment length in symbols, multiple of 4; 4 segments cover n
  bool any = false;
  for (int j0 = 0; j0 < p.nroots; j0 += 32) {
    const int j = j0 + lane;
    const uint32_t *T = mtab + (j0 / 32) * (32 << p.q) + lane;  // T[x * 32] = x * alpha^(root_j)
    unsigned v0 = 0, v1 = 0, v2 = 0, v3 = 0;
    for (int i = seg - 4; i >= 0; i -= 4) {
      const uint32_t w0 = *reinterpret_cast<const uint32_t *>(word + i);
      const uint32_t w1 = *reinterpret_cast<const uint32_t *>(word + seg + i);
      const uint32_t w2 = *reinterpret_cast<const uint32_t *>(word + 2 * seg + i);
      const uint32_t w3 = *reinterpret_cast<const uint32_t *>(word + 3 * seg + i);
#pragma unroll
      for (int b = 3; b >= 0; --b) {
        v0 = T[v0 * 32] ^ ((w0 >> (8 * b)) & 0xffu);
        v1 = T[v1 * 32] ^ ((w1 >> (8 * b)) & 0xffu);
        v2 = T[v2 * 32] ^ ((w2 >> (8 * b)) & 0xffu);
        v3 = T[v3 * 32] ^ ((w3 >> (8 * b)) & 0xffu);
      }
    }
    unsigned s = 0;
    if (j < p.nroots) {
      // S = v0 + v1 X^seg + v2 X^(2 seg) + v3 X^(3 seg),  X = alpha^(root_j)
      const unsigned e1 = (static_cast<unsigned>(rexp[j]) * seg) % p.n;
      unsigned e2 = e1 + e1, e3;
      if (e2 >= static_cast<unsigned>(p.n)) e2 -= p.n;
      e3 = e2 + e1;
      if (e3 >= static_cast<unsigned>(p.n)) e3 -= p.n;
      s = v0 ^ F.mul_alpha(v1, e1) ^ F.mul_alpha(v2, e2) ^ F.mul_alpha(v3, e3);
      synd[j] = static_cast<uint8_t>(s);
    }
    any |= __any_sync(kGfAll, s != 0);
  }
  __syncwarp();
  return any;
}

}  // namespace ccgpu
