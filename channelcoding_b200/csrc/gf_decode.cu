// gf_decode.cu -- K4: batched hard-decision (algebraic) decoding of primitive BCH / RS codes
// over GF(2^q), q <= 8, one warp per received word.
//
// Replaces  cyclic::correct_(b, erasures, hard_decision_tag)   reference codes/cyclic.h:207-252:
//   syndromes  s_j = b(alpha^(root_j))          cyclic.h:53-63 + math/polynomial.h:273-284 (Horner)
//   locator    error_locator_polynomial(...)    codes/hard_decision.h:61-196 (PGZ / BM / Euklid tags,
//              erasure positions folded in as in :127-131 / :171-172)
//   roots      zeroes(sigma) by exhaustive evaluation, #roots must equal deg sigma  cyclic.h:126-150
//   values     1 for binary BCH (codes/bch.h:80-83); for RS the reference solves a linear system
//              (codes/rs.h:41-78) -- here Forney's formula, which yields the same unique values
//   fix-up + re-syndrome check, failure if any syndrome is left   cyclic.h:237-248
// The locator is computed with (errors-and-erasures) Berlekamp-Massey, lane-parallel over the
// coefficients; the reference's three algorithm tags implement the same bounded-distance decoder
// (its own BM has an out-of-bounds read, SURVEY.md fact 8), so results are compared against Euklid.
//
// Work split inside the warp
//   syndromes   lane <-> syndrome index (gf_device.cuh).
//   BM          lane <-> locator coefficient, discrepancy by XOR butterfly.
//   roots       lane <-> codeword position (log/antilog tables in shared memory).
//   Forney      lane <-> error index.
// For RS and erasure-free BCH the re-syndrome check is implied (a locator of degree L <= t with L
// distinct roots reproduces all 2t syndromes, so the corrected word is a codeword; see DESIGN.md)
// and is skipped unless GfDevice::recheck is set; with erasures on a binary code the reference
// flips every erased position (bch.h:80-83), which only the check can validate, so it runs there.
#include <algorithm>
#include <vector>

#include "gf_decode.h"
#include "gf_device.cuh"

namespace ccgpu {

namespace {

constexpr int kGfThreads = 256;
constexpr int kGfWarps = kGfThreads / 32;
constexpr unsigned kAll = kGfAll;
constexpr int kWordBytes = 256;   // per-warp word buffer
constexpr int kWarpBytes = 512;   // word + syndromes + locator + evaluator + positions

struct GfParams {
  int q, n, t, nroots, binary, mu, recheck, max_erasures;
  const uint8_t *tables;
  const uint8_t *words;
  const uint8_t *erasure_pos;  // count x max_erasures (nullable)
  const uint8_t *erasure_cnt;  // count (nullable)
  unsigned long long count;
  uint8_t *corrected, *n_errors, *failed;
};

__global__ void __launch_bounds__(kGfThreads) gf_decode_kernel(const GfParams p) {
  extern __shared__ __align__(16) uint8_t sm[];
  const int size = 1 << p.q, n = p.n;
  const int ntab = (p.nroots + 31) / 32;
  // the table prologue of gf_fill_tables (gf_device.cuh), written out: routing it through that function changes this
  // kernel's instruction schedule
  uint32_t *mtab = reinterpret_cast<uint32_t *>(sm);                    // [ntab][size][32]
  uint8_t *s_exp = sm + size_t(ntab) * size * 32 * sizeof(uint32_t);  // [2*size]
  uint8_t *s_log = s_exp + 2 * size;                                  // [size]
  uint8_t *s_rexp = s_log + size;                                     // [64] root exponents
  uint8_t *per_warp = s_rexp + 64;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint8_t *word = per_warp + warp * kWarpBytes;  // [256], 16-byte aligned
  uint8_t *synd = word + kWordBytes;             // [64]
  uint8_t *lamv = synd + 64;                     // [32] locator coefficients
  uint8_t *llog = lamv + 32;                     // [32] their logarithms (0xff: zero coefficient)
  uint8_t *omega = llog + 32;                    // [32]
  uint8_t *pos = omega + 32;                     // [32] errata positions
  for (int i = threadIdx.x; i < 3 * size; i += blockDim.x) s_exp[i] = p.tables[i];
  if (threadIdx.x < 64) s_rexp[threadIdx.x] = static_cast<uint8_t>(threadIdx.x < p.nroots ? (p.mu + threadIdx.x) % n : 0);
  __syncthreads();
  for (int i = threadIdx.x; i < ntab * size * 32; i += blockDim.x) {
    const int tb = i / (size * 32), x = (i / 32) % size, j = tb * 32 + (i & 31);
    unsigned v = 0;
    if (x && j < p.nroots) v = s_exp[s_log[x] + s_rexp[j]];
    mtab[i] = v;
  }
  __syncthreads();
  const Gf F{ s_exp, s_log };
  const int seg4 = ((n + 15) / 16) * 16;  // bytes of the zero-padded word buffer in use (4 segments)

  const unsigned long long nwarps = static_cast<unsigned long long>(gridDim.x) * kGfWarps;
  for (unsigned long long w = static_cast<unsigned long long>(blockIdx.x) * kGfWarps + warp; w < p.count; w += nwarps) {
    const uint8_t *in = p.words + w * n;
    // the four Horner segments are [c*seg, (c+1)*seg): place symbol i at its natural index, zero the tail
    for (int i = lane; i < seg4; i += 32) word[i] = i < n ? in[i] : 0;
    const int rho = (p.erasure_cnt != nullptr) ? p.erasure_cnt[w] : 0;
    __syncwarp();
    bool failed = false;
    int nerr = 0;
    if (rho > p.max_erasures || rho > 30) {
      failed = true;
    } else if (syndromes(p, F, word, mtab, s_rexp, synd, lane)) {
      // ---------------- erasure locator Gamma(x) = prod (1 + X_e x), coefficient `lane`
      unsigned lam = lane == 0;
      for (int e = 0; e < rho; ++e) {
        const unsigned xe = p.erasure_pos[w * p.max_erasures + e] % n;  // X_e = alpha^position
        const unsigned up = __shfl_up_sync(kAll, lam, 1);
        lam ^= F.mul_alpha(lane ? up : 0u, xe);
      }
      // ---------------- Berlekamp-Massey from r = rho (hard_decision.h:123-152 in exact arithmetic)
      unsigned B = lam;
      int L = rho;
      for (int r = rho; r < p.nroots; ++r) {
        const unsigned bs = __shfl_up_sync(kAll, B, 1);
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
        if (L > 31) break;
      }
      failed = 2 * L > p.nroots + rho || L > 31 || L == 0;
      if (!failed) {
        lamv[lane] = static_cast<uint8_t>(lane <= L ? lam : 0);
        llog[lane] = static_cast<uint8_t>((lane <= L && lam) ? F.log[lam] : 0xff);
        __syncwarp();
        // ---------------- roots: Lambda(alpha^-i) == 0  <=>  errata at position i
        int found = 0;
        for (int i0 = 0; i0 < n; i0 += 32) {
          const int i = i0 + lane;
          unsigned v = 1;  // Lambda_0 = 1
          if (i < n) {
            const unsigned e = i ? n - i : 0;  // exponent of alpha^-i
            unsigned acc = 0;
            for (int k = 1; k <= L; ++k) {
              acc += e;
              if (acc >= static_cast<unsigned>(n)) acc -= n;
              const unsigned lg = llog[k];
              if (lg != 0xff) v ^= F.exp[lg + acc];
            }
          }
          const unsigned hit = __ballot_sync(kAll, i < n && v == 0);
          if (i < n && v == 0) {
            const int slot = found + __popc(hit & ((1u << lane) - 1u));
            if (slot < 32) pos[slot] = static_cast<uint8_t>(i);
          }
          found += __popc(hit);
        }
        __syncwarp();
        failed = found != L;
        if (!failed) {
          nerr = L;
          if (p.binary) {
            if (lane < L) word[pos[lane]] ^= 1;  // bch.h:80-83: every errata value is 1
          } else {
            // ---------------- Forney: Omega = S * Lambda mod x^(2t);  e = X^(1-mu) Omega(1/X) / Lambda'(1/X)
            if (lane < L) {
              unsigned o = 0;
              for (int j = 0; j <= lane; ++j) o ^= F.mul(lamv[j], synd[lane - j]);
              omega[lane] = static_cast<uint8_t>(o);
            }
            __syncwarp();
            if (lane < L) {
              const unsigned pk = pos[lane];
              const unsigned e = pk ? n - pk : 0;  // 1/X = alpha^-pos
              unsigned num = 0, den = 0, acc = 0;  // acc = exponent of (1/X)^k
              for (int k = 0; k < L; ++k) {
                num ^= F.mul_alpha(omega[k], acc);
                if ((k & 1) == 0) den ^= F.mul_alpha(lamv[k + 1], acc);  // Lambda' = sum_{k odd} Lambda_k x^(k-1)
                acc += e;
                if (acc >= static_cast<unsigned>(n)) acc -= n;
              }
              const unsigned xe = (pk * static_cast<unsigned>(((1 - p.mu) % n + n) % n)) % n;  // X^(1-mu)
              unsigned val = 0;
              if (den != 0 && num != 0) val = F.exp[(F.log[num] + n - F.log[den] + xe) % n];
              word[pk] ^= static_cast<uint8_t>(val);
              // a zero value at a non-erased position means the locator is not a true error locator;
              // an erased position may well carry the right symbol (value 0)
              if (val == 0) {
                bool erased = false;
                for (int e2 = 0; e2 < rho; ++e2) erased |= (p.erasure_pos[w * p.max_erasures + e2] % n) == pk;
                failed = !erased;
              }
            }
            failed = __any_sync(kAll, failed);
          }
          __syncwarp();
          // ---------------- cyclic.h:243-248: "Corrected word is not a codeword"
          if (!failed && (p.recheck || (p.binary && rho > 0))) failed = syndromes(p, F, word, mtab, s_rexp, synd, lane);
        }
      }
    }
    uint8_t *out = p.corrected + w * n;
    if (failed) {
      for (int i = lane; i < n; i += 32) out[i] = in[i];
    } else {
      for (int i = lane; i < n; i += 32) out[i] = word[i];
    }
    if (lane == 0) {
      p.failed[w] = failed ? 1 : 0;
      if (p.n_errors) p.n_errors[w] = static_cast<uint8_t>(failed ? 0 : nerr);
    }
    __syncwarp();
  }
}

size_t gf_smem_bytes(const GfDevice &d) { return gf_table_bytes(d.q, d.nroots) + size_t(kGfWarps) * kWarpBytes; }

}  // namespace

int gf_upload(const CodeSpec &spec, GfDevice *out) {
  *out = GfDevice();
  out->q = static_cast<int>(spec.q);
  out->n = static_cast<int>(spec.n);
  out->t = static_cast<int>(spec.t);
  out->nroots = static_cast<int>(spec.roots.size());
  out->binary = spec.family == 0;
  out->mu = spec.family == 0 ? 1 : static_cast<int>(spec.mu);
  out->step = spec.family == 0 ? 1 : static_cast<int>(spec.step);
  const size_t size = spec.F.size;
  std::vector<uint8_t> tab(3 * size);
  for (size_t i = 0; i < 2 * size; ++i) tab[i] = static_cast<uint8_t>(spec.F.exp[i]);
  for (size_t i = 0; i < size; ++i) tab[2 * size + i] = static_cast<uint8_t>(spec.F.log[i]);
  if (cudaMalloc(&out->tables, tab.size()) != cudaSuccess) return -1;
  if (cudaMemcpy(out->tables, tab.data(), tab.size(), cudaMemcpyHostToDevice) != cudaSuccess) return -1;
  return 0;
}

void gf_free(GfDevice *d) {
  if (d->tables) cudaFree(d->tables);
  *d = GfDevice();
}

int gf_launch(const GfDevice &d, const uint8_t *words, uint64_t count, const uint8_t *erasure_pos,
              const uint8_t *erasure_cnt, int max_erasures, uint8_t *corrected, uint8_t *n_errors, uint8_t *failed,
              int sm_count, cudaStream_t stream) {
  if (!d.tables || d.t > 31 || d.nroots > 64 || d.step != 1) return -3;
  GfParams p{ d.q, d.n, d.t, d.nroots, d.binary, d.mu, d.recheck, max_erasures, d.tables, words, erasure_pos, erasure_cnt,
              count, corrected, n_errors, failed };
  const size_t smem = gf_smem_bytes(d);
  if (cudaFuncSetAttribute(gf_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess)
    return -1;
  int occ = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gf_decode_kernel, kGfThreads, smem);
  const uint64_t want = (count + kGfWarps - 1) / kGfWarps;
  const unsigned grid = static_cast<unsigned>(std::min<uint64_t>(want, uint64_t(std::max(1, occ)) * sm_count));
  gf_decode_kernel<<<grid, kGfThreads, smem, stream>>>(p);
  return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

}  // namespace ccgpu
