/* tests/abp_ref.c -- a plain-C restatement of the ABP contract of include/ccgpu.h (ccgpu_decode_llr_abp), fast enough
 * for the full-size pools of tests/test_gpu_abp.py.  It is pinned bit for bit against the numpy restatement there.
 * Build: cc -O2 -ffp-contract=off -shared -fPIC (no FMA contraction: the contract multiplies and adds separately). */
#include <math.h>
#include <stdint.h>
#include <string.h>

#define ABP_B 1048576.0f
#define MAXN 128
#define MAXK 64

static float clamp_b(float v) { return fminf(fmaxf(v, -ABP_B), ABP_B); }

static void one_frame(const uint8_t *H, unsigned k, unsigned n, const float *y, unsigned max_iter, float gamma,
                      uint8_t *bits, float *Lout, uint8_t *iter, uint8_t *failed) {
  float L[MAXN], S[MAXN];
  uint8_t x[MAXN], M[MAXK][MAXN];
  unsigned order[MAXN], pick_row[MAXK];
  for (unsigned c = 0; c < n; ++c) L[c] = isnan(y[c]) ? 0.0f : clamp_b(y[c]);
  for (unsigned j = 0;; ++j) {
    int odd = 0;
    for (unsigned c = 0; c < n; ++c) x[c] = L[c] < 0.0f;
    for (unsigned r = 0; r < k && !odd; ++r) {
      unsigned p = 0;
      for (unsigned c = 0; c < n; ++c) p ^= H[r * n + c] & x[c];
      odd = p;
    }
    if (!odd || j == max_iter) {
      memcpy(bits, x, n);
      if (Lout) memcpy(Lout, L, n * sizeof(float));
      *iter = (uint8_t)j;
      *failed = (uint8_t)odd;
      return;
    }
    /* visiting order: insertion sort on the bits of |L_c|, stable, so ties keep ascending c */
    for (unsigned c = 0; c < n; ++c) {
      uint32_t kc;
      float a = fabsf(L[c]);
      memcpy(&kc, &a, 4);
      unsigned i = c;
      while (i > 0) {
        uint32_t kp;
        float b = fabsf(L[order[i - 1]]);
        memcpy(&kp, &b, 4);
        if (kp <= kc) break;
        order[i] = order[i - 1];
        --i;
      }
      order[i] = c;
    }
    /* Gauss-Jordan in the visiting order: the pivot row of the i-th pick is row i of A */
    uint8_t pivoted[MAXK] = { 0 };
    for (unsigned r = 0; r < k; ++r) memcpy(M[r], H + r * n, n);
    unsigned piv = 0;
    for (unsigned i = 0; i < n && piv < k; ++i) {
      const unsigned c = order[i];
      unsigned r = 0;
      while (r < k && !(M[r][c] && !pivoted[r])) ++r;
      if (r == k) continue;
      for (unsigned r2 = 0; r2 < k; ++r2)
        if (r2 != r && M[r2][c])
          for (unsigned cc = 0; cc < n; ++cc) M[r2][cc] ^= M[r][cc];
      pivoted[r] = 1;
      pick_row[piv++] = r;
    }
    /* check pass: the minimum and the sign parity over the other columns of the row, taken directly */
    for (unsigned c = 0; c < n; ++c) S[c] = 0.0f;
    for (unsigned i = 0; i < k; ++i) {
      const uint8_t *row = M[pick_row[i]];
      for (unsigned c = 0; c < n; ++c) {
        if (!row[c]) continue;
        float mu = INFINITY;
        unsigned s = 0;
        for (unsigned c2 = 0; c2 < n; ++c2) {
          if (!row[c2] || c2 == c) continue;
          if (fabsf(L[c2]) < mu) mu = fabsf(L[c2]);
          s ^= L[c2] < 0.0f;
        }
        if (mu == INFINITY) mu = 0.0f;
        S[c] = S[c] + (s ? -mu : mu);
      }
    }
    for (unsigned c = 0; c < n; ++c) {
      const float t = gamma * S[c];
      L[c] = clamp_b(L[c] + t);
    }
  }
}

/* H: k x n bytes (0/1), y: frames x n; bits frames x n, L (nullable) frames x n, iter and failed frames */
void abp_ref(const uint8_t *H, unsigned k, unsigned n, const float *y, uint64_t frames, unsigned max_iter, float gamma,
             uint8_t *bits, float *L, uint8_t *iter, uint8_t *failed) {
  for (uint64_t f = 0; f < frames; ++f)
    one_frame(H, k, n, y + f * n, max_iter, gamma, bits + f * n, L ? L + f * n : 0, iter + f, failed + f);
}
