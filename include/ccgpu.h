/* ccgpu.h -- C ABI of libccgpu.so, the B200 (sm_100a) engine behind the hot path of
 * hannesweisbach/channelcoding: iterative min-sum-family decoding of binary BCH codes on their
 * parity-check matrix inside an AWGN Monte-Carlo sweep, plus batched GF(2^q) algebraic BCH/RS
 * decoding.  Plain pointers and sizes only; no C++/torch types cross this boundary.
 *
 * The reference has no FFI: its boundary is C++ duck typing (SURVEY.md 8b).  Each entry point
 * below names the reference interface it replaces (paths relative to the reference's src/).
 * INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative ccgpu_status on error; the text of the
 *     last error of a context is available from ccgpu_last_error().  Nothing throws.
 *   - a per-frame decoding failure is DATA (failed[f] = 1), never an error code -- the
 *     reference's `decoding_failure` exception (codes/codes.h:28-36) is a normal outcome that the
 *     simulation counts (simulation/simulation.c++:133-135).
 *   - the caller owns every buffer.  Data pointers may be host or device pointers (detected with
 *     cudaPointerGetAttributes); host buffers are cut into chunks that rotate over three staging slots
 *     (copy in / decode / copy out overlap; pin the host memory to get asynchronous copies) and the
 *     call returns after the results are in the caller's buffer; with device buffers the work is
 *     enqueued on the context's stream and the call returns immediately (ccgpu_sync to wait).
 *   - a context is bound to one CUDA device and one stream and is internally locked, so the
 *     reference's pool threads (simulation/simulation.c++:240-273) may share it.
 *   - there is no CPU fallback: without a usable CUDA device ccgpu_create fails.
 */
#ifndef CCGPU_H
#define CCGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCGPU_ABI_VERSION 2 /* 2: ccgpu_ms_params grew the fixed-point fields; ccgpu_group_*; packed outputs */

typedef struct ccgpu_ctx ccgpu_ctx;
typedef struct ccgpu_code ccgpu_code;

typedef enum {
  CCGPU_OK = 0,
  CCGPU_ERR_INVALID = -1,     /* bad argument */
  CCGPU_ERR_CUDA = -2,        /* CUDA runtime error (text in ccgpu_last_error) */
  CCGPU_ERR_UNSUPPORTED = -3, /* valid request the engine has no kernel for */
  CCGPU_ERR_NO_DEVICE = -4    /* no CUDA device / extension not usable: there is no CPU fallback */
} ccgpu_status;

/* ---- decoder variants: the six soft-decision tags of codes/soft_decision.h:20-73 ------------- */
typedef enum {
  CCGPU_MS = 0,    /* min_sum_tag                  "MS"    soft_decision.h:20-23, :220-226 */
  CCGPU_NMS = 1,   /* normalized_min_sum_tag       "NMS"   :36-42, :228-237   r = alpha * min          */
  CCGPU_OMS = 2,   /* offset_min_sum_tag           "OMS"   :44-50, :239-253   r = max(min - beta, 0) in double */
  CCGPU_SCMS1 = 3, /* self_correcting_1_min_sum_tag "SCMS1" :52-56, :256-268                           */
  CCGPU_SCMS2 = 4, /* self_correcting_2_min_sum_tag "SCMS2" :58-62, :270-282                           */
  CCGPU_NMS2D = 5, /* normalized_2d_min_sum_tag    "2DNMS" :64-73, :284-295   r = alpha*min, q = beta*e + y */
  CCGPU_SPA = 6,   /* sum-product (tanh rule); extension, not in the reference                         */
  /* FIXED-POINT min-sum; extension, not in the reference (its decoders are float32): min_sum__ of
   * soft_decision.h:161-202 with integer messages, restated in oracle/ms_oracle.c (oracle_min_sum_fixed):
   *   y_i = clamp(rint(y * q_scale), -q_y_max, +q_y_max)      float32 product, ties to even, NaN -> 0
   *   q   = (S_c - r) + y_c                                   exact (wide accumulators, :135-136)
   *   r   = sign * fn_h(min(min_{others} |q|, q_msg_max))     three-valued signum as :75-77, :106-118
   *   L_c = S_c + y_c, b_c = L_c < 0, stop rules as for the float variants
   * with fn_h(m) = m (MS_Q), rne(A m / 1024), A = rint(alpha * 1024) (NMS_Q, ties to even),
   * max(m - B, 0), B = rint(beta * q_scale) (OMS_Q).  Hard decisions, iteration indices and failure flags are
   * bit-identical to that restatement; `L` returns the integer totals (units of 1 / q_scale) as floats.
   * The device kernel decodes TWO frames per lane in the 16-bit halves of every register (exact integer
   * arithmetic on the fp16x2 pipe) and therefore needs
   *   max_column_weight * fn_h(q_msg_max) + q_y_max <= 2048,  q_msg_max <= 1023,  alpha <= 1,  B <= 1024;
   * other parameter sets are rejected with CCGPU_ERR_UNSUPPORTED.  Cyclic (BCH) parity-check matrices only. */
  CCGPU_MS_Q = 7,
  CCGPU_NMS_Q = 8,
  CCGPU_OMS_Q = 9
} ccgpu_variant;

/* ---- stop rules (SURVEY.md fact 5) ------------------------------------------------------------ */
typedef enum {
  CCGPU_STOP_REF_ZERO_OVERLAP = 0, /* syndrome(H,b) of soft_decision.h:79-84 as executed: every row's
                                      integer overlap with b is 0 mod 256 (math/matrix.h:57-67)        */
  CCGPU_STOP_GF2_PARITY = 1,       /* H b^T = 0 over GF(2): what a syndrome check means               */
  CCGPU_STOP_NONE = 2              /* run exactly max_iter iterations, never fail (max_iter = 1 gives
                                      the behaviour of the reference's HEAD, math/matrix.h:50)         */
} ccgpu_stop_rule;

typedef struct {
  int32_t variant;    /* ccgpu_variant */
  int32_t stop_rule;  /* ccgpu_stop_rule */
  uint32_t max_iter;  /* template parameter Iterations of the reference's tags (50 in benchmark.c++) */
  uint32_t q_msg_max; /* fixed-point variants: check-node messages saturate at +-q_msg_max; 0 = default 31 */
  double alpha;       /* NMS / 2DNMS scale  (std::ratio parameter of the tag) */
  double beta;        /* OMS offset / 2DNMS variable-node scale; must be >= 0 for OMS */
  double q_scale;     /* fixed-point variants: quantiser steps per unit of y; 0 = default 8 */
  uint32_t q_y_max;   /* fixed-point variants: channel values saturate at +-q_y_max steps; 0 = default 31 */
  uint32_t reserved;
} ccgpu_ms_params;

/* error / iteration counters of one Monte-Carlo batch; all-zero codeword transmitted like
 * simulation.c++:113-131.  frame_errors is the reference's word_errors. */
typedef struct {
  uint64_t frames;
  uint64_t frame_errors; /* decoding failure OR any decided bit != 0 (simulation.c++:126-135) */
  uint64_t bit_errors;   /* decided bits != 0, failures included */
  uint64_t iterations;   /* decoder iterations executed, summed over frames */
  uint64_t failures;     /* decoding_failure (no stop within max_iter) */
  uint64_t undetected;   /* stop test passed on a non-zero word (impossible under REF_ZERO_OVERLAP) */
  uint64_t reserved[2];
} ccgpu_counters;

typedef struct {
  uint32_t family;     /* 0 = binary primitive BCH (codes/bch.h), 1 = RS (codes/rs.h), 2 = from dense H */
  uint32_t q;          /* field GF(2^q) */
  uint32_t n, l, k;    /* length, information symbols l = n - k, k = deg g (cyclic.h:104-105,273) */
  uint32_t dmin;       /* consecutive_zeroes(g) + 1 as computed by cyclic.h:186-204 (sic for RS) */
  uint32_t t;          /* correction_capability (codes.h:15-26) */
  uint32_t h_rows;     /* rows of the parity-check matrix in use */
  uint32_t row_weight; /* max row weight */
  uint32_t edges;      /* ones in H */
  uint32_t h_kind;     /* 0 = cyclic taps without wrap (cyclic.h:346-359), 1 = cyclic with wrap
                          (redundant rows), 2 = general (CSR) */
  uint32_t kernel;     /* 0 = host-only code, 1 = shape-specialised cyclic kernel (ms_cyclic / ms_cyclic_cta),
                          2 = general kernel (ms_csr) */
  double rate;         /* l / n (cyclic.h:274) */
} ccgpu_code_info;

/* ---- context ------------------------------------------------------------------------------------ */
int ccgpu_abi_version(void);
/* device: CUDA ordinal.  Replaces nothing in the reference (it has no device). */
int ccgpu_create(int device, ccgpu_ctx **out);
void ccgpu_destroy(ccgpu_ctx *ctx);
/* text of the context's last error; the pointer stays valid until the calling thread's next call of this function */
const char *ccgpu_last_error(const ccgpu_ctx *ctx);
/* use an existing cudaStream_t (e.g. torch's current stream) instead of the context's own */
int ccgpu_set_stream(ccgpu_ctx *ctx, void *cuda_stream);
void *ccgpu_get_stream(ccgpu_ctx *ctx);
int ccgpu_sync(ccgpu_ctx *ctx);
/* number of engine kernels launched through this context so far */
uint64_t ccgpu_kernel_launches(const ccgpu_ctx *ctx);
/* tuning overrides.  "quick": -1 the library decides per call whether frames with all-positive channel values are
 * retired without iterating (same results either way), 0 / 1 force it off / on -- the parity tests drive both paths
 * with it; "lane": -1 / 1 the n = 15 codes run on the lane-per-frame kernel, 0 on the general warp kernel (same results;
 * the tests compare the two); "work_batch": most frame indices a warp takes from the frame queue per atomic (0 = default).  The
 * environment variables CCGPU_QUICK / CCGPU_WORK_BATCH are read once, at ccgpu_create, as initial values. */
int ccgpu_set_option(ccgpu_ctx *ctx, const char *name, int64_t value);
/* "nvcc <version> sm_100a abi <n>": the toolkit the kernels were compiled with.  The bit-exactness of the ordered
 * column sums rests on properties of the generated code that tests/test_gpu_parity.py re-validates for every
 * compiled shape; a different toolkit must pass them again. */
const char *ccgpu_build_info(void);

/* ---- codes ---------------------------------------------------------------------------------------
 * cyclic::primitive_bch<q, Capability>() -- codes/bch.h:16-161 on top of codes/cyclic.h:67-386.
 * cap_kind 0 = errors<cap_value>, 1 = dmin<cap_value> (codes/codes.h:7-26).  Builds g (lcm of the
 * minimal polynomials of alpha^1, alpha^3, ...), h = (x^n+1)/g, k, l, dmin, rate and the k x n
 * parity-check matrix H() of cyclic.h:346-359, and uploads it.
 * For the three constructors ctx may be NULL: the result is then a host-only description
 * (info / to_string / H / poly / encode work, decoding calls are rejected). */
int ccgpu_bch_create(ccgpu_ctx *ctx, uint32_t q, int cap_kind, uint32_t cap_value, ccgpu_code **out);
/* cyclic::rs<q, errors<t>, Sigma, N, Coding, mu, step>() -- codes/rs.h:6-94. */
int ccgpu_rs_create(ccgpu_ctx *ctx, uint32_t q, uint32_t t, uint32_t mu, uint32_t step, ccgpu_code **out);
/* any dense 0/1 matrix exactly as matrix<uint8_t> from H<T>() / H_alt<T>() (math/matrix.h:11-70),
 * row-major rows x cols.  Cyclic-tap structure is detected; anything else runs on the CSR kernel.
 * rate is used for sigma(Eb/N0) only (simulation.c++:83-85). */
int ccgpu_code_from_dense(ccgpu_ctx *ctx, const uint8_t *H, uint32_t rows, uint32_t cols, double rate,
                          ccgpu_code **out);
/* switch a BCH code to the redundant H with `rows` cyclic shifts of the first row (k <= rows <= n);
 * extension: the reference only builds the k-row H (generate_n(k - 1), cyclic.h:353-356). */
int ccgpu_code_set_rows(ccgpu_code *code, uint32_t rows);
void ccgpu_code_destroy(ccgpu_code *code);
int ccgpu_code_get_info(const ccgpu_code *code, ccgpu_code_info *out);
/* "(n, l, dmin)-TAG" -- cyclic::to_string(), cyclic.h:282-287; it is the log-file name
 * (simulation.c++:98) and parsed by the CLI (benchmark.c++:214-240). */
int ccgpu_code_to_string(const ccgpu_code *code, const char *tag, char *buf, size_t cap);
int ccgpu_code_H(const ccgpu_code *code, uint8_t *out /* h_rows x n */);
/* cyclic::H_alt<T>() -- codes/cyclic.h:361-385, the parity-check matrix from the roots of g(x): t*q rows.
 * as_reference = 1 reproduces the reference bit for bit (its from_power reduces exponents mod 2^q,
 * math/galois.h:182-184, so rows are wrong for exponents >= 2^q); 0 reduces mod n (a valid matrix).
 * out may be NULL to query *rows.  Feed the result to ccgpu_code_from_dense to decode on it. */
int ccgpu_code_H_alt(const ccgpu_code *code, int as_reference, uint8_t *out, uint32_t *rows);
/* which: 0 = g(x), 1 = h(x); coefficients low degree first; returns the count or <0 */
int ccgpu_code_poly(const ccgpu_code *code, int which, uint16_t *out, size_t cap);
/* exp[2*2^q], log[2^q] of math::ef_element<2,q> (math/galois.h:269-301); poly 0 = default table :18-20 */
int ccgpu_gf_tables(uint32_t q, uint32_t poly, uint16_t *exp_out, uint16_t *log_out);
/* cyclic::encode with division_tag (cyclic.h:35-40, :289-311): count x l symbols -> count x n */
int ccgpu_encode(const ccgpu_code *code, const uint8_t *msgs, uint64_t count, uint8_t *words);

/* ---- decoding ----------------------------------------------------------------------------------
 * min_sum<float,uint8_t>(H, y, Tag{}) for `frames` frames -- codes/soft_decision.h:161-202,
 * :220-295, as reached from cyclic::correct_(.., soft_decision_tag) (cyclic.h:254-267) and
 * decoder::correct (simulation/simulation.h:62-65).
 *   y      frames x n   channel values, raw (the reference does not scale to LLRs)
 *   bits   frames x n   hard decision b of the last executed iteration (codes.h:43-52), 0/1
 *   L      frames x n   totals L of that iteration (soft_decision.h:180-182); nullable
 *   iter   frames       0-based iteration index at which the stop test passed
 *                       (std::get<2> of the reference's tuple); max_iter on failure; nullable
 *   failed frames       1 where the reference throws decoding_failure (soft_decision.h:201) */
int ccgpu_decode_llr(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, const float *y,
                     uint64_t frames, uint8_t *bits, float *L, uint8_t *iter, uint8_t *failed);

/* the same decode with a COMPACT output layout (opt-in; the byte-per-bit layout above is what correct() returns,
 * simulation/simulation.h:62-65, this one is what a batch consumer needs): the algorithmic output of SURVEY.md 8(d),
 * 4 * ceil(n/32) bytes of decided bits + one status byte per frame instead of n + 2 bytes.
 *   packed  frames x ceil(n/32) uint32   bit (c & 31) of word (c >> 5) is the decision of column c; unused bits 0
 *   status  frames                       0-based iteration index at which the stop test passed, 255 = decoding_failure
 * (max_iter <= 255, so a passing index is at most 254).  Host or device pointers like ccgpu_decode_llr. */
int ccgpu_decode_llr_packed(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, const float *y,
                            uint64_t frames, uint32_t *packed, uint8_t *status);

/* sigma of simulation.c++:83-85: 1 / sqrt(2 * rate * 10^(ebno_db/10)) */
double ccgpu_sigma(double rate, double ebno_db);
/* Shannon limit Eb/N0 [dB] of the binary-input AWGN channel at `rate` exactly as the reference looks it up: ebno(rate)
 * of simulation.c++:56-70 over its 131-entry table :21-52 (reproduced as data: the first point of every sweep, hence
 * every log file, derives from these numbers).  Pinned on 2028 rates dumped from the reference (tests/golden/shannon.json). */
double ccgpu_shannon_limit_db(double rate);
/* the same limit computed from the capacity of the channel (integral + bisection); a cross-check of the table and the
 * exact figure for rates between its entries.  Not used by the sweep. */
double ccgpu_shannon_limit_db_numeric(double rate);
/* first Eb/N0 point of a sweep, simulation.c++:105-107: (size_t(limit / step) + 1 / step) * step,
 * a negative limit counting as 0 */
double ccgpu_sweep_start_ebno(double rate, double step);
/* frames to simulate at a point given the previous point's word error rate, simulation.c++:91-93:
 * min(cap, 5e3 / wer); cap is 1e6 in the reference */
uint64_t ccgpu_sweep_samples(double previous_wer, uint64_t cap);

/* channel only: y[f][c] = 1 + sigma * z, z ~ N(0,1) from Philox4x32-10 keyed (seed, point),
 * counter (frame0 + f, c / 4)  -- replaces std::generate(b, noise) of simulation.c++:113-115, :125 */
int ccgpu_awgn_llr(ccgpu_ctx *ctx, uint32_t n, double sigma, uint64_t seed, uint32_t point, uint64_t frame0,
                   uint64_t frames, float *y);

/* one Eb/N0 point of awgn_simulation::operator() (simulation.c++:112-149) for global frames
 * [frame0, frame0 + frames): channel + decode + error test fused on chip; only counters leave
 * the GPU.  `out` may be a host or device pointer (device: accumulated into, caller zeroes).
 * The min-sum variants get the raw channel values y like the reference's decoders; for CCGPU_SPA the
 * values are scaled to log-likelihood ratios 2 y / sigma^2 first. */
int ccgpu_awgn_point(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, double ebno_db,
                     uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out);

/* EXTENSION (no reference implementation; BASELINE.json config 3 "multiple-bases parity-check matrices (cyclic-shift
 * rows)"): multiple-bases decoding.  The code is cyclic, so rotating the received word by s positions and decoding on
 * H (codes/cyclic.h:346-359) is decoding the word itself on H rotated the other way: `n_bases` rotations shifts[b] < n
 * give n_bases different parity-check matrices of the same code out of ONE kernel.  Every frame is decoded
 * n_bases times (y_b[c] = y[(c + shifts[b]) mod n], all candidates in one launch of the min-sum kernel with the
 * arithmetic of ccgpu_decode_llr), the candidates are rotated back, and the one with the largest correlation
 * sum_c y[c] (1 - 2 x[c]) (float32, c ascending) among the converged candidates is returned (ties: lowest base);
 * if none converged the frame is reported failed with the best non-converged candidate.  With n_bases = 1 and
 * shifts[0] = 0 the result equals ccgpu_decode_llr.  `iter` is the iteration index of the returned candidate,
 * `chosen` (nullable) the index of its base.  Pinned by tests/test_gpu_parity.py::test_mbbp_* against the CPU oracle
 * run on the rotated words with the same selection rule.  Host or device pointers like ccgpu_decode_llr; binary
 * BCH codes; use the GF(2) stop rule for non-zero codewords. */
int ccgpu_decode_llr_mbbp(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, const uint32_t *shifts,
                          uint32_t n_bases, const float *y, uint64_t frames, uint8_t *bits, float *L, uint8_t *iter,
                          uint8_t *failed, uint8_t *chosen);

/* one Eb/N0 point (frames [frame0, frame0 + frames) of the stream ccgpu_awgn_point draws) decoded with multiple
 * bases: channel kernel -> rotations -> decode -> selection -> counters, everything on the device.  `iterations`
 * counts the iterations executed over ALL bases (the work), the other counters refer to the returned word. */
int ccgpu_awgn_point_mbbp(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, const uint32_t *shifts,
                          uint32_t n_bases, double ebno_db, uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames,
                          ccgpu_counters *out);

/* one Eb/N0 point of awgn_simulation over the reference's `uncoded` pseudo-decoder (codes/uncoded.h:10-47: n symbols,
 * hard decision only, nominal rate 0.5 as in simulation/uncoded.c++:54): channel + decision + error test on the
 * device.  Same noise stream as ccgpu_awgn_point for the same (seed, point, frame).  Only frames, frame_errors and
 * bit_errors are counted. */
int ccgpu_awgn_point_uncoded(ccgpu_ctx *ctx, uint32_t n, double rate, double ebno_db, uint64_t seed, uint32_t point,
                             uint64_t frame0, uint64_t frames, ccgpu_counters *out);

/* the same Eb/N0 point for the HARD-decision tags (BM / PGZ / Euklid decoders of benchmark.c++:29-64 inside
 * awgn_simulation): channel, hard decision (codes/codes.h:43-52: bit = y < 0), algebraic decode
 * (cyclic.h:207-252) and the error test, all on the device; binary BCH codes.  iterations stays 0. */
int ccgpu_awgn_point_hard(ccgpu_ctx *ctx, const ccgpu_code *code, double ebno_db, uint64_t seed, uint32_t point,
                          uint64_t frame0, uint64_t frames, ccgpu_counters *out);

/* EXTENSION (no reference implementation): Chase-II soft-decision decoding of binary primitive BCH codes.  Per frame:
 *   h_c = (y_c < 0) as codes/codes.h:43-52 (0 for -0.0 and NaN);
 *   u_0 .. u_{p-1}: the p columns with the smallest (bits of fabsf(y_c) as uint32, c), ascending (ties: lower column;
 *   NaN sorts above +inf);
 *   test word m (m = 0 .. 2^p - 1) is h with u_j flipped for every set bit j of m, decoded errors-only exactly as
 *   ccgpu_gf_decode decodes it (bounded distance, same failure rules); a success x_m is a candidate;
 *   D_m = sum of fabsf(y_c) over the columns where x_m != h, float32, c ascending, starting from +0.0;
 *   the candidate with the smallest (bits of D_m as uint32, m) is returned.  Without a candidate: failed = 1,
 *   bits = h, chosen = 0.  p = 0 is ccgpu_gf_decode of the hard decision.
 * Binary BCH codes (t <= 31); 0 <= p <= 8 and p <= n.  bits frames x n, failed frames, chosen frames (nullable: index
 * m of the returned test pattern).  Host or device pointers like ccgpu_decode_llr. */
int ccgpu_decode_llr_chase(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t p, const float *y, uint64_t frames,
                           uint8_t *bits, uint8_t *failed, uint8_t *chosen);
/* one Eb/N0 point, frames [frame0, frame0 + frames) of the ccgpu_awgn_point noise stream, decoded with Chase-II on chip;
 * only counters leave (iterations stays 0).  `out` host or device pointer as in ccgpu_awgn_point. */
int ccgpu_awgn_point_chase(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t p, double ebno_db, uint64_t seed,
                           uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out);

/* EXTENSION (no reference implementation): ordered-statistics decoding (Fossorier-Lin OSD-i) of binary primitive BCH
 * codes, a near-maximum-likelihood decoder for short codes.  l information bits, k = n - l rows of the k-row H of
 * ccgpu_code_H at creation (codes/cyclic.h:346-359).  Per frame:
 *   1. h_c = (y_c < 0) as codes/codes.h:43-52 (0 for -0.0 and NaN);
 *   2. the columns are visited in ascending (bits of fabsf(y_c) as uint32, c): ties go to the lower column, NaN sorts
 *      above +inf (the order of ccgpu_decode_llr_chase);
 *   3. P = the columns picked greedily in that order, a column being picked when its H-column is not in the GF(2)
 *      span of the H-columns picked before it (|P| = rank H = k); I = the other l columns.  P depends on the code
 *      only, not on which rows H has, so ccgpu_code_set_rows does not change it; I is the "most reliable basis", the
 *      l columns picked greedily from a generator matrix in the reverse order;
 *   4. with i_0 < .. < i_{l-1} the columns of I, candidate e is the codeword x_e with x_e[I] = h[I] ^ 1_{E_e}; E_0 is
 *      empty, then come the sets {i_a} (a ascending), {i_a, i_b} (a < b, lexicographic) and {i_a, i_b, i_c}
 *      (lexicographic), none heavier than min(order, l): sum over w <= min(order, l) of C(l, w) candidates
 *      (1 / 37 / 667 / 7807 for BCH(63,36));
 *   5. D_e = sum of fabsf(y_c) over the columns where x_e != h, float32, c ascending, starting from +0.0; the winner
 *      is the smallest (K(D_e), e), K = the bits of D_e as uint32 with every NaN counted as 0x7fc00000;
 *   6. bits = x_winner, weight = |E_winner| <= order.  There is no failure: the result is always a codeword.
 * If h is a codeword it is returned with weight 0 (candidate 0 is h with D = +0.0).
 * Binary BCH codes with n <= 127 and k <= 64; 0 <= order <= 3 (order > 3: CCGPU_ERR_INVALID; RS, dense-H codes,
 * n = 255 or k > 64: CCGPU_ERR_UNSUPPORTED).  bits frames x n, weight frames (nullable).  Host or device pointers like
 * ccgpu_decode_llr, all of one kind. */
int ccgpu_decode_llr_osd(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t order, const float *y, uint64_t frames,
                         uint8_t *bits, uint8_t *weight);
/* one Eb/N0 point, frames [frame0, frame0 + frames) of the ccgpu_awgn_point noise stream, decoded with OSD on chip;
 * only counters leave: iterations = failures = 0, undetected = frame_errors.  `out` host or device pointer as in
 * ccgpu_awgn_point. */
int ccgpu_awgn_point_osd(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t order, double ebno_db, uint64_t seed,
                         uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out);

/* EXTENSION (no reference implementation): generalized minimum distance (GMD, Forney) soft-decision decoding of
 * Reed-Solomon codes over the AWGN channel, from the channel values of their binary image.  Symbol c (0 <= c < n) is
 * q bits; bit j of it is image position b = c q + j and equals (s_c >> j) & 1, with the symbol values of ccgpu_encode
 * and ccgpu_gf_decode.  A frame is n q channel values in the raw-y convention of ccgpu_decode_llr.  Per frame:
 *   1. h_b = (y_b < 0) as codes/codes.h:43-52 (0 for -0.0 and NaN); r_c = sum_j h_{cq+j} << j;
 *   2. kappa_c = min_j K(fabsf(y_{cq+j})), K = the bits as uint32 with every NaN counted as 0x7fc00000; the symbols
 *      are ranked in ascending (kappa_c, c);
 *   3. trial i = 0 .. F/2 (F = max_erasures) erases E_i, the first 2i symbols of that ranking, and decodes r with
 *      erasures E_i exactly as ccgpu_gf_decode_erasures would (bounded distance, 2e + 2i <= 2t, same failure rules;
 *      for even erasure counts this is the reference's Euklid decoder, DESIGN.md section 7); a success x_i is a
 *      candidate.  The 30-erasure limit of ccgpu_gf_decode_erasures does not apply: F = 2t = 32 is a pure erasure
 *      decode with 32 erasures;
 *   4. D_i = sum of fabsf(y_b) over the image positions b where the bit of x_i differs from h_b, float32, b ascending,
 *      starting from +0.0;
 *   5. the winner is the smallest (K(D_i), i).  If r is a codeword, trial 0 returns it with D = +0.0 and it wins;
 *   6. words = x_winner; without a candidate failed = 1 and words = r; chosen (nullable) = the winner's i, 0 when the
 *      frame failed.  F = 0 is ccgpu_gf_decode of r.
 * RS codes with 2t <= 32 and step 1 (binary BCH, dense-H codes, 2t > 32: CCGPU_ERR_UNSUPPORTED; F odd or F > 2t:
 * CCGPU_ERR_INVALID).  y frames x (n q), words frames x n, failed and chosen frames.  Host or device pointers like
 * ccgpu_decode_llr, all of one kind. */
int ccgpu_decode_llr_gmd(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t max_erasures, const float *y, uint64_t frames,
                         uint8_t *words, uint8_t *failed, uint8_t *chosen);
/* one Eb/N0 point, decoded with GMD on chip: frame f is what ccgpu_awgn_llr(n q, ccgpu_sigma(l / n, ebno_db), seed,
 * point, frame0, frames) writes for it (the all-zero word sent).  Only counters leave: frame_errors = failed or any
 * decided symbol non-zero, bit_errors = set bits of the decided binary image (r for a failed frame), failures = frames
 * without a candidate, undetected = decoded to a non-zero word, iterations = 0.  `out` host or device pointer as in
 * ccgpu_awgn_point.  With max_erasures = 0 this is the hard-decision RS curve. */
int ccgpu_awgn_point_gmd(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t max_erasures, double ebno_db, uint64_t seed,
                         uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out);

/* EXTENSION (no reference implementation): adaptive belief propagation (ABP, Jiang-Narayanan) of binary primitive BCH
 * codes with the min-sum check pass.  Before every check pass H is reduced so that the k least reliable independent
 * columns have weight one, which keeps errors on unreliable bits out of the short cycles of the dense H.  The k-row H of
 * ccgpu_code_H at creation is always used, whatever ccgpu_code_set_rows selected: the adapted matrix depends only on
 * the row space of H.  Per frame, with B = 2^20 and gamma_f = (float)gamma:
 *   1. L_c = y_c clamped to [-B, B]: NaN becomes +0.0, +-inf becomes +-B (every value is finite from here on);
 *   2. for j = 0, 1, ..: x_c = (L_c < 0); if H x = 0 over GF(2): bits = x, iter = j, failed = 0, stop.  If j = max_iter:
 *      bits = x, iter = max_iter, failed = 1, stop.  Otherwise apply 3-6 once;
 *   3. the columns are visited in ascending (bits of fabsf(L_c) as uint32, c) (the order of ccgpu_decode_llr_osd); P =
 *      p_0, .., p_{k-1} are the first k columns in that order whose H-columns are independent (OSD's step 3);
 *   4. A is the unique k x n matrix with the row space of H and A[:, P] = identity, row i the row with its one among
 *      the P columns at p_i;
 *   5. for each row i and each column c of row i: mu_{i,c} = min over the other columns c' of row i of fabsf(L_c')
 *      (+0.0 for a row of weight 1), s_{i,c} = parity of #{c' != c in row i : L_c' < 0}, m_{i,c} = s ? -mu : mu;
 *      S_c = +0.0 + m_{0,c} + m_{1,c} + .. over the rows holding c in ascending i, float32, no FMA;
 *   6. L_c <- fminf(fmaxf(L_c + gamma_f * S_c, -B), B), the product and the sum each rounded to nearest even.
 * Binary BCH codes with n <= 127 and k <= 64; 0 <= max_iter <= 255 (0: the syndrome check of the hard decision) and a
 * finite 0 < gamma <= 1, else CCGPU_ERR_INVALID; RS, dense-H codes, n = 255 or k > 64: CCGPU_ERR_UNSUPPORTED.  bits
 * frames x n, L (nullable) frames x n final soft values (they can be fed to ccgpu_decode_llr_osd), iter and failed
 * frames.  Host or device pointers like ccgpu_decode_llr, all of one kind. */
int ccgpu_decode_llr_abp(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t max_iter, double gamma, const float *y,
                         uint64_t frames, uint8_t *bits, float *L, uint8_t *iter, uint8_t *failed);
/* one Eb/N0 point, frames [frame0, frame0 + frames) of the ccgpu_awgn_point noise stream (raw y, no LLR scaling),
 * decoded with ABP on chip.  Only counters leave: iterations = sum of the updates applied (iter), failures = frames with
 * failed = 1, frame_errors = failed or any decided bit set, bit_errors = decided bits set, undetected = frames that
 * passed the stop test on a non-zero word.  `out` host or device pointer as in ccgpu_awgn_point. */
int ccgpu_awgn_point_abp(ccgpu_ctx *ctx, const ccgpu_code *code, uint32_t max_iter, double gamma, double ebno_db,
                         uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out);

/* EXTENSION (no reference implementation): maximum-likelihood decoding of high-rate binary primitive BCH codes by a
 * Viterbi search over the syndrome trellis of the k-row H (2^k states, n sections).  It returns a codeword closest to
 * the channel values in the metric of ccgpu_decode_llr_chase / _osd, with no approximation: the exact yardstick of the
 * other soft-decision decoders.  The k-row H of ccgpu_code_H at creation is always used, whatever
 * ccgpu_code_set_rows selected.  Per frame, with sigma_c = sum_r H[r][c] 2^r the k-bit syndrome of column c (never 0
 * for a BCH code):
 *   1. h_c = (y_c < 0) (codes/codes.h:43-52: 0 for -0.0 and NaN);
 *   2. w_c = fminf(fabsf(y_c), 2^20), NaN giving +0.0 (a NaN is an erasure; every w_c is finite);
 *   3. M_0(0) = +0.0, M_0(s) = +inf for s != 0;
 *   4. for c = 0 .. n-1 and every state s in [0, 2^k): the branch x_c = 0 comes from state s with cost [h_c != 0] w_c,
 *      the branch x_c = 1 from state s ^ sigma_c with cost [h_c != 1] w_c; M_{c+1}(s) is the smaller of the two sums
 *      M_c(pred) + cost, each one float32 add rounded to nearest even (no FMA); on equal sums the branch with
 *      x_c = h_c wins; d_c(s) is the x_c of the winning branch;
 *   5. traceback from s = 0: for c = n-1 down to 0: x_c = d_c(s), s ^= x_c sigma_c.  bits = x.
 * x is a codeword, its D (the float32 sum of w_c over the positions where x_c != h_c, c ascending, from +0.0) is M_n(0)
 * and at most the D of every codeword, and a codeword h is returned as it is.  There is no failure.  Binary BCH codes
 * with n <= 127 and 4 <= k <= 12 (BCH(15,11), (15,7), (15,5), (31,26), (31,21), (63,57), (63,51), (127,120)); RS,
 * dense-H codes, n = 255 or k > 12: CCGPU_ERR_UNSUPPORTED.  bits frames x n.  Host or device pointers like
 * ccgpu_decode_llr, all of one kind. */
int ccgpu_decode_llr_ml(ccgpu_ctx *ctx, const ccgpu_code *code, const float *y, uint64_t frames, uint8_t *bits);
/* one Eb/N0 point, frames [frame0, frame0 + frames) of the ccgpu_awgn_point noise stream (raw y, no LLR scaling),
 * decoded with ML on chip.  Only counters leave: frame_errors = frames with any decided bit set, bit_errors = decided
 * bits set, undetected = frame_errors, iterations = failures = 0.  `out` host or device pointer as in
 * ccgpu_awgn_point. */
int ccgpu_awgn_point_ml(ccgpu_ctx *ctx, const ccgpu_code *code, double ebno_db, uint64_t seed, uint32_t point,
                        uint64_t frame0, uint64_t frames, ccgpu_counters *out);

/* one weight class of bitflip_simulation::operator() (simulation.c++:156-213): all C(n, weight)
 * inputs x = -2*bit + 1, decoded and counted; patterns [first, first + count) in the
 * lexicographic order of std::next_permutation (count 0 = all). */
int ccgpu_bitflip_point(ccgpu_ctx *ctx, const ccgpu_code *code, const ccgpu_ms_params *params, uint32_t weight,
                        uint64_t first, uint64_t count, ccgpu_counters *out);

/* cyclic::correct_(.., hard_decision_tag) -- cyclic.h:207-252: syndromes (cyclic.h:53-63), error
 * locator (codes/hard_decision.h:61-196; the engine runs Berlekamp-Massey, which computes the same
 * bounded-distance result as the reference's PGZ/BM/Euklid tags), roots (cyclic.h:126-150), error
 * values (bch.h:80-83 / rs.h:41-78), correction and the re-syndrome check (cyclic.h:237-248).
 *   words     count x n  symbols (uint8)     corrected count x n (received word where failed)
 *   n_errors  count      number of corrected symbols (cyclic.h:237); nullable
 *   failed    count      1 where the reference throws decoding_failure */
int ccgpu_gf_decode(ccgpu_ctx *ctx, const ccgpu_code *code, const uint8_t *words, uint64_t count,
                    uint8_t *corrected, uint8_t *n_errors, uint8_t *failed);
/* the same with erasures -- the `erasures` argument of cyclic::correct (cyclic.h:331-344), folded into
 * the locator as in hard_decision.h:127-131 / :171-172.  Word w has erasure_cnt[w] (<= max_erasures <= 30)
 * erased positions erasure_pos[w * max_erasures + i]; e errors and f erasures are corrected when
 * 2e + f <= 2t.  n_errors counts errors + erasures like cyclic.h:237.  Deviation: with an odd f the
 * reference's Euklid stop rule (hard_decision.h:164: max = (2t + f) / 2, integer) also accepts locators one
 * degree beyond that bound, where the solution is not unique; the engine reports failed = 1 there.
 * For binary BCH the reference
 * flips EVERY erased position (error values are all 1, bch.h:80-83) and relies on the re-syndrome
 * check; the engine reproduces that. */
int ccgpu_gf_decode_erasures(ccgpu_ctx *ctx, const ccgpu_code *code, const uint8_t *words, uint64_t count,
                             const uint8_t *erasure_pos, const uint8_t *erasure_cnt, uint32_t max_erasures,
                             uint8_t *corrected, uint8_t *n_errors, uint8_t *failed);

/* binary BCH with erasures as the reference's PGZ decoder handles them (primitive_bch::correct(b, erasures,
 * peterson_gorenstein_zierler_tag), codes/bch.h:97-149): the erased positions are filled with zeros, then with
 * ones, both words are decoded errors-only (cyclic.h:207-252), and the success that corrected fewer positions is
 * returned (ties: the zero fill); failed = 1 when both fail or when a word has more than 2t erasures (:104-106).
 * erasure_cnt[w] = 0 is plain decoding.  n_errors is the count of the returned candidate (errors in the filled
 * word).  max_erasures <= 255; buffers as in ccgpu_gf_decode_erasures. */
int ccgpu_gf_decode_erasures_pgz(ccgpu_ctx *ctx, const ccgpu_code *code, const uint8_t *words, uint64_t count,
                                 const uint8_t *erasure_pos, const uint8_t *erasure_cnt, uint32_t max_erasures,
                                 uint8_t *corrected, uint8_t *n_errors, uint8_t *failed);
/* 1: always recompute the syndromes of the corrected word (cyclic.h:243-248).  Off by default: for
 * erasure-free words the check is implied by "deg Lambda <= t and deg Lambda distinct roots" (DESIGN.md 4). */
int ccgpu_code_set_recheck(ccgpu_code *code, int enable);

/* ---- device groups: several GPUs of one host behind one handle --------------------------------------------------
 * Replaces nothing in the reference (it has no device); it is where simulation.c++:112-149 decides how much work a
 * point is and waits for its word-error rate (:91-93 sizes the next point from it).  A group owns one context per
 * member device.  A sharded call splits the global unit range [first, first + units) (frames, patterns, words)
 * into contiguous parts, member m running the ordinary single-device entry point on its part from its own host
 * thread and stream, and merges the results inside the library: the eight counters are summed on the host
 * (the noise is keyed by the GLOBAL frame index, so the counters are identical for any number of devices);
 * batched decodes write disjoint slices of the caller's host buffers.  Ranges smaller than
 * ccgpu_group_set_min_frames (default 16384) per member use fewer members.  Codes are per device: `codes[m]` must
 * have been created on ccgpu_group_ctx(group, m) with the same parameters.  One group call runs at a time. */
typedef struct ccgpu_group ccgpu_group;
/* devices == NULL: CUDA ordinals 0 .. n_devices-1 */
int ccgpu_group_create(int n_devices, const int *devices, ccgpu_group **out);
void ccgpu_group_destroy(ccgpu_group *group);
int ccgpu_group_size(const ccgpu_group *group);
ccgpu_ctx *ccgpu_group_ctx(const ccgpu_group *group, int member);
const char *ccgpu_group_last_error(const ccgpu_group *group);
int ccgpu_group_set_min_frames(ccgpu_group *group, uint64_t frames_per_member);
/* the Monte-Carlo points of ccgpu_awgn_point / _hard / _chase / _osd / _gmd / _abp / _ml / _mbbp / _uncoded / ccgpu_bitflip_point, sharded; `out` is a
 * host pointer and holds the merged counters on return */
int ccgpu_group_awgn_point(ccgpu_group *group, ccgpu_code *const *codes, const ccgpu_ms_params *params, double ebno_db,
                           uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out);
int ccgpu_group_awgn_point_hard(ccgpu_group *group, ccgpu_code *const *codes, double ebno_db, uint64_t seed, uint32_t point,
                                uint64_t frame0, uint64_t frames, ccgpu_counters *out);
int ccgpu_group_awgn_point_chase(ccgpu_group *group, ccgpu_code *const *codes, uint32_t p, double ebno_db,
                                 uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out);
int ccgpu_group_awgn_point_osd(ccgpu_group *group, ccgpu_code *const *codes, uint32_t order, double ebno_db,
                               uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out);
int ccgpu_group_awgn_point_gmd(ccgpu_group *group, ccgpu_code *const *codes, uint32_t max_erasures, double ebno_db,
                               uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out);
int ccgpu_group_awgn_point_abp(ccgpu_group *group, ccgpu_code *const *codes, uint32_t max_iter, double gamma,
                               double ebno_db, uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames,
                               ccgpu_counters *out);
int ccgpu_group_awgn_point_ml(ccgpu_group *group, ccgpu_code *const *codes, double ebno_db, uint64_t seed,
                              uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out);
int ccgpu_group_awgn_point_mbbp(ccgpu_group *group, ccgpu_code *const *codes, const ccgpu_ms_params *params,
                                const uint32_t *shifts, uint32_t n_bases, double ebno_db, uint64_t seed, uint32_t point,
                                uint64_t frame0, uint64_t frames, ccgpu_counters *out);
int ccgpu_group_awgn_point_uncoded(ccgpu_group *group, uint32_t n, double rate, double ebno_db, uint64_t seed, uint32_t point,
                                   uint64_t frame0, uint64_t frames, ccgpu_counters *out);
int ccgpu_group_bitflip_point(ccgpu_group *group, ccgpu_code *const *codes, const ccgpu_ms_params *params, uint32_t weight,
                              uint64_t first, uint64_t count, ccgpu_counters *out);
/* ccgpu_decode_llr / ccgpu_gf_decode with HOST buffers, frames / words sharded over the members */
int ccgpu_group_decode_llr(ccgpu_group *group, ccgpu_code *const *codes, const ccgpu_ms_params *params, const float *y,
                           uint64_t frames, uint8_t *bits, float *L, uint8_t *iter, uint8_t *failed);
int ccgpu_group_gf_decode(ccgpu_group *group, ccgpu_code *const *codes, const uint8_t *words, uint64_t count,
                          uint8_t *corrected, uint8_t *n_errors, uint8_t *failed);

#ifdef __cplusplus
}
#endif
#endif /* CCGPU_H */
