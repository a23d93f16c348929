// cc/codes.h -- C++ host layer over the C ABI (ccgpu.h) that mirrors the reference's code types,
// so that a program written against hannesweisbach/channelcoding keeps its shape:
//
//   reference (src/)                                   this header
//   ------------------------------------------------   -------------------------------------------
//   errors<e>, dmin<d>, correction_capability          same names                     codes/codes.h:7-26
//   decoding_failure : std::runtime_error              same                           codes/codes.h:28-36
//   min_sum_tag<I>, normalized_min_sum_tag<I,R>, ...   same names, same to_string()   codes/soft_decision.h:20-73
//   cyclic::berlekamp_massey_tag / euklid_tag / PGZ    same names, same to_string()   codes/hard_decision.h:15-24
//   cyclic::primitive_bch<q, Capability, Tag>          cc::primitive_bch<q, Capability, Tag>   codes/bch.h:16-161
//   cyclic::rs<q, Capability, Tag>                     cc::rs<q, Capability, Tag>              codes/rs.h:6-94
//   (extension) Chase-II                               cc::primitive_bch<q, Capability, chase_tag<P> >
//   (extension) ordered-statistics decoding            cc::primitive_bch<q, Capability, osd_tag<Order> >
//   (extension) GMD decoding of RS codes               cc::rs<q, Capability, gmd_tag<F> >
//   (extension) adaptive belief propagation            cc::primitive_bch<q, Capability, abp_tag<Iterations, Gamma> >
//   (extension) maximum-likelihood (Viterbi) decoding  cc::primitive_bch<q, Capability, ml_tag>
//     .correct<R>(vector<float|uint>)  .to_string()  .rate  ::n  ::t  .H<T>()           codes/cyclic.h:282-359
//
// Differences a user sees: every object holds a ccgpu context/code handle (one GPU, or every GPU of the current
// cc::device_group -- Monte-Carlo points and batched decodes are then sharded over them), and there are
// batched entry points (correct_batch, awgn_point, bitflip_point) next to the single-frame
// `correct`, which is kept for drop-in compatibility (it costs a kernel launch per frame).
// All arithmetic runs in the CUDA kernels of libccgpu.so; this header only marshals.
#pragma once
#include <cstdint>
#include <memory>
#include <mutex>
#include <ratio>
#include <stdexcept>
#include <string>
#include <type_traits>
#include <vector>

#include "../ccgpu.h"

namespace cc {

// ---- codes/codes.h -------------------------------------------------------------------------------
template <unsigned e> struct errors { static constexpr unsigned value = e; };
template <unsigned d> struct dmin { static constexpr unsigned value = d; };
template <typename T> struct correction_capability;
template <unsigned v> struct correction_capability<dmin<v> > {
  static constexpr unsigned value = (v - 1) / 2;
  static constexpr int kind = 1;
  static constexpr unsigned raw = v;
};
template <unsigned v> struct correction_capability<errors<v> > {
  static constexpr unsigned value = v;
  static constexpr int kind = 0;
  static constexpr unsigned raw = v;
};

class decoding_failure : public std::runtime_error {
public:
  using std::runtime_error::runtime_error;
};

struct algorithm_tag {};
struct hard_decision_tag : algorithm_tag {};
struct soft_decision_tag : algorithm_tag {};

// ---- codes/soft_decision.h:20-73 -----------------------------------------------------------------
template <unsigned Iterations = 50> struct min_sum_tag : soft_decision_tag {
  static constexpr unsigned iterations = Iterations;
  static constexpr int variant = CCGPU_MS;
  static constexpr double alpha = 1.0, beta = 0.0;
  static std::string to_string() { return "MS"; }
};
template <unsigned Iterations, typename T = std::ratio<1> > struct normalized_min_sum_tag : soft_decision_tag {
  static constexpr unsigned iterations = Iterations;
  static constexpr int variant = CCGPU_NMS;
  static constexpr double alpha = static_cast<double>(T::num) / T::den, beta = 0.0;
  static std::string to_string() { return "NMS"; }
};
template <unsigned Iterations = 50, typename T = std::ratio<0> > struct offset_min_sum_tag : soft_decision_tag {
  static constexpr unsigned iterations = Iterations;
  static constexpr int variant = CCGPU_OMS;
  static constexpr double alpha = 1.0, beta = static_cast<double>(T::num) / T::den;
  static std::string to_string() { return "OMS"; }
};
template <unsigned Iterations = 50> struct self_correcting_1_min_sum_tag : soft_decision_tag {
  static constexpr unsigned iterations = Iterations;
  static constexpr int variant = CCGPU_SCMS1;
  static constexpr double alpha = 1.0, beta = 0.0;
  static std::string to_string() { return "SCMS1"; }
};
template <unsigned Iterations = 50> struct self_correcting_2_min_sum_tag : soft_decision_tag {
  static constexpr unsigned iterations = Iterations;
  static constexpr int variant = CCGPU_SCMS2;
  static constexpr double alpha = 1.0, beta = 0.0;
  static std::string to_string() { return "SCMS2"; }
};
// The reference computes beta = Beta::num / Alpha::den (soft_decision.h:71, on reduced ratios), so
// its default <50> is alpha = beta = 1.  `reference_beta` reproduces that; `beta` is the intended
// Beta::num / Beta::den.  primitive_bch uses reference_beta to stay bit-compatible.
template <unsigned Iterations = 50, typename Alpha = std::ratio<1>, typename Beta = std::ratio<1, 10> >
struct normalized_2d_min_sum_tag : soft_decision_tag {
  static constexpr unsigned iterations = Iterations;
  static constexpr int variant = CCGPU_NMS2D;
  static constexpr double alpha = static_cast<double>(Alpha::num) / Alpha::den;
  static constexpr double intended_beta = static_cast<double>(Beta::num) / Beta::den;
  static constexpr double beta = static_cast<double>(Beta::num) / Alpha::den;  // sic, as the reference
  static std::string to_string() { return "2DNMS"; }
};
// extension: sum-product (tanh rule); inputs must be LLRs (2 y / sigma^2)
template <unsigned Iterations = 50> struct sum_product_tag : soft_decision_tag {
  static constexpr unsigned iterations = Iterations;
  static constexpr int variant = CCGPU_SPA;
  static constexpr double alpha = 1.0, beta = 0.0;
  static std::string to_string() { return "SPA"; }
};

// extension (north_star "fixed-point min-sum"; CCGPU_MS_Q / NMS_Q / OMS_Q of ccgpu.h): the same loop with integer
// messages.  Quant = fixed_point<scale, y_max, msg_max>: y_int = clamp(rint(y * scale), +-y_max), check-node messages
// saturate at msg_max.  Two frames per GPU lane: about twice the edge throughput of the float tags.
template <unsigned Scale = 8, unsigned YMax = 31, unsigned MsgMax = 31> struct fixed_point {
  static constexpr double scale = Scale;
  static constexpr unsigned y_max = YMax, msg_max = MsgMax;
};
struct fixed_point_tag {};
template <unsigned Iterations = 50, typename Quant = fixed_point<> > struct fixed_min_sum_tag : soft_decision_tag, fixed_point_tag {
  using quant = Quant;
  static constexpr unsigned iterations = Iterations;
  static constexpr int variant = CCGPU_MS_Q;
  static constexpr double alpha = 1.0, beta = 0.0;
  static std::string to_string() { return "MSQ"; }
};
template <unsigned Iterations, typename T = std::ratio<1>, typename Quant = fixed_point<> >
struct fixed_normalized_min_sum_tag : soft_decision_tag, fixed_point_tag {
  using quant = Quant;
  static constexpr unsigned iterations = Iterations;
  static constexpr int variant = CCGPU_NMS_Q;
  static constexpr double alpha = static_cast<double>(T::num) / T::den, beta = 0.0;
  static std::string to_string() { return "NMSQ"; }
};
template <unsigned Iterations = 50, typename T = std::ratio<0>, typename Quant = fixed_point<> >
struct fixed_offset_min_sum_tag : soft_decision_tag, fixed_point_tag {
  using quant = Quant;
  static constexpr unsigned iterations = Iterations;
  static constexpr int variant = CCGPU_OMS_Q;
  static constexpr double alpha = 1.0, beta = static_cast<double>(T::num) / T::den;
  static std::string to_string() { return "OMSQ"; }
};

// ---- codes/hard_decision.h:15-24 -----------------------------------------------------------------
struct peterson_gorenstein_zierler_tag : hard_decision_tag { static std::string to_string() { return "PGZ"; } };
struct berlekamp_massey_tag : hard_decision_tag { static std::string to_string() { return "BM"; } };
struct euklid_tag : hard_decision_tag { static std::string to_string() { return "EUKLID"; } };

// ---- extension: Chase-II (ccgpu_decode_llr_chase).  The hard decision plus 2^P test patterns over the P least reliable
// positions, each decoded algebraically, the candidate closest to the channel values wins.  Neither a soft-decision
// (min-sum) nor a hard-decision tag: it takes channel values and decodes algebraically.
template <unsigned P> struct chase_tag : algorithm_tag {
  static_assert(P <= 8, "Chase-II takes at most 8 test positions");
  static constexpr unsigned p = P;
  static std::string to_string() { return "CHASE" + std::to_string(P); }
};
template <typename Tag> struct is_chase_tag : std::false_type {};
template <unsigned P> struct is_chase_tag<chase_tag<P> > : std::true_type {};

// ---- extension: ordered-statistics decoding OSD-i (ccgpu_decode_llr_osd).  Re-encodes the most reliable basis of the
// channel values with up to Order of its positions flipped; the candidate closest to the channel values wins.  Like
// Chase-II it takes channel values and is neither a soft-decision (min-sum) nor a hard-decision tag.
template <unsigned Order> struct osd_tag : algorithm_tag {
  static_assert(Order <= 3, "OSD takes order 0 .. 3");
  static constexpr unsigned order = Order;
  static std::string to_string() { return "OSD" + std::to_string(Order); }
};
template <typename Tag> struct is_osd_tag : std::false_type {};
template <unsigned Order> struct is_osd_tag<osd_tag<Order> > : std::true_type {};

// ---- extension: generalized minimum distance decoding of Reed-Solomon codes (ccgpu_decode_llr_gmd).  Takes the
// channel values of the binary image (n q per word), erases the 0, 2, .., F least reliable symbols in turn, decodes each
// trial with errors and erasures, and returns the candidate closest to the channel values.  F = 0 is hard-decision
// decoding.  Like Chase-II it is neither a soft-decision (min-sum) nor a hard-decision tag.
template <unsigned F> struct gmd_tag : algorithm_tag {
  static_assert(F % 2 == 0, "GMD erases symbols in pairs: F must be even");
  static constexpr unsigned max_erasures = F;
  static std::string to_string() { return "GMD" + std::to_string(F); }
};
template <typename Tag> struct is_gmd_tag : std::false_type {};
template <unsigned F> struct is_gmd_tag<gmd_tag<F> > : std::true_type {};

// ---- extension: adaptive belief propagation (ccgpu_decode_llr_abp).  Before each of at most Iterations min-sum check
// passes, H is reduced so that its least reliable independent columns have weight one; the soft values are updated
// with the damping factor Gamma (a std::ratio, 0 < Gamma <= 1).  It takes channel values but is not one of the min-sum
// variants of soft_decision_tag: it has its own entry points.
template <unsigned Iterations, typename Gamma = std::ratio<15, 100> > struct abp_tag : algorithm_tag {
  static_assert(Iterations <= 255, "ABP takes at most 255 iterations");
  static_assert(Gamma::num > 0 && Gamma::num <= Gamma::den, "ABP takes a damping factor 0 < Gamma <= 1");
  static constexpr unsigned iterations = Iterations;
  static constexpr double gamma = static_cast<double>(Gamma::num) / Gamma::den;
  static std::string to_string() { return "ABP" + std::to_string(Iterations); }
};
template <typename Tag> struct is_abp_tag : std::false_type {};
template <unsigned I, typename G> struct is_abp_tag<abp_tag<I, G> > : std::true_type {};

// ---- extension: maximum-likelihood decoding (ccgpu_decode_llr_ml).  A Viterbi search over the syndrome trellis of the
// k-row H returns a codeword closest to the channel values; high-rate codes only (n - l <= 12).  Like Chase-II it takes
// channel values and is neither a soft-decision (min-sum) nor a hard-decision tag.
struct ml_tag : algorithm_tag {
  static std::string to_string() { return "ML"; }
};
template <typename Tag> struct is_ml_tag : std::false_type {};
template <> struct is_ml_tag<ml_tag> : std::true_type {};

// ---- one GPU context shared by every code object of the process (per device) ------------------------
class gpu_error : public std::runtime_error {
public:
  using std::runtime_error::runtime_error;
};

enum class stop_rule : int {
  reference = CCGPU_STOP_REF_ZERO_OVERLAP,  // what the reference executes (SURVEY.md fact 5)
  gf2_parity = CCGPU_STOP_GF2_PARITY,
  none = CCGPU_STOP_NONE
};

// process-wide defaults picked up by code objects at construction (the reference's programs build their decoders
// as globals / in a catalogue, so a command-line flag has to act before that): the CUDA device of objects
// constructed without an explicit one, and the stop rule of soft decoders
namespace detail {
inline int &default_device_ref() {
  static int d = 0;
  return d;
}
inline stop_rule &default_stop_ref() {
  static stop_rule s = stop_rule::reference;
  return s;
}
}  // namespace detail
inline void set_default_device(int device) { detail::default_device_ref() = device; }
inline void set_default_stop_rule(stop_rule s) { detail::default_stop_ref() = s; }

class context {
  ccgpu_ctx *ctx_ = nullptr;
  bool owned_ = true;

public:
  explicit context(int device = 0) {
    if (ccgpu_create(device, &ctx_) != CCGPU_OK)
      throw gpu_error("ccgpu_create failed: no usable CUDA device (there is no CPU fallback)");
  }
  explicit context(ccgpu_ctx *borrowed) : ctx_(borrowed), owned_(false) {}  // a member of a device_group
  ~context() {
    if (owned_) ccgpu_destroy(ctx_);
  }
  context(const context &) = delete;
  context &operator=(const context &) = delete;
  ccgpu_ctx *get() const { return ctx_; }
  void check(int rc) const {
    if (rc != CCGPU_OK) throw gpu_error(std::string("ccgpu: ") + ccgpu_last_error(ctx_));
  }
  static std::shared_ptr<context> shared(int device = 0) {
    static std::mutex m;
    static std::shared_ptr<context> inst[16];
    std::lock_guard<std::mutex> g(m);
    if (!inst[device & 15]) inst[device & 15] = std::make_shared<context>(device);
    return inst[device & 15];
  }
};

// several GPUs of this host behind one handle (ccgpu_group): Monte-Carlo points and batched decodes of code objects
// created while a group is current are sharded over its devices, the counters are merged inside the library
// (identical to the one-GPU result: the noise is keyed by the global frame index).
//   cc::device_group::use(8);   // before the decoders are constructed; use(1) goes back to one device
class device_group {
  ccgpu_group *g_ = nullptr;

public:
  explicit device_group(int n_gpus, int first_device = 0) {
    std::vector<int> devs(static_cast<size_t>(n_gpus));
    for (int i = 0; i < n_gpus; ++i) devs[static_cast<size_t>(i)] = first_device + i;
    if (ccgpu_group_create(n_gpus, devs.data(), &g_) != CCGPU_OK)
      throw gpu_error("ccgpu_group_create failed: not enough usable CUDA devices");
  }
  // any list of CUDA ordinals; an ordinal may repeat (several members on one device: same results, used by the tests)
  explicit device_group(const std::vector<int> &devices) {
    if (ccgpu_group_create(static_cast<int>(devices.size()), devices.data(), &g_) != CCGPU_OK)
      throw gpu_error("ccgpu_group_create failed: not enough usable CUDA devices");
  }
  ~device_group() { ccgpu_group_destroy(g_); }
  device_group(const device_group &) = delete;
  device_group &operator=(const device_group &) = delete;
  ccgpu_group *get() const { return g_; }
  int size() const { return ccgpu_group_size(g_); }
  ccgpu_ctx *ctx(int member) const { return ccgpu_group_ctx(g_, member); }
  void check(int rc) const {
    if (rc != CCGPU_OK) throw gpu_error(std::string("ccgpu group: ") + ccgpu_group_last_error(g_));
  }
  static std::shared_ptr<device_group> &current() {
    static std::shared_ptr<device_group> g;
    return g;
  }
  static void use(int n_gpus, int first_device = 0) {
    current() = n_gpus > 1 ? std::make_shared<device_group>(n_gpus, first_device) : nullptr;
  }
  static void use(const std::vector<int> &devices) {
    current() = devices.empty() ? nullptr : std::make_shared<device_group>(devices);
  }
};

namespace detail {

struct code_handle {
  std::shared_ptr<device_group> grp;  // set when the code lives on every member of a group
  std::shared_ptr<context> ctx;       // the (first) device's context
  ccgpu_code *code = nullptr;         // == codes[0]
  std::vector<ccgpu_code *> codes;    // one per group member (one entry without a group)
  ccgpu_code_info info{};
  ~code_handle() {
    for (ccgpu_code *c : codes) ccgpu_code_destroy(c);
  }
  // creates the code through `create(ctx, &code)` on the current group's members, else on `device`
  template <typename Create> static std::shared_ptr<code_handle> make(int device, Create create) {
    auto h = std::make_shared<code_handle>();
    h->grp = device_group::current();
    if (h->grp) {
      h->ctx = std::make_shared<context>(h->grp->ctx(0));
      for (int m = 0; m < h->grp->size(); ++m) {
        ccgpu_code *c = nullptr;
        if (create(h->grp->ctx(m), &c) != CCGPU_OK) throw gpu_error(std::string("ccgpu: ") + ccgpu_last_error(h->grp->ctx(m)));
        h->codes.push_back(c);
      }
    } else {
      h->ctx = context::shared(device < 0 ? default_device_ref() : device);
      ccgpu_code *c = nullptr;
      h->ctx->check(create(h->ctx->get(), &c));
      h->codes.push_back(c);
    }
    h->code = h->codes[0];
    h->ctx->check(ccgpu_code_get_info(h->code, &h->info));
    return h;
  }
};

template <typename Tag, bool soft = std::is_base_of<soft_decision_tag, Tag>::value> struct params_of {
  static ccgpu_ms_params get(stop_rule) { return ccgpu_ms_params{}; }
};
template <typename Tag> struct params_of<Tag, true> {
  static ccgpu_ms_params get(stop_rule s) {
    ccgpu_ms_params p{};
    p.variant = Tag::variant;
    p.stop_rule = static_cast<int>(s);
    p.max_iter = Tag::iterations;
    p.alpha = Tag::alpha;
    p.beta = Tag::beta;
    set_quant(p, std::is_base_of<fixed_point_tag, Tag>());
    return p;
  }
  static void set_quant(ccgpu_ms_params &, std::false_type) {}
  template <typename U = Tag> static void set_quant(ccgpu_ms_params &p, std::true_type) {
    p.q_scale = U::quant::scale;
    p.q_y_max = U::quant::y_max;
    p.q_msg_max = U::quant::msg_max;
  }
};

}  // namespace detail

// common part of primitive_bch / rs: cyclic::cyclic<...> of codes/cyclic.h:67-386
template <typename Algorithm> class cyclic_base {
  static_assert(std::is_base_of<algorithm_tag, Algorithm>::value, "Algorithm must be a decoder tag");

protected:
  std::shared_ptr<detail::code_handle> h_;
  stop_rule stop_ = detail::default_stop_ref();

  explicit cyclic_base(std::shared_ptr<detail::code_handle> h) : h_(std::move(h)), rate(h_->info.rate) {}

public:
  const double rate;  // public data member like cyclic.h:111
  static constexpr bool soft_tag = std::is_base_of<soft_decision_tag, Algorithm>::value;
  static constexpr bool chase = is_chase_tag<Algorithm>::value;
  static constexpr bool osd = is_osd_tag<Algorithm>::value;
  static constexpr bool gmd = is_gmd_tag<Algorithm>::value;
  static constexpr bool abp = is_abp_tag<Algorithm>::value;
  static constexpr bool ml = is_ml_tag<Algorithm>::value;

  std::string to_string() const {  // cyclic.h:282-287
    char buf[96];
    h_->ctx->check(ccgpu_code_to_string(h_->code, Algorithm::to_string().c_str(), buf, sizeof(buf)));
    return buf;
  }
  const ccgpu_code_info &info() const { return h_->info; }
  ccgpu_code *handle() const { return h_->code; }
  const std::shared_ptr<context> &ctx() const { return h_->ctx; }
  void set_stop_rule(stop_rule s) { stop_ = s; }
  ccgpu_ms_params ms_params() const { return detail::params_of<Algorithm>::get(stop_); }

  // matrix<T> H<T>() of cyclic.h:346-359 as rows of a vector-of-vectors
  template <typename T> std::vector<std::vector<T> > H() const {
    std::vector<uint8_t> flat(static_cast<size_t>(h_->info.h_rows) * h_->info.n);
    h_->ctx->check(ccgpu_code_H(h_->code, flat.data()));
    std::vector<std::vector<T> > m(h_->info.h_rows, std::vector<T>(h_->info.n));
    for (unsigned r = 0; r < h_->info.h_rows; ++r)
      for (unsigned c = 0; c < h_->info.n; ++c) m[r][c] = T(flat[static_cast<size_t>(r) * h_->info.n + c]);
    return m;
  }

  // ---- batched soft decoding: frames x n channel values -> frames x n bits; failed[f] = 1 where the
  // reference would throw decoding_failure (soft_decision.h:201)
  void correct_batch(const float *y, uint64_t frames, uint8_t *bits, uint8_t *failed, uint8_t *iter = nullptr,
                     float *L = nullptr) const {
    static_assert(std::is_base_of<soft_decision_tag, Algorithm>::value, "soft-decision tag required");
    const ccgpu_ms_params p = ms_params();
    if (h_->grp)  // host buffers, frames sharded over the group's devices
      h_->grp->check(ccgpu_group_decode_llr(h_->grp->get(), h_->codes.data(), &p, y, frames, bits, L, iter, failed));
    else
      h_->ctx->check(ccgpu_decode_llr(h_->ctx->get(), h_->code, &p, y, frames, bits, L, iter, failed));
  }
  // ---- extension: multiple-bases decoding (ccgpu_decode_llr_mbbp): every frame is decoded on H rotated by each
  // of `rotations` and the best converged candidate is kept; chosen[f] (optional) is the index of its rotation
  void correct_batch_multiple_bases(const float *y, uint64_t frames, const std::vector<uint32_t> &rotations, uint8_t *bits,
                                    uint8_t *failed, uint8_t *iter = nullptr, float *L = nullptr,
                                    uint8_t *chosen = nullptr) const {
    static_assert(std::is_base_of<soft_decision_tag, Algorithm>::value, "soft-decision tag required");
    const ccgpu_ms_params p = ms_params();
    h_->ctx->check(ccgpu_decode_llr_mbbp(h_->ctx->get(), h_->code, &p, rotations.data(),
                                         static_cast<uint32_t>(rotations.size()), y, frames, bits, L, iter, failed, chosen));
  }
  // ---- batched algebraic decoding: count x n symbols
  void correct_batch(const uint8_t *words, uint64_t count, uint8_t *corrected, uint8_t *failed,
                     uint8_t *n_errors = nullptr) const {
    if (h_->grp)
      h_->grp->check(ccgpu_group_gf_decode(h_->grp->get(), h_->codes.data(), words, count, corrected, n_errors, failed));
    else
      h_->ctx->check(ccgpu_gf_decode(h_->ctx->get(), h_->code, words, count, corrected, n_errors, failed));
  }

  // ---- the reference's single-word entry point (cyclic.h:331-344): soft tags take channel values,
  // hard tags take symbols (or signed values that are hard-decided first, cyclic.h:163-171)
  template <typename Return_type = uint8_t, typename InputSequence>
  std::vector<Return_type> correct(const InputSequence &b) const {
    const unsigned n = h_->info.n;
    if (b.size() != n)
      throw std::runtime_error("Channel code word has the wrong size (" + std::to_string(b.size()) + "). Expected " +
                               std::to_string(n));
    std::vector<uint8_t> out(n);
    uint8_t failed = 0;
    correct_one(b, out.data(), &failed, std::is_base_of<soft_decision_tag, Algorithm>());
    if (failed) throw decoding_failure("Decoding failure");
    std::vector<Return_type> r;
    r.reserve(n);
    for (uint8_t v : out) r.push_back(Return_type(v));
    return r;
  }

  // ---- correct(b, erasures) of cyclic.h:331-344.  Soft tags: the channel value of every erased position is
  // set to 0 before decoding (cyclic.h:261-262).  Hard tags: errors-and-erasures decoding
  // (hard_decision.h:127-131 / :171-172) -- at most 30 erasures per word.
  template <typename Return_type = uint8_t, typename InputSequence>
  std::vector<Return_type> correct(const InputSequence &b, const std::vector<unsigned> &erasures) const {
    if (erasures.empty()) return correct<Return_type>(b);
    const unsigned n = h_->info.n;
    if (b.size() != n)
      throw std::runtime_error("Channel code word has the wrong size (" + std::to_string(b.size()) + "). Expected " +
                               std::to_string(n));
    std::vector<uint8_t> out(n);
    uint8_t failed = 0;
    correct_erased(b, erasures, out.data(), &failed, std::is_base_of<soft_decision_tag, Algorithm>());
    if (failed) throw decoding_failure("Decoding failure");
    std::vector<Return_type> r;
    r.reserve(n);
    for (uint8_t v : out) r.push_back(Return_type(v));
    return r;
  }

  // ---- one Eb/N0 point of awgn_simulation (simulation.c++:112-149), fused on the GPU
  // (frames are sharded over the devices of the group the code was created under, if any)
  ccgpu_counters awgn_point(double ebno_db, uint64_t frames, uint64_t seed = 0, uint32_t point = 0,
                            uint64_t frame0 = 0) const {
    const ccgpu_ms_params p = ms_params();
    ccgpu_counters c{};
    if (h_->grp)
      h_->grp->check(ccgpu_group_awgn_point(h_->grp->get(), h_->codes.data(), &p, ebno_db, seed, point, frame0, frames, &c));
    else
      h_->ctx->check(ccgpu_awgn_point(h_->ctx->get(), h_->code, &p, ebno_db, seed, point, frame0, frames, &c));
    return c;
  }
  // ---- the same point for a hard-decision tag: channel, hard decision (codes.h:43-52), algebraic decode and the
  // error test of simulation.c++:126-135 on the device
  ccgpu_counters awgn_point_hard(double ebno_db, uint64_t frames, uint64_t seed = 0, uint32_t point = 0,
                                 uint64_t frame0 = 0) const {
    ccgpu_counters c{};
    if (h_->grp)
      h_->grp->check(ccgpu_group_awgn_point_hard(h_->grp->get(), h_->codes.data(), ebno_db, seed, point, frame0, frames, &c));
    else
      h_->ctx->check(ccgpu_awgn_point_hard(h_->ctx->get(), h_->code, ebno_db, seed, point, frame0, frames, &c));
    return c;
  }
  // ---- one weight of bitflip_simulation (simulation.c++:156-213)
  ccgpu_counters bitflip_point(unsigned weight) const {
    const ccgpu_ms_params p = ms_params();
    ccgpu_counters c{};
    if (h_->grp)
      h_->grp->check(ccgpu_group_bitflip_point(h_->grp->get(), h_->codes.data(), &p, weight, 0, 0, &c));
    else
      h_->ctx->check(ccgpu_bitflip_point(h_->ctx->get(), h_->code, &p, weight, 0, 0, &c));
    return c;
  }

private:
  template <typename In>
  void correct_erased(const In &b, const std::vector<unsigned> &er, uint8_t *out, uint8_t *failed, std::true_type) const {
    std::vector<float> y(b.begin(), b.end());
    for (unsigned e : er) y.at(e) = 0.0f;
    correct_batch(y.data(), 1, out, failed);
  }
  template <typename In>
  void correct_erased(const In &b, const std::vector<unsigned> &er, uint8_t *out, uint8_t *failed, std::false_type) const {
    std::vector<uint8_t> w, pos(30, 0);
    for (const auto &e : b) w.push_back(std::is_signed<typename In::value_type>::value ? (e < 0 ? 1 : 0) : static_cast<uint8_t>(e));
    if (std::is_same<Algorithm, peterson_gorenstein_zierler_tag>::value && h_->info.family == 0) {
      // binary BCH + PGZ: the reference fills the erasures with zeros, then ones, and keeps the better decode (bch.h:97-149)
      if (er.size() > 255) throw decoding_failure("Number of erasures exceed error correction capability.");
      pos.assign(er.size(), 0);
      for (size_t i = 0; i < er.size(); ++i) pos[i] = static_cast<uint8_t>(er[i]);
      const uint8_t cnt = static_cast<uint8_t>(er.size());
      h_->ctx->check(ccgpu_gf_decode_erasures_pgz(h_->ctx->get(), h_->code, w.data(), 1, pos.data(), &cnt,
                                                  static_cast<uint32_t>(er.size()), out, nullptr, failed));
      return;
    }
    if (er.size() > 30) throw decoding_failure("Number of erasures exceed what the engine supports (30).");
    for (size_t i = 0; i < er.size(); ++i) pos[i] = static_cast<uint8_t>(er[i]);
    const uint8_t cnt = static_cast<uint8_t>(er.size());
    h_->ctx->check(ccgpu_gf_decode_erasures(h_->ctx->get(), h_->code, w.data(), 1, pos.data(), &cnt, 30, out, nullptr, failed));
  }
  template <typename In> void correct_one(const In &b, uint8_t *out, uint8_t *failed, std::true_type) const {
    std::vector<float> y(b.begin(), b.end());
    correct_batch(y.data(), 1, out, failed);
  }
  template <typename In> void correct_one(const In &b, uint8_t *out, uint8_t *failed, std::false_type) const {
    std::vector<uint8_t> w;
    w.reserve(b.size());
    for (const auto &e : b) {
      if (std::is_signed<typename In::value_type>::value) w.push_back(e < 0 ? 1 : 0);  // hard_decision, codes.h:43-52
      else w.push_back(static_cast<uint8_t>(e));
    }
    correct_batch(w.data(), 1, out, failed);
  }
};

namespace detail {
template <unsigned q, typename Capability> std::shared_ptr<code_handle> make_bch(int device) {
  return code_handle::make(device, [](ccgpu_ctx *ctx, ccgpu_code **out) {
    return ccgpu_bch_create(ctx, q, correction_capability<Capability>::kind, correction_capability<Capability>::raw, out);
  });
}
}  // namespace detail

// cyclic::primitive_bch<q, Capability, Sigma> -- codes/bch.h:16-161
template <unsigned q, typename Capability, typename Sigma = peterson_gorenstein_zierler_tag>
class primitive_bch : public cyclic_base<Sigma> {
public:
  static constexpr unsigned n = (1u << q) - 1;
  static constexpr unsigned t = correction_capability<Capability>::value;
  // device < 0: the process default (cc::set_default_device); under a current device_group the code lives on all its members
  explicit primitive_bch(int device = -1) : cyclic_base<Sigma>(detail::make_bch<q, Capability>(device)) {}
};

// extension: the same code decoded with Chase-II over the P least reliable positions (ccgpu_decode_llr_chase)
template <unsigned q, typename Capability, unsigned P>
class primitive_bch<q, Capability, chase_tag<P> > : public cyclic_base<chase_tag<P> > {
  using base = cyclic_base<chase_tag<P> >;

public:
  static constexpr unsigned n = (1u << q) - 1;
  static constexpr unsigned t = correction_capability<Capability>::value;
  explicit primitive_bch(int device = -1) : base(detail::make_bch<q, Capability>(device)) {}

  // frames x n channel values -> frames x n bits; failed[f] = 1 where no test pattern decoded; chosen[f] (optional) is
  // the index of the returned test pattern
  void correct_batch(const float *y, uint64_t frames, uint8_t *bits, uint8_t *failed, uint8_t *chosen = nullptr) const {
    this->h_->ctx->check(ccgpu_decode_llr_chase(this->h_->ctx->get(), this->h_->code, P, y, frames, bits, failed, chosen));
  }
  // one frame of channel values; throws decoding_failure when no test pattern decodes
  template <typename Return_type = uint8_t, typename InputSequence>
  std::vector<Return_type> correct(const InputSequence &b) const {
    if (b.size() != n)
      throw std::runtime_error("Channel code word has the wrong size (" + std::to_string(b.size()) + "). Expected " +
                               std::to_string(n));
    const std::vector<float> y(b.begin(), b.end());
    std::vector<uint8_t> out(n);
    uint8_t failed = 0;
    correct_batch(y.data(), 1, out.data(), &failed);
    if (failed) throw decoding_failure("Decoding failure");
    return std::vector<Return_type>(out.begin(), out.end());
  }
  // one Eb/N0 point (simulation.c++:112-149) decoded with Chase-II on the device, sharded over the code's group if any
  ccgpu_counters awgn_point(double ebno_db, uint64_t frames, uint64_t seed = 0, uint32_t point = 0, uint64_t frame0 = 0) const {
    ccgpu_counters c{};
    if (this->h_->grp)
      this->h_->grp->check(ccgpu_group_awgn_point_chase(this->h_->grp->get(), this->h_->codes.data(), P, ebno_db, seed, point,
                                                        frame0, frames, &c));
    else
      this->h_->ctx->check(ccgpu_awgn_point_chase(this->h_->ctx->get(), this->h_->code, P, ebno_db, seed, point, frame0, frames, &c));
    return c;
  }
};

// extension: the same code decoded with adaptive belief propagation (ccgpu_decode_llr_abp; n <= 127, n - l <= 64)
template <unsigned q, typename Capability, unsigned Iterations, typename Gamma>
class primitive_bch<q, Capability, abp_tag<Iterations, Gamma> > : public cyclic_base<abp_tag<Iterations, Gamma> > {
  using base = cyclic_base<abp_tag<Iterations, Gamma> >;
  using tag = abp_tag<Iterations, Gamma>;

public:
  static constexpr unsigned n = (1u << q) - 1;
  static constexpr unsigned t = correction_capability<Capability>::value;
  explicit primitive_bch(int device = -1) : base(detail::make_bch<q, Capability>(device)) {}

  // frames x n channel values -> frames x n bits, iter and failed per frame; L (optional) the final soft values
  void correct_batch(const float *y, uint64_t frames, uint8_t *bits, uint8_t *iter, uint8_t *failed,
                     float *L = nullptr) const {
    this->h_->ctx->check(ccgpu_decode_llr_abp(this->h_->ctx->get(), this->h_->code, Iterations, tag::gamma, y, frames,
                                              bits, L, iter, failed));
  }
  // one frame of channel values; throws decoding_failure when the stop test never passed
  template <typename Return_type = uint8_t, typename InputSequence>
  std::vector<Return_type> correct(const InputSequence &b) const {
    if (b.size() != n)
      throw std::runtime_error("Channel code word has the wrong size (" + std::to_string(b.size()) + "). Expected " +
                               std::to_string(n));
    const std::vector<float> y(b.begin(), b.end());
    std::vector<uint8_t> out(n);
    uint8_t iter = 0, failed = 0;
    correct_batch(y.data(), 1, out.data(), &iter, &failed);
    if (failed) throw decoding_failure("Decoding failure");
    return std::vector<Return_type>(out.begin(), out.end());
  }
  // one Eb/N0 point (simulation.c++:112-149) decoded with ABP on the device, sharded over the code's group if any
  ccgpu_counters awgn_point(double ebno_db, uint64_t frames, uint64_t seed = 0, uint32_t point = 0, uint64_t frame0 = 0) const {
    ccgpu_counters c{};
    if (this->h_->grp)
      this->h_->grp->check(ccgpu_group_awgn_point_abp(this->h_->grp->get(), this->h_->codes.data(), Iterations, tag::gamma,
                                                      ebno_db, seed, point, frame0, frames, &c));
    else
      this->h_->ctx->check(ccgpu_awgn_point_abp(this->h_->ctx->get(), this->h_->code, Iterations, tag::gamma, ebno_db, seed,
                                                point, frame0, frames, &c));
    return c;
  }
};

// extension: the same code decoded with maximum-likelihood decoding (ccgpu_decode_llr_ml; n <= 127, n - l <= 12)
template <unsigned q, typename Capability>
class primitive_bch<q, Capability, ml_tag> : public cyclic_base<ml_tag> {
  using base = cyclic_base<ml_tag>;

public:
  static constexpr unsigned n = (1u << q) - 1;
  static constexpr unsigned t = correction_capability<Capability>::value;
  explicit primitive_bch(int device = -1) : base(detail::make_bch<q, Capability>(device)) {}

  // frames x n channel values -> frames x n bits, always a codeword closest to the channel values
  void correct_batch(const float *y, uint64_t frames, uint8_t *bits) const {
    this->h_->ctx->check(ccgpu_decode_llr_ml(this->h_->ctx->get(), this->h_->code, y, frames, bits));
  }
  // one frame of channel values; ML never fails
  template <typename Return_type = uint8_t, typename InputSequence>
  std::vector<Return_type> correct(const InputSequence &b) const {
    if (b.size() != n)
      throw std::runtime_error("Channel code word has the wrong size (" + std::to_string(b.size()) + "). Expected " +
                               std::to_string(n));
    const std::vector<float> y(b.begin(), b.end());
    std::vector<uint8_t> out(n);
    correct_batch(y.data(), 1, out.data());
    return std::vector<Return_type>(out.begin(), out.end());
  }
  // one Eb/N0 point (simulation.c++:112-149) decoded with ML on the device, sharded over the code's group if any
  ccgpu_counters awgn_point(double ebno_db, uint64_t frames, uint64_t seed = 0, uint32_t point = 0, uint64_t frame0 = 0) const {
    ccgpu_counters c{};
    if (this->h_->grp)
      this->h_->grp->check(ccgpu_group_awgn_point_ml(this->h_->grp->get(), this->h_->codes.data(), ebno_db, seed, point,
                                                     frame0, frames, &c));
    else
      this->h_->ctx->check(ccgpu_awgn_point_ml(this->h_->ctx->get(), this->h_->code, ebno_db, seed, point, frame0, frames, &c));
    return c;
  }
};

// extension: the same code decoded with ordered-statistics decoding of order Order (ccgpu_decode_llr_osd; n <= 127,
// n - l <= 64)
template <unsigned q, typename Capability, unsigned Order>
class primitive_bch<q, Capability, osd_tag<Order> > : public cyclic_base<osd_tag<Order> > {
  using base = cyclic_base<osd_tag<Order> >;

public:
  static constexpr unsigned n = (1u << q) - 1;
  static constexpr unsigned t = correction_capability<Capability>::value;
  explicit primitive_bch(int device = -1) : base(detail::make_bch<q, Capability>(device)) {}

  // frames x n channel values -> frames x n bits, always a codeword; weight[f] (optional) is the number of information
  // positions the returned codeword flips
  void correct_batch(const float *y, uint64_t frames, uint8_t *bits, uint8_t *weight = nullptr) const {
    this->h_->ctx->check(ccgpu_decode_llr_osd(this->h_->ctx->get(), this->h_->code, Order, y, frames, bits, weight));
  }
  // one frame of channel values; OSD never fails
  template <typename Return_type = uint8_t, typename InputSequence>
  std::vector<Return_type> correct(const InputSequence &b) const {
    if (b.size() != n)
      throw std::runtime_error("Channel code word has the wrong size (" + std::to_string(b.size()) + "). Expected " +
                               std::to_string(n));
    const std::vector<float> y(b.begin(), b.end());
    std::vector<uint8_t> out(n);
    correct_batch(y.data(), 1, out.data());
    return std::vector<Return_type>(out.begin(), out.end());
  }
  // one Eb/N0 point (simulation.c++:112-149) decoded with OSD on the device, sharded over the code's group if any
  ccgpu_counters awgn_point(double ebno_db, uint64_t frames, uint64_t seed = 0, uint32_t point = 0, uint64_t frame0 = 0) const {
    ccgpu_counters c{};
    if (this->h_->grp)
      this->h_->grp->check(ccgpu_group_awgn_point_osd(this->h_->grp->get(), this->h_->codes.data(), Order, ebno_db, seed,
                                                      point, frame0, frames, &c));
    else
      this->h_->ctx->check(ccgpu_awgn_point_osd(this->h_->ctx->get(), this->h_->code, Order, ebno_db, seed, point, frame0,
                                                frames, &c));
    return c;
  }
};

// cyclic::rs<q, Capability, Sigma, N, Coding, mu, step> -- codes/rs.h:6-94
template <unsigned q, typename Capability, typename Sigma = peterson_gorenstein_zierler_tag, unsigned mu = 1,
          unsigned step = 1>
class rs : public cyclic_base<Sigma> {
  static_assert(std::is_base_of<hard_decision_tag, Sigma>::value, "RS codes are decoded algebraically");
  static std::shared_ptr<detail::code_handle> make(int device) {
    return detail::code_handle::make(device, [](ccgpu_ctx *ctx, ccgpu_code **out) {
      return ccgpu_rs_create(ctx, q, correction_capability<Capability>::value, mu, step, out);
    });
  }

public:
  static constexpr unsigned n = (1u << q) - 1;
  static constexpr unsigned t = correction_capability<Capability>::value;
  explicit rs(int device = -1) : cyclic_base<Sigma>(make(device)) {}
};

// extension: the same RS code decoded with GMD over up to F erased symbols from the channel values of its binary image
// (ccgpu_decode_llr_gmd; 2t <= 32).  A frame is n q channel values, bit j of symbol c at position c q + j.
template <unsigned q, typename Capability, unsigned F, unsigned mu, unsigned step>
class rs<q, Capability, gmd_tag<F>, mu, step> : public cyclic_base<gmd_tag<F> > {
  using base = cyclic_base<gmd_tag<F> >;
  static std::shared_ptr<detail::code_handle> make(int device) {
    return detail::code_handle::make(device, [](ccgpu_ctx *ctx, ccgpu_code **out) {
      return ccgpu_rs_create(ctx, q, correction_capability<Capability>::value, mu, step, out);
    });
  }

public:
  static constexpr unsigned n = (1u << q) - 1;
  static constexpr unsigned t = correction_capability<Capability>::value;
  static constexpr unsigned channel_length = n * q;  // channel values per word
  static_assert(F <= 2 * t, "GMD erases at most 2t symbols");
  explicit rs(int device = -1) : base(make(device)) {}

  // frames x (n q) channel values -> frames x n symbols; failed[f] = 1: no trial decoded, words = the hard decision;
  // chosen[f] (optional) = the winning trial i (2i symbols erased)
  void correct_batch(const float *y, uint64_t frames, uint8_t *words, uint8_t *failed, uint8_t *chosen = nullptr) const {
    this->h_->ctx->check(ccgpu_decode_llr_gmd(this->h_->ctx->get(), this->h_->code, F, y, frames, words, failed, chosen));
  }
  // one frame of n q channel values -> n symbols; throws decoding_failure when no trial decodes
  template <typename Return_type = uint8_t, typename InputSequence>
  std::vector<Return_type> correct(const InputSequence &b) const {
    if (b.size() != channel_length)
      throw std::runtime_error("Channel word has the wrong size (" + std::to_string(b.size()) + "). Expected " +
                               std::to_string(channel_length));
    const std::vector<float> y(b.begin(), b.end());
    std::vector<uint8_t> out(n);
    uint8_t failed = 0;
    correct_batch(y.data(), 1, out.data(), &failed);
    if (failed) throw decoding_failure("Decoding failure");
    return std::vector<Return_type>(out.begin(), out.end());
  }
  // one Eb/N0 point (simulation.c++:112-149) decoded with GMD on the device, sharded over the code's group if any
  ccgpu_counters awgn_point(double ebno_db, uint64_t frames, uint64_t seed = 0, uint32_t point = 0, uint64_t frame0 = 0) const {
    ccgpu_counters c{};
    if (this->h_->grp)
      this->h_->grp->check(ccgpu_group_awgn_point_gmd(this->h_->grp->get(), this->h_->codes.data(), F, ebno_db, seed, point,
                                                      frame0, frames, &c));
    else
      this->h_->ctx->check(ccgpu_awgn_point_gmd(this->h_->ctx->get(), this->h_->code, F, ebno_db, seed, point, frame0,
                                                frames, &c));
    return c;
  }
};

// codes/uncoded.h:10-47 -- the pseudo-decoder of simulation/uncoded.c++: n symbols, hard decision, nominal rate 0.5.
// `correct` is the decision itself (there is no arithmetic to offload); the Monte-Carlo point runs on the device.
class uncoded {
  std::shared_ptr<device_group> grp_;
  std::shared_ptr<context> ctx_;

public:
  static constexpr double rate = 0.5;
  const unsigned n;
  explicit uncoded(const unsigned l, int device = -1)
      : grp_(device_group::current()),
        ctx_(grp_ ? std::make_shared<context>(grp_->ctx(0)) : context::shared(device < 0 ? detail::default_device_ref() : device)),
        n(l) {}
  std::string to_string() const { return std::to_string(n) + "-uncoded"; }
  template <typename Return_type = uint8_t, typename InputSequence>
  std::vector<Return_type> correct(const InputSequence &b) const {
    std::vector<Return_type> r;
    r.reserve(n);
    for (const auto &e : b)
      r.push_back(Return_type(std::is_signed<typename InputSequence::value_type>::value ? (e < 0) : static_cast<bool>(e)));
    r.resize(n, Return_type(0));
    return r;
  }
  ccgpu_counters awgn_point(double ebno_db, uint64_t frames, uint64_t seed, uint32_t point, uint64_t frame0 = 0) const {
    ccgpu_counters c{};
    if (grp_)
      grp_->check(ccgpu_group_awgn_point_uncoded(grp_->get(), n, rate, ebno_db, seed, point, frame0, frames, &c));
    else
      ctx_->check(ccgpu_awgn_point_uncoded(ctx_->get(), n, rate, ebno_db, seed, point, frame0, frames, &c));
    return c;
  }
};

}  // namespace cc
