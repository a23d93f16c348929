// cc/simulation.h -- the reference's simulation layer (src/simulation/simulation.{h,c++}) on top
// of the GPU engine: same class names, same sweep schedule, same log-file format; the per-frame
// inner loop (simulation.c++:124-136: generate noise -> decoder.correct -> count) is replaced by
// one fused kernel launch per Eb/N0 point (ccgpu_awgn_point).
//
//   reference                                   here
//   -----------------------------------------   ---------------------------------------------------
//   class decoder (type erasure)                cc::decoder            simulation.h:23-69
//   class awgn_simulation                       cc::awgn_simulation    simulation.h:71-83, .c++:95-150
//   class bitflip_simulation                    cc::bitflip_simulation simulation.h:85-92, .c++:156-213
//   class thread_pool                           cc::thread_pool        simulation.h:94-117, .c++:219-273
//
// Deviations, all deliberate:  the noise is Philox-based (any frame of any point is addressable, so
// results do not depend on the number of GPUs), the `seed` really is forwarded (the reference parses
// --seed but never uses it, benchmark.c++:193-196), and next to "<name>.log" a "<name>.json" sidecar
// records frames, frame/bit errors, iterations and failures per point.
#pragma once
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <fstream>
#include <functional>
#include <iomanip>
#include <iostream>
#include <limits>
#include <list>
#include <memory>
#include <mutex>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include <sys/stat.h>

#include "codes.h"

namespace cc {

// ---- simulation.h:23-69: value-semantic, type-erased decoder ----------------------------------------
class decoder {
  class decoder_concept {
  public:
    virtual ~decoder_concept() = default;
    virtual std::vector<uint8_t> correct(const std::vector<float> &b) const = 0;
    virtual std::string to_string() const = 0;
    virtual double rate() const = 0;
    virtual unsigned n() const = 0;
    virtual bool soft() const = 0;
    virtual ccgpu_counters awgn_point(double ebno_db, uint64_t frames, uint64_t seed, uint32_t point,
                                      uint64_t frame0) const = 0;
    virtual ccgpu_counters bitflip_point(unsigned weight) const = 0;
  };
  template <typename T> class decoder_model : public decoder_concept {
    T implementation;

    // hard-decision tags: channel, hard decision (codes.h:43-52), algebraic decode and the error test of
    // simulation.c++:126-135 all on the device (ccgpu_awgn_point_hard)
    ccgpu_counters hard_point(double ebno_db, uint64_t frames, uint64_t seed, uint32_t point, uint64_t frame0) const {
      return implementation.awgn_point_hard(ebno_db, frames, seed, point, frame0);
    }
    template <typename U = T>
    ccgpu_counters point_impl(double e, uint64_t f, uint64_t s, uint32_t p, uint64_t f0, std::true_type) const {
      return implementation.awgn_point(e, f, s, p, f0);
    }
    template <typename U = T>
    ccgpu_counters point_impl(double e, uint64_t f, uint64_t s, uint32_t p, uint64_t f0, std::false_type) const {
      return hard_point(e, f, s, p, f0);
    }
    ccgpu_counters flips_impl(unsigned weight, std::true_type) const { return implementation.bitflip_point(weight); }
    ccgpu_counters flips_impl(unsigned weight, std::false_type) const {
      // enumerate the patterns on the host (std::next_permutation order like simulation.c++:181-199) and decode them
      // in bounded chunks: C(127, 6) patterns would not fit any memory in one piece, the reference streams them too
      const unsigned n_ = T::n;
      const size_t chunk = std::max<size_t>(1, (size_t(64) << 20) / n_);
      std::vector<int> b(n_ - weight, 0);
      b.insert(b.end(), weight, 1);
      std::vector<uint8_t> w, out, failed;
      w.reserve(chunk * n_);
      ccgpu_counters c{};
      auto flush = [&] {
        const uint64_t count = w.size() / n_;
        if (!count) return;
        out.resize(w.size());
        failed.resize(count);
        implementation.correct_batch(w.data(), count, out.data(), failed.data());
        for (uint64_t f = 0; f < count; ++f) {
          unsigned bits = 0;
          for (unsigned i = 0; i < n_; ++i) bits += out[f * n_ + i] != 0;
          c.frames++;
          c.failures += failed[f];
          c.bit_errors += bits;
          c.frame_errors += (failed[f] || bits) ? 1 : 0;
        }
        w.clear();
      };
      do {
        for (int bit : b) w.push_back(static_cast<uint8_t>(bit));
        if (w.size() >= chunk * n_) flush();
      } while (std::next_permutation(b.begin(), b.end()));
      flush();
      return c;
    }
  public:
    explicit decoder_model(T arg) : implementation(std::move(arg)) {}
    std::vector<uint8_t> correct(const std::vector<float> &b) const override { return implementation.template correct<uint8_t>(b); }
    std::string to_string() const override { return implementation.to_string(); }
    double rate() const override { return implementation.rate; }
    unsigned n() const override {  // channel values per frame: n q for GMD, which takes the binary image of RS words
      if constexpr (T::gmd)
        return T::channel_length;
      else
        return T::n;
    }
    bool soft() const override { return T::soft_tag; }
    ccgpu_counters awgn_point(double e, uint64_t f, uint64_t s, uint32_t p, uint64_t f0) const override {
      // soft tags, Chase-II, OSD, GMD, ABP and ML take the channel values: their own fused point
      return point_impl(e, f, s, p, f0,
                        std::integral_constant<bool, T::soft_tag || T::chase || T::osd || T::gmd || T::abp || T::ml>());
    }
    ccgpu_counters bitflip_point(unsigned weight) const override {
      if constexpr (T::chase)
        throw std::runtime_error(implementation.to_string() + ": bit-flip simulation has no channel reliabilities for Chase-II");
      else if constexpr (T::osd)
        throw std::runtime_error(implementation.to_string() + ": bit-flip simulation has no channel reliabilities for OSD");
      else if constexpr (T::gmd)
        throw std::runtime_error(implementation.to_string() + ": bit-flip simulation has no channel reliabilities for GMD");
      else if constexpr (T::abp)
        throw std::runtime_error(implementation.to_string() + ": bit-flip simulation has no channel reliabilities for ABP");
      else if constexpr (T::ml)
        throw std::runtime_error(implementation.to_string() + ": bit-flip simulation has no channel reliabilities for ML");
      else
        return flips_impl(weight, std::integral_constant<bool, T::soft_tag>());
    }
  };

  // codes/uncoded.h plugged into the simulations (simulation/uncoded.c++:54)
  class uncoded_model : public decoder_concept {
    uncoded implementation;

  public:
    explicit uncoded_model(uncoded arg) : implementation(std::move(arg)) {}
    std::vector<uint8_t> correct(const std::vector<float> &b) const override { return implementation.correct<uint8_t>(b); }
    std::string to_string() const override { return implementation.to_string(); }
    double rate() const override { return uncoded::rate; }
    unsigned n() const override { return implementation.n; }
    bool soft() const override { return false; }
    ccgpu_counters awgn_point(double e, uint64_t f, uint64_t s, uint32_t p, uint64_t f0) const override {
      return implementation.awgn_point(e, f, s, p, f0);
    }
    ccgpu_counters bitflip_point(unsigned weight) const override {  // every flipped pattern is a word error
      ccgpu_counters c{};
      double patterns = 1.0;
      for (unsigned i = 1; i <= weight; ++i) patterns = patterns * (implementation.n - weight + i) / i;
      c.frames = static_cast<uint64_t>(patterns + 0.5);
      c.frame_errors = weight ? c.frames : 0;
      c.bit_errors = c.frames * weight;
      return c;
    }
  };

  std::shared_ptr<const decoder_concept> _self;

public:
  template <typename T> decoder(T d) : _self(std::make_shared<decoder_model<T> >(std::move(d))) {}
  decoder(uncoded d) : _self(std::make_shared<uncoded_model>(std::move(d))) {}
  template <typename InputSequence> std::vector<uint8_t> correct(const InputSequence &b) const {
    return _self->correct(std::vector<float>(b.begin(), b.end()));
  }
  std::string to_string() const { return _self->to_string(); }
  double rate() const { return _self->rate(); }
  unsigned n() const { return _self->n(); }
  bool soft() const { return _self->soft(); }
  ccgpu_counters awgn_point(double ebno_db, uint64_t frames, uint64_t seed, uint32_t point, uint64_t frame0 = 0) const {
    return _self->awgn_point(ebno_db, frames, seed, point, frame0);
  }
  ccgpu_counters bitflip_point(unsigned weight) const { return _self->bitflip_point(weight); }
};

namespace detail {
inline bool file_exists(const std::string &fname) {
  struct stat buf;
  return stat(fname.c_str(), &buf) != -1;
}
inline std::ofstream open_file(const std::string &fname) {  // simulation.c++:72-81: never overwrite a log
  if (file_exists(fname)) throw std::runtime_error("File " + fname + " already exists.");
  return std::ofstream(fname.c_str(), std::ofstream::out);
}

// Shannon limit Eb/N0 [dB] of rate R on the binary-input AWGN channel (computed in the library;
// the reference tabulates it, simulation.c++:21-70)
inline double shannon_limit_db(double rate) { return ccgpu_shannon_limit_db(rate); }
}  // namespace detail

// ---- simulation.h:71-83, simulation.c++:95-150 -------------------------------------------------------
class awgn_simulation {
  const class decoder &decoder_;
  const double step;
  const uint64_t seed;
  uint64_t max_samples = 1000000;  // min(1e6, .) of simulation.c++:91-93
  std::string dir = ".";

public:
  awgn_simulation(const class decoder &d, const double step_ = 0.5, const uint64_t seed_ = 0)
      : decoder_(d), step(step_), seed(seed_) {}
  awgn_simulation &samples_cap(uint64_t cap) { max_samples = cap; return *this; }
  awgn_simulation &output_dir(const std::string &d) { dir = d; return *this; }

  // first simulated point: one full step above the (rounded-down) Shannon limit, simulation.c++:105-107;
  // a negative limit counts as 0 (the reference's size_t conversion of a negative is UB, SURVEY C12)
  static double start_ebno(double rate, double step) {
    return ccgpu_sweep_start_ebno(rate, step);
  }
  size_t samples(double wer) const { return static_cast<size_t>(std::min(double(max_samples), 5e3 / wer)); }

  void operator()() const {
    const size_t wer_width = std::numeric_limits<double>::digits10;
    const size_t ebno_width = 6;
    std::ofstream log_file(detail::open_file(dir + "/" + decoder_.to_string() + ".log"));
    std::ofstream json(dir + "/" + decoder_.to_string() + ".json");
    log_file << std::setw(ebno_width + 1) << "ebno" << " ";
    log_file << std::setw(wer_width + 6) << "wer" << std::endl;
    const double start = start_ebno(decoder_.rate(), step);
    const double max = std::max(8.0, start) + step / 2;
    double wer = 0.5;
    uint32_t point = 0;
    json << "[";
    for (double eb_no = start; eb_no < max; eb_no += step, ++point) {
      const size_t iterations = samples(wer);
      std::cout << std::this_thread::get_id() << " " << decoder_.to_string() << ": E_b/N_0 = " << eb_no << " with "
                << iterations << " … ";
      std::cout.flush();
      auto t0 = std::chrono::high_resolution_clock::now();
      const ccgpu_counters c = decoder_.awgn_point(eb_no, iterations, seed, point);
      auto seconds = std::chrono::duration_cast<std::chrono::seconds>(std::chrono::high_resolution_clock::now() - t0).count();
      std::cout << seconds << " s" << std::endl;
      wer = static_cast<double>(c.frame_errors) / iterations;
      log_file << std::setw(ebno_width + 1) << std::setprecision(ebno_width) << std::defaultfloat << eb_no << " ";
      log_file << std::setw(wer_width + 1) << std::setprecision(wer_width) << std::scientific << wer << std::endl;
      json << (point ? ",\n " : "") << "{\"ebno\": " << eb_no << ", \"frames\": " << c.frames << ", \"frame_errors\": "
           << c.frame_errors << ", \"bit_errors\": " << c.bit_errors << ", \"iterations\": " << c.iterations
           << ", \"failures\": " << c.failures << ", \"undetected\": " << c.undetected << "}";
      if (wer == 0.0) wer = 5e3 / double(max_samples);  // keep N at its cap instead of dividing by zero
    }
    json << "]\n";
  }
};

// ---- simulation.h:85-92, simulation.c++:156-213 ------------------------------------------------------
class bitflip_simulation {
  const class decoder &decoder_;
  const size_t errors;
  std::string dir = ".";

public:
  bitflip_simulation(const class decoder &d, const size_t errors_ = 0) : decoder_(d), errors(errors_) {}
  bitflip_simulation &output_dir(const std::string &d) { dir = d; return *this; }
  void operator()() const {
    const size_t wer_width = std::numeric_limits<double>::digits10;
    const size_t ebno_width = 6;
    std::ofstream log_file(detail::open_file(dir + "/" + decoder_.to_string() + ".log"));
    log_file << std::setw(ebno_width + 1) << "errors" << " ";
    log_file << std::setw(wer_width + 6) << "wer" << std::endl;
    for (size_t error = 0; error <= errors; error++) {
      std::cout << std::this_thread::get_id() << " " << decoder_.to_string() << ": errors = " << error << " … ";
      std::cout.flush();
      auto t0 = std::chrono::high_resolution_clock::now();
      const ccgpu_counters c = decoder_.bitflip_point(static_cast<unsigned>(error));
      auto seconds = std::chrono::duration_cast<std::chrono::seconds>(std::chrono::high_resolution_clock::now() - t0).count();
      std::cout << seconds << " s " << c.frame_errors << " " << c.frames << std::endl;
      log_file << std::setw(ebno_width + 1) << std::setprecision(ebno_width) << std::defaultfloat << error << " ";
      log_file << std::setw(wer_width + 1) << std::setprecision(wer_width) << std::scientific
               << static_cast<double>(c.frame_errors) / c.frames << std::endl;
    }
  }
};

// ---- simulation.h:94-117, simulation.c++:219-273: tasks = whole sweeps, one per decoder ---------------
class thread_pool {
  std::vector<std::thread> pool;
  std::mutex lock;
  std::condition_variable cv;
  std::list<std::function<void(void)> > queue;
  bool running = true;

  void thread_function() {
    for (;;) {
      std::function<void(void)> work;
      {
        std::unique_lock<std::mutex> m(lock);
        cv.wait(m, [&] { return !queue.empty() || !running; });
        if (queue.empty()) return;
        work = std::move(queue.front());
        queue.pop_front();
      }
      try {
        work();
      } catch (const std::exception &e) {  // a failing sweep is reported and dropped (simulation.c++:263-268)
        std::cerr << e.what() << std::endl;
      }
    }
  }

public:
  explicit thread_pool(const size_t pool_size = std::thread::hardware_concurrency()) {
    for (size_t i = 0; i < pool_size; i++) pool.emplace_back([this] { thread_function(); });
    std::cout << "Using " << pool.size() << " threads." << std::endl;
  }
  ~thread_pool() {
    {
      std::lock_guard<std::mutex> m(lock);
      running = false;
    }
    cv.notify_all();
    for (auto &&t : pool) t.join();
  }
  template <typename Functor> void push(Functor &&f) {
    {
      std::lock_guard<std::mutex> m(lock);
      queue.emplace_back(std::forward<Functor>(f));
    }
    cv.notify_one();
  }
};

}  // namespace cc
