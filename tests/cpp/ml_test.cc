// tests/cpp/ml_test.cc -- the ML decoders of the C++ layer (cc::primitive_bch<q, Capability, ml_tag>).
//   ml_test --host        no GPU needed: tag name and traits
//   ml_test --gpu <dir>   needs a B200: correct() against the C ABI batch, the AWGN point through cc::decoder,
//                         awgn_simulation's log, bit-flip simulation rejected
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <string>
#include <vector>

#include "cc/simulation.h"

using namespace cc;

#define CHECK(cond)                                                                  \
  do {                                                                               \
    if (!(cond)) {                                                                   \
      std::cerr << "CHECK failed: " #cond " at line " << __LINE__ << std::endl;      \
      return 1;                                                                      \
    }                                                                                \
  } while (0)

static bool same(const ccgpu_counters &a, const ccgpu_counters &b) {
  return a.frames == b.frames && a.frame_errors == b.frame_errors && a.bit_errors == b.bit_errors &&
         a.iterations == b.iterations && a.failures == b.failures && a.undetected == b.undetected;
}

static int host_tests() {
  CHECK(ml_tag::to_string() == "ML");
  static_assert(std::is_base_of<algorithm_tag, ml_tag>::value, "");
  static_assert(!std::is_base_of<soft_decision_tag, ml_tag>::value, "");
  static_assert(!std::is_base_of<hard_decision_tag, ml_tag>::value, "");
  static_assert(is_ml_tag<ml_tag>::value && !is_ml_tag<osd_tag<3> >::value && !is_osd_tag<ml_tag>::value, "");
  std::cout << "host ok" << std::endl;
  return 0;
}

static int gpu_tests(const std::string &dir) {
  using code_t = primitive_bch<6, dmin<5>, ml_tag>;
  const code_t code;
  CHECK(code.to_string() == "(63, 51, 5)-ML");
  CHECK(code_t::n == 63 && code_t::t == 2);
  // a few hundred frames of the Philox channel at 3 dB: single-frame correct() == the C ABI batch
  const unsigned n = code_t::n;
  const uint64_t frames = 400;
  std::vector<float> y(frames * n);
  CHECK(ccgpu_awgn_llr(code.ctx()->get(), n, ccgpu_sigma(code.rate, 3.0), 5, 0, 0, frames, y.data()) == CCGPU_OK);
  std::vector<uint8_t> bits(frames * n);
  CHECK(ccgpu_decode_llr_ml(code.ctx()->get(), code.handle(), y.data(), frames, bits.data()) == CCGPU_OK);
  std::vector<uint8_t> bits2(frames * n);
  code.correct_batch(y.data(), frames, bits2.data());
  CHECK(bits == bits2);
  unsigned changed = 0;
  for (uint64_t f = 0; f < frames; ++f) {
    const std::vector<float> one(y.begin() + f * n, y.begin() + (f + 1) * n);
    const std::vector<uint8_t> out = code.correct(one);
    CHECK(std::equal(out.begin(), out.end(), bits.begin() + f * n));
    bool differs = false;
    for (unsigned c = 0; c < n; ++c) differs |= out[c] != (one[c] < 0.0f ? 1 : 0);
    changed += differs;
  }
  CHECK(changed > 0 && changed < frames);
  // the AWGN point through the type-erased decoder is ccgpu_awgn_point_ml
  const decoder d(code);
  CHECK(!d.soft() && d.n() == 63 && d.to_string() == code.to_string());
  for (const double eb : { 3.0, 4.0 }) {
    ccgpu_counters direct{};
    CHECK(ccgpu_awgn_point_ml(code.ctx()->get(), code.handle(), eb, 7, 2, 1000, 20000, &direct) == CCGPU_OK);
    const ccgpu_counters via = d.awgn_point(eb, 20000, 7, 2, 1000);
    CHECK(same(direct, via) && direct.frames == 20000 && direct.iterations == 0 && direct.failures == 0 &&
          direct.undetected == direct.frame_errors && direct.frame_errors > 0);
  }
  // awgn_simulation writes the reference's log; its sidecar holds the counters of each point
  awgn_simulation(d, 0.5, 3).samples_cap(20000).output_dir(dir)();
  std::ifstream log(dir + "/(63, 51, 5)-ML.log");
  std::string header;
  CHECK(std::getline(log, header) && header == "   ebno                   wer");
  {
    std::string line;
    std::getline(log, line);
    const double eb = std::stod(line);
    const ccgpu_counters first = d.awgn_point(eb, awgn_simulation(d).samples_cap(20000).samples(0.5), 3, 0);
    std::ifstream js(dir + "/(63, 51, 5)-ML.json");
    const std::string text((std::istreambuf_iterator<char>(js)), std::istreambuf_iterator<char>());
    CHECK(text.find("\"frame_errors\": " + std::to_string(first.frame_errors) + ",") != std::string::npos);
  }
  // bit flips carry no reliabilities: rejected loudly
  bool rejected = false;
  try {
    d.bitflip_point(1);
  } catch (const std::runtime_error &) {
    rejected = true;
  }
  CHECK(rejected);
  std::cout << "gpu ok" << std::endl;
  return 0;
}

int main(int argc, char **argv) {
  if (argc >= 2 && std::string(argv[1]) == "--host") return host_tests();
  if (argc >= 3 && std::string(argv[1]) == "--gpu") return gpu_tests(argv[2]);
  std::cerr << "usage: ml_test --host | --gpu <scratch dir>" << std::endl;
  return 2;
}
