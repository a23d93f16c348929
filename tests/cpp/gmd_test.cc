// tests/cpp/gmd_test.cc -- the GMD decoders of the C++ layer (cc::rs<q, Capability, gmd_tag<F> >).
//   gmd_test --host        no GPU needed: tag names and traits
//   gmd_test --gpu <dir>   needs a B200: correct() against the C ABI batch, the AWGN point through cc::decoder (channel
//                          length n q), awgn_simulation's log, bit-flip simulation rejected, hard tags unchanged
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
  CHECK(gmd_tag<32>::to_string() == "GMD32" && gmd_tag<0>::to_string() == "GMD0");
  static_assert(gmd_tag<8>::max_erasures == 8, "");
  static_assert(std::is_base_of<algorithm_tag, gmd_tag<2> >::value, "");
  static_assert(!std::is_base_of<soft_decision_tag, gmd_tag<2> >::value, "");
  static_assert(!std::is_base_of<hard_decision_tag, gmd_tag<2> >::value, "");
  static_assert(is_gmd_tag<gmd_tag<4> >::value && !is_gmd_tag<chase_tag<4> >::value && !is_osd_tag<gmd_tag<2> >::value,
                "");
  using code_t = rs<4, errors<3>, gmd_tag<6> >;
  static_assert(code_t::n == 15 && code_t::t == 3 && code_t::channel_length == 60 && code_t::gmd && !code_t::chase, "");
  static_assert(!rs<8, errors<16>, euklid_tag>::gmd, "");
  std::cout << "host ok" << std::endl;
  return 0;
}

static int gpu_tests(const std::string &dir) {
  using code_t = rs<4, errors<3>, gmd_tag<6> >;
  const code_t code;
  CHECK(code.to_string().size() > 5 && code.to_string().substr(code.to_string().size() - 5) == "-GMD6");
  // a few hundred frames of the Philox channel at 5 dB: single-frame correct() == the C ABI batch
  const unsigned n = code_t::n, nq = code_t::channel_length;
  const uint64_t frames = 400;
  std::vector<float> y(frames * nq);
  CHECK(ccgpu_awgn_llr(code.ctx()->get(), nq, ccgpu_sigma(code.rate, 5.0), 5, 0, 0, frames, y.data()) == CCGPU_OK);
  std::vector<uint8_t> words(frames * n), failed(frames), chosen(frames);
  CHECK(ccgpu_decode_llr_gmd(code.ctx()->get(), code.handle(), 6, y.data(), frames, words.data(), failed.data(),
                             chosen.data()) == CCGPU_OK);
  std::vector<uint8_t> words2(frames * n), failed2(frames), chosen2(frames);
  code.correct_batch(y.data(), frames, words2.data(), failed2.data(), chosen2.data());
  CHECK(words == words2 && failed == failed2 && chosen == chosen2);
  unsigned erased = 0, failures = 0;
  for (uint64_t f = 0; f < frames; ++f) {
    const std::vector<float> one(y.begin() + f * nq, y.begin() + (f + 1) * nq);
    try {
      const std::vector<uint8_t> out = code.correct(one);
      CHECK(!failed[f] && std::equal(out.begin(), out.end(), words.begin() + f * n));
    } catch (const decoding_failure &) {
      CHECK(failed[f]);
      ++failures;
    }
    CHECK(chosen[f] <= 3);
    erased += chosen[f] != 0;
  }
  CHECK(erased > 0 && failures < frames);
  bool wrong_size = false;
  try {
    code.correct(std::vector<float>(n, 1.0f));
  } catch (const std::runtime_error &) {
    wrong_size = true;
  }
  CHECK(wrong_size);
  // the AWGN point through the type-erased decoder is ccgpu_awgn_point_gmd; its channel length is n q
  const decoder d(code);
  CHECK(!d.soft() && d.n() == nq && d.to_string() == code.to_string());
  CHECK(d.correct(std::vector<float>(nq, 1.0f)) == std::vector<uint8_t>(n, 0));
  for (const double eb : { 4.0, 5.0 }) {
    ccgpu_counters direct{};
    CHECK(ccgpu_awgn_point_gmd(code.ctx()->get(), code.handle(), 6, eb, 7, 2, 1000, 20000, &direct) == CCGPU_OK);
    const ccgpu_counters via = d.awgn_point(eb, 20000, 7, 2, 1000);
    CHECK(same(direct, via) && direct.frames == 20000 && direct.iterations == 0 && direct.frame_errors > 0 &&
          direct.frame_errors == direct.failures + direct.undetected);
  }
  // awgn_simulation writes the reference's log; its sidecar holds the counters of each point
  awgn_simulation(d, 0.5, 3).samples_cap(20000).output_dir(dir)();
  std::ifstream log(dir + "/" + code.to_string() + ".log");
  std::string header;
  CHECK(std::getline(log, header) && header == "   ebno                   wer");
  {
    std::string line;
    std::getline(log, line);
    const double eb = std::stod(line);
    const ccgpu_counters first = d.awgn_point(eb, awgn_simulation(d).samples_cap(20000).samples(0.5), 3, 0);
    std::ifstream js(dir + "/" + code.to_string() + ".json");
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
  // RS(255,223) with all 17 trials: a codeword with its 32 least reliable symbols garbled is recovered
  {
    using big_t = rs<8, errors<16>, gmd_tag<32> >;
    const big_t big;
    std::vector<float> yb(big_t::channel_length, 2.0f);
    for (unsigned c = 0; c < 32; ++c)
      for (unsigned j = 0; j < 8; ++j) yb[(7 * c) * 8 + j] = (j & 1) ? -0.1f : 0.1f;
    CHECK(big.correct(yb) == std::vector<uint8_t>(big_t::n, 0));
  }
  // the hard-decision RS tags keep their behaviour: ccgpu_awgn_point_hard still refuses RS codes
  {
    const decoder hard(rs<4, errors<3>, euklid_tag>{});
    CHECK(hard.n() == 15);
    bool refused = false;
    try {
      hard.awgn_point(5.0, 100, 0, 0);
    } catch (const std::runtime_error &) {
      refused = true;
    }
    CHECK(refused);
  }
  std::cout << "gpu ok" << std::endl;
  return 0;
}

int main(int argc, char **argv) {
  if (argc >= 2 && std::string(argv[1]) == "--host") return host_tests();
  if (argc >= 3 && std::string(argv[1]) == "--gpu") return gpu_tests(argv[2]);
  std::cerr << "usage: gmd_test --host | --gpu <scratch dir>" << std::endl;
  return 2;
}
