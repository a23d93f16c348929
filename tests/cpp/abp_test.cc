// tests/cpp/abp_test.cc -- the ABP decoders of the C++ layer (cc::primitive_bch<q, Capability, abp_tag<I, Gamma> >).
//   abp_test --host        no GPU needed: tag names and traits
//   abp_test --gpu <dir>   needs a B200: correct() against the C ABI batch, the AWGN point through cc::decoder,
//                          awgn_simulation's log, bit-flip simulation rejected
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
  CHECK(abp_tag<50>::to_string() == "ABP50" && (abp_tag<20, std::ratio<1, 10> >::to_string() == "ABP20"));
  static_assert(abp_tag<50>::iterations == 50 && abp_tag<50>::gamma == 0.15, "");
  static_assert(abp_tag<5, std::ratio<3, 10> >::gamma == 0.3 && abp_tag<1, std::ratio<1> >::gamma == 1.0, "");
  static_assert(std::is_base_of<algorithm_tag, abp_tag<5> >::value, "");
  static_assert(!std::is_base_of<soft_decision_tag, abp_tag<5> >::value, "");
  static_assert(!std::is_base_of<hard_decision_tag, abp_tag<5> >::value, "");
  static_assert(is_abp_tag<abp_tag<5> >::value && is_abp_tag<abp_tag<0, std::ratio<1, 2> > >::value, "");
  static_assert(!is_abp_tag<osd_tag<2> >::value && !is_osd_tag<abp_tag<2> >::value && !is_chase_tag<abp_tag<2> >::value, "");
  std::cout << "host ok" << std::endl;
  return 0;
}

static int gpu_tests(const std::string &dir) {
  using code_t = primitive_bch<6, dmin<11>, abp_tag<50> >;
  const code_t code;
  CHECK(code.to_string() == "(63, 36, 11)-ABP50");
  CHECK(code_t::n == 63 && code_t::t == 5);
  // a few hundred frames of the Philox channel at 2 dB: single-frame correct() == the C ABI batch
  const unsigned n = code_t::n;
  const uint64_t frames = 400;
  std::vector<float> y(frames * n);
  CHECK(ccgpu_awgn_llr(code.ctx()->get(), n, ccgpu_sigma(code.rate, 2.0), 5, 0, 0, frames, y.data()) == CCGPU_OK);
  std::vector<uint8_t> bits(frames * n), iter(frames), failed(frames);
  std::vector<float> L(frames * n);
  CHECK(ccgpu_decode_llr_abp(code.ctx()->get(), code.handle(), 50, 0.15, y.data(), frames, bits.data(), L.data(),
                             iter.data(), failed.data()) == CCGPU_OK);
  std::vector<uint8_t> bits2(frames * n), iter2(frames), failed2(frames);
  std::vector<float> L2(frames * n);
  code.correct_batch(y.data(), frames, bits2.data(), iter2.data(), failed2.data(), L2.data());
  CHECK(bits == bits2 && iter == iter2 && failed == failed2 && L == L2);
  unsigned updated = 0;
  for (uint64_t f = 0; f < frames; ++f) {
    const std::vector<float> one(y.begin() + f * n, y.begin() + (f + 1) * n);
    CHECK(!failed[f]);  // at 2 dB ABP (50, 0.15) reaches a codeword on every frame of this sample
    const std::vector<uint8_t> out = code.correct(one);
    CHECK(std::equal(out.begin(), out.end(), bits.begin() + f * n));
    updated += iter[f] != 0;
  }
  CHECK(updated > 0 && updated < frames);
  // one update at most: correct() throws exactly on the frames the C ABI reports as failed
  const primitive_bch<6, dmin<11>, abp_tag<1, std::ratio<1, 2> > > once;
  CHECK(ccgpu_decode_llr_abp(code.ctx()->get(), once.handle(), 1, 0.5, y.data(), frames, bits.data(), nullptr,
                             iter.data(), failed.data()) == CCGPU_OK);
  unsigned thrown = 0, n_failed = 0;
  for (uint64_t f = 0; f < frames; ++f) {
    const std::vector<float> one(y.begin() + f * n, y.begin() + (f + 1) * n);
    n_failed += failed[f];
    try {
      const std::vector<uint8_t> out = once.correct(one);
      CHECK(!failed[f] && std::equal(out.begin(), out.end(), bits.begin() + f * n));
    } catch (const decoding_failure &) {
      CHECK(failed[f] && iter[f] == 1);
      ++thrown;
    }
  }
  CHECK(thrown == n_failed && thrown > 0);
  // the AWGN point through the type-erased decoder is ccgpu_awgn_point_abp, iterations included
  const decoder d(code);
  CHECK(!d.soft() && d.n() == 63 && d.to_string() == code.to_string());
  for (const double eb : { 3.0, 4.0 }) {
    ccgpu_counters direct{};
    CHECK(ccgpu_awgn_point_abp(code.ctx()->get(), code.handle(), 50, 0.15, eb, 7, 2, 1000, 20000, &direct) == CCGPU_OK);
    const ccgpu_counters via = d.awgn_point(eb, 20000, 7, 2, 1000);
    CHECK(same(direct, via) && direct.frames == 20000 && direct.iterations > 0 && direct.frame_errors > 0 &&
          direct.frame_errors >= direct.failures);
  }
  // awgn_simulation writes the reference's log; its sidecar holds the counters of each point
  awgn_simulation(d, 0.5, 3).samples_cap(20000).output_dir(dir)();
  std::ifstream log(dir + "/(63, 36, 11)-ABP50.log");
  std::string header;
  CHECK(std::getline(log, header) && header == "   ebno                   wer");
  {
    std::string line;
    std::getline(log, line);
    const double eb = std::stod(line);
    const ccgpu_counters first = d.awgn_point(eb, awgn_simulation(d).samples_cap(20000).samples(0.5), 3, 0);
    std::ifstream js(dir + "/(63, 36, 11)-ABP50.json");
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
  std::cerr << "usage: abp_test --host | --gpu <scratch dir>" << std::endl;
  return 2;
}
