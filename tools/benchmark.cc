// tools/benchmark.cc -- the reference's `benchmark` program (src/simulation/benchmark.c++) on the GPU
// engine: the same catalogue of 108 decoders (q in {5,6,7} x dmin in {3,5,7,9} x 9 algorithms,
// benchmark.c++:28-161), the same getopt_long_only flags (:321-372) and the same set-intersection
// selection (:405-432); each selected decoder runs one AWGN sweep or one bit-flip enumeration and
// writes "<(n, l, dmin)-TAG>.log" in the reference's format.
//
//   g++ -std=c++17 -O2 -Iinclude tools/benchmark.cc -Lchannelcoding_b200 -lccgpu -Wl,-rpath,... -pthread
//
// Additions: --seed is honoured (the reference parses and drops it), --stop-rule ref|gf2 (stop test of the soft
// decoders: the reference's integer zero-overlap rule or the GF(2) syndrome), --max-samples N, --errors W (bit-flip
// weight, bitflips.c++ uses 6), --out DIR, --device D (first CUDA device), --gpus N (shard every point over N devices
// D .. D+N-1 through a ccgpu_group; the counters, hence the logs, are identical to the one-GPU run),
// --algorithm chase1 .. chase8 (Chase-II over 1 .. 8 test positions, "(n, l, dmin)-CHASE<P>.log"; built only when
// named, never part of "all" or of the default selection), --algorithm osd0 .. osd3 (ordered-statistics decoding of
// order 0 .. 3, "(n, l, dmin)-OSD<i>.log"; likewise only when named), --algorithm abp (adaptive belief propagation,
// 50 iterations, damping 0.15, "(n, l, dmin)-ABP50.log"; likewise only when named), --algorithm ml (maximum-likelihood
// decoding of the catalogue codes with n - l <= 12: (31,26,3), (31,21,5), (63,57,3), (63,51,5), (127,120,3);
// "(n, l, dmin)-ML.log"; likewise only when named).
#include <getopt.h>

#include <cmath>
#include <cstdlib>
#include <iostream>
#include <set>
#include <string>
#include <vector>

#include "cc/simulation.h"

using namespace cc;

template <unsigned Q, typename D> static void add_code(std::vector<decoder> &v) {
  v.emplace_back(primitive_bch<Q, D, berlekamp_massey_tag>());
  v.emplace_back(primitive_bch<Q, D, peterson_gorenstein_zierler_tag>());
  v.emplace_back(primitive_bch<Q, D, euklid_tag>());
  v.emplace_back(primitive_bch<Q, D, min_sum_tag<50> >());
  v.emplace_back(primitive_bch<Q, D, normalized_min_sum_tag<50, std::ratio<8, 10> > >());
  v.emplace_back(primitive_bch<Q, D, offset_min_sum_tag<50, std::ratio<1, 100> > >());
  v.emplace_back(primitive_bch<Q, D, self_correcting_1_min_sum_tag<50> >());
  v.emplace_back(primitive_bch<Q, D, self_correcting_2_min_sum_tag<50> >());
  v.emplace_back(primitive_bch<Q, D, normalized_2d_min_sum_tag<50> >());
}
// Chase-II decoders (extension): only built when --algorithm chase<P> asks for them, never part of "all"
template <unsigned Q, unsigned P> static void add_chase_power(std::vector<decoder> &v) {
  v.emplace_back(primitive_bch<Q, dmin<3>, chase_tag<P> >());
  v.emplace_back(primitive_bch<Q, dmin<5>, chase_tag<P> >());
  v.emplace_back(primitive_bch<Q, dmin<7>, chase_tag<P> >());
  v.emplace_back(primitive_bch<Q, dmin<9>, chase_tag<P> >());
}
template <unsigned P> static void add_chase(std::vector<decoder> &v) {
  add_chase_power<5, P>(v);
  add_chase_power<6, P>(v);
  add_chase_power<7, P>(v);
}
// OSD decoders (extension): only built when --algorithm osd<i> asks for them, never part of "all"
template <unsigned Q, unsigned O> static void add_osd_power(std::vector<decoder> &v) {
  v.emplace_back(primitive_bch<Q, dmin<3>, osd_tag<O> >());
  v.emplace_back(primitive_bch<Q, dmin<5>, osd_tag<O> >());
  v.emplace_back(primitive_bch<Q, dmin<7>, osd_tag<O> >());
  v.emplace_back(primitive_bch<Q, dmin<9>, osd_tag<O> >());
}
template <unsigned O> static void add_osd(std::vector<decoder> &v) {
  add_osd_power<5, O>(v);
  add_osd_power<6, O>(v);
  add_osd_power<7, O>(v);
}
// ABP decoders (extension): only built when --algorithm abp asks for them, never part of "all"
using abp_default = abp_tag<50>;
template <unsigned Q> static void add_abp_power(std::vector<decoder> &v) {
  v.emplace_back(primitive_bch<Q, dmin<3>, abp_default>());
  v.emplace_back(primitive_bch<Q, dmin<5>, abp_default>());
  v.emplace_back(primitive_bch<Q, dmin<7>, abp_default>());
  v.emplace_back(primitive_bch<Q, dmin<9>, abp_default>());
}
// ML decoders (extension): only built when --algorithm ml asks for them, never part of "all"; the catalogue codes with
// at most 12 parity checks, the bound of the Viterbi kernel
static void add_ml(std::vector<decoder> &v) {
  v.emplace_back(primitive_bch<5, dmin<3>, ml_tag>());
  v.emplace_back(primitive_bch<5, dmin<5>, ml_tag>());
  v.emplace_back(primitive_bch<6, dmin<3>, ml_tag>());
  v.emplace_back(primitive_bch<6, dmin<5>, ml_tag>());
  v.emplace_back(primitive_bch<7, dmin<3>, ml_tag>());
}
template <unsigned Q> static void add_power(std::vector<decoder> &v) {
  add_code<Q, dmin<3> >(v);
  add_code<Q, dmin<5> >(v);
  add_code<Q, dmin<7> >(v);
  add_code<Q, dmin<9> >(v);
}

[[noreturn]] static void usage() {
  std::cout << "--simulation [awgn|bitflip]  choose the simulation (default awgn)\n"
               "--algorithm <ms|nms|oms|scms1|scms2|2dnms|bm|pgz|euklid|all|chase1..chase8|osd0..osd3|abp|ml>\n"
               "             (repeatable; Chase-II, OSD, ABP and ML only when named, awgn only)\n"
               "--k <5|6|7|all>   code length n = 2^k - 1   (repeatable)\n"
               "--dmin <3|5|7|9|all>                          (repeatable)\n"
               "--seed <num>  --seed-time  --threads <num>\n"
               "--stop-rule <ref|gf2>  --max-samples <num>  --errors <num>  --out <dir>  --device <num>  --gpus <num>\n";
  std::exit(EXIT_FAILURE);
}

static std::string lower(std::string s) {
  for (auto &c : s) c = static_cast<char>(::tolower(c));
  return s;
}

int main(int argc, char *const argv[]) {
  std::set<std::string> algorithms;
  std::set<unsigned> ks, dmins;
  std::string simulation = "awgn", out = ".";
  uint64_t seed = 0, max_samples = 1000000;
  size_t threads = 1, errors = 6;  // the GPUs are shared: sweeps are serialised unless asked otherwise
  static struct option options[] = {
    { "simulation", required_argument, nullptr, 'i' }, { "algorithm", required_argument, nullptr, 'a' },
    { "k", required_argument, nullptr, 'k' },          { "dmin", required_argument, nullptr, 'd' },
    { "seed", required_argument, nullptr, 's' },       { "seed-time", no_argument, nullptr, 't' },
    { "threads", required_argument, nullptr, 'm' },    { "max-samples", required_argument, nullptr, 'x' },
    { "errors", required_argument, nullptr, 'e' },     { "out", required_argument, nullptr, 'o' },
    { "stop-rule", required_argument, nullptr, 'r' },  { "device", required_argument, nullptr, 'g' },
    { "gpus", required_argument, nullptr, 'n' },
    { nullptr, 0, nullptr, 0 },
  };
  std::string stop = "ref";
  int device = 0, gpus = 1;
  for (;;) {
    int idx = 0;
    const int c = getopt_long_only(argc, argv, "", options, &idx);
    if (c == -1) break;
    switch (c) {
    case 'i': simulation = lower(optarg); break;
    case 'a': algorithms.insert(lower(optarg)); break;
    case 'k': if (lower(optarg) != "all") ks.insert(static_cast<unsigned>(std::stoul(optarg))); break;
    case 'd': if (lower(optarg) != "all") dmins.insert(static_cast<unsigned>(std::stoul(optarg))); break;
    case 's': seed = strtoull(optarg, nullptr, 0); break;
    case 't': seed = static_cast<uint64_t>(std::chrono::high_resolution_clock::now().time_since_epoch().count()); break;
    case 'm': threads = std::stoull(optarg); break;
    case 'x': max_samples = std::stoull(optarg); break;
    case 'e': errors = std::stoull(optarg); break;
    case 'o': out = optarg; break;
    case 'r': stop = lower(optarg); break;
    case 'g': device = std::stoi(optarg); break;
    case 'n': gpus = std::stoi(optarg); break;
    default: usage();
    }
  }
  if (simulation != "awgn" && simulation != "bitflip") usage();
  if (stop != "ref" && stop != "gf2") usage();
  if (gpus < 1 || device < 0) usage();
  if (algorithms.count("all")) algorithms.clear();
  // the flags act on the decoders at construction: stop rule, first device, number of devices per point
  set_default_stop_rule(stop == "gf2" ? stop_rule::gf2_parity : stop_rule::reference);
  set_default_device(device);
  device_group::use(gpus, device);

  std::vector<decoder> decoders;
  add_power<5>(decoders);
  add_power<6>(decoders);
  add_power<7>(decoders);
  static void (*const chase[])(std::vector<decoder> &) = { add_chase<1>, add_chase<2>, add_chase<3>, add_chase<4>,
                                                           add_chase<5>, add_chase<6>, add_chase<7>, add_chase<8> };
  for (unsigned p = 1; p <= 8; ++p)
    if (algorithms.count("chase" + std::to_string(p))) chase[p - 1](decoders);
  static void (*const osd[])(std::vector<decoder> &) = { add_osd<0>, add_osd<1>, add_osd<2>, add_osd<3> };
  for (unsigned o = 0; o <= 3; ++o)
    if (algorithms.count("osd" + std::to_string(o))) osd[o](decoders);
  if (algorithms.count("abp")) {  // selected below by the name in the log: ABP50
    add_abp_power<5>(decoders);
    add_abp_power<6>(decoders);
    add_abp_power<7>(decoders);
    algorithms.insert(lower(abp_default::to_string()));
  }

  if (algorithms.count("ml")) add_ml(decoders);

  // selection by parsing to_string(), exactly like benchmark.c++:214-240
  std::vector<const decoder *> chosen;
  for (const auto &d : decoders) {
    const std::string str = d.to_string();
    const std::string name = lower(str.substr(str.find_last_of('-') + 1));
    const size_t end = str.find_last_of(')'), start = str.find_last_of(' ', end);
    const unsigned distance = static_cast<unsigned>(std::stoul(str.substr(start + 1, end - start - 1)));
    const unsigned n = static_cast<unsigned>(std::stoul(str.substr(str.find_first_of('(') + 1)));
    const unsigned power = static_cast<unsigned>(std::log2(n + 1));
    if (!algorithms.empty() && !algorithms.count(name)) continue;
    if (!ks.empty() && !ks.count(power)) continue;
    if (!dmins.empty() && !dmins.count(distance)) continue;
    chosen.push_back(&d);
  }
  if (chosen.empty()) {
    std::cout << "The selection is empty" << std::endl;
    usage();
  }
  thread_pool p(threads);
  for (const decoder *d : chosen) {
    if (simulation == "awgn")
      p.push([=] { awgn_simulation(*d, 0.5, seed).samples_cap(max_samples).output_dir(out)(); });
    else
      p.push([=] { bitflip_simulation(*d, errors).output_dir(out)(); });
  }
}
