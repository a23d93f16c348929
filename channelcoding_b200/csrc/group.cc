// group.cc -- ccgpu_group: several CUDA devices of one host behind ONE handle (include/ccgpu.h, "device groups").
//
// The reference has no notion of a device; what this replaces is the place where its simulation decides how much
// work a point is and waits for the result (simulation/simulation.c++:112-149: the frame loop of one Eb/N0 point and
// the word-error rate that sizes the next point, :91-93).  A group shards the global frame range of a point over its
// members by frame index -- the noise is keyed by the global frame index, so the counters do not depend on the
// number of devices -- and merges the eight counters inside the library.
//
// Mechanism: one persistent host thread per member device (member 0 is served by the calling thread).  A call hands
// every thread its frame range, each runs the ordinary single-device entry point on its own context / stream, and the
// caller adds the partial counters.  Measured against the alternative SURVEY.md 5 names (ncclAllReduce of the
// counters on the kernels' streams) in profiles/r2_notes.md: the host needs the merged counters anyway (the next
// point's sample count depends on them), so the all-reduce only adds its latency to the one device-to-host copy
// that both variants need; the multi-process path (torchrun, channelcoding_b200/simulation.py) keeps the NCCL
// all-reduce because there the counters live in different processes.
//
// Built on the public C ABI only (no access to context internals).
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <functional>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/ccgpu.h"

struct ccgpu_group {
  std::vector<ccgpu_ctx *> ctx;
  std::vector<int> device;
  std::vector<std::thread> workers;  // members 1 .. n-1
  std::mutex call_mu;                // one group call at a time
  std::mutex mu;
  std::condition_variable cv_job, cv_done;
  std::function<int(int)> job;       // member -> status
  uint64_t generation = 0;
  int participants = 0;              // members taking part in the current job (the first `participants`)
  int pending = 0;
  bool quit = false;
  std::vector<int> rc;
  std::string err;
  uint64_t min_frames_per_member = 16384;
};

namespace {

void worker_main(ccgpu_group *g, int member) {
  uint64_t seen = 0;
  for (;;) {
    std::function<int(int)> job;
    {
      std::unique_lock<std::mutex> lk(g->mu);
      g->cv_job.wait(lk, [&] { return g->quit || (g->generation != seen && member < g->participants); });
      if (g->quit) return;
      seen = g->generation;
      job = g->job;
    }
    const int rc = job(member);
    {
      std::lock_guard<std::mutex> lk(g->mu);
      g->rc[member] = rc;
      if (--g->pending == 0) g->cv_done.notify_all();
    }
  }
}

// run job(member) on the first `participants` members; member 0 on the calling thread.  Returns the first error.
int run(ccgpu_group *g, int participants, std::function<int(int)> job) {
  if (participants > 1) {
    std::lock_guard<std::mutex> lk(g->mu);
    g->job = job;
    g->participants = participants;
    g->pending = participants - 1;
    ++g->generation;
    g->cv_job.notify_all();
  }
  g->rc[0] = job(0);
  if (participants > 1) {
    std::unique_lock<std::mutex> lk(g->mu);
    g->cv_done.wait(lk, [&] { return g->pending == 0; });
    g->participants = 0;
  }
  for (int m = 0; m < participants; ++m)
    if (g->rc[m] != CCGPU_OK) {
      g->err = std::string("member ") + std::to_string(m) + " (device " + std::to_string(g->device[m]) + "): " +
               ccgpu_last_error(g->ctx[m]);
      return g->rc[m];
    }
  return CCGPU_OK;
}

int members_for(const ccgpu_group *g, uint64_t units) {
  const uint64_t want = units / g->min_frames_per_member;
  const uint64_t n = g->ctx.size();
  return static_cast<int>(want < 1 ? 1 : (want > n ? n : want));
}

// contiguous shard of [0, total) for member m of `parts`
void shard(uint64_t total, int parts, int m, uint64_t *off, uint64_t *cnt) {
  const uint64_t base = total / parts, rem = total % parts;
  *off = base * m + (static_cast<uint64_t>(m) < rem ? m : rem);
  *cnt = base + (static_cast<uint64_t>(m) < rem ? 1 : 0);
}

void add(ccgpu_counters *acc, const ccgpu_counters &c) {
  acc->frames += c.frames;
  acc->frame_errors += c.frame_errors;
  acc->bit_errors += c.bit_errors;
  acc->iterations += c.iterations;
  acc->failures += c.failures;
  acc->undetected += c.undetected;
}

int fail(ccgpu_group *g, int code, const char *msg) {
  if (g) g->err = msg;
  return code;
}

// the common shape of every sharded Monte-Carlo point: fn(member, first unit, units, partial counters)
int sharded_point(ccgpu_group *g, uint64_t units, ccgpu_counters *out,
                  const std::function<int(int, uint64_t, uint64_t, ccgpu_counters *)> &fn) {
  if (!g || !out) return fail(g, CCGPU_ERR_INVALID, "null argument");
  std::lock_guard<std::mutex> call(g->call_mu);
  const int parts = members_for(g, units);
  std::vector<ccgpu_counters> partial(parts);
  std::memset(partial.data(), 0, sizeof(ccgpu_counters) * parts);
  const int rc = run(g, parts, [&](int m) {
    uint64_t off, cnt;
    shard(units, parts, m, &off, &cnt);
    return fn(m, off, cnt, &partial[m]);
  });
  if (rc != CCGPU_OK) return rc;
  std::memset(out, 0, sizeof(*out));
  for (int m = 0; m < parts; ++m) add(out, partial[m]);
  return CCGPU_OK;
}

}  // namespace

extern "C" {

int ccgpu_group_create(int n_devices, const int *devices, ccgpu_group **out) {
  if (!out || n_devices < 1 || n_devices > 64) return CCGPU_ERR_INVALID;
  *out = nullptr;
  ccgpu_group *g = new (std::nothrow) ccgpu_group();
  if (!g) return CCGPU_ERR_CUDA;
  for (int i = 0; i < n_devices; ++i) {
    ccgpu_ctx *c = nullptr;
    const int dev = devices ? devices[i] : i;
    const int rc = ccgpu_create(dev, &c);
    if (rc != CCGPU_OK) {
      for (ccgpu_ctx *x : g->ctx) ccgpu_destroy(x);
      delete g;
      return rc;
    }
    g->ctx.push_back(c);
    g->device.push_back(dev);
  }
  g->rc.assign(n_devices, CCGPU_OK);
  try {
    for (int m = 1; m < n_devices; ++m) g->workers.emplace_back(worker_main, g, m);
  } catch (...) {
    ccgpu_group_destroy(g);
    return CCGPU_ERR_CUDA;
  }
  *out = g;
  return CCGPU_OK;
}

void ccgpu_group_destroy(ccgpu_group *g) {
  if (!g) return;
  {
    std::lock_guard<std::mutex> lk(g->mu);
    g->quit = true;
    g->cv_job.notify_all();
  }
  for (std::thread &t : g->workers)
    if (t.joinable()) t.join();
  for (ccgpu_ctx *c : g->ctx) ccgpu_destroy(c);
  delete g;
}

int ccgpu_group_size(const ccgpu_group *g) { return g ? static_cast<int>(g->ctx.size()) : 0; }

ccgpu_ctx *ccgpu_group_ctx(const ccgpu_group *g, int member) {
  return (g && member >= 0 && member < static_cast<int>(g->ctx.size())) ? g->ctx[member] : nullptr;
}

const char *ccgpu_group_last_error(const ccgpu_group *g) {
  thread_local std::string copy;
  copy = g ? g->err : std::string("no group");
  return copy.c_str();
}

int ccgpu_group_set_min_frames(ccgpu_group *g, uint64_t frames_per_member) {
  if (!g || frames_per_member == 0) return CCGPU_ERR_INVALID;
  std::lock_guard<std::mutex> call(g->call_mu);
  g->min_frames_per_member = frames_per_member;
  return CCGPU_OK;
}

int ccgpu_group_awgn_point(ccgpu_group *g, ccgpu_code *const *codes, const ccgpu_ms_params *params, double ebno_db,
                           uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!codes || !params) return fail(g, CCGPU_ERR_INVALID, "null argument");
  return sharded_point(g, frames, out, [&](int m, uint64_t off, uint64_t cnt, ccgpu_counters *c) {
    return ccgpu_awgn_point(g->ctx[m], codes[m], params, ebno_db, seed, point, frame0 + off, cnt, c);
  });
}

int ccgpu_group_awgn_point_hard(ccgpu_group *g, ccgpu_code *const *codes, double ebno_db, uint64_t seed, uint32_t point,
                                uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!codes) return fail(g, CCGPU_ERR_INVALID, "null argument");
  return sharded_point(g, frames, out, [&](int m, uint64_t off, uint64_t cnt, ccgpu_counters *c) {
    return ccgpu_awgn_point_hard(g->ctx[m], codes[m], ebno_db, seed, point, frame0 + off, cnt, c);
  });
}

int ccgpu_group_awgn_point_chase(ccgpu_group *g, ccgpu_code *const *codes, uint32_t p, double ebno_db, uint64_t seed,
                                 uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!codes) return fail(g, CCGPU_ERR_INVALID, "null argument");
  return sharded_point(g, frames, out, [&](int m, uint64_t off, uint64_t cnt, ccgpu_counters *c) {
    return ccgpu_awgn_point_chase(g->ctx[m], codes[m], p, ebno_db, seed, point, frame0 + off, cnt, c);
  });
}

int ccgpu_group_awgn_point_osd(ccgpu_group *g, ccgpu_code *const *codes, uint32_t order, double ebno_db, uint64_t seed,
                               uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!codes) return fail(g, CCGPU_ERR_INVALID, "null argument");
  return sharded_point(g, frames, out, [&](int m, uint64_t off, uint64_t cnt, ccgpu_counters *c) {
    return ccgpu_awgn_point_osd(g->ctx[m], codes[m], order, ebno_db, seed, point, frame0 + off, cnt, c);
  });
}

int ccgpu_group_awgn_point_gmd(ccgpu_group *g, ccgpu_code *const *codes, uint32_t max_erasures, double ebno_db,
                               uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!codes) return fail(g, CCGPU_ERR_INVALID, "null argument");
  return sharded_point(g, frames, out, [&](int m, uint64_t off, uint64_t cnt, ccgpu_counters *c) {
    return ccgpu_awgn_point_gmd(g->ctx[m], codes[m], max_erasures, ebno_db, seed, point, frame0 + off, cnt, c);
  });
}

int ccgpu_group_awgn_point_abp(ccgpu_group *g, ccgpu_code *const *codes, uint32_t max_iter, double gamma, double ebno_db,
                               uint64_t seed, uint32_t point, uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!codes) return fail(g, CCGPU_ERR_INVALID, "null argument");
  return sharded_point(g, frames, out, [&](int m, uint64_t off, uint64_t cnt, ccgpu_counters *c) {
    return ccgpu_awgn_point_abp(g->ctx[m], codes[m], max_iter, gamma, ebno_db, seed, point, frame0 + off, cnt, c);
  });
}

int ccgpu_group_awgn_point_ml(ccgpu_group *g, ccgpu_code *const *codes, double ebno_db, uint64_t seed, uint32_t point,
                              uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!codes) return fail(g, CCGPU_ERR_INVALID, "null argument");
  return sharded_point(g, frames, out, [&](int m, uint64_t off, uint64_t cnt, ccgpu_counters *c) {
    return ccgpu_awgn_point_ml(g->ctx[m], codes[m], ebno_db, seed, point, frame0 + off, cnt, c);
  });
}

int ccgpu_group_awgn_point_mbbp(ccgpu_group *g, ccgpu_code *const *codes, const ccgpu_ms_params *params,
                                const uint32_t *shifts, uint32_t n_bases, double ebno_db, uint64_t seed, uint32_t point,
                                uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  if (!codes || !params || !shifts) return fail(g, CCGPU_ERR_INVALID, "null argument");
  return sharded_point(g, frames, out, [&](int m, uint64_t off, uint64_t cnt, ccgpu_counters *c) {
    return ccgpu_awgn_point_mbbp(g->ctx[m], codes[m], params, shifts, n_bases, ebno_db, seed, point, frame0 + off, cnt, c);
  });
}

int ccgpu_group_awgn_point_uncoded(ccgpu_group *g, uint32_t n, double rate, double ebno_db, uint64_t seed, uint32_t point,
                                   uint64_t frame0, uint64_t frames, ccgpu_counters *out) {
  return sharded_point(g, frames, out, [&](int m, uint64_t off, uint64_t cnt, ccgpu_counters *c) {
    return ccgpu_awgn_point_uncoded(g->ctx[m], n, rate, ebno_db, seed, point, frame0 + off, cnt, c);
  });
}

int ccgpu_group_bitflip_point(ccgpu_group *g, ccgpu_code *const *codes, const ccgpu_ms_params *params, uint32_t weight,
                              uint64_t first, uint64_t count, ccgpu_counters *out) {
  if (!g || !codes || !params) return fail(g, CCGPU_ERR_INVALID, "null argument");
  ccgpu_code_info info;
  if (ccgpu_code_get_info(codes[0], &info) != CCGPU_OK) return fail(g, CCGPU_ERR_INVALID, "bad code");
  if (weight > info.n) return fail(g, CCGPU_ERR_INVALID, "weight > n");
  long double total = 1;
  for (unsigned i = 1; i <= weight; ++i) total = total * (info.n - weight + i) / i;
  if (total > 1.8e19L) return fail(g, CCGPU_ERR_UNSUPPORTED, "C(n, weight) does not fit 64 bits");
  const uint64_t patterns = static_cast<uint64_t>(total + 0.5L);
  if (first > patterns) return fail(g, CCGPU_ERR_INVALID, "first > C(n, weight)");
  if (count == 0 || count > patterns - first) count = patterns - first;
  if (count == 0) {
    std::memset(out, 0, sizeof(*out));
    return CCGPU_OK;
  }
  return sharded_point(g, count, out, [&](int m, uint64_t off, uint64_t cnt, ccgpu_counters *c) {
    return cnt ? ccgpu_bitflip_point(g->ctx[m], codes[m], params, weight, first + off, cnt, c) : CCGPU_OK;
  });
}

// batched decoding with HOST buffers, frames sharded over the members (device pointers belong to one device:
// use that member's context directly)
int ccgpu_group_decode_llr(ccgpu_group *g, ccgpu_code *const *codes, const ccgpu_ms_params *params, const float *y,
                           uint64_t frames, uint8_t *bits, float *L, uint8_t *iter, uint8_t *failed) {
  if (!g || !codes || !params || !y || !bits || !failed) return fail(g, CCGPU_ERR_INVALID, "null argument");
  ccgpu_code_info info;
  if (ccgpu_code_get_info(codes[0], &info) != CCGPU_OK) return fail(g, CCGPU_ERR_INVALID, "bad code");
  const uint64_t n = info.n;
  std::lock_guard<std::mutex> call(g->call_mu);
  const int parts = members_for(g, frames);
  return run(g, parts, [&](int m) {
    uint64_t off, cnt;
    shard(frames, parts, m, &off, &cnt);
    return ccgpu_decode_llr(g->ctx[m], codes[m], params, y + off * n, cnt, bits + off * n, L ? L + off * n : nullptr,
                            iter ? iter + off : nullptr, failed + off);
  });
}

int ccgpu_group_gf_decode(ccgpu_group *g, ccgpu_code *const *codes, const uint8_t *words, uint64_t count, uint8_t *corrected,
                          uint8_t *n_errors, uint8_t *failed) {
  if (!g || !codes || !words || !corrected || !failed) return fail(g, CCGPU_ERR_INVALID, "null argument");
  ccgpu_code_info info;
  if (ccgpu_code_get_info(codes[0], &info) != CCGPU_OK) return fail(g, CCGPU_ERR_INVALID, "bad code");
  const uint64_t n = info.n;
  std::lock_guard<std::mutex> call(g->call_mu);
  const int parts = members_for(g, count);
  return run(g, parts, [&](int m) {
    uint64_t off, cnt;
    shard(count, parts, m, &off, &cnt);
    return ccgpu_gf_decode(g->ctx[m], codes[m], words + off * n, cnt, corrected + off * n, n_errors ? n_errors + off : nullptr,
                           failed + off);
  });
}

}  // extern "C"
