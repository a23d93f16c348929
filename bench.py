#!/usr/bin/env python
"""bench.py -- headline benchmark of the hot path (BASELINE.json): decoded frames/s and info-bits/s,
BCH(63,36) normalised min-sum (alpha = 0.8, <= 50 iterations, early exit), 1/2/4/8 B200 vs host CPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--ebno 4.0] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step is one pass of the hot path over one batch of synthetic AWGN frames (all-zero codeword, like
the reference's simulation).  Three measurements per run:
  value   frames/s of ccgpu_decode_llr with the LLR batch resident in HBM (device pointers), CUDA
          events on the launching stream, max over ranks.  The batch (1.06 GB) is far larger than L2.
  e2e     the same call through the C ABI with HOST buffers: pinned y in, bits/iter/failed out,
          H2D + decode + D2H inside the timed region.
  fused   ccgpu_awgn_point (the Monte-Carlo product path: Philox channel + decode + counters fused,
          only 64 bytes leave the GPU), followed by the one NCCL all-reduce of the counters.
The CPU baseline is the reference's own decoder (oracle/_ref/libccref.so = the reference compiled by
oracle/build_ref.sh) running simulation.c++'s inner loop on all host cores; if that library is absent,
the C restatement in oracle/ (kind "port").  The same holds for the CPU baselines of the other configurations.
--dump-outputs DIR writes what the last timed step of `value` returned (see dump_outputs) for output-for-output
comparisons of two builds.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

Q, T, ALPHA, MAX_ITER = 6, 5, 0.8, 50
N, L_INFO, ROWS, W = 63, 36, 27, 18
EDGES = ROWS * W
ALGO_BYTES_PER_FRAME = 4 * N + 4 * ((N + 31) // 32) + 4  # SURVEY.md 8(d): LLR in, packed decisions + status out
WORKLOAD = ("BCH(63,36) t=5 normalised min-sum alpha=0.8, <=50 iterations, early exit with the reference's stop rule, "
            "AWGN Eb/N0=%g dB, all-zero codeword")


def csrc_hash():
    """sha256 over the library's kernel / host sources -- the stamp tools/ncu_summary.py puts into every capture"""
    import hashlib
    root = os.path.join(ROOT, "channelcoding_b200", "csrc")
    h = hashlib.sha256()
    for name in sorted(os.listdir(root)):
        if name.endswith((".cu", ".cuh", ".h", ".hpp", ".cc")):
            h.update(name.encode())
            with open(os.path.join(root, name), "rb") as f:
                h.update(f.read())
    return h.hexdigest()[:16]


CAPTURE = os.path.join(ROOT, "profiles", "r2_kernels.json")


def ncu_capture(label):
    """the committed ncu record of one kernel (tools/profile_r2.py + tools/ncu_summary.py) -> (record, current?) where
    `current` says that the capture was taken from exactly the sources the library was built from"""
    try:
        with open(CAPTURE) as f:
            recs = json.load(f)
        rec = [r for r in recs if r.get("label") == label][0]
        return rec, rec.get("csrc_sha") == csrc_hash()
    except Exception:
        return None, False


DUMP_FRAMES = 1 << 17  # 131072 frames x 63 decisions as float32 = 33 MB: a dump stays a few tens of MB at any --frames


def dump_outputs(path, out, np, torch):
    """what the timed decode returned to its caller in its last step -- decided bits (frames, n), iteration index and
    failure flag per frame -- for a fixed, seeded sample of the batch's frames, as float32 .npy files under `path`
    (frame_index.npy, float64, names the sampled frames).  The LLR batch is seeded too, so two builds run with the same
    arguments can be compared output for output."""
    bits, _, it, failed = out
    B = bits.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(B, min(B, DUMP_FRAMES), replace=False))
    sel = torch.from_numpy(idx).to(bits.device)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "frame_index.npy"), idx.astype(np.float64))
    for name, t in (("bits", bits), ("iterations", it), ("failed", failed)):
        np.save(os.path.join(path, name + ".npy"), t[sel].cpu().numpy().astype(np.float32))


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p.get("sm_max_mhz", 1965.0)), "measured"
    except Exception:
        return 6650.0, 1965.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)"""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_port_point(q, errors, variant_id, ebno, seconds, frames_per_thread=0, threads=None):
    """the C restatement in oracle/ standing in for the reference's soft decoder `variant_id` (ids of oracle/ccref.py) of
    BCH(2^q - 1, t = errors) where the reference library is not built: one python thread per core (ctypes releases the
    GIL) -> (frames, word_errors, seconds)"""
    import numpy as np
    import oracle
    from ccref import VARIANT_PARAMS
    from concurrent.futures import ThreadPoolExecutor
    variant, alpha, beta, max_iter = VARIANT_PARAMS[variant_id]
    threads = threads or (os.cpu_count() or 1)
    code = oracle.Code(0, q, errors)
    H = code.H()
    sig = oracle.sigma(code.rate, ebno)
    per = frames_per_thread or max(8, 12600 // code.n)  # 200 frames of BCH(63,36) between two looks at the clock

    def work(t):
        rng = np.random.default_rng(t)
        done = err = 0
        t0 = time.time()
        while True:
            y = (1 + sig * rng.standard_normal((per, code.n))).astype(np.float32)
            bits, _, _, failed = oracle.min_sum(H, y, variant, alpha, beta, max_iter)
            done += per
            err += int(((failed == 1) | bits.any(axis=1)).sum())
            if frames_per_thread or time.time() - t0 >= seconds:
                return done, err
    t0 = time.time()
    with ThreadPoolExecutor(threads) as ex:
        res = list(ex.map(work, range(threads)))
    return sum(r[0] for r in res), sum(r[1] for r in res), time.time() - t0


def cpu_reference(ebno, seconds, frames_per_thread=0, seed=0):
    """the reference's CPU decoder on all host cores -> (frames/s, cores, kind, word_errors, frames)"""
    cores = os.cpu_count() or 1
    import ccref
    if ccref.available():
        ref = ccref.Ref()
        frames, werr, el = ref.awgn_baseline(ccref.FAM_BCH, Q, ccref.CAP_ERRORS, T, ccref.ALG_SOFT0 + ccref.V_NMS, ebno,
                                             seed=seed, seconds=seconds, threads=cores,
                                             max_frames_per_thread=frames_per_thread)
        return frames / el, cores, "reference", werr, frames
    frames, werr, el = cpu_port_point(Q, T, ccref.V_NMS, ebno, seconds, frames_per_thread, cores)
    return frames / el, cores, "port", werr, frames


def cpu_reference_point(q, errors, variant_id, ebno, seconds, threads=None):
    """cpu_baseline leg for the other configurations (tools/bench_extra.py calls this instead of touching oracle/
    itself): the reference's soft decoder `variant_id` (0 MS, 1 NMS, ...) of BCH(2^q - 1, t = errors) on the host
    cores -> (frames, word_errors, seconds) or None when the reference library is not built"""
    import ccref
    if not ccref.available():
        return None
    ref = ccref.Ref()
    return ref.awgn_baseline(ccref.FAM_BCH, q, ccref.CAP_ERRORS, errors, ccref.ALG_SOFT0 + variant_id, ebno, seed=0,
                             seconds=seconds, threads=threads or (os.cpu_count() or 1))


def cpu_reference_rs(q, errors, words):
    """cpu_baseline leg: the reference's Euklid decoder of RS(2^q - 1, t = errors) on one core -> words/s or None"""
    import ccref
    if not ccref.available():
        return None
    ref = ccref.Ref()
    t0 = time.perf_counter()
    ref.hard_correct(ccref.FAM_RS, q, ccref.CAP_ERRORS, errors, ccref.ALG_EUKLID, words)
    return len(words) / (time.perf_counter() - t0)


def cpu_port_rs(q, errors, words):
    """the C restatement's Euklid decoder (oracle/gf_oracle.c) where the reference library is not built -> words/s"""
    import oracle
    code = oracle.Code(oracle.FAM_RS, q, errors)
    t0 = time.perf_counter()
    code.hard_correct(words)
    return len(words) / (time.perf_counter() - t0)


def other_configs(ctx, torch, dist, np, world, rank, dev, timed, args):
    """the other BASELINE.json configurations (bench.py's headline is configs[1]), one short measurement each in the same
    run so that the driver's BENCH / SCALE records carry them: every rank works on its own frames (weak scaling, no
    data-path collective), CUDA events on the launching stream, max over ranks.  Rank 0 adds the reference's CPU decoder
    of the same code on the host cores (a few seconds each) and the roofline figures -> list of records"""
    hbm_peak, sm_max, which = measured_peaks()
    alu_peak = 148 * 128 * sm_max * 1e6
    out = []
    cnt = torch.zeros(8, dtype=torch.int64, device=dev)

    def point(config, kernel, code, ebno, frames, variant, alpha=0.8, stop=0, quant=None, steps=3, cpu=None, note=None):
        state = {"s": 0}
        pt = int(round(ebno * 2)) + 64

        def step():
            f0 = (state["s"] * world + rank) * frames
            code.awgn_point(ebno, frames, variant, alpha, 0.0, MAX_ITER, stop, seed=3, point=pt, frame0=f0, out=cnt, quant=quant)
            state["s"] += 1
        cnt.zero_()
        ms = timed(step, steps, 1)
        c = cnt.clone()
        if world > 1:
            dist.all_reduce(c, op=dist.ReduceOp.SUM)
        c = c.cpu().numpy()
        done = int(c[0])
        value = world * frames * steps / (ms * 1e-3)
        iters = float(c[3]) / max(1, done)
        rec = {"config": config, "path": "ccgpu_awgn_point (Philox channel + decode + counters fused)", "kernel": kernel,
               "ebno_db": ebno, "variant": variant, "value": value, "unit": "frames/s", "info_bits_per_s": value * code.l,
               "ms_per_step": ms / steps, "frames_per_step_per_gpu": frames, "n_gpus": world,
               "wer": float(c[1]) / max(1, done), "ber": float(c[2]) / max(1, done) / code.n, "avg_iterations": iters,
               "edge_iterations_per_s": value * iters * code.edges,
               # SURVEY 8(d): the decoders are on-chip bound; HBM fraction as the contract asks, lane-op model beside it
               "roofline": {"bound": "hbm", "achieved": value / world * (4 * code.n + 4 * ((code.n + 31) // 32) + 4) / 1e9,
                            "peak": hbm_peak, "unit": "GB/s",
                            "frac": value / world * (4 * code.n + 4 * ((code.n + 31) // 32) + 4) / 1e9 / hbm_peak,
                            "traffic": 0, "note": "fused point: no LLR ever reaches HBM; bytes are what the streaming "
                                                  "form of the same decode would move"},
               "alu": {"model": "avg_iters*(11E+2n) lane-ops/frame (SURVEY 8d)",
                       "frac": value / world * iters * (11 * code.edges + 2 * code.n) / alu_peak}}
        if note:
            rec["note"] = note
        if rank == 0 and cpu is not None and not args.no_cpu:
            r, kind = cpu_reference_point(*cpu, ebno, 3.0), "reference"
            if r is None:
                r, kind = cpu_port_point(*cpu, ebno, 3.0), "port"
            f, w, el = r
            rec["cpu_baseline"] = {"value": f / el, "unit": "frames/s", "cores": os.cpu_count(), "kind": kind,
                                   "sample": "3 s wall = %d frames, WER %.4f" % (f, w / max(1, f))}
        out.append(rec)

    # ---- configs[0]: BCH(15,7) sum-product, Eb/N0 1..6 dB
    c15 = ctx.bch(4, errors=2)
    for eb in (1.0, 3.0, 6.0):
        point("configs[0] BCH(15,7) t=2 sum-product BP", "ms_cyclic_lane_kernel<bch_15_7, VN_SPA>", c15, eb, 1 << 24, "SPA", 1.0, stop=1,
              cpu=(4, 2, 0) if eb == 3.0 else None,
              note="the reference has no sum-product decoder: cpu_baseline is its min-sum decoder of the same code")
    # the same code with the reference's own decoder family (min-sum), the like-for-like line for its CPU baseline
    point("configs[0] BCH(15,7) t=2 min-sum (the reference's decoder of this code)", "ms_cyclic_lane_kernel<bch_15_7, VN_PLAIN>", c15, 3.0,
          1 << 25, "MS", 1.0, cpu=(4, 2, 0))
    # ---- configs[2]: BCH(127,64), H(), redundant H (127 cyclic shifts), multiple bases
    c127 = ctx.bch(7, errors=10)
    point("configs[2] BCH(127,64) t=10 NMS on H() (63 rows)", "ms_cyclic_kernel<bch_127_64, VN_PLAIN>", c127, 5.0, 1 << 20, "NMS",
          cpu=(7, 10, 1))
    point("configs[2] BCH(127,64) t=10 NMS_Q on H() (63 rows)", "ms_cyclic_q_kernel<bch_127_64>", c127, 5.0, 1 << 20, "NMS_Q",
          quant=(8.0, 31, 31))
    c127.set_rows(127)
    point("configs[2] BCH(127,64) t=10 NMS on the redundant H (127 cyclic-shift rows)",
          "ms_cyclic_cta_kernel<bch_127_64_red_cta, VN_PLAIN>", c127, 5.0, 1 << 19, "NMS", stop=1)
    point("configs[2] BCH(127,64) t=10 NMS_Q on the redundant H (127 cyclic-shift rows)",
          "ms_cyclic_cta_q_kernel<bch_127_64_red_cta>", c127, 5.0, 1 << 19, "NMS_Q", stop=1, quant=(8.0, 31, 31))
    c127.set_rows(63)
    nb, fr = 8, 1 << 18
    shifts = [(127 * i) // nb for i in range(nb)]
    state = {"s": 0, "c": None}

    def step_mbbp():
        state["c"] = c127.awgn_point_mbbp(5.0, fr, shifts, "NMS", 0.8, stop_rule=1, seed=3, point=99,
                                          frame0=(state["s"] * world + rank) * fr)
        state["s"] += 1
    ms = timed(step_mbbp, 3, 1)
    c = state["c"]
    out.append({"config": "configs[2] BCH(127,64) t=10 NMS, 8 bases (rotations of H), best converged candidate kept",
                "path": "ccgpu_awgn_point_mbbp (channel kernel -> rotate -> decode -> select -> count)",
                "kernel": "ms_cyclic_kernel<bch_127_64, VN_PLAIN> on 8 x frames candidates", "ebno_db": 5.0, "variant": "NMS",
                "value": world * fr * 3 / (ms * 1e-3), "unit": "frames/s", "candidate_decodes_per_s": nb * world * fr * 3 / (ms * 1e-3),
                "ms_per_step": ms / 3, "frames_per_step_per_gpu": fr, "n_gpus": world,
                "wer": c["frame_errors"] / max(1, c["frames"]), "wer_note": "last step of rank 0"})
    # ---- configs[4]: BCH(255,131) NMS
    c255 = ctx.bch(8, errors=18)
    point("configs[4] BCH(255,131) t=18 NMS", "ms_cyclic_cta_kernel<bch_255_131_cta, VN_PLAIN>", c255, 6.0, 1 << 18, "NMS",
          cpu=(8, 18, 1))
    point("configs[4] BCH(255,131) t=18 NMS", "ms_cyclic_cta_kernel<bch_255_131_cta, VN_PLAIN>", c255, 8.0, 1 << 20, "NMS")
    point("configs[4] BCH(255,131) t=18 NMS_Q", "ms_cyclic_cta_q_kernel<bch_255_131_cta>", c255, 6.0, 1 << 18, "NMS_Q",
          quant=(8.0, 31, 29))
    # ---- configs[3]: RS(255,223), 1e7 codewords over the job (at least 2.5e6 per GPU), 0..17 symbol errors
    rs = ctx.rs(8, 16)
    count = max(10_000_000 // world, 2_500_000)
    rng = np.random.default_rng(5)
    base = 4096
    words = rs.encode(rng.integers(0, 256, size=(base, rs.l)).astype(np.uint8))
    bad = words.copy()
    ne = rng.integers(0, 18, size=base)
    for i in range(base):
        pos = rng.choice(255, ne[i], replace=False)
        bad[i, pos] ^= rng.integers(1, 256, size=ne[i]).astype(np.uint8)
    d_words = torch.from_numpy(bad).to(dev).repeat((count + base - 1) // base, 1)[:count].contiguous()
    o = (torch.empty_like(d_words), torch.empty(count, dtype=torch.uint8, device=dev), torch.empty(count, dtype=torch.uint8, device=dev))
    ms = timed(lambda: rs.gf_decode(d_words, out=o), 3, 1)
    ok = o[2][:base].cpu().numpy() == 0
    assert np.array_equal(o[0][:base].cpu().numpy()[ok], words[ok]) and ok[ne <= 16].all() and not ok[ne > 16].any()
    value = world * count * 3 / (ms * 1e-3)
    ncu_rec, current = ncu_capture("K4 gf_decode RS(255,223) 0..17 errors")
    wf = ncu_rec.get("smem_wavefronts_per_unit") if (ncu_rec and current) else None
    rec = {"config": "configs[3] RS(255,223) over GF(2^8) batched hard decode, 1e7 codewords, 0..17 symbol errors (t = 16)",
           "path": "ccgpu_gf_decode, words resident in HBM", "kernel": "gf_decode_kernel", "value": value, "unit": "codewords/s",
           "ms_per_step": ms / 3, "codewords_per_step_per_gpu": count, "n_gpus": world,
           "roofline": {"bound": "hbm", "achieved": value / world * 511 / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": value / world * 511 / 1e9 / hbm_peak, "bytes_per_codeword": 511,
                        "traffic": (ncu_rec.get("dram_bytes_per_unit") * count) if (ncu_rec and current and ncu_rec.get("dram_bytes_per_unit")) else None},
           # the pipe that binds: table lookups in shared memory, one wavefront per SM per cycle
           "smem": {"wavefronts_per_codeword": wf, "frac": (value / world * wf / (148 * sm_max * 1e6)) if wf else None,
                    "capture": "profiles/r2_kernels.json" if (ncu_rec and current) else "no ncu capture of the current sources"}}
    del d_words, o
    # end to end: host buffers through the C ABI (chunked H2D / decode / D2H pipeline)
    nh = count // 4
    h_words = torch.from_numpy(bad).repeat((nh + base - 1) // base, 1)[:nh].contiguous().pin_memory()
    h_out = (torch.empty((nh, 255), dtype=torch.uint8).pin_memory().numpy(), torch.empty(nh, dtype=torch.uint8).pin_memory().numpy(),
             torch.empty(nh, dtype=torch.uint8).pin_memory().numpy())
    hw = h_words.numpy()
    rs.gf_decode(hw, out=h_out)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        rs.gf_decode(hw, out=h_out)
    el = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    rec["e2e"] = {"value": world * nh * 3 / float(el.item()), "unit": "codewords/s", "h2d_bytes_per_step": nh * 255,
                  "d2h_bytes_per_step": nh * 257, "path": "ccgpu_gf_decode with pinned host buffers"}
    if rank == 0 and not args.no_cpu:
        r, kind = cpu_reference_rs(8, 16, bad[:2048]), "reference"
        if r is None:
            r, kind = cpu_port_rs(8, 16, bad[:2048]), "port"
        rec["cpu_baseline"] = {"value": r, "unit": "codewords/s", "cores": 1, "kind": kind,
                               "sample": "2048 of the same words, euklid_tag, one thread (x %d cores = %.3g if every core ran one)"
                                         % (os.cpu_count(), r * os.cpu_count())}
    out.append(rec)
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_thread = 1000  # frames per thread per step: a bounded sample of the workload (0.6 s per step here)
    for _ in range(args.warmup):
        cpu_reference(args.ebno, 1e9, per_thread)
    t0 = time.time()
    frames = werr = 0
    for step in range(args.steps):
        rate, cores, kind, e, f = cpu_reference(args.ebno, 1e9, per_thread, seed=1 + step)  # fresh noise every step
        frames += f
        werr += e
    el = time.time() - t0
    value = frames / el
    line = {
        "impl": "reference", "metric": "decoded frames/s, BCH(63,36) normalised min-sum", "value": value,
        "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD % args.ebno, "ebno_db": args.ebno,
                   "frames_per_step": frames // max(1, args.steps)},
        "info_bits_per_s": value * L_INFO, "wer": werr / max(1, frames),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": kind,
                         "sample": "%d frames per thread per step, %d threads, simulation.c++ inner loop incl. noise "
                                   "generation" % (per_thread, cores)},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--ebno", type=float, default=4.0)
    ap.add_argument("--frames", type=int, default=1 << 22, help="frames per step per GPU (resident batch)")
    ap.add_argument("--e2e-frames", type=int, default=1 << 22, help="frames per step per GPU for the host-buffer path")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the table of the other BASELINE.json configurations")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (a fixed sample of frames) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    # stdout carries exactly ONE line, the JSON record.  Native libraries write to file descriptor 1 behind Python's
    # back (NCCL prints its version banner there whatever NCCL_DEBUG_FILE says): keep a private handle on the real
    # stdout for the record and point descriptor 1 at stderr for everything else.  The log LEVEL (NCCL_DEBUG) stays the
    # caller's -- the driver counts the ranks from that log, which now arrives on stderr in full.
    sys.stdout.flush()
    record_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    import numpy as np
    import torch
    import torch.distributed as dist
    import channelcoding_b200 as cc

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL logs to stdout by default: route it to stderr so that stdout stays the one JSON line; the log LEVEL
        # (NCCL_DEBUG) is left to the caller -- the driver counts the ranks from it
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx = cc.Context(local)
    ctx.use_torch_stream()
    code = ctx.bch(Q, errors=T)
    assert (code.n, code.l, code.h_rows, code.row_weight, code.kernel) == (N, L_INFO, ROWS, W, 1)
    B = args.frames
    sig = cc.sigma(code.rate, args.ebno)
    dev = torch.device("cuda", local)
    y = torch.empty((B, N), dtype=torch.float32, device=dev)
    ctx.awgn_llr(N, np.float32(sig), seed=0, point=int(round(args.ebno * 2)), frame0=rank * B, frames=B, out=y)
    out = (torch.empty((B, N), dtype=torch.uint8, device=dev), None, torch.empty(B, dtype=torch.uint8, device=dev),
           torch.empty(B, dtype=torch.uint8, device=dev))

    def step_resident():
        code.decode(y, "NMS", ALPHA, 0.0, MAX_ITER, out=out, want_L=False)

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ctx.kernel_launches
    ms_res = timed(step_resident, args.steps, args.warmup)
    launches = ctx.kernel_launches - launches0 - args.warmup
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / (ms_res * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, np, torch)

    # iteration statistics of the batch (for the ALU model and the log)
    it = out[2].to(torch.int64)
    failed = out[3].to(torch.int64)
    iters_exec = torch.where(failed == 1, torch.full_like(it, MAX_ITER), it + 1).double().mean().item()
    wer = ((failed == 1) | (out[0].sum(dim=1) > 0)).double().mean().item()

    # ---- e2e: host buffers through the C ABI
    Be = args.e2e_frames
    y_host = torch.empty((Be, N), dtype=torch.float32).pin_memory()
    y_host.copy_(y[:Be])
    h_bits = torch.empty((Be, N), dtype=torch.uint8).pin_memory()
    h_it = torch.empty(Be, dtype=torch.uint8).pin_memory()
    h_fail = torch.empty(Be, dtype=torch.uint8).pin_memory()
    e2e_out = (h_bits.numpy(), None, h_it.numpy(), h_fail.numpy())
    y_np = y_host.numpy()

    def step_e2e():
        code.decode(y_np, "NMS", ALPHA, 0.0, MAX_ITER, out=e2e_out, want_L=False)

    e2e_steps = max(3, args.steps // 2)
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()  # returns after the results are in the host buffers
    torch.cuda.synchronize()
    el = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    e2e_value = world * Be * e2e_steps / float(el.item())
    assert np.array_equal(h_fail.numpy(), out[3][:Be].cpu().numpy())

    # ---- the same end-to-end call with the compact output layout (ccgpu_decode_llr_packed: 8 B of decided bits + one
    # status byte per frame instead of 63 + 2): the device->host direction shrinks 7x, the input copy is unchanged
    h_packed = torch.empty((Be, (N + 31) // 32), dtype=torch.int32).pin_memory()
    h_status = torch.empty(Be, dtype=torch.uint8).pin_memory()
    packed_out = (h_packed.numpy().view(np.uint32), h_status.numpy())

    def step_e2e_packed():
        code.decode_packed(y_np, "NMS", ALPHA, 0.0, MAX_ITER, out=packed_out)

    for _ in range(2):
        step_e2e_packed()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e_packed()
    torch.cuda.synchronize()
    elp = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(elp, op=dist.ReduceOp.MAX)
    e2e_packed_value = world * Be * e2e_steps / float(elp.item())
    st = h_status.numpy()
    assert np.array_equal(st == 255, h_fail.numpy() == 1) and np.array_equal(st[st != 255], h_it.numpy()[st != 255])

    # ---- host-side ceiling of the e2e path: the same pinned buffer copied to the device and nothing else, all ranks at once
    d_copy = torch.empty((Be, N), dtype=torch.float32, device=dev)
    for _ in range(2):
        d_copy.copy_(y_host, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        d_copy.copy_(y_host, non_blocking=True)
    torch.cuda.synchronize()
    elc = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(elc, op=dist.ReduceOp.MAX)
    h2d_ceiling = world * Be * N * 4 * e2e_steps / float(elc.item()) / 1e9   # GB/s over all ranks
    del d_copy

    # ---- the fixed-point decoder (CCGPU_NMS_Q, two frames per lane) on the same resident batch; its decisions are those
    # of its own integer restatement, NOT the reference's float decoder, so it is reported next to the headline, not as it
    QUANT = (8.0, 31, 31)

    def step_fixed():
        code.decode(y, "NMS_Q", ALPHA, 0.0, MAX_ITER, out=out_q, want_L=False, quant=QUANT)

    out_q = (torch.empty((B, N), dtype=torch.uint8, device=dev), None, torch.empty(B, dtype=torch.uint8, device=dev),
             torch.empty(B, dtype=torch.uint8, device=dev))
    ms_fix = timed(step_fixed, max(3, args.steps // 2), args.warmup)
    fix_value = world * B * max(3, args.steps // 2) / (ms_fix * 1e-3)
    itq = torch.where(out_q[3] == 1, torch.full_like(out_q[2], MAX_ITER).to(torch.int64), out_q[2].to(torch.int64) + 1).double().mean().item()
    werq = ((out_q[3] == 1) | (out_q[0].sum(dim=1) > 0)).double().mean().item()
    fixed = {"variant": "NMS_Q alpha=0.8, quantiser scale 8 / y_max 31 / msg_max 31", "value": fix_value, "unit": "frames/s",
             "wer": werq, "avg_iterations": itq, "edge_iterations_per_s": fix_value * itq * EDGES,
             "float_edge_iterations_per_s": value * iters_exec * EDGES,
             "speedup_frames": fix_value / value, "speedup_edge_iterations": fix_value * itq / (value * iters_exec),
             "path": "ccgpu_decode_llr, resident LLRs, same batch as `value`"}

    # ---- fused Monte-Carlo point + the one all-reduce of the counters
    counters = torch.zeros(8, dtype=torch.int64, device=dev)
    point = int(round(args.ebno * 2))
    state = {"step": 0}

    per_point = torch.zeros(8, dtype=torch.int64, device=dev)

    def step_fused():
        # one Eb/N0 point of the sweep as the product runs it: every rank decodes its share of the point's frames, then
        # the eight counters are merged (the next point's sample count depends on the merged WER, simulation.c++:91-93),
        # so the all-reduce belongs INSIDE the timed step
        f0 = (state["step"] * world + rank) * B
        per_point.zero_()
        code.awgn_point(args.ebno, B, "NMS", ALPHA, 0.0, MAX_ITER, seed=0, point=point, frame0=f0, out=per_point)
        if world > 1:
            dist.all_reduce(per_point, op=dist.ReduceOp.SUM)
        counters.add_(per_point)
        state["step"] += 1

    ms_fused = timed(step_fused, args.steps, args.warmup)
    cnt = counters.cpu().numpy()
    fused_value = world * B * args.steps / (ms_fused * 1e-3)

    table = None if args.no_configs else other_configs(ctx, torch, dist, np, world, rank, dev, timed, args)

    if rank == 0:
        hbm_peak, sm_max, which = measured_peaks()
        kernel_ms = ms_res / args.steps
        achieved = B * ALGO_BYTES_PER_FRAME / (kernel_ms * 1e-3) / 1e9
        lane_ops = iters_exec * (11 * EDGES + 2 * N)
        alu_peak = 148 * 128 * sm_max * 1e6
        rec, current = ncu_capture("K2 ms_cyclic BCH(63,36) NMS 4 dB resident")
        # per-frame counts of the committed capture are only used when it describes THIS library (source hash matches)
        wf_frame = rec.get("smem_wavefronts_per_unit") if (rec and current) else None
        ins_frame = rec.get("warp_instructions_per_unit") if (rec and current) else None
        traffic_frame = rec.get("dram_bytes_per_unit") if (rec and current) else None
        rec_p, current_p = ncu_capture("K2 ms_cyclic BCH(63,36) NMS 4 dB resident, compact outputs")
        traffic_packed = rec_p.get("dram_bytes_per_unit") if (rec_p and current_p) else None
        capture_note = ("profiles/r2_kernels.json, csrc_sha %s" % rec.get("csrc_sha")) if (rec and current) else \
                       "no ncu capture of the current sources (csrc_sha %s): per-frame pipe counts withheld" % csrc_hash()
        line = {
            "metric": "decoded frames/s, BCH(63,36) normalised min-sum", "value": value, "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": kernel_ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD % args.ebno, "ebno_db": args.ebno, "frames_per_step_per_gpu": B,
                       "resident_batch": "%d frames per step per GPU resident in HBM (%.2f GB of LLRs)"
                                         % (B, B * N * 4 / 1e9),
                       "l2": "inputs larger than L2",
                       "sharding": "frames split across ranks, no data-path collective"},
            "info_bits_per_s": value * L_INFO, "wer": wer, "avg_iterations": iters_exec,
            "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": Be * N * 4,
                    "d2h_bytes_per_step": Be * (N + 2), "frames_per_step_per_gpu": Be,
                    "path": "ccgpu_decode_llr with pinned host buffers",
                    # the input copy is the bound of this path (252 B/frame in, 65 B/frame out on the other direction)
                    "h2d_gbs": e2e_value * N * 4 / 1e9, "h2d_ceiling_gbs": h2d_ceiling,
                    "frac_of_h2d_ceiling": e2e_value * N * 4 / 1e9 / h2d_ceiling,
                    "ceiling": "the same pinned buffer copied host->device by every rank at once, nothing else running"},
            "e2e_packed": {"value": e2e_packed_value, "unit": "frames/s", "h2d_bytes_per_step": Be * N * 4,
                           "d2h_bytes_per_step": Be * (4 * ((N + 31) // 32) + 1),
                           "path": "ccgpu_decode_llr_packed with pinned host buffers (bit-packed decisions + status byte)",
                           "frac_of_h2d_ceiling": e2e_packed_value * N * 4 / 1e9 / h2d_ceiling},
            "fused_monte_carlo": {"value": fused_value, "unit": "frames/s", "ms_per_step": ms_fused / args.steps,
                                  "wer": float(cnt[1]) / max(1, int(cnt[0])),
                                  "avg_iterations": float(cnt[3]) / max(1, int(cnt[0])), "frames": int(cnt[0]),
                                  "path": "ccgpu_awgn_point (Philox channel + decode + counters on chip) + one NCCL "
                                          "all-reduce of the 8 counters per step, inside the timed region"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak,
                         "traffic": (traffic_frame * B if traffic_frame else None), "capture": capture_note,
                         # DRAM bytes per frame measured by ncu: `value`'s layout (one byte per decided bit, as the
                         # reference's correct() returns them) and the compact layout the 264 algorithmic bytes assume
                         "traffic_bytes_per_frame": traffic_frame, "traffic_bytes_per_frame_compact_outputs": traffic_packed,
                         "peak_source": which, "kernel": "ms_cyclic_kernel<Shape<63,27,...>, VN_PLAIN>",
                         "bytes_per_frame": ALGO_BYTES_PER_FRAME,
                         "note": "the decoder is on-chip ALU/shared-memory bound, not HBM bound: see alu"},
            "alu": {"model": "avg_iters*(11E+2n) lane-ops/frame (SURVEY 8d)", "lane_ops_per_frame": lane_ops,
                    "achieved_lane_ops_per_s": value / world * lane_ops, "peak_lane_ops_per_s": alu_peak,
                    "frac": value / world * lane_ops / alu_peak},
            # the pipes that actually bind (ncu, profiles/r2_kernels.txt: issue 80 %, ALU 77 %, LSU 81 %):
            # shared-memory wavefronts against one per SM per cycle, warp instructions against four per SM per cycle;
            # the per-frame counts come from the committed ncu capture of this kernel at the same Eb/N0
            "smem": {"wavefronts_per_frame": wf_frame, "peak_wavefronts_per_s": 148 * sm_max * 1e6,
                     "achieved_wavefronts_per_s": (value / world * wf_frame) if wf_frame else None,
                     "frac": (value / world * wf_frame / (148 * sm_max * 1e6)) if wf_frame else None},
            "issue": {"warp_instructions_per_frame": ins_frame, "peak_per_s": 4 * 148 * sm_max * 1e6,
                      "achieved_per_s": (value / world * ins_frame) if ins_frame else None,
                      "frac": (value / world * ins_frame / (4 * 148 * sm_max * 1e6)) if ins_frame else None},
            "fixed_point": fixed,
            "clocks": clocks,
        }
        if table is not None:
            line["baseline_configs"] = table
        if not args.no_cpu:
            rate, cores, kind, werr, frames = cpu_reference(args.ebno, args.cpu_seconds)
            line["cpu_baseline"] = {"value": rate, "unit": "frames/s", "cores": cores, "kind": kind,
                                    "sample": "%.0f s wall on %d threads = %d frames of the same workload "
                                              "(simulation.c++ inner loop incl. noise generation), WER %.4f"
                                              % (args.cpu_seconds, cores, frames, werr / max(1, frames))}
        record_out.write(json.dumps(line) + "\n")
        record_out.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
