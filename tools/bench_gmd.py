#!/usr/bin/env python
"""tools/bench_gmd.py -- GMD decoding of Reed-Solomon codes (K7 gmd_kernel) on one GPU: rates and word-error rates,
one JSON line per configuration, plus a first line naming the card, its power limit and its maximum SM clock.

    python tools/bench_gmd.py [--frames 1048576] [--out FILE]

Per (code, Eb/N0): one "k4" line
  k4_words_per_s          ccgpu_gf_decode (K4) of the hard symbols of the same frames, device-resident: the
                          hard-decision yardstick, CUDA events around one launch after a warm-up launch
  wer_closed_form         P(more than t of the n hard symbols wrong), p_s = 1 - (1 - Q(1/sigma))^q: the exact WER of
                          any bounded-distance decoder of the hard decision
and per F one "gmd" line
  resident_words_per_s    ccgpu_decode_llr_gmd on device-resident channel values (frames x n q float32, larger than
                          the 126 MB L2 at the default size), CUDA events around one launch after a warm-up launch
  fused_words_per_s       ccgpu_awgn_point_gmd over the same frames (channel drawn on chip, only counters leave), host
                          clock around the synchronous call after a warm-up call
  trial_decodes_per_s     frames * (F/2 + 1) / resident time (frames whose hard decision is a codeword stop after the
                          syndromes on chip, so this counts the trials the contract defines, not the ones run)
  wer_gmd                 frame errors of the fused point over frames (F = 0: the hard-decision decoder)
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (q, t, Eb/N0 points, F values): RS(255,223) and RS(15,9)
CONFIGS = [(8, 16, (5.5, 6.0), (0, 8, 16, 32)), (4, 3, (5.0, 7.0), (0, 2, 4, 6))]
SEED, POINT = 1, 5


def card():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = r.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def closed_form_wer(n, q, t, sigma):
    from scipy import special, stats
    pb = 0.5 * special.erfc(1.0 / (sigma * 2 ** 0.5))
    return float(stats.binom.sf(t, n, 1.0 - (1.0 - pb) ** q))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1 << 20)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    import numpy as np
    import torch
    import channelcoding_b200 as cc
    if not torch.cuda.is_available():
        raise SystemExit("bench_gmd.py measures on a CUDA device; none is available")
    lines = [dict(card(), kind="card")]
    print(json.dumps(lines[0]), flush=True)
    ctx = cc.Context(0)
    ctx.use_torch_stream()
    N = a.frames

    def events(fn):
        fn()  # warm-up with the timed shapes
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3

    def emit(rec):
        rec["gpu"] = lines[0]["gpu"]
        lines.append(rec)
        print(json.dumps(rec), flush=True)

    for q, t, ebnos, Fs in CONFIGS:
        code = ctx.rs(q, t)
        n = code.n
        name = code.to_string("GMD")[:-len("-GMD")]
        y = torch.empty((N, n * q), dtype=torch.float32, device="cuda")
        words = torch.empty((N, n), dtype=torch.uint8, device="cuda")
        failed = torch.empty(N, dtype=torch.uint8, device="cuda")
        chosen = torch.empty(N, dtype=torch.uint8, device="cuda")
        nerr = torch.empty(N, dtype=torch.uint8, device="cuda")
        shifts = torch.arange(q, dtype=torch.int32, device="cuda")
        for ebno in ebnos:
            sigma = float(np.float32(cc.sigma(code.rate, ebno)))
            ctx.awgn_llr(n * q, sigma, SEED, POINT, 0, N, out=y)
            r = ((y < 0).view(N, n, q).to(torch.int32) << shifts).sum(dim=2).to(torch.uint8)
            t_k4 = events(lambda: code.gf_decode(r, out=(words, nerr, failed)))
            k4_wer = float(((failed != 0) | (words != 0).any(dim=1)).float().mean())
            emit({"kind": "k4", "code": name, "ebno_db": ebno, "frames": N, "k4_words_per_s": N / t_k4, "k4_s": t_k4,
                  "wer_k4": k4_wer, "wer_closed_form": closed_form_wer(n, q, t, sigma)})
            for F in Fs:
                t_res = events(lambda: code.decode_gmd(y, F, out=(words, failed, chosen)))
                code.awgn_point_gmd(ebno, min(N, 1 << 16), F, seed=SEED, point=POINT)  # warm-up
                t0 = time.perf_counter()
                g = code.awgn_point_gmd(ebno, N, F, seed=SEED, point=POINT)
                t_fused = time.perf_counter() - t0
                emit({"kind": "gmd", "code": name, "ebno_db": ebno, "F": F, "trials": F // 2 + 1, "frames": N,
                      "resident_words_per_s": N / t_res, "fused_words_per_s": N / t_fused,
                      "trial_decodes_per_s": N * (F // 2 + 1) / t_res, "wer_gmd": g["frame_errors"] / N,
                      "gmd_frame_errors": g["frame_errors"], "failures": g["failures"], "undetected": g["undetected"],
                      "resident_s": t_res, "fused_s": t_fused})
        del y, r, words, failed, chosen, nerr
        torch.cuda.empty_cache()
    ctx.close()
    if a.out:
        with open(a.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
