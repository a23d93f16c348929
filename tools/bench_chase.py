#!/usr/bin/env python
"""tools/bench_chase.py -- Chase-II (K5 chase_kernel) on one GPU: rates and word-error rates, one JSON line per
configuration, plus a first line naming the card and its power limit.

    python tools/bench_chase.py [--frames 4194304] [--out FILE]

Per (code, Eb/N0, p):
  resident_frames_per_s   ccgpu_decode_llr_chase on device-resident channel values (frames x n float32, larger than the
                          126 MB L2 at the default size), CUDA events around the timed launch
  fused_frames_per_s      ccgpu_awgn_point_chase over the same frames (channel drawn on chip, only counters leave)
  pattern_decodes_per_s   frames * 2^p / resident time: the test patterns a composition of 2^p separate decodes would
                          have to run (frames whose hard decision has a zero syndrome stop after pattern 0 on chip)
  k4_words_per_s          the yardstick: K4 (ccgpu_gf_decode) on the hard-decided words of the same frames, device
                          resident -- a lower bound on the cost of ONE of the 2^p passes of Chase composed from today's
                          entry points (no test-word construction, no selection)
  wer_chase / wer_hard / wer_nms   the same frames (seed, point) through Chase-II, ccgpu_awgn_point_hard and NMS 0.8
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (q, t, Eb/N0, p values): BCH(63,36), BCH(127,64), BCH(255,131)
CONFIGS = [(6, 5, 4.0, (2, 4, 6, 8)), (6, 5, 7.0, (2, 4, 6, 8)), (7, 10, 5.0, (4, 8)), (8, 18, 6.0, (4, 8))]
SEED, POINT = 1, 3


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1 << 22)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    import torch
    import channelcoding_b200 as cc
    if not torch.cuda.is_available():
        raise SystemExit("bench_chase.py measures on a CUDA device; none is available")
    lines = [dict(card(), kind="card")]
    print(json.dumps(lines[0]), flush=True)
    ctx = cc.Context(0)
    ctx.use_torch_stream()
    F = a.frames

    def events(fn):
        fn()  # warm-up with the timed shapes
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 1e3

    for q, t, ebno, ps in CONFIGS:
        code = ctx.bch(q, errors=t)
        n = code.n
        name = code.to_string("CHASE")[:-len("-CHASE")]
        y = torch.empty((F, n), dtype=torch.float32, device="cuda")
        ctx.awgn_llr(n, cc.sigma(code.rate, ebno), SEED, POINT, 0, F, out=y)
        words = (y < 0).to(torch.uint8)
        corrected, nerr, fl = torch.empty_like(words), torch.empty(F, dtype=torch.uint8, device="cuda"), \
            torch.empty(F, dtype=torch.uint8, device="cuda")
        t_k4 = events(lambda: code.gf_decode(words, out=(corrected, nerr, fl)))
        zero_syndrome = float((fl == 0).logical_and((corrected == words).all(dim=1)).float().mean())
        del corrected, nerr, fl
        hard = code.awgn_point_hard(ebno, F, seed=SEED, point=POINT)
        nms = code.awgn_point(ebno, F, "NMS", 0.8, seed=SEED, point=POINT)
        bits = torch.empty((F, n), dtype=torch.uint8, device="cuda")
        failed, chosen = torch.empty(F, dtype=torch.uint8, device="cuda"), torch.empty(F, dtype=torch.uint8, device="cuda")
        for p in ps:
            t_res = events(lambda: code.decode_chase(y, p, out=(bits, failed, chosen)))
            code.awgn_point_chase(ebno, min(F, 1 << 16), p, seed=SEED, point=POINT)  # warm-up
            t0 = time.perf_counter()
            ch = code.awgn_point_chase(ebno, F, p, seed=SEED, point=POINT)
            t_fused = time.perf_counter() - t0
            rec = {"kind": "chase", "code": name, "ebno_db": ebno, "p": p, "frames": F,
                   "resident_frames_per_s": F / t_res, "fused_frames_per_s": F / t_fused,
                   "pattern_decodes_per_s": F * (1 << p) / t_res, "k4_words_per_s": F / t_k4,
                   "pattern_decodes_over_k4": (F * (1 << p) / t_res) / (F / t_k4),
                   "hard_zero_syndrome_share": zero_syndrome,
                   "wer_chase": ch["frame_errors"] / F, "wer_hard": hard["frame_errors"] / F, "wer_nms": nms["frame_errors"] / F,
                   "chase_frame_errors": ch["frame_errors"], "hard_frame_errors": hard["frame_errors"],
                   "nms_frame_errors": nms["frame_errors"], "chase_failures": ch["failures"],
                   "resident_s": t_res, "fused_s": t_fused, "k4_s": t_k4, "gpu": lines[0]["gpu"]}
            lines.append(rec)
            print(json.dumps(rec), flush=True)
        del y, words, bits, failed, chosen
        torch.cuda.empty_cache()
    ctx.close()
    if a.out:
        with open(a.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
