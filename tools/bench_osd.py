#!/usr/bin/env python
"""tools/bench_osd.py -- ordered-statistics decoding (K6 osd_kernel) on one GPU: rates and word-error rates, one JSON
line per configuration, plus a first line naming the card and its power limit.

    python tools/bench_osd.py [--frames 4194304] [--out FILE]

Per (code, Eb/N0, order):
  resident_frames_per_s   ccgpu_decode_llr_osd on device-resident channel values (frames x n float32, larger than the
                          126 MB L2 at the default size), CUDA events around one launch after a warm-up launch
  fused_frames_per_s      ccgpu_awgn_point_osd over the same frames (channel drawn on chip, only counters leave)
  candidates_per_s        frames * N / resident time, N = sum over w <= order of C(l, w) candidates per frame (frames
                          whose hard decision is a codeword stop after the syndrome on chip)
  codeword_exit_share     share of frames whose hard decision is a codeword (the kernel's early exit)
  wer_osd / wer_chase4 / wer_chase8 / wer_hard / wer_nms   the same frames (seed, point) through OSD, Chase-II with
                          p = 4 and 8, ccgpu_awgn_point_hard and NMS 0.8
  ml_lower_bound          frames whose OSD word is nonzero and strictly closer to y than the all-zero word sent
                          (D < the sum of |y| over h), over frames: ML decoding errs on every such frame
"""
import argparse
import json
import os
import subprocess
import sys
import time
from math import comb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (q, t, Eb/N0, orders): BCH(63,36), BCH(127,64), BCH(31,16)
CONFIGS = [(6, 5, 4.0, (1, 2, 3)), (6, 5, 7.0, (1, 2, 3)), (7, 10, 5.0, (1, 2)), (5, 3, 4.0, (1, 2, 3))]
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
        raise SystemExit("bench_osd.py measures on a CUDA device; none is available")
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

    for q, t, ebno, orders in CONFIGS:
        code = ctx.bch(q, errors=t)
        n, l = code.n, round(code.rate * code.n)
        name = code.to_string("OSD")[:-len("-OSD")]
        y = torch.empty((F, n), dtype=torch.float32, device="cuda")
        ctx.awgn_llr(n, cc.sigma(code.rate, ebno), SEED, POINT, 0, F, out=y)
        h = y < 0
        absy = y.abs()
        # D of the all-zero word; compared only with D of the OSD word summed the same way
        d_zero = torch.where(h, absy, torch.zeros_like(absy)).sum(dim=1)
        bits = torch.empty((F, n), dtype=torch.uint8, device="cuda")
        weight = torch.empty(F, dtype=torch.uint8, device="cuda")
        code.decode_osd(y, 0, out=(bits, weight))
        codeword_exit = float((bits.bool() == h).all(dim=1).float().mean())
        hard = code.awgn_point_hard(ebno, F, seed=SEED, point=POINT)
        nms = code.awgn_point(ebno, F, "NMS", 0.8, seed=SEED, point=POINT)
        ch4 = code.awgn_point_chase(ebno, F, 4, seed=SEED, point=POINT)
        ch8 = code.awgn_point_chase(ebno, F, 8, seed=SEED, point=POINT)
        for order in orders:
            N = sum(comb(l, w) for w in range(order + 1))
            t_res = events(lambda: code.decode_osd(y, order, out=(bits, weight)))
            d_osd = torch.where(bits.bool() != h, absy, torch.zeros_like(absy)).sum(dim=1)
            ml = int((bits.bool().any(dim=1) & (d_osd < d_zero)).sum())
            code.awgn_point_osd(ebno, min(F, 1 << 16), order, seed=SEED, point=POINT)  # warm-up
            t0 = time.perf_counter()
            o = code.awgn_point_osd(ebno, F, order, seed=SEED, point=POINT)
            t_fused = time.perf_counter() - t0
            rec = {"kind": "osd", "code": name, "ebno_db": ebno, "order": order, "candidates": N, "frames": F,
                   "resident_frames_per_s": F / t_res, "fused_frames_per_s": F / t_fused,
                   "candidates_per_s": F * N / t_res, "codeword_exit_share": codeword_exit,
                   "wer_osd": o["frame_errors"] / F, "wer_chase4": ch4["frame_errors"] / F,
                   "wer_chase8": ch8["frame_errors"] / F, "wer_hard": hard["frame_errors"] / F,
                   "wer_nms": nms["frame_errors"] / F, "ml_lower_bound": ml / F,
                   "osd_frame_errors": o["frame_errors"], "chase4_frame_errors": ch4["frame_errors"],
                   "chase8_frame_errors": ch8["frame_errors"], "hard_frame_errors": hard["frame_errors"],
                   "nms_frame_errors": nms["frame_errors"], "ml_errors": ml,
                   "resident_s": t_res, "fused_s": t_fused, "gpu": lines[0]["gpu"]}
            lines.append(rec)
            print(json.dumps(rec), flush=True)
        del y, h, absy, d_zero, bits, weight
        torch.cuda.empty_cache()
    ctx.close()
    if a.out:
        with open(a.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
