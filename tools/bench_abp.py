#!/usr/bin/env python
"""tools/bench_abp.py -- adaptive belief propagation (K8 abp_kernel) on one GPU: rates and word-error rates, one JSON
line per configuration, plus a first line naming the card and its power limit.

    python tools/bench_abp.py [--frames 4194304] [--out FILE]

Per (code, Eb/N0, max_iter, gamma):
  resident_frames_per_s   ccgpu_decode_llr_abp on device-resident channel values (frames x n float32, larger than the
                          126 MB L2 at the default size; bits, L, iter and failed written), CUDA events around one
                          launch after a warm-up launch
  fused_frames_per_s      ccgpu_awgn_point_abp over the same frames (channel drawn on chip, only counters leave)
  avg_updates             updates (check pass + soft update) per frame
  codeword_exit_share     share of frames whose hard decision is already a codeword (zero updates)
  failed_share, undetected_share   frames that never passed the stop test / passed it on a wrong codeword
  wer_abp / wer_nms / wer_hard / wer_chase4 / wer_chase8 / wer_osd1 / wer_osd2   the same frames (seed, point) through
                          ABP, NMS 0.8 on H, ccgpu_awgn_point_hard, Chase-II with p = 4 and 8, OSD-1 and OSD-2
  ml_lower_bound          frames whose OSD-2 word is nonzero and strictly closer to y than the all-zero word sent, over
                          frames: ML decoding errs on every such frame (as tools/bench_osd.py)
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_osd import card  # noqa: E402

# (q, t, Eb/N0, ((max_iter, gamma), ..)): BCH(63,36), BCH(127,64), BCH(31,16)
SETTINGS_63 = ((20, 0.1), (50, 0.15), (50, 0.3))
CONFIGS = [(6, 5, 3.0, SETTINGS_63), (6, 5, 4.0, SETTINGS_63), (6, 5, 7.0, SETTINGS_63), (7, 10, 5.0, ((50, 0.15),)),
           (5, 3, 4.0, ((50, 0.15),))]
SEED, POINT = 1, 3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1 << 22)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    import torch
    import channelcoding_b200 as cc
    if not torch.cuda.is_available():
        raise SystemExit("bench_abp.py measures on a CUDA device; none is available")
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

    for q, t, ebno, settings in CONFIGS:
        code = ctx.bch(q, errors=t)
        n = code.n
        name = code.to_string("ABP")[:-len("-ABP")]
        y = torch.empty((F, n), dtype=torch.float32, device="cuda")
        ctx.awgn_llr(n, cc.sigma(code.rate, ebno), SEED, POINT, 0, F, out=y)
        h = y < 0
        absy = y.abs()
        d_zero = torch.where(h, absy, torch.zeros_like(absy)).sum(dim=1)
        bits = torch.empty((F, n), dtype=torch.uint8, device="cuda")
        weight = torch.empty(F, dtype=torch.uint8, device="cuda")
        code.decode_osd(y, 2, out=(bits, weight))
        d_osd = torch.where(bits.bool() != h, absy, torch.zeros_like(absy)).sum(dim=1)
        ml = int((bits.bool().any(dim=1) & (d_osd < d_zero)).sum())
        del d_osd, weight
        others = {"nms": code.awgn_point(ebno, F, "NMS", 0.8, seed=SEED, point=POINT),
                  "hard": code.awgn_point_hard(ebno, F, seed=SEED, point=POINT),
                  "chase4": code.awgn_point_chase(ebno, F, 4, seed=SEED, point=POINT),
                  "chase8": code.awgn_point_chase(ebno, F, 8, seed=SEED, point=POINT),
                  "osd1": code.awgn_point_osd(ebno, F, 1, seed=SEED, point=POINT),
                  "osd2": code.awgn_point_osd(ebno, F, 2, seed=SEED, point=POINT)}
        L = torch.empty((F, n), dtype=torch.float32, device="cuda")
        it = torch.empty(F, dtype=torch.uint8, device="cuda")
        failed = torch.empty(F, dtype=torch.uint8, device="cuda")
        for max_iter, gamma in settings:
            t_res = events(lambda: code.decode_abp(y, max_iter, gamma, out=(bits, L, it, failed)))
            exit_share = float((it == 0).float().mean())
            code.awgn_point_abp(ebno, min(F, 1 << 16), max_iter, gamma, seed=SEED, point=POINT)  # warm-up
            t0 = time.perf_counter()
            o = code.awgn_point_abp(ebno, F, max_iter, gamma, seed=SEED, point=POINT)
            t_fused = time.perf_counter() - t0
            rec = {"kind": "abp", "code": name, "ebno_db": ebno, "max_iter": max_iter, "gamma": gamma, "frames": F,
                   "resident_frames_per_s": F / t_res, "fused_frames_per_s": F / t_fused,
                   "avg_updates": o["iterations"] / F, "codeword_exit_share": exit_share,
                   "failed_share": o["failures"] / F, "undetected_share": o["undetected"] / F,
                   "wer_abp": o["frame_errors"] / F}
            rec.update({"wer_" + k: v["frame_errors"] / F for k, v in others.items()})
            rec["ml_lower_bound"] = ml / F
            rec["abp_frame_errors"] = o["frame_errors"]
            rec.update({k + "_frame_errors": v["frame_errors"] for k, v in others.items()})
            rec.update({"ml_errors": ml, "resident_s": t_res, "fused_s": t_fused, "gpu": lines[0]["gpu"]})
            lines.append(rec)
            print(json.dumps(rec), flush=True)
        del y, h, absy, d_zero, bits, L, it, failed
        torch.cuda.empty_cache()
    ctx.close()
    if a.out:
        with open(a.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
