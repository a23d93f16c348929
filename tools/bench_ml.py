#!/usr/bin/env python
"""tools/bench_ml.py -- maximum-likelihood (Viterbi) decoding (K9 ml_kernel) on one GPU: rates and word-error rates, one
JSON line per configuration, plus a first line naming the card, its power limit and its maximum SM clock.

    python tools/bench_ml.py [--frames 4194304] [--out FILE]

Per (code, Eb/N0):
  resident_frames_per_s   ccgpu_decode_llr_ml on device-resident channel values (frames x n float32, larger than the
                          126 MB L2 for n = 63 at the default size; bits written), CUDA events around one launch after a
                          warm-up launch
  butterflies_per_s       frames * n * 2^(k-1) / resident time (every frame counted, codeword exits included)
  fused_frames_per_s      ccgpu_awgn_point_ml over the same frames (channel drawn on chip, only counters leave), host
                          clock around the synchronising call
  codeword_exit_share     share of frames whose hard decision is already a codeword (the zero-syndrome exit)
  wer_ml / wer_osd1..3 / wer_chase4 / wer_chase8 / wer_hard / wer_nms / wer_abp   the same frames (seed, point) through
                          ML, OSD-1/2/3, Chase-II with p = 4 and 8, ccgpu_awgn_point_hard (BM), NMS 0.8 on the k-row H
                          and ABP (20, 0.1), with the frame-error counts
  ml_lower_bound          frames whose OSD-3 word is nonzero and strictly closer to y than the all-zero word sent, over
                          frames (as tools/bench_osd.py); bound_frames_not_ml_errors counts such frames that ML decoded
                          to the all-zero word (none, when ML is exact)
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

# (q, t, Eb/N0): BCH(63,51) x 3, BCH(63,57), BCH(31,21), BCH(127,120), BCH(15,7)
CONFIGS = [(6, 2, 4.0), (6, 2, 5.0), (6, 2, 6.0), (6, 1, 5.0), (5, 2, 4.0), (7, 1, 6.0), (4, 2, 3.0)]
SEED, POINT = 1, 3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1 << 22)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    import torch
    import channelcoding_b200 as cc
    if not torch.cuda.is_available():
        raise SystemExit("bench_ml.py measures on a CUDA device; none is available")
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

    for q, t, ebno in CONFIGS:
        code = ctx.bch(q, errors=t)
        n, k = code.n, code.n - code.l
        name = code.to_string("ML")[:-len("-ML")]
        y = torch.empty((F, n), dtype=torch.float32, device="cuda")
        ctx.awgn_llr(n, cc.sigma(code.rate, ebno), SEED, POINT, 0, F, out=y)
        h = y < 0
        absy = y.abs()
        bits = torch.empty((F, n), dtype=torch.uint8, device="cuda")
        t_res = events(lambda: code.decode_ml(y, out=bits))
        exit_share = float((bits.bool() == h).all(dim=1).float().mean())
        ml_wrong = bits.bool().any(dim=1)
        d_zero = torch.where(h, absy, torch.zeros_like(absy)).sum(dim=1)
        weight = torch.empty(F, dtype=torch.uint8, device="cuda")
        code.decode_osd(y, 3, out=(bits, weight))
        d_osd = torch.where(bits.bool() != h, absy, torch.zeros_like(absy)).sum(dim=1)
        bound = bits.bool().any(dim=1) & (d_osd < d_zero)
        ml_bound, not_ml = int(bound.sum()), int((bound & ~ml_wrong).sum())
        del d_osd, d_zero, weight, bound, ml_wrong, h, absy, y, bits
        torch.cuda.empty_cache()
        others = {"osd1": code.awgn_point_osd(ebno, F, 1, seed=SEED, point=POINT),
                  "osd2": code.awgn_point_osd(ebno, F, 2, seed=SEED, point=POINT),
                  "osd3": code.awgn_point_osd(ebno, F, 3, seed=SEED, point=POINT),
                  "chase4": code.awgn_point_chase(ebno, F, 4, seed=SEED, point=POINT),
                  "chase8": code.awgn_point_chase(ebno, F, 8, seed=SEED, point=POINT),
                  "hard": code.awgn_point_hard(ebno, F, seed=SEED, point=POINT),
                  "nms": code.awgn_point(ebno, F, "NMS", 0.8, seed=SEED, point=POINT),
                  "abp": code.awgn_point_abp(ebno, F, 20, 0.1, seed=SEED, point=POINT)}
        code.awgn_point_ml(ebno, min(F, 1 << 16), seed=SEED, point=POINT)  # warm-up
        t0 = time.perf_counter()
        o = code.awgn_point_ml(ebno, F, seed=SEED, point=POINT)
        t_fused = time.perf_counter() - t0
        rec = {"kind": "ml", "code": name, "k": k, "ebno_db": ebno, "frames": F,
               "resident_frames_per_s": F / t_res, "butterflies_per_s": F * n * (1 << (k - 1)) / t_res,
               "fused_frames_per_s": F / t_fused, "codeword_exit_share": exit_share, "wer_ml": o["frame_errors"] / F}
        rec.update({"wer_" + key: v["frame_errors"] / F for key, v in others.items()})
        rec["ml_lower_bound"] = ml_bound / F
        rec["ml_frame_errors"] = o["frame_errors"]
        rec.update({key + "_frame_errors": v["frame_errors"] for key, v in others.items()})
        rec.update({"ml_bound_frames": ml_bound, "bound_frames_not_ml_errors": not_ml, "resident_s": t_res,
                    "fused_s": t_fused, "gpu": lines[0]["gpu"]})
        lines.append(rec)
        print(json.dumps(rec), flush=True)
    ctx.close()
    if a.out:
        with open(a.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
