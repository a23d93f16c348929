#!/usr/bin/env python
"""tools/sweep.py -- Eb/N0 waterfall sweep sharded over GPUs (BASELINE.json config 5).

    python tools/sweep.py --q 8 --t 18 --variant NMS --alpha 0.8 --ebno-from 0 --ebno-to 8 --ebno-step 0.5
    python tools/sweep.py --q 6 --t 5 --chase 4 ...      # Chase-II over the 4 least reliable positions
    python tools/sweep.py --q 6 --t 5 --osd 2 ...        # ordered-statistics decoding of order 2
    python tools/sweep.py --q 8 --t 16 --gmd 32 ...      # RS(255,223), GMD with up to 32 erasures (--gmd 0: hard)
    python tools/sweep.py --q 6 --t 5 --abp 50 --gamma 0.15 ...  # adaptive belief propagation, 50 updates at most
    python tools/sweep.py --q 6 --t 2 --ml ...           # maximum-likelihood (Viterbi) decoding, n - l <= 12
    torchrun --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/sweep.py ...

Every Eb/N0 point is simulated in rounds of --batch frames (split evenly over the ranks by global frame
index) until --min-errors frame errors have been seen or --max-frames frames are spent; after each round
ONE all-reduce (NCCL) merges the eight counters.  Results do not depend on the number of GPUs: the noise of
a frame is keyed by (seed, point, global frame index).  Rank 0 prints one JSON line per point.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--q", type=int, default=8)
    ap.add_argument("--t", type=int, default=18)
    ap.add_argument("--variant", default="NMS")
    ap.add_argument("--alpha", type=float, default=0.8)
    ap.add_argument("--beta", type=float, default=0.0)
    ap.add_argument("--max-iter", type=int, default=50)
    ap.add_argument("--stop-rule", type=int, default=0)
    ap.add_argument("--ebno-from", type=float, default=0.0)  # (torchrun's own parser claims --start*)
    ap.add_argument("--ebno-to", type=float, default=8.0)
    ap.add_argument("--ebno-step", type=float, default=0.5)
    ap.add_argument("--batch", type=int, default=1 << 24)
    ap.add_argument("--min-errors", type=int, default=100)
    ap.add_argument("--max-frames", type=float, default=1e9)
    ap.add_argument("--seed", type=int, default=0)
    algo = ap.add_mutually_exclusive_group()
    algo.add_argument("--chase", type=int, default=None, metavar="P",
                      help="decode with Chase-II over the P least reliable positions (0..8) instead of the min-sum variant")
    algo.add_argument("--osd", type=int, default=None, metavar="ORDER",
                      help="decode with ordered-statistics decoding of order 0..3 instead of the min-sum variant")
    algo.add_argument("--gmd", type=int, default=None, metavar="F",
                      help="simulate the Reed-Solomon code RS(2^q - 1, 2^q - 1 - 2t) decoded with GMD over up to F "
                           "(even, <= 2t) erased symbols; 0 is hard-decision decoding")
    algo.add_argument("--abp", type=int, default=None, metavar="ITERS",
                      help="decode with adaptive belief propagation, at most ITERS (0..255) updates, instead of the "
                           "min-sum variant")
    algo.add_argument("--ml", action="store_true",
                      help="decode with maximum-likelihood (Viterbi) decoding on the syndrome trellis (n - l <= 12) "
                           "instead of the min-sum variant")
    ap.add_argument("--gamma", type=float, default=0.15, help="damping factor of --abp (0 < gamma <= 1)")
    a = ap.parse_args()

    import torch
    import torch.distributed as dist
    import channelcoding_b200 as cc
    from channelcoding_b200.simulation import shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL logs to stdout by default: route it to stderr so that stdout stays JSON lines; the log LEVEL is the caller's
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = cc.Context(local)
    ctx.use_torch_stream()
    code = ctx.rs(a.q, a.t) if a.gmd is not None else ctx.bch(a.q, errors=a.t)
    bits_per_frame = code.n * a.q if a.gmd is not None else code.n  # GMD counts the bits of the binary image
    dev = torch.device("cuda", local)
    tag = ("CHASE%d" % a.chase if a.chase is not None else "OSD%d" % a.osd if a.osd is not None else
           "GMD%d" % a.gmd if a.gmd is not None else "ABP%d" % a.abp if a.abp is not None else
           "ML" if a.ml else a.variant)
    point, eb = 0, a.ebno_from
    while eb < a.ebno_to + a.ebno_step / 2:
        total = torch.zeros(8, dtype=torch.int64, device=dev)
        done = 0
        t0 = time.perf_counter()
        while True:
            first, count = shard_range(a.batch, world, rank)
            part = torch.zeros(8, dtype=torch.int64, device=dev)
            if a.chase is not None:
                code.awgn_point_chase(eb, count, a.chase, seed=a.seed, point=point, frame0=done + first, out=part)
            elif a.osd is not None:
                code.awgn_point_osd(eb, count, a.osd, seed=a.seed, point=point, frame0=done + first, out=part)
            elif a.gmd is not None:
                code.awgn_point_gmd(eb, count, a.gmd, seed=a.seed, point=point, frame0=done + first, out=part)
            elif a.abp is not None:
                code.awgn_point_abp(eb, count, a.abp, a.gamma, seed=a.seed, point=point, frame0=done + first, out=part)
            elif a.ml:
                code.awgn_point_ml(eb, count, seed=a.seed, point=point, frame0=done + first, out=part)
            else:
                code.awgn_point(eb, count, a.variant, a.alpha, a.beta, a.max_iter, a.stop_rule, seed=a.seed, point=point,
                                frame0=done + first, out=part)
            if world > 1:
                dist.all_reduce(part, op=dist.ReduceOp.SUM)  # the one collective of the path
            total += part
            done += a.batch
            c = total.cpu().tolist()
            if c[1] >= a.min_errors or done >= a.max_frames:
                break
        el = time.perf_counter() - t0
        if rank == 0:
            print(json.dumps({"code": code.to_string(tag), "ebno_db": eb, "frames": c[0], "frame_errors": c[1],
                              "bit_errors": c[2], "wer": c[1] / c[0], "ber": c[2] / c[0] / bits_per_frame,
                              "avg_iterations": c[3] / c[0], "failures": c[4], "undetected": c[5], "n_gpus": world,
                              "seconds": el, "frames_per_s": c[0] / el}), flush=True)
        point += 1
        eb += a.ebno_step
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
