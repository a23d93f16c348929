"""The reference's AWGN sweep (src/simulation/simulation.c++:95-150) sharded over GPUs.

One process per GPU (torch.distributed).  Frames are independent units: rank r of W decodes the
global frame indices [r*N/W, (r+1)*N/W) of every Eb/N0 point (the noise is keyed by the global frame
index, so the totals do not depend on W), and one all-reduce (NCCL on GPUs, gloo in the CPU tests)
of the eight counters merges the point before the next point's sample count is derived from its
word-error rate (simulation.c++:91-93, :117, :143).  There is no other collective on this path.
"""
import os

from . import _lib


def shard_range(total, world, rank):
    """global frame range [first, first + count) of `rank`"""
    first = (total * rank) // world
    last = (total * (rank + 1)) // world
    return first, last - first


def sweep_points(rate, step=0.5, stop=8.0):
    """Eb/N0 points of simulation.c++:105-112: start one step above the Shannon limit, up to max(8, start)"""
    start = _lib.lib().ccgpu_sweep_start_ebno(float(rate), float(step))
    end = max(stop, start) + step / 2
    pts, eb = [], start
    while eb < end:
        pts.append(eb)
        eb += step
    return pts


def format_log_line(ebno, wer):
    """one line of "<name>.log": setw(7) setprecision(6) defaultfloat, setw(16) setprecision(15)
    scientific (simulation.c++:145-148)"""
    return "%7s %s" % ("%.6g" % ebno, "%.15e" % wer)


LOG_HEADER = "%7s %21s" % ("ebno", "wer")


def awgn_sweep(point_fn, name, rate, step=0.5, stop=8.0, cap=1000000, log_dir=None, dist=None, device=None,
               min_frames=0):
    """Runs the sweep.  point_fn(ebno_db, point_index, frame0, frames) -> 8 int64 counters (torch tensor on
    `device`) for the frames of THIS rank.  Returns a list of dicts (one per point), identical on every rank."""
    import torch
    world = dist.get_world_size() if dist is not None else 1
    rank = dist.get_rank() if dist is not None else 0
    wer = 0.5
    results = []
    log = None
    if log_dir is not None and rank == 0:
        path = os.path.join(log_dir, name + ".log")
        if os.path.exists(path):  # simulation.c++:72-81
            raise RuntimeError("File %s already exists." % path)
        log = open(path, "w")
        log.write(LOG_HEADER + "\n")
    for point, ebno in enumerate(sweep_points(rate, step, stop)):
        total = max(int(_lib.lib().ccgpu_sweep_samples(float(wer), int(cap))), int(min_frames))
        first, count = shard_range(total, world, rank)
        counters = point_fn(ebno, point, first, count)
        counters = counters.to(torch.int64)
        if dist is not None and world > 1:
            dist.all_reduce(counters, op=dist.ReduceOp.SUM)
        c = [int(v) for v in counters.cpu().tolist()]
        assert c[0] == total, (c[0], total)
        wer = c[1] / total
        results.append({"ebno": ebno, "frames": c[0], "frame_errors": c[1], "bit_errors": c[2], "iterations": c[3],
                        "failures": c[4], "undetected": c[5], "wer": wer})
        if log is not None:
            log.write(format_log_line(ebno, wer) + "\n")
            log.flush()
        if wer == 0.0:
            wer = 5e3 / cap
    if log is not None:
        log.close()
    return results


def gpu_point_fn(code, variant="MS", alpha=1.0, beta=0.0, max_iter=50, stop_rule=0, seed=0):
    """point_fn for awgn_sweep backed by ccgpu_awgn_point on the code's device"""
    import torch

    def fn(ebno, point, frame0, frames):
        out = torch.zeros(8, dtype=torch.int64, device="cuda:%d" % code.ctx.device)
        if frames > 0:
            code.awgn_point(ebno, frames, variant, alpha, beta, max_iter, stop_rule, seed=seed, point=point,
                            frame0=frame0, out=out)
            code.ctx.sync()  # the launch is asynchronous on the context's stream, not on torch's
        return out
    return fn


def chase_point_fn(code, p, seed=0):
    """point_fn for awgn_sweep backed by ccgpu_awgn_point_chase (Chase-II with p test positions) on the code's device"""
    import torch

    def fn(ebno, point, frame0, frames):
        out = torch.zeros(8, dtype=torch.int64, device="cuda:%d" % code.ctx.device)
        if frames > 0:
            code.awgn_point_chase(ebno, frames, p, seed=seed, point=point, frame0=frame0, out=out)
            code.ctx.sync()
        return out
    return fn


def osd_point_fn(code, order, seed=0):
    """point_fn for awgn_sweep backed by ccgpu_awgn_point_osd (OSD of the given order) on the code's device"""
    import torch

    def fn(ebno, point, frame0, frames):
        out = torch.zeros(8, dtype=torch.int64, device="cuda:%d" % code.ctx.device)
        if frames > 0:
            code.awgn_point_osd(ebno, frames, order, seed=seed, point=point, frame0=frame0, out=out)
            code.ctx.sync()
        return out
    return fn


def gmd_point_fn(code, max_erasures, seed=0):
    """point_fn for awgn_sweep backed by ccgpu_awgn_point_gmd (GMD of a Reed-Solomon code with up to max_erasures
    erasures; 0 = hard decision) on the code's device"""
    import torch

    def fn(ebno, point, frame0, frames):
        out = torch.zeros(8, dtype=torch.int64, device="cuda:%d" % code.ctx.device)
        if frames > 0:
            code.awgn_point_gmd(ebno, frames, max_erasures, seed=seed, point=point, frame0=frame0, out=out)
            code.ctx.sync()
        return out
    return fn


def abp_point_fn(code, max_iter=50, gamma=0.15, seed=0):
    """point_fn for awgn_sweep backed by ccgpu_awgn_point_abp (adaptive belief propagation) on the code's device"""
    import torch

    def fn(ebno, point, frame0, frames):
        out = torch.zeros(8, dtype=torch.int64, device="cuda:%d" % code.ctx.device)
        if frames > 0:
            code.awgn_point_abp(ebno, frames, max_iter, gamma, seed=seed, point=point, frame0=frame0, out=out)
            code.ctx.sync()
        return out
    return fn


def ml_point_fn(code, seed=0):
    """point_fn for awgn_sweep backed by ccgpu_awgn_point_ml (maximum-likelihood decoding) on the code's device"""
    import torch

    def fn(ebno, point, frame0, frames):
        out = torch.zeros(8, dtype=torch.int64, device="cuda:%d" % code.ctx.device)
        if frames > 0:
            code.awgn_point_ml(ebno, frames, seed=seed, point=point, frame0=frame0, out=out)
            code.ctx.sync()
        return out
    return fn
