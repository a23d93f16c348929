"""Every decoder's per-frame outputs against the oracle at the batch sizes the project is measured and used at.

The frame schedulers behave differently on large batches: the warp kernels take frame indices from the queue in batches
of up to 32 only while more than 2^work_shift x 32 frames remain, the host-buffer paths cut a batch into chunks that
rotate over three slot streams, multiple-bases decoding cuts it to fit its work arena.  A misrouted output -- a frame's
result written to another frame's row, a row never written, state left over from the frame a warp held before -- leaves
Monte-Carlo counters unchanged, so these paths are checked here output for output.

The oracle cannot decode millions of frames, but the decoders are per-frame functions, so a TILED check suffices:
  * a pool of M distinct frames (seeded AWGN on the all-zero codeword across the waterfall, so that iteration counts
    range from 1 to failures at max_iter, plus edge frames) is decoded once by the oracle on every core;
  * the batch of N frames is the pool tiled by a seeded index map src (every pool frame appears floor(N/M) or
    ceil(N/M) times, with random neighbours);
  * the outputs are prefilled with a sentinel, so a row the kernel never writes cannot match by chance;
  * out[f] == ref[src[f]] is required for every f and every output field (floats as bit patterns).
A CPU test checks the checker itself on the oracle's own outputs and a set of mutations."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle
from test_gpu_chase import chase_restatement
from test_gpu_parity import mbbp_restatement

gpu = pytest.mark.gpu

# sentinels the outputs are prefilled with, per field (as the integer the checker compares: floats as bit patterns)
SENT8 = 0xA5
SENTINEL = {"bits": SENT8, "iter": SENT8, "failed": SENT8, "status": SENT8, "chosen": SENT8, "corrected": SENT8,
            "nerr": SENT8, "L": 0x7FC0DEAD, "packed": int(np.uint32(0xA5A5A5A5).view(np.int32))}
MAX_ITER = 50


# ---------------------------------------------------------------------------------------------------- pools
def oracle_map(fn, y, chunk=1000):
    """fn(rows) -> tuple of per-row arrays, evaluated over chunks of y on every core (ctypes releases the GIL)"""
    threads = os.cpu_count() or 1
    chunk = max(1, min(chunk, -(-len(y) // (4 * threads))))
    parts = [y[i:i + chunk] for i in range(0, len(y), chunk)]
    with ThreadPoolExecutor(threads) as ex:
        outs = list(ex.map(fn, parts))
    return tuple(np.concatenate([o[k] for o in outs]) for k in range(len(outs[0])))


def edge_frames(n, rng, nonfinite=False):
    """all +1, all -1, zeros, exact magnitude ties, -0.0, the smallest subnormal, +-1e30, one negative value;
    +-inf and NaN only when `nonfinite`"""
    noisy = lambda: 1.0 + 0.8 * rng.standard_normal(n)  # noqa: E731
    cols = lambda k: rng.choice(n, k, replace=False)  # noqa: E731
    f = [np.ones(n), -np.ones(n), np.zeros(n), np.full(n, -0.0), np.full(n, 1e-45), np.full(n, -1e-45)]
    for k in (1, 3, 9):
        a = noisy()
        a[cols(k)] = 0.0
        f.append(a)
    for _ in range(6):
        f.append(rng.choice([-1.0, 1.0], n))                  # every |y| = 1
    a = noisy()
    a[cols(5)] = -0.0
    f.append(a)
    a = noisy()
    a[cols(4)] = 1e-45
    a[cols(2)] = -1e-45
    f.append(a)
    for k in (1, 4):
        a = noisy()
        a[cols(k)] = 1e30
        a[cols(k)] = -1e30
        f.append(a)
    for v in (-1.0, -0.25, -1e-45):
        a = np.ones(n)
        a[rng.integers(n)] = v                               # one negative value
        f.append(a)
    if nonfinite:
        f += [np.full(n, np.inf), np.full(n, -np.inf), np.full(n, np.nan)]
        for v in (np.inf, -np.inf, np.nan):
            a = noisy()
            a[cols(3)] = v
            f.append(a)
    return np.array(f, np.float32)


def awgn_pool(n, rate, M, ebnos, seed, nonfinite=False):
    """M distinct frames: the edge frames, then the all-zero codeword under seeded AWGN at each Eb/N0 in turn"""
    rng = np.random.default_rng(seed)
    edges = edge_frames(n, rng, nonfinite)
    k = M - len(edges)
    sig = np.resize(np.array([oracle.sigma(rate, eb) for eb in ebnos]), k)
    y = (1.0 + sig[:, None] * rng.standard_normal((k, n))).astype(np.float32)
    return np.concatenate([edges, y])


def ms_ref(H, y, variant, alpha=1.0, beta=0.0, max_iter=MAX_ITER, stop=0, quant=None):
    """oracle outputs of the pool as the decoder writes them: bits, L (fixed point: the integer totals as float32), iter,
    failed"""
    if variant.endswith("_Q"):
        q = quant or (8.0, 31, 31)
        b, L, it, f = oracle_map(lambda r: oracle.min_sum_fixed(H, r, variant, alpha, beta, max_iter, stop, *q), y)
        L = L.astype(np.float32)
    else:
        b, L, it, f = oracle_map(lambda r: oracle.min_sum(H, r, variant, alpha, beta, max_iter, stop), y)
    return {"bits": b, "L": L, "iter": it.astype(np.int32), "failed": f}


class Pool:
    def __init__(self, y, ref):
        self.y, self.ref = y, ref
        self.M = len(y)


# (q, t) of the binary BCH codes, and the pools: code, M, Eb/N0 (dB), seed, decoder (variant, alpha, beta, stop, quant)
BCH = {"bch_15_7": (4, 2), "bch_31_16": (5, 3), "bch_63_36": (6, 5), "bch_63_45": (6, 3), "bch_63_51": (6, 2),
       "bch_63_57": (6, 1), "bch_127_64": (7, 10), "bch_255_131": (8, 18)}
POOLS = {
    "63_36_NMS": ("bch_63_36", 32768, (1.0, 2.0, 3.0, 4.0, 5.0), 1, ("NMS", 0.8, 0.0, 0, None)),
    "63_36_SCMS2": ("bch_63_36", 16384, (1.0, 2.0, 3.0, 4.0, 5.0), 2, ("SCMS2", 1.0, 0.0, 1, None)),
    "63_36_2DNMS": ("bch_63_36", 16384, (1.0, 2.0, 3.0, 4.0, 5.0), 3, ("2DNMS", 0.9, 0.8, 0, None)),
    "63_36_NMS_Q": ("bch_63_36", 32768, (1.0, 2.0, 3.0, 4.0, 5.0), 4, ("NMS_Q", 0.8, 0.0, 0, None)),
    "63_36_MS_Q": ("bch_63_36", 32768, (1.0, 2.0, 3.0, 4.0, 5.0), 4, ("MS_Q", 1.0, 0.0, 1, None)),
    "63_51_NMS": ("bch_63_51", 16384, (1.0, 2.0, 3.0, 4.0, 5.0), 5, ("NMS", 0.8, 0.0, 0, None)),
    "63_57_NMS": ("bch_63_57", 16384, (0.0, 1.0, 2.0, 3.0, 4.0), 6, ("NMS", 0.8, 0.0, 0, None)),
    "127_64_NMS": ("bch_127_64", 4096, (3.5, 4.0, 4.5, 5.0, 5.5), 7, ("NMS", 0.8, 0.0, 0, None)),
    "255_131_NMS": ("bch_255_131", 256, (4.5, 5.0, 5.5, 6.0), 8, ("NMS", 0.8, 0.0, 0, None)),
    "255_131_NMS_Q": ("bch_255_131", 256, (4.5, 5.0, 5.5, 6.0), 9, ("NMS_Q", 0.8, 0.0, 0, (8.0, 31, 29))),
    "15_7_MS": ("bch_15_7", 65536, (-2.0, -1.0, 0.0, 1.0, 2.0, 3.0), 10, ("MS", 1.0, 0.0, 0, None)),
    "31_16_NMS": ("bch_31_16", 16384, (0.0, 1.0, 2.0, 3.0, 4.0), 11, ("NMS", 0.8, 0.0, 0, None)),
}


def bch_rate(name):
    q, t = BCH[name]
    oc = oracle.Code(0, q, t)
    return oc.n, oc.rate


def pool_y(name, M, ebnos, seed, nonfinite):
    n, rate = bch_rate(name)
    return awgn_pool(n, rate, M, ebnos, seed, nonfinite)


@pytest.fixture(scope="module")
def pools():
    """pools built on first use and kept for the module: key -> Pool"""
    return {}


def get_pool(pools, key):
    """the pool `key` of POOLS, decoded by the oracle"""
    if key not in pools:
        name, M, ebnos, seed, (variant, alpha, beta, stop, quant) = POOLS[key]
        y = pool_y(name, M, ebnos, seed, nonfinite=variant.endswith("_Q"))
        pools[key] = Pool(y, ms_ref(oracle.Code(0, *BCH[name]).H(), y, variant, alpha, beta, MAX_ITER, stop, quant))
    return pools[key]


def tiling(M, N, seed):
    """seeded index map of a batch of N frames onto a pool of M: every pool frame floor(N/M) or ceil(N/M) times"""
    rng = np.random.default_rng(seed)
    return rng.permutation(np.resize(rng.permutation(M), N))


# ---------------------------------------------------------------------------------------------------- the checker
def _ints(t):
    """a tensor as the integers the checker compares: float32 as its bit patterns"""
    import torch
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def mismatch_report(got, ref, src, limit=10, chunk=1 << 20):
    """got: field -> tensor [N, ...] (what the decoder wrote), ref: field -> tensor [M, ...] (the pool's expected
    outputs), src: int64 tensor [N], all on one device.  None if got[f] == ref[src[f]] for every row f and field, else a
    report: how many rows differ, and the first `limit` (f, src[f]) with whether the row still holds the sentinel
    (never written), equals the expected output of another pool frame (misrouted), or is something else."""
    import torch
    N = src.numel()
    g = {k: _ints(v) for k, v in got.items()}
    r = {k: _ints(v) for k, v in ref.items()}
    M = next(iter(r.values())).shape[0]
    bad = torch.zeros(N, dtype=torch.bool, device=src.device)
    for k in g:
        assert g[k].shape[0] == N and g[k].shape[1:] == r[k].shape[1:], k
        for a in range(0, N, chunk):
            d = g[k][a:a + chunk].to(r[k].dtype) != r[k][src[a:a + chunk]]
            bad[a:a + chunk] |= d.reshape(d.shape[0], -1).any(dim=1)
    nbad = int(bad.sum())
    if nbad == 0:
        return None
    lines = []
    for f in torch.nonzero(bad).flatten()[:limit].tolist():
        s = int(src[f])
        if all(bool((g[k][f] == SENTINEL[k]).all()) for k in g):
            kind = "sentinel: never written"
        else:
            same = torch.ones(M, dtype=torch.bool, device=src.device)
            for k in g:
                same &= (r[k] == g[k][f].to(r[k].dtype)).reshape(M, -1).all(dim=1)
            same[s] = False
            other = torch.nonzero(same).flatten()[:3].tolist()
            if other:
                rows = torch.nonzero(src == other[0]).flatten()[:3].tolist()
                kind = "misrouted: equals the output of pool frame %d (batch rows %s)" % (other[0], rows)
            else:
                kind = "something else: fields %s differ" % [k for k in g if not bool((g[k][f].to(r[k].dtype) == r[k][s]).all())]
        lines.append("  f=%d src=%d: %s" % (f, s, kind))
    return "%d of %d rows differ; the first %d:\n%s" % (nbad, N, len(lines), "\n".join(lines))


def check_tiled(got, ref, src, what):
    report = mismatch_report(got, ref, src)
    assert report is None, "%s: %s" % (what, report)


def to_dev(a, device="cuda"):
    """numpy or torch -> torch on `device`; uint32 words as int32"""
    import torch
    if isinstance(a, np.ndarray):
        a = torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a)
    return a.to(device)


def ref_on(pool_ref, device="cuda", fields=None):
    return {k: to_dev(v, device) for k, v in pool_ref.items() if fields is None or k in fields}


def sentinel_like(shape, dtype, field, lib="torch", device="cuda"):
    """an output buffer prefilled with the field's sentinel"""
    if lib == "numpy":
        a = np.empty(shape, dtype)
        a.view(np.int32 if a.itemsize == 4 else np.uint8)[...] = SENTINEL[field]
        return a
    import torch
    t = torch.empty(shape, dtype=dtype, device=device)
    (t.view(torch.int32) if t.element_size() == 4 else t).fill_(SENTINEL[field])
    return t


def ms_outputs(N, n, want_L, lib="torch", device="cuda"):
    import torch
    u8, f32 = (np.uint8, np.float32) if lib == "numpy" else (torch.uint8, torch.float32)
    mk = lambda shape, dt, k: sentinel_like(shape, dt, k, lib, device)  # noqa: E731
    return (mk((N, n), u8, "bits"), mk((N, n), f32, "L") if want_L else None, mk(N, u8, "iter"), mk(N, u8, "failed"))


def ms_got(out):
    bits, L, it, failed = out
    got = {"bits": bits, "iter": it, "failed": failed}
    if L is not None:
        got["L"] = L
    return {k: to_dev(v) for k, v in got.items()}


# ---------------------------------------------------------------------------------------------------- CPU self-test
def test_checker_rejects_misrouted_outputs():
    """the checker passes the oracle's own outputs of a tiled batch and rejects a row never written, two swapped rows,
    one flipped bit of L, an iteration index off by one and a row copied from its neighbour"""
    import torch
    oc = oracle.Code(0, 6, 5)
    y = awgn_pool(63, oc.rate, 160, (1.0, 3.0, 5.0), 99)
    ref = ms_ref(oc.H(), y, "NMS", 0.8)
    assert len(np.unique(ref["iter"])) > 5 and ref["failed"].any()
    N = 1000
    src = tiling(len(y), N, 5)
    ref_t = ref_on(ref, "cpu")
    src_t = torch.from_numpy(src)

    def tiled():
        out = ms_outputs(N, 63, True, "torch", "cpu")
        got = dict(zip(("bits", "L", "iter", "failed"), out))
        for k, v in got.items():
            v.copy_(ref_t[k][src_t].to(v.dtype) if k != "L" else ref_t[k][src_t])
        return got

    assert mismatch_report(tiled(), ref_t, src_t) is None

    def distinct_pair():
        for f in range(N - 1):
            a, b = int(src[f]), int(src[f + 1])
            if ref["iter"][a] != ref["iter"][b] and (ref["bits"][a] != ref["bits"][b]).any():
                return f, f + 1
        raise AssertionError("no neighbours with different outputs")

    f, f2 = distinct_pair()
    got = tiled()
    for k, v in got.items():
        (v.view(torch.int32) if k == "L" else v)[f] = SENTINEL[k]
    rep = mismatch_report(got, ref_t, src_t)
    assert rep is not None and rep.startswith("1 of 1000 rows differ") and "sentinel" in rep, rep

    got = tiled()
    for v in got.values():
        v[[f, f2]] = v[[f2, f]]
    rep = mismatch_report(got, ref_t, src_t)
    assert rep is not None and rep.startswith("2 of") and rep.count("misrouted") == 2, rep

    got = tiled()
    got["L"].view(torch.int32)[f, 17] ^= 1
    rep = mismatch_report(got, ref_t, src_t)
    assert rep is not None and rep.startswith("1 of") and "something else" in rep and "'L'" in rep, rep

    got = tiled()
    got["iter"][f] += 1
    rep = mismatch_report(got, ref_t, src_t)
    assert rep is not None and rep.startswith("1 of") and "'iter'" in rep, rep

    got = tiled()
    for v in got.values():
        v[f2] = v[f]
    rep = mismatch_report(got, ref_t, src_t)
    assert rep is not None and rep.startswith("1 of") and "misrouted" in rep, rep


def test_pool_and_tiling():
    """the pools contain every kind of edge frame and iteration counts across the whole range; the tiling uses every pool
    frame floor(N / M) or ceil(N / M) times"""
    src = tiling(1000, 4097, 3)
    c = np.bincount(src, minlength=1000)
    assert c.min() == 4 and c.max() == 5 and c.sum() == 4097
    y = awgn_pool(63, 36 / 63, 200, (1.0, 3.0), 0, nonfinite=True)
    assert len(np.unique(y.view(np.uint32), axis=0)) == len(y)
    assert np.isnan(y).any() and np.isinf(y).any() and (y == 1e30).any() and (y == -1e30).any()
    assert (np.signbit(y) & (y == 0)).any() and (y == np.float32(1e-45)).any()
    assert np.isfinite(awgn_pool(63, 36 / 63, 200, (1.0, 3.0), 0)).all()


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    import channelcoding_b200 as cc
    c = cc.Context(0)
    yield c
    c.close()


def gpu_bch(ctx, name):
    return ctx.bch(*BCH[name][:1], errors=BCH[name][1])


def decode_tiled(ctx, code, pool, N, seed, variant, alpha=1.0, beta=0.0, stop=0, quant=None, want_L=True, what=""):
    """decode the tiled batch from device memory into sentinel-filled outputs and check every row"""
    import torch
    src = torch.from_numpy(tiling(pool.M, N, seed)).cuda()
    y = to_dev(pool.y)[src]
    out = ms_outputs(N, code.n, want_L)
    code.decode(y, variant, alpha, beta, MAX_ITER, stop, want_L=want_L, out=out, quant=quant)
    torch.cuda.synchronize()
    del y
    got = ms_got(out)
    check_tiled(got, ref_on(pool.ref, fields=got.keys()), src, what)


@gpu
@pytest.mark.parametrize("N", [4194304, 3000017])
def test_headline_decode(ctx, pools, N):
    """bench.py's headline path: BCH(63,36) NMS 0.8, 50 iterations, stop rule 0, from torch tensors, totals requested"""
    pool = get_pool(pools, "63_36_NMS")
    decode_tiled(ctx, gpu_bch(ctx, "bch_63_36"), pool, N, N, "NMS", 0.8, what="BCH(63,36) NMS %d frames" % N)


@gpu
@pytest.mark.parametrize("option,value", [("work_batch", 1), ("work_batch", 5), ("work_batch", 1024), ("quick", 1)])
def test_headline_schedule_options(ctx, pools, option, value):
    """the same batch with other queue batch sizes (one frame per atomic, ragged batches, batches larger than a pool),
    and through the QUICK instantiation (all-positive frames retired without iterating; totals not requested)"""
    pool = get_pool(pools, "63_36_NMS")
    ctx.set_option(option, value)
    try:
        decode_tiled(ctx, gpu_bch(ctx, "bch_63_36"), pool, 4194304, 11 + value, "NMS", 0.8, want_L=option != "quick",
                     what="BCH(63,36) NMS %s=%d" % (option, value))
    finally:
        ctx.set_option(option, 0 if option == "work_batch" else -1)


@gpu
def test_headline_host_pipeline(ctx, pools):
    """numpy buffers: the chunks rotate over three slot streams, each with its own queue head; the byte layout and the
    compact layout (packed decisions + status byte)"""
    import torch
    pool = get_pool(pools, "63_36_NMS")
    code = gpu_bch(ctx, "bch_63_36")
    N = 4194304
    src_np = tiling(pool.M, N, 21)
    src = torch.from_numpy(src_np).cuda()
    y = pool.y[src_np]
    out = ms_outputs(N, 63, True, "numpy")
    code.decode(y, "NMS", 0.8, 0.0, MAX_ITER, 0, want_L=True, out=out)
    check_tiled(ms_got(out), ref_on(pool.ref), src, "BCH(63,36) NMS host buffers")
    del out
    packed = sentinel_like((N, 2), np.uint32, "packed", "numpy")
    status = sentinel_like(N, np.uint8, "status", "numpy")
    code.decode_packed(y, "NMS", 0.8, 0.0, MAX_ITER, 0, out=(packed, status))
    b = pool.ref["bits"].astype(np.uint64)
    words = (b << np.arange(63, dtype=np.uint64)).sum(axis=1, dtype=np.uint64)
    ref = {"packed": words.view(np.uint32).reshape(-1, 2),
           "status": np.where(pool.ref["failed"] == 1, 255, pool.ref["iter"]).astype(np.uint8)}
    check_tiled({"packed": to_dev(packed), "status": to_dev(status)}, ref_on(ref), src, "BCH(63,36) NMS packed, host buffers")


@gpu
@pytest.mark.parametrize("key", ["63_36_SCMS2", "63_36_2DNMS"])
def test_other_flavours(ctx, pools, key):
    """the self-correcting flavour (GF(2) stop rule) and the two-dimensional normalisation on the warp kernel"""
    pool = get_pool(pools, key)
    variant, alpha, beta, stop, _ = POOLS[key][4]
    decode_tiled(ctx, gpu_bch(ctx, "bch_63_36"), pool, 1048576, 31, variant, alpha, beta, stop, what=key)


@gpu
@pytest.mark.parametrize("key", ["63_36_NMS_Q", "63_36_MS_Q"])
def test_fixed_point(ctx, pools, key):
    """K2q, two frames per lane: NMS_Q with the default quantiser (what bench.py reports) and MS_Q with the GF(2) stop
    rule; +-inf and NaN included"""
    pool = get_pool(pools, key)
    variant, alpha, beta, stop, quant = POOLS[key][4]
    decode_tiled(ctx, gpu_bch(ctx, "bch_63_36"), pool, 4194304, 41, variant, alpha, beta, stop, quant, what=key)


@gpu
@pytest.mark.parametrize("key,name,fpw", [("63_51_NMS", "bch_63_51", 2), ("63_57_NMS", "bch_63_57", 4)])
def test_several_frames_per_warp(ctx, pools, key, name, fpw):
    """the grant path of take_frames: several frame groups of one warp refill from one pool of indices"""
    pool = get_pool(pools, key)
    decode_tiled(ctx, gpu_bch(ctx, name), pool, 4194304, 51 + fpw, "NMS", 0.8, what="%s (%d frames per warp)" % (name, fpw))


@gpu
def test_two_rows_per_lane(ctx, pools):
    pool = get_pool(pools, "127_64_NMS")
    decode_tiled(ctx, gpu_bch(ctx, "bch_127_64"), pool, 1048576, 61, "NMS", 0.8, what="BCH(127,64) NMS")


@gpu
@pytest.mark.parametrize("key", ["255_131_NMS", "255_131_NMS_Q"])
def test_cta_kernels(ctx, pools, key):
    """K2c and K2cq: one CTA per frame (BCH(255,131)), float and fixed point"""
    pool = get_pool(pools, key)
    variant, alpha, beta, stop, quant = POOLS[key][4]
    decode_tiled(ctx, gpu_bch(ctx, "bch_255_131"), pool, 262144, 71, variant, alpha, beta, stop, quant, what=key)


@gpu
def test_cta_kernel_redundant_H(ctx, pools):
    """K2c on BCH(127,64) with all 127 cyclic shifts as rows"""
    if "127_64_red" not in pools:
        H = oracle.Code(0, 7, 10).H(127)
        y = pool_y("bch_127_64", 1024, (3.0, 3.5, 4.0, 4.5, 5.0), 12, False)
        pools["127_64_red"] = Pool(y, ms_ref(H, y, "NMS", 0.8))
    code = gpu_bch(ctx, "bch_127_64")
    code.set_rows(127)
    assert code.h_rows == 127
    decode_tiled(ctx, code, pools["127_64_red"], 524288, 81, "NMS", 0.8, what="BCH(127,64) NMS, 127 rows")


@gpu
@pytest.mark.parametrize("key,name,N,variant,alpha", [("15_7_MS", "bch_15_7", 16777216, "MS", 1.0),
                                                       ("31_16_NMS", "bch_31_16", 4194304, "NMS", 0.8)])
def test_lane_kernel(ctx, pools, key, name, N, variant, alpha):
    """K2s, one lane per frame, FIFO refill of the lanes"""
    pool = get_pool(pools, key)
    code = gpu_bch(ctx, name)
    decode_tiled(ctx, code, pool, N, 91, variant, alpha, what=key)


@gpu
def test_csr_kernel(ctx, pools):
    """the general kernel on a row-permuted BCH(63,45) matrix"""
    oc = oracle.Code(0, 6, 3)
    H = oc.H()[np.random.default_rng(13).permutation(oc.k)]
    if "63_45_csr" not in pools:
        y = pool_y("bch_63_45", 4096, (2.0, 3.0, 4.0, 5.0, 6.0), 13, False)
        pools["63_45_csr"] = Pool(y, ms_ref(H, y, "NMS", 0.8))
    code = ctx.from_dense(H, oc.rate)
    assert code.kernel == 2
    decode_tiled(ctx, code, pools["63_45_csr"], 262144, 101, "NMS", 0.8, what="CSR BCH(63,45) NMS")


@gpu
def test_multiple_bases(ctx, pools):
    """bench.py's multiple-bases configuration (BCH(127,64) NMS, 8 bases, GF(2) stop rule): the batch is cut into chunks
    that fit the work arena"""
    import torch
    shifts = [(127 * i) // 8 for i in range(8)]
    oc = oracle.Code(0, 7, 10)
    H = oc.H()
    if "mbbp" not in pools:
        y = pool_y("bch_127_64", 512, (3.0, 3.5, 4.0, 4.5, 5.0), 14, False)
        b, L, it, f, ch = oracle_map(lambda r: mbbp_restatement(H, r, shifts, "NMS", 0.8, 0.0, MAX_ITER, 1), y, chunk=16)
        pools["mbbp"] = Pool(y, {"bits": b, "L": L, "iter": it.astype(np.int32), "failed": f, "chosen": ch})
    pool = pools["mbbp"]
    code = gpu_bch(ctx, "bch_127_64")
    N = 262144
    src = torch.from_numpy(tiling(pool.M, N, 111)).cuda()
    y = to_dev(pool.y)[src]
    out = ms_outputs(N, 127, True) + (sentinel_like(N, torch.uint8, "chosen"),)
    code.decode_mbbp(y, shifts, "NMS", 0.8, 0.0, MAX_ITER, 1, out=out)
    torch.cuda.synchronize()
    got = ms_got(out[:4])
    got["chosen"] = out[4]
    check_tiled(got, ref_on(pool.ref), src, "multiple bases")


@gpu
@pytest.mark.parametrize("path", ["host", "device"])
def test_chase(ctx, pools, path):
    """Chase-II p = 4 on BCH(63,36), host buffers (chunk loop over the slots) and torch tensors"""
    import torch
    if "chase" not in pools:
        y = pool_y("bch_63_36", 8192, (2.0, 3.0, 4.0, 5.0, 6.0), 15, False)
        b, f, ch, _ = oracle_map(lambda r: chase_restatement(oracle.Code(0, 6, 5), r, 4), y, chunk=256)
        pools["chase"] = Pool(y, {"bits": b, "failed": f, "chosen": ch})
    pool = pools["chase"]
    code = gpu_bch(ctx, "bch_63_36")
    N = 1048576
    src_np = tiling(pool.M, N, 121)
    src = torch.from_numpy(src_np).cuda()
    lib = "numpy" if path == "host" else "torch"
    u8 = np.uint8 if lib == "numpy" else torch.uint8
    out = (sentinel_like((N, 63), u8, "bits", lib), sentinel_like(N, u8, "failed", lib), sentinel_like(N, u8, "chosen", lib))
    y = pool.y[src_np] if lib == "numpy" else to_dev(pool.y)[src]
    code.decode_chase(y, 4, out=out)
    torch.cuda.synchronize()
    got = {k: to_dev(v) for k, v in zip(("bits", "failed", "chosen"), out)}
    check_tiled(got, ref_on(pool.ref), src, "Chase p=4 " + path)


@gpu
def test_gf_decode_host(ctx, pools):
    """RS(255,223) with 0 .. 20 symbol errors through the host chunk loop"""
    import torch
    if "rs" not in pools:
        rng = np.random.default_rng(16)
        oc = oracle.Code(1, 8, 16)
        words = oc.encode(rng.integers(0, 256, size=(8192, oc.l)).astype(np.uint8))
        for i, e in enumerate(rng.integers(0, 21, size=len(words))):
            pos = rng.choice(255, e, replace=False)
            words[i, pos] ^= rng.integers(1, 256, size=e).astype(np.uint8)
        out, nerr, status = oracle_map(lambda r: oracle.Code(1, 8, 16).hard_correct(r), words)
        failed = (status != 0).astype(np.uint8)
        pools["rs"] = Pool(words, {"corrected": np.where(failed[:, None] == 1, words, out),
                                   "nerr": np.where(failed == 1, 0, nerr).astype(np.uint8), "failed": failed})
        assert 0.05 < failed.mean() < 0.5
    pool = pools["rs"]
    code = ctx.rs(8, 16)
    N = 4194304
    src_np = tiling(pool.M, N, 131)
    out = (sentinel_like((N, 255), np.uint8, "corrected", "numpy"), sentinel_like(N, np.uint8, "nerr", "numpy"),
           sentinel_like(N, np.uint8, "failed", "numpy"))
    code.gf_decode(pool.y[src_np], out=out)
    got = {k: to_dev(v) for k, v in zip(("corrected", "nerr", "failed"), out)}
    check_tiled(got, ref_on(pool.ref), torch.from_numpy(src_np).cuda(), "RS(255,223) gf_decode host buffers")


def device_sets():
    import torch
    return [[0, 0, 0]] + ([list(range(torch.cuda.device_count()))] if torch.cuda.device_count() >= 2 else [])


@gpu
@pytest.mark.parametrize("which", [0, 1])
def test_group_decode(pools, which):
    """ccgpu_group_decode_llr: the batch sharded over three contexts on device 0, and over every device of the host"""
    import torch
    import channelcoding_b200 as cc
    sets = device_sets()
    if which >= len(sets):
        pytest.skip("one GPU only")
    pool = get_pool(pools, "63_36_NMS")
    N = 4194304
    src_np = tiling(pool.M, N, 141 + which)
    g = cc.Group(sets[which])
    try:
        code = g.bch(6, errors=5)
        out = ms_outputs(N, 63, True, "numpy")
        code.decode(pool.y[src_np], "NMS", 0.8, 0.0, MAX_ITER, 0, out=out)
    finally:
        g.close()
    check_tiled(ms_got(out), ref_on(pool.ref), torch.from_numpy(src_np).cuda(), "group %s" % sets[which])


# ---------------------------------------------------------------------------------------------------- fused == streaming
@gpu
@pytest.mark.parametrize("name,ebno,N,variant,alpha", [("bch_63_36", 4.0, 4194304, "NMS", 0.8),
                                                        ("bch_63_36", 7.0, 4194304, "NMS", 0.8),
                                                        ("bch_63_36", 4.0, 4194304, "NMS_Q", 0.8),
                                                        ("bch_15_7", 3.0, 16777216, "MS", 1.0),
                                                        ("bch_255_131", 6.0, 262144, "NMS", 0.8)])
def test_fused_point_equals_streaming_at_scale(ctx, name, ebno, N, variant, alpha):
    """ccgpu_awgn_point (with the host's own choice of instantiation: screening at 7 dB, the grouped CTA mode for
    BCH(255,131)) == channel kernel -> decode -> counters computed on the device, at sizes where full batches are taken"""
    import torch
    import channelcoding_b200 as cc
    code = gpu_bch(ctx, name)
    c = code.awgn_point(ebno, N, variant, alpha, seed=17, point=3, frame0=12345)
    y = torch.empty((N, code.n), dtype=torch.float32, device="cuda")
    ctx.awgn_llr(code.n, np.float32(cc.sigma(code.rate, ebno)), seed=17, point=3, frame0=12345, frames=N, out=y)
    bits, _, it, failed = code.decode(y, variant, alpha, 0.0, MAX_ITER, 0, want_L=False)
    torch.cuda.synchronize()
    del y
    nb = bits.sum(dim=1, dtype=torch.int64)
    fl = failed.to(torch.int64)
    expect = {"frames": N, "failures": int(fl.sum()), "bit_errors": int(nb.sum()),
              "frame_errors": int(((fl == 1) | (nb > 0)).sum()), "undetected": int(((fl == 0) & (nb > 0)).sum()),
              "iterations": int(torch.where(fl == 1, MAX_ITER, it.to(torch.int64) + 1).sum())}
    assert c == expect, (name, ebno, variant, c, expect)


@gpu
def test_bench_batch_against_the_oracle(ctx):
    """bench.py's rank-0 batch itself (seed 0, point 8, frames 0 .. 2^22 - 1 at 4 dB), decoded whole; a seeded sample of
    8192 of its frames -- all distinct -- against the oracle, and no row left unwritten"""
    import torch
    import channelcoding_b200 as cc
    code = gpu_bch(ctx, "bch_63_36")
    N = 1 << 22
    y = torch.empty((N, 63), dtype=torch.float32, device="cuda")
    ctx.awgn_llr(63, np.float32(cc.sigma(code.rate, 4.0)), seed=0, point=int(round(4.0 * 2)), frame0=0, frames=N, out=y)
    out = ms_outputs(N, 63, True)
    code.decode(y, "NMS", 0.8, 0.0, MAX_ITER, 0, want_L=True, out=out)
    torch.cuda.synchronize()
    assert int((out[3] > 1).sum()) == 0 and int((out[2] > MAX_ITER).sum()) == 0
    idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(N, 8192, replace=False))).cuda()
    ys = y[idx].cpu().numpy()
    ref = ms_ref(oracle.Code(0, 6, 5).H(), ys, "NMS", 0.8)
    got = {k: v[idx] for k, v in ms_got(out).items()}
    check_tiled(got, ref_on(ref), torch.arange(8192, device="cuda"), "bench.py batch sample")
