"""Ordered-statistics decoding of binary BCH codes (ccgpu_decode_llr_osd / ccgpu_awgn_point_osd, kernel K6).

The CPU restatement below implements the contract of include/ccgpu.h literally and by a route independent of the
kernel's: np.lexsort for the visiting order, a greedy GF(2) rank over the H-columns for the information set, the
candidates from a generator matrix G (oracle.Code.encode of the unit messages) solved on I as G' = G_I^-1 G (no
elimination of H), the float32 cumulative sum for the metric and the (K(D), e) minimum.  The tests without a gpu mark
check the restatement itself; the others pin the GPU against it bit for bit."""
import itertools
import os
import subprocess

import numpy as np
import pytest

import oracle

CODES = {"bch_15_7": (4, 2), "bch_15_5": (4, 3), "bch_31_16": (5, 3), "bch_31_21": (5, 2), "bch_63_36": (6, 5),
         "bch_63_45": (6, 3), "bch_127_64": (7, 10), "bch_127_106": (7, 3)}
NAN_KEY = np.uint32(0x7FC00000)


class Ref:
    """a code with the matrices the restatement needs: H (k x n) and G (l x n, row i = encode of unit message i)"""

    def __init__(self, name):
        self.oc = oracle.Code(0, *CODES[name])
        self.n, self.l, self.k = self.oc.n, self.oc.l, self.oc.n - self.oc.l
        self.H = self.oc.H()
        self.G = self.oc.encode(np.eye(self.l, dtype=np.uint8))


_REFS = {}


def ref(name):
    if name not in _REFS:
        _REFS[name] = Ref(name)
    return _REFS[name]


def visiting_order(y):
    """columns per frame in ascending (bits of |y_c| as uint32, c)"""
    key = np.abs(y).view(np.uint32)
    cols = np.broadcast_to(np.arange(y.shape[1]), y.shape)
    return np.lexsort((cols, key), axis=-1)


def greedy_pick(M, order, count):
    """the columns of M picked greedily in `order`, a column being picked when it is not in the GF(2) span of the
    columns picked before it; stops after `count` picks"""
    basis = {}  # leading bit -> vector, both as Python ints over the rows of M
    picked = []
    for c in order:
        v = int("".join("1" if b else "0" for b in M[:, c]) or "0", 2)
        while v:
            top = v.bit_length() - 1
            if top not in basis:
                basis[top] = v
                picked.append(int(c))
                break
            v ^= basis[top]
        if len(picked) == count:
            break
    return picked


def information_set(R, y_row):
    """I (ascending) of one frame: the complement of the greedy pick P over the H-columns"""
    P = set(greedy_pick(R.H, visiting_order(y_row[None])[0], R.k))
    assert len(P) == R.k
    return np.array([c for c in range(R.n) if c not in P])


def systematic_on(G, I):
    """G' = G_I^-1 G: the generator whose row a is the codeword with x[I] = unit vector a"""
    M = G.copy()
    for a, c in enumerate(I):
        r = a + int(np.nonzero(M[a:, c])[0][0])
        M[[a, r]] = M[[r, a]]
        hit = M[:, c].astype(bool)
        hit[a] = False
        M[hit] ^= M[a]
    return M


def subsets(l, order):
    """E_0, E_1, ..: empty, singles, pairs, triples .. up to min(order, l), each lexicographic"""
    out = []
    for w in range(min(order, l) + 1):
        out += list(itertools.combinations(range(l), w))
    return out


def metric(x, h, y):
    """D: float32 sum of |y_c| over the columns where x != h, ascending c, from +0.0"""
    return np.cumsum(np.where(x != h, np.abs(y), np.float32(0)), axis=-1, dtype=np.float32)[..., -1]


def key_of(D):
    """K(D): the bits of D as uint32, every NaN as 0x7fc00000"""
    k = np.asarray(D, np.float32).view(np.uint32).copy()
    k[np.isnan(D)] = NAN_KEY
    return k


def osd_restatement(R, y, order):
    """-> bits (frames, n) uint8, weight (frames,) uint8, D of the returned word (float32)"""
    y = np.ascontiguousarray(y, np.float32).reshape(-1, R.n)
    frames = y.shape[0]
    sets = subsets(R.l, order)
    wts = np.array([len(s) for s in sets], np.uint8)
    # flipped positions of each candidate, padded with index l (a zero row appended to G')
    E = np.full((len(sets), max(1, min(order, R.l))), R.l, np.int64)
    for e, s in enumerate(sets):
        E[e, :len(s)] = s
    bits = np.zeros((frames, R.n), np.uint8)
    weight = np.zeros(frames, np.uint8)
    D = np.zeros(frames, np.float32)
    for f in range(frames):
        h = (y[f] < 0).astype(np.uint8)
        I = information_set(R, y[f])
        Gs = systematic_on(R.G, I)
        x0 = (h[I].astype(np.int64) @ Gs.astype(np.int64) % 2).astype(np.uint8)  # the codeword with x[I] = h[I]
        Gz = np.concatenate([Gs, np.zeros((1, R.n), np.uint8)])
        X = np.bitwise_xor.reduce(Gz[E], axis=1) ^ x0              # x_e[I] = h[I] ^ 1_{E_e}
        De = metric(X, h[None, :], y[f][None, :])
        best = int(np.argmin(key_of(De)))                       # first index among equal keys: the smallest e
        bits[f], weight[f], D[f] = X[best], wts[best], De[best]
    return bits, weight, D


def noisy_codewords(oc, frames, ebno, rng, quantise=False):
    msgs = rng.integers(0, 2, size=(frames, oc.l)).astype(np.uint8)
    x = oc.encode(msgs)
    y = (1.0 - 2.0 * x + oracle.sigma(oc.rate, ebno) * rng.standard_normal(x.shape)).astype(np.float32)
    if quantise:
        y = (np.round(y * 4) / 4).astype(np.float32)
    return x, y


def special_values(frames, n, rng):
    """frames whose entries include +-0, +-inf and NaN"""
    y = (1.0 + 0.8 * rng.standard_normal((frames, n))).astype(np.float32)
    vals = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan], np.float32)
    mask = rng.random((frames, n)) < 0.06
    y[mask] = vals[rng.integers(0, len(vals), mask.sum())]
    return y


def is_codeword(R, x):
    return not ((R.H.astype(np.int64) @ x.astype(np.int64).T) % 2).any()


# ---------------------------------------------------------------- the restatement (CPU)

@pytest.mark.parametrize("name", ["bch_15_7", "bch_31_16", "bch_63_36", "bch_127_64"])
def test_information_set_duality(name):
    """matroid duality: I, the complement of the greedy pick over the H-columns in ascending order, is the set of l
    columns picked greedily over the G-columns in descending order; on noise, quantised ties, +-0, +-inf and NaN"""
    R = ref(name)
    rng = np.random.default_rng(1)
    _, y1 = noisy_codewords(R.oc, 20, 3.0, rng)
    _, y2 = noisy_codewords(R.oc, 20, 3.0, rng, quantise=True)
    ys = np.concatenate([y1, y2, special_values(20, R.n, rng), np.full((1, R.n), -0.0, np.float32)])
    for y in ys:
        I = information_set(R, y)
        from_G = sorted(greedy_pick(R.G, visiting_order(y[None])[0][::-1], R.l))
        assert I.tolist() == from_G


@pytest.mark.parametrize("name", ["bch_15_7", "bch_15_5"])
def test_full_order_is_maximum_likelihood(name):
    """order = l makes every codeword a candidate: D of the result is the smallest over a brute-force search of all
    2^l codewords, and the result is a codeword"""
    R = ref(name)
    rng = np.random.default_rng(2)
    _, y = noisy_codewords(R.oc, 200, 1.0, rng)
    y[:40] = (np.round(y[:40] * 2) / 2).astype(np.float32)
    every = R.oc.encode(np.array(list(itertools.product((0, 1), repeat=R.l)), np.uint8))
    bits, weight, D = osd_restatement(R, y, R.l)
    for f in range(len(y)):
        h = (y[f] < 0).astype(np.uint8)
        Dall = metric(every, h[None, :], y[f][None, :])
        assert key_of(D[f:f + 1])[0] == key_of(Dall).min()
        assert is_codeword(R, bits[f])


@pytest.mark.parametrize("name,order", [("bch_31_16", 1), ("bch_63_36", 2), ("bch_63_45", 3)])
def test_sent_codeword_within_order_is_beaten_or_matched(name, order):
    """when the sent codeword differs from h in at most `order` positions of I it is a candidate: D <= D(sent)"""
    R = ref(name)
    rng = np.random.default_rng(3)
    x, y = noisy_codewords(R.oc, 300, 2.0, rng)
    bits, _, D = osd_restatement(R, y, order)
    checked = 0
    for f in range(len(y)):
        h = (y[f] < 0).astype(np.uint8)
        I = information_set(R, y[f])
        if int((h[I] != x[f][I]).sum()) <= order:
            checked += 1
            assert key_of(D[f:f + 1])[0] <= key_of(metric(x[f], h, y[f]))
    assert checked > 100


def test_codeword_is_returned_unchanged():
    R = ref("bch_31_16")
    rng = np.random.default_rng(4)
    x, _ = noisy_codewords(R.oc, 50, 3.0, rng)
    y = ((1.0 - 2.0 * x) * rng.uniform(0.1, 2.0, x.shape)).astype(np.float32)
    bits, weight, D = osd_restatement(R, y, 2)
    assert np.array_equal(bits, x) and not weight.any() and not key_of(D).any()


# ---------------------------------------------------------------- the GPU against it

@pytest.fixture(scope="module")
def ctx():
    import channelcoding_b200 as cc
    c = cc.Context(0)
    yield c
    c.close()


def gpu_code(ctx, name):
    q, t = CODES[name]
    return ctx.bch(q, errors=t)


def assert_same(got, ref_out, what):
    bits, weight = (np.asarray(a.cpu()) if hasattr(a, "cpu") else a for a in got)
    rb, rw = ref_out[:2]
    assert np.array_equal(weight, rw), (what, "weight", int((weight != rw).sum()))
    assert np.array_equal(bits, rb), (what, "bits", int((bits != rb).any(axis=1).sum()))


# (code, Eb/N0 of the waterfall, frames per order 0..3): n = 127 at order 3 over ~100 frames keeps the restatement short
PARITY_CODES = {"bch_15_7": (2.0, (4099, 4099, 4099, 4099)), "bch_31_16": (2.5, (4099, 4099, 2000, 1000)),
                "bch_31_21": (3.0, (4099, 2000, 1000, 500)), "bch_63_36": (3.5, (4099, 2000, 1000, 300)),
                "bch_63_45": (4.0, (2000, 1000, 500, 200)), "bch_127_64": (4.0, (1000, 500, 200, 100)),
                "bch_127_106": (5.0, (1000, 300, 100, 100))}
PARITY = [(name, order) for name in PARITY_CODES for order in range(4)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,order", PARITY)
def test_restatement_parity(ctx, name, order):
    """bit-exact bits / weight: waterfall AWGN on random codewords (ragged counts), quantised values (order and metric
    ties), special values, a single frame; host buffers and torch CUDA tensors"""
    import torch
    R = ref(name)
    code = gpu_code(ctx, name)
    ebno, counts = PARITY_CODES[name]
    rng = np.random.default_rng(100 + order)
    _, y1 = noisy_codewords(R.oc, counts[order], ebno, rng)
    _, y2 = noisy_codewords(R.oc, 33, ebno, rng, quantise=True)
    y3 = special_values(33, R.n, rng)
    for what, y in (("waterfall", y1), ("quantised", y2), ("special", y3), ("one frame", y1[:1])):
        r = osd_restatement(R, y, order)
        assert_same(code.decode_osd(y, order), r, what + " host")
        got = code.decode_osd(torch.from_numpy(y).cuda(), order)
        torch.cuda.synchronize()
        assert_same(got, r, what + " torch")


@pytest.mark.gpu
@pytest.mark.parametrize("name,ebno,frames", [("bch_31_16", 3.0, 40000), ("bch_63_36", 4.0, 30001),
                                              ("bch_127_64", 5.0, 10000), ("bch_63_36", 8.0, 30000)])
def test_fused_point(ctx, name, ebno, frames):
    """ccgpu_awgn_point_osd == K1 -> ccgpu_decode_llr_osd -> host count; a device out accumulates; a group agrees"""
    import channelcoding_b200 as cc
    import torch
    code = gpu_code(ctx, name)
    order = 2
    y = ctx.awgn_llr(code.n, np.float32(cc.sigma(code.rate, ebno)), seed=9, point=4, frame0=77, frames=frames)
    bits, _ = code.decode_osd(y, order)
    nz = (bits != 0).sum(axis=1)
    c = code.awgn_point_osd(ebno, frames, order, seed=9, point=4, frame0=77)
    assert c["frames"] == frames and c["iterations"] == 0 and c["failures"] == 0
    assert c["bit_errors"] == int(nz.sum())
    assert c["frame_errors"] == int((nz > 0).sum()) == c["undetected"]
    dev = torch.tensor([5, 4, 3, 2, 1, 0, 7, 8], dtype=torch.int64, device="cuda:0")
    code.awgn_point_osd(ebno, frames, order, seed=9, point=4, frame0=77, out=dev)
    torch.cuda.synchronize()
    keys = ("frames", "frame_errors", "bit_errors", "iterations", "failures", "undetected")
    assert dev.cpu().tolist() == [v + c[k] for v, k in zip((5, 4, 3, 2, 1, 0), keys)] + [7, 8]
    g = cc.Group(list(range(torch.cuda.device_count())))
    g.set_min_frames(1000)
    gc = g.bch(CODES[name][0], errors=CODES[name][1])
    assert gc.awgn_point_osd(ebno, frames, order, seed=9, point=4, frame0=77) == c
    g.close()


@pytest.mark.gpu
def test_statistics_against_chase_and_hard_decoding(ctx):
    """BCH(63,36) at 4 dB, 1e5 frames of the same noise stream (seed 1, point 3): OSD-2 leaves fewer frame errors than
    Chase-II with p = 4 (expected about 60 against 560), OSD-1 fewer than hard decoding"""
    code = gpu_code(ctx, "bch_63_36")
    F = 100000
    o2 = code.awgn_point_osd(4.0, F, 2, seed=1, point=3)
    o1 = code.awgn_point_osd(4.0, F, 1, seed=1, point=3)
    ch = code.awgn_point_chase(4.0, F, 4, seed=1, point=3)
    bm = code.awgn_point_hard(4.0, F, seed=1, point=3)
    assert o2["frames"] == o1["frames"] == ch["frames"] == bm["frames"] == F
    assert 0 < o2["frame_errors"] < ch["frame_errors"], (o2, ch)
    assert o1["frame_errors"] < bm["frame_errors"], (o1, bm)


@pytest.mark.gpu
def test_errors_and_launches(ctx):
    import torch
    from channelcoding_b200 import CcgpuError
    from channelcoding_b200._lib import ERR_INVALID, ERR_UNSUPPORTED
    code = gpu_code(ctx, "bch_63_36")
    y = np.ones((4, 63), np.float32)
    for call in (lambda: code.decode_osd(y, 4), lambda: code.awgn_point_osd(4.0, 100, 4)):
        with pytest.raises(CcgpuError) as e:
            call()
        assert e.value.code == ERR_INVALID
    # RS, dense H, n = 255, k > 64 (BCH(127,57): k = 70)
    for other in (ctx.rs(8, 16), ctx.from_dense(code.H(), code.rate), ctx.bch(8, errors=18), ctx.bch(7, errors=11)):
        with pytest.raises(CcgpuError) as e:
            other.decode_osd(np.ones((4, other.n), np.float32), 1)
        assert e.value.code == ERR_UNSUPPORTED
        with pytest.raises(CcgpuError) as e:
            other.awgn_point_osd(4.0, 100, 1)
        assert e.value.code == ERR_UNSUPPORTED
    bits, weight = code.decode_osd(np.zeros((0, 63), np.float32), 3)
    assert bits.shape == (0, 63) and weight.shape == (0,)
    assert code.awgn_point_osd(4.0, 0, 3)["frames"] == 0
    yd = torch.ones((4, 63), dtype=torch.float32, device="cuda:0")
    with pytest.raises(CcgpuError) as e:
        code.decode_osd(yd, 1, out=(np.empty((4, 63), np.uint8), torch.empty(4, dtype=torch.uint8, device="cuda:0")))
    assert e.value.code == ERR_INVALID
    with pytest.raises(CcgpuError) as e:
        code.decode_osd(y, 1, out=(np.empty((4, 63), np.uint8), torch.empty(4, dtype=torch.uint8, device="cuda:0")))
    assert e.value.code == ERR_INVALID
    # set_rows does not change OSD; weight may be left out
    r = code.decode_osd(y, 2)
    code.set_rows(40)
    bits, weight = code.decode_osd(y, 2)
    assert np.array_equal(bits, r[0]) and np.array_equal(weight, r[1])
    # exactly one launch per device call
    yd = torch.from_numpy(noisy_codewords(ref("bch_63_36").oc, 5000, 3.0, np.random.default_rng(6))[1]).cuda()
    out = (torch.empty((5000, 63), dtype=torch.uint8, device="cuda:0"), torch.empty(5000, dtype=torch.uint8, device="cuda:0"))
    before = ctx.kernel_launches
    code.decode_osd(yd, 2, out=out)
    assert ctx.kernel_launches == before + 1
    dev = torch.zeros(8, dtype=torch.int64, device="cuda:0")
    code.awgn_point_osd(4.0, 100000, 2, out=dev)
    assert ctx.kernel_launches == before + 2
    torch.cuda.synchronize()


# ---------------------------------------------------------------- full size, tiled against the restatement

@pytest.mark.gpu
@pytest.mark.parametrize("path,N", [("device", 4194304), ("host", 1000003)])
def test_full_size_tiled(ctx, path, N):
    """OSD-2 on BCH(63,36) at full batch sizes: torch tensors, and host memory through the three-slot pipeline;
    every row against the restatement of the pool frame it holds, outputs prefilled with sentinels"""
    import torch
    import test_gpu_scale as scale
    scale.SENTINEL.setdefault("weight", scale.SENT8)
    R = ref("bch_63_36")
    y = scale.pool_y("bch_63_36", 4096, (2.0, 3.0, 4.0, 5.0, 6.0), 16, True)
    b, w, _ = scale.oracle_map(lambda rows: osd_restatement(R, rows, 2), y, chunk=64)
    pool = scale.Pool(y, {"bits": b, "weight": w})
    code = gpu_code(ctx, "bch_63_36")
    src_np = scale.tiling(pool.M, N, 122)
    src = torch.from_numpy(src_np).cuda()
    lib = "numpy" if path == "host" else "torch"
    u8 = np.uint8 if lib == "numpy" else torch.uint8
    out = (scale.sentinel_like((N, 63), u8, "bits", lib), scale.sentinel_like(N, u8, "weight", lib))
    yy = pool.y[src_np] if lib == "numpy" else scale.to_dev(pool.y)[src]
    code.decode_osd(yy, 2, out=out)
    torch.cuda.synchronize()
    got = {k: scale.to_dev(v) for k, v in zip(("bits", "weight"), out)}
    scale.check_tiled(got, scale.ref_on(pool.ref), src, "OSD-2 " + path)


# ---------------------------------------------------------------- the C++ layer

@pytest.fixture(scope="module")
def bins():
    from channelcoding_b200 import build as _build
    _build.build()
    return {os.path.basename(p): p for p in _build.build_tools()}


def test_cpp_osd_tags(bins):
    r = subprocess.run([bins["osd_test"], "--host"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_cpp_osd_decoder(bins, tmp_path):
    r = subprocess.run([bins["osd_test"], "--gpu", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_cli_osd(bins, tmp_path):
    """benchmark --algorithm osd1 writes "(63, 45, 7)-OSD1.log" in the reference's format, and only that log"""
    r = subprocess.run([bins["benchmark"], "--algorithm", "osd1", "--k", "6", "--dmin", "7", "--max-samples", "100000",
                        "--seed", "3", "--out", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert sorted(p.name for p in tmp_path.glob("*.log")) == ["(63, 45, 7)-OSD1.log"]
    lines = open(tmp_path / "(63, 45, 7)-OSD1.log").read().splitlines()
    assert lines[0] == "   ebno                   wer" and len(lines) >= 5
    wers = [float(x.split()[1]) for x in lines[1:]]
    assert wers[0] > wers[-1]
