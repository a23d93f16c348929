"""Maximum-likelihood decoding of high-rate binary BCH codes (ccgpu_decode_llr_ml / ccgpu_awgn_point_ml, kernel K9).

The CPU restatement below implements the contract of include/ccgpu.h literally, vectorised over frames x states in
float32: every state compares its two incoming sums M_c(pred) + cost as written (no butterflies, no zero-cost
shortcut), ties go to x_c = h_c, and the traceback walks the stored decisions from state 0.  The tests without a gpu
mark check the restatement against a brute-force search over every codeword and against OSD-3; the others pin the
GPU against it bit for bit."""
import os
import subprocess

import numpy as np
import pytest

import oracle
from test_gpu_osd import osd_restatement, noisy_codewords, special_values, key_of

# (q, t) of the eight supported codes (n <= 127, k = n - l <= 12)
CODES = {"bch_15_11": (4, 1), "bch_15_7": (4, 2), "bch_15_5": (4, 3), "bch_31_26": (5, 1), "bch_31_21": (5, 2),
         "bch_63_57": (6, 1), "bch_63_51": (6, 2), "bch_127_120": (7, 1)}
BOUND = np.float32(2.0 ** 20)


class Code:
    """a code with what the restatement needs: H (k x n), the column syndromes, and G (l x n) for the brute force"""

    def __init__(self, name):
        self.oc = oracle.Code(0, *CODES[name])
        self.n, self.l = self.oc.n, self.oc.l
        self.k = self.n - self.l
        self.H = self.oc.H()
        self.sigma = (self.H.astype(np.int64) << np.arange(self.k)[:, None]).sum(axis=0)
        self.G = self.oc.encode(np.eye(self.l, dtype=np.uint8))


_CODES = {}


def code_of(name):
    if name not in _CODES:
        _CODES[name] = Code(name)
    return _CODES[name]


def weights(y):
    """w_c = fminf(|y_c|, 2^20), NaN -> +0.0"""
    return np.where(np.isnan(y), np.float32(0), np.minimum(np.abs(y), BOUND)).astype(np.float32)


def metric(x, h, w):
    """D: float32 sum of w_c over the columns where x != h, ascending c, from +0.0 (sequential, not pairwise)"""
    return np.cumsum(np.where(x != h, w, np.float32(0)), axis=-1, dtype=np.float32)[..., -1]


def ml_restatement(R, y, chunk=256):
    """-> bits (frames, n) uint8, M_n(0) (frames,) float32"""
    y = np.ascontiguousarray(y, np.float32).reshape(-1, R.n)
    bits = np.zeros(y.shape, np.uint8)
    Mn = np.zeros(len(y), np.float32)
    states = np.arange(1 << R.k)
    zero = np.float32(0)
    for f0 in range(0, len(y), chunk):
        yy = y[f0:f0 + chunk]
        F = len(yy)
        h, w = yy < 0, weights(yy)
        M = np.full((F, 1 << R.k), np.inf, np.float32)
        M[:, 0] = 0
        d = np.zeros((R.n, F, 1 << R.k), bool)
        for c in range(R.n):
            hc = h[:, c:c + 1]
            s0 = M + np.where(hc, w[:, c:c + 1], zero)                       # x_c = 0 from s
            s1 = M[:, states ^ R.sigma[c]] + np.where(hc, zero, w[:, c:c + 1])  # x_c = 1 from s ^ sigma_c
            take1 = (s1 < s0) | ((s1 == s0) & hc)
            M = np.where(take1, s1, s0)
            d[c] = take1
        s = np.zeros(F, np.int64)
        rows = np.arange(F)
        for c in range(R.n - 1, -1, -1):
            x = d[c, rows, s]
            bits[f0:f0 + F, c] = x
            s ^= np.where(x, R.sigma[c], 0)
        Mn[f0:f0 + F] = M[:, 0]
    return bits, Mn


def is_codeword(R, x):
    return not ((R.H.astype(np.int64) @ np.atleast_2d(x).astype(np.int64).T) % 2).any()


def all_codewords(R):
    """the 2^l codewords as rows of bits, from the XOR span of G's rows packed as integers"""
    words = np.zeros(1, np.int64)
    for g in R.G:
        packed = int(sum(int(b) << c for c, b in enumerate(g)))
        words = np.concatenate([words, words ^ packed])
    return ((words[:, None] >> np.arange(R.n)) & 1).astype(np.uint8)


def mixed_inputs(R, frames, ebno, seed):
    """waterfall noise, quantised values (metric ties), special values (+-0, +-inf, NaN)"""
    rng = np.random.default_rng(seed)
    _, y1 = noisy_codewords(R.oc, frames, ebno, rng)
    _, y2 = noisy_codewords(R.oc, frames, ebno, rng, quantise=True)
    y3 = special_values(frames, R.n, rng)
    return {"waterfall": y1, "quantised": y2, "special": y3}


# ---------------------------------------------------------------- the restatement (CPU)

@pytest.mark.parametrize("name,frames", [("bch_15_11", 60), ("bch_15_7", 60), ("bch_15_5", 60), ("bch_31_21", 4)])
def test_restatement_is_maximum_likelihood(name, frames):
    """the restatement's word is a codeword, its D is M_n(0), and K(D) is the minimum over all 2^l codewords"""
    R = code_of(name)
    every = all_codewords(R)
    assert is_codeword(R, every)
    for what, y in mixed_inputs(R, frames, 1.0, 1).items():
        bits, Mn = ml_restatement(R, y)
        for f in range(len(y)):
            h, w = y[f] < 0, weights(y[f])
            assert is_codeword(R, bits[f]), (what, f)
            D = metric(bits[f], h, w)
            assert key_of(np.array([D], np.float32))[0] == key_of(Mn[f:f + 1])[0], (what, f)
            Dall = np.zeros(len(every), np.float32)
            for c in range(R.n):  # sequential float32 sum over every codeword at once
                Dall = Dall + np.where(every[:, c] != h[c], w[c], np.float32(0))
            assert key_of(Mn[f:f + 1])[0] == key_of(Dall).min(), (what, f)


def test_codeword_is_returned_unchanged():
    for name in ("bch_15_5", "bch_31_21", "bch_63_51"):
        R = code_of(name)
        rng = np.random.default_rng(4)
        x, _ = noisy_codewords(R.oc, 40, 3.0, rng)
        y = ((1.0 - 2.0 * x) * rng.uniform(0.1, 2.0, x.shape)).astype(np.float32)
        y[:5] = 1.0 - 2.0 * x[:5]  # equal magnitudes
        bits, Mn = ml_restatement(R, y)
        assert np.array_equal(bits, x) and not key_of(Mn).any()


@pytest.mark.parametrize("name,frames,ebno", [("bch_31_21", 200, 2.0), ("bch_63_57", 40, 3.0), ("bch_63_51", 30, 3.0)])
def test_restatement_beats_osd3(name, frames, ebno):
    """D(ML) <= D(OSD-3) on every frame, both measured with the contract's metric"""
    R = code_of(name)  # carries what osd_restatement reads: n, l, k, H, G
    rng = np.random.default_rng(5)
    _, y = noisy_codewords(R.oc, frames, ebno, rng)
    bits, Mn = ml_restatement(R, y)
    ob, _, _ = osd_restatement(R, y, 3)
    h, w = y < 0, weights(y)
    Dml, Dosd = metric(bits, h, w), metric(ob, h, w)
    assert (key_of(Dml) <= key_of(Dosd)).all()
    assert (key_of(Dml) == key_of(Mn)).all()


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


def as_np(a):
    return np.asarray(a.cpu()) if hasattr(a, "cpu") else a


# (code, Eb/N0 of the waterfall, frames): ragged counts
PARITY = {"bch_15_11": (2.0, 4099), "bch_15_7": (2.0, 4099), "bch_15_5": (1.0, 4099), "bch_31_26": (3.0, 4099),
          "bch_31_21": (3.0, 4099), "bch_63_57": (4.0, 3001), "bch_63_51": (4.0, 1001), "bch_127_120": (5.0, 2001)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PARITY))
def test_restatement_parity(ctx, name):
    """bit-exact bits: waterfall AWGN on random codewords (ragged counts), quantised values (metric ties), special
    values, a single frame; host buffers and torch CUDA tensors"""
    import torch
    R = code_of(name)
    code = gpu_code(ctx, name)
    ebno, frames = PARITY[name]
    ys = mixed_inputs(R, 33, ebno, 100)
    rng = np.random.default_rng(101)
    ys["waterfall"] = noisy_codewords(R.oc, frames, ebno, rng)[1]
    ys["one frame"] = ys["waterfall"][:1]
    for what, y in ys.items():
        rb, _ = ml_restatement(R, y)
        got = code.decode_ml(y)
        assert np.array_equal(got, rb), (what, "host", int((got != rb).any(axis=1).sum()))
        got = code.decode_ml(torch.from_numpy(y).cuda())
        torch.cuda.synchronize()
        got = as_np(got)
        assert np.array_equal(got, rb), (what, "torch", int((got != rb).any(axis=1).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("name,ebno", [("bch_63_51", 4.0), ("bch_63_57", 5.0), ("bch_31_21", 3.0)])
def test_kernel_against_kernels(ctx, name, ebno):
    """on the same frames of the AWGN stream: D(ML) <= D(OSD-3) and <= D(Chase p = 8) wherever Chase succeeds, and every
    frame of the OSD-3 ML lower bound (nonzero word strictly closer to y than the all-zero word sent) is an ML error"""
    import channelcoding_b200 as cc
    code = gpu_code(ctx, name)
    F = 20000
    y = ctx.awgn_llr(code.n, np.float32(cc.sigma(code.rate, ebno)), seed=1, point=3, frame0=0, frames=F)
    h, w = y < 0, weights(y)
    ml = code.decode_ml(y)
    osd, _ = code.decode_osd(y, 3)
    ch, failed, _ = code.decode_chase(y, 8)
    Dml, Dosd, Dch = metric(ml, h, w), metric(osd, h, w), metric(ch, h, w)
    Dzero = metric(np.zeros_like(ml), h, w)
    assert (Dml <= Dosd).all()
    ok = failed == 0
    assert ok.sum() > F // 2 and (Dml[ok] <= Dch[ok]).all()
    bound = osd.any(axis=1) & (Dosd < Dzero)
    assert bound.sum() > 0 or ebno >= 5.0
    assert ml.any(axis=1)[bound].all()
    assert ml.any(axis=1).sum() >= bound.sum()


@pytest.mark.gpu
@pytest.mark.parametrize("name,ebno,frames", [("bch_63_51", 4.0, 40000), ("bch_31_21", 3.0, 30001),
                                              ("bch_127_120", 6.0, 20000), ("bch_15_7", 3.0, 40000),
                                              ("bch_63_57", 9.0, 30000)])
def test_fused_point(ctx, name, ebno, frames):
    """ccgpu_awgn_point_ml == K1 -> ccgpu_decode_llr_ml -> host count; a device out accumulates; a group agrees"""
    import channelcoding_b200 as cc
    import torch
    code = gpu_code(ctx, name)
    y = ctx.awgn_llr(code.n, np.float32(cc.sigma(code.rate, ebno)), seed=9, point=4, frame0=77, frames=frames)
    nz = (code.decode_ml(y) != 0).sum(axis=1)
    c = code.awgn_point_ml(ebno, frames, seed=9, point=4, frame0=77)
    assert c["frames"] == frames and c["iterations"] == 0 and c["failures"] == 0
    assert c["bit_errors"] == int(nz.sum())
    assert c["frame_errors"] == int((nz > 0).sum()) == c["undetected"]
    dev = torch.tensor([5, 4, 3, 2, 1, 0, 7, 8], dtype=torch.int64, device="cuda:0")
    code.awgn_point_ml(ebno, frames, seed=9, point=4, frame0=77, out=dev)
    torch.cuda.synchronize()
    keys = ("frames", "frame_errors", "bit_errors", "iterations", "failures", "undetected")
    assert dev.cpu().tolist() == [v + c[k] for v, k in zip((5, 4, 3, 2, 1, 0), keys)] + [7, 8]
    g = cc.Group(list(range(torch.cuda.device_count())))
    g.set_min_frames(1000)
    gc = g.bch(CODES[name][0], errors=CODES[name][1])
    assert gc.awgn_point_ml(ebno, frames, seed=9, point=4, frame0=77) == c
    g.close()


@pytest.mark.gpu
def test_errors_and_launches(ctx):
    import torch
    from channelcoding_b200 import CcgpuError
    from channelcoding_b200._lib import ERR_INVALID, ERR_UNSUPPORTED
    code = gpu_code(ctx, "bch_63_51")
    # RS, dense H, k > 12 (BCH(31,16): k = 15, BCH(63,36): k = 27), n = 255 (BCH(255,247): k = 8)
    for other in (ctx.rs(8, 16), ctx.from_dense(code.H(), code.rate), ctx.bch(5, errors=3), ctx.bch(6, errors=5),
                  ctx.bch(8, errors=1)):
        with pytest.raises(CcgpuError) as e:
            other.decode_ml(np.ones((4, other.n), np.float32))
        assert e.value.code == ERR_UNSUPPORTED
        with pytest.raises(CcgpuError) as e:
            other.awgn_point_ml(4.0, 100)
        assert e.value.code == ERR_UNSUPPORTED
    y = np.ones((4, 63), np.float32)
    assert code.decode_ml(np.zeros((0, 63), np.float32)).shape == (0, 63)
    assert code.awgn_point_ml(4.0, 0)["frames"] == 0
    yd = torch.ones((4, 63), dtype=torch.float32, device="cuda:0")
    with pytest.raises(CcgpuError) as e:
        code.decode_ml(yd, out=np.empty((4, 63), np.uint8))
    assert e.value.code == ERR_INVALID
    with pytest.raises(CcgpuError) as e:
        code.decode_ml(y, out=torch.empty((4, 63), dtype=torch.uint8, device="cuda:0"))
    assert e.value.code == ERR_INVALID
    # set_rows does not change ML
    y = noisy_codewords(code_of("bch_63_51").oc, 3000, 3.0, np.random.default_rng(6))[1]
    r = code.decode_ml(y)
    code.set_rows(40)
    assert np.array_equal(code.decode_ml(y), r)
    # exactly one launch per device call and per fused point
    yd = torch.from_numpy(y).cuda()
    out = torch.empty((3000, 63), dtype=torch.uint8, device="cuda:0")
    before = ctx.kernel_launches
    code.decode_ml(yd, out=out)
    assert ctx.kernel_launches == before + 1
    dev = torch.zeros(8, dtype=torch.int64, device="cuda:0")
    code.awgn_point_ml(4.0, 100000, out=dev)
    assert ctx.kernel_launches == before + 2
    torch.cuda.synchronize()


# ---------------------------------------------------------------- full size, tiled against the restatement

@pytest.mark.gpu
@pytest.mark.parametrize("path,N", [("device", 4194304), ("host", 1000003)])
def test_full_size_tiled(ctx, path, N):
    """ML on BCH(63,51) at full batch sizes: torch tensors, and host memory through the three-slot pipeline; every row
    against the restatement of the pool frame it holds, outputs prefilled with sentinels"""
    import torch
    import test_gpu_scale as scale
    R = code_of("bch_63_51")
    y = scale.pool_y("bch_63_51", 4096, (2.0, 3.0, 4.0, 5.0, 6.0), 16, True)
    (b,) = scale.oracle_map(lambda rows: ml_restatement(R, rows, chunk=64)[:1], y, chunk=64)
    pool = scale.Pool(y, {"bits": b})
    code = gpu_code(ctx, "bch_63_51")
    src_np = scale.tiling(pool.M, N, 123)
    src = torch.from_numpy(src_np).cuda()
    lib = "numpy" if path == "host" else "torch"
    u8 = np.uint8 if lib == "numpy" else torch.uint8
    out = scale.sentinel_like((N, 63), u8, "bits", lib)
    yy = pool.y[src_np] if lib == "numpy" else scale.to_dev(pool.y)[src]
    code.decode_ml(yy, out=out)
    torch.cuda.synchronize()
    scale.check_tiled({"bits": scale.to_dev(out)}, scale.ref_on(pool.ref), src, "ML " + path)


# ---------------------------------------------------------------- the C++ layer

@pytest.fixture(scope="module")
def bins():
    from channelcoding_b200 import build as _build
    _build.build()
    return {os.path.basename(p): p for p in _build.build_tools()}


def test_cpp_ml_tag(bins):
    r = subprocess.run([bins["ml_test"], "--host"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_cpp_ml_decoder(bins, tmp_path):
    r = subprocess.run([bins["ml_test"], "--gpu", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_cli_ml(bins, tmp_path):
    """benchmark --algorithm ml writes "(63, 51, 5)-ML.log" in the reference's format, and only that log"""
    r = subprocess.run([bins["benchmark"], "--algorithm", "ml", "--k", "6", "--dmin", "5", "--max-samples", "100000",
                        "--seed", "3", "--out", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert sorted(p.name for p in tmp_path.glob("*.log")) == ["(63, 51, 5)-ML.log"]
    lines = open(tmp_path / "(63, 51, 5)-ML.log").read().splitlines()
    assert lines[0] == "   ebno                   wer" and len(lines) >= 5
    wers = [float(x.split()[1]) for x in lines[1:]]
    assert wers[0] > wers[-1]
