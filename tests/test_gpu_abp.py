"""Adaptive belief propagation of binary BCH codes (ccgpu_decode_llr_abp / ccgpu_awgn_point_abp, kernel K8).

Two CPU restatements of the contract of include/ccgpu.h:
- numpy, by a route independent of the kernel's: np.lexsort for the visiting order, the greedy GF(2) rank pick P of
  test_gpu_osd, A = (H[:, P])^-1 H by GF(2) inversion (no elimination in the visiting order), mu from a sort of the
  other columns' magnitudes (not from min1/min2), the float32 column sums in ascending row order;
- plain C (tests/abp_ref.c, compiled on first use), fast enough for the full-size pool.  A CPU test pins it bit for bit
  against the numpy one; the GPU tests compare the kernel against both."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oracle
from test_gpu_osd import greedy_pick, visiting_order

HERE = os.path.dirname(os.path.abspath(__file__))
CODES = {"bch_15_7": (4, 2), "bch_31_16": (5, 3), "bch_31_21": (5, 2), "bch_63_36": (6, 5), "bch_63_45": (6, 3),
         "bch_127_64": (7, 10), "bch_127_106": (7, 3)}
B = np.float32(2.0 ** 20)


class Ref:
    """a code with the matrices the restatements need: H (k x n) and G (l x n, row i = encode of unit message i)"""

    def __init__(self, name):
        self.oc = oracle.Code(0, *CODES[name])
        self.n, self.l, self.k = self.oc.n, self.oc.l, self.oc.n - self.oc.l
        self.H = np.ascontiguousarray(self.oc.H(), np.uint8)
        self.G = self.oc.encode(np.eye(self.l, dtype=np.uint8))


_REFS = {}


def ref(name):
    if name not in _REFS:
        _REFS[name] = Ref(name)
    return _REFS[name]


def gf2_inverse(M):
    """the inverse of a square GF(2) matrix by Gauss-Jordan on [M | I]"""
    k = M.shape[0]
    A = np.concatenate([M % 2, np.eye(k, dtype=np.uint8)], axis=1).astype(np.uint8)
    for col in range(k):
        r = col + int(np.nonzero(A[col:, col])[0][0])
        A[[col, r]] = A[[r, col]]
        hit = A[:, col].astype(bool)
        hit[col] = False
        A[hit] ^= A[col]
    return A[:, k:]


def adapted(R, L):
    """P (pick order) and A = (H[:, P])^-1 H for the soft values L of one frame"""
    P = greedy_pick(R.H, visiting_order(L[None])[0], R.k)
    assert len(P) == R.k
    A = (gf2_inverse(R.H[:, P]).astype(np.int64) @ R.H.astype(np.int64) % 2).astype(np.uint8)
    return P, A


def check_pass(A, L):
    """S_c = +0.0 + sum over the rows i holding c (ascending) of m_{i,c}, float32"""
    S = np.zeros(L.shape, np.float32)
    for row in A:
        cols = np.nonzero(row)[0]
        a = np.abs(L[cols])
        others = np.where(np.eye(len(cols), dtype=bool), np.float32(np.inf), a[None, :])
        mu = np.sort(others, axis=1)[:, 0] if len(cols) > 1 else np.zeros(1, np.float32)
        neg = (L[cols] < 0).astype(np.int64)
        s = (neg.sum() - neg) % 2
        S[cols] = S[cols] + np.where(s == 1, -mu, mu).astype(np.float32)
    return S


def abp_numpy(R, y, max_iter, gamma):
    """-> bits (frames, n) uint8, L (frames, n) float32, iter (frames,) uint8, failed (frames,) uint8"""
    y = np.ascontiguousarray(y, np.float32).reshape(-1, R.n)
    g = np.float32(gamma)
    out = (np.zeros(y.shape, np.uint8), np.zeros(y.shape, np.float32), np.zeros(len(y), np.uint8),
           np.zeros(len(y), np.uint8))
    for f in range(len(y)):
        L = np.where(np.isnan(y[f]), np.float32(0), np.clip(y[f], -B, B)).astype(np.float32)
        j = 0
        while True:
            x = (L < 0).astype(np.uint8)
            odd = bool((R.H.astype(np.int64) @ x % 2).any())
            if not odd or j == max_iter:
                break
            _, A = adapted(R, L)
            L = np.minimum(np.maximum(L + g * check_pass(A, L), -B), B).astype(np.float32)
            j += 1
        out[0][f], out[1][f], out[2][f], out[3][f] = x, L, j, odd
    return out


_CLIB = None


def clib():
    """tests/abp_ref.c compiled into a temporary directory"""
    global _CLIB
    if _CLIB is None:
        so = os.path.join(tempfile.mkdtemp(prefix="abp_ref_"), "abp_ref.so")
        subprocess.check_call(["cc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", "-o", so,
                               os.path.join(HERE, "abp_ref.c"), "-lm"])
        lib = C.CDLL(so)
        lib.abp_ref.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_void_p, C.c_uint64, C.c_uint, C.c_float, C.c_void_p,
                                C.c_void_p, C.c_void_p, C.c_void_p]
        lib.abp_ref.restype = None
        _CLIB = lib
    return _CLIB


def abp_c(R, y, max_iter, gamma):
    y = np.ascontiguousarray(y, np.float32).reshape(-1, R.n)
    F = len(y)
    bits, L = np.zeros((F, R.n), np.uint8), np.zeros((F, R.n), np.float32)
    it, failed = np.zeros(F, np.uint8), np.zeros(F, np.uint8)
    clib().abp_ref(R.H.ctypes.data, R.k, R.n, y.ctypes.data, F, max_iter, gamma, bits.ctypes.data, L.ctypes.data,
                   it.ctypes.data, failed.ctypes.data)
    return bits, L, it, failed


def abp_c_parallel(R, y, max_iter, gamma):
    import test_gpu_scale as scale
    return scale.oracle_map(lambda rows: abp_c(R, rows, max_iter, gamma), y, chunk=64)


def noisy_codewords(oc, frames, ebno, rng, quantise=False):
    msgs = rng.integers(0, 2, size=(frames, oc.l)).astype(np.uint8)
    x = oc.encode(msgs)
    y = (1.0 - 2.0 * x + oracle.sigma(oc.rate, ebno) * rng.standard_normal(x.shape)).astype(np.float32)
    if quantise:
        y = (np.round(y * 4) / 4).astype(np.float32)
    return x, y


def edge_frames(n, rng):
    """the edge frames of test_gpu_scale (+-0, ties, subnormals, +-1e30, +-inf, NaN)"""
    import test_gpu_scale as scale
    return scale.edge_frames(n, rng, nonfinite=True)


def same_outputs(got, want, what):
    bits, L, it, failed = (np.asarray(a.cpu()) if hasattr(a, "cpu") else a for a in got)
    wb, wL, wi, wf = want
    assert np.array_equal(failed, wf), (what, "failed", int((failed != wf).sum()))
    assert np.array_equal(it, wi), (what, "iter", int((it != wi).sum()))
    assert np.array_equal(bits, wb), (what, "bits", int((bits != wb).any(axis=1).sum()))
    assert np.array_equal(L.view(np.uint32), wL.view(np.uint32)), (what, "L", int((L.view(np.uint32) != wL.view(np.uint32)).any(axis=1).sum()))


# ---------------------------------------------------------------- the restatements (CPU)

@pytest.mark.parametrize("name", ["bch_15_7", "bch_31_16", "bch_63_36", "bch_127_64"])
def test_adapted_matrix(name):
    """A G^T = 0 (same row space as H, full rank k) and A[:, P] = I in pick order, on noise, ties and edge values"""
    R = ref(name)
    rng = np.random.default_rng(1)
    _, y1 = noisy_codewords(R.oc, 10, 2.0, rng)
    _, y2 = noisy_codewords(R.oc, 10, 2.0, rng, quantise=True)
    for y in np.concatenate([y1, y2, edge_frames(R.n, rng)]):
        L = np.where(np.isnan(y), np.float32(0), np.clip(y, -B, B)).astype(np.float32)
        P, A = adapted(R, L)
        assert not ((A.astype(np.int64) @ R.G.T.astype(np.int64)) % 2).any()
        assert np.array_equal(A[:, P], np.eye(R.k, dtype=np.uint8))


def test_codewords_stop_at_once():
    R = ref("bch_31_16")
    rng = np.random.default_rng(2)
    x, _ = noisy_codewords(R.oc, 40, 3.0, rng)
    y = ((1.0 - 2.0 * x) * rng.uniform(0.1, 2.0, x.shape)).astype(np.float32)
    bits, L, it, failed = abp_numpy(R, y, 50, 0.15)
    assert np.array_equal(bits, x) and not it.any() and not failed.any() and np.array_equal(L, y)


def test_max_iter_zero_is_the_syndrome_test():
    R = ref("bch_63_36")
    rng = np.random.default_rng(3)
    _, y = noisy_codewords(R.oc, 200, 4.0, rng)
    bits, L, it, failed = abp_numpy(R, y, 0, 0.15)
    h = (y < 0).astype(np.uint8)
    assert np.array_equal(bits, h) and not it.any()
    assert np.array_equal(failed, ((R.H.astype(np.int64) @ h.T.astype(np.int64)) % 2).any(axis=0).astype(np.uint8))
    assert 0 < failed.sum() < len(y)


def test_single_error_on_the_least_reliable_bit():
    """BCH(15,7): one wrong sign on the least reliable bit, every other bit reliable, is corrected by one update"""
    R = ref("bch_15_7")
    rng = np.random.default_rng(4)
    x, _ = noisy_codewords(R.oc, 50, 3.0, rng)
    y = ((1.0 - 2.0 * x) * rng.uniform(0.5, 1.5, x.shape)).astype(np.float32)
    pos = rng.integers(0, R.n, len(y))
    y[np.arange(len(y)), pos] = -np.sign(y[np.arange(len(y)), pos]) * np.float32(0.05)
    bits, _, it, failed = abp_numpy(R, y, 50, 0.15)
    assert np.array_equal(bits, x) and (it == 1).all() and not failed.any()


@pytest.mark.parametrize("name,max_iter,gamma", [("bch_15_7", 50, 0.15), ("bch_31_21", 5, 1.0), ("bch_63_36", 50, 0.15),
                                                 ("bch_63_45", 1, 0.05), ("bch_127_64", 5, 0.3)])
def test_c_restatement_equals_numpy(name, max_iter, gamma):
    """the C restatement is the numpy one, bit for bit: waterfall noise, quantised ties and the edge frames"""
    R = ref(name)
    rng = np.random.default_rng(5)
    frames = 40 if R.n == 127 else 150
    ebno = {15: 1.0, 31: 2.0, 63: 3.0, 127: 4.0}[R.n]
    _, y1 = noisy_codewords(R.oc, frames, ebno, rng)
    _, y2 = noisy_codewords(R.oc, 20, ebno, rng, quantise=True)
    y = np.concatenate([y1, y2, edge_frames(R.n, rng)])
    want = abp_numpy(R, y, max_iter, gamma)
    same_outputs(abp_c(R, y, max_iter, gamma), want, "C vs numpy")
    assert want[2].max() > min(1, max_iter - 1)


# ---------------------------------------------------------------- the GPU against them

@pytest.fixture(scope="module")
def ctx():
    import channelcoding_b200 as cc
    c = cc.Context(0)
    yield c
    c.close()


def gpu_code(ctx, name):
    q, t = CODES[name]
    return ctx.bch(q, errors=t)


# (code, Eb/N0 of the waterfall, waterfall frames)
PARITY_CODES = {"bch_15_7": (1.0, 4099), "bch_31_16": (2.0, 4099), "bch_31_21": (2.5, 4099), "bch_63_36": (3.0, 2003),
                "bch_63_45": (3.5, 2003), "bch_127_64": (4.0, 501), "bch_127_106": (5.0, 501)}
PARITY = [(name, m) for name in PARITY_CODES for m in (0, 1, 5, 50)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,max_iter", PARITY)
def test_restatement_parity(ctx, name, max_iter):
    """bit-exact bits / L / iter / failed for gamma in {0.05, 0.15, 1.0}: waterfall AWGN on random codewords (a ragged
    count), quantised values (order and minimum ties), the edge frames, a single frame; host buffers and torch CUDA
    tensors"""
    import torch
    R = ref(name)
    code = gpu_code(ctx, name)
    ebno, frames = PARITY_CODES[name]
    rng = np.random.default_rng(100 + max_iter)
    _, y1 = noisy_codewords(R.oc, frames, ebno, rng)
    _, y2 = noisy_codewords(R.oc, 33, ebno, rng, quantise=True)
    y3 = edge_frames(R.n, rng)
    for gamma in (0.05, 0.15, 1.0):
        for what, y in (("waterfall", y1), ("quantised", y2), ("edge", y3), ("one frame", y1[:1])):
            r = abp_c_parallel(R, y, max_iter, gamma)
            same_outputs(code.decode_abp(y, max_iter, gamma), r, "%s gamma=%g host" % (what, gamma))
            got = code.decode_abp(torch.from_numpy(y).cuda(), max_iter, gamma)
            torch.cuda.synchronize()
            same_outputs(got, r, "%s gamma=%g torch" % (what, gamma))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PARITY_CODES))
def test_numpy_restatement_parity(ctx, name):
    """the kernel against the numpy restatement directly, on a smaller sample"""
    R = ref(name)
    code = gpu_code(ctx, name)
    ebno, _ = PARITY_CODES[name]
    rng = np.random.default_rng(7)
    _, y = noisy_codewords(R.oc, 24 if R.n == 127 else 80, ebno, rng)
    y = np.concatenate([y, edge_frames(R.n, rng)])
    for max_iter, gamma in ((50, 0.15), (5, 1.0)):
        same_outputs(code.decode_abp(y, max_iter, gamma), abp_numpy(R, y, max_iter, gamma), "numpy %d %g" % (max_iter, gamma))


@pytest.mark.gpu
@pytest.mark.parametrize("name,ebno,frames,max_iter,gamma", [("bch_31_16", 3.0, 40000, 50, 0.15),
                                                             ("bch_63_36", 3.0, 30001, 20, 0.1),
                                                             ("bch_127_64", 5.0, 10000, 50, 0.15),
                                                             ("bch_63_36", 8.0, 30000, 50, 0.3)])
def test_fused_point(ctx, name, ebno, frames, max_iter, gamma):
    """ccgpu_awgn_point_abp == K1 -> ccgpu_decode_llr_abp -> host count; a device out accumulates; a group of one
    member and a group of every device agree"""
    import channelcoding_b200 as cc
    import torch
    code = gpu_code(ctx, name)
    y = ctx.awgn_llr(code.n, np.float32(cc.sigma(code.rate, ebno)), seed=9, point=4, frame0=77, frames=frames)
    bits, _, it, failed = code.decode_abp(y, max_iter, gamma)
    nz = (bits != 0).sum(axis=1)
    c = code.awgn_point_abp(ebno, frames, max_iter, gamma, seed=9, point=4, frame0=77)
    assert c["frames"] == frames
    assert c["iterations"] == int(it.astype(np.int64).sum())
    assert c["failures"] == int(failed.sum())
    assert c["frame_errors"] == int(((failed != 0) | (nz > 0)).sum())
    assert c["bit_errors"] == int(nz.sum())
    assert c["undetected"] == int(((failed == 0) & (nz > 0)).sum())
    dev = torch.tensor([5, 4, 3, 2, 1, 0, 7, 8], dtype=torch.int64, device="cuda:0")
    code.awgn_point_abp(ebno, frames, max_iter, gamma, seed=9, point=4, frame0=77, out=dev)
    torch.cuda.synchronize()
    keys = ("frames", "frame_errors", "bit_errors", "iterations", "failures", "undetected")
    assert dev.cpu().tolist() == [v + c[k] for v, k in zip((5, 4, 3, 2, 1, 0), keys)] + [7, 8]
    for devices in ([0], list(range(torch.cuda.device_count()))):
        g = cc.Group(devices)
        g.set_min_frames(1000)
        gc = g.bch(CODES[name][0], errors=CODES[name][1])
        assert gc.awgn_point_abp(ebno, frames, max_iter, gamma, seed=9, point=4, frame0=77) == c, devices
        g.close()


@pytest.mark.gpu
def test_gain_over_min_sum(ctx):
    """BCH(63,36) at 4 dB, 2e5 frames of the same noise stream: ABP (50, 0.15) leaves under a tenth of NMS 0.8's frame
    errors on the same H (about a fiftieth expected)"""
    code = gpu_code(ctx, "bch_63_36")
    F = 200000
    abp = code.awgn_point_abp(4.0, F, 50, 0.15, seed=1, point=3)
    nms = code.awgn_point(4.0, F, "NMS", 0.8, seed=1, point=3)
    assert abp["frames"] == nms["frames"] == F
    assert 0 < abp["frame_errors"] * 10 < nms["frame_errors"], (abp, nms)


@pytest.mark.gpu
def test_errors_and_launches(ctx):
    import torch
    from channelcoding_b200 import CcgpuError
    from channelcoding_b200._lib import ERR_INVALID, ERR_UNSUPPORTED
    code = gpu_code(ctx, "bch_63_36")
    y = np.ones((4, 63), np.float32)
    for max_iter, gamma in ((256, 0.15), (50, 0.0), (50, -0.1), (50, 1.01), (50, float("nan")), (50, float("inf"))):
        for call in (lambda: code.decode_abp(y, max_iter, gamma), lambda: code.awgn_point_abp(4.0, 100, max_iter, gamma)):
            with pytest.raises(CcgpuError) as e:
                call()
            assert e.value.code == ERR_INVALID, (max_iter, gamma)
    # RS, dense H, n = 255, k > 64 (BCH(127,57): k = 70)
    for other in (ctx.rs(8, 16), ctx.from_dense(code.H(), code.rate), ctx.bch(8, errors=18), ctx.bch(7, errors=11)):
        with pytest.raises(CcgpuError) as e:
            other.decode_abp(np.ones((4, other.n), np.float32))
        assert e.value.code == ERR_UNSUPPORTED
        with pytest.raises(CcgpuError) as e:
            other.awgn_point_abp(4.0, 100)
        assert e.value.code == ERR_UNSUPPORTED
    bits, L, it, failed = code.decode_abp(np.zeros((0, 63), np.float32))
    assert bits.shape == (0, 63) and it.shape == (0,)
    assert code.awgn_point_abp(4.0, 0)["frames"] == 0
    # a mixed host / device call is refused
    yd = torch.ones((4, 63), dtype=torch.float32, device="cuda:0")
    mixed = (np.empty((4, 63), np.uint8), None, torch.empty(4, dtype=torch.uint8, device="cuda:0"),
             torch.empty(4, dtype=torch.uint8, device="cuda:0"))
    for src in (yd, y):
        with pytest.raises(CcgpuError) as e:
            code.decode_abp(src, out=mixed)
        assert e.value.code == ERR_INVALID
    # set_rows does not change ABP; L may be left out
    _, y5 = noisy_codewords(ref("bch_63_36").oc, 300, 3.0, np.random.default_rng(6))
    r = code.decode_abp(y5)
    code.set_rows(40)
    out = (np.empty((300, 63), np.uint8), None, np.empty(300, np.uint8), np.empty(300, np.uint8))
    bits, _, it, failed = code.decode_abp(y5, out=out)
    assert np.array_equal(bits, r[0]) and np.array_equal(it, r[2]) and np.array_equal(failed, r[3])
    # exactly one launch per device call
    yd = torch.from_numpy(noisy_codewords(ref("bch_63_36").oc, 5000, 3.0, np.random.default_rng(6))[1]).cuda()
    before = ctx.kernel_launches
    code.decode_abp(yd)
    assert ctx.kernel_launches == before + 1
    dev = torch.zeros(8, dtype=torch.int64, device="cuda:0")
    code.awgn_point_abp(4.0, 100000, out=dev)
    assert ctx.kernel_launches == before + 2
    torch.cuda.synchronize()


# ---------------------------------------------------------------- full size, tiled against the C restatement

@pytest.mark.gpu
@pytest.mark.parametrize("path,N", [("device", 4194304), ("host", 1000003)])
def test_full_size_tiled(ctx, path, N):
    """ABP (50, 0.15) on BCH(63,36) at full batch sizes: torch tensors, and host memory through the three-slot
    pipeline; every row against the restatement of the pool frame it holds, outputs prefilled with sentinels"""
    import torch
    import test_gpu_scale as scale
    R = ref("bch_63_36")
    y = scale.pool_y("bch_63_36", 16384, (1.0, 2.0, 3.0, 4.0, 5.0), 17, True)
    assert len(np.unique(y.view(np.uint32), axis=0)) == len(y)
    b, L, it, f = abp_c_parallel(R, y, 50, 0.15)
    pool = scale.Pool(y, {"bits": b, "L": L, "iter": it, "failed": f})
    code = gpu_code(ctx, "bch_63_36")
    src_np = scale.tiling(pool.M, N, 123)
    src = torch.from_numpy(src_np).cuda()
    lib = "numpy" if path == "host" else "torch"
    out = scale.ms_outputs(N, 63, True, lib)
    yy = pool.y[src_np] if lib == "numpy" else scale.to_dev(pool.y)[src]
    code.decode_abp(yy, 50, 0.15, out=out)
    torch.cuda.synchronize()
    scale.check_tiled(scale.ms_got(out), scale.ref_on(pool.ref), src, "ABP " + path)


# ---------------------------------------------------------------- the C++ layer

@pytest.fixture(scope="module")
def bins():
    from channelcoding_b200 import build as _build
    _build.build()
    return {os.path.basename(p): p for p in _build.build_tools()}


def test_cpp_abp_tags(bins):
    r = subprocess.run([bins["abp_test"], "--host"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_cpp_abp_decoder(bins, tmp_path):
    r = subprocess.run([bins["abp_test"], "--gpu", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_cli_abp(bins, tmp_path):
    """benchmark --algorithm abp writes "(63, 45, 7)-ABP50.log" in the reference's format, and only that log"""
    r = subprocess.run([bins["benchmark"], "--algorithm", "abp", "--k", "6", "--dmin", "7", "--max-samples", "100000",
                        "--seed", "3", "--out", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert sorted(p.name for p in tmp_path.glob("*.log")) == ["(63, 45, 7)-ABP50.log"]
    lines = open(tmp_path / "(63, 45, 7)-ABP50.log").read().splitlines()
    assert lines[0] == "   ebno                   wer" and len(lines) >= 5
    wers = [float(x.split()[1]) for x in lines[1:]]
    assert wers[0] > wers[-1]
