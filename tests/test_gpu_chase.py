"""Chase-II soft-decision decoding of binary BCH codes (ccgpu_decode_llr_chase / ccgpu_awgn_point_chase, kernel K5).

The CPU restatement below implements the contract of include/ccgpu.h literally: np.lexsort for the reliability order,
every test word of every frame decoded in one batch of the C restatement of the bounded-distance decoder
(oracle.Code.hard_correct), the float32 cumulative sum for the metric and the (bits of D, m) minimum.  The tests
without a gpu mark check the restatement itself; the others pin the GPU against it bit for bit."""
import os
import subprocess

import numpy as np
import pytest

import oracle

CODES = {"bch_15_7": (4, 2), "bch_31_16": (5, 3), "bch_63_36": (6, 5), "bch_127_64": (7, 10), "bch_255_131": (8, 18)}


def least_reliable(y, p):
    """u_0 .. u_{p-1} per frame: the p smallest (bits of |y_c| as uint32, c)"""
    key = np.abs(y).view(np.uint32)
    cols = np.broadcast_to(np.arange(y.shape[1]), y.shape)
    return np.lexsort((cols, key), axis=-1)[:, :p]


def metric(x, h, y):
    """D: float32 sum of |y_c| over the columns where x != h, ascending c, from +0.0"""
    return np.cumsum(np.where(x != h, np.abs(y), np.float32(0)), axis=-1, dtype=np.float32)[..., -1]


def chase_restatement(oc, y, p):
    """-> bits (frames, n) uint8, failed (frames,) uint8, chosen (frames,) uint8, D of the returned word (float32)"""
    y = np.ascontiguousarray(y, np.float32)
    frames, n = y.shape
    h = (y < 0).astype(np.uint8)
    u = least_reliable(y, p)
    M = 1 << p
    tw = np.repeat(h[:, None, :], M, axis=1)
    rows = np.arange(frames)
    for m in range(M):
        for j in range(p):
            if (m >> j) & 1:
                tw[rows, m, u[:, j]] ^= 1
    out, _, status = oc.hard_correct(tw.reshape(-1, n))
    out = out.reshape(frames, M, n)
    ok = status.reshape(frames, M) == 0
    D = metric(out, h[:, None, :], y[:, None, :])
    key = (D.view(np.uint32).astype(np.uint64) << np.uint64(8)) | np.arange(M, dtype=np.uint64)
    key = np.where(ok, key, np.uint64(np.iinfo(np.uint64).max))
    best = key.argmin(axis=1)
    failed = ~ok.any(axis=1)
    bits = np.where(failed[:, None], h, out[rows, best])
    chosen = np.where(failed, 0, best).astype(np.uint8)
    return bits.astype(np.uint8), failed.astype(np.uint8), chosen, metric(bits, h, y)


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


# ---------------------------------------------------------------- the restatement (CPU)

def test_restatement_p0_is_hard_decoding():
    rng = np.random.default_rng(1)
    for name in ("bch_31_16", "bch_63_36"):
        oc = oracle.Code(0, *CODES[name])
        _, y = noisy_codewords(oc, 500, 3.0, rng)
        bits, failed, chosen, _ = chase_restatement(oc, y, 0)
        h = (y < 0).astype(np.uint8)
        out, _, status = oc.hard_correct(h)
        assert np.array_equal(failed, (status != 0).astype(np.uint8)) and not chosen.any()
        assert np.array_equal(bits, np.where((status != 0)[:, None], h, out))


@pytest.mark.parametrize("name", ["bch_31_16", "bch_63_36", "bch_127_64"])
def test_restatement_chase_guarantee(name):
    """at most t errors outside the p least reliable positions: the sent codeword is a candidate, so the frame decodes
    and the returned word is at least as close to y as the codeword sent"""
    q, t = CODES[name]
    oc = oracle.Code(0, q, t)
    rng = np.random.default_rng(2)
    frames, p, n = 300, 4, oc.n
    x = oc.encode(rng.integers(0, 2, size=(frames, oc.l)).astype(np.uint8))
    mag = rng.uniform(0.6, 1.5, size=(frames, n)).astype(np.float32)
    sign = np.ones((frames, n), np.float32)
    for f in range(frames):
        cols = rng.permutation(n)
        weak = cols[:p]                              # the p least reliable columns, any sign
        mag[f, weak] = rng.uniform(0.0, 0.5, p)
        sign[f, weak] = rng.choice([-1.0, 1.0], p)
        wrong = cols[p:p + rng.integers(0, t + 1)]   # at most t errors among the reliable ones
        sign[f, wrong] = -1.0
    y = ((1.0 - 2.0 * x) * sign * mag).astype(np.float32)
    bits, failed, _, D = chase_restatement(oc, y, p)
    assert not failed.any()
    D_sent = metric(x, (y < 0).astype(np.uint8), y)
    assert (D.view(np.uint32) <= D_sent.view(np.uint32)).all()
    assert (bits != x).any(axis=1).sum() < frames  # and mostly it is the codeword sent


def test_restatement_order_ties_and_special_values():
    y = np.full((1, 15), -0.5, np.float32)
    assert least_reliable(y, 4).tolist() == [[0, 1, 2, 3]]          # all |y| equal: lower columns first
    y = np.array([[1.0, -0.0, 0.0, np.inf, np.nan, -np.inf, 0.25, -0.25]], np.float32)
    assert least_reliable(y, 8).tolist() == [[1, 2, 6, 7, 0, 3, 5, 4]]  # +-0 tie by column, NaN above +-inf
    h = (y < 0).astype(np.uint8)
    assert h.tolist() == [[0, 0, 0, 0, 0, 1, 0, 1]]                   # -0.0 and NaN decide 0
    # the metric: +0.0 for an empty or all-zero difference, inf and NaN totals order above every finite one
    assert metric(h, h, y)[0].view(np.uint32) == 0
    z = h.copy()
    z[0, 1] ^= 1
    assert metric(z, h, y)[0].view(np.uint32) == 0                     # |-0.0| = +0.0
    z[0, 3] ^= 1
    assert np.isinf(metric(z, h, y)[0])
    z[0, 4] ^= 1
    d = metric(z, h, y)[0]
    assert np.isnan(d) and d.view(np.uint32) > np.float32(np.inf).view(np.uint32)


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


def assert_same(got, ref, what):
    bits, failed, chosen = (np.asarray(a.cpu()) if hasattr(a, "cpu") else a for a in got)
    rb, rf, rc = ref[:3]
    assert np.array_equal(failed, rf), (what, "failed", int((failed != rf).sum()))
    assert np.array_equal(chosen, rc), (what, "chosen", int((chosen != rc).sum()))
    assert np.array_equal(bits, rb), (what, "bits", int((bits != rb).any(axis=1).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bch_15_7", "bch_31_16", "bch_63_36", "bch_127_64", "bch_255_131"])
def test_p0_is_the_hard_path(ctx, name):
    code = gpu_code(ctx, name)
    oc = oracle.Code(0, *CODES[name])
    rng = np.random.default_rng(3)
    _, y = noisy_codewords(oc, 3000, 4.0, rng)
    y[:100] = special_values(100, oc.n, rng)
    bits, failed, chosen = code.decode_chase(y, 0)
    out, _, fl = code.gf_decode((y < 0).astype(np.uint8))
    assert np.array_equal(failed, fl) and np.array_equal(bits, out) and not chosen.any()


PARITY = [("bch_31_16", p, 2000, 2.5) for p in range(1, 6)] + [("bch_63_36", 4, 1000, 3.5), ("bch_63_36", 8, 1000, 3.5),
                                                                 ("bch_127_64", 6, 300, 3.0), ("bch_255_131", 8, 100, 3.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,p,frames,ebno", PARITY)
def test_restatement_parity(ctx, name, p, frames, ebno):
    """bit-exact bits / failed / chosen: waterfall noise (ragged count), quantised values (reliability and metric ties),
    special values; host buffers and torch CUDA tensors"""
    import torch
    code = gpu_code(ctx, name)
    oc = oracle.Code(0, *CODES[name])
    rng = np.random.default_rng(4 + p)
    _, y1 = noisy_codewords(oc, frames - 1, ebno, rng)
    _, y2 = noisy_codewords(oc, frames, ebno, rng, quantise=True)
    y3 = special_values(max(frames // 4, 32), oc.n, rng)
    for what, y in (("waterfall", y1), ("quantised", y2), ("special", y3)):
        ref = chase_restatement(oc, y, p)
        assert_same(code.decode_chase(y, p), ref, what + " host")
        got = code.decode_chase(torch.from_numpy(y).cuda(), p)
        torch.cuda.synchronize()
        assert_same(got, ref, what + " torch")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bch_63_36", "bch_127_64"])
def test_framewise_implication(ctx, name):
    """failed_chase => failed_hard, and where hard decoding succeeded the Chase word is at least as close to y"""
    code = gpu_code(ctx, name)
    oc = oracle.Code(0, *CODES[name])
    _, y = noisy_codewords(oc, 20000, 3.0, np.random.default_rng(5))
    bits, failed, _ = code.decode_chase(y, 5)
    h = (y < 0).astype(np.uint8)
    out, _, fl = code.gf_decode(h)
    assert not (failed.astype(bool) & ~fl.astype(bool)).any()
    ok = fl == 0
    assert (metric(bits[ok], h[ok], y[ok]).view(np.uint32) <= metric(out[ok], h[ok], y[ok]).view(np.uint32)).all()
    assert failed.sum() < fl.sum()


@pytest.mark.gpu
@pytest.mark.parametrize("name,ebno,frames", [("bch_31_16", 3.0, 40000), ("bch_63_36", 4.0, 30000),
                                              ("bch_127_64", 5.0, 10000), ("bch_255_131", 6.0, 3000),
                                              ("bch_63_36", 8.0, 30000)])
def test_fused_point(ctx, name, ebno, frames):
    """ccgpu_awgn_point_chase == K1 -> ccgpu_decode_llr_chase -> host count; halves add up; a device group agrees"""
    import channelcoding_b200 as cc
    import torch
    code = gpu_code(ctx, name)
    p = 4
    y = ctx.awgn_llr(code.n, np.float32(cc.sigma(code.rate, ebno)), seed=9, point=4, frame0=77, frames=frames)
    bits, failed, _ = code.decode_chase(y, p)
    nz = (bits != 0).sum(axis=1)
    c = code.awgn_point_chase(ebno, frames, p, seed=9, point=4, frame0=77)
    assert c["frames"] == frames and c["iterations"] == 0
    assert c["failures"] == int(failed.sum())
    assert c["bit_errors"] == int(nz.sum())
    assert c["frame_errors"] == int(((failed == 1) | (nz > 0)).sum())
    assert c["undetected"] == int(((failed == 0) & (nz > 0)).sum())
    halves = [code.awgn_point_chase(ebno, frames // 2, p, seed=9, point=4, frame0=77 + i * (frames // 2)) for i in range(2)]
    assert all(halves[0][k] + halves[1][k] == c[k] for k in c)
    dev = torch.zeros(8, dtype=torch.int64, device="cuda:0")
    code.awgn_point_chase(ebno, frames, p, seed=9, point=4, frame0=77, out=dev)
    torch.cuda.synchronize()
    assert dev.cpu().tolist()[:6] == [c[k] for k in ("frames", "frame_errors", "bit_errors", "iterations", "failures",
                                                         "undetected")]
    g = cc.Group(list(range(torch.cuda.device_count())))
    g.set_min_frames(1000)
    gc = g.bch(CODES[name][0], errors=CODES[name][1])
    assert gc.awgn_point_chase(ebno, frames, p, seed=9, point=4, frame0=77) == c
    g.close()


@pytest.mark.gpu
def test_statistics_against_hard_decoding(ctx):
    """BCH(63,36) at 5 dB, 1e5 frames of the same noise stream: Chase-II with p = 5 leaves fewer than half the frame
    errors of the hard-decision decoder.  Measured on a B200 (seed 1, point 0): 8 Chase frame errors against 949 hard
    ones; the factor of one half leaves a wide margin."""
    code = gpu_code(ctx, "bch_63_36")
    c = code.awgn_point_chase(5.0, 100000, 5, seed=1, point=0)
    h = code.awgn_point_hard(5.0, 100000, seed=1, point=0)
    assert c["frames"] == h["frames"] == 100000
    assert c["failures"] <= h["failures"]
    assert 0 < c["frame_errors"] < 0.5 * h["frame_errors"], (c, h)


@pytest.mark.gpu
def test_errors(ctx):
    import torch
    from channelcoding_b200 import CcgpuError
    from channelcoding_b200._lib import ERR_INVALID, ERR_UNSUPPORTED
    code = gpu_code(ctx, "bch_63_36")
    y = np.ones((4, 63), np.float32)
    with pytest.raises(CcgpuError) as e:
        code.decode_chase(y, 9)
    assert e.value.code == ERR_INVALID
    with pytest.raises(CcgpuError) as e:
        code.awgn_point_chase(4.0, 100, 9)
    assert e.value.code == ERR_INVALID
    for other in (ctx.rs(8, 16), ctx.from_dense(code.H(), code.rate)):
        with pytest.raises(CcgpuError) as e:
            other.decode_chase(np.ones((4, other.n), np.float32), 2)
        assert e.value.code == ERR_UNSUPPORTED
        with pytest.raises(CcgpuError) as e:
            other.awgn_point_chase(4.0, 100, 2)
        assert e.value.code == ERR_UNSUPPORTED
    bits, failed, chosen = code.decode_chase(np.zeros((0, 63), np.float32), 3)
    assert bits.shape == (0, 63) and failed.shape == (0,) and chosen.shape == (0,)
    assert code.awgn_point_chase(4.0, 0, 3)["frames"] == 0
    yd = torch.ones((4, 63), dtype=torch.float32, device="cuda:0")
    out = (np.empty((4, 63), np.uint8), torch.empty(4, dtype=torch.uint8, device="cuda:0"),
           torch.empty(4, dtype=torch.uint8, device="cuda:0"))
    with pytest.raises(CcgpuError) as e:
        code.decode_chase(yd, 3, out=out)
    assert e.value.code == ERR_INVALID


# ---------------------------------------------------------------- the C++ layer

@pytest.fixture(scope="module")
def bins():
    from channelcoding_b200 import build as _build
    _build.build()
    return {os.path.basename(p): p for p in _build.build_tools()}


def test_cpp_chase_tags(bins):
    r = subprocess.run([bins["chase_test"], "--host"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_cpp_chase_decoder(bins, tmp_path):
    r = subprocess.run([bins["chase_test"], "--gpu", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_cli_chase(bins, tmp_path):
    """benchmark --algorithm chase4 writes "(63, 45, 7)-CHASE4.log" in the reference's format, and only that log"""
    r = subprocess.run([bins["benchmark"], "--algorithm", "chase4", "--k", "6", "--dmin", "7", "--max-samples", "100000",
                        "--seed", "3", "--out", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert sorted(p.name for p in tmp_path.glob("*.log")) == ["(63, 45, 7)-CHASE4.log"]
    lines = open(tmp_path / "(63, 45, 7)-CHASE4.log").read().splitlines()
    assert lines[0] == "   ebno                   wer" and len(lines) >= 10
    wers = [float(x.split()[1]) for x in lines[1:]]
    assert wers[0] > wers[-1]
