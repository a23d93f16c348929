"""GMD soft-decision decoding of Reed-Solomon codes (ccgpu_decode_llr_gmd / ccgpu_awgn_point_gmd, kernel K7).

The CPU restatement below implements the contract of include/ccgpu.h literally: the binary image with bit j of symbol c
at position c*q + j, np.lexsort over (kappa, c) for the symbol ranking, every trial of every frame decoded by the C
restatement of the reference's Euklid decoder with that trial's erasures (oracle.Code.hard_correct, a different route
from the kernel's Berlekamp-Massey), the float32 cumulative sum over the image bits for the metric and the (K(D), i)
minimum.  For mu != 1, which the Euklid restatement does not decode, the trials run on ccgpu_gf_decode_erasures, the
decoder the contract names.  The tests without a gpu mark check the restatement itself; the others pin the GPU against
it bit for bit."""
import os
import subprocess

import numpy as np
import pytest

import oracle

# name -> (q, t, mu) of the RS codes
CODES = {"rs_7_3": (3, 2, 1), "rs_7_5": (3, 1, 1), "rs_15_9": (4, 3, 1), "rs_15_9_mu0": (4, 3, 0), "rs_255_223": (8, 16, 1)}
NAN_KEY = np.uint32(0x7fc00000)


def oracle_code(name):
    q, t, mu = CODES[name]
    return oracle.Code(oracle.FAM_RS, q, t, mu)


def image(words, q):
    """symbols (..., n) -> binary image (..., n*q): bit j of symbol c at position c*q + j"""
    w = np.asarray(words, np.uint8)
    return ((w[..., None] >> np.arange(q, dtype=np.uint8)) & 1).reshape(*w.shape[:-1], -1).astype(np.uint8)


def hard_symbols(y, q):
    """r_c = sum_j (y_{cq+j} < 0) << j"""
    h = (y < 0).astype(np.uint32).reshape(len(y), -1, q)
    return (h << np.arange(q, dtype=np.uint32)).sum(-1).astype(np.uint8)


def key_of(v):
    """K: the bits of fabsf(v) as uint32, every NaN counted as 0x7fc00000"""
    v = np.abs(np.asarray(v, np.float32))
    return np.where(np.isnan(v), NAN_KEY, v.view(np.uint32))


def ranking(y, q):
    """the symbols of every frame in ascending (kappa_c, c), kappa_c = min_j K(y_{cq+j})"""
    kappa = key_of(y).reshape(len(y), -1, q).min(-1)
    cols = np.broadcast_to(np.arange(kappa.shape[1]), kappa.shape)
    return np.lexsort((cols, kappa), axis=-1)


def metric(x_img, h_img, y):
    """D: float32 sum of |y_b| over the image positions where x != h, ascending b, from +0.0"""
    return np.cumsum(np.where(x_img != h_img, np.abs(y), np.float32(0)), axis=-1, dtype=np.float32)[..., -1]


def euklid_trials(oc):
    """the trial decoder of the restatement: the C restatement of the reference's Euklid decoder, word by word.
    r (frames, n), erased (frames, 2i) -> decoded words, success mask"""
    def decode(r, erased):
        if erased.shape[1] == 0:
            out, _, status = oc.hard_correct(r)
            return out, status == 0
        out, ok = np.zeros_like(r), np.zeros(len(r), bool)
        for f in range(len(r)):
            o, _, s = oc.hard_correct(r[f], [int(c) for c in erased[f]])
            out[f], ok[f] = o[0], s[0] == 0
        return out, ok
    return decode


def k4_trials(code):
    """the trial decoder as the contract words it, ccgpu_gf_decode_erasures itself: for codes with mu != 1, which the
    Euklid restatement does not decode (the reference's value solver assumes mu = 1)"""
    def decode(r, erased):
        if erased.shape[1] == 0:
            out, _, failed = code.gf_decode(r)
        else:
            cnt = np.full(len(r), erased.shape[1], np.uint8)
            out, _, failed = code.gf_decode(r, erasures=(np.ascontiguousarray(erased, np.uint8), cnt))
        return out, failed == 0
    return decode


def gmd_restatement(oc, y, F, trials=None):
    """-> words (frames, n) uint8, failed (frames,) uint8, chosen (frames,) uint8, D of the returned word (float32).
    trials: the errors-and-erasures decoder of one trial (default: euklid_trials(oc))"""
    q, n = oc.q, oc.n
    trials = trials or euklid_trials(oc)
    y = np.ascontiguousarray(y, np.float32).reshape(-1, n * q)
    frames, T = len(y), F // 2 + 1
    r = hard_symbols(y, q)
    order = ranking(y, q)
    cand = np.repeat(r[:, None, :], T, axis=1)
    ok = np.zeros((frames, T), bool)
    for i in range(T):
        cand[:, i], ok[:, i] = trials(r, order[:, :2 * i])
    h = image(r, q)
    D = metric(image(cand, q), h[:, None, :], y[:, None, :])
    key = (key_of(D).astype(np.uint64) << np.uint64(8)) | np.arange(T, dtype=np.uint64)
    key = np.where(ok, key, np.uint64(np.iinfo(np.uint64).max))
    best = key.argmin(axis=1)
    failed = ~ok.any(axis=1)
    rows = np.arange(frames)
    words = np.where(failed[:, None], r, cand[rows, best]).astype(np.uint8)
    chosen = np.where(failed, 0, best).astype(np.uint8)
    return words, failed.astype(np.uint8), chosen, metric(image(words, q), h, y)


def noisy_codewords(oc, frames, ebno, rng, quantise=False):
    x = oc.encode(rng.integers(0, 1 << oc.q, size=(frames, oc.l)).astype(np.uint8))
    y = (1.0 - 2.0 * image(x, oc.q) + oracle.sigma(oc.rate, ebno) * rng.standard_normal((frames, oc.n * oc.q)))
    y = y.astype(np.float32)
    if quantise:
        y = (np.round(y * 4) / 4).astype(np.float32)
    return x, y


def special_values(frames, nq, rng):
    """frames whose entries include +-0, +-inf and NaN"""
    y = (1.0 + 0.5 * rng.standard_normal((frames, nq))).astype(np.float32)
    vals = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan], np.float32)
    mask = rng.random((frames, nq)) < 0.03
    y[mask] = vals[rng.integers(0, len(vals), mask.sum())]
    return y


def bpsk(x, q, mag):
    return ((1.0 - 2.0 * image(x, q)) * mag).astype(np.float32)


# ---------------------------------------------------------------- the restatement (CPU)

@pytest.mark.parametrize("name", ["rs_7_3", "rs_15_9", "rs_255_223"])
def test_restatement_F0_is_hard_decoding(name):
    oc = oracle_code(name)
    _, y = noisy_codewords(oc, 300, 5.0, np.random.default_rng(1))
    words, failed, chosen, _ = gmd_restatement(oc, y, 0)
    r = hard_symbols(y, oc.q)
    out, _, status = oc.hard_correct(r)
    assert np.array_equal(failed, (status != 0).astype(np.uint8)) and not chosen.any()
    assert np.array_equal(words, np.where((status != 0)[:, None], r, out))
    assert 0 < failed.sum() < len(y)


@pytest.mark.parametrize("name", ["rs_7_3", "rs_15_9", "rs_255_223"])
def test_restatement_within_t_symbol_errors(name):
    """at most t symbol errors whose flipped bits are weak: the sent word is the candidate closest to y at every F
    (any other codeword differs from r in at least t + 1 symbols holding a strong bit)"""
    oc = oracle_code(name)
    q, t, n = oc.q, oc.t, oc.n
    rng = np.random.default_rng(2)
    frames = 60 if n == 255 else 200
    x = oc.encode(rng.integers(0, 1 << q, size=(frames, oc.l)).astype(np.uint8))
    mag = rng.uniform(0.6, 1.5, size=(frames, n * q)).astype(np.float32)
    sign = np.ones((frames, n * q), np.float32)
    for f in range(frames):
        for c in rng.choice(n, rng.integers(0, t + 1), replace=False):
            e = int(rng.integers(1, 1 << q))
            for j in range(q):
                if (e >> j) & 1:
                    sign[f, c * q + j] = -1.0
                    mag[f, c * q + j] = rng.uniform(0.01, 0.5 / q)
    y = bpsk(x, q, mag) * sign
    for F in range(0, 2 * t + 1, 2 if n < 255 else 16):
        words, failed, _, _ = gmd_restatement(oc, y, F)
        assert not failed.any() and np.array_equal(words, x), F


@pytest.mark.parametrize("name", ["rs_7_3", "rs_15_9", "rs_255_223"])
def test_restatement_recovers_2t_erasures(name):
    """2t wrong symbols that are the least reliable, no other error: the pure erasure trial F = 2t recovers the word
    and nothing closer to y exists"""
    oc = oracle_code(name)
    q, t, n = oc.q, oc.t, oc.n
    rng = np.random.default_rng(3)
    frames = 40 if n == 255 else 200
    x = oc.encode(rng.integers(0, 1 << q, size=(frames, oc.l)).astype(np.uint8))
    mag = rng.uniform(0.6, 1.5, size=(frames, n * q)).astype(np.float32)
    sent = x.copy()
    for f in range(frames):
        weak = rng.choice(n, 2 * t, replace=False)
        x[f, weak] ^= rng.integers(1, 1 << q, size=2 * t).astype(np.uint8)  # 2t symbol errors
        for c in weak:
            mag[f, c * q:(c + 1) * q] = rng.uniform(1e-4, 0.5 / (2 * t * q), size=q)
    y = bpsk(x, q, mag)
    words, failed, chosen, _ = gmd_restatement(oc, y, 2 * t)
    assert not failed.any() and np.array_equal(words, sent)
    assert (chosen == t).all()  # no earlier trial is within reach of the sent word


@pytest.mark.parametrize("name", ["rs_7_5", "rs_15_9", "rs_255_223"])
def test_restatement_codeword_inputs(name):
    oc = oracle_code(name)
    rng = np.random.default_rng(4)
    x = oc.encode(rng.integers(0, 1 << oc.q, size=(50, oc.l)).astype(np.uint8))
    y = bpsk(x, oc.q, rng.uniform(0.1, 2.0, size=(50, oc.n * oc.q)))
    words, failed, chosen, D = gmd_restatement(oc, y, 2 * oc.t)
    assert np.array_equal(words, x) and not failed.any() and not chosen.any() and not D.view(np.uint32).any()


def test_restatement_keys_and_image():
    assert image(np.array([[0b101, 0b010]], np.uint8), 3).tolist() == [[1, 0, 1, 0, 1, 0]]
    y = np.array([[-0.5, 0.25, -0.0, np.nan, np.inf, -1.0]], np.float32)
    assert hard_symbols(y, 3).tolist() == [[0b001, 0b100]]            # -0.0 and NaN decide 0
    assert ranking(y, 3).tolist() == [[0, 1]]
    y = np.array([[1.0, -2.0, np.nan, 3.0, 0.5, 0.5]], np.float32)
    assert ranking(y, 2).tolist() == [[2, 0, 1]]                      # kappa: 1.0, NaN, 0.5 (ties by column)
    assert key_of(np.float32(-np.nan)) == NAN_KEY and key_of(np.float32(-0.0)) == 0


# ---------------------------------------------------------------- the GPU against it

@pytest.fixture(scope="module")
def ctx():
    import channelcoding_b200 as cc
    c = cc.Context(0)
    yield c
    c.close()


def gpu_code(ctx, name):
    q, t, mu = CODES[name]
    return ctx.rs(q, t, mu=mu)


def assert_same(got, ref, what):
    words, failed, chosen = (np.asarray(a.cpu()) if hasattr(a, "cpu") else a for a in got)
    rw, rf, rc = ref[:3]
    assert np.array_equal(failed, rf), (what, "failed", int((failed != rf).sum()))
    assert np.array_equal(chosen, rc), (what, "chosen", int((chosen != rc).sum()))
    assert np.array_equal(words, rw), (what, "words", int((words != rw).any(axis=1).sum()))


PARITY = ([("rs_7_3", F, 1500, 3.0) for F in (0, 2, 4)] + [("rs_7_5", F, 1500, 4.0) for F in (0, 2)] +
          [("rs_15_9", F, 1500, 4.0) for F in (0, 2, 4, 6)] + [("rs_15_9_mu0", F, 1000, 4.0) for F in (0, 2, 4, 6)] +
          [("rs_255_223", F, 200, 5.5) for F in (0, 2, 16, 32)])


@pytest.mark.gpu
@pytest.mark.parametrize("name,F,frames,ebno", PARITY)
def test_restatement_parity(ctx, name, F, frames, ebno):
    """bit-exact words / failed / chosen: waterfall noise (ragged count), quantised values (ties in kappa and D),
    special values; host buffers, torch CUDA tensors and torch CPU tensors"""
    import torch
    code = gpu_code(ctx, name)
    oc = oracle_code(name)
    rng = np.random.default_rng(5 + F)
    _, y1 = noisy_codewords(oc, frames - 1, ebno, rng)
    _, y2 = noisy_codewords(oc, frames, ebno, rng, quantise=True)
    y3 = special_values(max(frames // 4, 33), oc.n * oc.q, rng)
    trials = k4_trials(code) if CODES[name][2] != 1 else None
    for what, y in (("waterfall", y1), ("quantised", y2), ("special", y3)):
        ref = gmd_restatement(oc, y, F, trials)
        assert_same(code.decode_gmd(y, F), ref, what + " host")
        got = code.decode_gmd(torch.from_numpy(y).cuda(), F)
        torch.cuda.synchronize()
        assert_same(got, ref, what + " torch")
        assert_same(code.decode_gmd(torch.from_numpy(y), F), ref, what + " torch cpu")
    if name == "rs_255_223" and F == 32:
        ref = gmd_restatement(oc, y1, F)
        assert (ref[2] == 16).any()  # the pure 32-erasure trial wins somewhere


@pytest.mark.gpu
def test_F0_is_gf_decode(ctx):
    code = gpu_code(ctx, "rs_255_223")
    oc = oracle_code("rs_255_223")
    _, y = noisy_codewords(oc, 3000, 5.0, np.random.default_rng(6))
    words, failed, chosen = code.decode_gmd(y, 0)
    out, _, fl = code.gf_decode(hard_symbols(y, oc.q))
    assert np.array_equal(failed, fl) and np.array_equal(words, out) and not chosen.any()


def host_count(words, failed, q):
    nz = (words != 0).sum(axis=1)
    bits = np.unpackbits(words, axis=1).sum(axis=1)
    return {"failures": int(failed.sum()), "bit_errors": int(bits.sum()),
            "frame_errors": int(((failed == 1) | (nz > 0)).sum()), "undetected": int(((failed == 0) & (nz > 0)).sum())}


@pytest.mark.gpu
@pytest.mark.parametrize("name,F,ebno,frames", [("rs_7_3", 4, 3.0, 40000), ("rs_15_9", 6, 5.0, 40000),
                                                ("rs_15_9_mu0", 2, 4.0, 40000), ("rs_255_223", 32, 5.5, 20000),
                                                ("rs_255_223", 0, 6.0, 20000)])
def test_fused_point(ctx, name, F, ebno, frames):
    """ccgpu_awgn_point_gmd == awgn_llr(n q) -> ccgpu_decode_llr_gmd -> host count; halves add up; a device group of one
    member and one of several agree"""
    import channelcoding_b200 as cc
    import torch
    code = gpu_code(ctx, name)
    nq = code.n * code.q
    y = ctx.awgn_llr(nq, np.float32(cc.sigma(code.rate, ebno)), seed=9, point=4, frame0=77, frames=frames)
    words, failed, _ = code.decode_gmd(y, F)
    c = code.awgn_point_gmd(ebno, frames, F, seed=9, point=4, frame0=77)
    assert c["frames"] == frames and c["iterations"] == 0
    for k, v in host_count(words, failed, code.q).items():
        assert c[k] == v, (k, c[k], v)
    assert c["frame_errors"] > 0
    halves = [code.awgn_point_gmd(ebno, frames // 2, F, seed=9, point=4, frame0=77 + i * (frames // 2)) for i in range(2)]
    assert all(halves[0][k] + halves[1][k] == c[k] for k in c)
    dev = torch.zeros(8, dtype=torch.int64, device="cuda:0")
    code.awgn_point_gmd(ebno, frames, F, seed=9, point=4, frame0=77, out=dev)
    torch.cuda.synchronize()
    assert dev.cpu().tolist()[:6] == [c[k] for k in ("frames", "frame_errors", "bit_errors", "iterations", "failures",
                                                         "undetected")]
    q, t, mu = CODES[name]
    members = list(range(torch.cuda.device_count())) if torch.cuda.device_count() >= 2 else [0, 0, 0]
    for devices in ([0], members):
        g = cc.Group(devices)
        g.set_min_frames(1000)
        gc = g.rs(q, t, mu=mu)
        assert gc.awgn_point_gmd(ebno, frames, F, seed=9, point=4, frame0=77) == c, devices
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,ebno,frames", [("rs_15_9", 5.0, 400000), ("rs_255_223", 5.5, 200000)])
def test_closed_form_hard_wer(ctx, name, ebno, frames):
    """F = 0 is a bounded-distance decoder: a frame is in error exactly when more than t symbols of its hard decision
    are wrong, P = P(Binomial(n, p_s) > t) with p_s = 1 - (1 - Q(1/sigma))^q.  The frame-error count lies inside the
    99.9 % binomial interval around it -- an independent check of the channel and the bit <-> symbol mapping."""
    import channelcoding_b200 as cc
    from scipy import special, stats
    code = gpu_code(ctx, name)
    q, t, _ = CODES[name]
    sigma = float(np.float32(cc.sigma(code.rate, ebno)))
    pb = 0.5 * special.erfc(1.0 / (sigma * np.sqrt(2.0)))
    ps = 1.0 - (1.0 - pb) ** q
    P = stats.binom.sf(t, code.n, ps)
    c = code.awgn_point_gmd(ebno, frames, 0, seed=11, point=1)
    lo, hi = stats.binom.interval(0.999, frames, P)
    assert lo <= c["frame_errors"] <= hi, (c["frame_errors"], frames * P, lo, hi)
    assert c["failures"] + c["undetected"] == c["frame_errors"]


@pytest.mark.gpu
def test_gmd_beats_hard_decoding(ctx):
    """RS(15,9) at 5 dB and RS(255,223) at 6 dB, the same noise stream: F = 2t leaves fewer frame errors than F = 0"""
    for name, ebno, frames in (("rs_15_9", 5.0, 200000), ("rs_255_223", 6.0, 200000)):
        code = gpu_code(ctx, name)
        g = code.awgn_point_gmd(ebno, frames, 2 * CODES[name][1], seed=1, point=0)
        h = code.awgn_point_gmd(ebno, frames, 0, seed=1, point=0)
        assert g["frames"] == h["frames"] == frames
        assert 0 < g["frame_errors"] < h["frame_errors"], (name, g, h)


@pytest.mark.gpu
def test_errors_and_launches(ctx):
    import torch
    from channelcoding_b200 import CcgpuError
    from channelcoding_b200._lib import ERR_INVALID, ERR_UNSUPPORTED, lib
    code = gpu_code(ctx, "rs_15_9")
    y = np.ones((4, 60), np.float32)
    for F in (1, 5, 8):
        for call in (lambda: code.decode_gmd(y, F), lambda: code.awgn_point_gmd(4.0, 100, F)):
            with pytest.raises(CcgpuError) as e:
                call()
            assert e.value.code == ERR_INVALID
    # binary BCH, dense H, 2t > 32 (a dense code has no symbol size, so its batch goes through the C ABI)
    L = lib()
    bch = ctx.bch(6, errors=5)
    yb = np.ones((4, 255 * 8), np.float32)
    wb = np.empty((4, 255), np.uint8)
    f = np.empty(4, np.uint8)
    for other in (bch, ctx.from_dense(bch.H(), bch.rate), ctx.rs(8, 17)):
        rc = L.ccgpu_decode_llr_gmd(ctx._h, other._h, 0, yb.ctypes.data, 4, wb.ctypes.data, f.ctypes.data, None)
        assert rc == ERR_UNSUPPORTED
        with pytest.raises(CcgpuError) as e:
            other.awgn_point_gmd(4.0, 100, 0)
        assert e.value.code == ERR_UNSUPPORTED
    with pytest.raises(CcgpuError) as e:
        bch.decode_gmd(np.ones((4, 63 * 6), np.float32), 0)
    assert e.value.code == ERR_UNSUPPORTED
    # ccgpu_awgn_point_hard still refuses RS codes
    with pytest.raises(CcgpuError) as e:
        code.awgn_point_hard(4.0, 100)
    assert e.value.code == ERR_UNSUPPORTED
    # null pointers
    w = np.empty((4, 15), np.uint8)
    assert L.ccgpu_decode_llr_gmd(ctx._h, code._h, 2, None, 4, w.ctypes.data, f.ctypes.data, None) == ERR_INVALID
    assert L.ccgpu_decode_llr_gmd(ctx._h, code._h, 2, y.ctypes.data, 4, None, f.ctypes.data, None) == ERR_INVALID
    assert L.ccgpu_decode_llr_gmd(ctx._h, code._h, 2, y.ctypes.data, 4, w.ctypes.data, None, None) == ERR_INVALID
    assert L.ccgpu_decode_llr_gmd(ctx._h, None, 2, y.ctypes.data, 4, w.ctypes.data, f.ctypes.data, None) == ERR_INVALID
    assert L.ccgpu_awgn_point_gmd(ctx._h, code._h, 2, 4.0, 0, 0, 0, 100, None) == ERR_INVALID
    # chosen is optional; empty batches
    L.ccgpu_decode_llr_gmd(ctx._h, code._h, 2, y.ctypes.data, 4, w.ctypes.data, f.ctypes.data, None)
    assert not w.any() and not f.any()
    words, failed, chosen = code.decode_gmd(np.zeros((0, 60), np.float32), 6)
    assert words.shape == (0, 15) and failed.shape == (0,) and chosen.shape == (0,)
    assert code.awgn_point_gmd(4.0, 0, 6)["frames"] == 0
    # mixed host and device buffers
    yd = torch.ones((4, 60), dtype=torch.float32, device="cuda:0")
    dev8 = lambda: torch.empty(4, dtype=torch.uint8, device="cuda:0")  # noqa: E731
    for args in ((yd, (np.empty((4, 15), np.uint8), dev8(), dev8())), (yd, (torch.empty((4, 15), dtype=torch.uint8,
                 device="cuda:0"), dev8(), np.empty(4, np.uint8))), (y, (np.empty((4, 15), np.uint8), dev8(),
                 np.empty(4, np.uint8)))):
        with pytest.raises(CcgpuError) as e:
            code.decode_gmd(args[0], 2, out=args[1])
        assert e.value.code == ERR_INVALID
    # exactly one launch per device call
    big = gpu_code(ctx, "rs_255_223")
    yd = torch.from_numpy(noisy_codewords(oracle_code("rs_255_223"), 2000, 5.5, np.random.default_rng(7))[1]).cuda()
    out = (torch.empty((2000, 255), dtype=torch.uint8, device="cuda:0"), dev8().new_empty(2000), dev8().new_empty(2000))
    before = ctx.kernel_launches
    big.decode_gmd(yd, 32, out=out)
    assert ctx.kernel_launches == before + 1
    dev = torch.zeros(8, dtype=torch.int64, device="cuda:0")
    big.awgn_point_gmd(5.5, 100000, 32, out=dev)
    assert ctx.kernel_launches == before + 2
    torch.cuda.synchronize()


# ---------------------------------------------------------------- full size, tiled against the restatement

@pytest.mark.gpu
@pytest.mark.parametrize("name,F,path,N", [("rs_15_9", 6, "device", 4194304), ("rs_15_9", 6, "host", 1000003),
                                           ("rs_255_223", 32, "device", 1048576)])
def test_full_size_tiled(ctx, name, F, path, N):
    """full batch sizes: torch tensors, and host memory through the three-slot pipeline; every row against the
    restatement of the pool frame it holds, outputs prefilled with sentinels"""
    import torch
    import test_gpu_scale as scale
    scale.SENTINEL.setdefault("words", scale.SENT8)
    oc = oracle_code(name)
    rng = np.random.default_rng(8)
    M = 4096 if oc.n < 255 else 1024
    ebnos = (3.0, 4.0, 5.0, 6.0) if oc.n < 255 else (5.0, 5.5, 6.0)
    parts = [noisy_codewords(oc, M // len(ebnos), e, rng)[1] for e in ebnos]
    parts.append(noisy_codewords(oc, M // 8, ebnos[1], rng, quantise=True)[1])
    parts.append(special_values(M // 8, oc.n * oc.q, rng))
    y = np.concatenate(parts)
    w, f, c, _ = scale.oracle_map(lambda rows: gmd_restatement(oracle_code(name), rows, F), y, chunk=64)
    pool = scale.Pool(y, {"words": w, "failed": f, "chosen": c})
    code = gpu_code(ctx, name)
    src_np = scale.tiling(pool.M, N, 123)
    src = torch.from_numpy(src_np).cuda()
    lib = "numpy" if path == "host" else "torch"
    u8 = np.uint8 if lib == "numpy" else torch.uint8
    out = (scale.sentinel_like((N, oc.n), u8, "words", lib), scale.sentinel_like(N, u8, "failed", lib),
           scale.sentinel_like(N, u8, "chosen", lib))
    yy = pool.y[src_np] if lib == "numpy" else scale.to_dev(pool.y)[src]
    code.decode_gmd(yy, F, out=out)
    torch.cuda.synchronize()
    got = {k: scale.to_dev(v) for k, v in zip(("words", "failed", "chosen"), out)}
    scale.check_tiled(got, scale.ref_on(pool.ref), src, "GMD %s F=%d %s" % (name, F, path))


# ---------------------------------------------------------------- the C++ layer and the sweep

@pytest.fixture(scope="module")
def bins():
    from channelcoding_b200 import build as _build
    _build.build()
    return {os.path.basename(p): p for p in _build.build_tools()}


def test_cpp_gmd_tags(bins):
    r = subprocess.run([bins["gmd_test"], "--host"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_cpp_gmd_decoder(bins, tmp_path):
    r = subprocess.run([bins["gmd_test"], "--gpu", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.gpu
def test_sweep_gmd():
    """tools/sweep.py --gmd: RS(15,9), tag GMD6, bit errors over the n q image bits; --gmd excludes --chase / --osd"""
    import json
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "tools", "sweep.py"), "--q", "4", "--t", "3", "--gmd", "6", "--ebno-from",
           "4", "--ebno-to", "5", "--ebno-step", "1", "--batch", "100000", "--min-errors", "10", "--max-frames", "1e6"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [json.loads(s) for s in r.stdout.splitlines()]
    assert [d["ebno_db"] for d in lines] == [4.0, 5.0]
    assert all(d["code"].startswith("(15, 9,") and d["code"].endswith("-GMD6") for d in lines)
    assert all(d["ber"] == d["bit_errors"] / d["frames"] / 60 for d in lines)
    assert lines[0]["wer"] > lines[1]["wer"] > 0
    r = subprocess.run(cmd + ["--chase", "2"], capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "not allowed with" in r.stderr
