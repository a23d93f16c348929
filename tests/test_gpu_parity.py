"""GPU parity tests (run on the B200 box: pytest -m gpu).  Every call goes through the C ABI
(include/ccgpu.h via channelcoding_b200.engine); the checker is the oracle (oracle/*.c, pinned
against the reference) and the committed golden vectors produced by the reference itself."""
import math
import os
import zlib

import numpy as np
import pytest

import oracle
from conftest import VARIANT_PARAMS, golden_H, load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import channelcoding_b200 as cc
    c = cc.Context(0)
    yield c
    c.close()


def make_code(ctx, e):
    if e["family"] == 0:
        return ctx.bch(e["q"], **({"errors": e["cap_value"]} if e["cap_kind"] == 0 else {"dmin": e["cap_value"]}))
    return ctx.rs(e["q"], e["t"])


def assert_same(gpu, ref, what):
    gb, gL, gi, gf = gpu
    ob, oL, oi, of = ref
    assert np.array_equal(gf, of), what + ": failed flags"
    assert np.array_equal(gi.astype(np.uint32), oi.astype(np.uint32)), what + ": iteration index"
    assert np.array_equal(gb, ob), what + ": bits"
    if gL is not None and oL is not None:
        assert np.array_equal(gL.view(np.uint32), oL.view(np.uint32)), what + ": totals L (bit pattern)"


# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["bch_15_7", "bch_31_16", "bch_63_36", "bch_127_64", "bch_255_131"])
def test_decode_golden(ctx, name, catalogue, golden_codes):
    """all variants on the reference's own dumped LLRs: bits, L, iteration index, failure flag bit-exact"""
    g = load_golden("minsum_%s.npz" % name)
    e = catalogue[name]
    code = make_code(ctx, e)
    assert np.array_equal(code.H(), golden_H(golden_codes, catalogue, name))
    assert code.kernel == 1  # every catalogue code has a shape-specialised cyclic kernel
    y = g["y"]
    n = e["n"]
    for v, (variant, alpha, beta, max_iter) in VARIANT_PARAMS.items():
        if "v%d.iter" % v not in g:
            continue
        bits, L, it, failed = code.decode(y, variant, alpha, beta, max_iter)
        assert np.array_equal(failed, g["v%d.failed" % v]), (name, v)
        assert np.array_equal(it, g["v%d.iter" % v]), (name, v)
        ok = failed == 0
        gb = np.unpackbits(g["v%d.bits" % v], axis=1)[:, :n]
        assert np.array_equal(bits[ok], gb[ok]), (name, v)
        if "v%d.L" % v in g:
            assert np.array_equal(L[ok].view(np.uint32), g["v%d.L" % v][ok].view(np.uint32)), (name, v)


@pytest.mark.parametrize("name,frames,ebnos", [("bch_15_7", 4000, (0.0, 2.0, 5.0)), ("bch_31_16", 2000, (1.0, 4.0)),
                                                ("bch_63_36", 1500, (1.0, 3.0, 5.0)), ("bch_63_45", 600, (3.0,)),
                                                ("bch_31_26", 1500, (4.0,)), ("bch_63_57", 400, (5.0,)),
                                                ("bch_127_64", 60, (3.5,)), ("bch_127_106", 60, (5.0,)),
                                                ("bch_255_131", 24, (5.5,))])
def test_decode_vs_oracle(ctx, name, frames, ebnos, catalogue):
    """fresh seeded noise, failures included (state at the throw), both stop rules"""
    e = catalogue[name]
    code = make_code(ctx, e)
    H = code.H()
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    for eb in ebnos:
        y = (1 + oracle.sigma(e["rate"], eb) * rng.standard_normal((frames, e["n"]))).astype(np.float32)
        y[0] = 0.0
        y[1] = -1.0
        for variant, alpha, beta, mi, stop in (("MS", 1, 0, 50, 0), ("NMS", 0.8, 0, 50, 0), ("OMS", 1, 0.01, 20, 0),
                                               ("SCMS1", 1, 0, 30, 0), ("SCMS2", 1, 0, 50, 0),
                                               ("2DNMS", 0.9, 0.8, 25, 0), ("NMS", 0.8, 0, 50, 1), ("MS", 1, 0, 4, 2),
                                               ("SCMS2", 1, 0, 12, 1)):
            sel = slice(0, frames if e["n"] <= 63 else max(6, frames // 4))
            gpu = code.decode(y[sel], variant, alpha, beta, mi, stop)
            ref = oracle.min_sum(H, y[sel], variant, alpha, beta, mi, stop)
            assert_same(gpu, ref, "%s %s stop=%d ebno=%g" % (name, variant, stop, eb))


def test_device_pointer_path(ctx, catalogue):
    """torch CUDA tensors (device path, async on the context's stream) == numpy (host path)"""
    import torch
    e = catalogue["bch_63_36"]
    code = make_code(ctx, e)
    rng = np.random.default_rng(3)
    y = (1 + 0.75 * rng.standard_normal((5000, 63))).astype(np.float32)
    host = code.decode(y, "NMS", 0.8)
    yt = torch.from_numpy(y).cuda()
    torch.cuda.synchronize()
    dev = code.decode(yt, "NMS", 0.8)
    ctx.sync()
    assert_same(tuple(t.cpu().numpy() for t in dev), host, "device path")


def test_csr_kernel_general_H(ctx, catalogue, golden_codes):
    """a matrix without cyclic structure (H_alt of the reference, and a row-permuted H) runs on the
    CSR kernel and matches the oracle; the same H in cyclic form gives identical decisions."""
    e = catalogue["bch_63_45"]
    rng = np.random.default_rng(9)
    H = golden_H(golden_codes, catalogue, "bch_63_45")
    Halt = golden_H(golden_codes, catalogue, "bch_63_45", alt=True)
    y = (1 + oracle.sigma(e["rate"], 4.0) * rng.standard_normal((300, 63))).astype(np.float32)
    for M in (Halt, H[rng.permutation(H.shape[0])]):
        code = ctx.from_dense(M, e["rate"])
        assert code.kernel == 2 and code.h_kind == 2
        for variant, alpha, beta, stop in (("MS", 1, 0, 0), ("NMS", 0.8, 0, 1), ("SCMS1", 1, 0, 0), ("OMS", 1, 0.05, 0)):
            assert_same(code.decode(y, variant, alpha, beta, 20, stop), oracle.min_sum(M, y, variant, alpha, beta, 20, stop),
                        "csr " + variant)
    code = ctx.from_dense(H, e["rate"])
    assert code.kernel == 1 and code.h_kind == 0


@pytest.mark.parametrize("name,rows", [("bch_15_7", 15), ("bch_31_16", 31), ("bch_63_36", 63), ("bch_63_36", 40),
                                       ("bch_127_64", 127), ("bch_255_131", 255), ("bch_255_131", 200)])
def test_redundant_rows(ctx, name, rows, catalogue):
    """redundant parity-check matrix: `rows` cyclic shifts with wrap-around (extension; parity unpinned
    by the reference, checked against the restatement which keeps the reference's loop order)"""
    e = catalogue[name]
    code = make_code(ctx, e)
    code.set_rows(rows)
    assert code.h_rows == rows and code.kernel == 1
    oc = oracle.Code(0, e["q"], e["t"])
    H = oc.H(rows)
    assert np.array_equal(code.H(), H)
    rng = np.random.default_rng(rows)
    frames = 400 if e["n"] <= 63 else (24 if e["n"] <= 127 else 6)
    y = (1 + oracle.sigma(e["rate"], 3.0) * rng.standard_normal((frames, e["n"]))).astype(np.float32)
    for variant, alpha, stop in (("NMS", 0.8, 1), ("MS", 1.0, 0), ("SCMS2", 1.0, 1)):
        assert_same(code.decode(y, variant, alpha, 0.0, 15, stop), oracle.min_sum(H, y, variant, alpha, 0.0, 15, stop),
                    "redundant %s %d %s" % (name, rows, variant))


SPA_TOL = 5e-2  # stated tolerance of the float32 sum-product totals: ||L - L64||_inf / ||L64||_inf per iteration (see below)


def _first_divergence(code, H, llr, kmax):
    """first iteration k at which the float32 kernel and the float64 yardstick decide a column differently ->
    (k, column, |L64| there, ||L64||_inf) or None"""
    for k in range(1, kmax + 1):
        gb, gL, _, _ = code.decode(llr[None, :], "SPA", max_iter=k, stop_rule=2)
        ob, oL, _, _ = oracle.spa_f64(H, llr[None, :], k, 2)
        diff = np.nonzero(gb[0] != ob[0])[0]
        if len(diff):
            c = int(diff[0])
            return k, c, abs(float(oL[0, c])), float(np.abs(oL[0]).max())
    return None


def test_sum_product_extension(ctx, catalogue):
    """SPA (tanh rule) is an extension: the reference has no such decoder, so parity is UNPINNED by it.  The yardstick
    is the same flooding loop in float64 (oracle_spa_f64).  north_star asks for "floating-point sum-product messages
    agree within a stated relative tolerance"; stated and checked here:
      * totals after k iterations (no stop rule): ||L_gpu - L64||_inf / ||L64||_inf <= 5e-2 for every frame and every
        k tested, median below 5e-3.  The bound is that loose only because of SATURATED messages: the exclusive tanh
        product is clamped to +-0.99999994, where one float32 ulp of the product moves 2 atanh by 0.35 -- on totals
        of magnitude 20..70; unsaturated messages agree to 1e-6.
      * BCH(15,7), 1..6 dB, 20 000 frames per point: hard decisions, iteration index and failure flag equal the
        float64 run on >= 99.95 % of the frames, and EVERY disagreeing frame sits on a decision boundary: at the first
        iteration where a decided bit differs, the float64 total of that column is inside the tolerance band.
      * the float32 restatement (ms_oracle.c, same prefix x suffix association as the kernel) is compared as well."""
    e = catalogue["bch_15_7"]
    code = make_code(ctx, e)
    H = code.H()
    rng = np.random.default_rng(4)
    total = agree = 0
    for eb in (1.0, 2.0, 3.0, 4.0, 5.0, 6.0):
        sig = oracle.sigma(e["rate"], eb)
        llr = (2.0 / sig ** 2 * (1 + sig * rng.standard_normal((20000, 15)))).astype(np.float32)
        gb, gL, gi, gf = code.decode(llr, "SPA", max_iter=50, stop_rule=1)
        ob, oL, oi, of = oracle.spa_f64(H, llr, 50, 1)
        same = (gi == oi) & (gf == of) & (gb == ob).all(axis=1)
        total += len(same)
        agree += int(same.sum())
        for f in np.nonzero(~same)[0][:20]:
            d = _first_divergence(code, H, llr[f], 50)
            assert d is not None, (eb, f)
            k, c, l64, linf = d
            assert l64 <= SPA_TOL * linf, "frame %d at %g dB diverges at iteration %d away from a decision boundary: |L|=%g of %g" % (f, eb, k, l64, linf)
        # per-iteration tolerance of the totals
        for k in (1, 2, 3, 5, 10, 20):
            _, La, _, _ = code.decode(llr[:3000], "SPA", max_iter=k, stop_rule=2)
            _, Lb, _, _ = oracle.spa_f64(H, llr[:3000], k, 2)
            rel = np.abs(La - Lb).max(axis=1) / np.abs(Lb).max(axis=1)
            assert rel.max() <= SPA_TOL and np.median(rel) <= 5e-3, (eb, k, rel.max(), np.median(rel))
        # float32 restatement vs the kernel: same association, only tanhf / atanhf differ in the last ulp
        rb, rL, ri, rf = oracle.min_sum(H, llr[:5000], "SPA", max_iter=50, stop_rule=1)
        same32 = (gi[:5000] == ri) & (gf[:5000] == rf) & (gb[:5000] == rb).all(axis=1)
        assert same32.mean() >= 0.9995, (eb, same32.mean())
    assert agree / total >= 0.9995, (agree, total)
    # the same on the general (CSR) kernel: rows permuted so that the cyclic structure is gone
    sig = oracle.sigma(e["rate"], 3.0)
    llr = (2.0 / sig ** 2 * (1 + sig * rng.standard_normal((4000, 15)))).astype(np.float32)
    perm = np.random.default_rng(2).permutation(code.h_rows)
    g = ctx.from_dense(H[perm], e["rate"])
    assert code.kernel == 1 and g.kernel == 2
    gb2, gL2, gi2, gf2 = g.decode(llr, "SPA", max_iter=10, stop_rule=1)
    ob2, oL2, oi2, of2 = oracle.spa_f64(H[perm], llr, 10, 1)
    same2 = (gi2 == oi2) & (gf2 == of2) & (gb2 == ob2).all(axis=1)
    assert same2.mean() >= 0.999
    # larger code on the cyclic kernel: agreement and the same decision-boundary argument
    e63 = catalogue["bch_63_36"]
    c63 = make_code(ctx, e63)
    H63 = c63.H()
    sig = oracle.sigma(e63["rate"], 4.0)
    llr = (2.0 / sig ** 2 * (1 + sig * rng.standard_normal((400, 63)))).astype(np.float32)
    gb, gL, gi, gf = c63.decode(llr, "SPA", max_iter=20, stop_rule=1)
    ob, oL, oi, of = oracle.spa_f64(H63, llr, 20, 1)
    same = (gi == oi) & (gf == of) & (gb == ob).all(axis=1)
    assert same.mean() >= 0.98, same.mean()
    for f in np.nonzero(~same)[0][:8]:
        d = _first_divergence(c63, H63, llr[f], 20)
        assert d is not None and d[2] <= SPA_TOL * d[3], (f, d)


# ---------------------------------------------------------------------------------------------------
def test_channel_kernel(ctx):
    """K1 against the CPU restatement: Philox stream identical, Box-Muller within MUFU tolerance"""
    for n, sigma_f in ((63, 0.75), (15, 1.1), (127, 0.5), (255, 0.66)):
        y = ctx.awgn_llr(n, sigma_f, seed=7, point=3, frame0=123456789012, frames=3001)
        ref = oracle.awgn(7, 3, 123456789012, 3001, n, sigma_f)
        err = np.abs(y - ref)
        assert err.max() < 2e-5 * max(1.0, sigma_f * 7), (n, err.max())
        assert np.median(err) < 5e-7
    # frame offsets address the same stream
    a = ctx.awgn_llr(63, 0.7, 1, 0, 0, 1000)
    b = ctx.awgn_llr(63, 0.7, 1, 0, 500, 500)
    assert np.array_equal(a[500:], b)


def test_channel_distribution(ctx):
    """the GPU channel kernel itself (Philox4x32-10 + MUFU Box-Muller), not its closeness to the CPU restatement:
    1.0e8 samples against the standard normal distribution -- four moments, the Kolmogorov-Smirnov distance on a
    4000-bin grid, tail probabilities and the lag-1 correlation, each within a 4-sigma band of its sampling error"""
    import math
    import torch
    n, frames, sigma_f = 63, 1600000, 0.75
    y = torch.empty((frames, n), dtype=torch.float32, device="cuda")
    ctx.awgn_llr(n, sigma_f, seed=11, point=5, frame0=10 ** 12, frames=frames, out=y)
    ctx.sync()
    z = ((y.double() - 1.0) / float(np.float32(sigma_f))).flatten()
    N = z.numel()
    assert N >= 10 ** 8
    m = z.mean().item()
    c = z - m
    var = (c * c).mean().item()
    skew = (c ** 3).mean().item() / var ** 1.5
    kurt = (c ** 4).mean().item() / var ** 2 - 3.0
    assert abs(m) < 4 / math.sqrt(N), m
    assert abs(var - 1.0) < 4 * math.sqrt(2.0 / N), var
    assert abs(skew) < 4 * math.sqrt(6.0 / N), skew
    assert abs(kurt) < 4 * math.sqrt(24.0 / N), kurt
    # Kolmogorov-Smirnov on a grid: sup |F_N - Phi| over 4000 bin edges in [-8, 8]; the 99.9 % critical value is 1.95 / sqrt(N)
    bins = 4000
    hist = torch.histc(z.float(), bins=bins, min=-8.0, max=8.0).double()
    below = (z < -8.0).sum().item()
    cdf = (torch.cumsum(hist, 0) + below) / N
    edges = torch.linspace(-8.0, 8.0, bins + 1, dtype=torch.float64, device="cuda")[1:]
    phi = 0.5 * (1.0 + torch.erf(edges / math.sqrt(2.0)))
    ks = (cdf - phi).abs().max().item()
    assert ks < 1.95 / math.sqrt(N) + 2e-6, ks  # (+ float32 binning of the grid)
    # tails (what the word error rate at high Eb/N0 lives on)
    for thr in (2.0, 3.0, 4.0, 4.5):
        p = 0.5 * math.erfc(thr / math.sqrt(2.0))
        for tail in ((z > thr), (z < -thr)):
            k = tail.sum().item()
            assert abs(k - N * p) < 4.5 * math.sqrt(N * p) + 1, (thr, k, N * p)
    # neighbouring samples (same Philox block / Box-Muller pair and across blocks) are uncorrelated
    zz = z.view(frames, n)
    for lag in (1, 2, 4):
        r = (zz[:, :-lag] * zz[:, lag:]).mean().item()
        assert abs(r) < 4.5 / math.sqrt(frames * (n - lag)), (lag, r)
    r = (zz[:-1, :] * zz[1:, :]).mean().item()   # same column of consecutive frames
    assert abs(r) < 4.5 / math.sqrt((frames - 1) * n), r


def test_fused_point_equals_streaming(ctx, catalogue):
    """ccgpu_awgn_point (channel + decode + count fused) == K1 -> ccgpu_decode_llr -> count on the host"""
    for name, eb, frames in (("bch_63_36", 3.0, 20000), ("bch_15_7", 2.0, 30000), ("bch_127_64", 4.0, 3000),
                             ("bch_255_131", 5.0, 600)):
        e = catalogue[name]
        code = make_code(ctx, e)
        import channelcoding_b200 as cc
        sig = cc.sigma(e["rate"], eb)
        y = ctx.awgn_llr(e["n"], np.float32(sig), seed=11, point=5, frame0=1000, frames=frames)
        bits, L, it, failed = code.decode(y, "NMS", 0.8)
        c = code.awgn_point(eb, frames, "NMS", 0.8, seed=11, point=5, frame0=1000)
        nb = bits.sum(axis=1)
        assert c["frames"] == frames
        assert c["failures"] == int(failed.sum())
        assert c["frame_errors"] == int(((failed == 1) | (nb > 0)).sum())
        assert c["bit_errors"] == int(nb.sum())
        assert c["iterations"] == int(np.where(failed == 1, 50, it.astype(np.int64) + 1).sum())
        assert c["undetected"] == 0
        # sharding by frame range gives the same totals (what N GPUs do)
        parts = [code.awgn_point(eb, frames // 4, "NMS", 0.8, seed=11, point=5, frame0=1000 + i * (frames // 4))
                 for i in range(4)]
        for k in c:
            assert sum(p[k] for p in parts) == c[k]


def test_bitflip_table3(ctx, kat, catalogue):
    """bitflips.c++ / report Table 3 on BCH(31,16,7), all C(31,w) patterns per weight"""
    code = make_code(ctx, catalogue["bch_31_16"])
    for w in range(0, 4):
        row = kat["bitflip_31_16_7"][str(w)]
        for v in range(6):
            variant, alpha, beta, mi = VARIANT_PARAMS[v]
            c = code.bitflip_point(w, variant, alpha, beta, mi)
            assert c["frames"] == row["patterns"] == math.comb(31, w)
            assert c["frame_errors"] == row[variant], (w, variant)
    # weights 4..6: published percentages of the parameter-free decoders (report p.33)
    for variant in ("MS", "SCMS1", "SCMS2"):
        for w in (4, 5, 6):
            c = code.bitflip_point(w, variant)
            pct = 100.0 * c["frame_errors"] / c["frames"]
            assert abs(pct - kat["table3_percent"][variant][w]) <= 0.06, (variant, w, pct)
    # pattern order = std::next_permutation order from 0..01..1
    first = code.bitflip_point(2, "MS", first=0, count=1)
    assert first["frames"] == 1


# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["rs_255_223", "rs_15_9", "rs_7_3", "rs_7_5", "bch_15_7", "bch_31_16", "bch_63_36",
                                  "bch_127_64", "bch_255_131"])
def test_gf_decode_golden(ctx, name, catalogue):
    g = load_golden("hard_%s.npz" % name)
    e = catalogue[name]
    code = make_code(ctx, e)
    assert np.array_equal(code.encode(g["msgs"]), g["words"])
    out, nerr, failed = code.gf_decode(g["received"])
    assert np.array_equal(failed, (g["status"] != 0).astype(np.uint8))
    ok = failed == 0
    assert np.array_equal(out[ok], g["corrected"][ok])
    assert np.array_equal(out[~ok], g["received"][~ok])
    assert np.array_equal(nerr[ok], (g["corrected"][ok] != g["received"][ok]).sum(axis=1))


@pytest.mark.parametrize("fam,q,t,count", [(1, 8, 16, 20000), (0, 8, 18, 4000), (0, 6, 5, 20000), (1, 4, 3, 20000)])
def test_gf_decode_vs_oracle(ctx, fam, q, t, count):
    rng = np.random.default_rng(q * 31 + t)
    oc = oracle.Code(fam, q, t)
    code = ctx.bch(q, errors=t) if fam == 0 else ctx.rs(q, t)
    msgs = rng.integers(0, (1 << q) if fam == 1 else 2, size=(count, oc.l)).astype(np.uint8)
    words = code.encode(msgs)
    assert np.array_equal(words[:200], oc.encode(msgs[:200]))
    bad = words.copy()
    ne = rng.integers(0, t + 4, size=count)
    for i in range(count):
        pos = rng.choice(oc.n, ne[i], replace=False)
        bad[i, pos] ^= (rng.integers(1, 1 << q, size=ne[i]).astype(np.uint8) if fam == 1 else 1)
    out, nerr, failed = code.gf_decode(bad)
    # bounded-distance property at full size
    within = ne <= t
    assert not failed[within].any() and np.array_equal(out[within], words[within])
    assert ((out[failed == 0] != bad[failed == 0]).sum(axis=1) <= t).all()
    # oracle (Euklid restatement) on a sample incl. every beyond-t word of the first 3000
    sel = np.arange(min(count, 3000))
    oo, on, os_ = oc.hard_correct(bad[sel])
    assert np.array_equal(failed[sel], (os_ != 0).astype(np.uint8))
    good = os_ == 0
    assert np.array_equal(out[sel][good], oo[good])


def test_exercises(ctx, kat, catalogue):
    """exercises.c++ tasks 6.1-6.10, errors-only cases"""
    for key, ex in kat["exercises"].items():
        if ex["erasures"]:
            continue
        code = make_code(ctx, catalogue[ex["code"]])
        out, nerr, failed = code.gf_decode(np.asarray([ex["received"]], np.uint8))
        if ex["expect"] == "unspecified":
            if not failed[0] and ex["status"] == 0:
                assert list(map(int, out[0])) == ex["corrected"], key
        elif ex["expect"] is None:
            assert failed[0] == 1, key
        else:
            assert failed[0] == 0 and list(map(int, out[0])) == ex["expect"], key


# ---------------------------------------------------------------------------------------------------
def test_wer_matches_reference_statistics(ctx, catalogue):
    """WER of the fused engine (Philox noise) vs the reference's own CPU simulation (mt19937_64
    noise) at the same Eb/N0: inside the 95 % interval of the difference of two proportions.  The
    reference's counts are the 1e5 frames per point it simulated of BCH(63,36) NMS (oracle/make_golden_wer.py
    -> tests/golden/ref_wer.json)."""
    import json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_wer.json")) as f:
        gold = [p for p in json.load(f)["points"] if p["code"] == "bch_63_36"]
    assert [(p["variant"], p["alpha"], p["max_iter"], p["ebno_db"]) for p in gold] == \
        [("NMS", 0.8, 50, eb) for eb in (2.0, 4.0, 5.0)]
    e = catalogue["bch_63_36"]
    code = make_code(ctx, e)
    for p in gold:
        eb, rf, rw = p["ebno_db"], p["frames"], p["word_errors"]
        c = code.awgn_point(eb, 2_000_000, "NMS", 0.8, seed=1, point=int(eb * 2))
        p1, p2 = rw / rf, c["frame_errors"] / c["frames"]
        se = math.sqrt(p1 * (1 - p1) / rf + p2 * (1 - p2) / c["frames"])
        assert abs(p1 - p2) <= 1.96 * se + 1e-9, (eb, p1, p2, se)


def test_wer_matches_reference_at_1e5_frames(ctx, catalogue):
    """the statistical leg with power: nine points (BCH(15,7) MS, BCH(63,36) NMS, BCH(127,64) NMS, three Eb/N0 each)
    for which the REFERENCE ITSELF simulated 1e5 frames with its own noise source (oracle/make_golden_wer.py ->
    tests/golden/ref_wer.json).  The engine simulates 1e7 frames per point (its own sampling error is a tenth of the
    reference's), so the comparison is against the binomial interval of the reference's finite sample:
    every point inside 3.3 sigma (99.9 %: nine comparisons at 95 % would fail a correct engine every third run),
    at least seven of the nine inside the 95 % interval, and no systematic bias (mean signed deviation small).
    A relative WER bias of 2 % in the channel kernel is 2.6 sigma at the WER = 0.64 point and would show."""
    import json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_wer.json")) as f:
        gold = json.load(f)
    assert len(gold["points"]) == 9 and all(p["frames"] >= 100000 for p in gold["points"])
    devs = []
    for i, p in enumerate(gold["points"]):
        e = catalogue[p["code"]]
        code = make_code(ctx, e)
        frames = 10_000_000 if e["n"] <= 63 else 4_000_000
        c = code.awgn_point(p["ebno_db"], frames, p["variant"], p["alpha"], 0.0, p["max_iter"], seed=77, point=i)
        pr, pg = p["word_errors"] / p["frames"], c["frame_errors"] / c["frames"]
        se = math.sqrt(pg * (1 - pg) / p["frames"] + pg * (1 - pg) / frames)
        devs.append((pr - pg) / se)
        assert abs(devs[-1]) <= 3.3, (p["code"], p["ebno_db"], pr, pg, devs[-1])
    devs = np.array(devs)
    assert (np.abs(devs) <= 1.96).sum() >= 7, devs
    assert abs(devs.mean()) <= 1.2, devs   # nine independent unit normals: the mean has sigma 1/3


# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fam,q,t,count", [(1, 4, 3, 6000), (1, 8, 16, 3000), (1, 3, 2, 3000), (0, 5, 3, 3000),
                                           (0, 6, 5, 2000)])
def test_gf_decode_erasures_vs_oracle(ctx, fam, q, t, count):
    """errors + erasures (cyclic::correct(b, erasures), hard_decision.h:171-172) against the Euklid
    restatement word by word, decodable and undecodable mixes; binary codes follow the reference's
    flip-every-erasure behaviour (bch.h:80-83)"""
    rng = np.random.default_rng(q * 1000 + t)
    oc = oracle.Code(fam, q, t)
    code = ctx.bch(q, errors=t) if fam == 0 else ctx.rs(q, t)
    n = oc.n
    max_e = min(2 * t + 2, 30)
    msgs = rng.integers(0, (1 << q) if fam == 1 else 2, size=(count, oc.l)).astype(np.uint8)
    words = code.encode(msgs)
    bad = words.copy()
    epos = np.zeros((count, max_e), np.uint8)
    ecnt = np.zeros(count, np.uint8)
    for i in range(count):
        f = int(rng.integers(0, max_e + 1))
        e = int(rng.integers(0, max(1, (2 * t - f) // 2 + 2)))
        e = min(e, n - f)
        pos = rng.choice(n, f + e, replace=False)
        if fam == 1:
            bad[i, pos[:f]] = rng.integers(0, 1 << q, size=f).astype(np.uint8) * (rng.random() < 0.5)
            bad[i, pos[f:]] ^= rng.integers(1, 1 << q, size=e).astype(np.uint8)
        else:
            bad[i, pos[:f]] = 0
            bad[i, pos[f:]] ^= 1
        epos[i, :f] = pos[:f]
        ecnt[i] = f
    out, nerr, failed = code.gf_decode(bad, erasures=(epos, ecnt))
    sel = np.arange(min(count, 1500))
    beyond = 0
    for i in sel:
        rho = int(ecnt[i])
        oo, on, os_ = oc.hard_correct(bad[i:i + 1], [int(x) for x in epos[i, :rho]])
        # bounded-distance region of errors-and-erasures decoding: 2 * errors + erasures <= 2t, i.e. the
        # errata locator has degree L with 2L <= 2t + rho.  There the engine equals the reference exactly.
        # With an ODD number of erasures the reference's Euklid stop rule (hard_decision.h:164,181:
        # max = (2t + rho) / 2 in integer arithmetic) also accepts degree L = (2t + rho + 1) / 2, one beyond
        # the guarantee, where the solution is not unique (it miscorrects in part of those cases); the
        # engine declares a decoding failure there (documented deviation, DESIGN.md 7).
        if os_[0] == 0 and 2 * int(on[0]) <= 2 * t + rho:
            assert failed[i] == 0 and np.array_equal(out[i], oo[0]) and nerr[i] == on[0], (i, rho)
        elif os_[0] == 0:
            assert rho % 2 == 1 and 2 * int(on[0]) == 2 * t + rho + 1 and failed[i] == 1, (i, rho, on[0])
            beyond += 1
        else:
            assert failed[i] == 1, (i, rho)
        if failed[i] == 0:
            assert os_[0] == 0
    # every word constructed inside the bound is recovered
    # erasure-only decoding up to 2t erasures recovers the word (RS); zero erasures == plain decode
    out0, nerr0, failed0 = code.gf_decode(bad[ecnt == 0]) if (ecnt == 0).any() else (None, None, None)
    if out0 is not None:
        assert np.array_equal(out0, out[ecnt == 0]) and np.array_equal(failed0, failed[ecnt == 0])


def test_exercises_with_erasures(ctx, kat, catalogue):
    """exercises.c++ tasks 6.7 / 6.8: RS(7,3) with erasures"""
    for key in ("6.7", "6.8"):
        ex = kat["exercises"][key]
        code = make_code(ctx, catalogue[ex["code"]])
        er = np.zeros((1, 4), np.uint8)
        er[0, :len(ex["erasures"])] = ex["erasures"]
        out, nerr, failed = code.gf_decode(np.asarray([ex["received"]], np.uint8),
                                           erasures=(er, np.asarray([len(ex["erasures"])], np.uint8)))
        assert failed[0] == 0 and list(map(int, out[0])) == ex["expect"], key


def test_gf_recheck_is_implied(ctx):
    """the re-syndrome check of cyclic.h:243-248 never changes an erasure-free result (it is implied by
    deg Lambda <= t with deg Lambda distinct roots): 2e5 RS(255,223) words with 0..24 errors, with and
    without the check, and every accepted word has all-zero syndromes"""
    rng = np.random.default_rng(77)
    code = ctx.rs(8, 16)
    oc = oracle.Code(1, 8, 16)
    count = 200000
    base = code.encode(rng.integers(0, 256, size=(512, code.l)).astype(np.uint8))
    bad = np.tile(base, (count // 512 + 1, 1))[:count].copy()
    ne = rng.integers(0, 25, size=count)
    rows = np.repeat(np.arange(count), ne)
    cols = rng.integers(0, 255, size=rows.size)
    bad[rows, cols] ^= rng.integers(1, 256, size=rows.size).astype(np.uint8)
    fast = code.gf_decode(bad)
    code.set_recheck(True)
    slow = code.gf_decode(bad)
    code.set_recheck(False)
    for a, b in zip(fast, slow):
        assert np.array_equal(a, b)
    ok = np.flatnonzero(fast[2] == 0)
    assert 0.5 < len(ok) / count < 0.8
    for i in ok[:: max(1, len(ok) // 400)]:
        assert not oc.syndromes(fast[0][i]).any()


def test_uncovered_columns_use_the_general_stop_test(ctx, catalogue, golden_codes):
    """a matrix whose rows do not cover every column: the reference's stop rule is then NOT equivalent to
    'decided word is all-zero' (bits in uncovered columns are ignored), the kernel must evaluate overlaps"""
    H = golden_H(golden_codes, catalogue, "bch_63_36")[:10]
    code = ctx.from_dense(H, 36 / 63)
    assert code.kernel == 1 and code.h_rows == 10
    rng = np.random.default_rng(12)
    y = (1 + 0.6 * rng.standard_normal((500, 63))).astype(np.float32)
    y[:, 50:] = -np.abs(y[:, 50:])  # uncovered columns decided as ones
    for stop in (0, 1):
        assert_same(code.decode(y, "NMS", 0.8, 0.0, 20, stop), oracle.min_sum(H, y, "NMS", 0.8, 0.0, 20, stop), "partial H")
    gb, gL, gi, gf = code.decode(y, "NMS", 0.8, 0.0, 20, 0)
    assert (gf == 0).any() and gb[gf == 0][:, 50:].all()


def test_hard_decision_awgn_point(ctx, catalogue):
    """ccgpu_awgn_point_hard (channel + hard decision + algebraic decode + count on the device) ==
    K1 -> host hard decision (codes.h:43-52) -> ccgpu_gf_decode -> host count (simulation.c++:126-135)"""
    import channelcoding_b200 as cc
    for name, eb, frames in (("bch_31_16", 3.0, 50000), ("bch_63_36", 4.0, 40000), ("bch_127_64", 5.0, 20000),
                             ("bch_255_131", 6.0, 5000)):
        e = catalogue[name]
        code = make_code(ctx, e)
        y = ctx.awgn_llr(e["n"], np.float32(cc.sigma(e["rate"], eb)), seed=9, point=4, frame0=77, frames=frames)
        out, nerr, failed = code.gf_decode((y < 0).astype(np.uint8))
        nz = (out != 0).sum(axis=1)
        c = code.awgn_point_hard(eb, frames, seed=9, point=4, frame0=77)
        assert c["frames"] == frames and c["iterations"] == 0
        assert c["failures"] == int(failed.sum())
        assert c["bit_errors"] == int(nz.sum())
        assert c["frame_errors"] == int(((failed == 1) | (nz > 0)).sum())
        assert c["undetected"] == int(((failed == 0) & (nz > 0)).sum())
        halves = [code.awgn_point_hard(eb, frames // 2, seed=9, point=4, frame0=77 + i * (frames // 2)) for i in range(2)]
        assert all(halves[0][k] + halves[1][k] == c[k] for k in c)


def test_edge_cases_and_errors(ctx, catalogue):
    """empty and single-frame batches, iteration limits, and the error contract of the ABI (an error code
    plus ccgpu_last_error text, never an exception across the boundary, never a silent fallback)"""
    import torch
    import channelcoding_b200 as cc
    code = make_code(ctx, catalogue["bch_63_36"])
    H = code.H()
    empty = code.decode(np.zeros((0, 63), np.float32), "NMS", 0.8)
    assert empty[0].shape == (0, 63) and empty[3].shape == (0,)
    assert code.awgn_point(4.0, 0, "NMS", 0.8)["frames"] == 0
    rng = np.random.default_rng(8)
    one = (1 + 0.8 * rng.standard_normal((1, 63))).astype(np.float32)
    assert_same(code.decode(one, "NMS", 0.8), oracle.min_sum(H, one, "NMS", 0.8), "single frame")
    y = (1 + 0.9 * rng.standard_normal((999, 63))).astype(np.float32)  # odd count: partial last warp / CTA
    for mi in (1, 2, 255):
        assert_same(code.decode(y, "OMS", 1.0, 0.02, mi), oracle.min_sum(H, y, "OMS", 1.0, 0.02, mi), "max_iter %d" % mi)
    # HEAD behaviour of the reference (matrix.h:50 bug): exactly one iteration, never a failure
    gb, gL, gi, gf = code.decode(y, "NMS", 0.8, 0.0, 1, cc.STOP_NONE)
    assert not gf.any() and not gi.any()
    for kwargs, text in (({"max_iter": 0}, "max_iter"), ({"max_iter": 256}, "max_iter"),
                         ({"variant": "OMS", "beta": -0.1}, "beta"), ({"stop_rule": 7}, "stop rule")):
        args = dict(variant="NMS", alpha=0.8, beta=0.0, max_iter=50, stop_rule=0)
        args.update(kwargs)
        with pytest.raises(cc.CcgpuError) as ei:
            code.decode(y, **args)
        assert ei.value.code == -1 and text in str(ei.value)
    with pytest.raises(cc.CcgpuError) as ei:  # device input with a host output buffer
        code.decode(torch.from_numpy(y).cuda(), "NMS", 0.8,
                    out=(np.empty((999, 63), np.uint8), None, np.empty(999, np.uint8), np.empty(999, np.uint8)))
    assert "device pointer" in str(ei.value)
    other = cc.Context(0)
    foreign = other.bch(6, errors=5)
    foreign.ctx = ctx  # hand the other context's code to this context: the ABI must refuse it
    with pytest.raises(cc.CcgpuError) as ei:
        foreign.decode(y, "NMS", 0.8)
    assert "not created on this context" in str(ei.value)
    foreign.ctx = other
    foreign.close()
    other.close()
    with pytest.raises(cc.CcgpuError):
        ctx.rs(8, 200)  # 2t >= n
    with pytest.raises(cc.CcgpuError):
        ctx.bch(9, errors=2)  # q > 8
    dense = ctx.from_dense(H, 36 / 63)
    with pytest.raises(cc.CcgpuError) as ei:
        dense.gf_decode(np.zeros((1, 63), np.uint8))
    assert ei.value.code == -3  # CCGPU_ERR_UNSUPPORTED: no field / roots behind a dense matrix


# ---------------------------------------------------------------------------------------------------
# multiple-bases decoding (extension, include/ccgpu.h ccgpu_decode_llr_mbbp)
def mbbp_restatement(H, y, shifts, variant, alpha, beta, max_iter, stop_rule):
    """the definition in include/ccgpu.h on the CPU: oracle decode of every rotation, rotate back, float32 correlation
    accumulated column by column, best converged candidate (ties: lowest base), else best failed candidate"""
    frames, n = y.shape
    cands = []
    for s in shifts:
        b, L, it, failed = oracle.min_sum(H, np.roll(y, -int(s), axis=1), variant, alpha, beta, max_iter, stop_rule)
        x = np.roll(b, int(s), axis=1)
        m = np.cumsum(np.where(x != 0, -y, y).astype(np.float32), axis=1, dtype=np.float32)[:, -1]
        cands.append((x, np.roll(L, int(s), axis=1), it, failed, m))
    bits = np.empty((frames, n), np.uint8)
    Lout = np.empty((frames, n), np.float32)
    it_out = np.empty(frames, np.uint32)
    failed_out = np.empty(frames, np.uint8)
    chosen = np.empty(frames, np.uint8)
    for f in range(frames):
        best = None
        for bi, (x, L, it, failed, m) in enumerate(cands):
            ok = failed[f] == 0
            if best is None or (ok and not best[1]) or (ok == best[1] and m[f] > best[2]):
                best = (bi, ok, m[f])
        bi = best[0]
        bits[f], Lout[f], it_out[f], failed_out[f], chosen[f] = cands[bi][0][f], cands[bi][1][f], cands[bi][2][f], 0 if best[1] else 1, bi
    return bits, Lout, it_out, failed_out, chosen


def test_mbbp_single_base_is_plain(ctx, catalogue):
    code = make_code(ctx, catalogue["bch_63_36"])
    rng = np.random.default_rng(41)
    y = (1 + oracle.sigma(36 / 63, 3.0) * rng.standard_normal((4000, 63))).astype(np.float32)
    plain = code.decode(y, "NMS", 0.8)
    b, L, it, failed, chosen = code.decode_mbbp(y, [0], "NMS", 0.8)
    assert_same((b, L, it, failed), plain, "one base, no rotation")
    assert not chosen.any()


@pytest.mark.parametrize("name,frames,ebno", [("bch_31_16", 1500, 3.0), ("bch_63_36", 800, 3.5), ("bch_127_64", 40, 4.0)])
def test_mbbp_matches_restatement(ctx, name, frames, ebno, catalogue):
    """random codewords, GF(2) stop rule, four rotations: every output equals the CPU restatement built on the oracle"""
    import torch
    e = catalogue[name]
    code = make_code(ctx, e)
    n = e["n"]
    rng = np.random.default_rng(zlib.crc32(("mbbp" + name).encode()))
    words = code.encode(rng.integers(0, 2, size=(frames, e["l"])).astype(np.uint8))
    y = ((1.0 - 2.0 * words) + oracle.sigma(e["rate"], ebno) * rng.standard_normal((frames, n))).astype(np.float32)
    shifts = [0, 5, n // 2, n - 3]
    for variant, alpha, beta, mi in (("NMS", 0.8, 0.0, 20), ("SCMS2", 1.0, 0.0, 15)):
        ref = mbbp_restatement(code.H(), y, shifts, variant, alpha, beta, mi, 1)
        got = code.decode_mbbp(y, shifts, variant, alpha, beta, mi, 1)
        assert np.array_equal(got[4], ref[4]), (name, variant, "chosen base")
        assert_same(got[:4], ref[:4], "%s %s multiple bases" % (name, variant))
        # device pointers give the same
        dev = code.decode_mbbp(torch.from_numpy(y).cuda(), shifts, variant, alpha, beta, mi, 1)
        ctx.sync()
        assert_same(tuple(t.cpu().numpy() for t in dev[:4]), ref[:4], "%s %s device path" % (name, variant))
        # more bases never lose a frame the first base decodes to a codeword with a better metric; here: the
        # multiple-bases word error rate is not worse than the single-base one
        single = code.decode(y, variant, alpha, beta, mi, 1)
        err_single = ((single[0] != words).any(axis=1) | (single[3] != 0)).mean()
        err_multi = ((got[0] != words).any(axis=1) | (got[3] != 0)).mean()
        assert err_multi <= err_single + 1e-9, (name, variant, err_single, err_multi)


def test_mbbp_point(ctx, catalogue):
    """fused point: counters equal channel kernel -> decode_mbbp -> host count, shards add up, and rotations help"""
    import channelcoding_b200 as cc
    code = make_code(ctx, catalogue["bch_63_36"])
    frames, eb, shifts = 40000, 4.0, [0, 7, 19, 31, 44, 58]
    c = code.awgn_point_mbbp(eb, frames, shifts, "NMS", 0.8, seed=5, point=2, frame0=64)
    y = ctx.awgn_llr(63, np.float32(cc.sigma(code.rate, eb)), seed=5, point=2, frame0=64, frames=frames)
    b, _, it, failed, _ = code.decode_mbbp(y, shifts, "NMS", 0.8, want_L=False)
    nz = b.any(axis=1)
    assert c["frames"] == frames and c["failures"] == int(failed.sum())
    assert c["frame_errors"] == int((nz | (failed != 0)).sum()) and c["bit_errors"] == int(b.sum())
    assert c["undetected"] == int((nz & (failed == 0)).sum())
    halves = [code.awgn_point_mbbp(eb, frames // 2, shifts, "NMS", 0.8, seed=5, point=2, frame0=64 + i * (frames // 2)) for i in range(2)]
    for k in ("frames", "frame_errors", "bit_errors", "iterations", "failures", "undetected"):
        assert c[k] == halves[0][k] + halves[1][k], k
    one = code.awgn_point(eb, frames, "NMS", 0.8, seed=5, point=2, frame0=64)
    assert c["frame_errors"] < 0.8 * one["frame_errors"], (c, one)
    assert c["iterations"] > one["iterations"]


def test_pgz_erasure_rule(ctx, catalogue):
    """ccgpu_gf_decode_erasures_pgz == the reference's primitive_bch<.., pgz_tag>::correct(b, erasures) (bch.h:97-149)
    on the vectors the reference produced (oracle/make_golden_pgz.py); host and device pointers"""
    import torch
    g = load_golden("hard_pgz_erasures.npz")
    for name in ("bch_15_7", "bch_31_16", "bch_63_36", "bch_63_45"):
        code = make_code(ctx, catalogue[name])
        rec, epos, ecnt = g[name + ".received"], g[name + ".epos"], g[name + ".ecnt"]
        out, nerr, failed = code.gf_decode(rec, erasures=(epos, ecnt), pgz_fill=True)
        clean = g[name + ".solver_defect"] == 0   # the reference's PGZ solver malfunctions on a few t = 5 words
        assert np.array_equal(failed[clean], (g[name + ".status"][clean] != 0).astype(np.uint8)), name
        ok = clean & (failed == 0)
        assert np.array_equal(out[ok], g[name + ".corrected"][ok]), name
        assert np.array_equal(out[failed != 0], rec[failed != 0])  # a failed word comes back as received
        # where the solver defect strikes, the engine still returns a codeword within the radius
        bad = ~clean
        assert (failed[bad] == 0).all() and np.array_equal(out[bad], g[name + ".words"][bad])
        dev = code.gf_decode(torch.from_numpy(rec).cuda(), erasures=(torch.from_numpy(epos).cuda(), torch.from_numpy(ecnt).cuda()),
                             pgz_fill=True)
        ctx.sync()
        assert np.array_equal(dev[0].cpu().numpy(), out) and np.array_equal(dev[2].cpu().numpy(), failed)
        assert np.array_equal(dev[1].cpu().numpy(), nerr)
        # no erasures: the plain decoder
        plain = code.gf_decode(rec)
        none = code.gf_decode(rec, erasures=(epos, np.zeros_like(ecnt)), pgz_fill=True)
        assert all(np.array_equal(a, b) for a, b in zip(plain, none))


def test_uncoded_point(ctx):
    """ccgpu_awgn_point_uncoded == hard decisions on the channel kernel's output for the same (seed, point, frames)"""
    import channelcoding_b200 as cc
    for n, eb in ((63, 3.0), (15, 6.0), (200, 5.0)):
        frames = 50000
        c = ctx.awgn_point_uncoded(n, eb, frames, seed=3, point=9, frame0=17)
        y = ctx.awgn_llr(n, np.float32(cc.sigma(0.5, eb)), seed=3, point=9, frame0=17, frames=frames)
        neg = y < 0
        assert c["frames"] == frames and c["bit_errors"] == int(neg.sum()) and c["frame_errors"] == int(neg.any(axis=1).sum())


@pytest.mark.parametrize("name,ebno", [("bch_15_7", 6.0), ("bch_31_16", 6.5), ("bch_63_36", 7.0), ("bch_63_57", 8.0),
                                       ("bch_127_64", 7.5), ("bch_255_131", 8.5)])
def test_all_positive_shortcut_is_exact(ctx, name, ebno, catalogue):
    """frames whose channel values are all positive are decided without executing iteration 0 when the totals L are
    not requested (ms_cyclic.cuh): same bits / iteration index / failure flag as the full path (L requested) and as
    the oracle, for every flavour and stop rule; zeros, infinities and NaNs never take the shortcut wrongly"""
    e = catalogue[name]
    code = make_code(ctx, e)
    n = e["n"]
    rng = np.random.default_rng(zlib.crc32(("quick" + name).encode()))
    frames = 6000 if n < 255 else 1500
    y = (1 + oracle.sigma(e["rate"], ebno) * rng.standard_normal((frames, n))).astype(np.float32)
    y[0] = 1.0
    y[1, 3] = 0.0            # a zero is not positive
    y[2] = np.inf
    y[3, 5] = np.nan
    y[4] = np.float32(1e-45)  # the smallest subnormal is positive
    y[5, n - 1] = -0.0
    allpos = (y > 0).all(axis=1)
    assert 0.2 < allpos.mean() < 0.98   # both kinds of frames are present
    for variant, alpha, beta, mi, stop in (("MS", 1, 0, 50, 0), ("NMS", 0.8, 0, 50, 0), ("OMS", 1, 0.3, 20, 0),
                                           ("SCMS1", 1, 0, 30, 1), ("SCMS2", 1, 0, 50, 0), ("2DNMS", 0.9, 0.8, 25, 1),
                                           ("NMS", 0.8, 0, 1, 0), ("MS", 1, 0, 5, 2)):
        full = code.decode(y, variant, alpha, beta, mi, stop, want_L=True)
        ctx.set_option("quick", 1)   # the QUICK instantiation (normally chosen by ccgpu_awgn_point at high Eb/N0)
        try:
            fast = code.decode(y, variant, alpha, beta, mi, stop, want_L=False)
        finally:
            ctx.set_option("quick", -1)
        assert fast[1] is None
        what = "%s %s stop=%d" % (name, variant, stop)
        assert np.array_equal(fast[0], full[0]) and np.array_equal(fast[2], full[2]) and np.array_equal(fast[3], full[3]), what
        if stop != 2:
            ok = allpos & ~np.isnan(y).any(axis=1)
            assert not fast[0][ok].any() and not fast[2][ok].any() and not fast[3][ok].any(), what
    hi = 1500 if n < 255 else 60
    ob, _, oi, of = oracle.min_sum(code.H(), y[6:hi], "NMS", 0.8, 0.0, 50, 0)   # (the rows with inf / nan left out)
    ctx.set_option("quick", 1)
    try:
        fast = code.decode(y[6:hi], "NMS", 0.8, 0.0, 50, 0, want_L=False)
        c1 = code.awgn_point(ebno, 300000 if n < 255 else 60000, "NMS", 0.8, seed=3, point=1)
        ctx.set_option("quick", 0)
        c0 = code.awgn_point(ebno, 300000 if n < 255 else 60000, "NMS", 0.8, seed=3, point=1)
    finally:
        ctx.set_option("quick", -1)
    assert np.array_equal(fast[0], ob) and np.array_equal(fast[2].astype(np.uint32), oi) and np.array_equal(fast[3], of)
    assert c0 == c1   # fused Monte-Carlo point: identical counters with and without the shortcut


@pytest.mark.parametrize("name", ["bch_31_16", "bch_63_36", "bch_63_45", "bch_127_64", "bch_127_106", "bch_255_131"])
def test_screening_gives_the_same_counters(ctx, name, catalogue):
    """Monte-Carlo points with counters only: the QUICK warp kernel screens frames in passes of 32 / NBLK (ms_cyclic.cuh
    SCREEN), the CTA kernel in groups of four (ms_cyclic_cta.cuh grouped mode); all-positive frames are counted without
    ever reaching the decoder.  The noise is keyed by the frame index, so the eight counters must equal those of the
    frame-at-a-time path (option quick = 0) exactly -- at low, medium and very high Eb/N0, for ragged frame counts (1, a
    few, not a multiple of the pass size), frame offsets, both stop rules and the self-correcting flavour."""
    e = catalogue[name]
    code = make_code(ctx, e)
    big = 200000 if e["n"] < 255 else 40000
    cases = [(4.0, big // 4, "NMS", 0.8, 0.0, 50, 0, 0), (7.0, big, "NMS", 0.8, 0.0, 50, 0, 5), (10.0, 4 * big + 3, "NMS", 0.8, 0.0, 50, 0, 0),
             (12.0, 4 * big + 1, "MS", 1.0, 0.0, 50, 1, 123456789012), (8.0, 1, "NMS", 0.8, 0.0, 50, 0, 7), (8.0, 3, "MS", 1.0, 0.0, 50, 0, 0),
             (8.0, 131, "OMS", 1.0, 0.3, 20, 0, 0), (7.5, big, "SCMS2", 1.0, 0.0, 50, 0, 0), (9.0, big, "2DNMS", 0.9, 0.8, 25, 1, 1),
             (9.0, big, "NMS", 0.8, 0.0, 1, 0, 0), (5.0, big // 4, "NMS_Q", 0.8, 0.0, 50, 0, 0), (9.0, big, "NMS_Q", 0.8, 0.0, 50, 0, 3),
             (12.0, 2 * big + 1, "MS_Q", 1.0, 0.0, 50, 1, 0), (10.0, 5, "NMS_Q", 0.8, 0.0, 50, 0, 0)]
    for ebno, frames, variant, alpha, beta, mi, stop, f0 in cases:
        res = []
        for quick in (1, 0):
            ctx.set_option("quick", quick)
            try:
                res.append(code.awgn_point(ebno, frames, variant, alpha, beta, mi, stop, seed=11, point=3, frame0=f0))
            finally:
                ctx.set_option("quick", -1)
        res.append(code.awgn_point(ebno, frames, variant, alpha, beta, mi, stop, seed=11, point=3, frame0=f0))  # the host's own choice
        what = "%s %s %.1f dB %d frames" % (name, variant, ebno, frames)
        assert res[0] == res[1] == res[2], (what, res)
        assert res[0]["frames"] == frames, what


def test_every_compiled_shape_keeps_the_reference_order(ctx, catalogue):
    """Guard for the ordered column sums (ms_cyclic.cuh VOLCS: program order through volatile shared-memory accesses
    instead of one __syncwarp per tap -- formally a race under independent thread scheduling, in practice decided by
    the SASS ptxas emits).  EVERY catalogue code (each has its own compiled shape) x every flavour: the totals L must
    carry the reference's float32 bit patterns, i.e. the rows were added in ascending order.  The toolkit is pinned
    by tests/test_host_abi.py::test_build_info; a new nvcc has to pass this test before it ships."""
    rng = np.random.default_rng(2024)
    seen = 0
    for name, e in sorted(catalogue.items()):
        if e["family"] != 0:
            continue
        code = make_code(ctx, e)
        assert code.kernel == 1, name
        H = code.H()
        frames = 96 if e["n"] <= 63 else (24 if e["n"] <= 127 else 8)
        y = (1 + oracle.sigma(e["rate"], 3.0) * rng.standard_normal((frames, e["n"]))).astype(np.float32)
        for variant, alpha, beta in (("MS", 1, 0), ("NMS", 0.8, 0), ("OMS", 1, 0.05), ("SCMS1", 1, 0), ("SCMS2", 1, 0),
                                     ("2DNMS", 0.9, 0.8)):
            assert_same(code.decode(y, variant, alpha, beta, 12, 0), oracle.min_sum(H, y, variant, alpha, beta, 12, 0),
                        "%s %s" % (name, variant))
        seen += 1
    assert seen >= 16


@pytest.mark.parametrize("name", ["bch_15_7", "bch_31_16", "bch_63_36", "bch_127_64", "bch_255_131", "bch_63_57"])
def test_packed_output_layout(ctx, name, catalogue):
    """ccgpu_decode_llr_packed (compact layout: ceil(n/32) words of decided bits + one status byte per frame, the
    algorithmic output of SURVEY 8d) carries exactly the information of ccgpu_decode_llr on every kernel: several
    frames per warp, several rows per lane, CTA per frame, the general (CSR) kernel, float and fixed-point flavours,
    host and device buffers"""
    import torch
    e = catalogue[name]
    code = make_code(ctx, e)
    n = e["n"]
    npw = (n + 31) // 32
    rng = np.random.default_rng(zlib.crc32(("packed" + name).encode()))
    frames = 3001 if n <= 63 else (301 if n <= 127 else 61)
    y = (1 + oracle.sigma(e["rate"], 4.0) * rng.standard_normal((frames, n))).astype(np.float32)
    y[0] = -1.0   # all-one word
    y[1, ::2] = -1.0
    codes = [code]
    if n == 63 and name == "bch_63_36":
        codes.append(ctx.from_dense(code.H()[rng.permutation(code.h_rows)], e["rate"]))  # CSR kernel
    quant = (8.0, 31, 29 if n == 255 else 31)
    for c in codes:
        for variant, alpha, mi, stop in (("NMS", 0.8, 50, 0), ("MS", 1.0, 7, 1), ("SCMS2", 1.0, 20, 2), ("NMS_Q", 0.8, 50, 0),
                                         ("MS_Q", 1.0, 6, 1)):
            if variant.endswith("_Q") and c.kernel != 1:
                continue
            q = quant if variant.endswith("_Q") else None
            bits, _, it, failed = c.decode(y, variant, alpha, 0.0, mi, stop, want_L=False, quant=q)
            packed, status = c.decode_packed(y, variant, alpha, 0.0, mi, stop, quant=q)
            assert packed.shape == (frames, npw) and packed.dtype == np.uint32
            unpacked = ((packed[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(frames, npw * 32).astype(np.uint8)
            what = "%s %s kernel %d" % (name, variant, c.kernel)
            assert np.array_equal(unpacked[:, :n], bits), what
            assert not unpacked[:, n:].any(), what + ": unused bits must be zero"
            assert np.array_equal(status, np.where(failed == 1, 255, it).astype(np.uint8)), what
            if c is code and variant in ("NMS", "NMS_Q"):
                yt = torch.from_numpy(y).cuda()
                pk, st = c.decode_packed(yt, variant, alpha, 0.0, mi, stop, quant=q)
                ctx.sync()
                assert np.array_equal(pk.cpu().numpy().view(np.uint32), packed) and np.array_equal(st.cpu().numpy(), status), what
