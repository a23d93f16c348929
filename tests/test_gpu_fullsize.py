"""Full-size runs of the BASELINE.json configurations, checked through size-independent properties
(the per-frame outputs at the benchmarked batch sizes are checked against the oracle in tests/test_gpu_scale.py):
shard-sum linearity of the counters, statistical agreement with a small oracle-checked run, all-zero-codeword round
trips for the linear RS code."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    import channelcoding_b200 as cc
    c = cc.Context(0)
    yield c
    c.close()


def test_bch_63_36_point_of_1e8_frames(ctx):
    """config[1]: BCH(63,36) NMS, 50 iterations, early exit, 1e8 frames at one Eb/N0 point"""
    code = ctx.bch(6, errors=5)
    total = 100_000_000
    whole = code.awgn_point(4.0, total, "NMS", 0.8, seed=3, point=8)
    assert whole["frames"] == total and whole["undetected"] == 0
    assert whole["failures"] <= whole["frame_errors"] <= whole["bit_errors"]
    assert whole["frames"] <= whole["iterations"] <= 50 * total
    # sharding by frame range (what 8 GPUs do) gives exactly the same totals
    parts = [code.awgn_point(4.0, total // 8, "NMS", 0.8, seed=3, point=8, frame0=i * (total // 8)) for i in range(8)]
    for k in whole:
        assert sum(p[k] for p in parts) == whole[k], k
    # the word error rate agrees with an independent seed within the 99.9 % interval of the difference
    other = code.awgn_point(4.0, 4_000_000, "NMS", 0.8, seed=4, point=8)
    p1, p2 = whole["frame_errors"] / total, other["frame_errors"] / other["frames"]
    se = math.sqrt(p1 * (1 - p1) / total + p2 * (1 - p2) / other["frames"])
    assert abs(p1 - p2) < 3.3 * se
    assert abs(p1 - 0.1803) < 0.002  # SURVEY 6.2: 0.181 with the reference's own noise source


def test_bch_255_131_waterfall_tail(ctx):
    """config[4]: BCH(255,131) towards the error floor: 2e8 frames at 8.5 dB in shards, every shard must
    account for all its frames; failures are rare and every one of them is a frame error"""
    code = ctx.bch(8, errors=18)
    shards = [code.awgn_point(8.5, 25_000_000, "NMS", 0.8, seed=1, point=17, frame0=i * 25_000_000) for i in range(8)]
    frames = sum(s["frames"] for s in shards)
    ferr = sum(s["frame_errors"] for s in shards)
    assert frames == 200_000_000
    assert 0 < ferr / frames < 5e-3
    assert all(s["failures"] <= s["frame_errors"] for s in shards)
    assert sum(s["iterations"] for s in shards) / frames < 3.0


def test_rs_255_223_ten_million_words(ctx):
    """config[3]: 1e7 RS(255,223) words.  The code is linear, so the all-zero codeword with e <= 16 symbol
    errors must come back as all-zero with n_errors = e, and e = 17 .. 20 must be reported as failures or
    (rarely) miscorrected to another codeword at distance <= 16 from the received word"""
    import torch
    code = ctx.rs(8, 16)
    count = 10_000_000
    g = torch.Generator(device="cuda").manual_seed(5)
    words = torch.zeros((count, 255), dtype=torch.uint8, device="cuda")
    ne = torch.randint(0, 21, (count,), device="cuda", generator=g)
    # positions: a random permutation prefix per word would be costly; draw e distinct positions by rejection-free
    # striding: start + i * step (mod 255) with step coprime to 255
    start = torch.randint(0, 255, (count,), device="cuda", generator=g)
    step = torch.tensor([1, 2, 4, 7, 8, 11, 13, 14], device="cuda")[torch.randint(0, 8, (count,), device="cuda", generator=g)]
    for i in range(20):
        sel = ne > i
        pos = (start + i * step) % 255
        val = torch.randint(1, 256, (count,), device="cuda", generator=g).to(torch.uint8)
        idx = torch.nonzero(sel).squeeze(1)
        words[idx, pos[idx]] = val[idx]
    torch.cuda.synchronize()
    out, nerr, failed = code.gf_decode(words)
    ctx.sync()
    ok = ne <= 16
    assert not failed[ok].any()
    assert not out[ok].any()
    assert torch.equal(nerr[ok].to(torch.int64), ne[ok])
    beyond = ~ok
    fb = failed[beyond].to(torch.bool)
    assert fb.float().mean() > 0.99                      # miscorrection probability is about 1/16! per word
    assert torch.equal(out[beyond][fb], words[beyond][fb])  # failed words are returned unchanged
    mis = beyond.nonzero().squeeze(1)[~fb]
    if mis.numel():
        assert ((out[mis] != words[mis]).sum(dim=1) <= 16).all()


def test_bch_15_7_sweep_monotone(ctx):
    """config[0]: BCH(15,7) over 1 .. 6 dB, min-sum and sum-product (LLR-scaled input): both curves fall
    monotonically and stay close to each other (on this dense parity-check matrix the tanh rule is slightly
    WORSE than min-sum, 0.210 vs 0.176 at 1 dB -- short cycles make it over-confident)"""
    code = ctx.bch(4, errors=2)
    prev = {"MS": 1.0, "SPA": 1.0}
    for i, eb in enumerate(np.arange(1.0, 6.01, 0.5)):
        ms = code.awgn_point(eb, 4_000_000, "MS", seed=2, point=i)
        spa = code.awgn_point(eb, 4_000_000, "SPA", seed=2, point=i, stop_rule=1)
        wer = ms["frame_errors"] / ms["frames"]
        wer_spa = spa["frame_errors"] / spa["frames"]
        assert wer < prev["MS"] * 1.02 and wer_spa < prev["SPA"] * 1.02
        assert 0.8 * wer < wer_spa < 1.3 * wer + 1e-5, (eb, wer_spa, wer)
        prev["MS"], prev["SPA"] = wer, wer_spa
    assert prev["MS"] < 1e-3 and prev["SPA"] < 1e-3


def test_bch_15_7_full_size_on_the_lane_kernel(ctx):
    """config[0] at full size on the lane-per-frame kernel: 2e8 frames per point.  Shard-sum linearity of every counter
    (what 8 GPUs do), equality with the warp kernel on a 2e7-frame slice, and the word error rate inside the 99.9 %
    interval of the reference's own CPU simulation (tests/golden/ref_wer.json, 1e5 frames per point)."""
    import json
    import os
    code = ctx.bch(4, errors=2)
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_wer.json")) as f:
        golden = json.load(f)
    total = 200_000_000
    for point, eb in enumerate((1.0, 3.0, 5.0)):
        whole = code.awgn_point(eb, total, "MS", seed=5, point=point)
        assert whole["frames"] == total and whole["failures"] <= whole["frame_errors"] <= whole["bit_errors"]
        assert whole["frames"] <= whole["iterations"] <= 50 * total
        parts = [code.awgn_point(eb, total // 8, "MS", seed=5, point=point, frame0=i * (total // 8)) for i in range(8)]
        for k in whole:
            assert sum(p[k] for p in parts) == whole[k], (eb, k)
        ctx.set_option("lane", 0)
        try:
            warp = code.awgn_point(eb, total // 10, "MS", seed=5, point=point, frame0=3 * (total // 10))
        finally:
            ctx.set_option("lane", -1)
        assert warp == code.awgn_point(eb, total // 10, "MS", seed=5, point=point, frame0=3 * (total // 10)), eb
        ref = [r for r in golden["points"] if r["code"] == "bch_15_7" and abs(r["ebno_db"] - eb) < 1e-9 and r["variant"] == "MS"]
        if ref:
            p1, n2 = whole["frame_errors"] / total, ref[0]["frames"]
            p2 = ref[0]["word_errors"] / n2
            assert abs(p1 - p2) < 3.3 * math.sqrt(p1 * (1 - p1) / total + p2 * (1 - p2) / n2 + 1e-12), (eb, p1, p2)


def test_bch_63_36_error_floor_with_screening(ctx):
    """config[1] towards the error floor: 2e9 frames at 10 dB (98 % of them are counted by the screening without reaching
    the decoder).  Every shard accounts for all its frames, the counters add up, one iteration per clean frame."""
    code = ctx.bch(6, errors=5)
    shard = 250_000_000
    shards = [code.awgn_point(10.0, shard, "NMS", 0.8, seed=9, point=20, frame0=i * shard) for i in range(8)]
    frames = sum(s["frames"] for s in shards)
    assert frames == 8 * shard and all(s["frames"] == shard for s in shards)
    ferr = sum(s["frame_errors"] for s in shards)
    assert ferr / frames < 2e-7 and all(s["failures"] <= s["frame_errors"] <= s["bit_errors"] for s in shards)
    it = sum(s["iterations"] for s in shards) / frames
    assert 1.0 <= it < 1.002
    ctx.set_option("quick", 0)
    try:
        plain = code.awgn_point(10.0, 20_000_000, "NMS", 0.8, seed=9, point=20, frame0=3 * shard)
    finally:
        ctx.set_option("quick", -1)
    assert plain == code.awgn_point(10.0, 20_000_000, "NMS", 0.8, seed=9, point=20, frame0=3 * shard)
