"""The host plumbing every entry point shares: where the Monte-Carlo counters go, and which mixes of host and device
buffers are refused.

* Counter accumulation: each of the six counter entry points, called through the C ABI with a device `out` that
  already holds values, adds exactly what the same call returns into a host `out`; the two reserved slots are left
  alone.  A device `out` is how the multi-GPU group sums its members, so a zeroing or overwrite there loses frames.
* Mixed residency: a device input with any output (or erasure input) in host memory is refused with ERR_INVALID, not
  decoded into the wrong address space; Chase-II refuses the reverse mix as well."""
import ctypes as C

import numpy as np
import pytest

gpu = pytest.mark.gpu

FIELDS = ("frames", "frame_errors", "bit_errors", "iterations", "failures", "undetected")
PREFILL = [101, 202, 303, 404, 505, 606, 707, 808]  # distinct, non-zero, all eight slots including the reserved two


@pytest.fixture(scope="module")
def ctx():
    import channelcoding_b200 as cc
    c = cc.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def bch(ctx):
    return ctx.bch(6, errors=5)  # BCH(63,36)


def counter_calls(ctx, code):
    """name -> fn(out pointer) -> return code of one call of that entry point, fixed arguments"""
    from channelcoding_b200 import _lib
    from channelcoding_b200.engine import ms_params
    L, h, c = _lib.lib(), ctx._h, code._h
    p = ms_params("NMS", 0.8)
    shifts = np.array([0, 9, 21], np.uint32)
    return {
        "awgn_point": lambda out: L.ccgpu_awgn_point(h, c, C.byref(p), 3.5, 7, 1, 100, 20000, out),
        "bitflip_point": lambda out: L.ccgpu_bitflip_point(h, c, C.byref(p), 4, 1000, 20000, out),
        "awgn_point_mbbp": lambda out: L.ccgpu_awgn_point_mbbp(h, c, C.byref(p), shifts.ctypes.data, len(shifts), 3.5, 7, 1,
                                                               100, 5000, out),
        "awgn_point_uncoded": lambda out: L.ccgpu_awgn_point_uncoded(h, code.n, code.rate, 3.5, 7, 1, 100, 20000, out),
        "awgn_point_hard": lambda out: L.ccgpu_awgn_point_hard(h, c, 5.0, 7, 1, 100, 20000, out),
        "awgn_point_chase": lambda out: L.ccgpu_awgn_point_chase(h, c, 3, 5.0, 7, 1, 100, 20000, out),
    }


@gpu
@pytest.mark.parametrize("name", ["awgn_point", "bitflip_point", "awgn_point_mbbp", "awgn_point_uncoded",
                                  "awgn_point_hard", "awgn_point_chase"])
def test_device_counters_accumulate(ctx, bch, name):
    import torch
    from channelcoding_b200._lib import Counters
    fn = counter_calls(ctx, bch)[name]
    host = Counters()
    ctx._check(fn(C.addressof(host)))
    want = host.as_dict()
    assert want["frames"] > 0
    dev = torch.tensor(PREFILL, dtype=torch.int64, device="cuda:0")
    ctx._follow_torch(dev)
    ctx._check(fn(dev.data_ptr()))
    torch.cuda.synchronize()
    assert dev.cpu().tolist() == [PREFILL[i] + want[k] for i, k in enumerate(FIELDS)] + PREFILL[6:]


def one_on_host(out):
    """every variant of the all-device tuple `out` with one of its tensors moved to host memory"""
    for i, t in enumerate(out):
        if t is not None:
            yield i, tuple(t.cpu().numpy() if j == i else u for j, u in enumerate(out))


def assert_refused(call, what):
    from channelcoding_b200 import CcgpuError
    from channelcoding_b200._lib import ERR_INVALID
    with pytest.raises(CcgpuError) as e:
        call()
    assert e.value.code == ERR_INVALID, what
    assert "device pointer" in str(e.value), (what, str(e.value))


@gpu
def test_mixed_residency_refused(ctx, bch):
    import torch
    frames, n = 64, bch.n
    dev = lambda shape, dt: torch.zeros(shape, dtype=dt, device="cuda:0")  # noqa: E731
    y = torch.ones((frames, n), dtype=torch.float32, device="cuda:0")
    u8 = torch.uint8
    shifts = [0, 9, 21]
    cases = [
        ("decode", lambda o: bch.decode(y, "NMS", 0.8, out=o),
         (dev((frames, n), u8), dev((frames, n), torch.float32), dev(frames, u8), dev(frames, u8))),
        ("decode_packed", lambda o: bch.decode_packed(y, "NMS", 0.8, out=o),
         (dev((frames, (n + 31) // 32), torch.int32), dev(frames, u8))),
        ("decode_mbbp", lambda o: bch.decode_mbbp(y, shifts, "NMS", 0.8, out=o),
         (dev((frames, n), u8), dev((frames, n), torch.float32), dev(frames, u8), dev(frames, u8), dev(frames, u8))),
        ("decode_chase", lambda o: bch.decode_chase(y, 3, out=o), (dev((frames, n), u8), dev(frames, u8), dev(frames, u8))),
    ]
    words = dev((frames, n), u8)
    epos, ecnt = dev((frames, 4), u8), dev(frames, u8)
    gf_out = (dev((frames, n), u8), dev(frames, u8), dev(frames, u8))
    cases.append(("gf_decode", lambda o: bch.gf_decode(words, out=o), gf_out))
    for pgz in (False, True):
        cases.append(("gf_decode(erasures, pgz_fill=%s)" % pgz,
                      lambda o, pgz=pgz: bch.gf_decode(words, out=o, erasures=(epos, ecnt), pgz_fill=pgz), gf_out))
    for what, call, out in cases:
        call(out)  # all on the device: accepted
        for i, o in one_on_host(out):
            assert_refused(lambda: call(o), "%s, output %d on the host" % (what, i))
    # the erasure inputs must follow the words too (through the ABI: Code.gf_decode takes them both from one side)
    from channelcoding_b200 import _lib
    from channelcoding_b200.engine import _ptr
    ctx._follow_torch(words)
    for fn in (_lib.lib().ccgpu_gf_decode_erasures, _lib.lib().ccgpu_gf_decode_erasures_pgz):
        for i, (ep, ec) in one_on_host((epos, ecnt)):
            assert_refused(lambda: ctx._check(fn(ctx._h, bch._h, _ptr(words), frames, _ptr(ep), _ptr(ec), 4,
                                                 *(_ptr(t) for t in gf_out))),
                           "%s, erasure input %d on the host" % (fn.__name__, i))
    # Chase-II refuses the reverse mix too: channel values on the host, one output on the device
    host_out = (np.zeros((frames, n), np.uint8), np.zeros(frames, np.uint8), np.zeros(frames, np.uint8))
    for i in range(3):
        o = tuple(torch.from_numpy(t).cuda() if j == i else t for j, t in enumerate(host_out))
        assert_refused(lambda: bch.decode_chase(y.cpu().numpy(), 3, out=o), "decode_chase, host y, output %d on the device" % i)
    torch.cuda.synchronize()
