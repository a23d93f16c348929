"""Thin object layer over the C ABI (include/ccgpu.h): Context (one CUDA device + stream) and Code
(a BCH / RS code or a dense parity-check matrix uploaded to the device).

Array arguments may be numpy arrays (host path: staged through the library, call returns when the
results are in the output arrays) or torch CUDA tensors (device path: enqueued on the context's
stream, no synchronisation)."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import CcgpuError, CodeInfo, Counters, MsParams

VARIANTS = {"MS": 0, "NMS": 1, "OMS": 2, "SCMS1": 3, "SCMS2": 4, "2DNMS": 5, "SPA": 6, "MS_Q": 7, "NMS_Q": 8, "OMS_Q": 9}
STOP_REF_ZERO_OVERLAP, STOP_GF2_PARITY, STOP_NONE = 0, 1, 2
CAP_ERRORS, CAP_DMIN = 0, 1


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _ptr(x):
    if x is None:
        return None
    if _is_torch(x):
        assert x.is_contiguous()
        return x.data_ptr()
    assert x.flags["C_CONTIGUOUS"]
    return x.ctypes.data


def ms_params(variant="MS", alpha=1.0, beta=0.0, max_iter=50, stop_rule=STOP_REF_ZERO_OVERLAP, quant=None):
    """quant: (q_scale, q_y_max, q_msg_max) of the fixed-point variants MS_Q / NMS_Q / OMS_Q; None = the defaults (8, 31, 31)"""
    v = VARIANTS[variant] if isinstance(variant, str) else int(variant)
    qs, qy, qm = quant if quant is not None else (0.0, 0, 0)
    return MsParams(v, int(stop_rule), int(max_iter), int(qm), float(alpha), float(beta), float(qs), int(qy), 0)


def _check(ctx, rc):
    if rc != 0:
        if ctx is not None:
            ctx._check(rc)
        raise CcgpuError(rc, "call failed (host-only code)")


def host_bch(q, errors=None, dmin=None):
    """host-only description of cyclic::primitive_bch<q, ..> (no CUDA device needed, no decoding)"""
    assert (errors is None) != (dmin is None)
    h = C.c_void_p()
    kind, val = (CAP_ERRORS, errors) if errors is not None else (CAP_DMIN, dmin)
    _check(None, _lib.lib().ccgpu_bch_create(None, q, kind, val, C.byref(h)))
    return Code(None, h)


def host_rs(q, errors, mu=1, step=1):
    h = C.c_void_p()
    _check(None, _lib.lib().ccgpu_rs_create(None, q, errors, mu, step, C.byref(h)))
    return Code(None, h)


def host_from_dense(H, rate):
    H = np.ascontiguousarray(H, np.uint8)
    h = C.c_void_p()
    _check(None, _lib.lib().ccgpu_code_from_dense(None, H.ctypes.data, H.shape[0], H.shape[1], float(rate), C.byref(h)))
    return Code(None, h)


class Context:
    def __init__(self, device=0):
        self._h = C.c_void_p()
        rc = _lib.lib().ccgpu_create(int(device), C.byref(self._h))
        if rc != 0:
            raise CcgpuError(rc, "ccgpu_create(device=%d) failed -- no usable CUDA device; there is no CPU "
                                 "fallback" % device)
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().ccgpu_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise CcgpuError(rc, _lib.lib().ccgpu_last_error(self._h).decode())

    def set_stream(self, cuda_stream_ptr):
        self._check(_lib.lib().ccgpu_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def use_torch_stream(self):
        import torch
        self.set_stream(torch.cuda.current_stream(self.device).cuda_stream)

    def set_option(self, name, value):
        """tuning overrides (ccgpu_set_option): "quick" -1 / 0 / 1, "work_batch" n"""
        self._check(_lib.lib().ccgpu_set_option(self._h, name.encode(), int(value)))

    def _follow_torch(self, *tensors):
        """Work on torch tensors must be ordered with torch's own work on them (allocation, fills, frees): run on
        torch's CURRENT stream of this device.  The context's private stream is non-blocking, so it orders with
        nothing torch does; a zero-fill issued by torch could land after the kernel's atomics."""
        if any(t is not None and _is_torch(t) for t in tensors):
            import torch
            cur = torch.cuda.current_stream(self.device).cuda_stream
            if _lib.lib().ccgpu_get_stream(self._h) != cur:
                self.set_stream(cur)

    def sync(self):
        self._check(_lib.lib().ccgpu_sync(self._h))

    @property
    def kernel_launches(self):
        return int(_lib.lib().ccgpu_kernel_launches(self._h))

    # ---- codes
    def bch(self, q, errors=None, dmin=None):
        """cyclic::primitive_bch<q, errors<e>> / <q, dmin<d>> (codes/bch.h:16-161)"""
        assert (errors is None) != (dmin is None)
        h = C.c_void_p()
        kind, val = (CAP_ERRORS, errors) if errors is not None else (CAP_DMIN, dmin)
        self._check(_lib.lib().ccgpu_bch_create(self._h, q, kind, val, C.byref(h)))
        return Code(self, h)

    def rs(self, q, errors, mu=1, step=1):
        """cyclic::rs<q, errors<e>, .., mu, step> (codes/rs.h:6-94)"""
        h = C.c_void_p()
        self._check(_lib.lib().ccgpu_rs_create(self._h, q, errors, mu, step, C.byref(h)))
        return Code(self, h)

    def from_dense(self, H, rate):
        H = np.ascontiguousarray(H, np.uint8)
        h = C.c_void_p()
        self._check(_lib.lib().ccgpu_code_from_dense(self._h, H.ctypes.data, H.shape[0], H.shape[1], float(rate),
                                                     C.byref(h)))
        return Code(self, h)

    # ---- channel
    def awgn_point_uncoded(self, n, ebno_db, frames, rate=0.5, seed=0, point=0, frame0=0):
        """one Eb/N0 point over the reference's `uncoded` pseudo-decoder (codes/uncoded.h) -> counters"""
        c = Counters()
        self._check(_lib.lib().ccgpu_awgn_point_uncoded(self._h, n, float(rate), float(ebno_db), seed, point, frame0, frames,
                                                        C.addressof(c)))
        return c.as_dict()

    def awgn_llr(self, n, sigma, seed, point, frame0, frames, out=None):
        if out is None:
            out = np.empty((frames, n), np.float32)
        self._follow_torch(out)
        self._check(_lib.lib().ccgpu_awgn_llr(self._h, n, float(sigma), seed, point, frame0, frames, _ptr(out)))
        return out


class Code:
    def __init__(self, ctx, handle):
        self.ctx = ctx
        self._h = handle
        self._refresh()

    def _refresh(self):
        info = CodeInfo()
        _check(self.ctx, _lib.lib().ccgpu_code_get_info(self._h, C.byref(info)))
        for k, _ in CodeInfo._fields_:
            setattr(self, k, getattr(info, k))

    def close(self):
        if getattr(self, "_h", None) and (self.ctx is None or getattr(self.ctx, "_h", None)):
            _lib.lib().ccgpu_code_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def to_string(self, tag):
        buf = C.create_string_buffer(128)
        _check(self.ctx, _lib.lib().ccgpu_code_to_string(self._h, tag.encode(), buf, 128))
        return buf.value.decode()

    def H(self):
        out = np.zeros((self.h_rows, self.n), np.uint8)
        _check(self.ctx, _lib.lib().ccgpu_code_H(self._h, out.ctypes.data))
        return out

    def H_alt(self, as_reference=False):
        """cyclic::H_alt<T>() (cyclic.h:361-385); as_reference reproduces the reference's exponent bug"""
        rows = C.c_uint32()
        _check(self.ctx, _lib.lib().ccgpu_code_H_alt(self._h, int(as_reference), None, C.byref(rows)))
        out = np.zeros((rows.value, self.n), np.uint8)
        _check(self.ctx, _lib.lib().ccgpu_code_H_alt(self._h, int(as_reference), out.ctypes.data, C.byref(rows)))
        return out

    def poly(self, which):
        out = np.zeros(1024, np.uint16)
        m = _lib.lib().ccgpu_code_poly(self._h, {"g": 0, "h": 1}[which], out.ctypes.data, 1024)
        if m < 0:
            raise CcgpuError(m, "ccgpu_code_poly")
        return out[:m].copy()

    def set_rows(self, rows):
        _check(self.ctx, _lib.lib().ccgpu_code_set_rows(self._h, rows))
        self._refresh()

    def encode(self, msgs):
        msgs = np.ascontiguousarray(msgs, np.uint8).reshape(-1, self.l)
        words = np.zeros((msgs.shape[0], self.n), np.uint8)
        _check(self.ctx, _lib.lib().ccgpu_encode(self._h, msgs.ctypes.data, msgs.shape[0], words.ctypes.data))
        return words

    # ---- decoding
    def decode(self, y, variant="MS", alpha=1.0, beta=0.0, max_iter=50, stop_rule=STOP_REF_ZERO_OVERLAP, want_L=True,
               out=None, quant=None):
        """min_sum<float,uint8_t>(H, y, Tag{}) per frame -> bits, L, iter, failed (ccgpu_decode_llr)"""
        p = ms_params(variant, alpha, beta, max_iter, stop_rule, quant)
        if _is_torch(y):
            import torch
            y = y.contiguous().view(-1, self.n)
            frames = y.shape[0]
            if out is None:
                bits = torch.empty((frames, self.n), dtype=torch.uint8, device=y.device)
                L = torch.empty((frames, self.n), dtype=torch.float32, device=y.device) if want_L else None
                it = torch.empty(frames, dtype=torch.uint8, device=y.device)
                failed = torch.empty(frames, dtype=torch.uint8, device=y.device)
            else:
                bits, L, it, failed = out
        else:
            y = np.ascontiguousarray(y, np.float32).reshape(-1, self.n)
            frames = y.shape[0]
            if out is None:
                bits = np.empty((frames, self.n), np.uint8)
                L = np.empty((frames, self.n), np.float32) if want_L else None
                it = np.empty(frames, np.uint8)
                failed = np.empty(frames, np.uint8)
            else:
                bits, L, it, failed = out
        self.ctx._follow_torch(y, bits)
        self.ctx._check(_lib.lib().ccgpu_decode_llr(self.ctx._h, self._h, C.byref(p), _ptr(y), frames, _ptr(bits),
                                                    _ptr(L), _ptr(it), _ptr(failed)))
        return bits, L, it, failed

    def decode_packed(self, y, variant="MS", alpha=1.0, beta=0.0, max_iter=50, stop_rule=STOP_REF_ZERO_OVERLAP, out=None,
                      quant=None):
        """ccgpu_decode_llr_packed: compact outputs -> packed (frames, ceil(n/32)) uint32, status (frames,) uint8
        [iteration index, 255 = failure]; numpy or torch like decode()"""
        p = ms_params(variant, alpha, beta, max_iter, stop_rule, quant)
        npw = (self.n + 31) // 32
        if _is_torch(y):
            import torch
            y = y.contiguous().view(-1, self.n)
            frames = y.shape[0]
            packed, status = out if out is not None else (torch.empty((frames, npw), dtype=torch.int32, device=y.device),
                                                          torch.empty(frames, dtype=torch.uint8, device=y.device))
        else:
            y = np.ascontiguousarray(y, np.float32).reshape(-1, self.n)
            frames = y.shape[0]
            packed, status = out if out is not None else (np.empty((frames, npw), np.uint32), np.empty(frames, np.uint8))
        self.ctx._follow_torch(y, packed)
        self.ctx._check(_lib.lib().ccgpu_decode_llr_packed(self.ctx._h, self._h, C.byref(p), _ptr(y), frames, _ptr(packed),
                                                           _ptr(status)))
        return packed, status

    def awgn_point(self, ebno_db, frames, variant="MS", alpha=1.0, beta=0.0, max_iter=50,
                   stop_rule=STOP_REF_ZERO_OVERLAP, seed=0, point=0, frame0=0, out=None, quant=None):
        """one Eb/N0 point of awgn_simulation (simulation.c++:112-149), fused on the GPU -> counters.
        out: optional torch uint64/int64 CUDA tensor of 8 slots that is accumulated into (no sync)."""
        p = ms_params(variant, alpha, beta, max_iter, stop_rule, quant)
        if out is not None:
            self.ctx._follow_torch(out)
            self.ctx._check(_lib.lib().ccgpu_awgn_point(self.ctx._h, self._h, C.byref(p), float(ebno_db), seed, point,
                                                        frame0, frames, _ptr(out)))
            return out
        c = Counters()
        self.ctx._check(_lib.lib().ccgpu_awgn_point(self.ctx._h, self._h, C.byref(p), float(ebno_db), seed, point,
                                                    frame0, frames, C.addressof(c)))
        return c.as_dict()

    def decode_mbbp(self, y, shifts, variant="MS", alpha=1.0, beta=0.0, max_iter=50, stop_rule=STOP_REF_ZERO_OVERLAP,
                    want_L=True, out=None):
        """multiple-bases decoding (extension, ccgpu_decode_llr_mbbp): every frame is decoded once per rotation in
        `shifts`, the best converged candidate is returned -> bits, L, iter, failed, chosen.
        out: optional (bits, L, iter, failed, chosen) buffers like decode()'s; L, iter and chosen may be None"""
        p = ms_params(variant, alpha, beta, max_iter, stop_rule)
        sh = np.ascontiguousarray(shifts, np.uint32)
        if _is_torch(y):
            import torch
            y = y.contiguous().view(-1, self.n)
            frames = y.shape[0]
            if out is None:
                mk = lambda shape, dt: torch.empty(shape, dtype=dt, device=y.device)  # noqa: E731
                bits, it, failed, chosen = mk((frames, self.n), torch.uint8), mk(frames, torch.uint8), mk(frames, torch.uint8), mk(frames, torch.uint8)
                L = mk((frames, self.n), torch.float32) if want_L else None
            else:
                bits, L, it, failed, chosen = out
        else:
            y = np.ascontiguousarray(y, np.float32).reshape(-1, self.n)
            frames = y.shape[0]
            if out is None:
                bits, it, failed, chosen = (np.empty((frames, self.n), np.uint8), np.empty(frames, np.uint8),
                                            np.empty(frames, np.uint8), np.empty(frames, np.uint8))
                L = np.empty((frames, self.n), np.float32) if want_L else None
            else:
                bits, L, it, failed, chosen = out
        self.ctx._follow_torch(y, bits)
        self.ctx._check(_lib.lib().ccgpu_decode_llr_mbbp(self.ctx._h, self._h, C.byref(p), sh.ctypes.data, len(sh), _ptr(y),
                                                         frames, _ptr(bits), _ptr(L), _ptr(it), _ptr(failed), _ptr(chosen)))
        return bits, L, it, failed, chosen

    def awgn_point_mbbp(self, ebno_db, frames, shifts, variant="MS", alpha=1.0, beta=0.0, max_iter=50,
                        stop_rule=STOP_REF_ZERO_OVERLAP, seed=0, point=0, frame0=0):
        """one Eb/N0 point decoded with multiple bases (ccgpu_awgn_point_mbbp) -> counters"""
        p = ms_params(variant, alpha, beta, max_iter, stop_rule)
        sh = np.ascontiguousarray(shifts, np.uint32)
        c = Counters()
        self.ctx._check(_lib.lib().ccgpu_awgn_point_mbbp(self.ctx._h, self._h, C.byref(p), sh.ctypes.data, len(sh),
                                                         float(ebno_db), seed, point, frame0, frames, C.addressof(c)))
        return c.as_dict()

    def awgn_point_hard(self, ebno_db, frames, seed=0, point=0, frame0=0):
        """one Eb/N0 point with hard decisions + algebraic decoding (the BM/PGZ/Euklid decoders in the sweep)"""
        c = Counters()
        self.ctx._check(_lib.lib().ccgpu_awgn_point_hard(self.ctx._h, self._h, float(ebno_db), seed, point, frame0, frames,
                                                         C.addressof(c)))
        return c.as_dict()

    def decode_chase(self, y, p, out=None):
        """Chase-II with the p least reliable positions (extension, ccgpu_decode_llr_chase; binary BCH codes,
        0 <= p <= 8) -> bits (frames, n) uint8, failed (frames,) uint8, chosen (frames,) uint8 [index of the returned
        test pattern]; numpy or torch CUDA tensors like decode()"""
        if _is_torch(y):
            import torch
            y = y.contiguous().view(-1, self.n)
            frames = y.shape[0]
            if out is None:
                out = (torch.empty((frames, self.n), dtype=torch.uint8, device=y.device),
                       torch.empty(frames, dtype=torch.uint8, device=y.device),
                       torch.empty(frames, dtype=torch.uint8, device=y.device))
        else:
            y = np.ascontiguousarray(y, np.float32).reshape(-1, self.n)
            frames = y.shape[0]
            if out is None:
                out = (np.empty((frames, self.n), np.uint8), np.empty(frames, np.uint8), np.empty(frames, np.uint8))
        bits, failed, chosen = out
        self.ctx._follow_torch(y, bits)
        self.ctx._check(_lib.lib().ccgpu_decode_llr_chase(self.ctx._h, self._h, int(p), _ptr(y), frames, _ptr(bits),
                                                          _ptr(failed), _ptr(chosen)))
        return bits, failed, chosen

    def awgn_point_chase(self, ebno_db, frames, p, seed=0, point=0, frame0=0, out=None):
        """one Eb/N0 point decoded with Chase-II on the GPU (ccgpu_awgn_point_chase) -> counters.
        out: optional torch uint64/int64 CUDA tensor of 8 slots that is accumulated into (no sync)."""
        if out is not None:
            self.ctx._follow_torch(out)
            self.ctx._check(_lib.lib().ccgpu_awgn_point_chase(self.ctx._h, self._h, int(p), float(ebno_db), seed, point, frame0,
                                                              frames, _ptr(out)))
            return out
        c = Counters()
        self.ctx._check(_lib.lib().ccgpu_awgn_point_chase(self.ctx._h, self._h, int(p), float(ebno_db), seed, point, frame0,
                                                          frames, C.addressof(c)))
        return c.as_dict()

    def decode_osd(self, y, order, out=None):
        """ordered-statistics decoding of order 0..3 (extension, ccgpu_decode_llr_osd; binary BCH codes with n <= 127,
        n - l <= 64) -> bits (frames, n) uint8, weight (frames,) uint8 [number of information positions the returned
        codeword flips]; numpy or torch CUDA tensors like decode()"""
        if _is_torch(y):
            import torch
            y = y.contiguous().view(-1, self.n)
            frames = y.shape[0]
            if out is None:
                out = (torch.empty((frames, self.n), dtype=torch.uint8, device=y.device),
                       torch.empty(frames, dtype=torch.uint8, device=y.device))
        else:
            y = np.ascontiguousarray(y, np.float32).reshape(-1, self.n)
            frames = y.shape[0]
            if out is None:
                out = (np.empty((frames, self.n), np.uint8), np.empty(frames, np.uint8))
        bits, weight = out
        self.ctx._follow_torch(y, bits)
        self.ctx._check(_lib.lib().ccgpu_decode_llr_osd(self.ctx._h, self._h, int(order), _ptr(y), frames, _ptr(bits),
                                                        _ptr(weight)))
        return bits, weight

    def awgn_point_osd(self, ebno_db, frames, order, seed=0, point=0, frame0=0, out=None):
        """one Eb/N0 point decoded with OSD of the given order on the GPU (ccgpu_awgn_point_osd) -> counters.
        out: optional torch uint64/int64 CUDA tensor of 8 slots that is accumulated into (no sync)."""
        if out is not None:
            self.ctx._follow_torch(out)
            self.ctx._check(_lib.lib().ccgpu_awgn_point_osd(self.ctx._h, self._h, int(order), float(ebno_db), seed, point,
                                                            frame0, frames, _ptr(out)))
            return out
        c = Counters()
        self.ctx._check(_lib.lib().ccgpu_awgn_point_osd(self.ctx._h, self._h, int(order), float(ebno_db), seed, point, frame0,
                                                        frames, C.addressof(c)))
        return c.as_dict()

    def decode_gmd(self, y, max_erasures, out=None):
        """GMD decoding of a Reed-Solomon code from the channel values of its binary image (extension,
        ccgpu_decode_llr_gmd; 2t <= 32): y (frames, n*q), bit j of symbol c at position c*q + j; trials erase the 0, 2,
        .., max_erasures least reliable symbols -> words (frames, n) uint8, failed (frames,) uint8, chosen (frames,)
        uint8 [index i of the winning trial]; numpy or torch CUDA tensors like decode()"""
        nq = self.n * self.q
        if _is_torch(y):
            import torch
            y = y.contiguous().view(-1, nq)
            frames = y.shape[0]
            if out is None:
                out = (torch.empty((frames, self.n), dtype=torch.uint8, device=y.device),
                       torch.empty(frames, dtype=torch.uint8, device=y.device),
                       torch.empty(frames, dtype=torch.uint8, device=y.device))
        else:
            y = np.ascontiguousarray(y, np.float32).reshape(-1, nq)
            frames = y.shape[0]
            if out is None:
                out = (np.empty((frames, self.n), np.uint8), np.empty(frames, np.uint8), np.empty(frames, np.uint8))
        words, failed, chosen = out
        self.ctx._follow_torch(y, words)
        self.ctx._check(_lib.lib().ccgpu_decode_llr_gmd(self.ctx._h, self._h, int(max_erasures), _ptr(y), frames,
                                                        _ptr(words), _ptr(failed), _ptr(chosen)))
        return words, failed, chosen

    def awgn_point_gmd(self, ebno_db, frames, max_erasures, seed=0, point=0, frame0=0, out=None):
        """one Eb/N0 point of a Reed-Solomon code decoded with GMD on the GPU (ccgpu_awgn_point_gmd; max_erasures = 0:
        hard-decision decoding) -> counters.  out: optional torch uint64/int64 CUDA tensor of 8 slots that is
        accumulated into (no sync)."""
        if out is not None:
            self.ctx._follow_torch(out)
            self.ctx._check(_lib.lib().ccgpu_awgn_point_gmd(self.ctx._h, self._h, int(max_erasures), float(ebno_db), seed,
                                                            point, frame0, frames, _ptr(out)))
            return out
        c = Counters()
        self.ctx._check(_lib.lib().ccgpu_awgn_point_gmd(self.ctx._h, self._h, int(max_erasures), float(ebno_db), seed, point,
                                                        frame0, frames, C.addressof(c)))
        return c.as_dict()

    def decode_abp(self, y, max_iter=50, gamma=0.15, out=None):
        """adaptive belief propagation with the min-sum check pass (extension, ccgpu_decode_llr_abp; binary BCH codes
        with n <= 127, n - l <= 64; 0 <= max_iter <= 255, 0 < gamma <= 1) -> bits, L, iter, failed like decode();
        out = (bits, L or None, iter, failed); numpy or torch CUDA tensors like decode()"""
        if _is_torch(y):
            import torch
            y = y.contiguous().view(-1, self.n)
            frames = y.shape[0]
            if out is None:
                out = (torch.empty((frames, self.n), dtype=torch.uint8, device=y.device),
                       torch.empty((frames, self.n), dtype=torch.float32, device=y.device),
                       torch.empty(frames, dtype=torch.uint8, device=y.device),
                       torch.empty(frames, dtype=torch.uint8, device=y.device))
        else:
            y = np.ascontiguousarray(y, np.float32).reshape(-1, self.n)
            frames = y.shape[0]
            if out is None:
                out = (np.empty((frames, self.n), np.uint8), np.empty((frames, self.n), np.float32),
                       np.empty(frames, np.uint8), np.empty(frames, np.uint8))
        bits, L, it, failed = out
        self.ctx._follow_torch(y, bits)
        self.ctx._check(_lib.lib().ccgpu_decode_llr_abp(self.ctx._h, self._h, int(max_iter), float(gamma), _ptr(y), frames,
                                                        _ptr(bits), _ptr(L), _ptr(it), _ptr(failed)))
        return bits, L, it, failed

    def awgn_point_abp(self, ebno_db, frames, max_iter=50, gamma=0.15, seed=0, point=0, frame0=0, out=None):
        """one Eb/N0 point decoded with ABP on the GPU (ccgpu_awgn_point_abp) -> counters.
        out: optional torch uint64/int64 CUDA tensor of 8 slots that is accumulated into (no sync)."""
        if out is not None:
            self.ctx._follow_torch(out)
            self.ctx._check(_lib.lib().ccgpu_awgn_point_abp(self.ctx._h, self._h, int(max_iter), float(gamma), float(ebno_db),
                                                            seed, point, frame0, frames, _ptr(out)))
            return out
        c = Counters()
        self.ctx._check(_lib.lib().ccgpu_awgn_point_abp(self.ctx._h, self._h, int(max_iter), float(gamma), float(ebno_db), seed,
                                                        point, frame0, frames, C.addressof(c)))
        return c.as_dict()

    def decode_ml(self, y, out=None):
        """maximum-likelihood decoding by a Viterbi search over the syndrome trellis of the k-row H (extension,
        ccgpu_decode_llr_ml; binary BCH codes with n <= 127, n - l <= 12) -> bits (frames, n) uint8, a codeword closest
        to y; out: the bits array to write; numpy or torch CUDA tensors like decode()"""
        if _is_torch(y):
            import torch
            y = y.contiguous().view(-1, self.n)
            frames = y.shape[0]
            if out is None:
                out = torch.empty((frames, self.n), dtype=torch.uint8, device=y.device)
        else:
            y = np.ascontiguousarray(y, np.float32).reshape(-1, self.n)
            frames = y.shape[0]
            if out is None:
                out = np.empty((frames, self.n), np.uint8)
        self.ctx._follow_torch(y, out)
        self.ctx._check(_lib.lib().ccgpu_decode_llr_ml(self.ctx._h, self._h, _ptr(y), frames, _ptr(out)))
        return out

    def awgn_point_ml(self, ebno_db, frames, seed=0, point=0, frame0=0, out=None):
        """one Eb/N0 point decoded with ML on the GPU (ccgpu_awgn_point_ml) -> counters.
        out: optional torch uint64/int64 CUDA tensor of 8 slots that is accumulated into (no sync)."""
        if out is not None:
            self.ctx._follow_torch(out)
            self.ctx._check(_lib.lib().ccgpu_awgn_point_ml(self.ctx._h, self._h, float(ebno_db), seed, point, frame0, frames,
                                                           _ptr(out)))
            return out
        c = Counters()
        self.ctx._check(_lib.lib().ccgpu_awgn_point_ml(self.ctx._h, self._h, float(ebno_db), seed, point, frame0, frames,
                                                       C.addressof(c)))
        return c.as_dict()

    def bitflip_point(self, weight, variant="MS", alpha=1.0, beta=0.0, max_iter=50,
                      stop_rule=STOP_REF_ZERO_OVERLAP, first=0, count=0, quant=None):
        """one error weight of bitflip_simulation (simulation.c++:156-213) -> counters"""
        p = ms_params(variant, alpha, beta, max_iter, stop_rule, quant)
        c = Counters()
        self.ctx._check(_lib.lib().ccgpu_bitflip_point(self.ctx._h, self._h, C.byref(p), weight, first, count,
                                                       C.addressof(c)))
        return c.as_dict()

    def set_recheck(self, enable):
        _check(self.ctx, _lib.lib().ccgpu_code_set_recheck(self._h, int(bool(enable))))

    def gf_decode(self, words, out=None, erasures=None, pgz_fill=False):
        """cyclic::correct_(.., hard_decision_tag) per word -> corrected, n_errors, failed.
        erasures: optional (positions[count, max_e] uint8, counts[count] uint8); pgz_fill=True handles them like the
        reference's PGZ decoder of binary BCH codes (zero fill / one fill, bch.h:97-149) instead of the
        errors-and-erasures locator"""
        if _is_torch(words):
            import torch
            words = words.contiguous().view(-1, self.n)
            cnt = words.shape[0]
            if out is None:
                out = (torch.empty_like(words), torch.empty(cnt, dtype=torch.uint8, device=words.device),
                       torch.empty(cnt, dtype=torch.uint8, device=words.device))
        else:
            words = np.ascontiguousarray(words, np.uint8).reshape(-1, self.n)
            cnt = words.shape[0]
            if out is None:
                out = (np.empty_like(words), np.empty(cnt, np.uint8), np.empty(cnt, np.uint8))
        corrected, nerr, failed = out
        self.ctx._follow_torch(words, corrected)
        if erasures is None:
            self.ctx._check(_lib.lib().ccgpu_gf_decode(self.ctx._h, self._h, _ptr(words), cnt, _ptr(corrected),
                                                       _ptr(nerr), _ptr(failed)))
        else:
            epos, ecnt = erasures
            if not _is_torch(epos):
                epos = np.ascontiguousarray(epos, np.uint8).reshape(cnt, -1)
                ecnt = np.ascontiguousarray(ecnt, np.uint8)
            fn = _lib.lib().ccgpu_gf_decode_erasures_pgz if pgz_fill else _lib.lib().ccgpu_gf_decode_erasures
            self.ctx._check(fn(self.ctx._h, self._h, _ptr(words), cnt, _ptr(epos), _ptr(ecnt), epos.shape[1],
                               _ptr(corrected), _ptr(nerr), _ptr(failed)))
        return corrected, nerr, failed


class Group:
    """several GPUs of this host behind one handle (ccgpu_group): Monte-Carlo points are sharded over the member
    devices by global frame index and the counters merged inside the library; `devices` may repeat an ordinal"""

    def __init__(self, devices):
        devices = list(range(devices)) if isinstance(devices, int) else list(devices)
        arr = (C.c_int * len(devices))(*devices)
        self._h = C.c_void_p()
        rc = _lib.lib().ccgpu_group_create(len(devices), arr, C.byref(self._h))
        if rc != 0:
            raise CcgpuError(rc, "ccgpu_group_create(%s) failed -- not enough usable CUDA devices" % devices)
        self.devices = devices
        self.members = [_Member(self, m) for m in range(len(devices))]
        self._codes = []

    def close(self):
        if getattr(self, "_h", None):
            for gc in self._codes:  # the codes live on the members' contexts: release them first
                for c in gc.codes:
                    c.close()
            for m in self.members:
                m._h = None
            _lib.lib().ccgpu_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise CcgpuError(rc, _lib.lib().ccgpu_group_last_error(self._h).decode())

    def set_min_frames(self, frames_per_member):
        self._check(_lib.lib().ccgpu_group_set_min_frames(self._h, int(frames_per_member)))

    def bch(self, q, errors=None, dmin=None):
        return GroupCode(self, [m.bch(q, errors=errors, dmin=dmin) for m in self.members])

    def rs(self, q, errors, mu=1, step=1):
        return GroupCode(self, [m.rs(q, errors, mu, step) for m in self.members])


class _Member(Context):
    """a member context of a Group (owned by the group)"""

    def __init__(self, group, member):
        self._h = C.c_void_p(_lib.lib().ccgpu_group_ctx(group._h, member))
        self.device = group.devices[member]
        self._group = group

    def close(self):
        self._h = None


class GroupCode:
    """one code replicated on every member of a Group"""

    def __init__(self, group, codes):
        self.group, self.codes = group, codes
        group._codes.append(self)
        self._arr = (C.c_void_p * len(codes))(*[c._h for c in codes])
        for k in ("n", "l", "k", "rate", "edges", "h_rows", "row_weight", "kernel"):
            setattr(self, k, getattr(codes[0], k))

    def to_string(self, tag):
        return self.codes[0].to_string(tag)

    def set_rows(self, rows):
        for c in self.codes:
            c.set_rows(rows)
        self.h_rows, self.edges = self.codes[0].h_rows, self.codes[0].edges

    def awgn_point(self, ebno_db, frames, variant="MS", alpha=1.0, beta=0.0, max_iter=50, stop_rule=STOP_REF_ZERO_OVERLAP,
                   seed=0, point=0, frame0=0, quant=None):
        p = ms_params(variant, alpha, beta, max_iter, stop_rule, quant)
        c = Counters()
        self.group._check(_lib.lib().ccgpu_group_awgn_point(self.group._h, self._arr, C.byref(p), float(ebno_db), seed, point,
                                                            frame0, frames, C.addressof(c)))
        return c.as_dict()

    def awgn_point_hard(self, ebno_db, frames, seed=0, point=0, frame0=0):
        c = Counters()
        self.group._check(_lib.lib().ccgpu_group_awgn_point_hard(self.group._h, self._arr, float(ebno_db), seed, point, frame0,
                                                                 frames, C.addressof(c)))
        return c.as_dict()

    def awgn_point_chase(self, ebno_db, frames, p, seed=0, point=0, frame0=0):
        c = Counters()
        self.group._check(_lib.lib().ccgpu_group_awgn_point_chase(self.group._h, self._arr, int(p), float(ebno_db), seed, point,
                                                                  frame0, frames, C.addressof(c)))
        return c.as_dict()

    def awgn_point_osd(self, ebno_db, frames, order, seed=0, point=0, frame0=0):
        c = Counters()
        self.group._check(_lib.lib().ccgpu_group_awgn_point_osd(self.group._h, self._arr, int(order), float(ebno_db), seed,
                                                                point, frame0, frames, C.addressof(c)))
        return c.as_dict()

    def awgn_point_gmd(self, ebno_db, frames, max_erasures, seed=0, point=0, frame0=0):
        c = Counters()
        self.group._check(_lib.lib().ccgpu_group_awgn_point_gmd(self.group._h, self._arr, int(max_erasures), float(ebno_db),
                                                                seed, point, frame0, frames, C.addressof(c)))
        return c.as_dict()

    def awgn_point_abp(self, ebno_db, frames, max_iter=50, gamma=0.15, seed=0, point=0, frame0=0):
        c = Counters()
        self.group._check(_lib.lib().ccgpu_group_awgn_point_abp(self.group._h, self._arr, int(max_iter), float(gamma),
                                                                float(ebno_db), seed, point, frame0, frames, C.addressof(c)))
        return c.as_dict()

    def awgn_point_ml(self, ebno_db, frames, seed=0, point=0, frame0=0):
        c = Counters()
        self.group._check(_lib.lib().ccgpu_group_awgn_point_ml(self.group._h, self._arr, float(ebno_db), seed, point,
                                                               frame0, frames, C.addressof(c)))
        return c.as_dict()

    def awgn_point_mbbp(self, ebno_db, frames, shifts, variant="MS", alpha=1.0, beta=0.0, max_iter=50,
                        stop_rule=STOP_REF_ZERO_OVERLAP, seed=0, point=0, frame0=0):
        p = ms_params(variant, alpha, beta, max_iter, stop_rule)
        sh = np.ascontiguousarray(shifts, np.uint32)
        c = Counters()
        self.group._check(_lib.lib().ccgpu_group_awgn_point_mbbp(self.group._h, self._arr, C.byref(p), sh.ctypes.data, len(sh),
                                                                 float(ebno_db), seed, point, frame0, frames, C.addressof(c)))
        return c.as_dict()

    def bitflip_point(self, weight, variant="MS", alpha=1.0, beta=0.0, max_iter=50, stop_rule=STOP_REF_ZERO_OVERLAP, first=0,
                      count=0, quant=None):
        p = ms_params(variant, alpha, beta, max_iter, stop_rule, quant)
        c = Counters()
        self.group._check(_lib.lib().ccgpu_group_bitflip_point(self.group._h, self._arr, C.byref(p), weight, first, count,
                                                               C.addressof(c)))
        return c.as_dict()

    def decode(self, y, variant="MS", alpha=1.0, beta=0.0, max_iter=50, stop_rule=STOP_REF_ZERO_OVERLAP, want_L=True, out=None,
               quant=None):
        """ccgpu_group_decode_llr: host (numpy) buffers, frames sharded over the members"""
        p = ms_params(variant, alpha, beta, max_iter, stop_rule, quant)
        y = np.ascontiguousarray(y, np.float32).reshape(-1, self.n)
        frames = y.shape[0]
        if out is None:
            out = (np.empty((frames, self.n), np.uint8), np.empty((frames, self.n), np.float32) if want_L else None,
                   np.empty(frames, np.uint8), np.empty(frames, np.uint8))
        bits, L, it, failed = out
        self.group._check(_lib.lib().ccgpu_group_decode_llr(self.group._h, self._arr, C.byref(p), _ptr(y), frames, _ptr(bits),
                                                            _ptr(L), _ptr(it), _ptr(failed)))
        return bits, L, it, failed

    def gf_decode(self, words, out=None):
        words = np.ascontiguousarray(words, np.uint8).reshape(-1, self.n)
        cnt = words.shape[0]
        if out is None:
            out = (np.empty_like(words), np.empty(cnt, np.uint8), np.empty(cnt, np.uint8))
        corrected, nerr, failed = out
        self.group._check(_lib.lib().ccgpu_group_gf_decode(self.group._h, self._arr, _ptr(words), cnt, _ptr(corrected),
                                                           _ptr(nerr), _ptr(failed)))
        return corrected, nerr, failed


def sigma(rate, ebno_db):
    return _lib.lib().ccgpu_sigma(float(rate), float(ebno_db))


def gf_tables(q, poly=0):
    size = 1 << q
    exp = np.zeros(2 * size, np.uint16)
    log = np.zeros(size, np.uint16)
    rc = _lib.lib().ccgpu_gf_tables(q, poly, exp.ctypes.data, log.ctypes.data)
    if rc != 0:
        raise CcgpuError(rc, "ccgpu_gf_tables")
    return exp, log
