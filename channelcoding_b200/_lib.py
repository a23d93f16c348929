"""ctypes binding of libccgpu.so (include/ccgpu.h).  There is no CPU fallback: if the CUDA
library was not built or no CUDA device is usable, importing / creating a context fails loudly."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CCGPU_LIB", os.path.join(_HERE, "libccgpu.so"))  # CCGPU_LIB: experimental builds

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED, ERR_NO_DEVICE = 0, -1, -2, -3, -4


class CcgpuError(RuntimeError):
    def __init__(self, code, text):
        super().__init__("ccgpu error %d: %s" % (code, text))
        self.code = code


class MsParams(C.Structure):
    _fields_ = [("variant", C.c_int32), ("stop_rule", C.c_int32), ("max_iter", C.c_uint32), ("q_msg_max", C.c_uint32),
                ("alpha", C.c_double), ("beta", C.c_double), ("q_scale", C.c_double), ("q_y_max", C.c_uint32),
                ("reserved", C.c_uint32)]


class Counters(C.Structure):
    _fields_ = [("frames", C.c_uint64), ("frame_errors", C.c_uint64), ("bit_errors", C.c_uint64),
                ("iterations", C.c_uint64), ("failures", C.c_uint64), ("undetected", C.c_uint64),
                ("reserved", C.c_uint64 * 2)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k in ("frames", "frame_errors", "bit_errors", "iterations", "failures",
                                                    "undetected")}


class CodeInfo(C.Structure):
    _fields_ = [(k, C.c_uint32) for k in ("family", "q", "n", "l", "k", "dmin", "t", "h_rows", "row_weight", "edges",
                                          "h_kind", "kernel")] + [("rate", C.c_double)]


_lib = None


def lib():
    """the loaded library; raises if it has not been built (python -m channelcoding_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError("channelcoding_b200: %s is missing -- build it with `python -m channelcoding_b200.build` "
                          "(nvcc, sm_100a).  There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, u8p, u64, u32, i32, dbl = C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int, C.c_double
    L.ccgpu_abi_version.restype = i32
    L.ccgpu_create.argtypes = [i32, C.POINTER(vp)]
    L.ccgpu_destroy.argtypes = [vp]
    L.ccgpu_destroy.restype = None
    L.ccgpu_last_error.argtypes = [vp]
    L.ccgpu_last_error.restype = C.c_char_p
    L.ccgpu_set_option.argtypes = [vp, C.c_char_p, C.c_int64]
    L.ccgpu_build_info.restype = C.c_char_p
    L.ccgpu_set_stream.argtypes = [vp, vp]
    L.ccgpu_get_stream.argtypes = [vp]
    L.ccgpu_get_stream.restype = vp
    L.ccgpu_sync.argtypes = [vp]
    L.ccgpu_kernel_launches.argtypes = [vp]
    L.ccgpu_kernel_launches.restype = u64
    L.ccgpu_bch_create.argtypes = [vp, u32, i32, u32, C.POINTER(vp)]
    L.ccgpu_rs_create.argtypes = [vp, u32, u32, u32, u32, C.POINTER(vp)]
    L.ccgpu_code_from_dense.argtypes = [vp, u8p, u32, u32, dbl, C.POINTER(vp)]
    L.ccgpu_code_set_rows.argtypes = [vp, u32]
    L.ccgpu_code_destroy.argtypes = [vp]
    L.ccgpu_code_destroy.restype = None
    L.ccgpu_code_get_info.argtypes = [vp, C.POINTER(CodeInfo)]
    L.ccgpu_code_to_string.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_size_t]
    L.ccgpu_code_H.argtypes = [vp, u8p]
    L.ccgpu_code_poly.argtypes = [vp, i32, vp, C.c_size_t]
    L.ccgpu_code_H_alt.argtypes = [vp, i32, vp, C.POINTER(u32)]
    L.ccgpu_gf_tables.argtypes = [u32, u32, vp, vp]
    L.ccgpu_encode.argtypes = [vp, u8p, u64, u8p]
    L.ccgpu_decode_llr.argtypes = [vp, vp, C.POINTER(MsParams), vp, u64, vp, vp, vp, vp]
    L.ccgpu_decode_llr_packed.argtypes = [vp, vp, C.POINTER(MsParams), vp, u64, vp, vp]
    L.ccgpu_sigma.argtypes = [dbl, dbl]
    L.ccgpu_sigma.restype = dbl
    L.ccgpu_shannon_limit_db.argtypes = [dbl]
    L.ccgpu_shannon_limit_db.restype = dbl
    L.ccgpu_shannon_limit_db_numeric.argtypes = [dbl]
    L.ccgpu_shannon_limit_db_numeric.restype = dbl
    L.ccgpu_sweep_start_ebno.argtypes = [dbl, dbl]
    L.ccgpu_sweep_start_ebno.restype = dbl
    L.ccgpu_sweep_samples.argtypes = [dbl, u64]
    L.ccgpu_sweep_samples.restype = u64
    L.ccgpu_awgn_llr.argtypes = [vp, u32, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_awgn_point.argtypes = [vp, vp, C.POINTER(MsParams), dbl, u64, u32, u64, u64, vp]
    L.ccgpu_awgn_point_hard.argtypes = [vp, vp, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_bitflip_point.argtypes = [vp, vp, C.POINTER(MsParams), u32, u64, u64, vp]
    L.ccgpu_awgn_point_uncoded.argtypes = [vp, u32, dbl, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_decode_llr_mbbp.argtypes = [vp, vp, C.POINTER(MsParams), vp, u32, vp, u64, vp, vp, vp, vp, vp]
    L.ccgpu_awgn_point_mbbp.argtypes = [vp, vp, C.POINTER(MsParams), vp, u32, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_decode_llr_chase.argtypes = [vp, vp, u32, vp, u64, vp, vp, vp]
    L.ccgpu_awgn_point_chase.argtypes = [vp, vp, u32, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_decode_llr_osd.argtypes = [vp, vp, u32, vp, u64, vp, vp]
    L.ccgpu_awgn_point_osd.argtypes = [vp, vp, u32, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_decode_llr_gmd.argtypes = [vp, vp, u32, vp, u64, vp, vp, vp]
    L.ccgpu_awgn_point_gmd.argtypes = [vp, vp, u32, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_decode_llr_abp.argtypes = [vp, vp, u32, dbl, vp, u64, vp, vp, vp, vp]
    L.ccgpu_awgn_point_abp.argtypes = [vp, vp, u32, dbl, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_decode_llr_ml.argtypes = [vp, vp, vp, u64, vp]
    L.ccgpu_awgn_point_ml.argtypes = [vp, vp, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_gf_decode.argtypes = [vp, vp, vp, u64, vp, vp, vp]
    L.ccgpu_gf_decode_erasures.argtypes = [vp, vp, vp, u64, vp, vp, u32, vp, vp, vp]
    L.ccgpu_gf_decode_erasures_pgz.argtypes = [vp, vp, vp, u64, vp, vp, u32, vp, vp, vp]
    L.ccgpu_code_set_recheck.argtypes = [vp, i32]
    cpp = C.POINTER(vp)
    L.ccgpu_group_create.argtypes = [i32, C.POINTER(i32), C.POINTER(vp)]
    L.ccgpu_group_destroy.argtypes = [vp]
    L.ccgpu_group_destroy.restype = None
    L.ccgpu_group_size.argtypes = [vp]
    L.ccgpu_group_ctx.argtypes = [vp, i32]
    L.ccgpu_group_ctx.restype = vp
    L.ccgpu_group_last_error.argtypes = [vp]
    L.ccgpu_group_last_error.restype = C.c_char_p
    L.ccgpu_group_set_min_frames.argtypes = [vp, u64]
    L.ccgpu_group_awgn_point.argtypes = [vp, cpp, C.POINTER(MsParams), dbl, u64, u32, u64, u64, vp]
    L.ccgpu_group_awgn_point_hard.argtypes = [vp, cpp, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_group_awgn_point_chase.argtypes = [vp, cpp, u32, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_group_awgn_point_osd.argtypes = [vp, cpp, u32, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_group_awgn_point_gmd.argtypes = [vp, cpp, u32, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_group_awgn_point_abp.argtypes = [vp, cpp, u32, dbl, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_group_awgn_point_ml.argtypes = [vp, cpp, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_group_awgn_point_mbbp.argtypes = [vp, cpp, C.POINTER(MsParams), vp, u32, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_group_awgn_point_uncoded.argtypes = [vp, u32, dbl, dbl, u64, u32, u64, u64, vp]
    L.ccgpu_group_bitflip_point.argtypes = [vp, cpp, C.POINTER(MsParams), u32, u64, u64, vp]
    L.ccgpu_group_decode_llr.argtypes = [vp, cpp, C.POINTER(MsParams), vp, u64, vp, vp, vp, vp]
    L.ccgpu_group_gf_decode.argtypes = [vp, cpp, vp, u64, vp, vp, vp]
    if L.ccgpu_abi_version() != 2:
        raise ImportError("libccgpu.so ABI version mismatch")
    _lib = L
    return L


# every symbol include/ccgpu.h declares (tests check that the library exports all of them)
EXPORTS = ["ccgpu_abi_version", "ccgpu_create", "ccgpu_destroy", "ccgpu_last_error", "ccgpu_set_option", "ccgpu_build_info", "ccgpu_set_stream",
           "ccgpu_get_stream", "ccgpu_sync", "ccgpu_kernel_launches", "ccgpu_bch_create", "ccgpu_rs_create",
           "ccgpu_code_from_dense", "ccgpu_code_set_rows", "ccgpu_code_destroy", "ccgpu_code_get_info",
           "ccgpu_code_to_string", "ccgpu_code_H", "ccgpu_code_H_alt", "ccgpu_code_poly", "ccgpu_gf_tables", "ccgpu_encode",
           "ccgpu_decode_llr", "ccgpu_decode_llr_packed", "ccgpu_sigma", "ccgpu_shannon_limit_db", "ccgpu_shannon_limit_db_numeric", "ccgpu_sweep_start_ebno", "ccgpu_sweep_samples", "ccgpu_awgn_llr", "ccgpu_awgn_point", "ccgpu_awgn_point_hard", "ccgpu_bitflip_point",
           "ccgpu_gf_decode", "ccgpu_gf_decode_erasures", "ccgpu_code_set_recheck", "ccgpu_decode_llr_mbbp", "ccgpu_awgn_point_uncoded", "ccgpu_gf_decode_erasures_pgz",
           "ccgpu_awgn_point_mbbp", "ccgpu_group_create", "ccgpu_group_destroy", "ccgpu_group_size", "ccgpu_group_ctx",
           "ccgpu_group_last_error", "ccgpu_group_set_min_frames", "ccgpu_group_awgn_point", "ccgpu_group_awgn_point_hard",
           "ccgpu_group_awgn_point_mbbp", "ccgpu_group_awgn_point_uncoded", "ccgpu_group_bitflip_point",
           "ccgpu_group_decode_llr", "ccgpu_group_gf_decode", "ccgpu_decode_llr_chase", "ccgpu_awgn_point_chase",
           "ccgpu_group_awgn_point_chase", "ccgpu_decode_llr_osd", "ccgpu_awgn_point_osd", "ccgpu_group_awgn_point_osd",
           "ccgpu_decode_llr_gmd", "ccgpu_awgn_point_gmd", "ccgpu_group_awgn_point_gmd",
           "ccgpu_decode_llr_abp", "ccgpu_awgn_point_abp", "ccgpu_group_awgn_point_abp",
           "ccgpu_decode_llr_ml", "ccgpu_awgn_point_ml", "ccgpu_group_awgn_point_ml"]
