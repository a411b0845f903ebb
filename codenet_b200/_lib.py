"""ctypes binding of libcodenet_b200.so (the C ABI declared in include/codenet_b200.h).

There is no CPU fallback: if the library is missing it is built with nvcc, and if that is impossible, or no
sm_100 device is visible when a device function is called, an exception is raised.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libcodenet_b200.so")
_lib = None


class CdnError(RuntimeError):
    pass


class Requant(C.Structure):
    _fields_ = [("M", C.POINTER(C.c_double)), ("B", C.POINTER(C.c_double)), ("lo", C.c_int), ("n", C.c_int)]


class DeformScale(C.Structure):
    _fields_ = [("ws", C.POINTER(C.c_int8)), ("Ms", C.c_double), ("bs", C.c_double), ("ss", C.c_double),
                ("zs", C.c_double), ("bound", C.c_int), ("mode", C.c_int)]


class PwChunk(C.Structure):
    _fields_ = [("col", C.c_int16), ("count", C.c_int16), ("pass_off", C.c_int16), ("dst_off", C.c_int16)]


class PwDesc(C.Structure):
    _fields_ = [("K", C.c_int), ("k_off", C.c_int), ("N", C.c_int), ("zx", C.c_int), ("wq", C.POINTER(C.c_int8)),
                ("rq", Requant), ("chunks", C.POINTER(PwChunk)), ("n_chunks", C.c_int),
                ("n_f32", C.c_int), ("Mf", C.POINTER(C.c_double)), ("bf", C.POINTER(C.c_double))]


# cdn_warp_desc (include/codenet_b200.h): one output image of cdn_warp_affine_u8_batch
WARP_DESC = np.dtype([("src_offset", np.int64), ("src_h", np.int32), ("src_w", np.int32), ("M", np.float64, (6,)),
                      ("dst_slot", np.int32), ("mirror_slot", np.int32)])
assert WARP_DESC.itemsize == 72
WARP_DESC_PER_LAUNCH = 454         # CDN_WARP_DESC_PER_LAUNCH
WARP_F32_DESC_PER_LAUNCH = 448     # CDN_WARP_F32_DESC_PER_LAUNCH (cdn_warp_affine_u8_f32_batch)

EXPORTS = {
    "cdn_last_error": (C.c_char_p, []),
    "cdn_version": (C.c_int, []),
    "cdn_check_device": (C.c_int, [C.c_int]),
    "cdn_set_debug_flags": (C.c_int, [C.c_uint]),
    "cdn_rq_int_solve": (C.c_int, [C.c_double, C.c_double, C.c_int, C.c_int64, C.c_int64, C.POINTER(C.c_int32),
                                   C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "cdn_stem_f32_i8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int8), C.c_int,
                                  C.POINTER(Requant), C.c_void_p, C.c_int, C.c_void_p]),
    "cdn_dw3x3_i8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int8),
                               C.c_int, C.c_int, C.POINTER(Requant), C.c_void_p, C.c_int, C.c_void_p]),
    "cdn_deform_dw_w4a8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(DeformScale),
                                     C.POINTER(C.c_int8), C.c_int, C.c_int, C.POINTER(Requant), C.c_void_p, C.c_int,
                                     C.c_void_p, C.c_void_p]),
    "cdn_deform_layer_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(DeformScale), C.POINTER(C.c_int8), C.c_int, C.c_int,
                                          C.c_int, C.POINTER(Requant)]),
    "cdn_deform_layer_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                       C.c_int, C.c_void_p, C.c_void_p]),
    "cdn_deform_layer_destroy": (C.c_int, [C.c_void_p]),
    "cdn_pw_gemm_i8": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.POINTER(PwDesc), C.c_void_p, C.c_int, C.c_void_p,
                                 C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "cdn_shuffle_unit_i8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(PwDesc), C.POINTER(C.c_int8),
                                      C.c_int, C.c_int, C.POINTER(Requant), C.POINTER(PwDesc), C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                      C.c_void_p]),
    "cdn_ctdet_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "cdn_ctdet_decode_prob": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "cdn_ctdet_decode_ws_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "cdn_ctdet_decode_ws": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_int, C.c_int,
                                      C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cdn_ctdet_post_affine": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "cdn_ctdet_flip_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                       C.c_void_p]),
    "cdn_deform_conv_forward_f32": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 16 + [C.c_void_p]),
    "cdn_deform_dw_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                    C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "cdn_deform_dw_up2_f32_ws": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                           C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cdn_deform_dw_f32_ws_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "cdn_deform_dw_f32_ws": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "cdn_pw_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "cdn_conv3x3_f32": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 7 + [C.c_void_p]),
    "cdn_dw3x3_f32": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 6 + [C.c_void_p]),
    "cdn_dw3x3_up2_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "cdn_pw_slice_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "cdn_pw_tf32x3_packed_floats": (C.c_size_t, [C.c_int, C.c_int]),
    "cdn_pw_tf32x3_pack": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "cdn_pw_slice_tf32x3": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                      C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "cdn_copy_channels_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_void_p]),
    "cdn_maxpool3s2_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "cdn_upsample2x_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "cdn_engine_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "cdn_engine_destroy": (C.c_int, [C.c_void_p]),
    "cdn_engine_add_tensor": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "cdn_engine_add_stem": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int8),
                                      C.c_int, C.POINTER(Requant)]),
    "cdn_engine_add_dw": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int8), C.c_int,
                                    C.c_int, C.POINTER(Requant)]),
    "cdn_engine_add_deform": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(DeformScale),
                                        C.POINTER(C.c_int8), C.c_int, C.c_int, C.POINTER(Requant)]),
    "cdn_engine_add_pw": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(PwDesc)]),
    "cdn_engine_set_heads": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "cdn_engine_finalize": (C.c_int, [C.c_void_p, C.c_int]),
    "cdn_engine_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "cdn_engine_run_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "cdn_engine_set_normalization": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "cdn_engine_run_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]),
    "cdn_engine_run_host_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "cdn_warp_affine_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "cdn_warp_affine_u8_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "cdn_warp_affine_u8_f32_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                               C.c_int, C.c_int, C.c_void_p]),
    "cdn_jpeg_parse": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "cdn_jpeg_decode_batch": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.c_void_p,
                                        C.c_int64, C.c_void_p, C.c_void_p]),
    "cdn_ctdet_group_by_class": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cdn_soft_nms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, C.c_void_p,
                               C.c_void_p]),
    "cdn_ctdet_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    "cdn_quantize_f32_i8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p, C.c_int, C.c_void_p]),
    "cdn_maxpool3s2_i8": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "cdn_engine_submit_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "cdn_engine_submit_host_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]),
    "cdn_engine_wait": (C.c_int, [C.c_void_p, C.c_int]),
    "cdn_engine_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "cdn_engine_read_tensor": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "cdn_engine_read_heads": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "cdn_engine_num_launches": (C.c_int, [C.c_void_p]),
    "cdn_engine_heads_fused": (C.c_int, [C.c_void_p]),
    "cdn_engine_units_fused": (C.c_int, [C.c_void_p]),
    "cdn_engine_op_fusion": (C.c_int, [C.c_void_p, C.c_int]),
    "cdn_engine_requant_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "cdn_engine_profile": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
}


def lib_path():
    return _LIB_PATH


def load():
    """Loads (building first if necessary) the shared library.  Raises if it cannot be produced."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        from . import build as _build
        _build.build()
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)                  # AttributeError if a declared symbol is not exported
        fn.restype, fn.argtypes = res, args
    if os.environ.get("CODENET_DEBUG_FLAGS"):        # kernel A/B experiments only (cdn_set_debug_flags)
        lib.cdn_set_debug_flags(int(os.environ["CODENET_DEBUG_FLAGS"]))
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise CdnError("codenet_b200: %s (status %d)" % (load().cdn_last_error().decode(), rc))


# ---- numpy -> ctypes helpers (keep the arrays alive for the duration of the call) --------------------------------
def i8p(a):
    return a.ctypes.data_as(C.POINTER(C.c_int8))


def f64p(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class Keep:
    """Collects the contiguous arrays whose pointers were handed to C."""

    def __init__(self):
        self.refs = []

    def i8(self, a):
        a = np.ascontiguousarray(a, dtype=np.int8); self.refs.append(a); return i8p(a)

    def f64(self, a):
        a = np.ascontiguousarray(a, dtype=np.float64); self.refs.append(a); return f64p(a)

    def requant(self, M, B, lo):
        M = np.ascontiguousarray(M, dtype=np.float64); B = np.ascontiguousarray(B, dtype=np.float64)
        self.refs += [M, B]
        r = Requant(f64p(M), f64p(B), int(lo), int(M.size))
        self.refs.append(r)
        return r

    def chunks(self, arr):
        arr = np.ascontiguousarray(arr, dtype=np.int16).reshape(-1, 4)
        self.refs.append(arr)
        return arr.ctypes.data_as(C.POINTER(PwChunk)), int(arr.shape[0])

    def pw_desc(self, a):
        d = PwDesc()
        d.K, d.k_off, d.N, d.zx = int(a["K"]), int(a["k_off"]), int(a["N"]), int(a["zx"])
        d.wq = self.i8(a["wq"])
        d.n_f32 = int(a.get("n_f32", 0))
        if d.n_f32:
            d.Mf, d.bf = self.f64(a["Mf"]), self.f64(a["bf"])
            d.rq = Requant(None, None, -128, 0)
            d.chunks, d.n_chunks = None, 0
        else:
            d.rq = self.requant(a["M"], a["B"], a["lo"])
            d.chunks, d.n_chunks = self.chunks(a["chunks"])
        self.refs.append(d)
        return d

    def deform_scale(self, a):
        s = DeformScale(self.i8(a["ws"]), float(a["Ms"]), float(a["bs"]), float(a["ss"]), float(a["zs"]),
                        int(a["bound"]), int(a["mode"]))
        self.refs.append(s)
        return s
