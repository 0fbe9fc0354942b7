"""ctypes binding of libvr180_b200.so (include/vr180_b200.h).

The product has no CPU fallback: if the shared object is missing or a call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = PKG / "libvr180_b200.so"

ABI_VERSION = 2
MAX_OPS = 12
MAX_OP_PARAMS = 12

# vr180_op_code
OP_NORMALIZE, OP_DENORMALIZE, OP_DENORMALIZE_INV, OP_ZOOM, OP_ZOOM_INV = 1, 2, 3, 4, 5
OP_EQUIRECT_ENC, OP_EQUIRECT_DEC, OP_FISHEYE_ENC, OP_FISHEYE_DEC = 6, 7, 8, 9
OP_RECTILINEAR_DEC, OP_RECTILINEAR_DEC_INV, OP_POLY, OP_ROT3 = 10, 11, 12, 13
MAPPING_CODES = {"rectilinear": 0, "stereographic": 1, "equidistant": 2, "equisolid": 3, "orthographic": 4}
MAPSRC_ANALYTIC, MAPSRC_FLOAT2, MAPSRC_FIXED, MAPSRC_PACKED = 0, 1, 2, 3
DEPTH_8U, DEPTH_16U = 0, 2  # OpenCV's depth codes (vr180_image_t.depth, vr180_host_job_t.depth)


class NativeError(RuntimeError):
    """A C-ABI call returned a negative vr180_status."""


class Op(C.Structure):
    _fields_ = [("code", C.c_int32), ("iparam", C.c_int32), ("p", C.c_double * MAX_OP_PARAMS)]


class Chain(C.Structure):
    _fields_ = [("n_ops", C.c_int32), ("reserved", C.c_int32), ("ops", Op * MAX_OPS)]


class Image(C.Structure):
    _fields_ = [("data", C.c_void_p), ("rows", C.c_int32), ("cols", C.c_int32), ("channels", C.c_int32),
                ("depth", C.c_int32), ("pitch", C.c_int64), ("frame_stride", C.c_int64)]


class MapSrc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("packed_interpolation", C.c_int32), ("chain", C.POINTER(Chain)),
                ("xmap", C.c_void_p), ("ymap", C.c_void_p), ("fixed", C.c_void_p), ("map_pitch", C.c_int64),
                ("radius_dev", C.c_void_p), ("packed", C.c_void_p)]


class View(C.Structure):
    _fields_ = [("src", Image), ("map", MapSrc), ("dst_x_offset", C.c_int32), ("reserved", C.c_int32)]


class RemapParams(C.Structure):
    _fields_ = [("n_views", C.c_int32), ("n_frames", C.c_int32), ("view", View * 2), ("share_map", C.c_int32),
                ("out_w", C.c_int32), ("out_h", C.c_int32), ("interpolation", C.c_int32), ("border_mode", C.c_int32),
                ("border_value", C.c_uint8 * 4), ("dst", C.c_void_p), ("dst_pitch", C.c_int64),
                ("dst_frame_stride", C.c_int64)]


class HostJob(C.Structure):
    _fields_ = [("n_views", C.c_int32), ("n_frames", C.c_int32), ("src", C.c_void_p * 2), ("src_rows", C.c_int32),
                ("src_cols", C.c_int32), ("channels", C.c_int32), ("depth", C.c_int32),
                ("src_pitch", C.c_int64 * 2), ("src_frame_stride", C.c_int64 * 2), ("map_kind", C.c_int32),
                ("share_map", C.c_int32), ("chain", C.POINTER(Chain) * 2), ("xmap", C.c_void_p * 2),
                ("ymap", C.c_void_p * 2), ("maps_cache_key", C.c_uint64), ("radius_mode", C.c_int32),
                ("reserved1", C.c_int32), ("threshold", C.c_double), ("out_w", C.c_int32), ("out_h", C.c_int32),
                ("interpolation", C.c_int32), ("border_mode", C.c_int32), ("border_value", C.c_uint8 * 4),
                ("dst", C.c_void_p), ("dst_pitch", C.c_int64), ("dst_frame_stride", C.c_int64),
                ("transitions_out", C.c_void_p), ("radius_out", C.c_void_p),
                ("src_frames", C.POINTER(C.c_void_p) * 2), ("dst_frames", C.POINTER(C.c_void_p)),
                ("staging", C.c_int32), ("copy_threads", C.c_int32), ("merge", C.c_int32), ("reserved2", C.c_int32)]


# every symbol include/vr180_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "vr180_abi_version": (C.c_int, []),
    "vr180_status_string": (C.c_char_p, [C.c_int]),
    "vr180_last_cuda_error": (C.c_char_p, []),
    "vr180_device_info": (C.c_int, [C.c_int, C.c_char_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                    C.POINTER(C.c_int)]),
    "vr180_launch_count": (C.c_uint64, []),
    "vr180_build_map": (C.c_int, [C.POINTER(Chain), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "vr180_pack_lut": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int64,
                                 C.c_void_p]),
    "vr180_packed_lut_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "vr180_pack_lut_tiles": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p]),
    "vr180_remap": (C.c_int, [C.POINTER(RemapParams), C.c_void_p]),
    "vr180_remap_ex": (C.c_int, [C.POINTER(RemapParams), C.POINTER(C.c_double), C.c_void_p]),
    "vr180_anaglyph": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64,
                                 C.c_int64, C.c_void_p]),
    "vr180_transform_points": (C.c_int, [C.POINTER(Chain), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "vr180_jpeg_available": (C.c_int, []),
    "vr180_jpeg_info": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "vr180_jpeg_decode": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p]),
    "vr180_jpeg_encode": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                    C.POINTER(C.c_size_t), C.c_void_p]),
    "vr180_get_radius": (C.c_int, [C.POINTER(Image), C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p,
                                   C.c_void_p]),
    "vr180_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "vr180_ctx_destroy": (C.c_int, [C.c_void_p]),
    "vr180_ctx_device": (C.c_int, [C.c_void_p]),
    "vr180_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "vr180_host_free": (C.c_int, [C.c_void_p]),
    "vr180_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "vr180_host_unregister": (C.c_int, [C.c_void_p]),
    "vr180_ctx_run": (C.c_int, [C.c_void_p, C.POINTER(HostJob)]),
    "vr180_ctx_run_ex": (C.c_int, [C.c_void_p, C.POINTER(HostJob), C.POINTER(C.c_double)]),
    "vr180_debug_weight_table": (C.c_int, [C.c_int, C.c_void_p]),
    "vr180_debug_set": (C.c_int, [C.c_int, C.c_int]),
    "vr180_debug_copy_ceiling": (C.c_int, [C.c_int, C.c_size_t, C.c_int, C.POINTER(C.c_double)]),
    "vr180_debug_host_copy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
}

_lib = None


def lib() -> C.CDLL:
    """Load the shared object (once).  Raises if it has not been built -- there is no fallback path."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python vr180-convert_b200/build.py` "
                "(or __graft_entry__.build()); vr180_convert_b200 has no CPU fallback")
        handle = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.vr180_abi_version() != ABI_VERSION:
            raise ImportError("libvr180_b200.so ABI version mismatch; rebuild")
        _lib = handle
    return _lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        handle = lib()
        msg = handle.vr180_status_string(status).decode()
        if status == -3:
            msg += ": " + handle.vr180_last_cuda_error().decode()
        raise NativeError(f"{what or 'vr180 call'} failed ({status}): {msg}")


def make_chain(ops) -> Chain:
    """Op tuples (the vocabulary of transformer.lower()) -> vr180_chain_t."""
    if not 1 <= len(ops) <= MAX_OPS:
        raise ValueError(f"chain must have 1..{MAX_OPS} ops, got {len(ops)}")
    ch = Chain()
    ch.n_ops = len(ops)
    for k, op in enumerate(ops):
        o = ch.ops[k]
        kind = op[0]
        params: list[float] = []
        if kind == "normalize":
            o.code = OP_NORMALIZE
            params = [op[1][0], op[1][1], op[2]]
        elif kind in ("denormalize", "denormalize_inv"):
            o.code = OP_DENORMALIZE if kind == "denormalize" else OP_DENORMALIZE_INV
            params = [op[1][0], op[1][1], op[2][0], op[2][1]]
        elif kind in ("zoom", "zoom_inv"):
            o.code = OP_ZOOM if kind == "zoom" else OP_ZOOM_INV
            params = [op[1]]
        elif kind in ("equirect_enc", "equirect_dec"):
            o.code = OP_EQUIRECT_ENC if kind == "equirect_enc" else OP_EQUIRECT_DEC
            o.iparam = 1 if op[1] else 0
        elif kind in ("fisheye_enc", "fisheye_dec"):
            o.code = OP_FISHEYE_ENC if kind == "fisheye_enc" else OP_FISHEYE_DEC
            o.iparam = MAPPING_CODES[op[1]]
        elif kind in ("rectilinear_dec", "rectilinear_dec_inv"):
            o.code = OP_RECTILINEAR_DEC if kind == "rectilinear_dec" else OP_RECTILINEAR_DEC_INV
            params = [op[1]]
        elif kind == "poly":
            coefs = [float(c) for c in op[1]]
            if len(coefs) > MAX_OP_PARAMS:
                raise ValueError(f"polynomial degree above {MAX_OP_PARAMS - 1} is not supported by the kernel")
            o.code = OP_POLY
            o.iparam = len(coefs)
            params = coefs
        elif kind == "rot3":
            o.code = OP_ROT3
            params = [float(v) for v in op[1]]
            if len(params) != 9:
                raise ValueError("rot3 needs a 3x3 matrix")
        else:
            raise ValueError(f"unknown chain op {kind!r}")
        for i, v in enumerate(params):
            o.p[i] = float(v)
    return ch
