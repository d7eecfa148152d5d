"""ctypes binding of libaeaj.so (include/aeaj.h).  Fails loudly: a missing library, a missing
symbol or a missing sm_100 device raises -- nothing here ever computes on the CPU."""
from __future__ import annotations

import ctypes as C
import os
import threading

import numpy as np

from . import tables

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG, "libaeaj.so")

EXPORTS = [
    "aeaj_last_error", "aeaj_version", "aeaj_create", "aeaj_destroy", "aeaj_set_color_tables", "aeaj_set_srgb_lut",
    "aeaj_color_forward", "aeaj_color_inverse", "aeaj_normalize", "aeaj_downsample_area", "aeaj_resize_linear",
    "aeaj_stage_workspace_bytes", "aeaj_cast_u8", "aeaj_clahe", "aeaj_gauss3", "aeaj_bilateral5",
    "aeaj_percentile_thresholds", "aeaj_canny_u8", "aeaj_canny", "aeaj_quadtree_caps", "aeaj_quadtree",
    "aeaj_dct_quant", "aeaj_dequant_idct", "aeaj_plan_create", "aeaj_plan_destroy", "aeaj_plan_get_info",
    "aeaj_plan_set_qtables", "aeaj_encode", "aeaj_decode", "aeaj_plan_last_launches",
    "aeaj_plan_enable_timing", "aeaj_plan_read_timing",
    "aeaj_plan_set_stream_layout", "aeaj_plan_set_tensor_dct", "aeaj_tensor_dct_status",
    "aeaj_states_to_leaves_host", "aeaj_pack_states_host",
    "aeaj_pack_coefficients", "aeaj_unpack_coefficients", "aeaj_pack_coefficients_host", "aeaj_unpack_coefficients_host",
    "aeaj_peer_alloc", "aeaj_peer_free", "aeaj_peer_export", "aeaj_peer_open", "aeaj_peer_close",
    "aeaj_plan_set_peers", "aeaj_copy_segments",
    "aeaj_encode_halo", "aeaj_decode_halo", "aeaj_set_fast_transfer",
    "aeaj_deflate_caps", "aeaj_deflate_coefficients", "aeaj_inflate_scratch_bytes", "aeaj_inflate_coefficients",
    "aeaj_decode_scaled_geometry", "aeaj_decode_scaled",
]


class AeajError(RuntimeError):
    pass


class PlanInfo(C.Structure):
    _fields_ = [("batch", C.c_int), ("height", C.c_int), ("width", C.c_int), ("space", C.c_int),
                ("block_min", C.c_int), ("block_max", C.c_int),
                ("layer_h", C.c_int * 3), ("layer_w", C.c_int * 3), ("root", C.c_int * 3),
                ("cap_leaves", C.c_int64 * 3), ("cap_states", C.c_int64 * 3), ("cap_coef", C.c_int64 * 3),
                ("workspace_bytes", C.c_int64)]


class EncodeIO(C.Structure):
    _fields_ = [("rgb", C.c_void_p), ("coef", C.c_void_p * 3), ("leaves", C.c_void_p * 3), ("states", C.c_void_p * 3),
                ("counts", C.c_void_p), ("tap_layers", C.c_void_p * 3), ("tap_edges", C.c_void_p * 3), ("status", C.c_void_p),
                ("packed_states", C.c_void_p * 3), ("rgb_u8", C.c_void_p)]


class DecodeIO(C.Structure):
    _fields_ = [("coef", C.c_void_p * 3), ("leaves", C.c_void_p * 3), ("counts", C.c_void_p), ("rgb", C.c_void_p),
                ("tap_layers", C.c_void_p * 3), ("rgb_u8", C.c_void_p), ("status", C.c_void_p)]


class PackedIO(C.Structure):
    _fields_ = [("mask", C.c_void_p * 3), ("vals", C.c_void_p * 3), ("counts", C.c_void_p)]


class DeflateIO(C.Structure):
    _fields_ = [("out", C.c_void_p * 3), ("lengths", C.c_void_p), ("status", C.c_void_p)]


class InflateIO(C.Structure):
    _fields_ = [("inp", C.c_void_p), ("offsets", C.c_void_p), ("lengths", C.c_void_p), ("coef", C.c_void_p * 3),
                ("status", C.c_void_p), ("out_bytes", C.c_void_p), ("segments", C.c_void_p)]


class Segment(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("bytes", C.c_int64)]


_lib = None
_lock = threading.Lock()


def load():
    """Load libaeaj.so; raises ImportError if it has not been built (python __graft_entry__.py build)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} not found: build it with `make -C {os.path.join(_PKG, 'csrc')}` "
                              "(or __graft_entry__.build()); there is no CPU fallback")
        lib = C.CDLL(LIB_PATH)
        missing = [s for s in EXPORTS if not hasattr(lib, s)]
        if missing:
            raise ImportError(f"libaeaj.so lacks symbols {missing}")
        lib.aeaj_last_error.restype = C.c_char_p
        lib.aeaj_stage_workspace_bytes.restype = C.c_size_t
        lib.aeaj_stage_workspace_bytes.argtypes = [C.c_int] * 4
        vp, i, sz, f = C.c_void_p, C.c_int, C.c_size_t, C.c_float
        lib.aeaj_create.argtypes = [i, C.POINTER(vp)]
        lib.aeaj_destroy.argtypes = [vp]
        lib.aeaj_set_color_tables.argtypes = [vp, i] + [vp] * 6
        lib.aeaj_set_srgb_lut.argtypes = [vp, vp]
        lib.aeaj_color_forward.argtypes = [vp, i, vp, vp, sz, vp]
        lib.aeaj_color_inverse.argtypes = [vp, i, vp, vp, sz, vp]
        lib.aeaj_normalize.argtypes = [vp, i, i, i, vp, vp, sz, vp]
        lib.aeaj_downsample_area.argtypes = [vp, vp, i, i, vp, i, i, vp]
        lib.aeaj_resize_linear.argtypes = [vp, vp, i, i, vp, i, i, vp]
        lib.aeaj_cast_u8.argtypes = [vp, vp, vp, sz, vp]
        for name in ("aeaj_clahe", "aeaj_gauss3", "aeaj_bilateral5"):
            getattr(lib, name).argtypes = [vp, vp, i, i, vp, vp, vp]
        lib.aeaj_percentile_thresholds.argtypes = [vp, vp, i, i, vp, vp, vp]
        lib.aeaj_canny_u8.argtypes = [vp, vp, i, i, vp, vp, vp, vp]
        lib.aeaj_canny.argtypes = [vp, vp, i, i, vp, vp, vp]
        lib.aeaj_quadtree_caps.argtypes = [i, i, i, i, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(i)]
        lib.aeaj_quadtree.argtypes = [vp, vp, i, i, i, i, vp, vp, vp, vp, vp]
        lib.aeaj_dct_quant.argtypes = [vp, vp, i, i, f, f, vp, vp, i, i, C.POINTER(vp), vp, vp, vp]
        lib.aeaj_dequant_idct.argtypes = [vp, vp, vp, vp, i, i, C.POINTER(vp), i, i, f, f, vp, vp, vp]
        lib.aeaj_plan_create.argtypes = [vp, i, i, i, i, i, i, C.POINTER(vp)]
        lib.aeaj_plan_destroy.argtypes = [vp]
        lib.aeaj_plan_get_info.argtypes = [vp, C.POINTER(PlanInfo)]
        lib.aeaj_plan_set_qtables.argtypes = [vp, vp, sz, vp]
        lib.aeaj_encode.argtypes = [vp, C.POINTER(EncodeIO), vp, vp]
        lib.aeaj_decode.argtypes = [vp, C.POINTER(DecodeIO), vp, vp]
        lib.aeaj_decode_scaled_geometry.argtypes = [vp, i, C.POINTER(i), C.POINTER(i), C.POINTER(i), C.POINTER(i), C.POINTER(C.c_int64)]
        lib.aeaj_decode_scaled.argtypes = [vp, C.POINTER(DecodeIO), i, vp, vp, vp]
        lib.aeaj_plan_last_launches.argtypes = [vp]
        lib.aeaj_plan_set_stream_layout.argtypes = [vp, i]
        lib.aeaj_plan_set_tensor_dct.argtypes = [vp, i]
        lib.aeaj_tensor_dct_status.argtypes = [vp, C.POINTER(i)]
        lib.aeaj_plan_enable_timing.argtypes = [vp, i]
        lib.aeaj_plan_read_timing.argtypes = [vp, C.c_char_p, sz, vp, i, C.POINTER(i)]
        lib.aeaj_states_to_leaves_host.argtypes = [vp, i, i, i, i, i, i, vp, C.POINTER(i), C.POINTER(C.c_int64)]
        lib.aeaj_pack_states_host.argtypes = [vp, i, vp]
        lib.aeaj_set_fast_transfer.argtypes = [vp, i]
        lib.aeaj_encode_halo.argtypes = [vp, C.POINTER(EncodeIO), vp, vp, i]
        lib.aeaj_decode_halo.argtypes = [vp, C.POINTER(DecodeIO), vp, vp, i]
        lib.aeaj_copy_segments.argtypes = [C.POINTER(Segment), i, vp, vp]
        lib.aeaj_peer_alloc.argtypes = [sz, C.POINTER(vp)]
        lib.aeaj_peer_free.argtypes = [vp]
        lib.aeaj_peer_export.argtypes = [vp, vp]
        lib.aeaj_peer_open.argtypes = [vp, C.POINTER(vp)]
        lib.aeaj_peer_close.argtypes = [vp]
        lib.aeaj_plan_set_peers.argtypes = [vp, i, i, C.POINTER(vp), C.POINTER(vp)]
        lib.aeaj_pack_coefficients.argtypes = [vp, C.POINTER(vp), vp, C.POINTER(PackedIO), vp, vp]
        lib.aeaj_unpack_coefficients.argtypes = [vp, C.POINTER(PackedIO), C.POINTER(vp), vp, vp]
        lib.aeaj_pack_coefficients_host.argtypes = [vp, C.c_int64, vp, vp, C.POINTER(C.c_int64), C.POINTER(i)]
        lib.aeaj_unpack_coefficients_host.argtypes = [vp, vp, C.c_int64, C.c_int64, vp]
        lib.aeaj_deflate_caps.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        lib.aeaj_deflate_coefficients.argtypes = [vp, C.POINTER(vp), vp, C.POINTER(DeflateIO), vp, vp]
        lib.aeaj_inflate_scratch_bytes.argtypes = [vp, C.c_int64, C.POINTER(C.c_int64)]
        lib.aeaj_inflate_coefficients.argtypes = [vp, C.POINTER(InflateIO), vp, C.c_int64, vp, vp]
        _lib = lib
        return lib


def check(rc: int, what: str = "libaeaj call"):
    if rc != 0:
        msg = load().aeaj_last_error().decode("utf-8", "replace")
        raise AeajError(f"{what} failed (code {rc}): {msg}")


_handles = {}


def handle(device: int = 0):
    """The per-device handle, created on first use with the host-derived colour tables uploaded."""
    lib = load()
    with _lock:
        if device in _handles:
            return _handles[device]
    h = C.c_void_p()
    check(lib.aeaj_create(device, C.byref(h)), "aeaj_create")
    keep = []
    for name, sid in tables.SPACE_ID.items():
        arrs = tables.color_tables(name)
        keep.append(arrs)
        check(lib.aeaj_set_color_tables(h, sid, *[a.ctypes.data for a in arrs]), "aeaj_set_color_tables")
    lut = tables.srgb_to_linear_lut()
    check(lib.aeaj_set_srgb_lut(h, lut.ctypes.data), "aeaj_set_srgb_lut")
    with _lock:
        _handles[device] = h
    return h


def states_to_leaves(states: np.ndarray, root: int, h: int, w: int, block_range=(0, 0)):
    """Host-side inverse of the state stream (jpeg.py:768-800 + 428-448): DFS pre-order 2-bit states
    -> (x, y, size, coefficient offset) per leaf.  Part of the entropy-decode side, runs on the host.
    The stream is untrusted: a root / leaf that does not fit the (h, w) layer or `block_range` raises ValueError."""
    lib = load()
    states = np.ascontiguousarray(states, dtype=np.uint8)
    leaves = np.empty((max(len(states), 1), 4), dtype=np.int32)
    n = C.c_int()
    ncoef = C.c_int64()
    rc = lib.aeaj_states_to_leaves_host(states.ctypes.data, len(states), int(root), int(h), int(w), int(block_range[0]), int(block_range[1]),
                                        leaves.ctypes.data, C.byref(n), C.byref(ncoef))
    if rc == -1:
        raise ValueError("corrupt quadtree header: " + lib.aeaj_last_error().decode("utf-8", "replace"))
    check(rc, "aeaj_states_to_leaves_host")
    return leaves[: n.value], int(ncoef.value)


def pack_coefficients_host(coef: np.ndarray):
    """int32 stream -> (mask uint32[ceil(n/32)], vals int16[nnz], overflow flag): the packed form of include/aeaj.h, on the CPU"""
    lib = load()
    coef = np.ascontiguousarray(coef, dtype=np.int32)
    mask = np.empty((coef.size + 31) // 32, dtype=np.uint32)
    vals = np.empty(max(coef.size, 1), dtype=np.int16)
    nnz, ovf = C.c_int64(), C.c_int()
    check(lib.aeaj_pack_coefficients_host(coef.ctypes.data, coef.size, mask.ctypes.data, vals.ctypes.data, C.byref(nnz), C.byref(ovf)),
          "aeaj_pack_coefficients_host")
    return mask, vals[: nnz.value], bool(ovf.value)


def unpack_coefficients_host(mask: np.ndarray, vals: np.ndarray, n_coef: int) -> np.ndarray:
    """inverse of the packed form: -> int32 stream of n_coef coefficients (what the .ajpg container stores, jpeg.py:590)"""
    lib = load()
    mask = np.ascontiguousarray(mask, dtype=np.uint32)
    vals = np.ascontiguousarray(vals, dtype=np.int16)
    if mask.size < (n_coef + 31) // 32:
        raise ValueError("packed stream: mask too short")
    out = np.empty(n_coef, dtype=np.int32)
    rc = lib.aeaj_unpack_coefficients_host(mask.ctypes.data, vals.ctypes.data, n_coef, vals.size, out.ctypes.data)
    if rc == -1:
        raise ValueError(lib.aeaj_last_error().decode("utf-8", "replace"))
    check(rc, "aeaj_unpack_coefficients_host")
    return out
