"""ctypes binding of the C-ABI library (include/gf_b200.h).

The product path has NO fallback: if ``libgf_b200.so`` is missing or fails to load, importing an
op raises.  Build it with ``python -m gaussianformer_b200.csrc.build`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_size_t, c_uint32, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# GF_B200_LIB: developer override to A/B an alternative build of the same library (tools/build_variant.py)
LIB_PATH = os.environ.get("GF_B200_LIB") or os.path.join(_HERE, "csrc", "libgf_b200.so")

GF_OK = 0
GF_SPLAT_BASE, GF_SPLAT_PROB = 0, 1
GF_FLAG_POINT_OUT_OF_GRID = 1
GF_FLAG_MEAN_OUT_OF_GRID = 2
GF_FLAG_RADIUS_LT_1 = 4
GF_FLAG_GENERIC_PATH = 256

DEBUG_EXPORTS = ("gf_debug_set_render_events", "gf_debug_gather_probe", "gf_debug_daf_forward_tma")   # include/gf_b200_debug.h: measurement hooks, not the drop-in boundary
EXPORTS = (
    "gf_abi_version", "gf_last_error", "gf_splat_supported_classes",
    "gf_splat_forward_workspace_bytes", "gf_splat_backward_workspace_bytes",
    "gf_splat_forward", "gf_splat_backward", "gf_splat_read_flags",
    "gf_daf_forward", "gf_daf_backward", "gf_daf_format", "gf_splat_ce_partials",
    "gf_daf_fused_supported", "gf_daf_fused_forward", "gf_daf_fused_backward",
    "gf_occ_loss_workspace_bytes", "gf_occ_loss_forward",
)
GF_OCC_LABEL_OUT_OF_RANGE = 1


class SplatDesc(Structure):
    _fields_ = [("G", c_int32), ("N", c_int32), ("C", c_int32), ("H", c_int32), ("W", c_int32), ("D", c_int32),
                ("variant", c_int32), ("radii_axes", c_int32), ("cov_stride", c_int32),
                ("pc_min", c_float * 3), ("grid_size", c_float), ("scale_multiplier", c_float),
                ("radii_min", c_int32), ("batch", c_int32), ("pts_shared", c_int32)]


class SplatInputs(Structure):
    _fields_ = [("pts", c_void_p), ("points_int", c_void_p), ("means", c_void_p), ("means_int", c_void_p),
                ("opacities", c_void_p), ("semantics", c_void_p), ("cov", c_void_p), ("radii", c_void_p),
                ("scales", c_void_p), ("rotations", c_void_p)]


class SplatOutputs(Structure):
    _fields_ = [("logits", c_void_p), ("bin_logits", c_void_p), ("density", c_void_p), ("probability", c_void_p),
                ("argmax", c_void_p), ("logits_cn", c_void_p), ("labels", c_void_p), ("class_weights", c_void_p),
                ("ce_partials", c_void_p)]


class SplatGrads(Structure):
    _fields_ = [("logits_grad", c_void_p), ("bin_logits_grad", c_void_p), ("density_grad", c_void_p),
                ("logits", c_void_p), ("bin_logits", c_void_p), ("probability", c_void_p),
                ("means_grad", c_void_p), ("opacity_grad", c_void_p), ("semantics_grad", c_void_p),
                ("cov_grad", c_void_p), ("scales_grad", c_void_p), ("rotations_grad", c_void_p)]


class DafDesc(Structure):
    _fields_ = [("batch", c_int32), ("num_cams", c_int32), ("num_feat", c_int32), ("num_embeds", c_int32),
                ("num_scale", c_int32), ("num_pts", c_int32), ("num_groups", c_int32)]


class DafFusedDesc(Structure):
    _fields_ = [("d", DafDesc), ("pts_per_anchor", c_int32)]


DAF_MAX_LEVELS = 8


class DafFormatDesc(Structure):
    _fields_ = [("batch_cams", c_int32), ("num_embeds", c_int32), ("num_scale", c_int32),
                ("hw", c_int32 * DAF_MAX_LEVELS)]


class OccLossDesc(Structure):
    _fields_ = [("B", c_int32), ("N", c_int32), ("C", c_int32), ("use_softmax", c_int32), ("ignore_index", c_int32),
                ("lovasz_ignore", c_int32), ("ignore_empty", c_int32), ("empty_label", c_int32),
                ("ce_weight", c_float), ("lovasz_weight", c_float), ("lovasz", c_int32)]


class GfError(RuntimeError):
    pass


_lib = None


def lib():
    """The loaded library; raises (never falls back) when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built "
                "(run `python -m gaussianformer_b200.csrc.build`). There is no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        L.gf_abi_version.restype = c_int
        L.gf_last_error.restype = c_char_p
        L.gf_splat_supported_classes.argtypes = [POINTER(c_int32), c_int]
        L.gf_splat_forward_workspace_bytes.restype = c_size_t
        L.gf_splat_forward_workspace_bytes.argtypes = [POINTER(SplatDesc)]
        L.gf_splat_backward_workspace_bytes.restype = c_size_t
        L.gf_splat_backward_workspace_bytes.argtypes = [POINTER(SplatDesc)]
        L.gf_splat_forward.argtypes = [POINTER(SplatDesc), POINTER(SplatInputs), POINTER(SplatOutputs), c_void_p,
                                       c_size_t, c_void_p]
        L.gf_splat_backward.argtypes = [POINTER(SplatDesc), POINTER(SplatInputs), POINTER(SplatGrads), c_void_p,
                                        c_size_t, c_void_p]
        L.gf_splat_read_flags.argtypes = [c_void_p, c_void_p, POINTER(c_uint32)]
        L.gf_debug_set_render_events.argtypes = [c_void_p, c_void_p]
        L.gf_debug_gather_probe.argtypes = [c_void_p, c_void_p, ctypes.c_int64, c_int32, c_void_p, c_void_p]
        L.gf_debug_daf_forward_tma.argtypes = [POINTER(DafDesc), c_void_p, POINTER(c_int32), POINTER(c_int32), c_void_p, c_void_p,
                                               c_void_p, c_void_p]
        L.gf_splat_ce_partials.argtypes = [POINTER(SplatDesc)]
        L.gf_splat_ce_partials.restype = c_int
        L.gf_daf_forward.argtypes = [POINTER(DafDesc)] + [c_void_p] * 7
        L.gf_daf_backward.argtypes = [POINTER(DafDesc)] + [c_void_p] * 10
        L.gf_daf_fused_supported.argtypes = [POINTER(DafFusedDesc)]
        L.gf_daf_fused_forward.argtypes = [POINTER(DafFusedDesc)] + [c_void_p] * 10
        L.gf_daf_fused_backward.argtypes = [POINTER(DafFusedDesc)] + [c_void_p] * 14
        L.gf_daf_format.argtypes = [POINTER(DafFormatDesc), POINTER(c_void_p), c_void_p, c_int, c_void_p]
        L.gf_occ_loss_workspace_bytes.restype = c_size_t
        L.gf_occ_loss_workspace_bytes.argtypes = [POINTER(OccLossDesc)]
        L.gf_occ_loss_forward.argtypes = [POINTER(OccLossDesc)] + [c_void_p] * 8 + [c_size_t, c_void_p]
        if L.gf_abi_version() != 2:
            raise ImportError("libgf_b200.so: ABI version mismatch")
        _lib = L
    return _lib


def check(rc: int):
    if rc != GF_OK:
        raise GfError(f"gf_b200 error {rc}: {lib().gf_last_error().decode()}")


def supported_classes():
    buf = (c_int32 * 32)()
    n = lib().gf_splat_supported_classes(buf, 32)
    return [int(buf[i]) for i in range(n)]
