"""ctypes binding of ``liboctm.so`` (the C ABI declared in ``include/octm.h``).

There is NO CPU fallback: if the CUDA library is missing, cannot be loaded, or a call fails, an
exception is raised.  ``python -m retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build``
(or ``__graft_entry__.build()``) compiles it in-tree for sm_100a.
"""
from __future__ import annotations

import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "liboctm.so")

OK = 0
NO_SEED = 0xFFFFFFFF
CF_TRUE_CLOSED, CF_PRED_CLOSED, CF_TRUE_OVERFLOW, CF_PRED_OVERFLOW = 1, 2, 4, 8
# column order of the device-derived per-class metrics (OCTM_M_* in include/octm.h)
CLASS_METRICS = ("accuracy", "sensitivity", "cm_precision", "specificity", "dice_coefficient", "iou_score",
                 "region_precision", "recall", "mean_squared_error", "root_mean_squared_error", "mad",
                 "vascularity_index", "thickness_difference", "hausdorff_distance", "hausdorff_distance_95", "assd")
BOUNDARY_METRICS = ("boundary_mse", "boundary_rmse", "boundary_mad")
DTYPE_F32, DTYPE_F16, DTYPE_BF16, DTYPE_F64, DTYPE_I32 = 0, 1, 2, 3, 4

_c = ctypes
_P = _c.c_void_p
_I64 = _c.c_int64
_INT = _c.c_int

# name -> (restype, argtypes); mirrors include/octm.h one to one (tests/test_abi.py checks that)
SIGNATURES = {
    "octm_abi_version": (_INT, []),
    "octm_last_error": (_c.c_char_p, []),
    "octm_launch_count": (_c.c_uint64, []),
    "octm_profile_enable": (_INT, [_INT]),
    "octm_profile_report": (_c.c_size_t, [_c.c_char_p, _c.c_size_t]),
    "octm_confusion_u8": (_INT, [_P, _P, _I64, _I64, _INT, _P, _P]),
    "octm_column_scan_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _P, _P, _P, _P, _P, _P]),
    "octm_boundary_error_i32": (_INT, [_P, _P, _I64, _INT, _INT, _P, _P, _P]),
    "octm_label_pass_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _P, _P, _P, _P, _P, _P, _P, _P]),
    "octm_label_pass_sorted_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "octm_label_pass_path": (_INT, [_INT, _INT, _INT, _P, _P]),
    "octm_label_pass_seed_policy": (_INT, [_INT]),
    "octm_validate_labels_u8": (_INT, [_P, _I64, _P, _P]),
    "octm_contour2d_workspace_bytes": (_c.c_size_t, [_I64, _INT, _INT, _INT, _INT]),
    "octm_contour2d_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _P, _INT, _P, _P, _P, _P, _P, _P, _c.c_size_t, _P]),
    "octm_contour2d_metrics_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _P, _P, _P, _P, _INT, _P, _P, _P, _P, _P, _P, _c.c_size_t, _P]),
    "octm_first_pos_u8": (_INT, [_P, _I64, _I64, _INT, _P, _P]),
    "octm_contour2d_trace_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _P, _P, _P, _INT, _P, _P, _P, _P]),
    "octm_contour2d_distance": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _INT, _P, _P, _P, _P, _INT, _P]),
    "octm_contour2d_distance_spacing": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _INT, _P, _P, _P, _P, _P, _INT, _P]),
    "octm_contour2d_all_vertices_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _INT, _P, _P, _P, _P]),
    "octm_contour2d_all_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _INT, _P, _P, _P, _P, _P, _P, _c.c_size_t, _P]),
    "octm_surface_dice_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _P, _INT, _P, _P, _P]),
    "octm_surface_dice_spacing_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _P, _P, _INT, _P, _P, _P]),
    "octm_components_u8": (_INT, [_P, _P, _I64, _INT, _INT, _INT, _INT, _P, _P, _P]),
    "octm_argmax_labels": (_INT, [_P, _INT, _I64, _INT, _I64, _INT, _P, _P]),
    "octm_auc_workspace_bytes": (_c.c_size_t, [_I64, _I64, _INT]),
    "octm_auc_u8": (_INT, [_P, _P, _INT, _I64, _I64, _c.c_double, _P, _P, _c.c_size_t, _P]),
    "octm_boundary_error_float": (_INT, [_P, _P, _INT, _I64, _INT, _I64, _P, _P, _P]),
    "octm_topology_violations_float": (_INT, [_P, _INT, _I64, _INT, _I64, _P, _P, _P]),
    "octm_surface3d_workspace_bytes": (_c.c_size_t, [_INT, _INT, _INT]),
    "octm_surface3d_u8": (_INT, [_P, _P, _INT, _INT, _INT, _INT, _INT, _INT, _P, _P, _P, _P, _P, _c.c_size_t, _P]),
    "octm_surface3d_spacing_workspace_bytes": (_c.c_size_t, [_INT, _INT, _INT]),
    "octm_surface3d_spacing_u8": (_INT, [_P, _P, _INT, _INT, _INT, _INT, _INT, _INT, _P, _P, _INT, _P, _P, _P, _P, _P, _P,
                                         _P, _c.c_size_t, _P]),
    "octm_host_pack_nibbles": (_INT, [_P, _P, _c.c_size_t, _INT]),
    "octm_unpack_nibbles_u8": (_INT, [_P, _I64, _P, _P]),
    "octm_labels_from_boundaries": (_INT, [_P, _INT, _I64, _INT, _INT, _INT, _P, _P]),
    "octm_totals_len": (_INT, [_INT]),
    "octm_totals_sum_len": (_INT, [_INT]),
    "octm_derive_metrics": (_INT, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _INT, _INT, _INT, _P, _P, _P, _P]),
    "octm_derive_metrics_spacing": (_INT, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _INT, _INT, _INT, _P, _P, _P, _P,
                                           _P]),
}

_lib = None


class OctmError(RuntimeError):
    """A liboctm entry point returned a negative status."""


def load():
    """Load liboctm.so once; raises if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run "
            "`python -m retinal_oct_image_segmentation_via_deep_learning_b200.csrc.build`. "
            "This package has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.octm_abi_version() != 1:
        raise RuntimeError("liboctm.so ABI version mismatch; rebuild it")
    _lib = lib
    return lib


def call(name, *args):
    """Invoke an int-returning entry point; raise OctmError with the library's message on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != OK:
        raise OctmError(f"{name} failed ({rc}): {lib.octm_last_error().decode(errors='replace')}")
    return rc


def launch_count():
    return int(load().octm_launch_count())


class kernel_profile:
    """``with kernel_profile() as prof: ...`` -> ``prof.kernels`` = {kernel: (launches, total ms)} of every liboctm
    kernel launched inside the block (CUDA events on the launch streams; for benchmarks, outside timed regions)."""

    def __enter__(self):
        load().octm_profile_enable(1)
        self.kernels = {}
        return self

    def __exit__(self, *exc):
        lib = load()
        buf = ctypes.create_string_buffer(1 << 16)
        lib.octm_profile_report(buf, len(buf))
        for line in buf.value.decode().splitlines():
            name, n, ms = line.split()
            self.kernels[name] = (int(n), float(ms))
        lib.octm_profile_enable(0)
        return False
