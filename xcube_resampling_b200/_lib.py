"""ctypes binding of ``libxrs.so`` (the C ABI declared in ``include/xrs.h``).

There is no CPU fallback: if the shared library is missing or cannot be loaded
the first call raises.  Build it with ``python -m xcube_resampling_b200.build``.
"""

from __future__ import annotations

import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# XRS_LIB selects an experimental build variant (build.py); the product library otherwise
LIB_PATH = os.environ.get("XRS_LIB") or os.path.join(_HERE, "libxrs.so")

c_int = ctypes.c_int
c_i32 = ctypes.c_int32
c_i64 = ctypes.c_int64
c_f64 = ctypes.c_double
c_p = ctypes.c_void_p


class XrsError(RuntimeError):
    """A libxrs call returned a non-zero status."""


class XrsProj(ctypes.Structure):
    """``struct xrs_proj`` of include/xrs.h."""

    _fields_ = [("kind", c_i32), ("_pad", c_i32), ("a", c_f64), ("inv_f", c_f64), ("lon0", c_f64),
                ("lat0", c_f64), ("k0", c_f64), ("fe", c_f64), ("fn", c_f64)]

    @classmethod
    def from_crs(cls, crs) -> "XrsProj":
        kind, a, inv_f, lon0, lat0, k0, fe, fn = crs.proj_params()
        return cls(kind, 0, a, inv_f, lon0, lat0, k0, fe, fn)


class XrsZarrCF(ctypes.Structure):
    """``struct xrs_zarr_cf`` of include/xrs.h."""

    MAX_FILLS = 16
    _fields_ = [("out_dtype", c_i32), ("n_fills", c_i32), ("has_scale", c_i32), ("has_offset", c_i32),
                ("scale", c_f64), ("offset", c_f64), ("fills", ctypes.c_uint64 * MAX_FILLS)]

    @classmethod
    def from_params(cls, out_dtype: int, fills, scale, offset) -> "XrsZarrCF":
        """``fills``: numpy array of the stored type; ``scale`` / ``offset``: ``None`` when absent."""
        cf = cls(out_dtype, len(fills), scale is not None, offset is not None, scale or 0.0, offset or 0.0)
        for k, f in enumerate(fills):
            cf.fills[k] = int.from_bytes(f.tobytes(), "little")
        return cf


# name -> (restype, argtypes); must list every symbol of include/xrs.h
SIGNATURES = {
    "xrs_version": (c_int, []),
    "xrs_device_count": (c_int, []),
    "xrs_last_error": (ctypes.c_char_p, []),
    "xrs_launch_count": (ctypes.c_uint64, []),
    "xrs_profile_enable": (c_int, [c_i32]),
    "xrs_profile_collect": (c_i32, [c_p, c_i64, c_p, c_p, c_i32]),
    "xrs_tile_src_bboxes_workspace_bytes": (c_i64, [c_i32, c_i32]),
    "xrs_tile_src_bboxes": (c_int, [c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p, c_i32, c_p, c_p, c_i32, c_i32, c_p,
                                    c_p, c_p]),
    "xrs_rectify_ij_workspace_bytes": (c_i64, [c_i64, c_i64, c_i64, c_i64]),
    "xrs_rectify_ij": (c_int, [c_p, c_p, c_i64, c_i64, c_i64, c_p, c_p, c_i64, c_i64, c_i32, c_i32, c_f64, c_f64,
                               c_f64, c_f64, c_f64, c_i32, c_f64, c_i64, c_i64, c_p, c_p, c_p]),
    "xrs_gather_ij": (c_int, [c_p, c_p, c_i32, c_i32, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_p, c_i64,
                              c_i64, c_i32, c_f64, c_p]),
    "xrs_gather_ij2": (c_int, [c_p, c_p, c_p, c_i32, c_i32, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_p, c_i64,
                               c_i64, c_i32, c_f64, c_f64, c_p]),
    "xrs_rectify_gather": (c_int, [c_p, c_p, c_i64, c_i64, c_i64, c_p, c_i64, c_i64, c_i32, c_i32, c_f64, c_f64, c_f64,
                                   c_f64, c_f64, c_i32, c_f64, c_i64, c_i64, c_p, c_p, c_p, c_p, c_i32, c_i32, c_i64, c_i64,
                                   c_i64, c_i64, c_i64, c_i32, c_f64, c_p]),
    "xrs_minform_init": (c_int, [c_p, c_i64, c_p]),
    "xrs_tile_src_bboxes_partial": (c_int, [c_p, c_p, c_i64, c_i64, c_i64, c_i64, c_p, c_p, c_i32, c_p, c_p, c_i32,
                                            c_p, c_p, c_p]),
    "xrs_tile_src_bboxes_finalize": (c_int, [c_p, c_i32, c_i32, c_i64, c_i64, c_p, c_p]),
    "xrs_quad_row_group": (c_i32, []),
    "xrs_band_quad_footprints": (c_int, [c_p, c_p, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_f64, c_f64,
                                         c_f64, c_f64, c_f64, c_i32, c_p, c_i32, c_p, c_p]),
    "xrs_coords_stats": (c_int, [c_p, c_p, c_i64, c_i64, c_i64, c_i32, c_p, c_p]),
    "xrs_lon_360": (c_int, [c_p, c_i64, c_i64, c_i64, c_p]),
    "xrs_copy2d_slices": (c_int, [c_p, c_i64, c_i64, c_p, c_i64, c_i64, c_i64, c_i64, c_i64, c_p]),
    "xrs_transform_points": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_p]),
    "xrs_reproject": (c_int, [c_p, c_p, c_i32, c_i32, c_i32, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_p, c_p,
                              c_p, c_p, c_i64, c_i64, c_i32, c_i32, c_p, c_p, c_p, c_p, c_i32, c_i32, c_f64, c_f64,
                              c_i32, c_f64, c_i64, c_i64, c_p]),
    "xrs_affine": (c_int, [c_p, c_p, c_i32, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_f64, c_f64, c_f64, c_f64,
                           c_i32, c_f64, c_i32, c_i32, c_i32, c_i32, c_p]),
    "xrs_has_nan": (c_int, [c_p, c_i32, c_i64, c_i64, c_i64, c_i64, c_i64, c_p, c_p]),
    "xrs_affine_recover": (c_int, [c_p, c_p, c_i32, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_f64, c_f64, c_f64,
                                   c_f64, c_f64, c_i32, c_i32, c_i32, c_i32, c_p]),
    "xrs_coarsen": (c_int, [c_p, c_p, c_i32, c_i64, c_i64, c_i64, c_i64, c_i64, c_i32, c_i32, c_i32, c_p]),
    "xrs_zarr_decode_workspace_bytes": (c_i64, [c_p, c_i64, c_i64, c_i64, c_i64, c_i32]),
    "xrs_zarr_decode": (c_int, [c_p, c_i64, c_p, c_i64, c_i64, c_i64, c_i64, c_i32, c_i32, ctypes.c_uint64, c_p, c_i64,
                                c_i64, c_p, c_i64, c_i64, c_i64, c_i64, c_i64, c_i64, c_p, c_i64, c_p, c_p]),
}

_lock = threading.Lock()
_lib = None


def load() -> ctypes.CDLL:
    """Load libxrs.so (once) and type every entry point.  Fails loudly."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise XrsError(
                f"{LIB_PATH} not found: the CUDA extension is not built. Run "
                "`python -m xcube_resampling_b200.build` (needs nvcc); there is no CPU fallback."
            )
        lib = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is missing
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
        return lib


def check(rc: int, what: str = "libxrs call"):
    if rc != 0:
        msg = load().xrs_last_error().decode("utf-8", "replace")
        raise XrsError(f"{what} failed (status {rc}): {msg}")


def profile_enable(on: bool):
    """Switch per-kernel event timing of libxrs on or off (include/xrs.h: xrs_profile_enable)."""
    load().xrs_profile_enable(1 if on else 0)


def profile_collect() -> dict:
    """{kernel name: (total ms, launches)} since the last collect; waits for the kernels."""
    lib = load()
    n_max = 64
    names = ctypes.create_string_buffer(4096)
    ms = (ctypes.c_double * n_max)()
    cnt = (ctypes.c_int64 * n_max)()
    n = lib.xrs_profile_collect(ctypes.cast(names, c_p), 4096, ctypes.cast(ms, c_p), ctypes.cast(cnt, c_p), n_max)
    keys = names.value.decode().split("\n")[:n]
    return {k: (ms[i], cnt[i]) for i, k in enumerate(keys)}
