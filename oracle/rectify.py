"""Oracle restatement of the rectify path (test infrastructure only).

Follows ``rectify.py:312-419`` (tile loop, xy_border, tile-local offsets),
``gridmapping/base.py:565-629`` + ``gridmapping/bboxes.py:28-106`` (source
windows) and ``rectify.py:579-734`` (gather).  The per-pixel arithmetic lives
in ``xrs_oracle.c``.
"""

import numpy as np

from ._lib import lib, ptr
from .grid import RegularGrid, tile_xy_bboxes

UV_DELTA = 1e-3  # constants.py:80

METHODS = {"nearest": 0, "bilinear": 1, "triangular": 2, 0: 0, 1: 1}

DTYPE_CODES = {
    np.dtype(np.float32): 0, np.dtype(np.float64): 1, np.dtype(np.uint8): 2, np.dtype(np.int8): 3,
    np.dtype(np.uint16): 4, np.dtype(np.int16): 5, np.dtype(np.int32): 6, np.dtype(np.uint32): 7,
    np.dtype(np.int64): 8,
}


def ij_bboxes(x, y, xy_boxes, xy_border=0.0, ij_border=0):
    """gridmapping/bboxes.py:28-106 via gridmapping/base.py:565-629."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    xy_boxes = np.ascontiguousarray(xy_boxes, dtype=np.float64)
    out = np.full(xy_boxes.shape, -1, dtype=np.int64)
    h, w = x.shape
    lib().xrso_ij_bboxes(ptr(x), ptr(y), h, w, ptr(xy_boxes), xy_boxes.shape[0], float(xy_border),
                         int(ij_border), ptr(out))
    return out


def xy_border_for(g: RegularGrid) -> float:
    """rectify.py:329-340."""
    num_tiles_x = g.width / g.tile_w
    num_tiles_y = g.height / g.tile_h
    return min(
        min(2 * num_tiles_x * g.x_res, 2 * num_tiles_y * g.y_res),
        min(0.5 * (g.x_max - g.x_min), 0.5 * (g.y_max - g.y_min)),
    )


def source_windows(x, y, g: RegularGrid) -> np.ndarray:
    """rectify.py:342-345: per-tile source ij boxes, ij_border=1."""
    return ij_bboxes(x, y, tile_xy_bboxes(g), xy_border=xy_border_for(g), ij_border=1)


def rectify_ij(x, y, g: RegularGrid, uv_delta: float = UV_DELTA, windows=None) -> np.ndarray:
    """rectify.py:312-419: the (2, H, W) float64 source-index image."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    if windows is None:
        windows = source_windows(x, y, g)
    windows = np.ascontiguousarray(windows, dtype=np.int64)
    out = np.empty((2, g.height, g.width), dtype=np.float64)
    h, w = x.shape
    lib().xrso_rectify_ij(ptr(x), ptr(y), h, w, ptr(windows), ptr(out), g.height, g.width, g.tile_h, g.tile_w,
                          float(g.x_min), float(g.y_min), float(g.y_max), float(g.x_res), float(g.y_res),
                          int(g.is_j_axis_up), float(uv_delta))
    return out


def rectify_ij_block(x_win, y_win, src_i_min, src_j_min, dst_h, dst_w, x_off, y_off, x_scale, y_scale,
                     uv_delta=UV_DELTA) -> np.ndarray:
    """rectify.py:424-576 on one tile (same argument meaning as the numba kernel)."""
    x_win = np.ascontiguousarray(x_win, dtype=np.float64)
    y_win = np.ascontiguousarray(y_win, dtype=np.float64)
    out = np.empty((2, dst_h, dst_w), dtype=np.float64)
    wh, ww = x_win.shape
    lib().xrso_rectify_ij_block(ptr(x_win), ptr(y_win), wh, ww, ww, int(src_i_min), int(src_j_min), ptr(out),
                                dst_h, dst_w, dst_w, dst_h * dst_w, float(x_off), float(y_off), float(x_scale),
                                float(y_scale), float(uv_delta))
    return out


def _full(shape, fill_value, dtype) -> np.ndarray:
    """rectify.py:618,621: ``np.full(shape, fill_value, dtype=src dtype)``.  numpy 2 refuses a Python int outside the
    dtype's range -- the default integer fill -1 (utils.py:307-316) of a uint32 variable raises OverflowError -- where
    numpy 1.x wrapped it modulo 2**bits (-1 -> 0xFFFFFFFF); this returns numpy 1.x's value."""
    try:
        return np.full(shape, fill_value, dtype=dtype)
    except OverflowError:
        return np.full(shape, np.array(fill_value).astype(dtype), dtype=dtype)


def gather(src, ij, method, fill_value) -> np.ndarray:
    """rectify.py:579-734: (bands, h, w) or (h, w) source -> target via the ij image."""
    if method not in METHODS:
        raise NotImplementedError(
            f"interp_methods must be one of 0, 1, 'nearest', 'bilinear', 'triangular', was '{method}'."
        )
    src = np.asarray(src)
    squeeze = src.ndim == 2
    src3 = np.ascontiguousarray(src[None] if squeeze else src)
    code = DTYPE_CODES[src3.dtype]
    ij = np.ascontiguousarray(ij, dtype=np.float64)
    bands, sh, sw = src3.shape
    _, dh, dw = ij.shape
    out = _full((bands, dh, dw), fill_value, src3.dtype)
    rc = lib().xrso_gather_ij(ptr(src3), code, bands, sh, sw, ptr(ij), ptr(out), dh, dw, METHODS[method])
    assert rc == 0
    return out[0] if squeeze else out


def rectify(x, y, src, g: RegularGrid, method, fill_value, uv_delta=UV_DELTA):
    """ij image + gather: what rectify_dataset computes per variable (rectify.py:146,159-174)."""
    ij = rectify_ij(x, y, g, uv_delta)
    return gather(src, ij, method, fill_value), ij
