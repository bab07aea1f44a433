"""Shared test helpers: golden loading, synthetic swaths, oracle grids."""

import hashlib
import os

import numpy as np

from oracle import grid as ogrid

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def grid_from_golden(vec) -> ogrid.RegularGrid:
    w, h, tw, th, x_min, y_min, x_max, y_max, x_res, y_res, j_up = vec
    return ogrid.RegularGrid(int(w), int(h), int(tw), int(th), float(x_min), float(y_min), float(x_max),
                             float(y_max), float(x_res), float(y_res), bool(j_up))


from xcube_resampling_b200.synthetic import covering_grid_args, swath  # noqa: E402,F401


def assert_same(a, b, what=""):
    """Bit-exact comparison with NaN == NaN."""
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} != {b.shape}"
    assert a.dtype == b.dtype, f"{what}: dtype {a.dtype} != {b.dtype}"
    if not np.array_equal(a, b, equal_nan=a.dtype.kind == "f"):
        bad = ~((a == b) | ((a != a) & (b != b))) if a.dtype.kind == "f" else (a != b)
        idx = np.argwhere(bad)[:5]
        raise AssertionError(f"{what}: {bad.sum()} of {a.size} elements differ, first at {idx.tolist()}: "
                             f"{a[bad][:5]} vs {b[bad][:5]}")


def assert_bits(a, b, what="", skip=None):
    """Equal dtypes, shapes and bit patterns, every NaN taken as one NaN: unlike ``assert_same`` the sign of zero
    counts.  ``skip``: boolean mask of elements left out (only for documented deviations)."""
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} != {b.shape}"
    assert a.dtype == b.dtype, f"{what}: dtype {a.dtype} != {b.dtype}"
    ua, ub = (np.ascontiguousarray(x).view(f"u{a.dtype.itemsize}") for x in (a, b))
    if a.dtype.kind == "f":
        canon = np.array([np.nan], dtype=a.dtype).view(ua.dtype)[0]
        ua, ub = np.where(np.isnan(a), canon, ua), np.where(np.isnan(b), canon, ub)
    bad = ua != ub
    if skip is not None:
        bad &= ~np.asarray(skip, dtype=bool)
    if bad.any():
        idx = np.argwhere(bad)[:5]
        raise AssertionError(f"{what}: {bad.sum()} of {a.size} elements differ, first at {idx.tolist()}: "
                             f"{a[bad][:5]} vs {b[bad][:5]}")


def digest(a) -> str:
    """64-bit SHA-256 prefix of dtype, shape and values; every NaN hashes as one NaN and -0.0 as 0.0, so
    equal digests stand for ``assert_same``: equal dtypes, shapes and ``np.array_equal(..., equal_nan=True)``."""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a + 0).astype(a.dtype, copy=False)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()[:16]


def dual_swath():
    """(x, y, grid, bands) on which tests/test_oracle_dual.py holds the two-method gather against the
    reference's kernels (tests/golden/dual_swath_digests.json, written by make_golden.py)."""
    x, y = swath(220, 180, theta=20.0, seed=5)
    res = 0.0027
    size, xy_min = covering_grid_args(x, y, res)
    g = ogrid.regular_grid(size, xy_min, res, tile_size=64)
    data = np.random.default_rng(5).random((3, 180, 220)).astype(np.float32)
    data[1, 60:70, 80:120] = np.nan
    return x, y, g, data


INT32_MAX = np.iinfo(np.int32).max


def quad_footprints_np(x, y, g, band_edges, group=32, rows=None):
    """numpy restatement of ``xrs_band_quad_footprints`` (csrc/bands.cu) -- our own partition logic,
    not reference code: per target row band and per group of ``group`` source quad rows, the
    min-form (c_min, -c_max) over the quads whose grown pixel box overlaps the band.  ``rows``
    restricts the scan to the quad rows of vertex rows [rows[0], rows[1]) (a slab)."""
    h, w = x.shape
    n_bands = len(band_edges) - 1
    n_groups = -(-(h - 1) // group)
    out = np.full((n_bands, n_groups, 2), INT32_MAX, dtype=np.int32)
    r0, r1 = (0, h) if rows is None else rows
    inv_xr, inv_yr = 1.0 / g.x_res, 1.0 / g.y_res
    with np.errstate(invalid="ignore", over="ignore"):
        fx = (x[r0:r1] - g.x_min) * inv_xr
        fy = (y[r0:r1] - g.y_min) * inv_yr if g.is_j_axis_up else (g.y_max - y[r0:r1]) * inv_yr
        ok = (np.abs(fx) < 1e15) & (np.abs(fy) < 1e15)
    corners = [(slice(0, -1), slice(0, -1)), (slice(0, -1), slice(1, None)), (slice(1, None), slice(0, -1)),
               (slice(1, None), slice(1, None))]
    n_ok = sum(ok[c].astype(np.int32) for c in corners)
    lo_x = np.minimum.reduce([np.where(ok[c], fx[c], np.inf) for c in corners])
    hi_x = np.maximum.reduce([np.where(ok[c], fx[c], -np.inf) for c in corners])
    lo_y = np.minimum.reduce([np.where(ok[c], fy[c], np.inf) for c in corners])
    hi_y = np.maximum.reduce([np.where(ok[c], fy[c], -np.inf) for c in corners])
    with np.errstate(invalid="ignore"):
        mrg = 2.0 + 0.01 * np.maximum(hi_x - lo_x, hi_y - lo_y)
        lo_x, hi_x = np.floor(lo_x) - mrg, np.floor(hi_x) + mrg
        lo_y, hi_y = np.floor(lo_y) - mrg, np.floor(hi_y) + mrg
        hit = (n_ok >= 3) & (hi_x >= 0.0) & (lo_x < g.width) & (hi_y >= 0.0) & (lo_y < g.height)
        r_lo = np.where(hit, np.maximum(lo_y, 0.0), 0).astype(np.int64)
        r_hi = np.where(hit, np.minimum(hi_y, g.height - 1.0), -1).astype(np.int64)
    qj, qi = np.nonzero(hit)
    for b in range(n_bands):
        e0, e1 = band_edges[b], band_edges[b + 1]
        if e0 >= e1:
            continue
        sel = (r_lo[qj, qi] < e1) & (r_hi[qj, qi] >= e0)
        gj = (qj[sel] + r0) // group
        for gi in np.unique(gj):
            cols = qi[sel][gj == gi]
            out[b, gi, 0] = min(out[b, gi, 0], cols.min())
            out[b, gi, 1] = min(out[b, gi, 1], -cols.max())
    return out


def two_method_gather_np(src, ij, method):
    """numpy restatement of what ONE thread of ``k2_gather_dual`` (csrc/gather_dual.cu) does per band and
    pixel -- our own kernel's logic, not reference code: the four taps (i0, j0) .. (i1, j1) of the
    interpolated sample, the nearest sample PICKED among them (column i1 when u > 0.5, row j1 when
    v > 0.5), float64 arithmetic in the reference's order, one cast.  Returns (interp, nearest) with
    NaN / 0 where ij has no source (the caller applies its fill values)."""
    src = np.asarray(src)
    src3 = src[None] if src.ndim == 2 else src
    h, w = src3.shape[-2:]
    fi, fj = np.asarray(ij[0], dtype=np.float64), np.asarray(ij[1], dtype=np.float64)
    valid = ~(np.isnan(fi) | np.isnan(fj))
    fi0, fj0 = np.where(valid, fi, 0.0), np.where(valid, fj, 0.0)
    i0, j0 = fi0.astype(np.int64), fj0.astype(np.int64)
    u, v = fi0 - i0, fj0 - j0
    i1, j1 = np.minimum(np.maximum(i0 + 1, 0), w - 1), np.minimum(np.maximum(j0 + 1, 0), h - 1)
    right, lower = u > 0.5, v > 0.5
    r00, r01, r10, r11 = src3[:, j0, i0], src3[:, j0, i1], src3[:, j1, i0], src3[:, j1, i1]
    near = np.where(lower, np.where(right, r11, r10), np.where(right, r01, r00))
    v00, v01, v10, v11 = (a.astype(np.float64) for a in (r00, r01, r10, r11))
    with np.errstate(invalid="ignore", over="ignore"):
        if method == "bilinear":
            a = v00 + u * (v01 - v00)
            b = v10 + u * (v11 - v10)
            val = a + v * (b - a)
        elif method == "triangular":
            val = np.where(u + v < 1.0, v00 + u * (v01 - v00) + v * (v10 - v00),
                           v11 + (1.0 - u) * (v10 - v11) + (1.0 - v) * (v01 - v11))
        else:
            raise ValueError(method)
        if src3.dtype.kind == "f":
            interp = val.astype(src3.dtype)
        else:  # C cast: float64 -> int64 (truncation) -> T
            interp = np.where(valid, val, 0.0).astype(np.int64).astype(src3.dtype)
    return interp, near, valid


def hand_made_ij(smooth: bool, h, w, H, W):
    """ij planes with exact half-pixel fractions (ties keep the lower index, rectify.py:693-698), the
    last row / column (neighbour taps clamp at the image edge), zeros, NaN in one plane only.
    ``smooth``: neighbouring target pixels reach neighbouring source pixels (every tile's box fits the
    staging buffers); otherwise random positions (every tile takes the global-tap branch)."""
    rng = np.random.default_rng(4)
    if smooth:
        fi = np.clip(np.arange(W)[None, :] * 0.7 + rng.random((H, W)), 0, w - 1)
        fj = np.clip(np.arange(H)[:, None] * 0.6 + rng.random((H, W)), 0, h - 1)
    else:
        fi = rng.random((H, W)) * (w - 1)
        fj = rng.random((H, W)) * (h - 1)
    fi[::3, ::2] = np.minimum(np.floor(fi[::3, ::2]) + 0.5, w - 1)      # ties in i
    fj[1::3, ::2] = np.minimum(np.floor(fj[1::3, ::2]) + 0.5, h - 1)    # ties in j
    fi[:, W - 2:] = w - 1                                 # last column: i1 == i0
    fj[H - 2:, :] = h - 1                                 # last row: j1 == j0
    fi[40, W - 6:] = w - 1 - 0.25
    fj[H - 5, 10:20] = h - 1 - 0.75
    fi[:, :2] = 0.0
    fj[:2, :] = 0.0
    fi[20:24, 30:40] = np.nan
    fj[20:24, 30:40] = np.nan
    fi[30, 50] = np.nan                                      # NaN in one plane only: still "no source"
    fj[31, 51] = np.nan
    fi[32:64, 64:96] = np.nan                                # one whole 32x32 tile without a source (CTA early out)
    return np.stack([fi, fj])
