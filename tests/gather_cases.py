"""Cases of the gather family shared by the host build (test_host_k2k3_dtypes.py) and the GPU
(test_gather_reproject_dtypes_gpu.py): K2 (csrc/gather.cu, csrc/gather_dual.cu) through an ij image and K3
(csrc/reproject.cu) on an identity transform, every dtype at full range, with the oracle's answer
(oracle/rectify.py, oracle/reproject.py: rectify.py:579-734, reproject.py:268-530).

Values: half of the bands span the dtype's full range, the other half are drawn from its exact extremes
(INT64_MIN / MAX, 2^53 +- 1, UINT32_MAX, -128 / 127, +-0.0, NaN, +-inf, subnormals, +-FLT_MAX side by side, so
that bilinear samples overflow to inf or round to 2^63).  Geometries: ``hand_made_ij`` smooth (every tile copies
its source box into the staging buffers) and scattered (no tile does: the staged kernels take their global-tap
branch), a rotated swath through K1 (the fused kernel applies), a resident window with poison outside, 1 / 5 / 25
bands.  Fills per dtype, extremes included.

``skip`` masks the elements of a documented deviation (DESIGN.md section 5): an int64 fill beyond 2^53 reaches
the kernels as a double and is rounded.
"""

import dataclasses
import functools
import warnings
from unittest import mock

import numpy as np

from oracle import grid as ogrid
from oracle import rectify as orect
from oracle import reproject as orep
from oracle import proj as oproj

from .helpers import covering_grid_args, hand_made_ij, swath

nan, inf = np.nan, np.inf
DTYPES = (np.float32, np.float64, np.uint8, np.int8, np.uint16, np.int16, np.int32, np.uint32, np.int64)
METHODS = ("nearest", "bilinear", "triangular")
SRC_HW, DST_HW = (70, 96), (64, 80)   # hand_made_ij geometry


def extremes(dtype) -> np.ndarray:
    dt = np.dtype(dtype)
    if dt.kind == "f":
        fi = np.finfo(dt)
        tiny = fi.smallest_subnormal
        return np.array([0.0, -0.0, nan, inf, -inf, fi.max, -fi.max, fi.max, -fi.max, tiny, -tiny, fi.tiny, 1.0, -1.0],
                        dtype=dt)
    ii = np.iinfo(dt)
    v = [ii.min, ii.max, ii.min + 1, ii.max - 1, 0, 1]
    if dt == np.int64:
        v += [2**53 - 1, 2**53, 2**53 + 1, -(2**53) - 1, 2**63 - 512, 2**63 - 513, 2**62 + 1]
    if dt == np.uint32:
        v += [2**31, 2**31 - 1]
    if dt.kind == "i" and dt != np.int64:
        v += [-1]
    return np.array(v, dtype=dt)


def values(dtype, shape, rng, family: str) -> np.ndarray:
    """``full``: the whole range of the dtype (floats: magnitudes log-uniform over the normal range, both signs,
    a few specials); ``extremes``: drawn from :func:`extremes` only."""
    dt = np.dtype(dtype)
    if family == "extremes":
        return rng.choice(extremes(dt), size=shape)
    if dt.kind == "f":
        fi = np.finfo(dt)
        e = rng.uniform(np.log10(fi.tiny), np.log10(fi.max), shape)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            a = (np.where(rng.random(shape) < 0.5, -1.0, 1.0) * 10.0 ** e).astype(dt)
        a.ravel()[rng.choice(a.size, a.size // 50, replace=False)] = rng.choice(extremes(dt), a.size // 50)
        return a
    ii = np.iinfo(dt)
    return rng.integers(ii.min, ii.max, shape, dtype=dt, endpoint=True)


def source(dtype, n_bands, h, w, seed=0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    return np.stack([values(dtype, (h, w), rng, "extremes" if b % 2 else "full") for b in range(n_bands)])


def default_fill(dtype):
    """The product's default fill of a variable (utils.py:307-316): uint8 255, uint16 65535, other integers -1,
    floats NaN."""
    dt = np.dtype(dtype)
    return 255 if dt == np.uint8 else 65535 if dt == np.uint16 else -1 if dt.kind in "iu" else nan


def fills(dtype):
    """Fill values worth a case: the default, NaN (x86's conversion into integers), each extreme that a fill
    can take, and for int64 values beyond 2^53 (rounded: a documented deviation)."""
    dt = np.dtype(dtype)
    if dt.kind == "f":
        fi = np.finfo(dt)
        return [nan, -0.0, inf, -inf, float(fi.max), float(fi.smallest_subnormal)]
    ii = np.iinfo(dt)
    out = [default_fill(dt), nan, int(ii.min), int(ii.max), 0]
    if dt == np.int64:
        out += [2**53, 2**53 + 1, -(2**53) - 1]
    return list(dict.fromkeys(out))   # unsigned: the minimum is 0, the default may be the maximum


def fill_rounded(dtype, fill) -> bool:
    """The fill reaches the C ABI as float(fill): does that change it?  (int64 beyond 2^53, INT64_MAX)"""
    return np.dtype(dtype).kind in "iu" and isinstance(fill, int) and int(float(fill)) != fill


@dataclasses.dataclass
class GatherCase:
    id: str
    src: np.ndarray       # (bands, h, w), the full source image
    ij: np.ndarray        # (2, H, W) fractional source indices
    method: str
    fill: object          # as the user passes it; the C ABI gets float(fill)
    want: np.ndarray      # oracle: rectify.py's gather with `method`
    want_near: np.ndarray  # oracle with nearest and the same fill (the second output of the dual kernel)
    skip: object          # mask of elements left out (documented deviation) or None
    staged: str           # which branch the staged kernels take: "box" (some tiles stage their source box), "global"
    window: tuple = None  # (i0, j0, i1, j1): only this part of the source is resident, poison elsewhere
    swath: tuple = None   # (x, y, size, xy_min, res, tile): ij comes from K1 over these coordinates

    @property
    def resident(self) -> np.ndarray:
        """The source as the kernels see it: outside ``window`` every element is the dtype's largest value."""
        if self.window is None:
            return self.src
        i0, j0, i1, j1 = self.window
        dt = self.src.dtype
        poison = np.finfo(dt).max if dt.kind == "f" else np.iinfo(dt).max
        out = np.full_like(self.src, poison)
        out[:, j0:j1, i0:i1] = self.src[:, j0:j1, i0:i1]
        return out


def _case(id, src, ij, method, fill, staged, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)   # np.full of NaN into an integer dtype
        want = orect.gather(src, ij, method, fill)
        near = orect.gather(src, ij, "nearest", fill) if method != "nearest" else want
    skip = None
    if fill_rounded(src.dtype, fill):
        skip = np.broadcast_to(np.isnan(ij[0]) | np.isnan(ij[1]), want.shape)
    return GatherCase(id, src, ij, method, fill, want, near, skip, staged, **kw)


@functools.lru_cache(maxsize=None)
def _swath_scene():
    w, h = 120, 90
    x, y = swath(w, h, theta=20.0, seed=3)
    x[40:43, 30:60] = nan   # a hole: pixels without a source inside covered tiles
    res, tile = 0.0027, 64
    size, xy_min = covering_grid_args(x, y, res)
    g = ogrid.regular_grid(size, xy_min, res, tile_size=tile)
    return (x, y, size, xy_min, res, tile), orect.rectify_ij(x, y, g)


@functools.lru_cache(maxsize=None)
def gather_cases() -> tuple:
    (h, w), (H, W) = SRC_HW, DST_HW
    cases = []
    geo = {"smooth": hand_made_ij(True, h, w, H, W), "scattered": hand_made_ij(False, h, w, H, W)}
    sw, sw_ij = _swath_scene()
    for k, dt in enumerate(DTYPES):
        name = np.dtype(dt).name
        src = source(dt, 3, h, w, seed=10 + k)
        src_sw = source(dt, 3, 90, 120, seed=20 + k)
        for method in METHODS:
            for g, ij in geo.items():
                cases.append(_case(f"{name}-{method}-{g}", src, ij, method, default_fill(dt),
                                   "box" if g == "smooth" else "global"))
            cases.append(_case(f"{name}-{method}-swath", src_sw, sw_ij, method, default_fill(dt), "box", swath=sw))
        # a row band of the target that sees one corner of the swath: only that part of the source is resident
        band_ij = sw_ij[:, 0:30]
        fi, fj = band_ij
        win = (int(np.nanmin(fi)) // 32 * 32, int(np.nanmin(fj)), min(120, int(np.nanmax(fi)) + 2),
               min(90, int(np.nanmax(fj)) + 2))
        for method in ("nearest", "bilinear"):
            cases.append(_case(f"{name}-{method}-window", src_sw, band_ij, method, default_fill(dt), "box", window=win))
        for f in fills(dt):
            for method in ("nearest", "bilinear"):
                cases.append(_case(f"{name}-{method}-fill={f!r}", src, geo["smooth"], method, f, "box"))
    for dt in (np.float32, np.uint32, np.int8, np.int64):
        for nb in (1, 5, 25):
            src = source(dt, nb, h, w, seed=nb)
            for method in ("nearest", "bilinear"):
                cases.append(_case(f"{np.dtype(dt).name}-{method}-bands={nb}", src, geo["smooth"], method,
                                   default_fill(dt), "box"))
    return tuple(cases)


def gather_case_ids():
    return [c.id for c in gather_cases()]


def gather_case(case_id) -> GatherCase:
    return {c.id: c for c in gather_cases()}[case_id]


# ---------------------------------------------------------------------------
# K3 on an identity transform (geographic source, shifted / rescaled geographic target poking out of the source on
# two sides): the separable kernel, row-block form for bilinear, per-pixel blends, padding
# ---------------------------------------------------------------------------
@dataclasses.dataclass
class ReprojectCase:
    id: str
    src: np.ndarray
    method: str
    fill: object
    out_f64: bool     # bilinear: the reference's float64 result, else the source dtype
    tile: object
    want: np.ndarray
    skip: object = None   # uint32 results outside [0, 2^32) (documented deviation) or None


def reproject_grids(GridMapping, tile):
    """(source, target) GridMappings of the identity cases, built with the product's class."""
    src_gm = GridMapping.regular((90, 64), (10.0, 50.0), 0.01, "EPSG:4326")
    tgt_gm = GridMapping.regular((70, 53), (10.0 + 0.013 - 0.05, 50.0 - 0.021 - 0.03), 0.0113, "OGC:CRS84",
                                 tile_size=tile)
    return src_gm, tgt_gm


def reproject_fill(dtype):
    """In-range fills (the reference's np.pad refuses -1 for unsigned types and NaN for integers): the dtype's
    minimum for integers, so that a padded tap reads an extreme, NaN for floats."""
    dt = np.dtype(dtype)
    return nan if dt.kind == "f" else int(np.iinfo(dt).min) if dt.kind == "i" else int(np.iinfo(dt).max)


def _triangular_f64(xx, yy, window, x0, y0, x_res, y_res, method):
    """oracle.reproject.sample_window's triangular blend before its cast back to the window's dtype."""
    fx = (xx - np.float32(x0)) / x_res
    fy = (yy - np.float32(y0)) / -y_res
    i_lo, i_hi = np.floor(fx).astype(np.int64), np.ceil(fx).astype(np.int64)
    j_lo, j_hi = np.floor(fy).astype(np.int64), np.ceil(fy).astype(np.int64)
    u, v = fx - i_lo, fy - j_lo
    p00, p01 = window[:, j_lo, i_lo], window[:, j_lo, i_hi]
    p10, p11 = window[:, j_hi, i_lo], window[:, j_hi, i_hi]
    near = p00 + u * (p01 - p00) + v * (p10 - p00)
    far = p11 + (1.0 - u) * (p10 - p11) + (1.0 - v) * (p01 - p11)
    return np.where((u + v < 1.0)[None], near, far)


def _uint32_out_of_range(f64) -> np.ndarray:
    """Where a float64 result cast back to uint32 lies outside [0, 2^32): undefined in C, and numpy's result depends
    on its build (DESIGN.md section 5) -- a documented deviation."""
    with np.errstate(invalid="ignore"):
        return ~((f64 >= 0) & (f64 < 2.0**32))


@functools.lru_cache(maxsize=None)
def reproject_cases(GridMapping) -> tuple:
    cases = []
    geo = oproj.from_epsg(4326)
    for k, dt in enumerate(DTYPES):
        name = np.dtype(dt).name
        for tile in (None, (32, 16)):
            src_gm, tgt_gm = reproject_grids(GridMapping, tile)
            src = source(dt, 3, src_gm.height, src_gm.width, seed=40 + k)
            g = ogrid.regular_grid(tgt_gm.size, (tgt_gm.x_min, tgt_gm.y_min), tgt_gm.xy_res, tile_size=tgt_gm.tile_size,
                                   is_j_axis_up=tgt_gm.is_j_axis_up)
            xs, ys = src_gm.x_values, src_gm.y_values
            fill = reproject_fill(dt)
            def oracle(method):
                with np.errstate(all="ignore"), warnings.catch_warnings():
                    warnings.simplefilter("ignore", RuntimeWarning)
                    return orep.reproject(src, float(xs[0]), float(ys[0]), src_gm.x_res, src_gm.y_res,
                                          float(ys[1] - ys[0]), g, geo, geo, method, fill)

            tid = "tile" if tile else "one-tile"
            for method in METHODS:
                want, skip = oracle(method), None
                if method == "triangular" and dt == np.uint32:
                    with mock.patch.object(orep, "sample_window", _triangular_f64):
                        skip = _uint32_out_of_range(oracle(method))
                cases.append(ReprojectCase(f"{name}-{method}-{tid}", src, method, fill, method == "bilinear", tile, want,
                                           skip))
                if method == "bilinear":  # cast once to the source dtype (numpy's astype) instead of float64
                    with np.errstate(all="ignore"), warnings.catch_warnings():
                        warnings.simplefilter("ignore", RuntimeWarning)
                        w32 = want.astype(np.dtype(dt))
                    skip = _uint32_out_of_range(want) if dt == np.uint32 else None
                    cases.append(ReprojectCase(f"{name}-bilinear-as-source-{tid}", src, method, fill, False, tile, w32,
                                               skip))
    return tuple(cases)
