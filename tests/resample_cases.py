"""Cases of the affine / coarsen family (csrc/resample.cu, csrc/resample_fast.cu) shared by the host build
(test_host_k4k5_kernels.py) and the GPU (test_resample_edges_gpu.py): inputs with their memory layout, the C ABI
call, the oracle's answer (oracle/resample.py: scipy + numpy) and the kernel expected to run.

The expected kernel comes from :func:`expected_kernel`, a restatement of the dispatch rules of
``launch_affine_fast`` written here from their intent (which kernel may run for which alignment), not imported
from the product.  Values span each dtype's full range: int64 around +-1.7e18 and up to 2^63 - 1024, uint32 above
2^31, int8 at -128 / 127, floats with +-0, +-inf and NaN.
"""

import dataclasses
import warnings

import numpy as np

from oracle import resample as ores

nan, inf = np.nan, np.inf
ALL_AGGS = ("center", "count", "first", "last", "max", "mean", "median", "mode", "min", "prod", "std", "sum", "var")
DTYPES = (np.float32, np.float64, np.uint8, np.int8, np.uint16, np.int16, np.int32, np.uint32, np.int64)
SORTABLE = (np.float32, np.float64, np.uint8, np.int16, np.uint16, np.int32)  # k5_window_reduce<sort> types


@dataclasses.dataclass
class Layout:
    """Memory layout of the (n, h, w) source: row pitch = w + pitch_pad, slice stride = h * pitch + slice_pad, the
    first element ``elem_off`` elements past a 256-byte boundary."""
    pitch_pad: int = 0
    slice_pad: int = 0
    elem_off: int = 0

    def strides(self, shape):
        n, h, w = shape
        pitch = w + self.pitch_pad
        return pitch, h * pitch + self.slice_pad

    def slice_stride_seen(self, shape):
        """What the Python layer passes as slice stride: h * pitch when there is one slice."""
        pitch, ss = self.strides(shape)
        return ss if shape[0] > 1 else shape[1] * pitch


@dataclasses.dataclass
class Case:
    id: str
    kind: str        # "coarsen" | "affine" | "recover" | "has_nan"
    src: np.ndarray  # (n, h, w)
    layout: Layout
    args: dict
    want: object
    skip: object     # mask of elements excluded from the comparison (documented deviation) or None
    kernel: str      # expected kernel name


# ---------------------------------------------------------------------------
# dispatch rules of launch_affine_fast, restated
# ---------------------------------------------------------------------------
def _int_offset(v):
    return v >= 0 and float(v) == int(v)


def expected_kernel(kind, dtype, shape, layout, args):
    dtype = np.dtype(dtype)
    if kind == "has_nan":
        return "k4_has_nan" if dtype.kind == "f" else ""
    if kind == "recover":
        return "k4_affine_recover"
    n, h, w = shape
    es = dtype.itemsize
    flt = dtype.kind == "f"
    if kind == "coarsen":
        f_j, f_i = args["factors"]
        order, scale, off, out_hw, blend, exact = 0, (1.0, 1.0), (0.0, 0.0), (h // f_j, w // f_i), False, True
    else:
        f_j, f_i = args["factors"]
        order, scale, off, out_hw = args["order"], args["scale"], args["offset"], args["out_hw"]
        blend, exact = args["slice_blend"], False
    agg = args["agg"]
    generic = "k4_affine_generic"
    if f_j != f_i or f_j not in (2, 4, 8) or tuple(scale) != (1.0, 1.0):
        return generic
    if not (_int_offset(off[0]) and _int_offset(off[1])):
        return generic
    j_off, i_off = int(off[0]), int(off[1])
    if j_off + out_hw[0] * f_j > h or i_off + out_hw[1] * f_i > w:
        return generic  # some sample is cval
    if order == 1 and flt and blend:
        return generic  # next-slice taps (for one slice the slice itself)
    if order == 0 and not exact and (flt or dtype == np.int64):
        return generic  # scipy's float64 round trip: -0.0 -> +0.0, int64 beyond 2^53 rounded
    if order == 1 and dtype == np.int64:
        return generic
    pitch = w + layout.pitch_pad
    sstride = layout.slice_stride_seen(shape)
    F, dst_w = f_j, out_hw[1]

    def aligned(nbytes):  # view start, rows, slices and the column offset on `nbytes`
        return all(v % nbytes == 0 for v in (layout.elem_off * es, pitch * es, sstride * es, i_off * es))

    if dtype == np.uint8:
        if agg in ("median", "mode") and dst_w % 2 == 0 and aligned(2 * F):
            return "k5_u8x2_sort"  # 2 windows of F bytes per row
        if agg not in ("prod", "std", "var") and dst_w % 4 == 0 and aligned(8 if F == 2 else 16):
            return "k5_u8x4_reduce"  # 4 windows per thread, 8- / 16-byte row loads
    if agg in ("median", "mode"):
        return "k5_window_reduce<sort>" if dtype.type in SORTABLE else generic
    if flt and order == 1 and F == 2 and agg != "count" and dst_w % 4 == 0 and aligned(16):
        return "k5_blend2_x4"
    return "k5_window_reduce<simple>"


# ---------------------------------------------------------------------------
# the oracle
# ---------------------------------------------------------------------------
def _lib_dtype(a):
    """numpy's uint64 sums / products are the library's int64 plane viewed as uint64 by affine.py."""
    a = np.asarray(a)
    return a.view(np.int64) if a.dtype == np.uint64 else a


def _zero_sign_mix(fine, f_j, f_i, agg):
    """Float min / max windows holding both +0.0 and -0.0: numpy's nanmin / nanmax returns a sign that depends
    on its SIMD reduction order, the kernels the first one found (DESIGN section 5, known deviations)."""
    if agg not in ("min", "max") or fine.dtype.kind != "f":
        return None
    *lead, H, W = fine.shape
    b = fine.reshape(*lead, H // f_j, f_j, W // f_i, f_i)
    z = b == 0
    neg = np.signbit(b)
    ax = (b.ndim - 3, b.ndim - 1)
    return np.any(z & neg, axis=ax) & np.any(z & ~neg, axis=ax)


def oracle(kind, src, args):
    """(want, skip) for one case."""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if kind == "has_nan":
            return bool(np.isnan(src).any()) if src.dtype.kind == "f" else False, None
        if kind == "coarsen":
            f_j, f_i = args["factors"]
            want = _lib_dtype(ores.coarsen(src, f_j, f_i, args["agg"]))
            return want, _zero_sign_mix(src, f_j, f_i, args["agg"])
        f_j, f_i = args["factors"]
        (sj, si), (oj, oi) = args["scale"], args["offset"]
        matrix = ((si, 0.0, oi), (0.0, sj, oj))
        big = (args["out_hw"][0] * f_j, args["out_hw"][1] * f_i)
        recover = kind == "recover"
        order = 1 if recover else args["order"]
        if args["slice_blend"]:
            fine = ores.upscale(src, matrix, (src.shape[0],) + big, order, recover, args["cval"])
        else:
            fine = np.stack([ores.upscale(s, matrix, big, order, recover, args["cval"]) for s in src])
        if recover:
            assert fine.dtype == np.float64, "NaN recovery needs a NaN in the source"
        if f_j * f_i == 1:
            return fine, None
        return _lib_dtype(ores.coarsen(fine, f_j, f_i, args["agg"])), _zero_sign_mix(fine, f_j, f_i, args["agg"])


def make(id, kind, src, args, layout=None):
    src = np.asarray(src)
    if src.ndim == 2:
        src = src[None]
    layout = layout or Layout()
    want, skip = oracle(kind, src, args)
    return Case(id, kind, src, layout, args, want, skip, expected_kernel(kind, src.dtype, src.shape, layout, args))


def affine_args(scale, offset, out_hw, order, cval=0.0, agg="mean", factors=(1, 1), slice_blend=False):
    return dict(scale=tuple(float(v) for v in scale), offset=tuple(float(v) for v in offset), out_hw=tuple(out_hw),
                order=order, cval=cval, agg=agg, factors=tuple(factors), slice_blend=slice_blend)


# ---------------------------------------------------------------------------
# values
# ---------------------------------------------------------------------------
def values(dtype, shape, rng, kind="full"):
    """``full``: the dtype's range with its edges; ``classes``: a few values next to the dtype's maximum (mode
    ties; the oracle's histogram spans max - min); ``moderate``: int64 sums of 4 and products stay in range."""
    dtype = np.dtype(dtype)
    if dtype.kind == "f":
        a = rng.normal(size=shape) * 1e3
        r = rng.random(shape)
        a[r < 0.06] = nan
        a[(r >= 0.06) & (r < 0.09)] = inf
        a[(r >= 0.09) & (r < 0.12)] = -inf
        a[(r >= 0.12) & (r < 0.2)] = 0.0
        a[(r >= 0.2) & (r < 0.28)] = -0.0
        big = np.finfo(dtype).max
        a[(r >= 0.28) & (r < 0.3)] = big
        a[(r >= 0.3) & (r < 0.32)] = -big
        return a.astype(dtype)
    info = np.iinfo(dtype)
    if kind == "classes":
        return (info.max - rng.integers(0, 4, size=shape)).astype(dtype)
    if dtype == np.int64:
        lim = 2.2e18 if kind == "moderate" else 1.7e18
        a = (rng.uniform(-1, 1, size=shape) * lim).astype(np.int64)
        if kind == "moderate":
            return a
        r = rng.random(shape)
        a[r < 0.05] = np.iinfo(np.int64).max - 1024
        a[(r >= 0.05) & (r < 0.1)] = -(2 ** 62) - 1
        a[(r >= 0.1) & (r < 0.15)] = 2 ** 52 + 1  # float64 + 0.5 rounds half to even: scipy gives 2^52 + 2
        a[(r >= 0.15) & (r < 0.2)] = 1_700_000_000_123_456_789
        return a
    a = rng.integers(int(info.min), int(info.max), size=shape, endpoint=True, dtype=np.int64)
    r = rng.random(shape)
    a[r < 0.08] = info.min
    a[(r >= 0.08) & (r < 0.16)] = info.max
    a[(r >= 0.16) & (r < 0.22)] = 0
    if dtype == np.uint32:
        a[(r >= 0.22) & (r < 0.5)] = rng.integers(2 ** 31, 2 ** 32, size=int(((r >= 0.22) & (r < 0.5)).sum()))
    return a.astype(dtype)


# ---------------------------------------------------------------------------
# the table
# ---------------------------------------------------------------------------
def _aggs_for(dtype, f):
    dt = np.dtype(dtype)
    out = [a for a in ALL_AGGS if not (a == "mode" and dt.kind == "f")]
    if dt == np.int64:  # sums / products of +-1.7e18 wrap; the "moderate" cases below cover them
        out = [a for a in out if a not in ("sum", "prod")]
    if dt in (np.int32, np.uint32, np.int64):  # a variance beyond the dtype's range (DESIGN section 5)
        out = [a for a in out if a != "var"]
    return [a for a in out if a != "mode"]  # mode: the "classes" cases


def cases():
    out = []
    rng = np.random.default_rng(2024)
    # ---- every dtype, full range, F = 2 / 4 / 8 and odd factors, through xrs_coarsen --------------------------
    for dt in DTYPES:
        name = np.dtype(dt).name
        for f in (2, 4, 8, 3, (1, 3), 5):
            f_j, f_i = (f, f) if isinstance(f, int) else f
            src = values(dt, (2, 3 * f_j, 7 * f_i), rng)
            for agg in _aggs_for(dt, f):
                out.append(make(f"coarsen-{name}-{f}-{agg}", "coarsen", src, dict(factors=(f_j, f_i), agg=agg)))
            if np.dtype(dt).kind != "f":
                cls = values(dt, (1, 2 * f_j, 8 * f_i), rng, "classes")
                out.append(make(f"coarsen-{name}-{f}-mode", "coarsen", cls, dict(factors=(f_j, f_i), agg="mode")))
        if dt == np.int64:
            for f in (2, 3):
                src = values(dt, (1, 2 * f, 6 * f), rng, "moderate") // (4 if f == 3 else 1)
                out.append(make(f"coarsen-int64-{f}-sum", "coarsen", src, dict(factors=(f, f), agg="sum")))
    # int64 odd-count median around 1.7e18 (numpy's float64 middle value, rounded and cast back)
    big = (1_700_000_000_000_000_000 + rng.integers(-10 ** 6, 10 ** 6, size=(1, 6, 9))).astype(np.int64)
    out.append(make("coarsen-int64-3x3-median-1.7e18", "coarsen", big, dict(factors=(3, 3), agg="median")))

    # ---- aligned fast paths: every branch of launch_affine_fast, layouts ---------------------------------------
    # (dst_w, i_off, pitch_pad, slice_pad, elem_off, n)
    layouts = [(8, 0, 0, 0, 0, 1), (9, 0, 0, 0, 0, 1), (10, 0, 0, 0, 0, 1), (11, 0, 0, 0, 0, 1), (8, 1, 0, 0, 0, 1),
               (8, "align", 0, 0, 0, 1), (8, 0, 3, 0, 0, 1), (8, 0, 0, 0, 1, 1), (8, 0, 0, 0, "15B", 1),
               (8, 0, 0, 0, 0, 3), (8, 0, 0, 5, 0, 3), (12, "align", 4, 16, "align", 3), (8, "8B", 0, 0, 0, 1),
               (8, 0, 0, 0, "8B", 1)]
    kinds = [(np.uint8, "mean", 0), (np.uint8, "sum", 0), (np.uint8, "count", 0), (np.uint8, "median", 0),
             (np.uint8, "mode", 0), (np.uint8, "std", 0), (np.float32, "mean", 1), (np.float64, "max", 1),
             (np.float32, "median", 1), (np.float64, "median", 0), (np.int16, "mode", 0), (np.int16, "mean", 0),
             (np.float32, "count", 1), (np.uint32, "min", 0), (np.int64, "mean", 1), (np.int64, "first", 0)]
    for f in (2, 4, 8):
        for dt, agg, order in kinds:
            es = np.dtype(dt).itemsize
            for k, (dst_w, i_off, ppad, spad, eoff, n) in enumerate(layouts):
                if (f == 8 and k % 2) or (f == 4 and k % 3 == 1):
                    continue  # the full layout list at F = 2, a part of it at 4 and 8
                align = 16 // es
                i_off = {"align": align, "8B": max(1, 8 // es)}.get(i_off, i_off)
                eoff = {"15B": max(1, 15 // es), "align": align, "8B": max(1, 8 // es)}.get(eoff, eoff)
                dst_h, j_off = 3, (1 if k % 4 == 3 else 0)
                h, w = j_off + dst_h * f + (k % 2), i_off + dst_w * f + (k % 3)
                if dt == np.uint8 and agg in ("mode", "median"):
                    src = rng.integers(0, 3 if agg == "mode" else 256, size=(n, h, w)).astype(dt)
                else:
                    src = values(dt, (n, h, w), rng, "classes" if agg == "mode" else "full")
                args = affine_args((1, 1), (j_off, i_off), (dst_h, dst_w), order, nan if order else 0.0, agg, (f, f))
                lay = Layout(ppad, spad, eoff)
                out.append(make(f"fast-{np.dtype(dt).name}-{agg}-o{order}-f{f}-L{k}", "affine", src, args, lay))
    # 3-D order-1 float input with slice_blend: next-slice taps -> generic kernel
    src = values(np.float32, (3, 8, 16), rng)
    out.append(make("fast-3d-slice-blend-falls-back", "affine", src,
                    affine_args((1, 1), (0, 0), (4, 8), 1, nan, "mean", (2, 2), slice_blend=True)))

    # ---- uint8 packed kernels -----------------------------------------------------------------------------------
    for f in (2, 4, 8):
        a = np.zeros((2, 2 * f, 8 * f), np.uint8)
        a[0, :, 4 * f:] = 255  # windows all 0 / all 255 (8 x 8: sum 16 320)
        a[1, :f, :] = rng.integers(0, 256, size=(f, 8 * f))
        # medians whose middle values have an odd sum, with both parities of the floor: (3, 4) -> 4, (5, 6) -> 6
        lo = f * f // 2
        for win, (x, y) in enumerate(((3, 4), (5, 6), (254, 255), (0, 1))):
            vals = np.array([0] * (lo - 1) + [x, y] + [255] * (f * f - lo - 1), np.uint8)
            a[1, f:, win * f:(win + 1) * f] = rng.permutation(vals).reshape(f, f)
        for agg in ("sum", "mean", "median", "count", "max", "min"):
            out.append(make(f"u8-edges-f{f}-{agg}", "coarsen", a, dict(factors=(f, f), agg=agg)))
        # mode ties placed first, middle and last in sort order (two values c times each, the rest fewer times)
        m = np.zeros((1, f, 8 * f), np.uint8)
        n_win, c = f * f, (f * f + 2) // 3
        rest = n_win - 2 * c
        for win, (tie, filler) in enumerate((((0, 9), np.arange(100, 100 + rest)),
                                             ((4, 9), np.array([0] * (rest // 2) + [255] * (rest - rest // 2))),
                                             ((200, 255), np.arange(10, 10 + rest)),
                                             ((7, 8), np.arange(20, 20 + rest)))):
            vals = np.concatenate([[tie[0]] * c, [tie[1]] * c, filler]).astype(np.uint8)
            m[0, :, win * f:(win + 1) * f] = rng.permutation(vals).reshape(f, f)
        m[0, :, 4 * f:] = rng.integers(0, 2, size=(f, 4 * f))
        out.append(make(f"u8-mode-ties-f{f}", "coarsen", m, dict(factors=(f, f), agg="mode")))
        out.append(make(f"u8-count-zeros-f{f}", "coarsen", m, dict(factors=(f, f), agg="count")))

    # ---- K4 generic ---------------------------------------------------------------------------------------------
    for f in (3, (1, 3), (2, 4), 5, 16, (2, 128), (16, 16)):
        f_j, f_i = (f, f) if isinstance(f, int) else f
        for dt, agg in ((np.float32, "median"), (np.float64, "mean"), (np.int32, "median"), (np.int64, "median"),
                        (np.uint8, "max"), (np.int8, "min")):
            src = values(dt, (1, 2 * f_j + 1, 2 * f_i + 3), rng)
            args = affine_args((0.93, 1.07), (0.25, -0.5), (2, 2), 1, nan, agg, (f_j, f_i))
            out.append(make(f"generic-{np.dtype(dt).name}-{f_j}x{f_i}-{agg}", "affine", src, args))
    for dt in DTYPES:
        name = np.dtype(dt).name
        src = values(dt, (1, 9, 13), rng)
        for order in (0, 1):
            # scales / offsets that land exactly on len - 1, just beyond it, and negative offsets
            for sc, off, hw in (((1.0, 1.0), (0.0, 0.0), (9, 13)), ((2.0, 3.0), (0.0, 0.0), (5, 5)),
                                ((1.0, 1.0), (1e-12, -1e-12), (9, 13)), ((0.5, 0.5), (-0.75, -1.0), (19, 27)),
                                ((1.5, 0.75), (0.3, 2.2), (7, 15))):
                args = affine_args(sc, off, hw, order, 3.0)
                out.append(make(f"edge-{name}-o{order}-{sc}-{off}", "affine", src, args))
        if np.dtype(dt).kind in "iu":
            for cval in (nan, inf, -inf, 1e300, -1e300, 2.0 ** 63, 2.0 ** 31 - 0.5, 2.0 ** 31 + 0.5, 2.0 ** 32 - 0.5):
                args = affine_args((1.0, 1.0), (-2.0, 5.0), (9, 13), 0, cval)
                out.append(make(f"cval-{name}-{cval!r}", "affine", src, args))
    # int64 finding cases: order 0 (float64 round trip), aligned order 1 / 2 (generic, rounded)
    i64 = values(np.int64, (1, 8, 16), rng)
    out.append(make("int64-order0-identity", "affine", i64, affine_args((1, 1), (0, 0), (8, 16), 0)))
    out.append(make("int64-order1-aligned-div2", "affine", i64, affine_args((1, 1), (0, 0), (4, 8), 1, -1.0, "mean", (2, 2))))
    out.append(make("int64-order0-aligned-2x2-first", "affine", i64,
                    affine_args((1, 1), (0, 0), (4, 8), 0, -1.0, "first", (2, 2))))
    # 3-D slice_blend for n = 1..4 with NaN / +-inf in the (mirrored) next slice
    for n in (1, 2, 3, 4):
        for dt in (np.float32, np.float64):
            src = rng.normal(size=(n, 7, 9)).astype(dt)
            src[n - 1, 2, 3] = nan
            src[max(n - 2, 0), 4, 4] = inf
            src[0, 6, 8] = -inf
            args = affine_args((0.8, 1.25), (0.1, -0.2), (8, 7), 1, nan, slice_blend=True)
            out.append(make(f"slice-blend-n{n}-{np.dtype(dt).name}", "affine", src, args))
            args = affine_args((1, 1), (0, 0), (3, 4), 1, nan, "max", (2, 2), slice_blend=True)
            out.append(make(f"slice-blend-n{n}-{np.dtype(dt).name}-2x2", "affine", src, args))

    # ---- recover_nans -------------------------------------------------------------------------------------------
    for dt in (np.float32, np.float64):
        name = np.dtype(dt).name
        src = rng.normal(size=(1, 12, 15)).astype(dt)
        src[0, 3, 4] = nan
        src[0, 7:9, 10:12] = nan
        src[0, 11, 14] = nan
        for cval in (nan, 5.0):  # numeric fill: the reference divides cval by cval outside the source
            for tag, a in (("upscale", affine_args((0.5, 0.5), (-0.25, -0.25), (26, 32), 1, cval)),
                           ("half-pixel", affine_args((1, 1), (0.5, 0.5), (12, 15), 1, cval)),
                           ("div2", affine_args((1, 1), (0, 0), (6, 7), 1, cval, "mean", (2, 2))),
                           ("div3", affine_args((1, 1), (-0.5, 0.25), (4, 5), 1, cval, "median", (3, 3)))):
                out.append(make(f"recover-{name}-{tag}-{cval}", "recover", src, a))
        s3 = rng.normal(size=(3, 6, 7)).astype(dt)
        s3[0, 1, 1] = nan
        s3[1, 2, 2] = inf     # next slice of slice 0: +-inf contaminates after the zero filling
        s3[2, 3, 3] = nan     # next slice of slice 1: NaN is zero filled and does not
        s3[1, 4, 5] = -inf
        out.append(make(f"recover-{name}-3d", "recover", s3,
                        affine_args((0.9, 0.9), (0.2, 0.1), (6, 7), 1, nan, slice_blend=True)))

    # ---- has_nan ------------------------------------------------------------------------------------------------
    for dt in (np.float32, np.float64):
        name = np.dtype(dt).name
        a = np.zeros((1, 1, 16384 + 300), dt)
        a[0, 0, 16384 + 277] = nan  # beyond the 64-block column cap, lane 21 of its warp
        out.append(make(f"has-nan-{name}-wide", "has_nan", a, {}))
        a = np.zeros((1, 1100, 40), dt)
        a[0, 1090, 37] = nan  # beyond the 1024-row cap, lane 5
        out.append(make(f"has-nan-{name}-tall", "has_nan", a, {}))
        a = np.zeros((3, 20, 50), dt)
        a[2, 19, 45] = nan  # last slice only, lane 13
        out.append(make(f"has-nan-{name}-last-slice", "has_nan", a, {}, Layout(3, 7, 0)))
        out.append(make(f"has-nan-{name}-none", "has_nan", np.zeros((2, 5, 40), dt), {}))
    for dt in (np.uint8, np.int32, np.int64):
        out.append(make(f"has-nan-{np.dtype(dt).name}", "has_nan", values(dt, (1, 4, 40), rng), {}))
    return out
