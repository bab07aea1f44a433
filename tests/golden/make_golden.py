"""Generate tests/golden/*.npz by running the REFERENCE's own kernels.

Runs only where the reference package is installed (the directories of
``oracle/refkernels.py``'s ``REF_DIRS``, ``oracle/_ref`` first): the
reference's numba / numpy kernels are imported from there (third-party packages
that are not installed -- dask, xarray, pyproj, affine, zarr, dask_image -- are
replaced by inert stub modules, numba JIT stays on) and executed on small seeded
inputs.  The resulting input/output vectors are committed; the GPU box and the
CPU test-suite only ever read the ``.npz`` files.

    python tests/golden/make_golden.py

The tile loops below restate ``rectify.py:373-419`` / ``605-635`` only as far as
needed to feed the reference kernels with the slices the reference would pass.
"""

import os
import sys
import types

os.environ.setdefault("NUMBA_CACHE_DIR", "/tmp/numba_cache_golden")
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


class _Any:
    def __init__(self, *a, **k):
        pass

    def __getattr__(self, n):
        if n.startswith("__") and n.endswith("__"):
            raise AttributeError(n)
        return _Any()

    def __call__(self, *a, **k):
        return _Any()

    def __or__(self, o):
        return self

    def __ror__(self, o):
        return self

    def __getitem__(self, k):
        return _Any()

    def __mro_entries__(self, bases):
        return ()


class _Stub(types.ModuleType):
    def __getattr__(self, n):
        if n.startswith("__") and n.endswith("__"):
            raise AttributeError(n)
        return _Any()


def reference_dir():
    """The first directory of ``oracle.refkernels.REF_DIRS`` that holds the reference package."""
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    from oracle.refkernels import REF_DIRS

    where = next((d for d in REF_DIRS if os.path.isdir(os.path.join(d, "xcube_resampling"))), None)
    if where is None:
        raise SystemExit(f"the reference package (xcube_resampling) is in none of {list(REF_DIRS)}")
    return where


def install_reference():
    for name in ["dask", "dask.array", "dask.array.core", "xarray", "pyproj", "pyproj.crs", "pyproj.transformer",
                 "dask_image", "dask_image.ndinterp", "affine", "zarr", "zarr.convenience"]:
        if name not in sys.modules:
            m = _Stub(name)
            m.__path__ = []
            sys.modules[name] = m
    where = reference_dir()
    if where not in sys.path:
        sys.path.insert(0, where)


# ---------------------------------------------------------------------------
# synthetic inputs
# ---------------------------------------------------------------------------
def swath(width, height, res=0.0027, theta=12.0, seed=0, lon0=10.0, lat0=45.0):
    """OLCI-like rotated swath with a smooth sub-pixel perturbation (SURVEY.md 8d, C2)."""
    i = np.arange(width, dtype=np.float64)[None, :]
    j = np.arange(height, dtype=np.float64)[:, None]
    a = (i - width / 2) * res
    b = (height / 2 - j) * res
    th = np.deg2rad(theta)
    lat = lat0 + a * np.sin(th) + b * np.cos(th)
    lon = lon0 + (a * np.cos(th) - b * np.sin(th)) / np.cos(np.deg2rad(lat))
    lon = lon + 0.1 * res * np.sin(i / 37.0 + seed) * np.cos(j / 29.0)
    lat = lat + 0.1 * res * np.cos(i / 31.0) * np.sin(j / 41.0 + seed)
    return lon, lat


def regular_params(x, y, res, tile, j_up=False):
    """Target grid covering the swath; returns a plain dict (no reference types needed)."""
    xf, yf = x[np.isfinite(x)], y[np.isfinite(y)]
    x_min = float(xf.min()) - res / 2
    y_min = float(yf.min()) - res / 2
    w = int(np.ceil((xf.max() - xf.min()) / res)) + 1
    h = int(np.ceil((yf.max() - yf.min()) / res)) + 1
    tw, th = (w, h) if tile is None else ((tile, tile) if isinstance(tile, int) else tile)
    return dict(width=w, height=h, tile_w=min(tw, w), tile_h=min(th, h), x_min=x_min, y_min=y_min,
                x_max=x_min + res * w, y_max=y_min + res * h, x_res=res, y_res=res, j_up=j_up)


def tile_boxes(g):
    nty = -(-g["height"] // g["tile_h"])
    ntx = -(-g["width"] // g["tile_w"])
    ij = np.array([[tx * g["tile_w"], ty * g["tile_h"], min((tx + 1) * g["tile_w"], g["width"]),
                    min((ty + 1) * g["tile_h"], g["height"])] for ty in range(nty) for tx in range(ntx)],
                  dtype=np.int64)
    if g["j_up"]:
        off = np.array([g["x_min"], g["y_min"], g["x_min"], g["y_min"]])
        sc = np.array([g["x_res"], g["y_res"], g["x_res"], g["y_res"]])
        xy = off + sc * ij
    else:
        off = np.array([g["x_min"], g["y_max"], g["x_min"], g["y_max"]])
        sc = np.array([g["x_res"], -g["y_res"], g["x_res"], -g["y_res"]])
        xy = off + sc * ij
        xy[:, [1, 3]] = xy[:, [3, 1]]
    return ij, xy


def reference_rectify(R, B, x, y, g, uv_delta=1e-3):
    """windows + ij image through the reference kernels, tile by tile."""
    ij_boxes, xy_boxes = tile_boxes(g)
    ntx_f, nty_f = g["width"] / g["tile_w"], g["height"] / g["tile_h"]
    border = min(min(2 * ntx_f * g["x_res"], 2 * nty_f * g["y_res"]),
                 min(0.5 * (g["x_max"] - g["x_min"]), 0.5 * (g["y_max"] - g["y_min"])))
    windows = np.full((len(ij_boxes), 4), -1, dtype=np.int64)
    B.compute_ij_bboxes(x, y, xy_boxes, border, 1, windows)
    ij = np.full((2, g["height"], g["width"]), np.nan)
    for k, (i0, j0, i1, j1) in enumerate(ij_boxes):
        bb = windows[k]
        if bb[0] == -1:
            continue
        xs = np.ascontiguousarray(x[bb[1]:bb[3] + 1, bb[0]:bb[2] + 1])
        ys = np.ascontiguousarray(y[bb[1]:bb[3] + 1, bb[0]:bb[2] + 1])
        blk = np.empty((2, j1 - j0, i1 - i0))
        x_off = g["x_min"] + i0 * g["x_res"]
        y_off = g["y_min"] + j0 * g["y_res"] if g["j_up"] else g["y_max"] - j0 * g["y_res"]
        R._compute_target_source_ij_sequential(xs, ys, bb[0], bb[1], blk, x_off, y_off, g["x_res"],
                                               g["y_res"] if g["j_up"] else -g["y_res"], uv_delta)
        ij[:, j0:j1, i0:i1] = blk
    return windows, ij


def reference_gather(R, src, ij, g, method, fill):
    """rectify.py:605-635 per reference tile."""
    src3 = src if src.ndim == 3 else src[None]
    out = np.full((src3.shape[0], g["height"], g["width"]), fill, dtype=src3.dtype)
    ij_boxes, _ = tile_boxes(g)
    for (i0, j0, i1, j1) in ij_boxes:
        blk_ij = np.ascontiguousarray(ij[:, j0:j1, i0:i1])
        if np.all(np.isnan(blk_ij[0])):
            continue
        bbox = (int(np.nanmin(blk_ij[0])), int(np.nanmin(blk_ij[1])),
                min(int(np.nanmax(blk_ij[0])) + 2, src3.shape[-1]), min(int(np.nanmax(blk_ij[1])) + 2, src3.shape[-2]))
        win = src3[..., bbox[1]:bbox[3], bbox[0]:bbox[2]].astype(np.float64)
        dst = np.full((src3.shape[0], j1 - j0, i1 - i0), fill, dtype=src3.dtype)
        R._compute_var_image_sequential(win, blk_ij, dst, bbox, method)
        out[:, j0:j1, i0:i1] = dst
    return out if src.ndim == 3 else out[0]


def make_rectify(R, B):
    out = {}
    cases = []
    rng = np.random.default_rng(7)
    # (name, width, height, theta, tile, j_up, nan_coords)
    specs = [
        ("swath_single", 96, 80, 12.0, None, False, False),
        ("swath_tiled32", 96, 80, 12.0, 32, False, False),
        ("swath_tiled_17x40_jup", 96, 80, -25.0, (17, 40), True, False),
        ("swath_nan_coords", 70, 60, 33.0, 48, False, True),
        ("swath_fine_target", 40, 36, 5.0, 64, False, False),
    ]
    for name, w, h, theta, tile, j_up, nan_coords in specs:
        x, y = swath(w, h, theta=theta, seed=len(cases))
        if nan_coords:
            x = x.copy()
            y = y.copy()
            m = rng.random(x.shape) < 0.03
            x[m] = np.nan
            y[m & (rng.random(x.shape) < 0.5)] = np.nan
            x[5, 7] = np.inf
            y[9, 11] = -np.inf
        res = 0.0027 if name != "swath_fine_target" else 0.0027 / 3.1
        g = regular_params(x, y, res, tile, j_up)
        windows, ij = reference_rectify(R, B, x, y, g)
        f32 = rng.random((3, h, w)).astype(np.float32)
        f32[0, rng.random((h, w)) < 0.02] = np.nan
        u8 = rng.integers(0, 200, (h, w)).astype(np.uint8)
        i16 = rng.integers(-3000, 3000, (2, h, w)).astype(np.int16)
        f64 = rng.random((h, w))
        out[f"{name}/x"], out[f"{name}/y"] = x, y
        out[f"{name}/grid"] = np.array([g["width"], g["height"], g["tile_w"], g["tile_h"], g["x_min"], g["y_min"],
                                        g["x_max"], g["y_max"], g["x_res"], g["y_res"], float(g["j_up"])])
        out[f"{name}/windows"], out[f"{name}/ij"] = windows, ij
        for vname, src, fill in (("f32", f32, np.nan), ("u8", u8, 255), ("i16", i16, -1), ("f64", f64, np.nan)):
            out[f"{name}/src_{vname}"] = src
            for method in ("nearest", "bilinear", "triangular"):
                out[f"{name}/out_{vname}_{method}"] = reference_gather(R, src, ij, g, method, fill)
        cases.append(name)
    out["cases"] = np.array(cases)
    np.savez_compressed(os.path.join(HERE, "rectify.npz"), **out)
    print("rectify.npz:", cases)


def make_rectify_f32_coords(R, B):
    """float32 coordinate images fed to the reference kernels as they are (rectify.py:480-501 builds
    its vertex arrays in the coordinates' dtype).  Pins that up-casting float32 coordinates to
    float64 first, as the C ABI requires, changes nothing."""
    out = {}
    cases = []
    for name, w, h, theta, tile, j_up in [("f32_tiled32", 96, 80, 12.0, 32, False),
                                          ("f32_tiled_17x40_jup", 70, 64, -25.0, (17, 40), True)]:
        x, y = swath(w, h, theta=theta, seed=3)
        x32, y32 = x.astype(np.float32), y.astype(np.float32)
        g = regular_params(x32.astype(np.float64), y32.astype(np.float64), 0.0027, tile, j_up)
        windows, ij = reference_rectify(R, B, x32, y32, g)
        out[f"{name}/x"], out[f"{name}/y"] = x32, y32
        out[f"{name}/grid"] = np.array([g["width"], g["height"], g["tile_w"], g["tile_h"], g["x_min"], g["y_min"],
                                        g["x_max"], g["y_max"], g["x_res"], g["y_res"], float(g["j_up"])])
        out[f"{name}/windows"], out[f"{name}/ij"] = windows, ij
        cases.append(name)
    out["cases"] = np.array(cases)
    np.savez_compressed(os.path.join(HERE, "rectify_f32coords.npz"), **out)
    print("rectify_f32coords.npz:", cases)


def make_ij_bboxes(B):
    """compute_ij_bboxes on the fixture of tests/gridmapping/test_bboxes.py plus random boxes."""
    out = {}
    lon, lat = np.meshgrid(np.linspace(10.0, 20.0, 11), np.linspace(50.0, 60.0, 11))
    out["x"], out["y"] = lon, lat
    rng = np.random.default_rng(3)
    k = 0
    for border, ij_border in [(0.0, 0), (0.5, 0), (1.0, 0), (2.0, 0), (2.0, 2), (0.3, 1)]:
        lo = rng.uniform(8.0, 18.0, (6, 1))
        boxes = np.concatenate([lo, 48.0 + (lo - 8.0), lo + rng.uniform(0.1, 6.0, (6, 1)),
                                48.0 + (lo - 8.0) + rng.uniform(0.1, 6.0, (6, 1))], axis=1)
        boxes = np.concatenate([boxes, [[12.4, 51.6, 12.6, 51.7], [10.0, 50.0, 20.0, 60.0], [31.0, 71.0, 36.0, 76.0]]])
        res = np.full(boxes.shape, -1, dtype=np.int64)
        B.compute_ij_bboxes(lon, lat, boxes, border, ij_border, res)
        out[f"case{k}/boxes"], out[f"case{k}/params"], out[f"case{k}/result"] = boxes, np.array([border, ij_border]), res
        k += 1
    out["n_cases"] = np.array(k)
    np.savez_compressed(os.path.join(HERE, "ij_bboxes.npz"), **out)
    print("ij_bboxes.npz:", k, "cases")


def make_dual_swath():
    """Digests of the reference's three gathers, tile by tile, of the swath tests/test_oracle_dual.py holds
    the two-method gather against (too large to commit as arrays)."""
    import json

    from oracle import refkernels
    from tests.helpers import digest, dual_swath

    x, y, g, data = dual_swath()
    methods = ("nearest", "bilinear", "triangular")
    _, ref = refkernels.rectify_pass(x, y, data, g, methods, n_threads=4, keep_outputs=True)
    out = {m: digest(ref[m]) for m in methods}
    out["source"] = "the reference's own kernels (tests/golden/make_golden.py)"
    with open(os.path.join(HERE, "dual_swath_digests.json"), "w") as fh:
        json.dump(out, fh, indent=0, sort_keys=True)
    print("dual_swath_digests.json")


def main():
    install_reference()
    import xcube_resampling.gridmapping.bboxes as B
    import xcube_resampling.rectify as R

    make_rectify(R, B)
    make_rectify_f32_coords(R, B)
    make_ij_bboxes(B)
    make_dual_swath()
    try:
        from make_golden_resample import make_all as make_resample  # added with the affine/coarsen/reproject paths
    except ImportError:
        make_resample = None
    if make_resample is not None:
        make_resample()


if __name__ == "__main__":
    sys.path.insert(0, HERE)
    main()
