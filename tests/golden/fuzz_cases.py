"""The seeded fuzz cases of the oracle / reference comparison and the digest both sides are reduced to.

Shared by ``fuzz_oracle_vs_reference.py`` (the oracle against the reference's own kernels, where the
reference package is installed; it also writes ``fuzz_digests.json``) and ``tests/test_oracle_fuzz.py``
(the oracle against those digests, anywhere).  The cases are drawn from ONE generator in a fixed order --
rectify, then reproject, then coarsen -- so both sides see the same inputs for the same seed.
"""

import numpy as np

import make_golden as mg
from tests.helpers import digest  # noqa: F401

SEED, N_CASES = 11, 120
METHODS = ("nearest", "bilinear", "triangular")


def n_secondary(n_cases: int) -> int:
    """Number of reproject and of coarsen cases that follow ``n_cases`` rectify cases."""
    return max(20, n_cases // 3)


def rectify_cases(rng, n_cases):
    """(k, x, y, grid dict, src) of random small swaths -- rotations, NaN holes, folds, coordinates snapped to
    the pixel raster (pixel centres exactly on triangle edges), duplicated columns -- on random target
    resolutions, tilings and axis directions.  Cases whose grid is degenerate or too large are skipped."""
    for k in range(n_cases):
        w, h = int(rng.integers(3, 70)), int(rng.integers(3, 70))
        theta = float(rng.uniform(-180, 180))
        x, y = mg.swath(w, h, theta=theta, seed=int(rng.integers(0, 100)), lat0=float(rng.uniform(-60, 60)),
                        lon0=float(rng.uniform(-150, 150)))
        kind = rng.integers(0, 6)
        if kind == 1:   # NaN holes
            m = rng.random(x.shape) < 0.05
            x = x.copy()
            y = y.copy()
            x[m] = np.nan
            y[m & (rng.random(x.shape) < 0.5)] = np.nan
        elif kind == 2:  # strong perturbation (folds)
            x = x + rng.normal(0, 0.0027 * 0.7, x.shape)
            y = y + rng.normal(0, 0.0027 * 0.7, y.shape)
        elif kind == 3:  # coordinates snapped to the pixel raster (pixel centres on edges)
            x = np.round(x / 0.00135) * 0.00135
            y = np.round(y / 0.00135) * 0.00135
        elif kind == 4:  # duplicated rows / columns
            x[:, w // 2] = x[:, w // 2 - 1]
            y[:, w // 2] = y[:, w // 2 - 1]
        res = 0.0027 * float(rng.choice([0.31, 0.5, 1.0, 1.0, 1.7, 3.3]))
        tile = [None, int(rng.integers(5, 40)), (int(rng.integers(4, 50)), int(rng.integers(4, 50)))][int(rng.integers(0, 3))]
        j_up = bool(rng.integers(0, 2))
        try:
            g = mg.regular_params(x, y, res, tile, j_up)
        except ValueError:
            continue
        if g["width"] * g["height"] > 400000 or g["width"] < 2 or g["height"] < 2:
            continue
        src = rng.random((2, h, w)).astype(np.float32)
        yield k, x, y, g, src


def reproject_cases(rng, n):
    """(k, xx, yy, arr, x_coord, y_coord, xres, yres) of random ``_reproject_block`` windows over six dtypes,
    with target points exactly on source pixel centres and exactly half way between them."""
    for k in range(n):
        ww, wh, tw, th = (int(v) for v in rng.integers(3, 40, 4))
        xres, yres = float(rng.choice([0.0001, 0.01, 10.0, 0.25])), float(rng.choice([0.0001, 0.01, 10.0, 0.5]))
        xo, yo = float(rng.uniform(-170, 170) * (1 if xres < 1 else 3000)), float(rng.uniform(-80, 80) * (1 if yres < 1 else 70000))
        x_coord = (xo + xres * np.arange(ww)).astype(np.float32).reshape(ww, 1, 1)
        y_coord = (yo - yres * np.arange(wh)).astype(np.float32).reshape(wh, 1, 1)
        fx = rng.uniform(0.0, ww - 1.001, size=(th, tw))
        fy = rng.uniform(0.0, wh - 1.001, size=(th, tw))
        fx[0, : min(tw, ww - 1)] = np.arange(min(tw, ww - 1))           # exactly on pixel centres
        fy[-1, : min(tw, wh - 1)] = np.arange(min(tw, wh - 1)) + 0.5     # exactly half way (rint ties)
        xx = np.float64(x_coord[0, 0, 0]) + fx * xres
        yy = np.float64(y_coord[0, 0, 0]) - fy * yres
        dtype = [np.float32, np.float64, np.uint8, np.int16, np.int32, np.int64][int(rng.integers(0, 6))]
        if np.issubdtype(dtype, np.floating):
            arr = rng.normal(size=(2, wh, ww)).astype(dtype)
            arr[0, rng.random((wh, ww)) < 0.05] = np.nan
        else:
            info = np.iinfo(dtype)
            arr = rng.integers(max(info.min, -2**40), min(info.max, 2**40), size=(2, wh, ww)).astype(dtype)
        yield k, xx, yy, arr, x_coord, y_coord, xres, yres


def coarsen_cases(rng, n):
    """(k, a, f_j, f_i) of random blocks, factors 1-8 and seven dtypes, with NaN shares of 0 / 10 / 60 % and
    integer blocks of few classes (mode ties)."""
    for k in range(n):
        f_j, f_i = int(rng.integers(1, 9)), int(rng.integers(1, 9))
        h, w = f_j * int(rng.integers(1, 7)), f_i * int(rng.integers(1, 7))
        dtype = [np.float32, np.float64, np.uint8, np.int16, np.uint16, np.int32, np.int64][int(rng.integers(0, 7))]
        if np.issubdtype(dtype, np.floating):
            a = (rng.normal(size=(h, w)) * 10.0 ** int(rng.integers(-3, 4))).astype(dtype)
            a[rng.random((h, w)) < rng.choice([0.0, 0.1, 0.6])] = np.nan
        else:
            info = np.iinfo(dtype)
            a = rng.integers(max(info.min, -500), min(info.max, 500), size=(h, w)).astype(dtype)
            if rng.random() < 0.5:
                a = (a % 5).astype(dtype)  # few classes: mode ties
        yield k, a, f_j, f_i
