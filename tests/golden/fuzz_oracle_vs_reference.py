"""Fuzz the CPU oracle against the REFERENCE's own numba kernels (needs the reference package where
make_golden.py's ``reference_dir`` finds it -- oracle/_ref first; third-party packages are stubbed as there).

    python tests/golden/fuzz_oracle_vs_reference.py [seed] [n_cases] [--write-digests | --check-digests]

The cases are those of ``fuzz_cases.py``: random small swaths through the source windows, the ij image
and the three gathers, random windows / dtypes / methods through ``_reproject_block`` and random blocks /
factors / dtypes through every ``AGG_METHODS`` reducer; oracle and reference must agree bit for bit.
Round 1: seeds 1-5, 21, 31-33: 5550 rectify, 1000 reproject-block and 1000 coarsen cases, 0 mismatches.
``--write-digests`` writes the digests of the REFERENCE's outputs to fuzz_digests.json, which
tests/test_oracle_fuzz.py holds the oracle against on machines without the reference; ``--check-digests``
compares them with that file instead (tests/test_oracle_fuzz.py runs it wherever the reference is installed).
"""
import json
import os
import sys
import time
import warnings

os.environ.setdefault("NUMBA_CACHE_DIR", "/tmp/numba_cache_golden")
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import fuzz_cases as fc  # noqa: E402
import make_golden as mg  # noqa: E402

mg.install_reference()
import xcube_resampling.gridmapping.bboxes as B  # noqa: E402
import xcube_resampling.rectify as R  # noqa: E402
from xcube_resampling import reproject as P  # noqa: E402
from xcube_resampling.constants import AGG_METHODS  # noqa: E402

from oracle import grid as ogrid, rectify as orect, reproject as orep, resample as ores  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
seed = int(args[0]) if args else fc.SEED
n_cases = int(args[1]) if len(args) > 1 else fc.N_CASES
rng = np.random.default_rng(seed)
digests = {"seed": seed, "n_cases": n_cases, "rectify": {}, "reproject": {}, "coarsen": {}}

bad = 0
t0 = time.time()
for k, x, y, g, src in fc.rectify_cases(rng, n_cases):
    win_ref, ij_ref = mg.reference_rectify(R, B, x, y, g)
    og = ogrid.RegularGrid(g["width"], g["height"], g["tile_w"], g["tile_h"], g["x_min"], g["y_min"], g["x_max"], g["y_max"], g["x_res"], g["y_res"], g["j_up"])
    win_or = orect.source_windows(x, y, og)
    ij_or = orect.rectify_ij(x, y, og)
    ok = np.array_equal(win_ref, win_or) and np.array_equal(ij_ref, ij_or, equal_nan=True)
    d = digests["rectify"][str(k)] = {"windows": fc.digest(win_ref), "ij": fc.digest(ij_ref)}
    for method in fc.METHODS:
        a = mg.reference_gather(R, src, ij_ref, g, method, np.nan)
        b = orect.gather(src, ij_ref, method, np.nan)
        d[method] = fc.digest(a)
        if not np.array_equal(a, b, equal_nan=True):
            ok = False; print("gather mismatch", method)
    if not ok:
        bad += 1
        print("MISMATCH case", k, "windows", np.array_equal(win_ref, win_or),
              "ij differing", int(np.sum(~((ij_ref == ij_or) | (np.isnan(ij_ref) & np.isnan(ij_or))))))
print(f"{n_cases} cases, {bad} mismatches, {time.time()-t0:.1f} s")

# ---------------------------------------------------------------------------
# reproject: oracle.reproject.sample_window vs the reference's _reproject_block (reproject.py:268-335)
# ---------------------------------------------------------------------------
bad_p = 0
n_p = fc.n_secondary(n_cases)
for k, xx, yy, arr, x_coord, y_coord, xres, yres in fc.reproject_cases(rng, n_p):
    for method in fc.METHODS:
        with np.errstate(all="ignore"):
            a = P._reproject_block(xx, yy, arr, x_coord, y_coord, xres, yres, method)
            b = orep.sample_window(xx, yy, arr, x_coord[0, 0, 0], y_coord[0, 0, 0], xres, yres, method)
        digests["reproject"][f"{k}/{method}"] = fc.digest(a)
        if a.dtype != b.dtype or not np.array_equal(a, b, equal_nan=a.dtype.kind == "f"):
            bad_p += 1
            print("REPROJECT MISMATCH", k, method, arr.dtype.name, a.dtype, b.dtype)
print(f"reproject: {n_p} cases, {bad_p} mismatches")

# ---------------------------------------------------------------------------
# coarsen: oracle.resample.coarsen vs the reference's AGG_METHODS reducers (coarsen.py, constants.py:51-65)
# ---------------------------------------------------------------------------
bad_c = 0
n_c = fc.n_secondary(n_cases)
for k, a, f_j, f_i in fc.coarsen_cases(rng, n_c):
    h, w = a.shape
    block = a.reshape(h // f_j, f_j, w // f_i, f_i)
    for agg, fn in AGG_METHODS.items():
        if agg == "mode" and a.dtype.kind == "f":
            continue
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            want = np.asarray(fn(block, (1, 3)))
            got = np.asarray(ores.coarsen(a, f_j, f_i, agg))
        digests["coarsen"][f"{k}/{agg}"] = fc.digest(want)
        if want.dtype != got.dtype or not np.array_equal(want, got, equal_nan=want.dtype.kind == "f"):
            bad_c += 1
            print("COARSEN MISMATCH", k, agg, a.dtype.name, (f_j, f_i), want.dtype, got.dtype)
print(f"coarsen: {n_c} cases, {bad_c} mismatches")

bad_d = 0
if "--write-digests" in sys.argv:
    digests["source"] = "the reference's own kernels (tests/golden/fuzz_oracle_vs_reference.py --write-digests)"
    with open(os.path.join(HERE, "fuzz_digests.json"), "w") as fh:
        json.dump(digests, fh, indent=0, sort_keys=True)
elif "--check-digests" in sys.argv:
    with open(os.path.join(HERE, "fuzz_digests.json")) as fh:
        stored = json.load(fh)
    keys = ("seed", "n_cases", "rectify", "reproject", "coarsen")
    bad_d = sum(stored[k] != digests[k] for k in keys)
    print(f"stored digests: {bad_d} of {len(keys)} parts differ from the reference's")
sys.exit(1 if (bad or bad_p or bad_c or bad_d) else 0)
