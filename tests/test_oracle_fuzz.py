"""Short fuzz campaign of the oracle against the reference's own kernels on the seeded cases of
tests/golden/fuzz_cases.py: source windows, ij image and the three gathers of random swaths,
``_reproject_block`` windows, every ``AGG_METHODS`` reducer -- bit for bit, dtypes included.

Everywhere, the oracle's outputs are held against the digests in tests/golden/fuzz_digests.json (their
``source`` says what produced them).  Where the reference package is installed (``oracle.refkernels.REF_DIRS``),
tests/golden/fuzz_oracle_vs_reference.py also runs the cases through the reference's kernels in a subprocess
(importing the reference installs stub modules for dask / xarray / pyproj): the oracle must equal them, and
their digests must equal the stored ones."""

import importlib.util
import json
import os
import subprocess
import sys
import warnings

import numpy as np

from oracle import grid as ogrid
from oracle import rectify as orect
from oracle import reproject as orep
from oracle import resample as ores
from oracle.refkernels import REF_DIRS
from xcube_resampling_b200.constants import AGG_METHODS

from .helpers import GOLDEN

sys.path.insert(0, GOLDEN)
import fuzz_cases as fc  # noqa: E402  (tests/golden is a script directory, not a package)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _mismatches(want, got):
    return [key for key in want if got.get(key) != want[key]] + [key for key in got if key not in want]


def test_oracle_equals_reference_kernels_on_random_swaths():
    with open(os.path.join(GOLDEN, "fuzz_digests.json")) as fh:
        golden = json.load(fh)
    assert (golden["seed"], golden["n_cases"]) == (fc.SEED, fc.N_CASES)
    rng = np.random.default_rng(fc.SEED)

    got = {}
    for k, x, y, g, src in fc.rectify_cases(rng, fc.N_CASES):
        og = ogrid.RegularGrid(g["width"], g["height"], g["tile_w"], g["tile_h"], g["x_min"], g["y_min"], g["x_max"],
                               g["y_max"], g["x_res"], g["y_res"], g["j_up"])
        ij = orect.rectify_ij(x, y, og)
        d = got[str(k)] = {"windows": fc.digest(orect.source_windows(x, y, og)), "ij": fc.digest(ij)}
        for method in fc.METHODS:
            d[method] = fc.digest(orect.gather(src, ij, method, np.nan))
    bad = [f"{k}/{part}" for k in golden["rectify"] for part in _mismatches(golden["rectify"][k], got.get(k, {}))]
    assert len(got) == len(golden["rectify"]) and not bad, f"rectify: {len(got)} cases, mismatches {bad[:20]}"

    got = {}
    for k, xx, yy, arr, x_coord, y_coord, xres, yres in fc.reproject_cases(rng, fc.n_secondary(fc.N_CASES)):
        for method in fc.METHODS:
            with np.errstate(all="ignore"):
                out = orep.sample_window(xx, yy, arr, x_coord[0, 0, 0], y_coord[0, 0, 0], xres, yres, method)
            got[f"{k}/{method}"] = fc.digest(out)
    bad = _mismatches(golden["reproject"], got)
    assert not bad, f"reproject: {len(got)} cases, mismatches {bad[:20]}"

    got = {}
    for k, a, f_j, f_i in fc.coarsen_cases(rng, fc.n_secondary(fc.N_CASES)):
        for agg in AGG_METHODS:
            if agg == "mode" and a.dtype.kind == "f":
                continue
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                got[f"{k}/{agg}"] = fc.digest(ores.coarsen(a, f_j, f_i, agg))
    bad = _mismatches(golden["coarsen"], got)
    assert not bad, f"coarsen: {len(got)} cases, mismatches {bad[:20]}"

    if importlib.util.find_spec("numba") is None or not any(
            os.path.isdir(os.path.join(d, "xcube_resampling")) for d in REF_DIRS):
        return  # the reference cannot run here: the stored digests above stand for it
    r = subprocess.run([sys.executable, os.path.join(GOLDEN, "fuzz_oracle_vs_reference.py"), "--check-digests"],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    for line in (f"{fc.N_CASES} cases, 0 mismatches", "reproject: 40 cases, 0 mismatches",
                 "coarsen: 40 cases, 0 mismatches", "stored digests: 0 of 5 parts differ"):
        assert line in r.stdout, r.stdout[-2000:]
