"""CPU pin of the two-method gather's algorithm (``k2_gather_dual`` / ``xrs_gather_ij2``): "the
nearest-neighbour sample is one of the four taps of the bilinear / triangular one" is checked, without a
GPU, against the oracle's ``_compute_var_image`` restatement and against the REFERENCE's own numba kernel
(``rectify.py:640-734``: through ``oracle/refkernels.py`` where it is installed, its golden outputs, stored
digests).  The GPU tests then only have to show that the CUDA kernel equals the oracle."""

import json
import os

import numpy as np
import pytest

from oracle import grid as ogrid
from oracle import rectify as orect

from .helpers import (GOLDEN, assert_same, covering_grid_args, digest, dual_swath, hand_made_ij, swath,
                      two_method_gather_np)

nan = np.nan


def _apply_fill(arr, valid, fill):
    out = arr.copy()
    out[:, ~valid] = fill
    return out


@pytest.mark.parametrize("smooth", [True, False])
@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.uint8, np.int16, np.uint16, np.int64])
def test_picked_tap_equals_oracle_on_ties_edges_and_holes(smooth, dtype):
    h, w = 40, 70
    ij = hand_made_ij(smooth, h, w, 64, 96)
    data = (np.random.default_rng(6).random((3, h, w)) * 200).astype(dtype)
    if np.dtype(dtype).kind == "f":
        data[0, 3:6, 10:30] = nan
        data[1, 20, 20] = np.inf
    fill = nan if np.dtype(dtype).kind == "f" else 9
    for method in ("bilinear", "triangular"):
        interp, near, valid = two_method_gather_np(data, ij, method)
        assert_same(_apply_fill(interp, valid, fill), orect.gather(data, ij, method, fill), f"{method} {dtype}")
        assert_same(_apply_fill(near, valid, fill), orect.gather(data, ij, "nearest", fill), f"nearest {dtype}")


@pytest.mark.parametrize("theta,seed", [(12.0, 1), (-40.0, 2), (85.0, 3)])
def test_picked_tap_equals_oracle_on_swaths(theta, seed):
    x, y = swath(260, 200, theta=theta, seed=seed)
    res = 0.0027
    size, xy_min = covering_grid_args(x, y, res)
    g = ogrid.regular_grid(size, xy_min, res, tile_size=96)
    data = np.random.default_rng(seed).random((2, 200, 260)).astype(np.float32)
    ij = orect.rectify_ij(x, y, g)
    for method in ("bilinear", "triangular"):
        interp, near, valid = two_method_gather_np(data, ij, method)
        assert_same(_apply_fill(interp, valid, nan), orect.gather(data, ij, method, nan), method)
        assert_same(_apply_fill(near, valid, nan), orect.gather(data, ij, "nearest", nan), "nearest")


def test_picked_tap_equals_the_reference_kernels():
    """The same against the reference's own ``_compute_var_image_sequential`` (tile by tile, as the
    reference runs it): against its outputs where the reference package and numba load (whose digests must
    then equal the stored ones), and everywhere against tests/golden/dual_swath_digests.json (its ``source``
    says what produced it)."""
    from oracle import refkernels

    x, y, g, data = dual_swath()
    with open(os.path.join(GOLDEN, "dual_swath_digests.json")) as fh:
        stored = json.load(fh)
    try:
        refkernels.load()
    except ImportError:
        ref = None
    else:
        _, ref = refkernels.rectify_pass(x, y, data, g, ("nearest", "bilinear", "triangular"), n_threads=4,
                                         keep_outputs=True)
        assert {m: digest(out) for m, out in ref.items()} == {m: stored[m] for m in ref}, "stored digests"
    ij = orect.rectify_ij(x, y, g)
    for method in ("bilinear", "triangular"):
        interp, near, valid = two_method_gather_np(data, ij, method)
        interp, near = _apply_fill(interp, valid, nan), _apply_fill(near, valid, nan)
        if ref is not None:
            assert_same(interp, ref[method], f"{method} vs reference kernel")
            assert_same(near, ref["nearest"], "nearest vs reference kernel")
        assert digest(interp) == stored[method], f"{method} vs stored digest"
        assert digest(near) == stored["nearest"], "nearest vs stored digest"
    assert valid.mean() > 0.3


def _golden_cases():
    from .helpers import load_golden

    return [str(c) for c in load_golden("rectify.npz")["cases"]]


@pytest.mark.parametrize("case", _golden_cases())
def test_picked_tap_equals_the_reference_goldens(case):
    """The committed outputs of the reference's own kernels (tests/golden/rectify.npz): the two-method
    logic reproduces the nearest AND the bilinear / triangular golden of every variable from the golden ij."""
    from .helpers import load_golden

    z = load_golden("rectify.npz")
    ij = z[f"{case}/ij"]
    for vname, fill in (("f32", nan), ("u8", 255), ("i16", -1), ("f64", nan)):
        src = z[f"{case}/src_{vname}"]
        for method in ("bilinear", "triangular"):
            interp, near, valid = two_method_gather_np(src, ij, method)
            interp, near = _apply_fill(interp, valid, fill), _apply_fill(near, valid, fill)
            if src.ndim == 2:
                interp, near = interp[0], near[0]
            assert_same(interp, z[f"{case}/out_{vname}_{method}"], f"{case} {vname}/{method}")
            assert_same(near, z[f"{case}/out_{vname}_nearest"], f"{case} {vname}/nearest")


def test_picked_tap_at_the_full_size_of_config_c2():
    """BASELINE config C2 at full size (4865 x 4091 swath -> 7992 x 5013, 28 M valid target pixels): the
    picked tap equals the oracle's nearest gather and the shared taps its bilinear gather, one band."""
    from xcube_resampling_b200 import synthetic as syn

    w, h, res = syn.OLCI_WIDTH, syn.OLCI_HEIGHT, syn.OLCI_RES_DEG
    lon, lat = syn.swath(w, h, res=res, theta=12.0, seed=0)
    size, xy_min = syn.covering_grid_args(lon, lat, res)
    g = ogrid.regular_grid(size, xy_min, res, tile_size=512)
    ij = orect.rectify_ij(lon, lat, g)
    band = syn.band_stack(1, h, w, seed=0)
    interp, near, valid = two_method_gather_np(band, ij, "bilinear")
    assert 0.6 < valid.mean() < 0.8
    assert_same(_apply_fill(interp, valid, nan), orect.gather(band, ij, "bilinear", nan), "C2 bilinear")
    assert_same(_apply_fill(near, valid, nan), orect.gather(band, ij, "nearest", nan), "C2 nearest")
