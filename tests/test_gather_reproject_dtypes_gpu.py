"""The shared gather / reprojection case table (tests/gather_cases.py) on the GPU through the C ABI --
``xrs_gather_ij``, ``xrs_gather_ij2``, ``xrs_rectify_gather`` and ``xrs_reproject`` -- on pitched sources (16-byte
row pitch: the TMA-staged kernels) and unpitched ones (an odd row pitch: the direct kernel, the two-pass fallback
of the dual gather), bit for bit with the sign of zero counted.  Plus one ``rectify_dataset`` case per finding:
int64 nearest samples beyond 2^53, int64 interpolations that round to 2^63 (the device's own conversion would
saturate), NaN fills into integer variables, the default fill of uint32.  (K3's nearest path copies the stored
value, as the reference's direct indexing does; its int64 cases are in the table.)"""

import numpy as np
import pytest

from oracle import rectify as orect

from xcube_resampling_b200 import GridMapping

from . import gather_cases as gc
from .helpers import assert_bits

pytestmark = pytest.mark.gpu
nan = np.nan


@pytest.fixture(scope="module")
def xrs():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import xcube_resampling_b200 as pkg
    from xcube_resampling_b200 import _dev, rectify, reproject

    pkg.dev, pkg.rect, pkg.rep = _dev, rectify, reproject
    return pkg


def _to_device(xrs, a, pitched: bool):
    """Pitched: 16-byte aligned rows (TMA can describe them); unpitched: a row pitch of w + 1 elements, which no
    dtype makes a multiple of 16 bytes."""
    if pitched:
        return xrs.dev.to_device_pitched(a)
    n, h, w = a.shape
    wide = np.zeros((n, h, w + 1), dtype=a.dtype)
    wide[:, :, :w] = a
    return xrs.dev.to_device(wide)[:, :, :w]


def _resident(xrs, c, pitched):
    """(device source, window_origin, full_size) as the kernels get it for case ``c``."""
    nb, h, w = c.src.shape
    if c.window is None:
        return _to_device(xrs, c.src, pitched), (0, 0), (w, h)
    i0, j0, i1, j1 = c.window
    return _to_device(xrs, np.ascontiguousarray(c.src[:, j0:j1, i0:i1]), pitched), (i0, j0), (w, h)


@pytest.mark.parametrize("pitched", [True, False])
@pytest.mark.parametrize("case_id", gc.gather_case_ids())
def test_gather_ij_and_ij2(xrs, case_id, pitched):
    c = gc.gather_case(case_id)
    sd, origin, full = _resident(xrs, c, pitched)
    ij = xrs.dev.to_device(c.ij)
    got = xrs.rect.gather_ij(sd, ij, c.method, c.fill, window_origin=origin, full_size=full)
    assert_bits(xrs.dev.to_host(got), c.want, f"{case_id}: xrs_gather_ij, pitched={pitched}", skip=c.skip)
    if c.method != "nearest":
        got_i, got_n = xrs.rect.gather_ij_pair(sd, ij, c.method, c.fill, c.fill, window_origin=origin, full_size=full)
        assert_bits(xrs.dev.to_host(got_i), c.want, f"{case_id}: xrs_gather_ij2 {c.method}, pitched={pitched}", skip=c.skip)
        assert_bits(xrs.dev.to_host(got_n), c.want_near, f"{case_id}: xrs_gather_ij2 nearest, pitched={pitched}",
                    skip=c.skip)


@pytest.mark.parametrize("pitched", [True, False])
@pytest.mark.parametrize("case_id", [i for i in gc.gather_case_ids() if i.endswith("-swath")])
def test_rectify_gather(xrs, case_id, pitched):
    c = gc.gather_case(case_id)
    x, y, size, xy_min, res, tile = c.swath
    gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=tile)
    xd, yd = xrs.dev.to_device(x), xrs.dev.to_device(y)
    got = xrs.rect.RectifyPlan(gm, xd.device).rectify_gather(xd, yd, _to_device(xrs, c.src, pitched), c.method, c.fill)
    assert_bits(xrs.dev.to_host(got), c.want, f"{case_id}: xrs_rectify_gather, pitched={pitched}", skip=c.skip)


@pytest.mark.parametrize("pitched", [True, False])
@pytest.mark.parametrize("case_id", [c.id for c in gc.reproject_cases(GridMapping)])
def test_reproject(xrs, case_id, pitched):
    c = {c.id: c for c in gc.reproject_cases(xrs.GridMapping)}[case_id]
    src_gm, tgt_gm = gc.reproject_grids(xrs.GridMapping, c.tile)
    plan = xrs.rep.ReprojectPlan(src_gm, tgt_gm)
    out_dtype = None if c.out_f64 or c.method != "bilinear" else c.src.dtype
    got = plan.run(_to_device(xrs, c.src, pitched), c.method, c.fill, out_dtype=out_dtype)
    assert_bits(xrs.dev.to_host(got), c.want, f"{case_id}: xrs_reproject, pitched={pitched}", skip=c.skip)


# ---------------------------------------------------------------------------
# one dataset-level case per finding
# ---------------------------------------------------------------------------
def _swath_dataset(xrs, **data_vars):
    (x, y, size, xy_min, res, tile), ij = gc._swath_scene()
    ds = xrs.Dataset(data_vars={k: (("y", "x"), v) for k, v in data_vars.items()},
                     coords=dict(lon=(("y", "x"), x), lat=(("y", "x"), y)))
    src_gm = xrs.GridMapping.from_coords(x, y, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
    tgt_gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=tile)
    return ds, src_gm, tgt_gm, ij


def test_rectify_dataset_int64_nearest_and_rounding_to_2_63(xrs):
    """int64 nearest samples beyond 2^53 are rounded (INT64_MAX -> INT64_MIN); bilinear samples between values within
    512 of INT64_MAX round to 2^63 and store INT64_MIN, as x86 does."""
    rng = np.random.default_rng(3)
    big = rng.choice(np.array([2**63 - 1, 2**63 - 512, 2**53 + 1, 2526497193922298463], dtype=np.int64), (90, 120))
    ds, src_gm, tgt_gm, ij = _swath_dataset(xrs, near=big, lin=big)
    out = xrs.rectify_dataset(ds, target_gm=tgt_gm, source_gm=src_gm, interp_methods={"near": "nearest", "lin": "bilinear"})
    assert_bits(out["near"].values, orect.gather(big, ij, "nearest", -1), "int64 nearest")
    want = orect.gather(big, ij, "bilinear", -1)
    assert (want == -(2**63)).any()
    assert_bits(out["lin"].values, want, "int64 bilinear")


def test_rectify_dataset_nan_and_uint32_fills(xrs):
    """NaN fills into integer variables take x86's conversion; uint32's default fill -1 is 0xFFFFFFFF."""
    rng = np.random.default_rng(4)
    i32 = rng.integers(-2**31, 2**31, (90, 120), dtype=np.int32)
    i64 = rng.integers(-2**62, 2**62, (90, 120), dtype=np.int64)
    u32 = rng.integers(0, 2**32, (90, 120), dtype=np.uint32)
    ds, src_gm, tgt_gm, ij = _swath_dataset(xrs, i32=i32, i64=i64, u32=u32)
    out = xrs.rectify_dataset(ds, target_gm=tgt_gm, source_gm=src_gm, interp_methods="bilinear",
                              fill_values={"i32": nan, "i64": nan})
    no_src = np.isnan(ij[0]) | np.isnan(ij[1])
    assert no_src.any()
    assert (out["i32"].values[no_src] == -(2**31)).all() and (out["i64"].values[no_src] == -(2**63)).all()
    assert (out["u32"].values[no_src] == 0xFFFFFFFF).all()
    import warnings

    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        for name, a, fill in (("i32", i32, nan), ("i64", i64, nan), ("u32", u32, -1)):
            assert_bits(out[name].values, orect.gather(a, ij, "bilinear", fill), name)

