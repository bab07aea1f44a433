"""The case table of tests/resample_cases.py on the B200: the same inputs, memory layouts and C ABI calls as
test_host_k4k5_kernels.py runs on the host build, through the Python layer (affine_resample_dev, coarsen_dev,
has_nan_dev), held to the same oracle bit for bit and to the same expected kernel (profiler names).  Then one
affine_transform_dataset case per int64 / fill finding: nearest int64, aligned bilinear int64 / 2, int64 3 x 3
median, int32 with fill_values=NaN."""

import numpy as np
import pytest

from oracle import resample as ores

from . import resample_cases
from .helpers import assert_bits

pytestmark = pytest.mark.gpu
CASES = resample_cases.cases()


@pytest.fixture(scope="module")
def xrs():
    import torch

    assert torch.cuda.is_available()
    import xcube_resampling_b200 as pkg
    from xcube_resampling_b200 import _dev, _lib, affine

    pkg.dev, pkg.aff, pkg.lib = _dev, affine, _lib
    return pkg


def _device_view(xrs, case):
    """The case's source on the device with its layout: a 256-byte aligned buffer, the view elem_off elements in."""
    import torch

    src = case.src
    n, h, w = src.shape
    pitch, sstride = case.layout.strides(src.shape)
    es = src.dtype.itemsize
    n_el = case.layout.elem_off + (n - 1) * sstride + (h - 1) * pitch + w
    host = np.zeros(n_el, dtype=src.dtype)
    np.lib.stride_tricks.as_strided(host[case.layout.elem_off:], src.shape, (sstride * es, pitch * es, es))[...] = src
    raw = torch.from_numpy(host.view(np.uint8)).cuda()
    flat = raw.view(xrs.dev.torch_dtype(src.dtype))
    assert flat.data_ptr() % 256 == 0
    return torch.as_strided(flat, (n, h, w), (sstride, pitch, 1), case.layout.elem_off)


def _run(xrs, case):
    lib = xrs.lib
    lib.profile_collect()
    lib.profile_enable(True)
    try:
        v, a = _device_view(xrs, case), case.args
        if case.kind == "has_nan":
            out = xrs.aff.has_nan_dev(v)
        elif case.kind == "coarsen":
            out = xrs.dev.to_host(xrs.aff.coarsen_dev(v, a["factors"], a["agg"]))
        else:
            out = xrs.dev.to_host(xrs.aff.affine_resample_dev(v, a["scale"], a["offset"], a["out_hw"], a.get("order", 1),
                                                              a["cval"], a["agg"], a["factors"], a["slice_blend"],
                                                              recover=case.kind == "recover"))
    finally:
        lib.profile_enable(False)
    return out, list(lib.profile_collect())


@pytest.mark.parametrize("chunk", range(8))
def test_cases_on_the_gpu(xrs, chunk):
    failures = []
    for case in CASES[chunk::8]:
        got, kernels = _run(xrs, case)
        try:
            assert kernels == ([case.kernel] if case.kernel else []), f"ran {kernels}, expected {case.kernel}"
            if case.kind == "has_nan":
                assert got == case.want
            else:
                assert_bits(got, np.asarray(case.want), case.id, case.skip)
        except AssertionError as e:
            failures.append(f"{case.id}: {e}")
    assert not failures, f"{len(failures)} cases fail:\n" + "\n".join(failures[:20])


def _dataset(xrs, values):
    h, w = values.shape  # 0.5-degree cells, x from 0, y from 6 down: every grid matrix below is exact
    coords = dict(lon=0.25 + 0.5 * np.arange(w), lat=6.0 - 0.25 - 0.5 * np.arange(h))
    return xrs.Dataset(data_vars=dict(v=(("lat", "lon"), values)), coords=coords)


def test_affine_transform_dataset_int64_and_fill_findings(xrs):
    rng = np.random.default_rng(3)
    big = (rng.uniform(-1, 1, (12, 18)) * 1.7e18).astype(np.int64)
    big[::3, ::4] = 2 ** 52 + 1
    big[1, 1] = 1_700_000_000_123_456_789
    ds = _dataset(xrs, big)
    gm = xrs.GridMapping.from_dataset(ds)
    # nearest (the default for integers), shifted by two cells: float64 round trip, fill -1 outside
    out = xrs.affine_transform_dataset(ds, xrs.GridMapping.regular((18, 12), (1.0, -1.0), 0.5, gm.crs), source_gm=gm)
    want = ores.resample_array(big, ((1.0, 0.0, 2.0), (0.0, 1.0, 2.0)), (12, 18), 0, "center", False, -1)
    assert_bits(out["v"].values, want, "int64 nearest")
    # bilinear 2x down-scaling on aligned grids: the generic kernel, samples rounded like scipy's
    out = xrs.affine_transform_dataset(ds, xrs.GridMapping.regular((9, 6), (0.0, 0.0), 1.0, gm.crs), source_gm=gm,
                                       interp_methods="bilinear", agg_methods="mean")
    want = ores.resample_array(big, ((2.0, 0.0, 0.0), (0.0, 2.0, 0.0)), (6, 9), 1, "mean", False, -1)
    assert_bits(out["v"].values, want, "int64 bilinear / 2")
    # 3 x 3 median of values around 1.7e18: numpy's float64 middle value, rounded and cast back
    near = (1_700_000_000_000_000_000 + rng.integers(-10 ** 6, 10 ** 6, (12, 18))).astype(np.int64)
    ds3 = _dataset(xrs, near)
    out = xrs.affine_transform_dataset(ds3, xrs.GridMapping.regular((6, 4), (0.0, 0.0), 1.5, gm.crs), source_gm=gm,
                                       interp_methods="bilinear", agg_methods="median")
    want = ores.resample_array(near, ((3.0, 0.0, 0.0), (0.0, 3.0, 0.0)), (4, 6), 1, "median", False, -1)
    assert_bits(out["v"].values, want, "int64 3x3 median")
    # int32 with fill_values=NaN: scipy's conversion of NaN is INT32_MIN
    i32 = rng.integers(-2 ** 31, 2 ** 31, (12, 18)).astype(np.int32)
    ds4 = _dataset(xrs, i32)
    out = xrs.affine_transform_dataset(ds4, xrs.GridMapping.regular((18, 12), (1.0, -1.0), 0.5, gm.crs), source_gm=gm,
                                       fill_values=np.nan)
    want = ores.resample_array(i32, ((1.0, 0.0, 2.0), (0.0, 1.0, 2.0)), (12, 18), 0, "center", False, np.nan)
    assert (want == np.iinfo(np.int32).min).any()
    assert_bits(out["v"].values, want, "int32 NaN fill")
