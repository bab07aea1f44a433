"""K2 and K3 as kernels on the host across all nine dtypes at full range (tests/gather_cases.py), bit for bit with
the sign of zero counted: k2_gather_staged / k2_gather_direct / k2_gather_dual / the fused staged gather
(csrc/gather.cu, csrc/gather_dual.cu) and k3_reproject (csrc/reproject.cu), each compiled unchanged for the host
(tests/hostmath.build_k2 / build_k3), against the oracle.

The cases pin what the reference stores:
* int64 nearest samples take the float64 round trip of the reference's source window (rectify.py:628-630): values
  beyond 2^53 are rounded, INT64_MAX becomes INT64_MIN;
* float64 -> integer stores and fills have x86's results (xrs_casts.h): an int64 interpolation that rounds to 2^63
  is INT64_MIN, NaN fills are INT32_MIN / INT64_MIN for int32 / int64 and 0 for the other integer types, the
  default fill -1 of a uint32 variable is 0xFFFFFFFF.
"""

import numpy as np
import pytest

import xcube_resampling_b200 as xrs
from oracle import grid as ogrid
from oracle import rectify as orect

from . import gather_cases as gc
from .helpers import assert_bits
from .test_host_k3 import _case_utm_from_geographic, _fake_transform_points, _oracle

nan = np.nan


def _build(tmp_path_factory, name):
    from . import hostmath

    try:
        return getattr(hostmath, f"build_{name}")(str(tmp_path_factory.mktemp(f"{name}host_dtypes")))
    except RuntimeError as e:
        if "g++ not available" in str(e):
            pytest.skip(str(e))
        raise


@pytest.fixture(scope="module")
def k2_so(tmp_path_factory):
    return _build(tmp_path_factory, "k2")


@pytest.fixture(scope="module")
def k1_so(tmp_path_factory):
    return _build(tmp_path_factory, "k1")


@pytest.fixture(scope="module")
def k3_so(tmp_path_factory):
    return _build(tmp_path_factory, "k3")


@pytest.mark.parametrize("case_id", gc.gather_case_ids())
def test_k2_staged_and_direct(k2_so, case_id):
    from . import hostmath

    c = gc.gather_case(case_id)
    for staged in (True, False):
        out, (boxes, _) = hostmath.k2_gather(k2_so, c.resident, c.ij, c.method, c.fill, staged=staged, window=c.window)
        assert_bits(out, c.want, f"{case_id}: k2_gather_{'staged' if staged else 'direct'}", skip=c.skip)
        if staged:
            assert (boxes > 0) is (c.staged == "box"), boxes


@pytest.mark.parametrize("case_id", [i for i in gc.gather_case_ids() if "-nearest-" not in i])
def test_k2_dual(k2_so, case_id):
    """Both outputs of one k2_gather_dual launch: the interpolated bands and the nearest ones picked among its taps."""
    from . import hostmath

    c = gc.gather_case(case_id)
    out_i, out_n, (boxes, _) = hostmath.k2_gather_dual(k2_so, c.resident, c.ij, c.method, c.fill, c.fill, window=c.window)
    assert_bits(out_i, c.want, f"{case_id}: dual, {c.method}", skip=c.skip)
    assert_bits(out_n, c.want_near, f"{case_id}: dual, nearest", skip=c.skip)
    assert (boxes > 0) is (c.staged == "box")


@pytest.mark.parametrize("case_id", [i for i in gc.gather_case_ids() if i.endswith("-swath")])
def test_k2_fused(k2_so, k1_so, case_id):
    """K1's claim stage, then the staged gather resolving the claim words in registers (xrs_rectify_gather)."""
    from . import hostmath

    c = gc.gather_case(case_id)
    x, y, size, xy_min, res, tile = c.swath
    g = ogrid.regular_grid(size, xy_min, res, tile_size=tile)
    windows = orect.source_windows(x, y, g)
    _, claims, _ = hostmath.k1(k1_so, x, y, windows, g)
    got = hostmath.k2_gather_fused(k2_so, c.src, x, y, windows, claims, g, c.method, c.fill)
    assert_bits(got, c.want, f"{case_id}: fused", skip=c.skip)


def test_int64_nearest_takes_the_float64_round_trip(k2_so):
    """The finding itself, spelled out: INT64_MAX reads back as INT64_MIN, 2^53 + 1 as 2^53, and a value beyond 2^53
    as its nearest double -- in all three K2 kernels."""
    from . import hostmath

    v = np.array([2**63 - 1, 2**53 + 1, 2526497193922298463, -(2**63), 5], dtype=np.int64)
    want = np.array([-(2**63), 2**53, 2526497193922298368, -(2**63), 5], dtype=np.int64)
    src = np.tile(v, (1, 4, 1))                       # (1, 4, 5)
    ij = np.stack(np.meshgrid(np.arange(5.0), np.arange(4.0)))
    for staged in (True, False):
        out, _ = hostmath.k2_gather(k2_so, src, ij, "nearest", -1, staged=staged)
        assert_bits(out[0], np.tile(want, (4, 1)), f"staged={staged}")
    _, out_n, _ = hostmath.k2_gather_dual(k2_so, src, ij, "bilinear", -1, -1)
    assert_bits(out_n[0], np.tile(want, (4, 1)), "dual")


def test_int64_interpolation_rounding_to_2_63_is_int64_min(k2_so):
    """A bilinear sample between INT64_MAX - 511 and INT64_MAX rounds to 2^63 in float64: x86 stores INT64_MIN
    (where the device's saturating conversion would give INT64_MAX)."""
    from . import hostmath

    src = np.array([[[2**63 - 512, 2**63 - 1], [2**63 - 1, 2**63 - 1]]], dtype=np.int64)
    ij = np.array([[[0.5]], [[0.5]]])
    for method in ("bilinear", "triangular"):
        out, _ = hostmath.k2_gather(k2_so, src, ij, method, 0, staged=True)
        assert out[0, 0, 0] == -(2**63) == orect.gather(src, ij, method, 0)[0, 0, 0], method


def test_fills_take_x86_conversions(k2_so):
    """NaN into integers, -1 into uint32 (the default integer fill), and int64 fills beyond 2^53 (rounded: the one
    remaining fill deviation, DESIGN.md section 5)."""
    from . import hostmath

    ij = np.full((2, 1, 3), nan)
    want = {np.int8: 0, np.uint8: 0, np.int16: 0, np.uint16: 0, np.int32: -(2**31), np.uint32: 0, np.int64: -(2**63)}
    for dt, v in want.items():
        out, _ = hostmath.k2_gather(k2_so, np.zeros((1, 2, 2), dt), ij, "bilinear", nan)
        assert (out == v).all(), dt
    out, _ = hostmath.k2_gather(k2_so, np.zeros((1, 2, 2), np.uint32), ij, "nearest", -1)
    assert (out == 0xFFFFFFFF).all() and (orect.gather(np.zeros((1, 2, 2), np.uint32), ij, "nearest", -1) == out).all()
    out, _ = hostmath.k2_gather(k2_so, np.zeros((1, 2, 2), np.int64), ij, "nearest", 2**53 + 1)
    assert (out == 2**53).all()


# ---------------------------------------------------------------------------
# K3
# ---------------------------------------------------------------------------
@pytest.fixture()
def rep(monkeypatch):
    import xcube_resampling_b200.reproject as rep

    monkeypatch.setattr(rep, "transform_points", _fake_transform_points)
    return rep


@pytest.mark.parametrize("case_id", [c.id for c in gc.reproject_cases(xrs.GridMapping)])
def test_k3_identity_transform(k3_so, rep, case_id):
    """Separable kernel (row-block form for bilinear): diff_as_f64's wrapping differences and cast_like_numpy inside
    the kernel, full-range values, padded taps reading the fill."""
    from . import hostmath

    c = {c.id: c for c in gc.reproject_cases(xrs.GridMapping)}[case_id]
    src_gm, tgt_gm = gc.reproject_grids(xrs.GridMapping, c.tile)
    w = rep.get_source_windows(src_gm, tgt_gm)
    got, (plan, sep, nodes) = hostmath.k3_reproject(k3_so, c.src, src_gm, tgt_gm, w, c.method, c.fill, out_f64=c.out_f64)
    assert sep and not nodes
    assert_bits(got, c.want, case_id, skip=c.skip)


@pytest.mark.parametrize("dtype,method", [(dt, m) for dt in (np.int64, np.int8, np.uint32, np.float64)
                                          for m in ("nearest", "bilinear", "triangular")
                                          if (dt, m) != (np.uint32, "triangular")])  # uint32 wraps out of range
def test_k3_lattice_and_exact_forms(k3_so, rep, dtype, method):
    """A real projection (geographic source -> UTM target): the lattice and the exact per-pixel forms, with the
    tolerances of test_host_k3.py (libm stands in for CUDA's math library: nearest may pick the other tap at a
    rounding tie, interpolations agree to 1e-6 relative)."""
    from . import hostmath

    src_gm, tgt_gm = _case_utm_from_geographic(n=96)
    data = gc.source(dtype, 2, src_gm.height, src_gm.width, seed=7)
    # band 0 smooth over the full range (a real projection moves the taps a little, so only a smooth band can be held
    # to a tolerance); band 1 extremes, for nearest
    lo, hi = (np.iinfo(dtype).min, np.iinfo(dtype).max) if np.dtype(dtype).kind in "iu" else (-np.finfo(dtype).max / 4, np.finfo(dtype).max / 4)
    ramp = np.clip(np.linspace(lo, hi, data[0].size).round(), lo, np.nextafter(float(hi), 0.0))   # float(INT64_MAX) is 2^63
    data[0] = ramp.reshape(data[0].shape).astype(dtype)
    fill = gc.reproject_fill(dtype)
    w = rep.get_source_windows(src_gm, tgt_gm)
    with np.errstate(all="ignore"):
        want = _oracle(src_gm, tgt_gm, data, method, fill, 4326, 32632)
    for kw in ({}, dict(exact_only=True)):
        got, (plan, sep, nodes) = hostmath.k3_reproject(k3_so, data, src_gm, tgt_gm, w, method, fill, **kw)
        assert not sep and got.dtype == want.dtype
        if method == "nearest":
            same = (got == want) | (np.isnan(got) & np.isnan(want) if got.dtype.kind == "f" else False)
            assert float(np.mean(~same)) < 1e-3, kw
        else:
            g64, w64 = got[0].astype(np.float64), want[0].astype(np.float64)
            np.testing.assert_allclose(g64, w64, rtol=1e-6, atol=np.abs(w64[np.isfinite(w64)]).max() * 1e-9,
                                       equal_nan=True, err_msg=str(kw))
