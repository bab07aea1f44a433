"""The pieces shared by the affine / coarsen kernels -- the text of csrc/resample_common.cuh compiled for the
HOST (tests/hostmath) -- against numpy and scipy themselves, bit for bit, without a GPU:

* ``numpy_window_sum``: numpy's summation order over the two window axes of the (h, f_j, w, f_i) view that
  ``dask.array.coarsen`` hands to the reducers (coarsen.py:50-111) -- pairwise blocks of 8 along the innermost
  axis, rows accumulated sequentially;
* ``scipy_cast``: the output conversion of ``scipy.ndimage.affine_transform`` (ni_interpolation.c
  CASE_INTERP_OUT*) for integer outputs (affine.py:353-362);
* ``axis_order1``: the two taps and weights of scipy's order-1 filter incl. the mirrored tap at the upper edge.
"""

import ctypes

import numpy as np
import pytest
from scipy import ndimage


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    from . import hostmath

    try:
        return ctypes.CDLL(hostmath.build_resample(str(tmp_path_factory.mktemp("resamplehost"))))
    except RuntimeError as e:
        if "g++ not available" in str(e):
            pytest.skip(str(e))
        raise


def _p(a):
    return ctypes.c_void_p(a.ctypes.data)


@pytest.mark.parametrize("dtype,fn", [(np.float32, "xrsh_window_sums_f32"), (np.float64, "xrsh_window_sums_f64")])
@pytest.mark.parametrize("f_j,f_i", [(2, 2), (4, 4), (8, 8), (16, 16), (3, 5), (5, 9), (1, 7), (8, 3), (2, 32), (7, 100),
                                     (16, 15), (3, 128)])
def test_window_sums_follow_numpys_summation_order(lib, dtype, fn, f_j, f_i):
    rng = np.random.default_rng(f_j * 1000 + f_i)
    h, w = 7, 5
    a = ((rng.random((h * f_j, w * f_i)) - 0.3) * 1000).astype(dtype)
    want = np.sum(a.reshape(h, f_j, w, f_i), axis=(1, 3))  # what np.nansum / np.nanmean reduce, coarsen.py:72-90
    wins = np.ascontiguousarray(a.reshape(h, f_j, w, f_i).transpose(0, 2, 1, 3)).reshape(h * w, f_j * f_i)
    out = np.empty(h * w, dtype=dtype)
    getattr(lib, fn)(_p(wins), f_j, f_i, ctypes.c_long(h * w), _p(out))
    assert np.array_equal(out.reshape(h, w), want)
    assert want.dtype == dtype


def test_integer_output_conversion_is_scipys(lib):
    """All nine dtypes, including what C leaves undefined and scipy on x86 defines: NaN, +-inf, 2^63 after the
    +0.5 (INT64_MIN), beyond it (INT64_MAX), and values whose +0.5 rounds half to even in float64."""
    v = np.concatenate([np.linspace(-70000.0, 70000.0, 2801), np.arange(-6, 7) + 0.5, np.arange(-6, 7) - 0.5,
                        [0.0, -0.0, 0.49999999999999994, 254.5, 255.5, 32767.5, -32768.5, 65535.49, 65535.5, 2147483647.5,
                         -2147483648.5, 4e9, -4e9, 127.5, -128.5, 128.5, -129.5, 2.0 ** 31 - 0.5, 2.0 ** 31 + 0.5,
                         2.0 ** 32 - 0.5, 2.0 ** 32 + 0.5, np.nan, -np.nan, np.inf, -np.inf, 1e300, -1e300, 2.0 ** 63,
                         2.0 ** 63 - 1024, 2.0 ** 63 + 2048, 2.0 ** 64, -2.0 ** 63, -2.0 ** 63 - 4096, 2.0 ** 52 + 1,
                         -2.0 ** 52 - 1, 2.0 ** 53 + 2, 1.7e18]])
    n = v.size
    dtypes = (np.float32, np.float64, np.uint8, np.int8, np.uint16, np.int16, np.int32, np.uint32, np.int64)
    out = np.zeros(sum(np.dtype(d).itemsize for d in dtypes) * n, np.uint8)
    lib.xrsh_scipy_cast(_p(v), ctypes.c_long(n), _p(out))
    off = 0
    for dt in dtypes:  # scipy's own conversion: an identity affine_transform of the float64 values
        got = out[off:off + np.dtype(dt).itemsize * n].view(dt)
        off += np.dtype(dt).itemsize * n
        want = ndimage.affine_transform(v, [1.0], output=dt, order=0, mode="constant")
        assert np.array_equal(got, want, equal_nan=np.dtype(dt).kind == "f"), dt


@pytest.mark.parametrize("length", [2, 3, 8, 100])
def test_order1_taps_and_weights_are_scipys(lib, length):
    """One axis of scipy's order-1 filter, probed through affine_transform on unit impulses: the weight scipy
    gives source sample k at coordinate c is the response to an impulse at k."""
    rng = np.random.default_rng(length)
    c = np.concatenate([rng.random(200) * (length - 1), np.arange(length, dtype=np.float64), [length - 1 - 1e-12, 1e-12]])
    n = c.size
    k0, k1 = np.empty(n, np.int64), np.empty(n, np.int64)
    w0, w1 = np.empty(n), np.empty(n)
    inside = np.empty(n, np.uint8)
    lib.xrsh_axis_order1(_p(c), ctypes.c_long(n), ctypes.c_long(length), _p(k0), _p(k1), _p(w0), _p(w1), _p(inside))
    assert inside.all()
    ours = np.zeros((n, length))
    np.add.at(ours, (np.arange(n), k0), w0)
    np.add.at(ours, (np.arange(n), k1), w1)
    for k in range(length):
        impulse = np.zeros(length)
        impulse[k] = 1.0
        resp = ndimage.map_coordinates(impulse, [c], order=1, mode="constant", cval=0.0)
        assert np.array_equal(resp, ours[:, k]), (length, k)
    # outside the image: scipy returns cval
    out = np.array([-1e-9, length - 1 + 1e-9, -5.0, length + 3.0])
    lib.xrsh_axis_order1(_p(out), ctypes.c_long(4), ctypes.c_long(length), _p(k0), _p(k1), _p(w0), _p(w1), _p(inside))
    assert not inside[:4].any()
    assert np.array_equal(ndimage.map_coordinates(np.ones(length), [out], order=1, mode="constant", cval=-7.0), [-7.0] * 4)
