"""The affine / coarsen family as kernels on the host: csrc/resample.cu and csrc/resample_fast.cu compiled
unchanged for the CPU (tests/hostmath.build_resample_kernels), launch code and C ABI included, run over the case
table of tests/resample_cases.py.  For every case: the output equals the oracle's bit for bit (sign of zero
included), the kernel that ran is the one the table's restatement of the dispatch rules expects, and no load is
misaligned for its width -- a misaligned vector load is a fault on the GPU, which x86 would let pass.  The
SIMD-in-a-word intrinsics of the shim are held to a numpy model of each lane."""

import numpy as np
import pytest

from . import resample_cases
from .helpers import assert_bits

CASES = resample_cases.cases()


@pytest.fixture(scope="module")
def rsk(tmp_path_factory):
    from . import hostmath

    try:
        so = hostmath.build_resample_kernels(str(tmp_path_factory.mktemp("rskhost")))
    except RuntimeError as e:
        if "g++ not available" in str(e):
            pytest.skip(str(e))
        raise
    return hostmath.ResampleKernels(so)


def run_case(rsk, case):
    from . import hostmath

    pitch, sstride = case.layout.strides(case.src.shape)
    view = hostmath.aligned_view(case.src, pitch, sstride, case.layout.elem_off)
    a = case.args
    if case.kind == "coarsen":
        return rsk.coarsen(view, a["factors"], a["agg"])
    if case.kind == "has_nan":
        return rsk.has_nan(view)
    if case.kind == "recover":
        return rsk.affine_recover(view, a["scale"], a["offset"], a["out_hw"], a["cval"], a["agg"], a["factors"],
                                  a["slice_blend"])
    return rsk.affine(view, a["scale"], a["offset"], a["out_hw"], a["order"], a["cval"], a["agg"], a["factors"],
                      a["slice_blend"])


def test_case_table_is_complete():
    kernels = {c.kernel for c in CASES}
    assert kernels >= {"k4_affine_generic", "k4_affine_recover", "k4_has_nan", "k5_window_reduce<simple>",
                       "k5_window_reduce<sort>", "k5_blend2_x4", "k5_u8x4_reduce", "k5_u8x2_sort"}
    assert {c.src.dtype for c in CASES} == {np.dtype(d) for d in resample_cases.DTYPES}


@pytest.mark.parametrize("chunk", range(8))
def test_cases_on_the_host_build(rsk, chunk):
    failures = []
    for case in CASES[chunk::8]:
        got, kernels, misaligned = run_case(rsk, case)
        try:
            assert misaligned == 0, f"{misaligned} misaligned loads"
            assert kernels == ([case.kernel] if case.kernel else []), f"ran {kernels}, expected {case.kernel}"
            if case.kind == "has_nan":
                assert got == case.want
            else:
                want = np.asarray(case.want)
                assert_bits(got, want if want.ndim == 3 else want.reshape(got.shape), case.id, case.skip)
        except AssertionError as e:
            failures.append(f"{case.id}: {e}")
    assert not failures, f"{len(failures)} cases fail:\n" + "\n".join(failures[:20])


LANE_WORDS = np.array([0x00000000, 0x7f7f7f7f, 0x80808080, 0xffffffff, 0x00ff7f80, 0x807fff00, 0x01010101, 0xfefefefe,
                       0x0000ffff, 0xffff0000, 0x7fff8000, 0x00800080], dtype=np.uint32)


def _lanes(v, bits):
    v = np.asarray(v, dtype=np.uint64)
    return [(v >> np.uint64(bits * k)) & np.uint64((1 << bits) - 1) for k in range(32 // bits)]


def _pack(lanes, bits):
    r = np.zeros_like(lanes[0])
    for k, x in enumerate(lanes):
        r |= (x & np.uint64((1 << bits) - 1)) << np.uint64(bits * k)
    return r.astype(np.uint32)


def _model(op, a, b, c):
    if op == "byte_perm":
        v = (b.astype(np.uint64) << np.uint64(32)) | a.astype(np.uint64)
        sel = _lanes(c, 4)
        return _pack([(v >> (np.uint64(8) * sel[k])) & np.uint64(0xff) for k in range(4)], 8)
    if op == "dp4a":
        return (c.astype(np.uint64) + sum(x * y for x, y in zip(_lanes(a, 8), _lanes(b, 8)))).astype(np.uint32)
    bits = 16 if op.endswith("2") else 8
    fn = {"vminu": np.minimum, "vmaxu": np.maximum, "vhaddu": lambda x, y: (x + y) >> np.uint64(1),
          "vadd": lambda x, y: x + y, "vcmpeq": lambda x, y: np.where(x == y, 0xff, 0).astype(np.uint64),
          "vcmpne": lambda x, y: np.where(x != y, 0xff, 0).astype(np.uint64),
          "vcmpgtu": lambda x, y: np.where(x > y, 0xff, 0).astype(np.uint64)}[op[:-1]]
    return _pack([fn(x, y) for x, y in zip(_lanes(a, bits), _lanes(b, bits))], bits)


@pytest.mark.parametrize("op", ["byte_perm", "vminu4", "vmaxu4", "vminu2", "vmaxu2", "vhaddu4", "vadd4", "vcmpeq4",
                                "vcmpne4", "vcmpgtu4", "dp4a"])
def test_simd_intrinsics_lane_by_lane(rsk, op):
    """Random words, the 0x00 / 0x7f / 0x80 / 0xff lanes and pairs whose lane sums carry (must not cross lanes)."""
    rng = np.random.default_rng(11)
    a = np.concatenate([rng.integers(0, 2 ** 32, 4000, dtype=np.uint64).astype(np.uint32), np.repeat(LANE_WORDS, 12)])
    b = np.concatenate([rng.integers(0, 2 ** 32, 4000, dtype=np.uint64).astype(np.uint32), np.tile(LANE_WORDS, 12)])
    if op == "byte_perm":  # default mode: selector nibbles 0..7
        c = _pack([rng.integers(0, 8, a.size).astype(np.uint64) for _ in range(8)], 4)
        c[:16] = [0x5140, 0x7362, 0x5410, 0x7632, 0x6420, 0x7531, 0x2200, 0x3311, 0x4400, 0x5511, 0x6622, 0x7733,
                  0x3210, 0x7654, 0x0000, 0x7777]
    else:
        c = rng.integers(0, 2 ** 32, a.size, dtype=np.uint64).astype(np.uint32)
    got = rsk.simd(op, a, b, c)
    want = _model(op, a, b, c)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, f"{op}: {bad.size} words differ, first a={a[bad[0]]:#x} b={b[bad[0]]:#x}: " \
                          f"{got[bad[0]]:#x} vs {want[bad[0]]:#x}"


@pytest.mark.parametrize("f", [2, 4, 8])
def test_u8x4_kernel_on_its_own(rsk, f):
    """k5_u8x4_reduce launched directly with every aggregation it implements: its median / mode (byte-wise sorting
    network, half-to-even of the middle pair, run lengths with the lowest value winning ties) sit behind
    k5_u8x2_sort in the dispatch, which takes every layout they could get."""
    from . import hostmath

    cases = [c for c in CASES if c.kind == "coarsen" and c.src.dtype == np.uint8 and c.args["factors"] == (f, f)
             and c.src.shape[2] % (4 * f) == 0]
    assert cases
    failures = []
    for case in cases:
        agg = case.args["agg"]
        if agg in ("prod", "std", "var"):
            continue
        n, h, w = case.src.shape
        got, kernels, misaligned = rsk.u8x4(hostmath.aligned_view(case.src, w, h * w, 0), f, agg)
        try:
            assert kernels == ["k5_u8x4_reduce"] and misaligned == 0, (kernels, misaligned)
            assert_bits(got, np.asarray(case.want).astype(got.dtype), case.id)
        except AssertionError as e:
            failures.append(f"{case.id}: {e}")
    assert not failures, "\n".join(failures[:20])
