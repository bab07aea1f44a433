"""The device decode of compressed Zarr chunks as kernels on the host: csrc/decode.cu compiled unchanged for the CPU
(tests/hostmath/zarr_decode.py), launch code and C ABI included, run over the case table of tests/zarr_decode_cases.py.

Every slot equals the host decode (``ZarrV2Source.read_bands`` / ``DecodedSource.read_bands``) bit for bit, with the
poison around it and the canary after the workspace intact, and no launch exceeds CUDA's grid and block limits (the
launch shim refuses what the device would refuse).  Every malformed case is reported with its reason and
chunk, writes nothing outside its slot or workspace, and reads nothing past the end of its file: the file ends at a
page that may not be read."""

import ctypes
import mmap

import numpy as np
import pytest

from xcube_resampling_b200._pipeline import decode_error, zarr_decode, zarr_workspace_bytes

from . import zarr_decode_cases

CASES = zarr_decode_cases.cases()
POISON, CANARY = 0x5A, 0xC3


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    from .hostmath.zarr_decode import build_decode

    try:
        so = build_decode(str(tmp_path_factory.mktemp("decodehost")))
    except RuntimeError as e:
        if "g++ not available" in str(e):
            pytest.skip(str(e))
        raise
    from xcube_resampling_b200._lib import SIGNATURES

    lib = ctypes.CDLL(so)
    for name in ("xrs_zarr_decode", "xrs_zarr_decode_workspace_bytes", "xrs_last_error"):
        fn = getattr(lib, name)  # attribute access caches the function object; lib[name] would not
        fn.restype, fn.argtypes = SIGNATURES[name]
    lib.xrsh_bad_launches.restype, lib.xrsh_bad_launches.argtypes = ctypes.c_long, []
    return lib


class Guarded:
    """``data`` copied so that its last byte is the last readable one: the next page is mapped PROT_NONE."""

    def __init__(self, data: bytes):
        page = mmap.PAGESIZE
        n = -(-max(len(data), 1) // page) * page
        self.map = mmap.mmap(-1, n + page)
        base = ctypes.addressof(ctypes.c_char.from_buffer(self.map))
        libc = ctypes.CDLL(None)
        libc.mprotect.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
        assert libc.mprotect(ctypes.c_void_p(base + n), page, 0) == 0
        self.addr = base + n - len(data)
        ctypes.memmove(self.addr, data, len(data))


def run_case(lib, case, root):
    """Decode ``case`` through ``lib``; returns (slot, expected, error word, paths, intact)."""
    source = case.source(root)
    b0, nb, window = case.read()
    buf, n_bytes, table, paths = source.device_read(b0, nb, [(window[0], window[1], 0, source.shape[-1])], window)
    data = Guarded(buf[:n_bytes].tobytes())
    ws_bytes = zarr_workspace_bytes(lib, source, table)
    ws = np.full(ws_bytes + 4096, CANARY, np.uint8)
    win_h, w = window[1] - window[0], source.shape[-1]
    wp = w + 5
    dt = np.dtype(source.dtype).newbyteorder("=")
    slot = np.frombuffer(np.full((nb + 2) * (win_h + 2) * wp * dt.itemsize, POISON, np.uint8), dt)
    slot = slot.reshape(nb + 2, win_h + 2, wp)
    err = np.zeros(1, np.uint32)
    rc = zarr_decode(lib, source, data.addr, n_bytes, table, slot[1:, 1:].ctypes.data, wp, (win_h + 2) * wp, window,
                     b0, nb, ws.ctypes.data, ws_bytes, err.ctypes.data, None)
    assert rc == 0, lib.xrs_last_error()
    assert lib.xrsh_bad_launches() == 0, "a launch beyond CUDA's grid or block limits"
    inner = np.zeros(slot.shape, bool)
    inner[1:nb + 1, 1:win_h + 1, :w] = True
    poison = np.full(1, 0, dt)
    poison.view(np.uint8)[:] = POISON
    intact = bool(np.all(slot.view(np.uint8).reshape(slot.shape + (-1,))[~inner] == POISON)) and \
        bool(np.all(ws[ws_bytes:] == CANARY))
    return slot[1:nb + 1, 1:win_h + 1, :w], case.expected(source) if not case.error else None, int(err[0]), paths, intact


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.dtype(f"u{a.dtype.itemsize}"))


def test_case_table_is_complete():
    names = {c.name for c in CASES}
    for dt in ("float32", "float64", "uint8", "int8", "uint16", "int16", "int32", "uint32", "int64"):
        assert {f"{dt}_split", f"{dt}_dont_split", f"{dt}_no_shuffle", f"{dt}_lz4"} <= names
    assert sum(c.error != 0 for c in CASES) >= 9 and len({c.error for c in CASES if c.error}) == 7


@pytest.mark.parametrize("case", [c for c in CASES if not c.error], ids=lambda c: c.name)
def test_decode_equals_the_host_decode(lib, case, tmp_path):
    got, want, err, _, intact = run_case(lib, case, str(tmp_path))
    assert err == 0, decode_error(err, [])
    assert intact, "a byte outside the slot or the workspace changed"
    assert got.dtype == want.dtype
    assert np.array_equal(_bits(got), _bits(want)), case.name


@pytest.mark.parametrize("case", [c for c in CASES if c.error], ids=lambda c: c.name)
def test_malformed_chunks_are_reported(lib, case, tmp_path):
    _, _, err, paths, intact = run_case(lib, case, str(tmp_path))
    assert err >> 24 == case.error, decode_error(err, paths)
    assert (err & 0xFFFFFF) - 1 == 0
    assert paths[0] in decode_error(err, paths)
    assert intact, "a malformed chunk wrote outside its slot or the workspace"


def test_header_checks_name_the_chunk(lib, tmp_path):
    """A file the call can reject from its header alone fails the call, naming the chunk."""
    case = next(c for c in CASES if c.name == "float32_lz4")
    source = case.source(str(tmp_path))
    buf, n_bytes, table, paths = source.device_read(0, 1, [(0, 21, 0, 37)], (0, 21))
    table[1]["header"][:4] = np.frombuffer((5).to_bytes(4, "little"), np.uint8)
    assert lib.xrs_zarr_decode_workspace_bytes(table.ctypes.data, len(table), 1, 8, 16, 0) == -1
    assert b"chunk 1" in lib.xrs_last_error()


def test_host_checks_raise_the_host_paths_errors(tmp_path):
    """Bit-shuffled and BloscLZ frames raise the errors of ``blosc_decompress``."""
    from xcube_resampling_b200.io import ZarrV2Source

    from .test_host_io import _blosc_frame

    case = next(c for c in CASES if c.name == "float32_split")
    path = case.write(str(tmp_path))
    raw = np.zeros(2 * 8 * 17, np.float32).tobytes()
    frame = bytearray(_blosc_frame(raw, 4, 512, True, "lz4"))
    frame[2] |= 0x4
    open(f"{path}/0.0.0", "wb").write(bytes(frame))
    with pytest.raises(NotImplementedError, match="bit-shuffled"):
        ZarrV2Source(path).device_read(0, 1, [(0, 8, 0, 17)], (0, 8))
    frame[2] = frame[2] & 0x1F & ~0x4
    open(f"{path}/0.0.0", "wb").write(bytes(frame))
    with pytest.raises(NotImplementedError, match="BloscLZ"):
        ZarrV2Source(path).device_read(0, 1, [(0, 8, 0, 17)], (0, 8))
