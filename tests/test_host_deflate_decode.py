"""The device decode of Deflate-compressed Zarr chunks as kernels on the host: csrc/decode.cu (k_inflate and the launch
code around it) compiled for the CPU (tests/hostmath/deflate_decode.py), run over the case table of
tests/deflate_decode_cases.py.

Every slot equals the host decode bit for bit, the poison around it and the canary after the workspace stay intact,
and nothing is read past the end of a file (it ends at a page that may not be read).  Every malformed case is reported
with its reason and chunk, and the host path rejects the same file.  The kernel's test hook shows that the corpus
reaches every block type, every length and distance code at both ends of its extra bits, every repeat code and both
wrappers."""

import ctypes

import numpy as np
import pytest

from xcube_resampling_b200._pipeline import decode_error

from . import deflate_decode_cases as dc
from .test_host_zarr_decode import _bits, run_case

CASES = dc.cases()


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    from .hostmath.deflate_decode import build_deflate_decode

    try:
        so = build_deflate_decode(str(tmp_path_factory.mktemp("deflatedecodehost")))
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
    lib.xrsh_deflate_events_take.restype, lib.xrsh_deflate_events_take.argtypes = None, [ctypes.c_void_p]
    return lib


def test_case_table_is_complete():
    names = {c.name for c in CASES}
    for dt in ("float32", "float64", "uint8", "int8", "uint16", "int16", "int32", "uint32", "int64"):
        assert {f"{dt}_zlib_split", f"{dt}_zlib_dont_split", f"{dt}_zlib_no_shuffle", f"{dt}_zlib",
                f"{dt}_gzip"} <= names
    reasons = {c.error for c in CASES if c.error}
    assert {dc.OFFSET_BEFORE_START, dc.LITERALS_OVERRUN, dc.MATCH_OVERRUN, dc.INPUT_OVERRUN, dc.SHORT,
            dc.BAD_FRAME_HEADER, dc.TRAILING_BYTES, dc.CHECKSUM, dc.BAD_BLOCK, dc.BAD_CODES,
            dc.BAD_SYMBOL} == reasons


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
    source = case.source(str(tmp_path / "host"))
    out = np.empty((1,) + tuple(source.shape[-2:]), np.dtype(source.dtype).newbyteorder("="))
    with pytest.raises(Exception):
        source.read_bands(0, 1, out)


def test_corpus_reaches_every_block_type_code_and_wrapper(lib, tmp_path):
    events = (ctypes.c_long * 128)()
    total = np.zeros(128, np.int64)
    lib.xrsh_deflate_events_take(events)
    for case in CASES:
        if not case.error:
            _, _, err, _, _ = run_case(lib, case, str(tmp_path / case.name))
            assert err == 0
            lib.xrsh_deflate_events_take(events)
            total += np.ctypeslib.as_array(events)
    names = ["stored", "fixed", "dynamic"] + [f"length code {257 + c} {e}" for c in range(29) for e in ("low", "high")]
    names += [f"distance code {c} {e}" for c in range(30) for e in ("low", "high")]
    names += ["repeat 16", "repeat 17", "repeat 18", "zlib", "gzip", "length 258 from code 284", "no distance codes"]
    missing = [name for name, n in zip(names, total) if n == 0]
    assert not missing, missing


def test_header_checks_raise_the_host_paths_errors(tmp_path):
    """zlib files with a bad header, FDICT or too short, gzip files that are not gzip, of another method or too
    short, and Blosc frames of another inner codec than the store's cname fail the device read with the errors the
    host path raises for them."""
    import gzip
    import zlib

    from xcube_resampling_b200.io import ZarrV2Source, chunk_decoder

    case = next(c for c in CASES if c.name == "float32_zlib")
    path = case.write(str(tmp_path / "z"))
    fdict = bytes([0x78, 0x20 + (31 - (0x7820 % 31)) % 31])
    for data in (b"\x78\x02" + bytes(20), fdict + bytes(20), b"\x78\x01\x03", b"\x79\x01" + bytes(20)):
        open(f"{path}/0.0", "wb").write(data)
        with pytest.raises(zlib.error):
            ZarrV2Source(path).device_read(0, 1, [(0, 8, 0, 16)], (0, 8))
        with pytest.raises(zlib.error):
            chunk_decoder(case.compressor)(data)
    case = next(c for c in CASES if c.name == "float32_gzip")
    path = case.write(str(tmp_path / "g"))
    for data, err in ((b"\x1f\x8c" + bytes(30), gzip.BadGzipFile), (b"\x1f\x8b\x07" + bytes(30), gzip.BadGzipFile),
                      (b"\x1f\x8b\x08" + bytes(12), zlib.error), (b"\x1f\x8b\x08" + bytes(3), EOFError)):
        open(f"{path}/0.0", "wb").write(data)
        with pytest.raises(err):
            ZarrV2Source(path).device_read(0, 1, [(0, 8, 0, 16)], (0, 8))
        with pytest.raises(err):
            chunk_decoder(case.compressor)(data)
    case = next(c for c in CASES if c.name == "float32_zlib_split")
    path = case.write(str(tmp_path / "b"))
    from .test_host_io import _blosc_frame

    open(f"{path}/0.0.0", "wb").write(_blosc_frame(np.zeros(2 * 8 * 17, np.float32).tobytes(), 4, 512, True, "zstd"))
    with pytest.raises(ValueError, match="not the store's Zlib"):
        ZarrV2Source(path).device_read(0, 1, [(0, 8, 0, 17)], (0, 8))


def test_a_store_of_each_codec_reads_for_the_device(tmp_path):
    from xcube_resampling_b200.io import CHUNK_BLOSC, CHUNK_GZIP, CHUNK_ZLIB, ZarrV2Source

    for name, codec in (("float32_zlib", CHUNK_ZLIB), ("float32_gzip", CHUNK_GZIP), ("float32_zlib_split", CHUNK_BLOSC)):
        src = ZarrV2Source(next(c for c in CASES if c.name == name).write(str(tmp_path)))
        assert src.device_decodable and src.device_codec == codec
