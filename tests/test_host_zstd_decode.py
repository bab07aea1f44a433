"""The device decode of Zstd-compressed Zarr chunks as kernels on the host: csrc/decode.cu (k_zstd_decode and the
launch code around it) compiled for the CPU (tests/hostmath/zstd_decode.py), run over the case table of
tests/zstd_decode_cases.py.

Every slot equals the host decode bit for bit, the poison around it and the canary after the workspace stay intact,
and nothing is read past the end of a file (it ends at a page that may not be read).  Every malformed case is reported
with its reason and chunk, and the host path rejects the same file.  The corpus is shown to exercise every block type,
literals type and sequence-table mode (read from the frame headers) and every repeat-offset rule (counted by the
kernel's test hook)."""

import ctypes

import numpy as np
import pytest

from xcube_resampling_b200._pipeline import decode_error

from . import zstd_decode_cases as zc
from .test_host_zarr_decode import _bits, run_case

CASES = zc.cases()


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    from .hostmath.zstd_decode import build_zstd_decode

    try:
        so = build_zstd_decode(str(tmp_path_factory.mktemp("zstddecodehost")))
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
    lib.xrsh_zstd_events_take.restype, lib.xrsh_zstd_events_take.argtypes = None, [ctypes.c_void_p]
    return lib


def test_case_table_is_complete():
    names = {c.name for c in CASES}
    for dt in ("float32", "float64", "uint8", "int8", "uint16", "int16", "int32", "uint32", "int64"):
        assert {f"{dt}_zstd_split", f"{dt}_zstd_dont_split", f"{dt}_zstd_no_shuffle", f"{dt}_zstd"} <= names
    reasons = {c.error for c in CASES if c.error}
    assert set(range(2, 16)) <= reasons, sorted(set(range(2, 16)) - reasons)


def test_libzstd_cases_present():
    if zc.libzstd() is None:
        pytest.skip(zc.LIBZSTD_MISSING)
    assert sum(c.name.startswith(("libzstd", "blosc_libzstd")) for c in CASES) == 5


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


def _frames(case, root):
    """The zstd frames of a case's chunk files (each Blosc stream that is not stored)."""
    import os

    path = case.write(root)
    out = []
    for key in sorted(os.listdir(path)):
        if key.startswith("."):
            continue
        data = open(os.path.join(path, key), "rb").read()
        if case.compressor["id"] == "zstd":
            out.append(data)
            continue
        nbytes, blocksize = (int.from_bytes(data[k:k + 4], "little") for k in (4, 8))
        nblocks = -(-nbytes // blocksize)
        starts = [int.from_bytes(data[16 + 4 * b:20 + 4 * b], "little") for b in range(nblocks)]
        for b, pos in enumerate(starts):
            end = starts[b + 1] if b + 1 < nblocks else len(data)
            while pos < end:
                n = int.from_bytes(data[pos:pos + 4], "little")
                if data[pos + 4:pos + 8] == zc.MAGIC:
                    out.append(data[pos + 4:pos + 4 + n])
                pos += 4 + n
    return out


def test_corpus_exercises_every_block_literals_and_table_mode(tmp_path):
    blocks = [b for c in CASES if not c.error for f in _frames(c, str(tmp_path)) for b in zc.walk(f)]
    assert {b["type"] for b in blocks} == {0, 1, 2}
    lits = {(b["literals"], b.get("streams")) for b in blocks if b["type"] == 2}
    assert {(0, None), (1, None), (2, 1), (2, 4), (3, 1), (3, 4)} <= lits, lits
    for k, name in enumerate(("literal lengths", "offsets", "match lengths")):
        assert {b["modes"][k] for b in blocks if "modes" in b} == {0, 1, 2, 3}, name


def test_every_repeat_offset_rule_occurs(lib, tmp_path):
    """Repeat offsets 1 / 2 / 3 after literals (events 0-2) and, after none, Repeat_Offset2 / 3 / Repeat_Offset1 - 1
    (events 4-6): all of them in the hand-assembled frame, all but the last in a level-19 libzstd frame."""
    events = (ctypes.c_long * 8)()
    for name, want in (("hand_repeat_offsets", (0, 1, 2, 4, 5, 6)), ("level_19_multi_block", (0, 1, 2, 4, 5))):
        lib.xrsh_zstd_events_take(events)
        _, _, err, _, _ = run_case(lib, next(c for c in CASES if c.name == name), str(tmp_path / name))
        assert err == 0
        lib.xrsh_zstd_events_take(events)
        assert all(events[k] > 0 for k in want), (name, list(events))


def test_header_checks_raise_the_host_paths_errors(tmp_path):
    """A numcodecs zstd file that is not a frame, has no content size or the wrong one fails the device read with the
    host path's errors; a Blosc frame of another inner codec than the store's cname too."""
    from xcube_resampling_b200.io import ZarrV2Source, chunk_decoder

    case = next(c for c in CASES if c.name == "float32_zstd")
    path = case.write(str(tmp_path))
    raw = np.zeros(8 * 16, np.float32).tobytes()
    for data, err, match in ((b"\x00" * 20, ValueError, "not a zstd frame"),
                             (zc.frame([zc.block(0, raw, True)], None, window=0x20), NotImplementedError,
                              "without a content size"),
                             (zc.frame([zc.block(0, raw[:-4], True)], len(raw) - 4, 2), ValueError, "holds 508")):
        open(f"{path}/0.0", "wb").write(data)
        with pytest.raises(err, match=match):
            ZarrV2Source(path).device_read(0, 1, [(0, 8, 0, 16)], (0, 8))
        with pytest.raises(Exception):
            np.frombuffer(chunk_decoder(case.compressor)(data), np.float32).reshape(8, 16)
    case = next(c for c in CASES if c.name == "float32_zstd_split")
    path = case.write(str(tmp_path))
    from .test_host_io import _blosc_frame

    open(f"{path}/0.0.0", "wb").write(_blosc_frame(np.zeros(2 * 8 * 17, np.float32).tobytes(), 4, 512, True, "lz4"))
    with pytest.raises(ValueError, match="not the store's Zstd"):
        ZarrV2Source(path).device_read(0, 1, [(0, 8, 0, 17)], (0, 8))
