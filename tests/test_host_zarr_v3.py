"""Zarr v3 stores on the host: ``io.crc32c``, ``ZarrV3Source`` over the hand-written stores of tests/zarr_v3_cases.py
(every codec chain, sharding, fill values, key encodings), ``open_zarr_dataset`` on v3 groups, ``add_spatial_ref`` on
them, the rejections, and the device decode of the case table -- CRC-32C check included -- as kernels on the host
(csrc/decode.cu with decode_crc32c.cuh, tests/hostmath/crc32c_decode.py)."""

import ctypes
import json
import os

import numpy as np
import pytest

from xcube_resampling_b200.io import ZarrV2Source, ZarrV3Source, crc32c, open_zarr_dataset, write_zarr_array

from . import zarr_v3_cases as v3
from .test_host_zarr_decode import _bits, run_case

CASES = v3.cases()
GOOD = [c for c in CASES if not c.error]
BAD = [c for c in CASES if c.error]


def _bitwise_crc32c(data: bytes) -> int:
    c = 0xFFFFFFFF
    for b in data:
        c ^= b
        for _ in range(8):
            c = (c >> 1) ^ 0x82F63B78 if c & 1 else c >> 1
    return c ^ 0xFFFFFFFF


@pytest.fixture(scope="module")
def sse42(tmp_path_factory):
    fn = v3.sse42_crc32c(str(tmp_path_factory.mktemp("sse42")))
    if fn is None:
        pytest.skip("needs gcc and an x86 CPU with SSE4.2")
    return fn


KNOWN = v3.KNOWN


@pytest.mark.parametrize("data,want", KNOWN, ids=["check", "zeros", "ones", "incrementing", "decrementing"])
def test_crc32c_known_answers(data, want, sse42):
    assert crc32c(data) == want
    assert _bitwise_crc32c(data) == want and sse42(data) == want


def test_crc32c_random_lengths_and_alignments(sse42):
    rng = np.random.default_rng(5)
    blob = rng.integers(0, 256, (1 << 20) + 200, dtype=np.uint8).tobytes()
    lengths = [0, 1, 2, 3, 4, 5, 7, 8, 31, 32, 33, 63, 64, 65, 127, 128, 129, 191, 192, 193, 4095, 4096, 4097,
               64 * 3 + 63, 64 * 1000 + 1] + rng.integers(0, 1 << 20, 12).tolist() + [1 << 20]
    for k, n in enumerate(lengths):
        off = k % 13  # odd alignments of the view
        view = memoryview(blob)[off:off + n]
        assert crc32c(view) == sse42(view), n
        if n <= 5000:
            assert crc32c(view) == _bitwise_crc32c(view), n


def _expected_array(case) -> np.ndarray:
    """The case's array with its missing chunks (or inner chunks, or whole shards) at the fill value."""
    a = np.array(case.array)
    unit = case.shard["chunk_shape"] if case.shard else case.chunks
    value = v3.spelled_fill(case.fill_value, a.dtype)[0]
    for m in case.missing:
        if m[0] == "shard":
            sl = tuple(slice(s * c, (s + 1) * c) for s, c in zip(m[1:], case.chunks))
        else:
            sl = tuple(slice(i * u, (i + 1) * u) for i, u in zip(m, unit))
        a[sl] = value
    return a


@pytest.mark.parametrize("case", GOOD, ids=lambda c: c.name)
def test_v3_store_equals_the_array_and_the_v2_store(case, tmp_path):
    src = ZarrV3Source(case.write(str(tmp_path)))
    want = _expected_array(case)
    assert src.dtype == case.array.dtype and src.shape == case.array.shape
    got = src.read_all()
    assert np.array_equal(_bits(got), _bits(want)), case.name
    nb = min(2, case.array.shape[0] - 1)
    out = np.empty((nb,) + case.array.shape[1:], dtype=src.dtype)
    src.read_bands(1, nb, out)
    assert np.array_equal(_bits(out), _bits(want[1:1 + nb]))
    if isinstance(case.fill_value, str) and case.fill_value.startswith("0x"):
        return  # v2 has no spelling for a float's raw bits
    unit = case.shard["chunk_shape"] if case.shard else case.chunks
    p2 = str(tmp_path / "v2")
    write_zarr_array(p2, want, unit, ("band", "y", "x"))
    meta = json.load(open(os.path.join(p2, ".zarray")))
    meta["fill_value"] = case.fill_value
    json.dump(meta, open(os.path.join(p2, ".zarray"), "w"))
    assert np.array_equal(_bits(ZarrV2Source(p2).read_all()), _bits(got))


def test_fill_value_spellings(tmp_path):
    a = np.zeros((4, 4), np.float32)
    for fill, want in [("NaN", np.float32(np.nan)), ("Infinity", np.float32(np.inf)),
                       ("-Infinity", np.float32(-np.inf)), (2.5, np.float32(2.5)), (-3, np.float32(-3)),
                       ("0x7fc00001", np.array([0x7FC00001], np.uint32).view(np.float32)[0]),
                       ("0xff800000", np.float32(-np.inf))]:
        p = str(tmp_path / str(fill))
        v3.write_v3_array(p, a, (2, 2), ("y", "x"), fill_value=fill, missing=((1, 1),))
        got = ZarrV3Source(p).read_all()
        assert _bits(got[2:, 2:]).tolist() == [[_bits(np.array([want]))[0]] * 2] * 2, fill
        assert np.all(got[:2, :] == 0)
    p = str(tmp_path / "i64")
    v3.write_v3_array(p, np.zeros((2, 2), np.int64), (1, 2), ("y", "x"), fill_value=-2 ** 63, missing=((1, 0),))
    assert ZarrV3Source(p).read_all()[1].tolist() == [-2 ** 63] * 2


def test_shard_index_is_read_once_per_shard(tmp_path):
    case = next(c for c in CASES if c.name == "shard_end_crc")
    src = ZarrV3Source(case.write(str(tmp_path)))

    class Counting(dict):
        sets = 0

        def __setitem__(self, k, v):
            Counting.sets += 1
            super().__setitem__(k, v)

    src._indexes = Counting()
    out = np.empty((1,) + case.array.shape[1:], np.float32)
    for b in range(3):
        src.read_bands(b, 1, out)
    assert Counting.sets == len(src._indexes) == 8  # 2 x 2 x 2 shards, one a missing file


def test_device_read_reads_only_the_inner_chunks(tmp_path):
    """Ranged reads: the bytes of the inner chunks that intersect the segments, never a whole shard."""
    case = next(c for c in CASES if c.name == "shard_end_crc")
    src = ZarrV3Source(case.write(str(tmp_path)))
    segments, window = [(9, 15, 20, 30)], (8, 16)
    buf, n_bytes, table, paths = src.device_read(0, 2, segments, window)
    # bands 0-1, inner row 1, inner columns 1 (pixels 17-33): inner chunks (0, 1, 1) [missing] and (1, 1, 1)
    assert len(table) == 2 and table[0]["codec"] == 0
    p = os.path.join(src.path, "c", "0", "0", "0")
    index = v3.shard_index(p, 8, start=False, crc=True)
    k = int(np.ravel_multi_index((1, 1, 1), (2, 2, 2)))  # its place in the shard's inner grid
    assert n_bytes == int(index[k, 1]) < os.path.getsize(p)
    raw = open(p, "rb").read()
    assert buf[:n_bytes].tobytes() == raw[int(index[k, 0]):int(index[k, 0]) + n_bytes]
    assert table[1]["codec"] == 3 | 0x100 and table[1]["length"] == n_bytes
    assert "inner chunk (1, 1, 1)" in paths[1] and paths[1].startswith(p)


def _write(tmp_path, name, **kw):
    p = str(tmp_path / name)
    args = dict(array=np.arange(2 * 6 * 8, dtype=np.float32).reshape(2, 6, 8), chunks=(1, 6, 8),
                dims=("band", "y", "x"))
    args.update(kw)
    v3.write_v3_array(p, **args)
    return p


def _edit(path, fn):
    meta = json.load(open(os.path.join(path, "zarr.json")))
    fn(meta)
    json.dump(meta, open(os.path.join(path, "zarr.json"), "w"))


def test_rejections_name_the_file(tmp_path):
    shard = {"chunk_shape": (1, 3, 4), "index_crc": True}
    p = _write(tmp_path, "short_index", codecs=("bytes", "zstd"), shard=shard)
    f = os.path.join(p, "c", "0", "0", "0")
    open(f, "wb").write(open(f, "rb").read()[-20:])
    with pytest.raises(ValueError, match=f"{f}.*index"):
        ZarrV3Source(p).read_all()
    p = _write(tmp_path, "index_crc", codecs=("bytes", "zstd"), shard=shard)
    f = os.path.join(p, "c", "1", "0", "0")
    raw = bytearray(open(f, "rb").read())
    raw[-10] ^= 1
    open(f, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match=f"{f}: shard index: CRC-32C mismatch"):
        ZarrV3Source(p).read_all()
    p = _write(tmp_path, "outside", codecs=("bytes", "zstd"), shard={"chunk_shape": (1, 3, 4), "index_crc": False})
    f = os.path.join(p, "c", "0", "0", "0")
    raw = bytearray(open(f, "rb").read())
    raw[-16 * 4 + 8:-16 * 4 + 16] = (len(raw) + 1).to_bytes(8, "little")  # nbytes of inner chunk 0
    open(f, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match=f"{f}: a shard index entry points outside the file"):
        ZarrV3Source(p).read_all()
    p = _write(tmp_path, "chunk_crc", codecs=("bytes", "gzip", "crc32c"), shard=shard)
    f = os.path.join(p, "c", "0", "0", "0")
    raw = bytearray(open(f, "rb").read())
    raw[30] ^= 1
    open(f, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match=r"c/0/0/0 \(inner chunk \(0, 0, 0\)\): CRC-32C mismatch"):
        ZarrV3Source(p).read_all()
    p = _write(tmp_path, "plain_crc", codecs=("bytes", "crc32c"))
    f = os.path.join(p, "c", "1", "0", "0")
    raw = bytearray(open(f, "rb").read())
    raw[0] ^= 1
    open(f, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match=f"{f}: CRC-32C mismatch"):
        ZarrV3Source(p).read_all()


@pytest.mark.parametrize("edit,error,match", [
    (lambda m: m.update(chunk_grid={"name": "rectilinear", "configuration": {}}), NotImplementedError, "rectilinear"),
    (lambda m: m.update(data_type="string"), NotImplementedError, "'string'"),
    (lambda m: m.update(data_type="r16"), NotImplementedError, "'r16'"),
    (lambda m: m.update(storage_transformers=[{"name": "x"}]), NotImplementedError, "storage transformers"),
    (lambda m: m.update(codecs=[{"name": "transpose", "configuration": {"order": [0, 2, 1]}}, "bytes"]),
     NotImplementedError, "transpose"),
    (lambda m: m.update(codecs=[{"name": "bytes", "configuration": {"endian": "little"}},
                                {"name": "blosc", "configuration": {"cname": "lz4", "shuffle": "bitshuffle"}}]),
     NotImplementedError, "bit-shuffled"),
    (lambda m: m.update(codecs=[{"name": "bytes", "configuration": {"endian": "little"}}, {"name": "bitshuffle"}]),
     NotImplementedError, "bit-shuffled"),
    (lambda m: m.update(codecs=[{"name": "bytes", "configuration": {"endian": "little"}}, {"name": "jpeg"}]),
     NotImplementedError, "'jpeg'"),
    (lambda m: m.update(codecs=[{"name": "bytes"}]), ValueError, "endian"),
    (lambda m: m.update(codecs=[{"name": "bytes", "configuration": {"endian": "little"}}, "zstd", "gzip"]),
     NotImplementedError, "gzip"),
    (lambda m: m.update(codecs=[{"name": "sharding_indexed", "configuration": {
        "chunk_shape": [1, 3, 4], "codecs": [{"name": "sharding_indexed", "configuration": {}}],
        "index_codecs": [{"name": "bytes", "configuration": {"endian": "little"}}]}}]),
     NotImplementedError, "nested"),
    (lambda m: m.update(chunk_key_encoding={"name": "custom"}), NotImplementedError, "custom"),
])
def test_unsupported_metadata_raises(tmp_path, edit, error, match):
    p = _write(tmp_path, "a", codecs=("bytes", "zstd"))
    _edit(p, edit)
    with pytest.raises(error, match=match) as e:
        ZarrV3Source(p).read_all()
    assert p in str(e.value) or error is ValueError


def test_host_checks_see_the_payload(tmp_path):
    """The device read checks each header on the payload, the CRC-32C trailer excluded, with the host path's errors."""
    p = _write(tmp_path, "a", codecs=("bytes", "zstd", "crc32c"))
    f = os.path.join(p, "c", "0", "0", "0")
    raw = bytearray(open(f, "rb").read())
    raw[0] ^= 1  # not a zstd frame
    open(f, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match="not a zstd frame"):
        ZarrV3Source(p).device_read(0, 1, [(0, 6, 0, 8)], (0, 6))
    src = ZarrV3Source(_write(tmp_path, "b", codecs=("bytes", "zstd", "crc32c")))
    buf, n, table, _ = src.device_read(0, 2, [(0, 6, 0, 8)], (0, 6))
    assert bytes(table[0]["header"][:4]) == b"\x28\xb5\x2f\xfd" and table[0]["codec"] == 3 | 0x100
    assert not ZarrV3Source(_write(tmp_path, "c", codecs=("bytes", "crc32c"))).device_decodable


def test_dimension_names_and_fallbacks(tmp_path):
    root = str(tmp_path / "s.zarr")
    v3.write_v3_group(root, {"title": "t"})
    a = np.ones((3, 4), np.float32)
    v3.write_v3_array(os.path.join(root, "named"), a, (3, 4), ("lat", "lon"))
    v3.write_v3_array(os.path.join(root, "attr"), a, (3, 4), None, attributes={"_ARRAY_DIMENSIONS": ["y", "x"],
                                                                               "units": "m"})
    v3.write_v3_array(os.path.join(root, "none"), a, (3, 4), None, dimension_names=False)
    v3.write_v3_array(os.path.join(root, "partial"), a, (3, 4), (None, "x"))
    ds = open_zarr_dataset(root)
    assert ds.attrs == {"title": "t"}
    assert ds["named"].dims == ("lat", "lon") and ds["attr"].dims == ("y", "x")
    assert ds["attr"].attrs == {"units": "m"}
    assert ds["none"].dims == ("dim_0", "dim_1") and ds["partial"].dims == ("dim_0", "x")


def test_small_arrays_and_coordinates(tmp_path):
    root = str(tmp_path / "s.zarr")
    v3.write_v3_group(root)
    v3.write_v3_array(os.path.join(root, "scalar"), np.array(3.5, ">f8"), (), (), codecs=("bytes", "crc32c"))
    v3.write_v3_array(os.path.join(root, "scalar_v2key"), np.array(7, np.int16), (), (),
                      key_encoding={"name": "v2"})
    v3.write_v3_array(os.path.join(root, "missing"), np.array(0, np.float32), (), (), fill_value="NaN",
                      missing=((),))
    x = np.arange(50, dtype=np.float64) * 0.5
    v3.write_v3_array(os.path.join(root, "x"), x, (16,), ("x",), codecs=("bytes", "zstd"), missing=((2,),),
                      fill_value=-1)
    v3.write_v3_array(os.path.join(root, "y"), x[:37], (20,), ("y",), codecs=("bytes", "gzip", "crc32c"),
                      shard={"chunk_shape": (5,), "index_location": "start", "index_crc": True})
    ds = open_zarr_dataset(root)
    assert ds["scalar"].values == 3.5 and ds["scalar"].dims == ()
    assert ds["scalar_v2key"].values == 7 and np.isnan(ds["missing"].values)
    want = x.copy()
    want[32:48] = -1
    assert np.array_equal(ds["x"].values, want) and ds["x"].dims == ("x",)
    assert np.array_equal(ds["y"].values, x[:37])


def test_open_zarr_dataset_v3_mask_and_scale_and_grid_mapping(tmp_path):
    from xcube_resampling_b200 import GridMapping
    from xcube_resampling_b200.cfconv import add_spatial_ref
    from xcube_resampling_b200.crs import CRS
    from xcube_resampling_b200.io import DecodedSource, LazyDataArray

    root = str(tmp_path / "s.zarr")
    v3.write_v3_group(root, {"source": "test"})
    x = 10.0 + np.arange(40) * 0.01
    y = 50.0 - np.arange(30) * 0.01
    v3.write_v3_array(os.path.join(root, "lon"), x, (40,), ("lon",), codecs=("bytes", "zstd"))
    v3.write_v3_array(os.path.join(root, "lat"), y, (30,), ("lat",), codecs=("bytes", "zstd"))
    raw = np.random.default_rng(1).integers(0, 1000, (2, 30, 40)).astype(np.uint16)
    raw[0, 0, :5] = 65535
    v3.write_v3_array(os.path.join(root, "rad"), raw, (2, 16, 20), ("band", "lat", "lon"),
                      codecs=("bytes", "zstd", "crc32c"), shard={"chunk_shape": (1, 8, 10), "index_crc": True},
                      attributes={"scale_factor": 0.5, "add_offset": 1.0, "_FillValue": 65535})
    v3.write_v3_array(os.path.join(root, "other"), np.zeros((30, 2), np.uint8), (30, 2), ("lat", "k"))
    # consolidated metadata, as zarr-python writes it
    meta = json.load(open(os.path.join(root, "zarr.json")))
    meta["consolidated_metadata"] = {"kind": "inline", "must_understand": False, "metadata": {
        n: json.load(open(os.path.join(root, n, "zarr.json"))) for n in ("lon", "lat", "rad", "other")}}
    json.dump(meta, open(os.path.join(root, "zarr.json"), "w"))

    ds = open_zarr_dataset(root, mask_and_scale=True)
    assert isinstance(ds["rad"], LazyDataArray) and isinstance(ds["rad"].source, DecodedSource)
    want = raw.astype(np.float32)
    want[raw == 65535] = np.nan
    want = want * np.float32(0.5) + np.float32(1.0)
    assert np.array_equal(ds["rad"].values, want, equal_nan=True) and "scale_factor" not in ds["rad"].attrs
    assert ds.attrs == {"source": "test"}

    add_spatial_ref(root, CRS.from_string("EPSG:4326"), xy_dim_names=("lon", "lat"))
    sr = json.load(open(os.path.join(root, "spatial_ref", "zarr.json")))
    assert sr["zarr_format"] == 3 and sr["shape"] == [] and sr["data_type"] == "uint8"
    assert sr["codecs"] == [{"name": "bytes"}] and os.path.isfile(os.path.join(root, "spatial_ref", "c"))
    assert json.load(open(os.path.join(root, "rad", "zarr.json")))["attributes"]["grid_mapping"] == "spatial_ref"
    assert "grid_mapping" not in json.load(open(os.path.join(root, "other", "zarr.json")))["attributes"]
    consolidated = json.load(open(os.path.join(root, "zarr.json")))["consolidated_metadata"]["metadata"]
    assert set(consolidated) == {"lon", "lat", "rad", "other", "spatial_ref"}
    assert consolidated["rad"]["attributes"]["grid_mapping"] == "spatial_ref"
    ds = open_zarr_dataset(root)
    assert ds["spatial_ref"].values == 0 and ds["rad"].attrs["grid_mapping"] == "spatial_ref"
    gm = GridMapping.from_dataset(ds)
    assert gm.crs.is_geographic and gm.size == (40, 30)


def test_add_spatial_ref_uses_the_stores_key_encoding(tmp_path):
    from xcube_resampling_b200.cfconv import add_spatial_ref
    from xcube_resampling_b200.crs import CRS

    root = str(tmp_path / "s.zarr")
    v3.write_v3_group(root)
    v3.write_v3_array(os.path.join(root, "v"), np.zeros((3, 4), np.float32), (3, 4), ("y", "x"),
                      key_encoding={"name": "v2"})
    add_spatial_ref(root, CRS.from_string("EPSG:3035"))
    assert os.path.isfile(os.path.join(root, "spatial_ref", "0"))
    assert json.load(open(os.path.join(root, "spatial_ref", "zarr.json")))["chunk_key_encoding"]["name"] == "v2"
    assert open_zarr_dataset(root)["spatial_ref"].values == 0


# --- the device decode as kernels on the host --------------------------------------------------------------------


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    from .hostmath.crc32c_decode import build_crc32c_decode

    try:
        so = build_crc32c_decode(str(tmp_path_factory.mktemp("crc32chost")))
    except RuntimeError as e:
        if "g++ not available" in str(e):
            pytest.skip(str(e))
        raise
    from xcube_resampling_b200._lib import SIGNATURES

    lib = ctypes.CDLL(so)
    for name in ("xrs_zarr_decode", "xrs_zarr_decode_workspace_bytes", "xrs_last_error"):
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = SIGNATURES[name]
    lib.xrsh_bad_launches.restype, lib.xrsh_bad_launches.argtypes = ctypes.c_long, []
    lib.xrsh_take_log.restype = ctypes.c_long
    return lib


def _kernels(lib) -> list:
    names, err = ctypes.create_string_buffer(4096), ctypes.create_string_buffer(4096)
    lib.xrsh_take_log(names, 4096, err, 4096)
    return names.value.decode().split(";")


@pytest.mark.parametrize("case", GOOD, ids=lambda c: c.name)
def test_host_build_decodes_the_case_table(lib, case, tmp_path):
    source = case.source(str(tmp_path))
    if not getattr(source, "device_decodable", False):
        pytest.skip("decoded on the host path")
    _kernels(lib)
    got, want, err, _, intact = run_case(lib, case, str(tmp_path / "run"))
    assert err == 0 and intact, case.name
    assert np.array_equal(_bits(got), _bits(want)), case.name
    ran = _kernels(lib)
    assert ("zarr_crc32c" in ran) == ("crc32c" in str(case.codecs)), ran


@pytest.mark.parametrize("case", BAD, ids=lambda c: c.name)
def test_host_build_reports_a_crc_mismatch(lib, case, tmp_path):
    _, _, err, paths, intact = run_case(lib, case, str(tmp_path))
    assert err >> 24 == v3.CRC32C_MISMATCH and (err & 0xFFFFFF) - 1 == 0 and intact
    from xcube_resampling_b200._pipeline import decode_error

    assert "CRC-32C" in decode_error(err, paths) and paths[0] in decode_error(err, paths)


@pytest.mark.parametrize("where", ["payload", "trailer"])
def test_host_build_names_the_right_chunk(lib, tmp_path, where):
    """A flipped byte in file k of the table (of its payload, or of its trailer) is reported for chunk k."""
    from xcube_resampling_b200._pipeline import zarr_decode, zarr_workspace_bytes

    from .test_host_zarr_decode import Guarded

    case = next(c for c in CASES if c.name == "shard_end_crc")
    source = ZarrV3Source(case.write(str(tmp_path)))
    buf, n_bytes, table, paths = source.device_read(0, 3, [(0, 21, 0, 37)], (0, 21))
    present = [k for k in range(len(table)) if table[k]["codec"]]
    k = present[len(present) // 2]
    data = bytearray(buf[:n_bytes].tobytes())
    t = table[k]
    data[int(t["offset"]) + (int(t["length"]) - 2 if where == "trailer" else 40)] ^= 0x01
    g = Guarded(bytes(data))
    ws_bytes = zarr_workspace_bytes(lib, source, table)
    ws = np.zeros(ws_bytes, np.uint8)
    slot = np.zeros((3, 21, 40), np.float32)
    err = np.zeros(1, np.uint32)
    rc = zarr_decode(lib, source, g.addr, n_bytes, table, slot.ctypes.data, 40, 21 * 40, (0, 21), 0, 3,
                     ws.ctypes.data, ws_bytes, err.ctypes.data, None)
    assert rc == 0, lib.xrs_last_error()
    assert err[0] >> 24 == v3.CRC32C_MISMATCH and (int(err[0]) & 0xFFFFFF) - 1 == k


def test_base_host_build_refuses_flagged_chunks(tmp_path):
    """Without the CRC-32C check compiled in, a flagged table fails the call instead of skipping the check."""
    from xcube_resampling_b200._lib import SIGNATURES

    from .hostmath.zarr_decode import build_decode

    try:
        so = build_decode(str(tmp_path))
    except RuntimeError as e:
        pytest.skip(str(e))
    lib = ctypes.CDLL(so)
    for name in ("xrs_zarr_decode", "xrs_zarr_decode_workspace_bytes", "xrs_last_error"):
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = SIGNATURES[name]
    case = next(c for c in CASES if c.name == "v3_blosc_lz4_crc32c")
    source = case.source(str(tmp_path))
    buf, n_bytes, table, _ = source.device_read(0, 1, [(0, 21, 0, 37)], (0, 21))
    ws_bytes = lib.xrs_zarr_decode_workspace_bytes(table.ctypes.data, len(table), 2, 8, 17, 0)
    assert ws_bytes > 0
    ws = np.zeros(ws_bytes, np.uint8)
    slot = np.zeros((1, 21, 37), np.float32)
    err = np.zeros(1, np.uint32)
    from xcube_resampling_b200._pipeline import zarr_decode

    rc = zarr_decode(lib, source, buf.ctypes.data, n_bytes, table, slot.ctypes.data, 37, 21 * 37, (0, 21), 0, 1,
                     ws.ctypes.data, ws_bytes, err.ctypes.data, None)
    assert rc != 0 and b"no CRC-32C check" in lib.xrs_last_error()


def test_flag_on_a_missing_or_short_file_fails_the_call(lib, tmp_path):
    case = next(c for c in CASES if c.name == "v3_zstd_crc32c")
    source = case.source(str(tmp_path))
    _, _, table, _ = source.device_read(0, 2, [(0, 21, 0, 37)], (0, 21))
    t = table.copy()
    t[0]["length"] = 3
    assert lib.xrs_zarr_decode_workspace_bytes(t.ctypes.data, len(t), 2, 8, 17, 0) == -1
    assert b"chunk 0" in lib.xrs_last_error() and b"CRC-32C" in lib.xrs_last_error()
    t = table.copy()
    t[1]["codec"] = 0x100
    assert lib.xrs_zarr_decode_workspace_bytes(t.ctypes.data, len(t), 2, 8, 17, 0) == -1


def _flagged_files(payloads, trailers):
    """The payloads, each followed by its 4-byte trailer, at odd offsets of one buffer (1 ... 7 bytes apart), and a
    chunk table flagging every one of them XRS_CHUNK_CRC32C."""
    from xcube_resampling_b200.io import CHUNK_CRC32C, CHUNK_LZ4, CHUNK_TABLE_DTYPE

    data, table = bytearray(), np.zeros(len(payloads), CHUNK_TABLE_DTYPE)
    for k, (p, t) in enumerate(zip(payloads, trailers)):
        data += bytes(k % 7 + 1)
        table[k]["offset"], table[k]["length"] = len(data), len(p) + 4
        table[k]["codec"] = CHUNK_LZ4 | CHUNK_CRC32C
        data += p + t.to_bytes(4, "little")
    return bytes(data), table


def _sweep_payloads():
    rng = np.random.default_rng(9)
    return [v for v, _ in v3.KNOWN] + [rng.integers(0, 256, n, dtype=np.uint8).tobytes()
                                       for n in v3.crc_sweep_lengths()]


def _host_crc32c(lib, data, table):
    from .test_host_zarr_decode import Guarded

    g = Guarded(data)  # the last trailer ends at a page that may not be read
    err = np.zeros(1, np.uint32)
    fn = lib.xrsh_crc32c
    fn.restype, fn.argtypes = ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_void_p]
    assert fn(g.addr, table.ctypes.data, len(table), err.ctypes.data) == 0
    assert lib.xrsh_bad_launches() == 0
    return int(err[0])


def test_host_build_k_crc32c_known_answers_and_sweep(lib, sse42):
    """k_crc32c itself on the known answers and on payloads of 0 ... 64 bytes, multiples of 32 and one either side,
    and random lengths up to 1 MiB at odd offsets, against the SSE4.2 instruction; a flipped bit in the payload or the
    trailer of any one file is reported for that file."""
    payloads = _sweep_payloads()
    for v, want in v3.KNOWN:
        assert sse42(v) == want
    trailers = [sse42(p) for p in payloads]
    data, table = _flagged_files(payloads, trailers)
    t = table.copy()
    assert _host_crc32c(lib, data, t) == 0
    assert np.all(t["codec"] == 2) and np.array_equal(t["length"], table["length"] - 4)  # flag and trailer dropped
    wrong = [trailers[k] ^ (1 << (k % 32)) for k in range(len(trailers))]  # every file alone with a wrong trailer
    for k in range(len(payloads)):
        d, tab = _flagged_files(payloads, trailers[:k] + [wrong[k]] + trailers[k + 1:])
        word = _host_crc32c(lib, d, tab)
        assert word >> 24 == v3.CRC32C_MISMATCH and (word & 0xFFFFFF) - 1 == k, (k, len(payloads[k]))
    for k in [k for k, p in enumerate(payloads) if len(p)][::7]:  # a flipped payload bit
        d = bytearray(data)
        d[int(table[k]["offset"]) + (len(payloads[k]) * 5) // 7] ^= 0x08
        word = _host_crc32c(lib, bytes(d), table.copy())
        assert word >> 24 == v3.CRC32C_MISMATCH and (word & 0xFFFFFF) - 1 == k, (k, len(payloads[k]))


def test_an_unknown_fill_value_names_the_array(tmp_path):
    p = _write(tmp_path, "a", codecs=("bytes", "zstd"))
    _edit(p, lambda m: m.update(fill_value="Nonsense"))
    with pytest.raises(ValueError, match=f"{p}: unknown fill_value 'Nonsense'"):
        ZarrV3Source(p)
