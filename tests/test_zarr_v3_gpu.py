"""Zarr v3 stores decoded on the device: the case table of tests/zarr_v3_cases.py bit for bit against the host decode,
CRC-32C mismatches reported by ``k_crc32c``, and the band pipeline fed from a sharded zstd + crc32c store and from a
Blosc-LZ4 store giving exactly what the same arrays give as a v2 store and in memory."""

import os
import zlib

import numpy as np
import pytest

from . import zarr_v3_cases as v3
from .helpers import assert_same, covering_grid_args, swath
from .test_host_io import _blosc_frame, _compress_store
from .test_zarr_decode_gpu import _bits, _device_decode, xrs  # noqa: F401  (xrs: the module fixture)

pytestmark = pytest.mark.gpu
CASES = v3.cases()
SHARDED_ZSTD = (("bytes", "zstd", "crc32c"), {"chunk_shape": (3, 50, 64), "index_crc": True})
BLOSC_LZ4 = (("bytes", v3.blosc("lz4")), None)
STORES = {"sharded-zstd-crc32c": SHARDED_ZSTD, "blosc-lz4": BLOSC_LZ4}


@pytest.mark.parametrize("case", [c for c in CASES if not c.error], ids=lambda c: c.name)
def test_device_decode_equals_the_host_decode(xrs, case, tmp_path):  # noqa: F811
    source = case.source(str(tmp_path / "probe"))
    if not source.device_decodable:
        pytest.skip("decoded on the host path")
    got, source, word, _, intact = _device_decode(case, str(tmp_path))
    assert word == 0 and intact
    assert np.array_equal(_bits(got), _bits(case.expected(source))), case.name


@pytest.mark.parametrize("case", [c for c in CASES if c.error], ids=lambda c: c.name)
def test_device_reports_a_crc_mismatch(xrs, case, tmp_path):  # noqa: F811
    _, _, word, paths, intact = _device_decode(case, str(tmp_path))
    assert word >> 24 == v3.CRC32C_MISMATCH and (word & 0xFFFFFF) == 1 and intact


def _scene(tmp_path, kind):
    """The same scene as a v3 store of ``kind``, as a Blosc-LZ4 v2 store and as arrays."""
    from xcube_resampling_b200.io import write_zarr_array

    x, y = swath(300, 240, theta=15.0, seed=11)
    rng = np.random.default_rng(6)
    h, w = x.shape
    rad = (rng.integers(0, 400, (7, h, w)) / 16).astype(np.float32)
    cls = rng.integers(0, 9, (h, w)).astype(np.int16)
    codecs, shard = STORES[kind]
    store = str(tmp_path / f"{kind}.zarr")
    v3.write_v3_group(store)
    v3.write_v3_array(os.path.join(store, "lon"), x, (64, 64), ("y", "x"), codecs=("bytes", "zstd"))
    v3.write_v3_array(os.path.join(store, "lat"), y, (64, 64), ("y", "x"), codecs=("bytes", "zstd"))
    v3.write_v3_array(os.path.join(store, "rad"), rad, (6, 100, 128) if shard else (3, 50, 64), ("band", "y", "x"),
                      codecs=codecs, shard=shard)
    cls_shard = dict(shard, chunk_shape=(50, 64)) if shard else None
    v3.write_v3_array(os.path.join(store, "cls"), cls, (100, 128) if shard else (50, 64), ("y", "x"),
                      codecs=tuple(c if c != v3.blosc("lz4") else v3.blosc("lz4", typesize=2) for c in codecs),
                      shard=cls_shard)
    v2 = tmp_path / f"{kind}_v2.zarr"
    write_zarr_array(str(v2 / "lon"), x, (64, 64), ("y", "x"))
    write_zarr_array(str(v2 / "lat"), y, (64, 64), ("y", "x"))
    write_zarr_array(str(v2 / "rad"), rad, (3, 50, 64), ("band", "y", "x"))
    write_zarr_array(str(v2 / "cls"), cls, (50, 64), ("y", "x"))
    meta = {"id": "blosc", "cname": "lz4", "clevel": 5, "shuffle": 1, "blocksize": 0}
    _compress_store(str(v2 / "rad"), lambda r: _blosc_frame(r, 4, 16384, True, "lz4"), meta)
    _compress_store(str(v2 / "cls"), lambda r: _blosc_frame(r, 2, 16384, True, "lz4"), meta)
    return x, y, rad, cls, store, str(v2)


def _memory(xrs, x, y, rad, cls):  # noqa: F811
    return xrs.Dataset(data_vars={"rad": (("band", "y", "x"), rad), "cls": (("y", "x"), cls)},
                       coords={"lon": (("y", "x"), x), "lat": (("y", "x"), y)})


@pytest.mark.parametrize("devices", [None, [0, 0]])
@pytest.mark.parametrize("kind", sorted(STORES))
def test_rectify_from_a_v3_store(xrs, tmp_path, kind, devices):  # noqa: F811
    from xcube_resampling_b200.io import open_zarr_dataset

    x, y, rad, cls, store, v2 = _scene(tmp_path, kind)
    res = 0.0027
    size, xy_min = covering_grid_args(x, y, res)
    tgt_gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=128)
    src_gm = xrs.GridMapping.from_coords(x, y, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
    interp = {"rad": "bilinear", "cls": "nearest"}
    ds = open_zarr_dataset(store)
    assert ds["rad"].source.device_decodable and ds["cls"].source.device_decodable
    got = xrs.rectify_dataset(ds, target_gm=tgt_gm, source_gm=src_gm, interp_methods=interp, devices=devices)
    from_v2 = xrs.rectify_dataset(open_zarr_dataset(v2), target_gm=tgt_gm, source_gm=src_gm, interp_methods=interp,
                                  devices=devices)
    from_mem = xrs.rectify_dataset(_memory(xrs, x, y, rad, cls), target_gm=tgt_gm, source_gm=src_gm,
                                   interp_methods=interp, devices=devices)
    for name in interp:
        assert_same(got[name].values, from_v2[name].values, f"{name} from the {kind} store vs v2, devices={devices}")
        assert_same(got[name].values, from_mem[name].values, f"{name} from the {kind} store vs memory")


@pytest.mark.parametrize("devices", [None, [0, 0]])
@pytest.mark.parametrize("kind", sorted(STORES))
def test_reproject_from_a_v3_store(xrs, tmp_path, kind, devices):  # noqa: F811
    from xcube_resampling_b200.io import open_zarr_dataset, write_zarr_array

    src_gm = xrs.GridMapping.regular((400, 360), (9.0, 47.0), 0.01, "EPSG:4326")
    tgt_gm = xrs.GridMapping.regular((560, 760), (4180000.0, 2660000.0), 450.0, "EPSG:3035", tile_size=96)
    rng = np.random.default_rng(3)
    data = (rng.integers(0, 300, (5, src_gm.height, src_gm.width)) / 8).astype(np.float32)
    codecs, shard = STORES[kind]
    store = str(tmp_path / "r.zarr")
    v3.write_v3_group(store)
    v3.write_v3_array(os.path.join(store, "lon"), src_gm.x_values, (400,), ("lon",), codecs=("bytes", "zstd"))
    v3.write_v3_array(os.path.join(store, "lat"), src_gm.y_values, (360,), ("lat",), codecs=("bytes", "zstd"))
    v3.write_v3_array(os.path.join(store, "v"), data, (4, 256, 256) if shard else (2, 128, 128),
                      ("band", "lat", "lon"), codecs=codecs,
                      shard=dict(shard, chunk_shape=(2, 128, 128)) if shard else None)
    v2 = tmp_path / "r_v2.zarr"
    write_zarr_array(str(v2 / "lon"), src_gm.x_values, (400,), ("lon",))
    write_zarr_array(str(v2 / "lat"), src_gm.y_values, (360,), ("lat",))
    write_zarr_array(str(v2 / "v"), data, (2, 128, 128), ("band", "lat", "lon"))
    mem = xrs.Dataset(data_vars={"v": (("band", "lat", "lon"), data)},
                      coords={"lon": (("lon",), src_gm.x_values), "lat": (("lat",), src_gm.y_values)})
    for method in ("nearest", "bilinear"):
        got = xrs.reproject_dataset(open_zarr_dataset(store), tgt_gm, source_gm=src_gm, interp_methods=method,
                                    devices=devices)
        for other, what in ((open_zarr_dataset(str(v2)), "v2"), (mem, "memory")):
            want = xrs.reproject_dataset(other, tgt_gm, source_gm=src_gm, interp_methods=method, devices=devices)
            assert_same(got["v"].values, want["v"].values, f"{method} from the {kind} store vs {what}")


def test_h2d_bytes_are_the_inner_chunks(xrs, tmp_path):  # noqa: F811
    """Only the inner chunks that intersect the segments cross PCIe (plus the chunk table), never whole shards."""
    import torch

    from xcube_resampling_b200._pipeline import GatherPipeline, SourceGroup, Target
    from xcube_resampling_b200.io import ZarrV3Source

    rng = np.random.default_rng(2)
    a = (rng.integers(0, 100, (4, 90, 130)) / 4).astype(np.float32)
    path = str(tmp_path / "a")
    v3.write_v3_array(path, a, (2, 64, 80), ("band", "y", "x"), codecs=("bytes", "zstd", "crc32c"),
                      shard={"chunk_shape": (1, 32, 40), "index_crc": True})
    src = ZarrV3Source(path)
    segments = [(10, 40, 20, 50), (40, 70, 85, 130)]
    window = (10, 70)
    pipe = GatherPipeline(0, (90, 130), 8, (0, 8), src_window=window, segments=segments)
    seen = []

    def process(src_view, target, out_view, b0):
        seen.append((b0, src_view.clone()))

    out = np.zeros((4, 8, 8), np.float32)
    pipe.run([SourceGroup(src, [Target("a", "nearest", 0.0, out)])], process)
    torch.cuda.synchronize()
    tiles = {(kj, ki) for (j0, j1, i0, i1) in segments for kj in range(j0 // 32, -(-j1 // 32))
             for ki in range(i0 // 40, -(-i1 // 40))}
    per = (2, 2, 2)  # inner chunks per shard (2, 64, 80) / (1, 32, 40)

    def inner_size(kb, kj, ki):  # from the shard's index, parsed here
        shard = os.path.join(path, "c", str(kb // 2), str(kj // 2), str(ki // 2))
        index = v3.shard_index(shard, 8, start=False, crc=True)
        return int(index[np.ravel_multi_index((kb % 2, kj % 2, ki % 2), per), 1])

    inner = sum(inner_size(kb, kj, ki) for kb in range(4) for (kj, ki) in tiles)
    shards = sum(os.path.getsize(os.path.join(dp, f)) for dp, _, fs in os.walk(os.path.join(path, "c")) for f in fs)
    assert pipe.h2d_bytes == inner < shards
    for b0, view in seen:
        v = view.cpu().numpy()
        for (j0, j1, i0, i1) in segments:
            assert np.array_equal(v[:, j0 - window[0]:j1 - window[0], i0:i1], a[b0:b0 + len(v), j0:j1, i0:i1])


def test_a_bad_crc_raises_naming_the_shard_and_inner_chunk(xrs, tmp_path):  # noqa: F811
    from xcube_resampling_b200._lib import XrsError
    from xcube_resampling_b200.io import open_zarr_dataset

    x, y, rad, cls, store, _ = _scene(tmp_path, "sharded-zstd-crc32c")
    # inner chunk (1, 1, 2) of rad's (3, 50, 64) inner chunks: shard (0, 0, 1) of (6, 100, 128), place (1, 1, 0)
    shard_file = os.path.join(store, "rad", "c", "0", "0", "1")
    off, size = (int(v) for v in v3.shard_index(shard_file, 8, start=False, crc=True)[
        np.ravel_multi_index((1, 1, 0), (2, 2, 2))])
    data = bytearray(open(shard_file, "rb").read())
    data[off + size - 3] ^= 0x40  # a bit of the inner chunk's CRC-32C trailer
    open(shard_file, "wb").write(bytes(data))
    res = 0.0027
    size_, xy_min = covering_grid_args(x, y, res)
    tgt_gm = xrs.GridMapping.regular(size_, xy_min, res, "EPSG:4326", tile_size=128)
    src_gm = xrs.GridMapping.from_coords(x, y, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
    with pytest.raises(XrsError, match=r"c/0/0/1 \(inner chunk \(1, 1, 2\)\).*CRC-32C"):
        xrs.rectify_dataset(open_zarr_dataset(store), target_gm=tgt_gm, source_gm=src_gm,
                            interp_methods={"rad": "bilinear"}, variables="rad")


class _Bytes1D:
    """A (1, n) uint8 array of (1, 1) chunks: the geometry xrs_zarr_decode gets for the CRC-32C sweep."""

    def __init__(self, n):
        self.shape, self.chunks, self.dtype = (1, n), (1, 1), np.dtype(np.uint8)

    def device_fill_bits(self):
        return 0


def _sweep_files(sse42, wrong=None):
    """Flagged chunk files whose payloads follow the CRC-32C sweep, each decoding to one byte: real lz4 / zlib / zstd
    streams of 6 to 10 bytes, then Blosc frames stored whole (a 16-byte header and the byte) padded to every sweep length
    from 17 bytes on, the known-answer vectors as padding of five of them.  Files sit at odd offsets; ``wrong``: the
    file whose trailer is off by one bit.  Returns (data, table, the decoded bytes)."""
    import pyarrow as pa

    from xcube_resampling_b200.io import (CHUNK_BLOSC, CHUNK_CRC32C, CHUNK_LZ4, CHUNK_TABLE_DTYPE, CHUNK_ZLIB,
                                          CHUNK_ZSTD)

    rng = np.random.default_rng(4)
    files = [(CHUNK_LZ4, (1).to_bytes(4, "little") + bytes([0x10, 11])),
             (CHUNK_ZLIB, zlib.compress(bytes([12]))),
             (CHUNK_ZSTD, pa.Codec("zstd").compress(bytes([13])).to_pybytes())]
    pads = [v for v, _ in v3.KNOWN] + [rng.integers(0, 256, n - 17, dtype=np.uint8).tobytes()
                                       for n in v3.crc_sweep_lengths() if n >= 17]
    for k, pad in enumerate(pads):
        n = 17 + len(pad)
        head = bytes([2, 1, 0x2, 1]) + (1).to_bytes(4, "little") + (1).to_bytes(4, "little") + n.to_bytes(4, "little")
        files.append((CHUNK_BLOSC, head + bytes([k % 251]) + pad))
    data, table, values = bytearray(), np.zeros(len(files), CHUNK_TABLE_DTYPE), []
    for k, (codec, payload) in enumerate(files):
        data += bytes(k % 7 + 1)
        crc = sse42(payload) ^ (1 << (k % 32) if k == wrong else 0)
        table[k]["offset"], table[k]["length"], table[k]["col"] = len(data), len(payload) + 4, k
        table[k]["codec"] = codec | CHUNK_CRC32C
        table[k]["header"][:min(16, len(payload))] = np.frombuffer(payload[:16], np.uint8)
        data += payload + crc.to_bytes(4, "little")
        values.append(payload[16] if codec == CHUNK_BLOSC else payload[-1] if codec == CHUNK_LZ4 else 11 + k)
    return bytes(data), table, values


def _run_decode(lib, data, table):
    import torch

    from xcube_resampling_b200 import _dev
    from xcube_resampling_b200._pipeline import zarr_decode, zarr_workspace_bytes

    source = _Bytes1D(len(table))
    d = torch.from_numpy(np.frombuffer(data, np.uint8).copy()).cuda()
    ws_bytes = zarr_workspace_bytes(lib, source, table)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    wp = -(-len(table) // 128) * 128
    slot = torch.zeros(wp, dtype=torch.uint8, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    rc = zarr_decode(lib, source, d.data_ptr(), len(data), table, slot.data_ptr(), wp, wp, (0, 1), 0, 1,
                     ws.data_ptr(), ws_bytes, err.data_ptr(), _dev.stream_ptr())
    assert rc == 0, lib.xrs_last_error()
    torch.cuda.synchronize()
    return int(err.cpu().numpy().view(np.uint32)[0]), slot.cpu().numpy()[:len(table)]


def test_k_crc32c_sweep_on_the_device(xrs, tmp_path):  # noqa: F811
    """k_crc32c on the device over payloads of the CRC-32C sweep at odd offsets, trailers from the SSE4.2 instruction:
    every file passes and decodes; a wrong trailer bit or a flipped payload bit of any one file is reported for it."""
    from xcube_resampling_b200._lib import load

    sse42 = v3.sse42_crc32c(str(tmp_path))
    if sse42 is None:
        pytest.skip("needs gcc and an x86 CPU with SSE4.2")
    lib = load()
    data, table, values = _sweep_files(sse42)
    word, got = _run_decode(lib, data, table.copy())
    assert word == 0 and got.tolist() == values
    for k in range(len(table)):
        d, t, _ = _sweep_files(sse42, wrong=k)
        word, _ = _run_decode(lib, d, t)
        assert word >> 24 == v3.CRC32C_MISMATCH and (word & 0xFFFFFF) - 1 == k, (k, int(t[k]["length"]))
    for k in range(3, len(table), 5):  # a flipped bit in the padding of a stored frame
        d = bytearray(data)
        n = int(table[k]["length"]) - 4
        if n > 17:
            d[int(table[k]["offset"]) + 17 + (n - 17) // 2] ^= 0x20
            word, _ = _run_decode(lib, bytes(d), table.copy())
            assert word >> 24 == v3.CRC32C_MISMATCH and (word & 0xFFFFFF) - 1 == k, (k, n)
