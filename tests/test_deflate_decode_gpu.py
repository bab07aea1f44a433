"""Deflate-compressed Zarr chunks decoded on the device (``k_inflate``, csrc/decode.cu): the case table of
tests/deflate_decode_cases.py bit for bit against the host decode, malformed files reported, and the band pipeline fed
from numcodecs-zlib, numcodecs-gzip and Blosc-Zlib stores giving exactly what the host-decoded call gives."""

import gzip
import json
import os
import zlib

import numpy as np
import pytest

from . import deflate_decode_cases as dc
from .helpers import assert_same, covering_grid_args, swath
from .test_host_io import _blosc_frame, _compress_store
from .test_zarr_decode_gpu import _bits, _device_decode, xrs  # noqa: F401  (xrs: the module fixture)
from .test_zstd_decode_gpu import _host_only

pytestmark = pytest.mark.gpu
CASES = dc.cases()
STORES = {"zlib": (lambda r, t: zlib.compress(r, 1), {"id": "zlib", "level": 1}),
          "gzip": (lambda r, t: gzip.compress(r, 1, mtime=0), {"id": "gzip", "level": 1}),
          "blosc-zlib": (lambda r, t: _blosc_frame(r, t, 16384, True, "zlib"), dc.BLOSC_ZLIB)}


@pytest.mark.parametrize("case", [c for c in CASES if not c.error], ids=lambda c: c.name)
def test_device_decode_equals_the_host_decode(xrs, case, tmp_path):  # noqa: F811
    got, source, word, _, intact = _device_decode(case, str(tmp_path))
    assert word == 0 and intact
    assert np.array_equal(_bits(got), _bits(case.expected(source))), case.name


@pytest.mark.parametrize("case", [c for c in CASES if c.error], ids=lambda c: c.name)
def test_device_rejects_malformed_chunks(xrs, case, tmp_path):  # noqa: F811
    _, _, word, paths, intact = _device_decode(case, str(tmp_path))
    assert word >> 24 == case.error and (word & 0xFFFFFF) == 1 and intact


def _scene(tmp_path, kind):
    from xcube_resampling_b200.io import write_zarr_array

    x, y = swath(300, 240, theta=15.0, seed=11)
    h, w = x.shape
    rng = np.random.default_rng(6)
    rad = (rng.integers(0, 400, (7, h, w)) / 16).astype(np.float32)
    cls = rng.integers(0, 9, (h, w)).astype(np.int16)
    store = tmp_path / f"{kind}.zarr"
    write_zarr_array(str(store / "lon"), x, (64, 64), ("y", "x"))
    write_zarr_array(str(store / "lat"), y, (64, 64), ("y", "x"))
    write_zarr_array(str(store / "rad"), rad, (3, 100, 128), ("band", "y", "x"))
    write_zarr_array(str(store / "cls"), cls, (64, 300), ("y", "x"))
    enc, meta = STORES[kind]
    _compress_store(str(store / "rad"), lambda r: enc(r, 4), meta)
    _compress_store(str(store / "cls"), lambda r: enc(r, 2), meta)
    return x, y, str(store)


@pytest.mark.parametrize("devices", [None, [0, 0]])
@pytest.mark.parametrize("kind", sorted(STORES))
def test_rectify_from_a_deflate_store(xrs, tmp_path, kind, devices):  # noqa: F811
    from xcube_resampling_b200.io import open_zarr_dataset

    x, y, store = _scene(tmp_path, kind)
    res = 0.0027
    size, xy_min = covering_grid_args(x, y, res)
    tgt_gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=128)
    src_gm = xrs.GridMapping.from_coords(x, y, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
    interp = {"rad": "bilinear", "cls": "nearest"}
    ds = open_zarr_dataset(store)
    assert ds["rad"].source.device_decodable and ds["cls"].source.device_decodable
    got = xrs.rectify_dataset(ds, target_gm=tgt_gm, source_gm=src_gm, interp_methods=interp, devices=devices)
    want = xrs.rectify_dataset(_host_only(open_zarr_dataset(store)), target_gm=tgt_gm, source_gm=src_gm,
                               interp_methods=interp, devices=devices)
    for name in interp:
        assert_same(got[name].values, want[name].values, f"{name} from the {kind} store, devices={devices}")


@pytest.mark.parametrize("devices", [None, [0, 0]])
@pytest.mark.parametrize("kind", sorted(STORES))
def test_reproject_from_a_deflate_store(xrs, tmp_path, kind, devices):  # noqa: F811
    from xcube_resampling_b200.io import open_zarr_dataset, write_zarr_array

    src_gm = xrs.GridMapping.regular((400, 360), (9.0, 47.0), 0.01, "EPSG:4326")
    tgt_gm = xrs.GridMapping.regular((560, 760), (4180000.0, 2660000.0), 450.0, "EPSG:3035", tile_size=96)
    rng = np.random.default_rng(3)
    data = (rng.integers(0, 300, (5, src_gm.height, src_gm.width)) / 8).astype(np.float32)
    store = tmp_path / "r.zarr"
    write_zarr_array(str(store / "lon"), src_gm.x_values, (400,), ("lon",))
    write_zarr_array(str(store / "lat"), src_gm.y_values, (360,), ("lat",))
    write_zarr_array(str(store / "v"), data, (2, 128, 128), ("band", "lat", "lon"))
    enc, meta = STORES[kind]
    _compress_store(str(store / "v"), lambda r: enc(r, 4), meta)
    for method in ("nearest", "bilinear"):
        want = xrs.reproject_dataset(_host_only(open_zarr_dataset(str(store))), tgt_gm, source_gm=src_gm,
                                     interp_methods=method)
        got = xrs.reproject_dataset(open_zarr_dataset(str(store)), tgt_gm, source_gm=src_gm, interp_methods=method,
                                    devices=devices)
        assert_same(got["v"].values, want["v"].values, f"{method} from the {kind} store, devices={devices}")


@pytest.mark.parametrize("kind", sorted(STORES))
def test_packed_uint16_store_decodes_like_the_host(xrs, tmp_path, kind):  # noqa: F811
    """open_zarr_dataset(mask_and_scale=True) over a packed uint16 store: CF unpacking in the scatter equals the
    host-decoded call."""
    from xcube_resampling_b200.io import open_zarr_dataset, write_zarr_array

    x, y = swath(200, 160, theta=10.0, seed=4)
    rng = np.random.default_rng(9)
    packed = rng.integers(0, 2000, (4, 160, 200)).astype(np.uint16)
    packed[:, 20:30, 40:90] = 65535
    packed[1, 60:70, :] = 7
    store = tmp_path / "p.zarr"
    write_zarr_array(str(store / "lon"), x, (64, 64), ("y", "x"))
    write_zarr_array(str(store / "lat"), y, (64, 64), ("y", "x"))
    write_zarr_array(str(store / "rad"), packed, (1, 64, 100), ("band", "y", "x"))
    enc, meta = STORES[kind]
    _compress_store(str(store / "rad"), lambda r: enc(r, 2), meta)
    attrs = json.load(open(store / "rad" / ".zattrs"))
    attrs.update(scale_factor=0.02, add_offset=-1.5, _FillValue=65535, missing_value=[7])
    json.dump(attrs, open(store / "rad" / ".zattrs", "w"))
    (store / "rad" / "2.1.1").unlink()  # a missing chunk: the fill value, masked
    res = 0.004
    size, xy_min = covering_grid_args(x, y, res)
    tgt_gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=128)
    src_gm = xrs.GridMapping.from_coords(x, y, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
    dev = open_zarr_dataset(str(store), mask_and_scale=True)
    assert dev["rad"].source.device_decodable and dev["rad"].dtype == np.float32
    for method in ("nearest", "bilinear"):
        got = xrs.rectify_dataset(dev, target_gm=tgt_gm, source_gm=src_gm, interp_methods=method)
        want = xrs.rectify_dataset(_host_only(open_zarr_dataset(str(store), mask_and_scale=True)), target_gm=tgt_gm,
                                   source_gm=src_gm, interp_methods=method)
        assert_same(got["rad"].values, want["rad"].values, method)
        assert np.isnan(got["rad"].values).any() and np.isfinite(got["rad"].values).mean() > 0.3


@pytest.mark.parametrize("kind", sorted(STORES))
def test_h2d_bytes_are_the_compressed_chunk_files(xrs, tmp_path, kind):  # noqa: F811
    import torch

    from xcube_resampling_b200._pipeline import GatherPipeline, SourceGroup, Target
    from xcube_resampling_b200.io import ZarrV2Source, write_zarr_array

    rng = np.random.default_rng(2)
    a = (rng.integers(0, 100, (4, 90, 130)) / 4).astype(np.float32)
    path = str(tmp_path / "a")
    write_zarr_array(path, a, (1, 32, 40), ("band", "y", "x"))
    enc, meta = STORES[kind]
    _compress_store(path, lambda r: enc(r, 4), meta)
    src = ZarrV2Source(path)
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
    files = sum(os.path.getsize(os.path.join(path, f"{kb}.{kj}.{ki}")) for kb in range(4) for (kj, ki) in tiles)
    assert pipe.h2d_bytes == files
    for b0, view in seen:
        v = view.cpu().numpy()
        for (j0, j1, i0, i1) in segments:
            assert np.array_equal(v[:, j0 - window[0]:j1 - window[0], i0:i1], a[b0:b0 + len(v), j0:j1, i0:i1])


@pytest.mark.parametrize("kind", sorted(STORES))
def test_a_malformed_deflate_chunk_raises_naming_the_file(xrs, tmp_path, kind):  # noqa: F811
    from xcube_resampling_b200._lib import XrsError
    from xcube_resampling_b200.io import open_zarr_dataset

    x, y, store = _scene(tmp_path, kind)
    bad = store + "/rad/1.1.1"
    data = bytearray(open(bad, "rb").read())
    if kind == "blosc-zlib":  # the Adler-32 of the first stream of the first block that is not stored
        pos = int.from_bytes(data[16:20], "little")
        while data[pos + 4] != 0x78:
            pos += 4 + int.from_bytes(data[pos:pos + 4], "little")
        end = pos + 4 + int.from_bytes(data[pos:pos + 4], "little")
        data[end - 1] ^= 1
    else:  # the Adler-32 / the CRC-32
        data[-1 if kind == "zlib" else -8] ^= 1
    open(bad, "wb").write(bytes(data))
    res = 0.0027
    size, xy_min = covering_grid_args(x, y, res)
    tgt_gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=128)
    src_gm = xrs.GridMapping.from_coords(x, y, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
    with pytest.raises(XrsError, match="1.1.1.*checksum mismatch"):
        xrs.rectify_dataset(open_zarr_dataset(store), target_gm=tgt_gm, source_gm=src_gm,
                            interp_methods={"rad": "bilinear"}, variables="rad")
