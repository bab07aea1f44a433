"""Compressed Zarr chunks decoded on the device (``xrs_zarr_decode``, csrc/decode.cu): the case table of
tests/zarr_decode_cases.py bit for bit against the host decode, malformed files reported, and the band pipeline fed
from Blosc-LZ4 stores giving exactly what uncompressed stores and in-memory arrays give."""

import numpy as np
import pytest

from . import zarr_decode_cases
from .helpers import assert_same, covering_grid_args, swath
from .test_host_io import _blosc_frame, _compress_store

pytestmark = pytest.mark.gpu
CASES = zarr_decode_cases.cases()
POISON = 0x5A


@pytest.fixture(scope="module")
def xrs():
    import torch

    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import xcube_resampling_b200 as pkg

    return pkg


def _device_decode(case, root):
    import torch

    from xcube_resampling_b200 import _dev
    from xcube_resampling_b200._lib import load
    from xcube_resampling_b200._pipeline import zarr_decode, zarr_workspace_bytes

    lib = load()
    source = case.source(root)
    b0, nb, window = case.read()
    buf, n_bytes, table, paths = source.device_read(b0, nb, [(window[0], window[1], 0, source.shape[-1])], window)
    data = torch.from_numpy(buf[:max(n_bytes, 1)].copy()).cuda()
    ws_bytes = zarr_workspace_bytes(lib, source, table)
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device="cuda")
    win_h, w = window[1] - window[0], source.shape[-1]
    wp = -(-w // 32) * 32 + 32
    dt = np.dtype(source.dtype).newbyteorder("=")
    slot = torch.full(((nb + 2) * (win_h + 2) * wp * dt.itemsize,), POISON, dtype=torch.uint8, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    base = slot.data_ptr() + ((win_h + 2) * wp + wp) * dt.itemsize  # band 1, row 1 of the poisoned block
    rc = zarr_decode(lib, source, data.data_ptr(), n_bytes, table, base, wp, (win_h + 2) * wp, window, b0, nb,
                     ws.data_ptr(), ws_bytes, err.data_ptr(), _dev.stream_ptr())
    assert rc == 0, lib.xrs_last_error()
    torch.cuda.synchronize()
    host = slot.cpu().numpy().view(dt).reshape(nb + 2, win_h + 2, wp)
    inner = np.zeros(host.shape, bool)
    inner[1:nb + 1, 1:win_h + 1, :w] = True
    intact = bool(np.all(host.view(np.uint8).reshape(host.shape + (-1,))[~inner] == POISON))
    word = int(err.cpu().numpy().view(np.uint32)[0])
    return host[1:nb + 1, 1:win_h + 1, :w], source, word, paths, intact


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.dtype(f"u{a.dtype.itemsize}"))


@pytest.mark.parametrize("case", [c for c in CASES if not c.error], ids=lambda c: c.name)
def test_device_decode_equals_the_host_decode(xrs, case, tmp_path):
    got, source, word, _, intact = _device_decode(case, str(tmp_path))
    assert word == 0 and intact
    assert np.array_equal(_bits(got), _bits(case.expected(source))), case.name


@pytest.mark.parametrize("case", [c for c in CASES if c.error], ids=lambda c: c.name)
def test_device_rejects_malformed_chunks(xrs, case, tmp_path):
    _, _, word, paths, intact = _device_decode(case, str(tmp_path))
    assert word >> 24 == case.error and (word & 0xFFFFFF) == 1 and intact


def _blosc_store(path, shuffle_typesize, blocksize):
    _compress_store(path, lambda r: _blosc_frame(r, shuffle_typesize, blocksize, True, "lz4"),
                    {"id": "blosc", "cname": "lz4", "clevel": 5, "shuffle": 1, "blocksize": 0})


def _scene_stores(tmp_path):
    from xcube_resampling_b200.io import write_zarr_array

    x, y = swath(300, 240, theta=15.0, seed=11)
    h, w = x.shape
    rng = np.random.default_rng(6)
    rad = (rng.integers(0, 400, (7, h, w)) / 16).astype(np.float32)
    cls = rng.integers(0, 30, (h, w)).astype(np.uint8)
    stores = {}
    for kind in ("plain", "blosc"):
        store = tmp_path / f"{kind}.zarr"
        write_zarr_array(str(store / "lon"), x, (64, 64), ("y", "x"))
        write_zarr_array(str(store / "lat"), y, (64, 64), ("y", "x"))
        write_zarr_array(str(store / "rad"), rad, (3, 100, 128), ("band", "y", "x"))  # depth 3 vs chunks 1, 2, 4
        write_zarr_array(str(store / "cls"), cls, (64, 300), ("y", "x"))
        if kind == "blosc":
            _blosc_store(str(store / "rad"), 4, 4096)
            _blosc_store(str(store / "cls"), 1, 8192)
        stores[kind] = str(store)
    return x, y, rad, cls, stores


@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_rectify_from_a_blosc_store(xrs, tmp_path, devices):
    from xcube_resampling_b200.io import open_zarr_dataset

    x, y, rad, cls, stores = _scene_stores(tmp_path)
    res = 0.0027
    size, xy_min = covering_grid_args(x, y, res)
    tgt_gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=128)
    src_gm = xrs.GridMapping.from_coords(x, y, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
    eager = xrs.Dataset(data_vars=dict(rad=(("band", "y", "x"), rad), cls=(("y", "x"), cls)),
                        coords=dict(lon=(("y", "x"), x), lat=(("y", "x"), y)))
    interp = {"rad": "bilinear", "cls": "nearest"}
    want = xrs.rectify_dataset(eager, target_gm=tgt_gm, source_gm=src_gm, interp_methods=interp, devices=devices)
    for kind in ("plain", "blosc"):
        ds = open_zarr_dataset(stores[kind])
        assert ds["rad"].source.device_decodable == (kind == "blosc")
        got = xrs.rectify_dataset(ds, target_gm=tgt_gm, source_gm=src_gm, interp_methods=interp, devices=devices)
        for name in interp:
            assert_same(got[name].values, want[name].values, f"{name} from the {kind} store, devices={devices}")


@pytest.mark.parametrize("devices", [None, [0, 0]])
def test_reproject_from_a_blosc_store(xrs, tmp_path, devices):
    from xcube_resampling_b200.io import open_zarr_dataset, write_zarr_array

    src_gm = xrs.GridMapping.regular((400, 360), (9.0, 47.0), 0.01, "EPSG:4326")
    tgt_gm = xrs.GridMapping.regular((560, 760), (4180000.0, 2660000.0), 450.0, "EPSG:3035", tile_size=96)
    rng = np.random.default_rng(3)
    data = (rng.integers(0, 300, (5, src_gm.height, src_gm.width)) / 8).astype(np.float32)
    store = tmp_path / "r.zarr"
    write_zarr_array(str(store / "lon"), src_gm.x_values, (400,), ("lon",))
    write_zarr_array(str(store / "lat"), src_gm.y_values, (360,), ("lat",))
    write_zarr_array(str(store / "v"), data, (2, 128, 128), ("band", "lat", "lon"))
    _blosc_store(str(store / "v"), 4, 16384)
    eager = xrs.Dataset(data_vars=dict(v=xrs.DataArray(data, dims=("band", "lat", "lon"))),
                        coords=dict(lon=xrs.DataArray(src_gm.x_values, dims="lon"),
                                    lat=xrs.DataArray(src_gm.y_values, dims="lat")))
    for method in ("nearest", "bilinear"):
        want = xrs.reproject_dataset(eager, tgt_gm, source_gm=src_gm, interp_methods=method)
        got = xrs.reproject_dataset(open_zarr_dataset(str(store)), tgt_gm, source_gm=src_gm, interp_methods=method,
                                    devices=devices)
        assert_same(got["v"].values, want["v"].values, f"{method}, devices={devices}")


def test_packed_uint16_store_decodes_like_the_host(xrs, tmp_path):
    """open_zarr_dataset(mask_and_scale=True): CF unpacking in the scatter equals DecodedSource.read_bands."""
    import json

    from xcube_resampling_b200.io import LazySource, open_zarr_dataset, write_zarr_array

    x, y = swath(200, 160, theta=10.0, seed=4)
    rng = np.random.default_rng(9)
    packed = rng.integers(0, 2000, (4, 160, 200)).astype(np.uint16)
    packed[:, 20:30, 40:90] = 65535
    packed[1, 60:70, :] = 7
    store = tmp_path / "p.zarr"
    write_zarr_array(str(store / "lon"), x, (64, 64), ("y", "x"))
    write_zarr_array(str(store / "lat"), y, (64, 64), ("y", "x"))
    write_zarr_array(str(store / "rad"), packed, (1, 64, 100), ("band", "y", "x"))
    _blosc_store(str(store / "rad"), 2, 4096)
    attrs = json.load(open(store / "rad" / ".zattrs"))
    attrs.update(scale_factor=0.02, add_offset=-1.5, _FillValue=65535, missing_value=[7])
    json.dump(attrs, open(store / "rad" / ".zattrs", "w"))
    os_remove = store / "rad" / "2.1.1"
    os_remove.unlink()  # a missing chunk: the fill value, masked

    class HostOnly(LazySource):
        def __init__(self, src):
            self.src, self.shape, self.dtype = src, src.shape, src.dtype

        def read_bands(self, b0, nb, out):
            self.src.read_bands(b0, nb, out)

    res = 0.004
    size, xy_min = covering_grid_args(x, y, res)
    tgt_gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=128)
    src_gm = xrs.GridMapping.from_coords(x, y, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
    dev = open_zarr_dataset(str(store), mask_and_scale=True)
    assert dev["rad"].source.device_decodable and dev["rad"].dtype == np.float32
    host = open_zarr_dataset(str(store), mask_and_scale=True)
    host = xrs.Dataset(data_vars=dict(rad=type(host["rad"])(HostOnly(host["rad"].source), dims=host["rad"].dims)),
                       coords=dict(host.coords))
    for method in ("nearest", "bilinear"):
        got = xrs.rectify_dataset(dev, target_gm=tgt_gm, source_gm=src_gm, interp_methods=method)
        want = xrs.rectify_dataset(host, target_gm=tgt_gm, source_gm=src_gm, interp_methods=method)
        assert_same(got["rad"].values, want["rad"].values, method)
        assert np.isnan(got["rad"].values).any() and np.isfinite(got["rad"].values).mean() > 0.3


def test_h2d_bytes_are_the_intersecting_chunk_files(xrs, tmp_path):
    import os

    import torch

    from xcube_resampling_b200._pipeline import GatherPipeline, SourceGroup, Target
    from xcube_resampling_b200.io import ZarrV2Source, write_zarr_array

    rng = np.random.default_rng(2)
    a = (rng.integers(0, 100, (4, 90, 130)) / 4).astype(np.float32)
    path = str(tmp_path / "a")
    write_zarr_array(path, a, (1, 32, 40), ("band", "y", "x"))
    _blosc_store(path, 4, 2048)
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
    for b0, view in seen:  # the segments are in place, at their true position in the window
        v = view.cpu().numpy()
        for (j0, j1, i0, i1) in segments:
            assert np.array_equal(v[:, j0 - window[0]:j1 - window[0], i0:i1], a[b0:b0 + len(v), j0:j1, i0:i1])


def test_a_malformed_chunk_raises_naming_the_file(xrs, tmp_path):
    from xcube_resampling_b200._lib import XrsError
    from xcube_resampling_b200.io import open_zarr_dataset

    x, y, rad, cls, stores = _scene_stores(tmp_path)
    bad = stores["blosc"] + "/rad/1.1.1"
    frame = bytearray(open(bad, "rb").read())
    pos = int.from_bytes(frame[16:20], "little")
    frame[pos:pos + 4] = (len(frame)).to_bytes(4, "little")
    open(bad, "wb").write(bytes(frame))
    res = 0.0027
    size, xy_min = covering_grid_args(x, y, res)
    tgt_gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=128)
    src_gm = xrs.GridMapping.from_coords(x, y, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
    with pytest.raises(XrsError, match="1.1.1"):
        xrs.rectify_dataset(open_zarr_dataset(stores["blosc"]), target_gm=tgt_gm, source_gm=src_gm,
                            interp_methods={"rad": "bilinear"}, variables="rad")
