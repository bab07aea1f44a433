"""Store-fed rectify_dataset: compressed chunks decoded on the host vs on the device (csrc/decode.cu).

Writes a seeded, OLCI-shaped scene (21 x 4091 x 4865 float32, compressible radiance-like values) as Zarr-v2 stores
of the chosen ``--codec``, plus a packed uint16 variant with CF attributes, into a temporary directory:

* ``blosc-lz4`` (default): Blosc-LZ4, byte-shuffled, with 32 KiB and 256 KiB blocks;
* ``blosc-zstd``: the same with Zstd streams (``--zstd-level``);
* ``zstd``: numcodecs ``zstd``, one frame per 1 MiB chunk (``--zstd-level``);
* ``blosc-zlib``: Blosc with Zlib streams (``--zlib-level``, default 1 as numcodecs');
* ``zlib`` / ``gzip``: numcodecs ``zlib`` / ``gzip``, one stream or member per 1 MiB chunk (``--zlib-level``).

``--zarr-format 3`` writes the same scene as Zarr v3 arrays instead (``zarr.json``, ``c/...`` chunk keys, codecs
``bytes`` then the compressor: ``zstd``, ``gzip``, ``blosc`` or ``numcodecs.zlib``); ``--crc32c`` appends the ``crc32c``
codec; ``--shard BANDS,ROWS,COLS`` wraps the chunks into ``sharding_indexed`` shards of that shape (index at the end,
followed by its CRC-32C, as zarr-python writes it).  The device decode then reports ``k_crc32c``'s time beside the
decode kernels'.

  Then times one rectify_dataset call (nearest + bilinear of the same bands) three ways:

* ``memory``: the bands as page-locked in-memory arrays;
* ``host_decode``: the store through a plain LazySource that offers only ``read_bands`` (chunks decoded by
  the store's host decoder (``io.chunk_decoder``) on the pipeline's reader thread);
* ``device_decode``: the store itself (chunk files uploaded compressed, decoded by xrs_zarr_decode).

Also reports the decode kernels' time (CUDA events, one profiled call), GB/s of decoded and of compressed bytes,
the band bytes each path uploads (the band pipeline's ``h2d_bytes`` counter), the device name and power limit, and whether host- and device-decoded outputs are identical.

    python tools/zarr_decode_bench.py --steps 3 --out zarr_decode_bench.json
    python tools/zarr_decode_bench.py --codec zstd --zstd-level 3 --steps 3
    python tools/zarr_decode_bench.py --codec gzip --zlib-level 1 --steps 3
    python tools/zarr_decode_bench.py --codec zstd --zarr-format 3 --shard 1,2048,2048 --crc32c --steps 3
"""

from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _compressor(codec: str, level: int):
    """``bytes -> bytes`` of one Blosc stream or numcodecs chunk, and the Blosc inner codec number."""
    import pyarrow as pa

    if codec == "blosc-lz4":
        c = pa.Codec("lz4_raw")
        return (lambda raw: c.compress(raw).to_pybytes()), 1
    if codec in ("blosc-zlib", "zlib"):
        return (lambda raw: zlib.compress(raw, level)), 3
    if codec == "gzip":
        import gzip

        return (lambda raw: gzip.compress(raw, level, mtime=0)), None
    c = pa.Codec("zstd", compression_level=level)
    return (lambda raw: c.compress(raw).to_pybytes()), 4


def blosc_frame(raw: bytes, typesize: int, blocksize: int, codec: str = "blosc-lz4", level: int = 3) -> bytes:
    """A Blosc-1 frame (byte shuffle, split streams) as numcodecs writes it, per io.blosc_decompress's layout."""
    compress, fmt = _compressor(codec, level)
    flags = (fmt << 5) | 0x1
    nblocks = -(-len(raw) // blocksize)
    parts, starts, pos = [], [], 16 + 4 * nblocks
    for b in range(nblocks):
        block = np.frombuffer(raw, np.uint8, count=min(blocksize, len(raw) - b * blocksize), offset=b * blocksize)
        n = len(block) // typesize
        block = np.concatenate([block[:n * typesize].reshape(n, typesize).T.reshape(-1), block[n * typesize:]])
        split = typesize <= 16 and blocksize // typesize >= 128 and len(block) == blocksize
        ns = typesize if split else 1
        ne = len(block) // ns
        starts.append(pos)
        for k in range(ns):
            part = block[k * ne:(k + 1) * ne].tobytes()
            comp = compress(part)
            if len(comp) >= ne:
                comp = part
            parts.append(len(comp).to_bytes(4, "little") + comp)
            pos += 4 + len(comp)
    head = bytes([2, 1, flags, typesize]) + len(raw).to_bytes(4, "little") + blocksize.to_bytes(4, "little")
    return head + pos.to_bytes(4, "little") + b"".join(s.to_bytes(4, "little") for s in starts) + b"".join(parts)


NUMCODECS = ("zstd", "zlib", "gzip")  # one compressed stream per chunk file, no Blosc container


def _v3_codecs(codec: str, level: int, typesize: int, blocksize: int, crc: bool) -> list:
    """The Zarr v3 codec chain of a store written with ``codec``."""
    if codec == "zstd":
        comp = {"name": "zstd", "configuration": {"level": level, "checksum": False}}
    elif codec == "gzip":
        comp = {"name": "gzip", "configuration": {"level": level}}
    elif codec == "zlib":
        comp = {"name": "numcodecs.zlib", "configuration": {"level": level}}
    else:
        comp = {"name": "blosc", "configuration": {"cname": codec[len("blosc-"):], "clevel": level, "shuffle": "shuffle",
                                                   "typesize": typesize, "blocksize": blocksize}}
    return [{"name": "bytes", "configuration": {"endian": "little"}}, comp] + ([{"name": "crc32c"}] if crc else [])


def write_store(path, array, chunks, blocksize, attrs=None, codec="blosc-lz4", level=3, zarr_format=2, crc=False,
                shard=None):
    os.makedirs(path, exist_ok=True)
    if zarr_format == 3:
        return _write_store_v3(path, array, chunks, blocksize, attrs, codec, level, crc, shard)
    if codec in NUMCODECS:
        compressor = {"id": codec, "level": level}
    else:
        compressor = {"id": "blosc", "cname": codec[len("blosc-"):],
                      "clevel": 5 if codec == "blosc-lz4" else level, "shuffle": 1, "blocksize": blocksize}
    meta = {"chunks": list(chunks), "compressor": compressor,
            "dtype": array.dtype.str, "fill_value": None, "filters": None, "order": "C", "shape": list(array.shape),
            "zarr_format": 2}
    json.dump(meta, open(os.path.join(path, ".zarray"), "w"))
    json.dump(dict(attrs or {}, _ARRAY_DIMENSIONS=["band", "y", "x"]), open(os.path.join(path, ".zattrs"), "w"))
    grid = [range(-(-n // c)) for n, c in zip(array.shape, chunks)]

    def one(idx):
        block = np.zeros(chunks, dtype=array.dtype)
        sl = tuple(slice(k * c, min(n, (k + 1) * c)) for k, c, n in zip(idx, chunks, array.shape))
        part = array[sl]
        block[tuple(slice(0, s) for s in part.shape)] = part
        if codec in NUMCODECS:
            frame = _compressor(codec, level)[0](block.tobytes())
        else:
            frame = blosc_frame(block.tobytes(), array.dtype.itemsize, blocksize, codec, level)
        with open(os.path.join(path, ".".join(str(k) for k in idx)), "wb") as fh:
            fh.write(frame)
        return len(frame)

    with ThreadPoolExecutor(os.cpu_count() or 4) as pool:
        return sum(pool.map(one, np.ndindex(*[len(g) for g in grid])))


def _encode(array, chunks, idx, blocksize, codec, level) -> bytes:
    """The compressed bytes of chunk ``idx`` (edge chunks padded with zeros)."""
    block = np.zeros(chunks, dtype=array.dtype)
    sl = tuple(slice(k * c, min(n, (k + 1) * c)) for k, c, n in zip(idx, chunks, array.shape))
    part = array[sl]
    block[tuple(slice(0, s) for s in part.shape)] = part
    if codec in NUMCODECS:
        return _compressor(codec, level)[0](block.tobytes())
    return blosc_frame(block.tobytes(), array.dtype.itemsize, blocksize, codec, level)


def _write_store_v3(path, array, chunks, blocksize, attrs, codec, level, crc, shard):
    """A Zarr v3 array: chunks (inner chunks of ``shard``-shaped shards) under ``c/``, each followed by its CRC-32C
    when ``crc``; a shard file ends in its index of (offset, nbytes) uint64 pairs and the index's CRC-32C."""
    from xcube_resampling_b200.io import crc32c

    def encode(idx):
        data = _encode(array, chunks, idx, blocksize, codec, level)
        return data + crc32c(data).to_bytes(4, "little") if crc else data

    def put(idx, data):
        p = os.path.join(path, "c", *[str(k) for k in idx])
        os.makedirs(os.path.dirname(p), exist_ok=True)
        with open(p, "wb") as fh:
            fh.write(data)
        return len(data)

    inner = _v3_codecs(codec, level, array.dtype.itemsize, blocksize, crc)
    if shard is None:
        codecs, grid_chunks = inner, list(chunks)

        def one(idx):
            return put(idx, encode(idx))
        units = np.ndindex(*[-(-n // c) for n, c in zip(array.shape, chunks)])
    else:
        per = tuple(s // c for s, c in zip(shard, chunks))
        index_codecs = [{"name": "bytes", "configuration": {"endian": "little"}}, {"name": "crc32c"}]
        codecs = [{"name": "sharding_indexed", "configuration": {
            "chunk_shape": list(chunks), "codecs": inner, "index_codecs": index_codecs, "index_location": "end"}}]
        grid_chunks = list(shard)

        def one(sidx):
            index = np.full((int(np.prod(per)), 2), 2 ** 64 - 1, np.uint64)
            body = bytearray()
            for k, local in enumerate(np.ndindex(*per)):
                idx = tuple(s * p + q for s, p, q in zip(sidx, per, local))
                if all(i * c < n for i, c, n in zip(idx, chunks, array.shape)):
                    data = encode(idx)
                    index[k] = (len(body), len(data))
                    body += data
            raw = index.astype("<u8").tobytes()
            return put(sidx, bytes(body) + raw + crc32c(raw).to_bytes(4, "little"))
        units = np.ndindex(*[-(-n // c) for n, c in zip(array.shape, shard)])
    meta = {"zarr_format": 3, "node_type": "array", "shape": list(array.shape), "data_type": array.dtype.name,
            "chunk_grid": {"name": "regular", "configuration": {"chunk_shape": grid_chunks}},
            "chunk_key_encoding": {"name": "default", "configuration": {"separator": "/"}}, "fill_value": 0,
            "codecs": codecs, "attributes": dict(attrs or {}), "dimension_names": ["band", "y", "x"]}
    json.dump(meta, open(os.path.join(path, "zarr.json"), "w"))
    with ThreadPoolExecutor(os.cpu_count() or 4) as pool:
        return sum(pool.map(one, units))


def radiance(nb, h, w, seed):
    """Smooth fields plus noise, quantised to 1/64: float32 whose low mantissa bytes shuffle into long runs."""
    rng = np.random.default_rng(seed)
    j = np.linspace(0, 6, h, dtype=np.float32)[:, None]
    i = np.linspace(0, 9, w, dtype=np.float32)[None, :]
    out = np.empty((nb, h, w), np.float32)
    for b in range(nb):
        base = 40 + 20 * np.sin(j + b * 0.3) * np.cos(i * 0.7) + 5 * b
        out[b] = np.round((base + rng.normal(0, 0.5, (h, w)).astype(np.float32)) * 64) / 64
    return out


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                            os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="scene size relative to OLCI (1.0: 4865 x 4091)")
    ap.add_argument("--bands", type=int, default=21)
    ap.add_argument("--codec", choices=("blosc-lz4", "blosc-zstd", "zstd", "blosc-zlib", "zlib", "gzip"),
                    default="blosc-lz4")
    ap.add_argument("--zstd-level", type=int, default=3, help="zstd compression level (blosc-zstd, zstd)")
    ap.add_argument("--zlib-level", type=int, default=1, help="zlib compression level (blosc-zlib, zlib, gzip)")
    ap.add_argument("--zarr-format", type=int, choices=(2, 3), default=2, help="write Zarr v2 or v3 stores")
    ap.add_argument("--shard", default=None, help="BANDS,ROWS,COLS: v3 sharding_indexed shards of that shape")
    ap.add_argument("--crc32c", action="store_true", help="v3: the crc32c codec after the compressor")
    ap.add_argument("--out", default=None, help="JSON result file (default: print only)")
    ap.add_argument("--dir", default=None, help="where the stores are written (default: a temporary directory)")
    args = ap.parse_args()
    shard = tuple(int(v) for v in args.shard.split(",")) if args.shard else None
    if args.zarr_format == 2 and (shard or args.crc32c):
        ap.error("--shard and --crc32c need --zarr-format 3")

    import torch

    import xcube_resampling_b200 as xrs
    from xcube_resampling_b200 import _dev, _lib, _pipeline, synthetic as syn
    from xcube_resampling_b200.io import DecodedSource, LazyDataArray, LazySource, ZarrV2Source, ZarrV3Source

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU path and has no CPU fallback")
    w = max(64, int(round(syn.OLCI_WIDTH * args.scale)))
    h = max(64, int(round(syn.OLCI_HEIGHT * args.scale)))
    nb = args.bands
    res = syn.OLCI_RES_DEG
    lon, lat = syn.swath(w, h, res=res, theta=12.0, seed=0)
    size, xy_min = syn.covering_grid_args(lon, lat, res)
    target_gm = xrs.GridMapping.regular(size, xy_min, res, "EPSG:4326", tile_size=512)
    lon_p, lat_p = _dev.pinned_empty(lon.shape, np.float64), _dev.pinned_empty(lat.shape, np.float64)
    lon_p[...], lat_p[...] = lon, lat
    source_gm = xrs.GridMapping.from_coords(lon_p, lat_p, "EPSG:4326", xy_res=res, xy_dim_names=("x", "y"))
    coords = dict(lon=(("y", "x"), lon_p), lat=(("y", "x"), lat_p))
    interp = {"near": "nearest", "bil": "bilinear"}

    root = args.dir or tempfile.mkdtemp(prefix="zarr_decode_bench_")
    rad = radiance(nb, h, w, seed=1)
    chunks = (1, 512, 512)
    if shard and any(s % c for s, c in zip(shard, chunks)):
        raise SystemExit(f"--shard {args.shard} is not a multiple of the chunks {chunks}")
    t0 = time.perf_counter()
    stores = {}
    deflate = args.codec in ("blosc-zlib", "zlib", "gzip")
    kw = dict(codec=args.codec, level=args.zlib_level if deflate else args.zstd_level, zarr_format=args.zarr_format,
              crc=args.crc32c, shard=shard)
    blocks = (("f32", 0),) if args.codec in NUMCODECS else (("f32_block256k", 256 << 10), ("f32_block32k", 32 << 10))
    for label, bs in blocks:
        stores[label] = (os.path.join(root, label), write_store(os.path.join(root, label), rad, chunks, bs, **kw),
                         None)
    packed = np.round((rad + 1.5) / 0.02).astype(np.uint16)
    packed[:, h // 3:h // 3 + 40, :] = 65535
    cf = {"scale_factor": 0.02, "add_offset": -1.5, "_FillValue": 65535}
    stores["u16_cf" if args.codec in NUMCODECS else "u16_cf_block256k"] = (
        os.path.join(root, "u16"), write_store(os.path.join(root, "u16"), packed, chunks, 256 << 10, cf, **kw), cf)
    write_s = time.perf_counter() - t0

    class HostOnly(LazySource):
        """The store behind a source that offers only read_bands: chunks decode on the host."""

        def __init__(self, src):
            self.src, self.shape, self.dtype = src, src.shape, src.dtype

        def read_bands(self, b0, n, out):
            self.src.read_bands(b0, n, out)

    def dataset(values):
        return xrs.Dataset(data_vars={k: (("band", "y", "x"), values) if isinstance(values, np.ndarray)
                                      else LazyDataArray(values, dims=("band", "y", "x")) for k in interp},
                           coords=coords)

    # the band bytes each call uploads, as the band pipeline counts them (GatherPipeline.h2d_bytes)
    uploaded = []
    run = _pipeline.GatherPipeline.run

    def counted_run(self, *a, **k):
        before = self.h2d_bytes
        run(self, *a, **k)
        uploaded.append(self.h2d_bytes - before)

    _pipeline.GatherPipeline.run = counted_run

    def timed(ds, steps):
        """(outputs, ms per call, band H2D bytes of the last call)"""
        out = xrs.rectify_dataset(ds, target_gm=target_gm, source_gm=source_gm, interp_methods=interp)  # warm-up
        times = []
        for _ in range(steps):
            torch.cuda.synchronize()
            uploaded.clear()
            t = time.perf_counter()
            out = xrs.rectify_dataset(ds, target_gm=target_gm, source_gm=source_gm, interp_methods=interp)
            torch.cuda.synchronize()
            times.append((time.perf_counter() - t) * 1e3)
        return out, times, int(sum(uploaded))

    result = {"tool": "tools/zarr_decode_bench.py", "device": torch.cuda.get_device_name(0),
              "power_limit": power_limit(), "scene": {"bands": nb, "height": h, "width": w, "chunks": list(chunks)},
              "target": list(target_gm.size), "store_write_s": round(write_s, 1), "codec": args.codec,
              "zstd_level": None if args.codec == "blosc-lz4" or deflate else args.zstd_level,
              "zarr_format": args.zarr_format, "shard": list(shard) if shard else None, "crc32c": args.crc32c,
              "paths": {}}
    if deflate:
        result["zlib_level"] = args.zlib_level
    mem = _dev.pinned_empty(rad.shape, np.float32)
    mem[...] = rad
    _, t_mem, up_mem = timed(dataset(mem), args.steps)
    result["paths"]["memory_f32"] = {"ms": t_mem, "ms_median": float(np.median(t_mem)), "band_h2d_bytes": up_mem}
    for label, (path, file_bytes, attrs) in stores.items():
        Source = ZarrV3Source if args.zarr_format == 3 else ZarrV2Source
        base = Source(path)
        dev_src = DecodedSource(base, attrs) if attrs else base
        host_src = HostOnly(DecodedSource(Source(path), attrs) if attrs else Source(path))
        assert dev_src.device_decodable
        out_h, t_h, up_h = timed(dataset(host_src), args.steps)
        out_d, t_d, up_d = timed(dataset(dev_src), args.steps)
        same = all(np.array_equal(out_h[k].values.view(np.uint32), out_d[k].values.view(np.uint32)) for k in interp)
        _lib.profile_enable(True)
        xrs.rectify_dataset(dataset(dev_src), target_gm=target_gm, source_gm=source_gm, interp_methods=interp)
        torch.cuda.synchronize()
        prof = _lib.profile_collect()
        _lib.profile_enable(False)
        dec = {k: v for k, v in prof.items() if k.startswith("zarr_")}
        dec_ms = sum(v[0] for v in dec.values())
        decoded = nb * (-(-h // chunks[1]) * chunks[1]) * (-(-w // chunks[2]) * chunks[2]) * base.dtype.itemsize
        result["paths"][label] = {
            "store_file_bytes": int(file_bytes), "decoded_chunk_bytes": int(decoded),
            "host_decode": {"ms": t_h, "ms_median": float(np.median(t_h)), "band_h2d_bytes": up_h},
            "device_decode": {"ms": t_d, "ms_median": float(np.median(t_d)), "band_h2d_bytes": up_d,
                              "decode_kernels_ms": {k: {"ms": v[0], "launches": v[1]} for k, v in dec.items()},
                              "decode_ms": dec_ms,
                              "crc32c_ms": dec.get("zarr_crc32c", (0.0,))[0],
                              "crc32c_share_of_decode": dec.get("zarr_crc32c", (0.0,))[0] / dec_ms if dec_ms else None,
                              "decoded_GBps": decoded / dec_ms / 1e6 if dec_ms else None,
                              "compressed_GBps": up_d / dec_ms / 1e6 if dec_ms else None},
            "host_vs_device_outputs_identical": bool(same)}
        print(json.dumps({label: result["paths"][label]}), flush=True)
    if not args.dir:
        shutil.rmtree(root, ignore_errors=True)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(text)


if __name__ == "__main__":
    main()
