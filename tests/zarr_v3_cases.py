"""Zarr v3 stores written by hand, and the case table of their decode shared by the host tests
(test_host_zarr_v3.py) and the GPU (test_zarr_v3_gpu.py).

The ``zarr`` / ``numcodecs`` packages are not in this build, so :func:`write_v3_array` assembles stores from the Zarr v3
core specification and its ``sharding_indexed`` and ``crc32c`` codec specifications: ``zarr.json`` metadata, chunk keys
of the ``default`` or ``v2`` encoding, and chunk files run through the codec chain in order (``bytes`` with its
endianness, one compressor, a 4-byte little-endian CRC-32C).  A shard file holds its encoded inner chunks back to back and
an index of one little-endian uint64 (offset, nbytes) pair per inner chunk in C order, (2^64 - 1, 2^64 - 1) for an
absent one, at its end or start, optionally followed by the index's CRC-32C.  Compressed streams come from the
standard library, pyarrow and test_host_io's Blosc assembler.

A case is a store plus one read (bands ``b0 : b0 + nb`` of a row ``window``), with the ``Case`` interface of
tests/zarr_decode_cases.py; ``expected`` is the host decode (``read_bands``), which the host tests also compare with the
numpy array and with the same array written as v2."""

from __future__ import annotations

import ctypes
import gzip
import json
import os
import shutil
import subprocess
import zlib
from dataclasses import dataclass, field

import numpy as np

from xcube_resampling_b200.io import DecodedSource, ZarrV3Source, crc32c

from .test_host_io import _blosc_frame
from .zarr_decode_cases import _values, numcodecs_lz4

CRC32C_MISMATCH = 19  # enum xrs_decode_error
MISSING = 2 ** 64 - 1


def _zstd(raw: bytes) -> bytes:
    import pyarrow as pa

    return pa.Codec("zstd").compress(raw).to_pybytes()


def _encoder(codec, typesize: int):
    """bytes -> bytes of one compressor entry of a v3 codec list."""
    name = codec if isinstance(codec, str) else codec["name"]
    conf = {} if isinstance(codec, str) else codec.get("configuration", {})
    if name in ("zstd", "numcodecs.zstd"):
        return _zstd
    if name in ("gzip", "numcodecs.gzip"):
        return lambda r: gzip.compress(r, 5)
    if name == "numcodecs.zlib":
        return lambda r: zlib.compress(r, 5)
    if name == "numcodecs.lz4":
        return numcodecs_lz4
    if name in ("blosc", "numcodecs.blosc"):
        shuffle = conf.get("shuffle", "noshuffle")
        shuffle = shuffle in ("shuffle", 1)
        ts = conf.get("typesize") or typesize
        return lambda r: _blosc_frame(r, ts, 128 * ts, shuffle, conf.get("cname", "lz4"))
    raise ValueError(name)


def encode_chain(raw: bytes, codecs, typesize: int) -> bytes:
    """Run the bytes of one chunk (already in the ``bytes`` codec's byte order) through the bytes -> bytes codecs."""
    for c in codecs:
        name = c if isinstance(c, str) else c["name"]
        if name in ("bytes", "transpose"):
            continue
        if name == "crc32c":
            raw = raw + crc32c(raw).to_bytes(4, "little")
        else:
            raw = _encoder(c, typesize)(raw)
    return raw


def _key(encoding, idx) -> str:
    name = encoding["name"]
    sep = encoding.get("configuration", {}).get("separator", "/" if name == "default" else ".")
    parts = [str(i) for i in idx]
    return sep.join(["c"] + parts) if name == "default" else (sep.join(parts) if parts else "0")


def _write_file(path: str, key: str, data: bytes) -> None:
    p = os.path.join(path, *key.split("/"))
    os.makedirs(os.path.dirname(p), exist_ok=True)
    open(p, "wb").write(data)


def write_v3_array(path: str, array: np.ndarray, chunks, dims=None, codecs=("bytes",), shard=None,
                   key_encoding=None, fill_value=0, attributes=None, missing=(), dimension_names=True,
                   corrupt=None) -> None:
    """A Zarr v3 array.  ``codecs``: the chain (``"bytes"`` becomes ``bytes`` with the array's endianness); ``shard``:
    ``{"chunk_shape", "index_location", "index_crc"}`` -- then ``chunks`` is the shard shape and ``codecs`` the inner
    chain; ``missing``: chunk (or inner chunk) indices not written, whole shards when sharded and an index is listed
    with ``"shard"`` first; ``corrupt(raw) -> raw``: applied to the file of the first chunk written."""
    array = np.asarray(array)
    os.makedirs(path, exist_ok=True)
    key_encoding = key_encoding or {"name": "default", "configuration": {"separator": "/"}}
    endian = {"<": "little", ">": "big", "=": "little", "|": None}[array.dtype.byteorder]

    def chain(cs):
        out = []
        for c in cs:
            if c == "bytes":
                out.append({"name": "bytes", "configuration": {"endian": endian}} if endian else {"name": "bytes"})
            else:
                out.append(c if isinstance(c, dict) else {"name": c, "configuration": {}})
        return out

    inner_chain = chain(codecs)
    unit = tuple(shard["chunk_shape"]) if shard else tuple(chunks)
    typesize = array.dtype.itemsize

    def encoded(idx):
        block = np.zeros(unit, dtype=array.dtype)
        sl = tuple(slice(k * c, min(n, (k + 1) * c)) for k, c, n in zip(idx, unit, array.shape))
        part = array[sl]
        block[tuple(slice(0, s) for s in part.shape)] = part
        return encode_chain(block.tobytes(), inner_chain, typesize)

    first = [True]

    def write(key, data):
        if corrupt is not None and first[0]:
            data = corrupt(data)
        first[0] = False
        _write_file(path, key, data)

    grid = tuple(-(-n // c) for n, c in zip(array.shape, chunks))
    if shard is None:
        for idx in np.ndindex(*grid):
            if idx not in missing:
                write(_key(key_encoding, idx), encoded(idx))
        codec_meta = inner_chain
    else:
        per = tuple(c // i for c, i in zip(chunks, unit))
        n = int(np.prod(per, dtype=np.int64))
        index_bytes = 16 * n + (4 if shard.get("index_crc") else 0)
        start = shard.get("index_location", "end") == "start"
        for sidx in np.ndindex(*grid):
            if ("shard",) + sidx in missing:
                continue
            index = np.full((n, 2), MISSING, np.uint64)
            body = bytearray()
            base = index_bytes if start else 0
            for k, local in enumerate(np.ndindex(*per)):
                idx = tuple(s * p + q for s, p, q in zip(sidx, per, local))
                if idx in missing or any(i * u >= d for i, u, d in zip(idx, unit, array.shape)):
                    continue
                data = encoded(idx)
                index[k] = (base + len(body), len(data))
                body += data
            raw_index = index.astype("<u8").tobytes()
            if shard.get("index_crc"):
                raw_index += crc32c(raw_index).to_bytes(4, "little")
            write(_key(key_encoding, sidx), bytes(raw_index + body) if start else bytes(body + raw_index))
        index_codecs = [{"name": "bytes", "configuration": {"endian": "little"}}]
        if shard.get("index_crc"):
            index_codecs.append({"name": "crc32c", "configuration": {}})
        conf = {"chunk_shape": list(unit), "codecs": inner_chain, "index_codecs": index_codecs}
        if "index_location" in shard:
            conf["index_location"] = shard["index_location"]
        codec_meta = [{"name": "sharding_indexed", "configuration": conf}]
    names = {"float32": "float32", "float64": "float64"}.get(array.dtype.name, array.dtype.name)
    meta = {"zarr_format": 3, "node_type": "array", "shape": list(array.shape), "data_type": names,
            "chunk_grid": {"name": "regular", "configuration": {"chunk_shape": list(chunks)}},
            "chunk_key_encoding": key_encoding, "fill_value": fill_value, "codecs": codec_meta,
            "attributes": dict(attributes or {}), "storage_transformers": []}
    if dimension_names:
        meta["dimension_names"] = list(dims) if dims is not None else None
    json.dump(meta, open(os.path.join(path, "zarr.json"), "w"))


def write_v3_group(path: str, attributes=None) -> None:
    os.makedirs(path, exist_ok=True)
    json.dump({"zarr_format": 3, "node_type": "group", "attributes": dict(attributes or {})},
              open(os.path.join(path, "zarr.json"), "w"))


BLOSC = {"name": "blosc", "configuration": {"cname": "lz4", "clevel": 5, "shuffle": "shuffle", "typesize": 4,
                                            "blocksize": 0}}


def blosc(cname: str, shuffle: str = "shuffle", typesize: int = 4) -> dict:
    return {"name": "blosc", "configuration": {"cname": cname, "clevel": 5, "shuffle": shuffle, "typesize": typesize,
                                               "blocksize": 0}}


def sse42_crc32c(out_dir: str):
    """CRC-32C through the SSE4.2 ``crc32`` instruction, from a small C helper built in ``out_dir``: the reference the
    kernel and ``io.crc32c`` are checked against; ``None`` without gcc or an x86 CPU with SSE4.2."""
    gcc = shutil.which("gcc")
    if gcc is None or not os.path.isfile("/proc/cpuinfo") or "sse4_2" not in open("/proc/cpuinfo").read():
        return None
    src = os.path.join(out_dir, "crc.c")
    open(src, "w").write("#include <nmmintrin.h>\n#include <stddef.h>\n#include <stdint.h>\n"
                         "uint32_t crc32c_sse42(const uint8_t *p, size_t n) {\n"
                         "    uint32_t c = 0xFFFFFFFFu;\n"
                         "    for (size_t k = 0; k < n; ++k) c = _mm_crc32_u8(c, p[k]);\n"
                         "    return c ^ 0xFFFFFFFFu;\n}\n")
    so = os.path.join(out_dir, "libcrc.so")
    subprocess.run([gcc, "-O2", "-msse4.2", "-shared", "-fPIC", src, "-o", so], check=True)
    fn = ctypes.CDLL(so).crc32c_sse42
    fn.restype, fn.argtypes = ctypes.c_uint32, [ctypes.c_char_p, ctypes.c_size_t]
    return lambda data: fn(bytes(data), len(data))


# CRC-32C known answers: "123456789" and the RFC 3720 B.4 vectors
KNOWN = [(b"123456789", 0xE3069283), (bytes(32), 0x8A9136AA), (b"\xff" * 32, 0x62A8AB43),
         (bytes(range(32)), 0x46DD794E), (bytes(range(31, -1, -1)), 0x113FDB5C)]


def crc_sweep_lengths(seed: int = 11) -> list:
    """Payload lengths of the CRC-32C sweep: 0 ... 64 (a warp's 32 lanes get empty or one-byte segments), multiples of
    32 and one either side up to 64 KiB, and random lengths up to 1 MiB, 1 MiB included."""
    rng = np.random.default_rng(seed)
    lengths = list(range(65))
    for k in (3, 4, 5, 7, 8, 31, 32, 33, 100, 1024, 2048):
        lengths += [32 * k - 1, 32 * k, 32 * k + 1]
    lengths += sorted(rng.integers(1 << 10, 1 << 20, 10).tolist()) + [1 << 20]
    return lengths


def spelled_fill(fill, dtype) -> np.ndarray:
    """A v3 ``fill_value`` as a one-element array of ``dtype``, read from its spelling here, not by io.py."""
    dtype = np.dtype(dtype)
    if isinstance(fill, str) and fill.startswith("0x"):
        return np.array([int(fill, 16)], dtype=f"u{dtype.itemsize}").view(dtype.newbyteorder("=")).astype(dtype)
    value = {"NaN": np.nan, "Infinity": np.inf, "-Infinity": -np.inf}.get(fill, fill) if isinstance(fill, str) else fill
    return np.array([value], dtype=dtype)


def shard_index(path: str, n_inner: int, start: bool, crc: bool) -> np.ndarray:
    """(n_inner, 2) uint64 (offset, nbytes) index of a shard file, parsed here as write_v3_array lays it out."""
    raw = open(path, "rb").read()
    size = 16 * n_inner + (4 if crc else 0)
    index = raw[:size] if start else raw[len(raw) - size:]
    return np.frombuffer(index[:16 * n_inner], "<u8").reshape(n_inner, 2)


@dataclass
class Case:
    name: str
    array: np.ndarray
    chunks: tuple                       # chunk shape, or shard shape when `shard` is given
    codecs: tuple = ("bytes",)
    shard: dict | None = None
    key_encoding: dict | None = None
    fill_value: object = 0
    missing: tuple = ()
    attrs: dict = field(default_factory=dict)  # CF attributes: read through DecodedSource
    b0: int = 0
    nb: int = 0
    window: tuple | None = None
    corrupt: object = None
    error: int = 0                      # the reason xrs_zarr_decode must report

    def write(self, root: str) -> str:
        path = os.path.join(root, self.name)
        dims = ("band", "y", "x")[-self.array.ndim:]
        write_v3_array(path, self.array, self.chunks, dims, self.codecs, self.shard, self.key_encoding,
                       self.fill_value, missing=self.missing, corrupt=self.corrupt)
        return path

    def source(self, root: str):
        src = ZarrV3Source(self.write(root))
        return DecodedSource(src, self.attrs) if self.attrs else src

    def read(self):
        bands = 1 if self.array.ndim == 2 else self.array.shape[0]
        window = self.window or (0, self.array.shape[-2])
        return self.b0, self.nb or bands - self.b0, window

    def expected(self, source) -> np.ndarray:
        b0, nb, (j0, j1) = self.read()
        out = np.empty((nb,) + tuple(source.shape[-2:]), dtype=np.dtype(source.dtype).newbyteorder("="))
        source.read_bands(b0, nb, out)
        return out[:, j0:j1]


def _flip(pos: int):
    """corrupt: flip one bit of byte ``pos`` of the file (negative: from its end)."""
    def corrupt(raw):
        raw = bytearray(raw)
        raw[pos] ^= 0x10
        return bytes(raw)
    return corrupt


def cases() -> list[Case]:
    """Stores the device decodes (every compressor chain, sharded and not), then malformed ones."""
    a = _values("float32", (3, 21, 37), seed=31)
    i16 = _values("int16", (3, 21, 37), seed=32)
    out = []
    chains = {
        "zstd": ("bytes", "zstd"),
        "zstd_crc32c": ("bytes", "zstd", "crc32c"),
        "gzip": ("bytes", "gzip"),
        "gzip_crc32c": ("bytes", "gzip", "crc32c"),
        "blosc_lz4": ("bytes", blosc("lz4")),
        "blosc_lz4_crc32c": ("bytes", blosc("lz4"), "crc32c"),
        "blosc_zstd_noshuffle": ("bytes", blosc("zstd", "noshuffle")),
        "blosc_zlib_crc32c": ("bytes", blosc("zlib"), "crc32c"),
        "numcodecs_zlib": ("bytes", "numcodecs.zlib"),
        "numcodecs_lz4_crc32c": ("bytes", "numcodecs.lz4", "crc32c"),
        "numcodecs_zstd": ("bytes", "numcodecs.zstd"),
        "numcodecs_gzip": ("bytes", "numcodecs.gzip"),
        "numcodecs_blosc": ("bytes", {"name": "numcodecs.blosc", "configuration": {"cname": "lz4", "shuffle": 1}}),
        "transpose_identity": ({"name": "transpose", "configuration": {"order": [0, 1, 2]}}, "bytes", "zstd"),
    }
    for name, chain in chains.items():
        out.append(Case(f"v3_{name}", a, (2, 8, 17), chain, fill_value="NaN", missing=((1, 1, 0),), b0=1, nb=2,
                        window=(3, 19)))
    # big-endian bytes codec, 1-byte types without an endian
    out.append(Case("v3_big_endian_f4", a.astype(">f4"), (2, 8, 17), ("bytes", "zstd", "crc32c"), fill_value="NaN"))
    out.append(Case("v3_big_endian_i2", i16.astype(">i2"), (2, 8, 17), ("bytes", blosc("lz4", typesize=2)),
                    fill_value=-7, missing=((0, 1, 1),)))
    out.append(Case("v3_uint8_gzip", _values("uint8", (2, 21, 37), seed=33), (1, 8, 17), ("bytes", "gzip", "crc32c"),
                    fill_value=9, missing=((1, 0, 0),)))
    # sharded: index at the end / start, with and without its CRC-32C; missing inner chunks and shards; ragged shards
    sh = lambda loc, crc: {"chunk_shape": (1, 8, 17), "index_location": loc, "index_crc": crc}  # noqa: E731
    out += [
        Case("shard_end_crc", a, (2, 16, 34), ("bytes", "zstd", "crc32c"), sh("end", True), fill_value="NaN",
             missing=((0, 1, 1), ("shard", 1, 1, 1))),
        Case("shard_start", a, (2, 16, 34), ("bytes", "zstd"), sh("start", False), fill_value="Infinity",
             missing=((2, 0, 0),), b0=1, nb=2, window=(5, 20)),
        Case("shard_start_crc_blosc", a, (2, 16, 34), ("bytes", blosc("lz4"), "crc32c"), sh("start", True),
             fill_value="0x7fc00001", missing=(("shard", 0, 0, 1),)),
        Case("shard_end_gzip", i16, (3, 16, 34), ("bytes", "gzip"), sh("end", False), fill_value=-3,
             missing=((1, 1, 2),)),
        Case("shard_default_location_dot_keys", a, (2, 16, 34), ("bytes", "zstd", "crc32c"),
             {"chunk_shape": (2, 8, 17), "index_crc": True}, key_encoding={"name": "default",
                                                                           "configuration": {"separator": "."}}),
        Case("v2_keys_dot", a, (2, 8, 17), ("bytes", "zstd"), key_encoding={"name": "v2"}, fill_value="-Infinity",
             missing=((0, 0, 0),)),
        Case("v2_keys_slash", a, (2, 8, 17), ("bytes", blosc("lz4"), "crc32c"),
             key_encoding={"name": "v2", "configuration": {"separator": "/"}}),
        Case("cf_shard_uint16", _values("uint16", (3, 21, 37), seed=34), (2, 16, 34),
             ("bytes", "zstd", "crc32c"), {"chunk_shape": (1, 8, 17), "index_crc": True}, fill_value=65535,
             missing=((0, 2, 0),), attrs={"scale_factor": 0.01, "add_offset": -5.0, "_FillValue": 65535,
                                          "missing_value": [3]}),
    ]
    # a flipped bit in the payload and one in the trailer: reason 19 for chunk 0, the first file of the table
    out += [
        Case("bad_crc_payload", a[:1], (1, 8, 17), ("bytes", "zstd", "crc32c"), corrupt=_flip(20),
             error=CRC32C_MISMATCH),
        Case("bad_crc_trailer", a[:1], (1, 8, 17), ("bytes", blosc("lz4"), "crc32c"), corrupt=_flip(-2),
             error=CRC32C_MISMATCH),
        Case("bad_crc_shard_inner", a[:1], (1, 16, 34), ("bytes", "gzip", "crc32c"),
             {"chunk_shape": (1, 8, 17), "index_crc": True}, corrupt=_flip(3), error=CRC32C_MISMATCH),
    ]
    return out
