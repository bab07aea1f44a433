"""The I/O edge: chunked arrays on disk -> page-locked host staging -> H2D, overlapped.

The reference opens Zarr / NetCDF through xarray + dask and lets the dask chunks flow into its tile
tasks.  Here a data variable may be a :class:`LazyDataArray` whose bands live in a chunked store;
the band-chunk pipeline (``_pipeline.GatherPipeline``) then reads band chunk k+1 from the store into
one of two page-locked staging buffers on a reader thread while chunk k is being copied to the
device and chunk k-1 is being gathered -- decode / read, PCIe upload, kernels and download all
overlap, and the host never holds more than two chunks of a variable.

Stores understood without third-party packages:

* :class:`ZarrV2Source` -- a Zarr-v2 array in a directory store (C order, any chunking): what
  ``add_spatial_ref`` (``cfconv.py``) and the reference's Zarr helpers operate on.  Chunks may be
  uncompressed (``"compressor": null``: read straight into the staging buffer) or compressed with a
  codec whose stream format the standard library or pyarrow decodes (numcodecs ids ``zlib``, ``gzip``,
  ``bz2``, ``lzma``, ``zstd``, ``lz4``, and ``blosc`` -- zarr's default -- with an LZ4 / LZ4HC / Snappy /
  Zlib / Zstd inner codec, byte shuffle or none: :func:`blosc_decompress`), decoded on the reader thread.
  BloscLZ or bit-shuffled Blosc frames and Zarr filters need the ``zarr`` / ``numcodecs`` packages, which
  this build does not have; open such stores with xarray and pass the arrays instead.
  Blosc-LZ4 / LZ4HC / Zstd / Zlib stores (byte shuffle or none) and numcodecs ``lz4`` / ``zstd`` / ``zlib`` / ``gzip``
  stores are not decoded on the host in the band pipeline: their chunk files are read as they are
  (:meth:`ZarrV2Source.device_read`), uploaded compressed and decoded, unshuffled and CF-unpacked on the device
  (``xrs_zarr_decode``, ``csrc/decode.cu``).  ``read_bands`` stays the host decode, for ``values`` / ``read_all``
  and every other codec.
* :class:`ZarrV3Source` -- a Zarr v3 array in a directory store (``zarr.json``), sharded (``sharding_indexed``)
  or not, with the ``bytes`` codec (either byte order), at most one compressor (``zstd``, ``gzip``, ``blosc``, or the
  ``numcodecs.<id>`` twin of a :func:`chunk_decoder` codec) and optionally the ``crc32c`` checksum, checked by
  :func:`crc32c` on the host path.  Written from the Zarr v3 core specification and its ``sharding_indexed`` and
  ``crc32c`` codec specifications.  It shares the chunk loops of :class:`ZarrV2Source`; only where a chunk's bytes
  are (a file, or a range of a shard file named by the shard's index) and how they are framed differ.  Stores whose
  compressor the device decodes reach it the same way, one inner chunk at a time, their CRC-32C checked on the
  device.
* :class:`NpySource` -- a ``.npy`` file, memory-mapped.
* :class:`NetCDF3Source` -- a variable of a NetCDF classic / 64-bit-offset file (CDF-1 / CDF-2), memory-mapped
  through ``scipy.io.netcdf_file``; its big-endian values are byte-swapped by the copy into the staging
  buffer.  NetCDF-4 files are HDF5 containers and need ``netCDF4`` / ``h5py``, which this build does not
  have; open them with xarray and pass the arrays instead.

:func:`open_zarr_dataset` / :func:`open_netcdf_dataset` assemble a :class:`~xcube_resampling_b200.dataset.Dataset` from a
directory store (Zarr v2, or a Zarr v3 group): coordinate arrays (1-D, or 2-D named like coordinates) are read eagerly, every
other array becomes a lazy variable.
"""

from __future__ import annotations

import json
import os
from collections.abc import Mapping

import numpy as np

from .dataset import DataArray, Dataset


def _pyarrow_codec(name: str):
    try:
        import pyarrow as pa
    except ImportError as e:  # pragma: no cover - pyarrow is part of the image
        raise NotImplementedError(f"{name}-compressed Zarr chunks need pyarrow (or the zarr package)") from e
    return pa.Codec(name)


def chunk_decoder(compressor: dict | None):
    """``bytes -> bytes`` for a Zarr-v2 ``compressor`` entry (numcodecs configuration), ``None`` for
    uncompressed chunks; ``NotImplementedError`` for codecs this build cannot decode."""
    if compressor is None:
        return None
    cid = compressor.get("id")
    if cid == "zlib":
        import zlib

        return zlib.decompress
    if cid == "gzip":
        import gzip

        return gzip.decompress
    if cid == "bz2":
        import bz2

        return bz2.decompress
    if cid == "lzma":
        import lzma

        fmt, filters = compressor.get("format", lzma.FORMAT_XZ), compressor.get("filters")
        return lambda raw: lzma.decompress(raw, format=fmt, filters=filters)
    if cid == "zstd":
        codec = _pyarrow_codec("zstd")

        def zstd(raw):  # a standard frame; its header carries the decoded size
            size = _zstd_content_size(raw)
            if size is None:
                raise NotImplementedError("zstd frame without a content size")
            return codec.decompress(raw, decompressed_size=size).to_pybytes()

        return zstd
    if cid == "lz4":
        codec = _pyarrow_codec("lz4_raw")

        def lz4(raw):  # numcodecs: little-endian int32 decoded size, then one raw LZ4 block
            size = int.from_bytes(raw[:4], "little", signed=True)
            return codec.decompress(raw[4:], decompressed_size=size).to_pybytes()

        return lz4
    if cid == "blosc":
        return blosc_decompress
    raise NotImplementedError(f"Zarr chunks compressed with {cid!r} need the zarr package, which this build does not "
                              "have; open the store with xarray and pass the arrays instead")


_BLOSC_MAX_SPLITS, _BLOSC_MIN_BUFFERSIZE = 16, 128


def _blosc_stream_decoder(fmt: int):
    """``(bytes, decoded size) -> bytes`` of the inner codec a Blosc-1 frame names in bits 5-7 of its flags."""
    if fmt == 1:  # LZ4 / LZ4HC: one raw LZ4 block per stream
        codec = _pyarrow_codec("lz4_raw")
        return lambda raw, n: codec.decompress(raw, decompressed_size=n).to_pybytes()
    if fmt == 2:
        codec = _pyarrow_codec("snappy")
        return lambda raw, n: codec.decompress(raw, decompressed_size=n).to_pybytes()
    if fmt == 3:
        import zlib

        return lambda raw, n: zlib.decompress(raw)
    if fmt == 4:
        codec = _pyarrow_codec("zstd")
        return lambda raw, n: codec.decompress(raw, decompressed_size=n).to_pybytes()
    raise NotImplementedError("Blosc frames compressed with BloscLZ need the zarr / blosc packages, which this build "
                              "does not have (lz4, lz4hc, snappy, zlib and zstd frames are decoded)")


def blosc_decompress(frame: bytes) -> bytes:
    """Decode one Blosc-1 frame (what numcodecs' ``Blosc`` -- zarr-v2's default compressor -- writes per chunk),
    following the container layout c-blosc publishes (README_HEADER.rst, ``blosc_d`` in blosc.c):

    * 16-byte header: version, versionlz, flags, typesize, then little-endian uint32 ``nbytes`` (decoded size),
      ``blocksize``, ``cbytes`` (size of the whole frame).  Flags: bit 0 byte shuffle, bit 1 the payload is a
      plain copy, bit 2 bit shuffle, bit 4 blocks are not split, bits 5-7 the inner codec
      (0 BloscLZ, 1 LZ4 / LZ4HC, 2 Snappy, 3 Zlib, 4 Zstd).
    * ``ceil(nbytes / blocksize)`` int32 block offsets (from the start of the frame), then the blocks.  A block
      is ``typesize`` streams (one per byte position of the shuffled block) when splitting applies -- not the
      last, partial block; ``typesize <= 16``; at least 128 bytes per stream -- else one stream.  A stream is an
      int32 compressed size followed by the data, stored verbatim when that size equals the decoded size.
    * byte shuffle within a block of ``n`` elements: byte ``j`` of element ``i`` sits at ``j * n + i``; the
      ``blocksize % typesize`` trailing bytes are not shuffled.

    The inner codecs come from the standard library / pyarrow; there is no Blosc library in this image, so
    the tests assemble their frames by hand from this description.  Bit-shuffled frames and BloscLZ raise
    ``NotImplementedError``."""
    if len(frame) < 16:
        raise ValueError("not a Blosc frame: shorter than its 16-byte header")
    version, _, flags, typesize = frame[0], frame[1], frame[2], frame[3]
    nbytes, blocksize, cbytes = (int.from_bytes(frame[k:k + 4], "little") for k in (4, 8, 12))
    if version != 2 or cbytes > len(frame) or (nbytes and blocksize == 0):
        raise ValueError(f"not a Blosc-1 frame (version {version}, cbytes {cbytes} of {len(frame)} bytes)")
    if nbytes == 0:
        return b""
    if flags & 0x2:  # stored
        if 16 + nbytes > len(frame):
            raise ValueError("truncated Blosc frame")
        return bytes(frame[16:16 + nbytes])
    if flags & 0x4:
        raise NotImplementedError("bit-shuffled Blosc frames need the zarr / blosc packages, which this build does "
                                  "not have")
    decode = _blosc_stream_decoder(flags >> 5)
    typesize = max(typesize, 1)
    shuffled = bool(flags & 0x1) and typesize > 1
    nblocks = -(-nbytes // blocksize)
    starts = np.frombuffer(frame, dtype="<i4", count=nblocks, offset=16)
    out = np.empty(nbytes, dtype=np.uint8)
    for b in range(nblocks):
        bsize = min(blocksize, nbytes - b * blocksize)
        leftover = bsize != blocksize
        split = (not flags & 0x10 and typesize <= _BLOSC_MAX_SPLITS
                 and blocksize // typesize >= _BLOSC_MIN_BUFFERSIZE and not leftover)
        nstreams = typesize if split else 1
        neblock = bsize // nstreams
        pos, parts = int(starts[b]), []
        for _ in range(nstreams):
            if pos < 16 or pos + 4 > len(frame):
                raise ValueError("corrupt Blosc frame: stream outside the frame")
            csize = int.from_bytes(frame[pos:pos + 4], "little", signed=True)
            pos += 4
            if csize < 0 or pos + csize > len(frame):
                raise ValueError("corrupt Blosc frame: stream outside the frame")
            raw = frame[pos:pos + csize]
            pos += csize
            part = bytes(raw) if csize == neblock else decode(raw, neblock)
            if len(part) != neblock:
                raise ValueError("corrupt Blosc frame: stream decodes to the wrong size")
            parts.append(part)
        block = np.frombuffer(b"".join(parts), dtype=np.uint8)
        dst = out[b * blocksize:b * blocksize + bsize]
        if shuffled:
            n = bsize // typesize
            dst[:n * typesize] = block[:n * typesize].reshape(typesize, n).T.reshape(-1)
            dst[n * typesize:] = block[n * typesize:]
        else:
            dst[:] = block
    return out.tobytes()


def _zstd_content_size(raw: bytes) -> int | None:
    """Frame_Content_Size of a zstd frame header (RFC 8878, 3.1.1.1), ``None`` if the frame omits it."""
    if len(raw) < 6 or raw[:4] != b"\x28\xb5\x2f\xfd":
        raise ValueError("not a zstd frame")
    desc = raw[4]
    fcs_flag, single_segment, dict_flag = desc >> 6, (desc >> 5) & 1, desc & 3
    pos = 5 + (0 if single_segment else 1) + (0, 1, 2, 4)[dict_flag]
    n = (1 if single_segment else 0, 2, 4, 8)[fcs_flag]
    if n == 0:
        return None
    value = int.from_bytes(raw[pos:pos + n], "little")
    return value + 256 if n == 2 else value


_CRC32C_POLY = 0x82F63B78  # CRC-32C (Castagnoli), reflected
_CRC_SEGMENT = 64  # bytes of one segment of crc32c's vectorised pass


def _crc_mul(a: int, b, poly: int = _CRC32C_POLY):
    """``a * b`` modulo the reflected polynomial ``poly`` (bit 31 is x^0; zlib's multmodp); ``b`` may be a uint32
    array, multiplied element by element."""
    p = b ^ b
    for k in range(32):
        if a & (0x80000000 >> k):
            p = p ^ b
        b = (b >> 1) ^ ((b & 1) * poly)
    return p


def _crc_shift(n: int, poly: int = _CRC32C_POLY) -> int:
    """x^(8n) modulo ``poly``: the operator that runs a CRC register over ``n`` zero bytes (zlib's x2nmodp)."""
    p, x = 0x80000000, 0x00800000  # x^0, x^8
    while n:
        if n & 1:
            p = _crc_mul(x, p, poly)
        x = _crc_mul(x, x, poly)
        n >>= 1
    return p


_crc32c_tables: dict = {}


def _crc32c_table(shift_bytes: int) -> np.ndarray:
    """(4, 256) uint32: row k maps byte v to x^(8 * shift_bytes) * (v << 8k), so that a register ``c`` run over
    ``shift_bytes`` zero bytes is the XOR of ``table[k][(c >> 8k) & 255]``; ``shift_bytes`` 0 gives the byte table of
    CRC-32C itself (register ``c`` over one byte ``v`` is ``table0[(c ^ v) & 255] ^ (c >> 8)``)."""
    if shift_bytes not in _crc32c_tables:
        v = np.arange(256, dtype=np.uint32)
        if shift_bytes == 0:
            for _ in range(8):
                v = (v >> 1) ^ ((v & 1) * np.uint32(_CRC32C_POLY))
            _crc32c_tables[0] = v
        else:
            by = (v[None, :] << (8 * np.arange(4, dtype=np.uint32))[:, None]).astype(np.uint32)
            _crc32c_tables[shift_bytes] = _crc_mul(_crc_shift(shift_bytes), by).astype(np.uint32)
    return _crc32c_tables[shift_bytes]


def crc32c(data) -> int:
    """CRC-32C (Castagnoli, reflected polynomial 0x82F63B78, init and final XOR 0xFFFFFFFF) of ``data`` -- the
    checksum of Zarr v3's ``crc32c`` codec and of its shard indexes.

    The bytes are cut into segments of 64 bytes that are run through the byte table side by side (one numpy step per
    byte position, over all segments at once); the segment registers are then combined pairwise, level by level,
    with the GF(2) shift ``x^(8 * 64 * 2^level)`` (the linearity crc32_combine uses), and the tail of fewer than 64
    bytes runs through the table last.  No Python loop runs per byte of the bulk."""
    buf = np.frombuffer(memoryview(data).cast("B"), dtype=np.uint8)
    n_seg = len(buf) // _CRC_SEGMENT
    table = _crc32c_table(0)
    reg = np.uint32(0xFFFFFFFF)
    if n_seg:
        levels = max(n_seg - 1, 0).bit_length()
        # leading zero segments are free: with a zero register they leave it zero
        segs = np.zeros((1 << levels, _CRC_SEGMENT), np.uint8)
        segs[(1 << levels) - n_seg:] = buf[:n_seg * _CRC_SEGMENT].reshape(n_seg, _CRC_SEGMENT)
        cols = np.ascontiguousarray(segs.T)
        c = np.zeros(1 << levels, np.uint32)
        c[(1 << levels) - n_seg] = reg
        for col in cols:
            c = table[(c ^ col) & 0xFF] ^ (c >> 8)
        for level in range(levels):
            t = _crc32c_table(_CRC_SEGMENT << level)
            a, b = c[0::2], c[1::2]
            c = t[0][a & 0xFF] ^ t[1][(a >> 8) & 0xFF] ^ t[2][(a >> 16) & 0xFF] ^ t[3][a >> 24] ^ b
        reg = c[0]
    reg = int(reg)
    for v in buf[n_seg * _CRC_SEGMENT:].tolist():
        reg = int(table[(reg ^ v) & 0xFF]) ^ (reg >> 8)
    return reg ^ 0xFFFFFFFF


def _check_crc32c(raw, where: str) -> memoryview:
    """The payload of a chunk that ends in the crc32c codec's 4-byte little-endian CRC-32C; ``ValueError`` naming
    ``where`` when the file is too short or the checksum does not match."""
    raw = memoryview(raw)
    if len(raw) < 4:
        raise ValueError(f"{where}: shorter than its 4-byte CRC-32C")
    if crc32c(raw[:-4]) != int.from_bytes(raw[-4:], "little"):
        raise ValueError(f"{where}: CRC-32C mismatch")
    return raw[:-4]


class LazySource:
    """A (bands, h, w) or (h, w) array that can deliver whole bands into a caller's buffer."""

    shape: tuple
    dtype: np.dtype

    def read_bands(self, b0: int, nb: int, out: np.ndarray) -> None:  # pragma: no cover - interface
        """Fill ``out[:nb]`` (shape (>= nb, h, w), C-contiguous rows) with bands ``b0 : b0 + nb``."""
        raise NotImplementedError

    @property
    def ndim(self) -> int:
        return len(self.shape)

    @property
    def nbytes(self) -> int:
        return int(np.prod(self.shape)) * np.dtype(self.dtype).itemsize

    def read_all(self) -> np.ndarray:
        bands = 1 if len(self.shape) == 2 else self.shape[0]
        out = np.empty((bands,) + tuple(self.shape[-2:]), dtype=self.dtype)
        self.read_bands(0, bands, out)
        return out[0] if len(self.shape) == 2 else out


class NpySource(LazySource):
    """A ``.npy`` file read through a memory map."""

    def __init__(self, path: str):
        self._mm = np.load(path, mmap_mode="r")
        if self._mm.ndim not in (2, 3):
            raise ValueError(f"{path}: expected a 2-D or 3-D array, got {self._mm.ndim} dimensions")
        self.shape, self.dtype = tuple(self._mm.shape), self._mm.dtype

    def read_bands(self, b0, nb, out):
        src = self._mm[None] if self._mm.ndim == 2 else self._mm
        out[:nb] = src[b0:b0 + nb]


class NetCDF3Source(LazySource):
    """One 2-D or 3-D variable of an open ``scipy.io.netcdf_file`` (``mmap=True``).  The file object is kept
    alive by the source; values are delivered as stored, in native byte order."""

    def __init__(self, nc_file, name: str):
        self._file = nc_file  # owns the memory map the variable's data points into
        self._var = nc_file.variables[name]
        if len(self._var.shape) not in (2, 3):
            raise ValueError(f"{name}: expected a 2-D or 3-D variable, got shape {self._var.shape}")
        self.shape = tuple(int(n) for n in self._var.shape)
        self.dtype = self._var.data.dtype.newbyteorder("=")

    def read_bands(self, b0, nb, out):
        data = self._var.data
        out[:nb] = (data[None] if data.ndim == 2 else data)[b0:b0 + nb]


# one chunk file of a device read: ``struct xrs_zarr_chunk`` of include/xrs.h
CHUNK_TABLE_DTYPE = np.dtype([("offset", "<i8"), ("length", "<i8"), ("band", "<i8"), ("row", "<i8"), ("col", "<i8"),
                              ("codec", "<i4"), ("n_streams", "<i4"), ("stream_base", "<i8"), ("scratch", "<i8"),
                              ("header", "u1", 16)])
assert CHUNK_TABLE_DTYPE.itemsize == 80
CHUNK_MISSING, CHUNK_BLOSC, CHUNK_LZ4, CHUNK_ZSTD, CHUNK_ZLIB, CHUNK_GZIP = 0, 1, 2, 3, 4, 5  # enum xrs_chunk_codec
CHUNK_CRC32C = 0x100  # flag: the file ends in a CRC-32C of its payload
_BLOSC_INNER = {"lz4": 1, "lz4hc": 1, "zlib": 3, "zstd": 4}  # Blosc flags bits 5-7 of a store's cname
_BLOSC_INNER_NAMES = {1: "LZ4", 3: "Zlib", 4: "Zstd"}
_NUMCODECS_DEVICE = {"lz4": CHUNK_LZ4, "zstd": CHUNK_ZSTD, "zlib": CHUNK_ZLIB, "gzip": CHUNK_GZIP}
_ZSTD_HEADER_MAX = 18  # magic, descriptor, window, dictionary ID (4), content size (8)
_GZIP_MIN = 19  # a gzip member's 10-byte header, one byte of Deflate, CRC-32 and ISIZE


def _device_codec(compressor: dict | None) -> int | None:
    """The codec of ``xrs_zarr_decode`` a ``.zarray`` compressor maps to, ``None`` when chunks decode on the host."""
    if not compressor:
        return None
    if compressor.get("id") in _NUMCODECS_DEVICE:
        return _NUMCODECS_DEVICE[compressor["id"]]
    if compressor.get("id") == "blosc" and compressor.get("cname") in _BLOSC_INNER and \
            compressor.get("shuffle", 1) in (0, 1):
        return CHUNK_BLOSC
    return None


def _check_device_header(path: str, codec: int, head: bytes, size: int, chunk_bytes: int, inner: int = 1) -> None:
    """The checks :func:`blosc_decompress` / the numcodecs lz4, zstd, zlib and gzip decoders make before decoding, on
    a file's header only, with the same errors; the device decode checks the streams.  ``inner``: the Blosc inner
    codec the store's ``cname`` names (1 LZ4, 3 Zlib, 4 Zstd); ``head``: the first 16 bytes of the file, 18 for
    zstd, 19 for gzip."""
    if codec == CHUNK_LZ4:
        if size < 4 or int.from_bytes(head[:4], "little", signed=True) != chunk_bytes:
            raise ValueError(f"{path}: the lz4 chunk's size prefix does not match the chunk size {chunk_bytes}")
        return
    if codec == CHUNK_ZSTD:
        content = _zstd_content_size(head)
        if content is None:
            raise NotImplementedError("zstd frame without a content size")
        if content != chunk_bytes:
            raise ValueError(f"{path}: the zstd frame holds {content} bytes, the chunk {chunk_bytes}")
        return
    if codec in (CHUNK_ZLIB, CHUNK_GZIP):
        name = "zlib" if codec == CHUNK_ZLIB else "gzip"
        if codec == CHUNK_ZLIB:  # CMF, FLG without FDICT, and room for one byte of Deflate and the Adler-32
            ok = size >= 7 and (head[0] & 15) == 8 and head[0] >> 4 <= 7 and (head[0] * 256 + head[1]) % 31 == 0 \
                and not head[1] & 0x20
        else:  # magic and method 8, and room for one byte of Deflate, the CRC-32 and ISIZE
            ok = size >= 19 and bytes(head[:3]) == b"\x1f\x8b\x08"
        if not ok:  # the host decoder's own error for the file's start (all of it, when the file is that short)
            chunk_decoder({"id": name})(bytes(head))
            raise ValueError(f"{path}: a {name} chunk file of {size} bytes does not decode to {chunk_bytes} bytes")
        return
    if size < 16:
        raise ValueError(f"{path}: not a Blosc frame: shorter than its 16-byte header")
    version, flags = head[0], head[2]
    nbytes, blocksize, cbytes = (int.from_bytes(head[k:k + 4], "little") for k in (4, 8, 12))
    if version != 2 or cbytes > size or (nbytes and blocksize == 0):
        raise ValueError(f"{path}: not a Blosc-1 frame (version {version}, cbytes {cbytes} of {size} bytes)")
    if nbytes != chunk_bytes:
        raise ValueError(f"{path}: the Blosc frame holds {nbytes} bytes, the chunk {chunk_bytes}")
    if flags & 0x2:
        if 16 + nbytes > size:
            raise ValueError(f"{path}: truncated Blosc frame")
        return
    if flags & 0x4:
        raise NotImplementedError("bit-shuffled Blosc frames need the zarr / blosc packages, which this build does "
                                  "not have")
    if flags >> 5 != inner:
        _blosc_stream_decoder(flags >> 5)  # BloscLZ: the host path's error
        raise ValueError(f"{path}: the Blosc frame's inner codec ({flags >> 5}) is not the store's "
                         f"{_BLOSC_INNER_NAMES[inner]}")


class _ZarrSource(LazySource):
    """What Zarr v2 and v3 arrays share: the loops of :meth:`read_bands` and :meth:`device_read` over the chunk grid.
    A subclass says where the bytes of one chunk are and how they are framed (:meth:`_locate`, :meth:`_payload`) and
    sets ``path``, ``shape``, ``chunks`` (the unit of decoding), ``dtype``, ``device_codec``, ``_device_inner`` and
    ``_fill`` (the value of a missing chunk)."""

    _crc = False  # chunk files end in a CRC-32C of the bytes in front of it (Zarr v3's crc32c codec)

    def _locate(self, idx) -> tuple[str, str, int, int] | None:  # pragma: no cover - interface
        """(file, name for messages, offset, size) of chunk ``idx``'s bytes; ``None`` for a missing chunk."""
        raise NotImplementedError

    def _payload(self, raw, where: str) -> bytes:  # pragma: no cover - interface
        """The decoded bytes of a chunk file ``raw``."""
        raise NotImplementedError

    @property
    def device_decodable(self) -> bool:
        """Whether :meth:`device_read` applies: the store's compressor is one ``xrs_zarr_decode`` decodes."""
        return self.device_codec is not None

    def device_fill_bits(self) -> int:
        """The stored value of a missing chunk (what :meth:`_chunk` fills in), native byte order, as an integer."""
        v = np.full(1, self._fill, dtype=self.dtype.newbyteorder("="))
        return int.from_bytes(v.tobytes(), "little")

    def device_read(self, b0: int, nb: int, segments, window, buffer=None):
        """The chunk files behind bands ``b0 : b0 + nb`` of the (j0, j1, i0, i1) ``segments`` inside the row
        ``window``, read as they are on disk into a page-locked byte buffer, followed by their chunk table
        (:data:`CHUNK_TABLE_DTYPE`).  Only each file's header is checked here.  ``buffer`` (the previous
        result's) is reused when it is large enough.  Returns ``(buffer, n_file_bytes, table, paths)``."""
        from . import _dev

        three_d = len(self.shape) == 3
        cb = self.chunks[0] if three_d else 1
        ch, cw = self.chunks[-2:]
        chunk_bytes = int(np.prod(self.chunks)) * self.dtype.itemsize
        tiles = set()
        for (j0, j1, i0, i1) in segments:
            j0, j1 = max(j0, window[0]), min(j1, window[1])
            if j0 >= j1 or i0 >= i1:
                continue
            tiles.update((kj, ki) for kj in range(j0 // ch, -(-j1 // ch)) for ki in range(i0 // cw, -(-i1 // cw)))
        keys = [(kb, kj, ki) for kb in range(b0 // cb, -(-(b0 + nb) // cb)) for (kj, ki) in sorted(tiles)]
        locs = [self._locate((kb, kj, ki) if three_d else (kj, ki)) for (kb, kj, ki) in keys]
        paths = [loc[1] if loc else self._missing_name((kb, kj, ki) if three_d else (kj, ki))
                 for (kb, kj, ki), loc in zip(keys, locs)]
        n_bytes = sum(loc[3] for loc in locs if loc)
        table_at = -(-n_bytes // 8) * 8
        need = table_at + len(keys) * CHUNK_TABLE_DTYPE.itemsize
        if buffer is None or buffer.nbytes < need:
            buffer = _dev.pinned_empty((max(need, 1 << 20) + (need >> 3),), np.uint8)  # an eighth to grow into
        table = buffer[table_at:need].view(CHUNK_TABLE_DTYPE)
        table[...] = 0
        pos = 0
        trailer = 4 if self._crc else 0
        for k, ((kb, kj, ki), loc, p) in enumerate(zip(keys, locs, paths)):
            t = table[k]
            t["band"], t["row"], t["col"] = kb * cb, kj * ch, ki * cw
            if loc is None:  # a missing chunk is all fill value
                t["codec"] = CHUNK_MISSING
                continue
            file, _, offset, size = loc
            with open(file, "rb") as fh:
                fh.seek(offset)
                got = fh.readinto(memoryview(buffer[pos:pos + size]))
            if got != size:
                raise ValueError(f"{p}: short read ({got} of {size} bytes)")
            if size < trailer:
                raise ValueError(f"{p}: shorter than its 4-byte CRC-32C")
            n_head = {CHUNK_ZSTD: _ZSTD_HEADER_MAX, CHUNK_GZIP: _GZIP_MIN}.get(self.device_codec, 16)
            head = buffer[pos:pos + min(size - trailer, n_head)].tobytes()  # of the payload: the trailer excluded
            _check_device_header(p, self.device_codec, head, size - trailer, chunk_bytes, self._device_inner)
            t["offset"], t["length"] = pos, size
            t["codec"] = self.device_codec | (CHUNK_CRC32C if self._crc else 0)
            t["header"][:min(len(head), 16)] = np.frombuffer(head[:16], np.uint8)
            pos += size
        return buffer, n_bytes, table, paths

    def _missing_name(self, idx) -> str:  # pragma: no cover - interface
        """Where chunk ``idx`` would be, for messages about a table that lists it as missing."""
        raise NotImplementedError

    def _chunk(self, idx):
        loc = self._locate(idx)
        if loc is None:  # a missing chunk is all fill value
            return np.full(self.chunks, self._fill, dtype=self.dtype)
        file, where, offset, size = loc
        with open(file, "rb") as fh:
            fh.seek(offset)
            raw = fh.read(size)
        if len(raw) != size:
            raise ValueError(f"{where}: short read ({len(raw)} of {size} bytes)")
        return np.frombuffer(self._payload(raw, where), dtype=self.dtype).reshape(self.chunks)

    def read_bands(self, b0, nb, out):
        three_d = len(self.shape) == 3
        cb = self.chunks[0] if three_d else 1
        ch, cw = self.chunks[-2:]
        h, w = self.shape[-2:]
        for kb in range(b0 // cb, -(-(b0 + nb) // cb)):
            lo, hi = max(b0, kb * cb), min(b0 + nb, (kb + 1) * cb)
            for kj in range(-(-h // ch)):
                for ki in range(-(-w // cw)):
                    block = self._chunk((kb, kj, ki) if three_d else (kj, ki))
                    if not three_d:
                        block = block[None]
                    j0, i0 = kj * ch, ki * cw
                    j1, i1 = min(h, j0 + ch), min(w, i0 + cw)
                    out[lo - b0:hi - b0, j0:j1, i0:i1] = block[lo - kb * cb:hi - kb * cb, :j1 - j0, :i1 - i0]


class ZarrV2Source(_ZarrSource):
    """One Zarr-v2 array of a directory store (2-D or 3-D, C order; uncompressed or with a codec of
    :func:`chunk_decoder`).  Blosc-LZ4 / LZ4HC / Zstd / Zlib (byte shuffle or none) and numcodecs ``lz4`` / ``zstd`` /
    ``zlib`` / ``gzip`` stores can also be read for the device (:meth:`device_read`): the band pipeline then decodes
    the chunks there."""

    def __init__(self, path: str):
        meta = json.load(open(os.path.join(path, ".zarray")))
        if meta.get("zarr_format") != 2:
            raise ValueError(f"{path}: not a Zarr v2 array")
        if meta.get("filters"):
            raise NotImplementedError(f"{path}: filtered Zarr arrays need the zarr package, which this "
                                      "build does not have; open the store with xarray and pass the arrays instead")
        try:
            self._decode = chunk_decoder(meta.get("compressor"))
        except NotImplementedError as e:
            raise NotImplementedError(f"{path}: {e}") from None
        if meta.get("order", "C") != "C":
            raise NotImplementedError(f"{path}: only C-order chunks are supported")
        self.path = path
        self.shape = tuple(int(n) for n in meta["shape"])
        if len(self.shape) not in (2, 3):
            raise ValueError(f"{path}: expected a 2-D or 3-D array, got shape {self.shape}")
        self.chunks = tuple(int(n) for n in meta["chunks"])
        self.dtype = np.dtype(meta["dtype"])
        self.fill = meta.get("fill_value")
        self._fill = _fill_value(self.fill, self.dtype)
        self.sep = meta.get("dimension_separator", ".")
        attrs_path = os.path.join(path, ".zattrs")
        self.attrs = json.load(open(attrs_path)) if os.path.isfile(attrs_path) else {}
        self.device_codec = _device_codec(meta.get("compressor"))
        self._device_inner = _BLOSC_INNER.get((meta.get("compressor") or {}).get("cname"), 1)

    def _locate(self, idx):
        p = os.path.join(self.path, self.sep.join(str(i) for i in idx))
        return (p, p, 0, os.path.getsize(p)) if os.path.isfile(p) else None

    def _missing_name(self, idx):
        return os.path.join(self.path, self.sep.join(str(i) for i in idx))

    def _payload(self, raw, where):
        return raw if self._decode is None else self._decode(raw)


_V3_TYPES = ("bool", "int8", "int16", "int32", "int64", "uint8", "uint16", "uint32", "uint64", "float16", "float32",
             "float64", "complex64", "complex128")
_V3_SHUFFLE = {"noshuffle": 0, "shuffle": 1}
_MISSING = 2 ** 64 - 1  # offset and size of an inner chunk a shard does not hold


def _v3_codec(entry) -> tuple[str, dict]:
    """(name, configuration) of one entry of a v3 ``codecs`` list (a bare name stands for no configuration)."""
    if isinstance(entry, str):
        return entry, {}
    return entry.get("name"), dict(entry.get("configuration") or {})


def _v3_compressor(name: str, conf: dict) -> dict:
    """The numcodecs configuration (what :func:`chunk_decoder` / :func:`_device_codec` take) of a v3 bytes -> bytes
    compressor."""
    if name == "zstd":
        return {"id": "zstd", "level": conf.get("level", 0)}
    if name == "gzip":
        return {"id": "gzip", "level": conf.get("level", 5)}
    if name == "blosc":
        shuffle = conf.get("shuffle", "noshuffle")
        if shuffle == "bitshuffle":
            raise NotImplementedError("bit-shuffled Blosc frames need the zarr / blosc packages, which this build "
                                      "does not have")
        if shuffle not in _V3_SHUFFLE:
            raise ValueError(f"unknown Blosc shuffle {shuffle!r}")
        return {"id": "blosc", "cname": conf.get("cname", "lz4"), "clevel": conf.get("clevel", 5),
                "shuffle": _V3_SHUFFLE[shuffle], "typesize": conf.get("typesize"), "blocksize": conf.get("blocksize", 0)}
    if name.startswith("numcodecs.") and name[10:] in ("zlib", "gzip", "bz2", "lzma", "zstd", "lz4", "blosc"):
        return dict(conf, id=name[10:])
    if name in ("bitshuffle", "numcodecs.bitshuffle"):
        raise NotImplementedError("bit-shuffled chunks need the zarr / numcodecs packages, which this build does not "
                                  "have; open the store with xarray and pass the arrays instead")
    raise NotImplementedError(f"Zarr v3 codec {name!r} needs the zarr package, which this build does not have; open "
                              "the store with xarray and pass the arrays instead")


def _v3_chain(codecs, data_type: str, ndim: int, nested: bool = False) -> dict:
    """The rules of a v3 codec chain this build reads: an identity ``transpose`` at most, exactly one array -> bytes
    codec (``bytes``, or ``sharding_indexed`` when not ``nested``), then at most one compressor, then ``crc32c``.
    Returns ``{"endian", "compressor", "crc", "sharding"}``."""
    out = {"endian": None, "compressor": None, "crc": False, "sharding": None}
    stage = 0  # 0 before the array -> bytes codec, 1 after it, 2 after the compressor, 3 after crc32c
    for entry in codecs or ():
        name, conf = _v3_codec(entry)
        if name == "transpose" and stage == 0:
            if list(conf.get("order", ())) != list(range(ndim)):
                raise NotImplementedError(f"a transpose codec of order {conf.get('order')} (only the identity order "
                                          "is read)")
        elif name in ("bytes", "sharding_indexed") and stage == 0:
            if name == "sharding_indexed":
                if nested:
                    raise NotImplementedError("nested sharding_indexed codecs are not read")
                out["sharding"] = conf
            else:
                endian = conf.get("endian")
                if endian is None and np.dtype(data_type).itemsize > 1:
                    raise ValueError(f"the bytes codec of a {data_type} array needs an endian")
                if endian not in (None, "little", "big"):
                    raise ValueError(f"unknown endian {endian!r} of the bytes codec")
                out["endian"] = endian
            stage = 1
        elif name == "crc32c" and stage in (1, 2):
            out["crc"] = True
            stage = 3
        elif stage == 1 and name not in ("transpose", "bytes", "sharding_indexed", "crc32c", "vlen-utf8",
                                         "vlen-bytes"):
            out["compressor"] = _v3_compressor(name, conf)
            stage = 2
        elif stage == 0 and name not in ("bytes", "sharding_indexed", "transpose"):
            raise NotImplementedError(f"array -> array codec {name!r} (only an identity transpose is read)")
        else:
            raise NotImplementedError(f"codec {name!r} at this place of the chain (read: [transpose], bytes or "
                                      "sharding_indexed, [one compressor], [crc32c])")
    if stage == 0:
        raise ValueError("the codec chain has no array -> bytes codec")
    if out["sharding"] is not None and stage != 1:
        raise NotImplementedError("codecs after sharding_indexed are not read")
    return out


def _v3_fill(fill, dtype: np.dtype):
    """The value of a v3 ``fill_value``: a number, ``"NaN"`` / ``"Infinity"`` / ``"-Infinity"``, or ``"0x..."`` -- a
    float's raw bits."""
    if isinstance(fill, str) and fill.startswith("0x"):
        bits = np.array([int(fill, 16)], dtype=f"u{dtype.itemsize}")
        return bits.view(dtype.newbyteorder("="))[0]
    if isinstance(fill, str):
        special = {"NaN": np.nan, "Infinity": np.inf, "-Infinity": -np.inf}
        if fill not in special:
            raise ValueError(f"unknown fill_value {fill!r}")
        return dtype.newbyteorder("=").type(special[fill])
    if isinstance(fill, list) and dtype.kind == "c":
        return dtype.newbyteorder("=").type(complex(_v3_fill(fill[0], np.dtype("f8")), _v3_fill(fill[1], np.dtype("f8"))))
    return dtype.newbyteorder("=").type(0 if fill is None else fill)


def _v3_key(encoding, idx) -> str:
    """The key of chunk ``idx`` under a v3 ``chunk_key_encoding`` (``default``: ``c/1/2`` or ``c.1.2``, ``c`` for a
    0-D array; ``v2``: ``1.2``, ``0`` for a 0-D array), as a relative path."""
    name, conf = _v3_codec(encoding or {"name": "default"})
    if name == "default":
        sep = conf.get("separator", "/")
        key = sep.join(["c"] + [str(i) for i in idx])
    elif name == "v2":
        sep = conf.get("separator", ".")
        key = sep.join(str(i) for i in idx) if idx else "0"
    else:
        raise NotImplementedError(f"chunk_key_encoding {name!r}")
    if sep not in ("/", "."):
        raise ValueError(f"chunk key separator {sep!r}")
    return key.replace("/", os.sep)


def _v3_meta(path: str) -> dict:
    meta = json.load(open(os.path.join(path, "zarr.json")))
    if meta.get("zarr_format") != 3 or meta.get("node_type") != "array":
        raise ValueError(f"{path}: not a Zarr v3 array")
    return meta


def v3_dimension_names(meta: dict) -> list:
    """``dimension_names``, else ``attributes._ARRAY_DIMENSIONS``, else ``dim_k``; a null name becomes ``dim_k``."""
    names = meta.get("dimension_names") or (meta.get("attributes") or {}).get("_ARRAY_DIMENSIONS")
    ndim = len(meta["shape"])
    if not names or len(names) != ndim:
        names = [None] * ndim
    return [n if n is not None else f"dim_{k}" for k, n in enumerate(names)]


class _ZarrV3Array(_ZarrSource):
    """A Zarr v3 array of a directory store of any rank (:class:`ZarrV3Source` is the 2-D / 3-D lazy source).
    Written from the Zarr v3 core specification and its ``sharding_indexed`` and ``crc32c`` codec specifications.

    * ``zarr.json``: ``shape``, a ``regular`` chunk grid, a numeric ``data_type``, ``fill_value``,
      ``chunk_key_encoding`` (``default`` or ``v2``), ``attributes``, ``dimension_names``; no storage transformers.
    * Codecs (:func:`_v3_chain`): [identity ``transpose``], ``bytes`` (its ``endian`` sets the byte order), at most one
      compressor (``zstd``, ``gzip``, ``blosc`` or ``numcodecs.<id>`` of :func:`chunk_decoder`), [``crc32c``].
    * ``sharding_indexed`` (not nested): a shard file holds inner chunks (``chunk_shape``, inner ``codecs``) and an
      index of one little-endian uint64 (offset, nbytes) pair per inner chunk in C order, (2^64 - 1, 2^64 - 1) for
      an absent one, at the ``end`` (default) or ``start`` of the file and optionally followed by its CRC-32C.  The
      index of each shard is read once, with one ranged read, and kept; inner chunks are read with ranged reads.
      A missing shard file is all fill value.

    ``chunks`` is the unit of decoding: the inner chunk of a sharded array."""

    def __init__(self, path: str):
        meta = _v3_meta(path)
        self.path = path
        self.shape = tuple(int(n) for n in meta["shape"])
        grid_name, grid = _v3_codec(meta.get("chunk_grid") or {})
        if grid_name != "regular":
            raise NotImplementedError(f"{path}: chunk grid {grid_name!r} (only regular grids are read)")
        outer = tuple(int(n) for n in grid["chunk_shape"])
        data_type = meta.get("data_type")
        if data_type not in _V3_TYPES:
            raise NotImplementedError(f"{path}: Zarr v3 data type {data_type!r} is not read (numeric types only)")
        if meta.get("storage_transformers"):
            raise NotImplementedError(f"{path}: storage transformers are not read")
        self._encoding = meta.get("chunk_key_encoding")
        self.attrs = dict(meta.get("attributes") or {})
        self.dimension_names = v3_dimension_names(meta)
        try:
            _v3_key(self._encoding, (0,) * len(self.shape))
            chain = _v3_chain(meta.get("codecs"), data_type, len(self.shape))
            self._shard = None
            if chain["sharding"] is not None:
                conf = chain["sharding"]
                inner = tuple(int(n) for n in conf["chunk_shape"])
                if len(inner) != len(outer) or any(o % i for o, i in zip(outer, inner)):
                    raise ValueError(f"inner chunks {inner} do not tile the shard {outer}")
                index = _v3_chain(conf.get("index_codecs"), "uint64", len(outer) + 1, nested=True)
                if index["compressor"] is not None or index["endian"] not in ("little", None):
                    raise NotImplementedError("a shard index other than little-endian bytes [+ crc32c]")
                location = conf.get("index_location", "end")
                if location not in ("start", "end"):
                    raise ValueError(f"unknown index_location {location!r}")
                per = tuple(o // i for o, i in zip(outer, inner))
                n_inner = int(np.prod(per, dtype=np.int64))
                self._shard = {"per": per, "n": n_inner, "start": location == "start",
                               "index_bytes": 16 * n_inner + (4 if index["crc"] else 0), "index_crc": index["crc"]}
                self._indexes: dict = {}
                chain = _v3_chain(conf.get("codecs"), data_type, len(outer), nested=True)
                self.chunks = inner
            else:
                self.chunks = outer
            self._decode = chunk_decoder(chain["compressor"])
            dtype = np.dtype(data_type)
            self.dtype = dtype.newbyteorder(">" if chain["endian"] == "big" else "<") if dtype.itemsize > 1 else dtype
            self._fill = _v3_fill(meta.get("fill_value"), self.dtype)
        except (NotImplementedError, ValueError) as e:
            raise type(e)(f"{path}: {e}") from None
        self._crc = chain["crc"]
        self.device_codec = _device_codec(chain["compressor"])
        self._device_inner = _BLOSC_INNER.get((chain["compressor"] or {}).get("cname"), 1)

    def _key_path(self, idx) -> str:
        return os.path.join(self.path, _v3_key(self._encoding, idx))

    def _missing_name(self, idx):
        if self._shard is None:
            return self._key_path(idx)
        shard = tuple(i // p for i, p in zip(idx, self._shard["per"]))
        return f"{self._key_path(shard)} (inner chunk {tuple(int(i) for i in idx)})"

    def _index(self, shard) -> tuple[str, np.ndarray | None]:
        """(file, (n, 2) uint64 index) of a shard, ``None`` for a missing shard file; checked once and cached."""
        if shard not in self._indexes:
            p = self._key_path(shard)
            if not os.path.isfile(p):
                self._indexes[shard] = (p, None)
                return self._indexes[shard]
            sh = self._shard
            size = os.path.getsize(p)
            if size < sh["index_bytes"]:
                raise ValueError(f"{p}: a shard of {size} bytes cannot hold its {sh['index_bytes']}-byte index")
            with open(p, "rb") as fh:
                fh.seek(0 if sh["start"] else size - sh["index_bytes"])
                raw = fh.read(sh["index_bytes"])
            if len(raw) != sh["index_bytes"]:
                raise ValueError(f"{p}: short read of the shard index")
            if sh["index_crc"]:
                raw = _check_crc32c(raw, f"{p}: shard index")
            index = np.frombuffer(raw, dtype="<u8").reshape(sh["n"], 2).astype(np.uint64)
            present = ~((index[:, 0] == _MISSING) & (index[:, 1] == _MISSING))
            off, nbytes = index[present, 0], index[present, 1]
            if np.any(off > size) or np.any(nbytes > np.uint64(size) - off):
                raise ValueError(f"{p}: a shard index entry points outside the file of {size} bytes")
            self._indexes[shard] = (p, index)
        return self._indexes[shard]

    def _locate(self, idx):
        if self._shard is None:
            p = self._key_path(idx)
            return (p, p, 0, os.path.getsize(p)) if os.path.isfile(p) else None
        per = self._shard["per"]
        p, index = self._index(tuple(i // q for i, q in zip(idx, per)))
        if index is None:
            return None
        k = int(np.ravel_multi_index(tuple(i % q for i, q in zip(idx, per)), per)) if per else 0
        off, nbytes = int(index[k, 0]), int(index[k, 1])
        if off == _MISSING and nbytes == _MISSING:
            return None
        return p, f"{p} (inner chunk {tuple(int(i) for i in idx)})", off, nbytes

    def _payload(self, raw, where):
        if self._crc:
            raw = _check_crc32c(raw, where)
        return raw if self._decode is None else self._decode(bytes(raw))


class ZarrV3Source(_ZarrV3Array):
    """One 2-D or 3-D Zarr v3 array of a directory store (:class:`_ZarrV3Array`), sharded or not.  Chunks compressed
    with a codec ``xrs_zarr_decode`` decodes (``zstd``, ``gzip``, ``blosc`` with an LZ4 / Zstd / Zlib inner codec and
    byte shuffle or none, and their ``numcodecs.*`` twins) can be read for the device (:meth:`device_read`); a
    ``crc32c`` trailer is then checked there too."""

    def __init__(self, path: str):
        super().__init__(path)
        if len(self.shape) not in (2, 3):
            raise ValueError(f"{self.path}: expected a 2-D or 3-D array, got shape {self.shape}")


def cf_decoded_dtype(dtype: np.dtype, attrs: Mapping) -> np.dtype | None:
    """The float type CF mask-and-scale decoding gives a variable, ``None`` when its attributes ask for none:
    float32 for integers of up to 16 bits and floats of up to 32 bits (float32 holds them exactly), float64
    otherwise -- xarray's ``open_dataset(mask_and_scale=True)`` rule for variables without ``add_offset``
    (with one, xarray's choice has varied between releases; this build keeps the same rule)."""
    if not any(k in attrs for k in ("scale_factor", "add_offset", "_FillValue", "missing_value")):
        return None
    dtype = np.dtype(dtype)
    small = (dtype.kind in "iu" and dtype.itemsize <= 2) or (dtype.kind == "f" and dtype.itemsize <= 4)
    return np.dtype(np.float32 if small else np.float64)


class DecodedSource(LazySource):
    """CF mask-and-scale decoding of another source on the reader thread: ``_FillValue`` / ``missing_value``
    become NaN, then ``raw * scale_factor + add_offset`` in the decoded float type (:func:`cf_decoded_dtype`)."""

    def __init__(self, source: LazySource, attrs: Mapping):
        self.source, self.shape = source, tuple(source.shape)
        self.dtype = cf_decoded_dtype(source.dtype, attrs)
        if self.dtype is None:
            raise ValueError("the variable's attributes ask for no decoding")
        self._fills = []
        for key in ("_FillValue", "missing_value"):
            for f in np.asarray(attrs.get(key, [])).ravel().tolist():
                try:  # JSON attributes may spell the float specials as strings ("NaN"); those mask nothing new
                    f = float(f) if not isinstance(f, (int, np.integer)) else int(f)
                except (TypeError, ValueError):
                    continue
                if f == f and (source.dtype.kind == "f" or float(f).is_integer()):
                    self._fills.append(f)
        self._scale, self._offset = attrs.get("scale_factor"), attrs.get("add_offset")

    def _raw_fills(self) -> np.ndarray:
        """The fill values :meth:`read_bands` masks, as values of the stored type (native byte order)."""
        raw = np.dtype(self.source.dtype).newbyteorder("=")
        keep = [f for f in self._fills if raw.kind == "f" or np.iinfo(raw).min <= f <= np.iinfo(raw).max]
        with np.errstate(over="ignore"):
            return np.array([raw.type(f) for f in keep], dtype=raw)

    @property
    def device_decodable(self) -> bool:
        return bool(getattr(self.source, "device_decodable", False)) and len(self._raw_fills()) <= 16

    def device_read(self, b0, nb, segments, window, buffer=None):
        """The stored chunk files, as :meth:`ZarrV2Source.device_read`; :meth:`device_cf` gives the decoding."""
        return self.source.device_read(b0, nb, segments, window, buffer)

    def device_fill_bits(self) -> int:
        return self.source.device_fill_bits()

    def device_cf(self) -> dict:
        """What ``xrs_zarr_decode`` needs to apply this decoding: decoded dtype, fills (stored type), scale, offset."""
        return {"out_dtype": self.dtype, "fills": self._raw_fills(),
                "scale": None if self._scale is None else float(self._scale),
                "offset": None if self._offset is None else float(self._offset)}

    def read_bands(self, b0, nb, out):
        raw = np.empty((nb,) + self.shape[-2:], dtype=self.source.dtype)
        self.source.read_bands(b0, nb, raw)
        res = out[:nb]
        np.copyto(res, raw, casting="unsafe")
        for f in self._fills:  # a NaN fill value of float data is NaN already and is not in the list
            if raw.dtype.kind == "f" or np.iinfo(raw.dtype).min <= f <= np.iinfo(raw.dtype).max:
                res[raw == raw.dtype.type(f)] = np.nan
        if self._scale is not None:
            np.multiply(res, self.dtype.type(self._scale), out=res)
        if self._offset is not None:
            np.add(res, self.dtype.type(self._offset), out=res)


_CF_CODING_ATTRS = ("scale_factor", "add_offset", "_FillValue", "missing_value")


def _lazy_variable(source: LazySource, dims, attrs, name, mask_and_scale: bool) -> "LazyDataArray":
    if mask_and_scale and cf_decoded_dtype(source.dtype, attrs) is not None:
        source = DecodedSource(source, attrs)
        attrs = {k: v for k, v in attrs.items() if k not in _CF_CODING_ATTRS}  # moved to the encoding, as in xarray
    return LazyDataArray(source, dims=dims, attrs=attrs, name=name)


class LazyDataArray(DataArray):
    """A dataset variable whose values stay in a chunked store until a pipeline streams them (``source``);
    ``values`` materialises the whole array for anything that is not a streaming consumer."""

    __slots__ = ("source",)

    def __init__(self, source: LazySource, dims, attrs=None, name=None):
        self.source = source
        stand_in = np.broadcast_to(np.zeros((), dtype=source.dtype), source.shape)  # shape / dtype without memory
        DataArray.__init__(self, stand_in, dims=dims, attrs=attrs, name=name)

    @property
    def values(self) -> np.ndarray:
        return self.source.read_all()

    data = values


def _fill_value(fill, dtype: np.dtype):
    """The value of a missing chunk: ``fill_value`` of ``.zarray`` (``"NaN"`` / ``"Infinity"`` /
    ``"-Infinity"`` are the JSON spellings of the float specials; ``null`` leaves it undefined -- zero here)."""
    if isinstance(fill, str) or fill is None:
        return {"NaN": np.nan, "Infinity": np.inf, "-Infinity": -np.inf}.get(fill, 0) if dtype.kind == "f" else 0
    return fill


def _read_small_array(arr_dir: str, meta: dict) -> np.ndarray:
    """A 0-D or 1-D Zarr array (``spatial_ref``, axis coordinates), chunks decoded like those of
    :class:`ZarrV2Source` / :class:`ZarrV3Source` (``meta``: its ``.zarray`` or ``zarr.json``); missing chunks hold the
    fill value."""
    if meta.get("zarr_format") == 3:
        arr = _ZarrV3Array(arr_dir)
        if not arr.shape:
            return arr._chunk(())[()].copy()
        n, c = arr.shape[0], arr.chunks[0]
        parts = [arr._chunk((k,))[:min(c, n - k * c)] for k in range(-(-n // c))]
        return np.concatenate(parts) if n else np.empty(0, arr.dtype)
    if meta.get("filters"):
        raise NotImplementedError(f"{arr_dir}: filtered Zarr arrays need the zarr package, which this build does not "
                                  "have; open the store with xarray and pass the arrays instead")
    try:
        decode = chunk_decoder(meta.get("compressor"))
    except NotImplementedError as e:
        raise NotImplementedError(f"{arr_dir}: {e}") from None
    dt = np.dtype(meta["dtype"])
    fill = _fill_value(meta.get("fill_value"), dt)

    def chunk(name, count):
        p = os.path.join(arr_dir, name)
        if not os.path.isfile(p):
            return np.full(count, fill, dtype=dt)
        raw = open(p, "rb").read()
        return np.frombuffer(raw if decode is None else decode(raw), dtype=dt)[:count]

    shape = tuple(int(n) for n in meta["shape"])
    if not shape:
        return chunk("0", 1)[0].copy()
    n, c = shape[0], int(meta["chunks"][0])
    return np.concatenate([chunk(str(k), c)[:min(c, n - k * c)] for k in range(-(-n // c))]) if n else np.empty(0, dt)


def open_zarr_dataset(path: str, coord_names=("lon", "lat", "x", "y", "longitude", "latitude",
                                              "transformed_x", "transformed_y"), mask_and_scale: bool = False) -> Dataset:
    """A Zarr-v2 directory store as a :class:`Dataset`: scalar, 1-D and coordinate-named arrays are read
    now, every other 2-D / 3-D array becomes a :class:`LazyDataArray`.  By default values are delivered
    as stored (what ``xarray.open_zarr(..., mask_and_scale=False)`` gives): ``scale_factor`` /
    ``add_offset`` / ``_FillValue`` attributes are passed through, not applied.  ``mask_and_scale=True``
    decodes the lazy variables that carry such attributes on the reader thread (:class:`DecodedSource`).

    A Zarr v3 store (a root ``zarr.json`` of ``node_type`` group) is read the same way, each child array from its
    own ``zarr.json`` (:class:`ZarrV3Source`); the group attributes come from the root, and consolidated metadata is
    not used for reading."""
    root = os.path.join(path, "zarr.json")
    if os.path.isfile(root):
        group = json.load(open(root))
        if group.get("zarr_format") != 3 or group.get("node_type") != "group":
            raise ValueError(f"{path}: not a Zarr v3 group")
        return _open_zarr_v3(path, group, coord_names, mask_and_scale)
    data_vars, coords = {}, {}
    for item in sorted(os.listdir(path)):
        arr_dir = os.path.join(path, item)
        if not os.path.isfile(os.path.join(arr_dir, ".zarray")):
            continue
        meta = json.load(open(os.path.join(arr_dir, ".zarray")))
        attrs_path = os.path.join(arr_dir, ".zattrs")
        attrs = json.load(open(attrs_path)) if os.path.isfile(attrs_path) else {}
        dims = attrs.pop("_ARRAY_DIMENSIONS", None) or [f"dim_{k}" for k in range(len(meta["shape"]))]
        shape = tuple(meta["shape"])
        if len(shape) <= 1:
            coords[item] = DataArray(_read_small_array(arr_dir, meta), dims=dims if shape else (), attrs=attrs, name=item)
        else:
            src = ZarrV2Source(arr_dir)
            if item in coord_names:
                coords[item] = DataArray(src.read_all(), dims=dims, attrs=attrs, name=item)
            else:
                data_vars[item] = _lazy_variable(src, dims, attrs, item, mask_and_scale)
    group_attrs = os.path.join(path, ".zattrs")
    return Dataset(data_vars=data_vars, coords=coords, attrs=json.load(open(group_attrs)) if os.path.isfile(group_attrs) else {})


def _open_zarr_v3(path: str, group: dict, coord_names, mask_and_scale: bool) -> Dataset:
    """:func:`open_zarr_dataset` for a Zarr v3 group: its child arrays, by the same rules as a v2 store."""
    data_vars, coords = {}, {}
    for item in sorted(os.listdir(path)):
        arr_dir = os.path.join(path, item)
        meta_path = os.path.join(arr_dir, "zarr.json")
        if not os.path.isfile(meta_path):
            continue
        meta = json.load(open(meta_path))
        if meta.get("zarr_format") != 3 or meta.get("node_type") != "array":
            continue
        dims = v3_dimension_names(meta)
        attrs = dict(meta.get("attributes") or {})
        attrs.pop("_ARRAY_DIMENSIONS", None)
        shape = tuple(meta["shape"])
        if len(shape) <= 1:
            coords[item] = DataArray(_read_small_array(arr_dir, meta), dims=dims, attrs=attrs, name=item)
        else:
            src = ZarrV3Source(arr_dir)
            if item in coord_names:
                coords[item] = DataArray(src.read_all(), dims=dims, attrs=attrs, name=item)
            else:
                data_vars[item] = _lazy_variable(src, dims, attrs, item, mask_and_scale)
    return Dataset(data_vars=data_vars, coords=coords, attrs=dict(group.get("attributes") or {}))


def open_netcdf_dataset(path: str, coord_names=("lon", "lat", "x", "y", "longitude", "latitude",
                                                "transformed_x", "transformed_y"), mask_and_scale: bool = False) -> Dataset:
    """A NetCDF classic file as a :class:`Dataset`, with the rules of :func:`open_zarr_dataset`: scalar, 1-D
    and coordinate-named variables are read now, every other 2-D / 3-D variable becomes a
    :class:`LazyDataArray` over the file's memory map.  Values as stored unless ``mask_and_scale=True``
    (then as in :func:`open_zarr_dataset`); ``bytes`` attributes are decoded to ``str`` as xarray does."""
    from scipy.io import netcdf_file

    with open(path, "rb") as fh:
        magic = fh.read(4)
    if magic[:3] != b"CDF":
        kind = "a NetCDF-4 / HDF5 file, which needs the netCDF4 or h5py package (not in this build); open it with " \
               "xarray and pass the arrays instead" if magic == b"\x89HDF" else "not a NetCDF classic file"
        raise NotImplementedError(f"{path}: {kind}")

    class MappedFile(netcdf_file):
        """Lazy variables keep views of the memory map for as long as they live, so the map is released by
        the garbage collector, not by close(): scipy's warning about exactly that is not news here."""

        def close(self):
            import warnings

            with warnings.catch_warnings():
                warnings.simplefilter("ignore", RuntimeWarning)
                super().close()

        __del__ = close

    nc = MappedFile(path, "r", mmap=True, maskandscale=False)

    def text(v):
        return v.decode("utf-8", "replace") if isinstance(v, bytes) else v

    data_vars, coords = {}, {}
    for name, var in nc.variables.items():
        attrs = {k: text(v) for k, v in var._attributes.items()}
        dims = tuple(var.dimensions)
        if len(var.shape) in (2, 3) and name not in coord_names:
            data_vars[name] = _lazy_variable(NetCDF3Source(nc, name), dims, attrs, name, mask_and_scale)
            continue
        values = np.array(var.data, dtype=var.data.dtype.newbyteorder("="))  # a copy: independent of the map
        (coords if len(var.shape) <= 2 else data_vars)[name] = DataArray(values, dims=dims, attrs=attrs, name=name)
    return Dataset(data_vars=data_vars, coords=coords, attrs={k: text(v) for k, v in nc._attributes.items()})


def write_zarr_array(path: str, array: np.ndarray, chunks, dims) -> None:
    """Write ``array`` as an uncompressed Zarr-v2 array (test fixtures, synthetic benchmark stores)."""
    os.makedirs(path, exist_ok=True)
    array = np.asarray(array)
    chunks = tuple(int(c) for c in chunks)
    json.dump({"chunks": list(chunks), "compressor": None, "dtype": array.dtype.str, "fill_value": None, "filters": None,
               "order": "C", "shape": list(array.shape), "zarr_format": 2}, open(os.path.join(path, ".zarray"), "w"))
    json.dump({"_ARRAY_DIMENSIONS": list(dims)}, open(os.path.join(path, ".zattrs"), "w"))
    if array.ndim == 0:
        array.reshape(1).tofile(os.path.join(path, "0"))
        return
    grid = [range(-(-n // c)) for n, c in zip(array.shape, chunks)]
    for idx in np.ndindex(*[len(g) for g in grid]):
        block = np.zeros(chunks, dtype=array.dtype)
        sl = tuple(slice(k * c, min(n, (k + 1) * c)) for k, c, n in zip(idx, chunks, array.shape))
        part = array[sl]
        block[tuple(slice(0, s) for s in part.shape)] = part
        block.tofile(os.path.join(path, ".".join(str(k) for k in idx)))
