"""Case table of the device decode of compressed Zarr chunks (csrc/decode.cu, ``xrs_zarr_decode``), shared by the host
build (test_host_zarr_decode.py) and the GPU (test_zarr_decode_gpu.py).

A case is a store written to a temporary directory plus one read: bands ``b0 : b0 + nb`` of the row ``window``.  The
expected slot is what ``ZarrV2Source.read_bands`` / ``DecodedSource.read_bands`` -- the host decode -- gives for those
rows.  Frames come from test_host_io's Blosc assembler and pyarrow's ``lz4_raw``; LZ4 blocks the compressors may never
emit (every literal / match length class, overlapping offsets) are assembled by hand.  Malformed cases name the
rejection ``xrs_zarr_decode`` must report (``include/xrs.h``, enum xrs_decode_error)."""

from __future__ import annotations

import json
import os
from dataclasses import dataclass, field

import numpy as np

from xcube_resampling_b200.io import DecodedSource, ZarrV2Source, write_zarr_array

from .test_host_io import _blosc_frame

BAD_LAYOUT, OFFSET_ZERO, OFFSET_BEFORE_START, LITERALS_OVERRUN, MATCH_OVERRUN, INPUT_OVERRUN, SHORT = range(1, 8)

BLOSC_LZ4 = {"id": "blosc", "cname": "lz4", "clevel": 5, "shuffle": 1, "blocksize": 0}
LZ4 = {"id": "lz4", "acceleration": 1}


def lz4_raw(raw: bytes) -> bytes:
    import pyarrow as pa

    return pa.Codec("lz4_raw").compress(raw).to_pybytes()


def numcodecs_lz4(raw: bytes) -> bytes:
    return len(raw).to_bytes(4, "little") + lz4_raw(raw)


def _length(n: int) -> bytes:
    """LZ4 length extension bytes for a nibble of 15: runs of 255, then the rest."""
    return b"\xff" * (n // 255) + bytes([n % 255])


def lz4_block(seqs, last: bytes) -> tuple[bytes, bytes]:
    """An LZ4 block from ``seqs`` of (literals, offset, match length) and the final literals; returns the block and
    what it decodes to (copied byte by byte, as the format defines overlapping matches)."""
    block, out = bytearray(), bytearray()
    for lit, off, ml in list(seqs) + [(last, None, None)]:
        ln = min(len(lit), 15)
        mn = 0 if ml is None else min(ml - 4, 15)
        block.append((ln << 4) | mn)
        if ln == 15:
            block += _length(len(lit) - 15)
        block += lit
        out += lit
        if ml is None:
            break
        block += off.to_bytes(2, "little")
        if mn == 15:
            block += _length(ml - 19)
        for _ in range(ml):
            out.append(out[len(out) - off] if off <= len(out) else 0)
    return bytes(block), bytes(out)


@dataclass
class Case:
    name: str
    array: np.ndarray                 # values as stored (its dtype is the .zarray dtype, byte order included)
    chunks: tuple
    compressor: dict | None
    encode: object = None             # (raw chunk bytes, chunk key) -> file bytes, None: file missing
    attrs: dict = field(default_factory=dict)  # CF attributes: read through DecodedSource
    b0: int = 0
    nb: int = 0                       # 0: every band
    window: tuple | None = None       # source rows; None: all
    error: int = 0                    # the reason xrs_zarr_decode must report

    def write(self, root: str) -> str:
        path = os.path.join(root, self.name)
        dims = ("band", "y", "x")[-self.array.ndim:]
        write_zarr_array(path, self.array, self.chunks, dims)
        for key in os.listdir(path):
            if key.startswith("."):
                continue
            raw = open(os.path.join(path, key), "rb").read()
            data = self.encode(raw, key)
            if data is None:
                os.remove(os.path.join(path, key))
            else:
                open(os.path.join(path, key), "wb").write(data)
        meta = json.load(open(os.path.join(path, ".zarray")))
        meta["compressor"] = self.compressor
        if self.array.dtype.kind == "f":
            meta["fill_value"] = "NaN"
        elif self.array.dtype.kind in "iu":
            meta["fill_value"] = 7
        json.dump(meta, open(os.path.join(path, ".zarray"), "w"))
        return path

    def source(self, root: str):
        src = ZarrV2Source(self.write(root))
        return DecodedSource(src, self.attrs) if self.attrs else src

    def read(self):
        bands = 1 if self.array.ndim == 2 else self.array.shape[0]
        h = self.array.shape[-2]
        window = self.window or (0, h)
        return self.b0, self.nb or bands - self.b0, window

    def expected(self, source) -> np.ndarray:
        b0, nb, (j0, j1) = self.read()
        out = np.empty((nb,) + tuple(source.shape[-2:]), dtype=np.dtype(source.dtype).newbyteorder("="))
        source.read_bands(b0, nb, out)
        return out[:, j0:j1]


def _values(dtype, shape, seed) -> np.ndarray:
    """Compressible values with runs, plus a sprinkling of the dtype's extremes (NaN, -0.0, inf for floats)."""
    rng = np.random.default_rng(seed)
    dt = np.dtype(dtype)
    n = int(np.prod(shape))
    if dt.kind == "f":
        v = (rng.integers(0, 40, n) / 8).astype(dt)
        specials = np.array([np.nan, -0.0, np.inf, -np.inf, np.finfo(dt).max, np.finfo(dt).tiny / 4], dtype=dt)
    else:
        info = np.iinfo(dt)
        v = rng.integers(0, 9, n).astype(dt)
        specials = np.array([info.min, info.max, 0, 1], dtype=dt)
    v[np.repeat(rng.random(-(-n // 8)) < 0.3, 8)[:n]] = 3  # runs
    idx = rng.choice(n, size=min(n, 40), replace=False)
    v[idx] = specials[np.arange(len(idx)) % len(specials)]
    return v.reshape(shape)


def _blosc(typesize, blocksize, shuffle=True, dont_split=False, store_streams=False, missing=()):
    def encode(raw, key):
        if key in missing:
            return None
        return _blosc_frame(raw, typesize, blocksize, shuffle, "lz4", dont_split=dont_split, store_streams=store_streams)
    return encode


def _stored_frame(raw, key):
    """A Blosc frame holding the chunk as a plain copy (flag bit 1), shuffle flag set: it does not apply."""
    head = bytes([2, 1, 0x2 | 0x1 | (1 << 5), 4]) + len(raw).to_bytes(4, "little") + len(raw).to_bytes(4, "little")
    return head + (16 + len(raw)).to_bytes(4, "little") + raw


def _hand(block: bytes, size: int):
    return lambda raw, key: size.to_bytes(4, "little") + block


def cases() -> list[Case]:
    out = []
    nine = ("float32", "float64", "uint8", "int8", "uint16", "int16", "int32", "uint32", "int64")
    for dt in nine:
        isz = np.dtype(dt).itemsize
        a = _values(dt, (3, 21, 37), seed=isz)
        # 2 x 8 x 17 = 272 elements: two full blocks of 128 elements (split: typesize streams) and a partial one
        out.append(Case(f"{dt}_split", a, (2, 8, 17), BLOSC_LZ4, _blosc(isz, 128 * isz), b0=1, nb=2, window=(3, 19)))
        out.append(Case(f"{dt}_dont_split", a, (2, 8, 17), BLOSC_LZ4, _blosc(isz, 128 * isz, dont_split=True)))
        out.append(Case(f"{dt}_no_shuffle", a, (2, 8, 17), dict(BLOSC_LZ4, shuffle=0),
                        _blosc(isz, 64 * isz, shuffle=False)))
        out.append(Case(f"{dt}_lz4", a[0], (8, 16), LZ4, lambda raw, key: numcodecs_lz4(raw)))
    f32 = _values("float32", (5, 30, 45), seed=3)
    out += [
        Case("stored_streams", f32, (2, 16, 32), BLOSC_LZ4, _blosc(4, 1024, store_streams=True)),
        Case("stored_frame", f32, (2, 16, 32), BLOSC_LZ4, _stored_frame),
        # typesize 4 over uint8 chunks of 45 bytes, blocks of 16: the last block holds 3 elements and 1 tail byte
        Case("tail_not_an_element", _values("uint8", (2, 11, 23), seed=4), (1, 5, 9), BLOSC_LZ4, _blosc(4, 16)),
        # typesize 8 over int16 chunks of 70 bytes, blocks of 64: a last block of 6 bytes, not one whole element
        Case("typesize_above_itemsize", _values("int16", (13, 20), seed=5), (5, 7), BLOSC_LZ4, _blosc(8, 64)),
        Case("missing_chunks", f32, (2, 16, 32), BLOSC_LZ4, _blosc(4, 1024, missing=("0.0.1", "2.1.0", "1.0.0"))),
        Case("missing_chunks_int", _values("int32", (3, 30, 45), seed=6), (1, 16, 32), BLOSC_LZ4,
             _blosc(4, 1024, missing=("0.1.1", "2.0.0"))),
        Case("ragged_edges_window", f32, (2, 16, 32), BLOSC_LZ4, _blosc(4, 512), b0=2, nb=3, window=(7, 29)),
        # 90000 chunk files in one call: more than a launch's 65535 grid rows
        Case("many_chunk_files", _values("uint8", (300, 300), seed=12), (1, 1), BLOSC_LZ4, _blosc(1, 16)),
        Case("band_depth_3_of_1", f32, (3, 16, 32), BLOSC_LZ4, _blosc(4, 1024), b0=0, nb=1),
        Case("band_depth_3_of_2", f32, (3, 16, 32), BLOSC_LZ4, _blosc(4, 1024), b0=1, nb=2),
        Case("band_depth_3_of_4", f32, (3, 16, 32), BLOSC_LZ4, _blosc(4, 1024), b0=1, nb=4),
    ]
    for dt in (">f4", ">i2", ">f8", ">u4"):
        a = _values(np.dtype(dt).newbyteorder("="), (3, 21, 37), seed=9).astype(dt)
        isz = a.dtype.itemsize
        out.append(Case(f"big_endian_{dt[1:]}", a, (2, 8, 17), BLOSC_LZ4, _blosc(isz, 128 * isz)))
    # CF mask-and-scale: the decoded type, NaN for _FillValue / missing_value, * scale, + offset
    cf = [("uint16", {"scale_factor": 0.01, "add_offset": -5.0, "_FillValue": 3, "missing_value": [8, 65535]}),
          ("int16", {"scale_factor": 2.5e-4, "add_offset": 1.25, "_FillValue": -32768, "missing_value": [3, 70000]}),
          ("uint8", {"scale_factor": 0.5, "_FillValue": 255, "missing_value": [3]}),
          ("int32", {"scale_factor": 1e-3, "add_offset": 100.0, "_FillValue": -2147483648, "missing_value": [3]}),
          ("float32", {"scale_factor": 3.0, "add_offset": 0.5, "_FillValue": "NaN", "missing_value": [3.0]}),
          ("float32", {"_FillValue": 0.0}),
          ("uint16", {"add_offset": 0.0})]
    for k, (dt, attrs) in enumerate(cf):
        isz = np.dtype(dt).itemsize
        a = _values(dt, (3, 21, 37), seed=20 + k)
        out.append(Case(f"cf_{k}_{dt}", a, (2, 8, 17), BLOSC_LZ4, _blosc(isz, 128 * isz, missing=("1.1.0",)),
                        attrs=attrs, b0=1, nb=2))
    # hand-assembled LZ4 blocks: literal lengths 0 / 14 / 15 / 270 / >= 510, match lengths 4 / 18 / 19 / >= 274,
    # offsets 1 ... 65535, overlapping copies; numcodecs lz4 chunks of uint8 (1, n)
    rng = np.random.default_rng(7)
    lits = lambda n: rng.integers(0, 256, n, dtype=np.uint8).tobytes()  # noqa: E731
    hand = [
        ("lz4_lengths", [(lits(14), 1, 4), (lits(15), 2, 18), (b"", 3, 19), (lits(270), 4, 300), (lits(600), 7, 4),
                         (lits(1), 8, 5), (lits(2), 31, 40), (lits(3), 32, 64), (lits(4), 33, 33)], lits(5)),
        ("lz4_offset_65535", [(lits(70000), 65535, 1000), (lits(509), 65535, 274), (lits(510), 9, 529)], lits(12)),
        ("lz4_literals_only", [], lits(300)),
    ]
    for name, seqs, last in hand:
        block, dec = lz4_block(seqs, last)
        arr = np.frombuffer(dec, np.uint8).reshape(1, -1)
        out.append(Case(name, arr, arr.shape, LZ4, _hand(block, len(dec))))
    # malformed: one chunk each, its size prefix the chunk size
    n = len(lz4_block([(b"abcdefgh", 8, 4)], b"xyzuvwa")[1])  # 19 bytes
    bad = [
        ("bad_offset_zero", bytes([0x80]) + b"abcdefgh" + b"\x00\x00" + bytes([0x30]) + b"xyz", OFFSET_ZERO),
        ("bad_offset_before_start", bytes([0x80]) + b"abcdefgh" + b"\x09\x00" + bytes([0x30]) + b"xyz",
         OFFSET_BEFORE_START),
        ("bad_literals_past_size", bytes([0x80]) + b"abcdefgh" + b"\x08\x00" + bytes([0x80]) + b"xyzuvwab",
         LITERALS_OVERRUN),
        ("bad_match_past_size", bytes([0x8f]) + b"abcdefgh" + b"\x08\x00" + b"\x05" + bytes([0x30]) + b"xyz",
         MATCH_OVERRUN),
        ("bad_extension_past_input", bytes([0xf0]) + b"\xff\xff", INPUT_OVERRUN),
        ("bad_match_extension_past_input", bytes([0x8f]) + b"abcdefgh" + b"\x08\x00" + b"\xff", INPUT_OVERRUN),
        ("bad_ends_after_match", bytes([0x80]) + b"abcdefgh" + b"\x08\x00", INPUT_OVERRUN),
        ("bad_short", bytes([0x80]) + b"abcdefgh" + b"\x08\x00" + bytes([0x20]) + b"xy", SHORT),
    ]
    for name, block, reason in bad:
        arr = np.zeros((1, n), np.uint8)
        out.append(Case(name, arr, arr.shape, LZ4, _hand(block, n), error=reason))

    a = _values("float32", (1, 16, 32), seed=11)

    def stream_past_frame(raw, key):
        f = bytearray(_blosc_frame(raw, 4, 1024, True, "lz4"))
        pos = int.from_bytes(f[16:20], "little")
        f[pos:pos + 4] = (len(f) - pos).to_bytes(4, "little")  # its data would end 4 bytes past the frame
        return bytes(f)

    def block_offset_past_frame(raw, key):
        f = bytearray(_blosc_frame(raw, 4, 1024, True, "lz4"))
        f[16:20] = (len(f) - 2).to_bytes(4, "little")
        return bytes(f)

    out.append(Case("bad_stream_past_frame", a, (1, 16, 32), BLOSC_LZ4, stream_past_frame, error=BAD_LAYOUT))
    out.append(Case("bad_block_offset_past_frame", a, (1, 16, 32), BLOSC_LZ4, block_offset_past_frame,
                    error=BAD_LAYOUT))
    return out
