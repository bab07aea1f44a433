"""Case table of the device decode of Deflate-compressed Zarr chunks (numcodecs ``zlib`` / ``gzip`` and Blosc-Zlib;
csrc/decode.cu, ``k_inflate``), shared by the host build (test_host_deflate_decode.py) and the GPU
(test_deflate_decode_gpu.py).

Cases are :class:`zarr_decode_cases.Case`.  Streams come from ``zlib.compressobj`` (levels 0-9, every strategy,
window bits 9-15, memLevel 1 and 9), ``gzip.compress`` / ``gzip.GzipFile`` and pyarrow's ``gzip`` codec; Blosc-Zlib
frames from test_host_io's assembler.  Streams with stored / fixed / dynamic blocks the compressors may never emit --
every length and distance code at both ends of its extra bits, 15-bit codes, every repeat code at both ends of its
count, a single distance code, no distance codes -- are written here with a small bit writer (RFC 1951), and gzip
files with every header field and several members.  Malformed files name the reason ``xrs_zarr_decode`` must report
(``include/xrs.h``, enum xrs_decode_error); the host path rejects each of them too."""

from __future__ import annotations

import gzip
import io
import random
import zlib

import numpy as np

from .test_host_io import _blosc_frame
from .zarr_decode_cases import Case, _values

(OFFSET_BEFORE_START, LITERALS_OVERRUN, MATCH_OVERRUN, INPUT_OVERRUN, SHORT, BAD_FRAME_HEADER) = (3, 4, 5, 6, 7, 8)
TRAILING_BYTES, CHECKSUM, BAD_BLOCK, BAD_CODES, BAD_SYMBOL = 14, 15, 16, 17, 18

ZLIB = {"id": "zlib", "level": 1}
GZIP = {"id": "gzip", "level": 1}
BLOSC_ZLIB = {"id": "blosc", "cname": "zlib", "clevel": 5, "shuffle": 1, "blocksize": 0}


# ---- a Deflate writer (RFC 1951) ----

class Bits:
    """LSB-first bit writer; Huffman codes go most significant bit first."""

    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def bits(self, v: int, n: int):
        assert 0 <= v < (1 << n) or n == v == 0
        self.acc |= v << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def code(self, c: int, n: int):
        self.bits(int(format(c, f"0{n}b")[::-1], 2), n)

    def align(self):
        if self.n:
            self.bits(0, 8 - self.n)

    def done(self) -> bytes:
        self.align()
        return bytes(self.out)


LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195,
            227, 258]
LEN_EXTRA = [0] * 8 + [k // 4 for k in range(4, 24)] + [0]
DIST_BASE = [1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073,
             4097, 6145, 8193, 12289, 16385, 24577]
DIST_EXTRA = [0, 0, 0, 0] + [k // 2 for k in range(2, 28)]


def canonical(lengths) -> dict:
    """symbol -> (code, length) of the canonical Huffman code with these lengths (RFC 1951 3.2.2)."""
    count = [0] * 16
    for n in lengths:
        count[n] += 1
    count[0] = 0
    code, nxt = 0, [0] * 16
    for b in range(1, 16):
        code = (code + count[b - 1]) << 1
        nxt[b] = code
    out = {}
    for s, n in enumerate(lengths):
        if n:
            out[s] = (nxt[n], n)
            nxt[n] += 1
    return out


FIXED_LIT = canonical([8] * 144 + [9] * 112 + [7] * 24 + [8] * 8)
FIXED_DIST = canonical([5] * 32)


def _match_codes(length: int, dist: int, len_code: int | None = None):
    lc = len_code if len_code is not None else max(c for c in range(29) if LEN_BASE[c] <= length and
                                                   (c != 27 or length < 258))
    dc = max(c for c in range(30) if DIST_BASE[c] <= dist)
    return lc, length - LEN_BASE[lc], dc, dist - DIST_BASE[dc]


def huffman_block(w: Bits, ops, out: bytearray, lit_codes, dist_codes):
    """``ops``: bytes (literals) or (length, distance[, length code]) matches; appends what they decode to."""
    for op in ops:
        if isinstance(op, (bytes, bytearray)):
            for b in op:
                w.code(*lit_codes[b])
                out.append(b)
            continue
        length, dist = op[0], op[1]
        lc, le, dc, de = _match_codes(length, dist, op[2] if len(op) > 2 else None)
        w.code(*lit_codes[257 + lc])
        w.bits(le, LEN_EXTRA[lc])
        w.code(*dist_codes[dc])
        w.bits(de, DIST_EXTRA[dc])
        for _ in range(length):
            out.append(out[len(out) - dist])
    w.code(*lit_codes[256])


def stored_block(w: Bits, data: bytes, out: bytearray, last: bool):
    w.bits(int(last), 1)
    w.bits(0, 2)
    w.align()
    w.bits(len(data), 16)
    w.bits(len(data) ^ 0xFFFF, 16)
    for b in data:
        w.bits(b, 8)
    out += data


def fixed_block(w: Bits, ops, out: bytearray, last: bool):
    w.bits(int(last), 1)
    w.bits(1, 2)
    huffman_block(w, ops, out, FIXED_LIT, FIXED_DIST)


def tokens(lengths):
    """Code-length symbols for ``lengths``: runs of zeros as 18 (11-138) / 17 (3-10), repeats of the previous
    length as 16 (3-6), greedily, as (symbol, extra bits, extra value)."""
    out, i = [], 0
    while i < len(lengths):
        v, r = lengths[i], 1
        while i + r < len(lengths) and lengths[i + r] == v:
            r += 1
        i += r
        if v == 0:
            while r >= 11:
                k = min(r, 138)
                out.append((18, 7, k - 11))
                r -= k
            if r >= 3:
                out.append((17, 3, r - 3))
                r = 0
            out += [(0, 0, 0)] * r
            continue
        out.append((v, 0, 0))
        r -= 1
        while r >= 3:
            k = min(r, 6)
            out.append((16, 2, k - 3))
            r -= k
        out += [(v, 0, 0)] * r
    return out


# a complete code-length code over all 19 symbols: 13 of 4 bits, 6 of 5 bits
CL_ORDER = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
CL_LENGTHS = [4] * 13 + [5] * 6


def dynamic_block(w: Bits, lit_lengths, dist_lengths, ops, out: bytearray, last: bool, toks=None):
    w.bits(int(last), 1)
    w.bits(2, 2)
    w.bits(len(lit_lengths) - 257, 5)
    w.bits(len(dist_lengths) - 1, 5)
    w.bits(19 - 4, 4)
    for k in range(19):
        w.bits(CL_LENGTHS[k], 3)
    cl = canonical([CL_LENGTHS[CL_ORDER.index(s)] for s in range(19)])
    for sym, nb, val in (toks if toks is not None else tokens(list(lit_lengths) + list(dist_lengths))):
        w.code(*cl[sym])
        w.bits(val, nb)
    huffman_block(w, ops, out, canonical(lit_lengths), canonical(dist_lengths))


def zlib_wrap(raw: bytes, out: bytes) -> bytes:
    return b"\x78\x01" + raw + zlib.adler32(out).to_bytes(4, "big")


def gzip_member(raw: bytes, out: bytes, flags: int = 0, header_fields: bytes = b"") -> bytes:
    return (b"\x1f\x8b\x08" + bytes([flags]) + (123456).to_bytes(4, "little") + b"\x00\x03" + header_fields + raw +
            zlib.crc32(out).to_bytes(4, "little") + (len(out) & 0xFFFFFFFF).to_bytes(4, "little"))


# ---- hand-assembled streams ----

def _rand(n: int, seed: int) -> bytes:
    return random.Random(seed).randbytes(n)


def every_length_and_distance() -> tuple[bytes, bytes]:
    """One stored block of 33000 random bytes, then fixed blocks with every length code at its lowest and highest
    extra value (284 + 31 = 258 too, and 285) and every distance code at both ends, 32768 included."""
    w, out = Bits(), bytearray()
    stored_block(w, _rand(33000, 1), out, False)
    ops = []
    for c in range(29):
        for length in {LEN_BASE[c], LEN_BASE[c] + (1 << LEN_EXTRA[c]) - 1}:
            ops += [(length, 1000 + c), b"x"]
    ops += [(258, 77, 27), b"y"]  # code 284 with extra 31
    for c in range(30):
        for dist in {DIST_BASE[c], DIST_BASE[c] + (1 << DIST_EXTRA[c]) - 1}:
            ops += [(5 + c % 7, dist), bytes([c])]
    fixed_block(w, ops, out, False)
    fixed_block(w, [b"run", (258, 1), (3, 1), (100, 1), b"z"], out, True)  # distance 1
    return w.done(), bytes(out)


def stored_and_mixed() -> tuple[bytes, bytes]:
    """Stored blocks of 0 and 65535 bytes and every block type in turn, their boundaries inside a byte."""
    w, out = Bits(), bytearray()
    stored_block(w, b"", out, False)
    fixed_block(w, [b"abc", (7, 2)], out, False)  # ends inside a byte
    stored_block(w, _rand(65535, 2), out, False)
    lit = [0] * 286
    for s in range(256):
        lit[s] = 9 if s < 224 else 8  # 224 / 512 + 32 / 256 = 9 / 16: the rest below
    lit[256:286] = [6] * 26 + [7] * 4
    dynamic_block(w, lit, [4, 4] + [5] * 28, [b"dynamic", (10, 3), b"!" * 5, (40, 300)], out, False)
    fixed_block(w, [b"q"], out, False)
    stored_block(w, b"tail", out, True)
    return w.done(), bytes(out)


def fifteen_bit_codes() -> tuple[bytes, bytes]:
    """A dynamic block with codes of 1 to 15 bits (the longest two reach subtables) and a single distance code of
    length 1."""
    lit = [0] * 258
    for k, s in enumerate(range(65, 79)):  # 'A'..'N' get 1..14 bits
        lit[s] = k + 1
    lit[256] = lit[257] = 15
    w, out = Bits(), bytearray()
    ops = [b"ABCDEFGHIJKLMN" * 3, b"N" * 5, (3, 1), b"MA", (3, 1)]
    dynamic_block(w, lit, [1], ops, out, True)
    return w.done(), bytes(out)


def no_distance_codes() -> tuple[bytes, bytes]:
    """A dynamic block with one distance length of 0 (no distance codes) and literals only."""
    lit = [0] * 257
    lit[ord("a")], lit[ord("b")], lit[256] = 1, 2, 2
    w, out = Bits(), bytearray()
    dynamic_block(w, lit, [0], [b"abba" * 50], out, True)
    return w.done(), bytes(out)


def repeat_codes() -> tuple[bytes, bytes]:
    """Code lengths with 17 at 3 and 10, 18 at 11 and 138, 16 at 3 and 6, and a 16 crossing from the litlen to the
    distance lengths."""
    lit = [0] * 286
    lit[3:10] = [7] * 7          # 7, then 16 x 6
    lit[20:24] = [7] * 4         # 7, then 16 x 3
    lit[35] = 7
    lit[174:178] = [6] * 4
    lit[178:286] = [7] * 108     # runs on into the distance lengths: a 16 covers 281-286
    # zeros: 0-2 (17 x 3), 10-19 (17 x 10), 24-34 (18 x 11), 36-173 (18 x 138)
    dist = [7, 7, 6, 5, 4, 3, 2, 1] + [0] * 22
    toks = tokens(lit + dist)
    assert (17, 3, 0) in toks and (17, 3, 7) in toks and (18, 7, 0) in toks and (18, 7, 127) in toks
    assert (16, 2, 0) in toks and (16, 2, 3) in toks
    w, out = Bits(), bytearray()
    ops = [bytes([3, 4, 5, 20, 35, 174, 200, 255]), (3, 1), (10, 5), bytes([9, 21]), (20, 16), (258, 8),
           bytes([23, 177])]
    dynamic_block(w, lit, dist, ops, out, True, toks)
    return w.done(), bytes(out)


HAND = {"hand_every_length_and_distance": every_length_and_distance, "hand_stored_and_mixed": stored_and_mixed,
        "hand_15_bit_codes": fifteen_bit_codes, "hand_no_distance_codes": no_distance_codes,
        "hand_repeat_codes": repeat_codes}


# ---- the table ----

def _per_chunk(fn):
    return lambda raw, key: fn(raw)


def _blosc_zlib(typesize, blocksize, shuffle=True, dont_split=False, store_streams=False, missing=()):
    def encode(raw, key):
        if key in missing:
            return None
        return _blosc_frame(raw, typesize, blocksize, shuffle, "zlib", dont_split=dont_split,
                            store_streams=store_streams)
    return encode


def _stored_frame(raw, key):
    """A Blosc-Zlib frame holding the chunk as a plain copy (flag bit 1)."""
    head = bytes([2, 1, 0x2 | 0x1 | (3 << 5), 4]) + len(raw).to_bytes(4, "little") + len(raw).to_bytes(4, "little")
    return head + (16 + len(raw)).to_bytes(4, "little") + raw


def compressobj(level=6, strategy=zlib.Z_DEFAULT_STRATEGY, wbits=15, mem_level=8):
    def enc(raw):
        c = zlib.compressobj(level, zlib.DEFLATED, wbits, mem_level, strategy)
        return c.compress(raw) + c.flush()
    return enc


def gzip_file_with_name(raw: bytes) -> bytes:
    buf = io.BytesIO()
    with gzip.GzipFile(filename="chunk.bin", mode="wb", fileobj=buf, mtime=1700000000) as f:
        f.write(raw)
    return buf.getvalue()


def pyarrow_gzip(raw: bytes) -> bytes:
    import pyarrow as pa

    return pa.Codec("gzip").compress(raw).to_pybytes()


def _gzip_variants(raw: bytes, kind: str) -> bytes:
    """gzip files with header fields, several members (one empty) and NUL padding, over the chunk ``raw``."""
    half = len(raw) // 2
    d1, d2 = zlib.compressobj(6, zlib.DEFLATED, -15), zlib.compressobj(1, zlib.DEFLATED, -15)
    a, b = d1.compress(raw[:half]) + d1.flush(), d2.compress(raw[half:]) + d2.flush()
    e = zlib.compressobj(6, zlib.DEFLATED, -15)
    empty = e.compress(b"") + e.flush()
    if kind == "fields":  # FEXTRA, FNAME, FCOMMENT, FHCRC and the reserved bits 5-7
        fields = (4).to_bytes(2, "little") + b"XY\x00\x00" + b"name.bin\x00" + b"a comment\x00" + b"\xde\xad"
        return gzip_member(a, raw[:half], 0x04 | 0x08 | 0x10 | 0x02 | 0xE0, fields) + gzip_member(b, raw[half:])
    if kind == "members":
        return gzip_member(a, raw[:half]) + gzip_member(empty, b"") + gzip_member(b, raw[half:])
    return gzip_member(a, raw[:half]) + b"\x00" * 7 + gzip_member(b, raw[half:]) + b"\x00" * 5


def cases() -> list[Case]:
    out = []
    nine = ("float32", "float64", "uint8", "int8", "uint16", "int16", "int32", "uint32", "int64")
    for k, dt in enumerate(nine):
        isz = np.dtype(dt).itemsize
        a = _values(dt, (3, 21, 37), seed=60 + isz)
        out.append(Case(f"{dt}_zlib_split", a, (2, 8, 17), BLOSC_ZLIB, _blosc_zlib(isz, 128 * isz), b0=1, nb=2,
                        window=(3, 19)))
        out.append(Case(f"{dt}_zlib_dont_split", a, (2, 8, 17), BLOSC_ZLIB, _blosc_zlib(isz, 128 * isz,
                                                                                       dont_split=True)))
        out.append(Case(f"{dt}_zlib_no_shuffle", a, (2, 8, 17), dict(BLOSC_ZLIB, shuffle=0),
                        _blosc_zlib(isz, 64 * isz, shuffle=False)))
        out.append(Case(f"{dt}_zlib", a[0], (8, 16), dict(ZLIB, level=k + 1),
                        _per_chunk(lambda raw, lv=k + 1: zlib.compress(raw, lv))))
        out.append(Case(f"{dt}_gzip", a[0], (8, 16), dict(GZIP, level=9 - k),
                        _per_chunk(lambda raw, lv=9 - k: gzip.compress(raw, lv, mtime=0))))
    # a 2 x 200 x 128 float32 field (200 KiB chunks): zlib's encoder settings
    rng = np.random.default_rng(61)
    field = (np.sin(np.arange(400 * 128) / 300.0).reshape(4, 100, 128) * 1000).astype(np.float32)
    field += rng.integers(0, 4, field.shape).astype(np.float32)
    big = np.concatenate([field, field[::-1]], axis=1)
    for level in range(10):
        out.append(Case(f"zlib_level_{level}", big, (2, 200, 128), dict(ZLIB, level=level),
                        _per_chunk(compressobj(level))))
    for name, strategy in (("filtered", zlib.Z_FILTERED), ("huffman_only", zlib.Z_HUFFMAN_ONLY),
                           ("rle", zlib.Z_RLE), ("fixed", zlib.Z_FIXED)):
        out.append(Case(f"zlib_strategy_{name}", big, (2, 200, 128), ZLIB, _per_chunk(compressobj(6, strategy))))
    f32 = _values("float32", (5, 30, 45), seed=62)
    text = _values("uint8", (40, 1000), seed=63)
    for wbits in range(9, 16):
        out.append(Case(f"zlib_wbits_{wbits}", text, (20, 1000), ZLIB, _per_chunk(compressobj(9, wbits=wbits))))
    for mem in (1, 9):
        out.append(Case(f"zlib_mem_level_{mem}", big, (2, 200, 128), ZLIB, _per_chunk(compressobj(6, mem_level=mem))))
    out += [
        Case("gzip_mtime", f32, (2, 16, 32), GZIP, _per_chunk(lambda r: gzip.compress(r, 6, mtime=1234567890))),
        Case("gzip_file_name", f32, (2, 16, 32), GZIP, _per_chunk(gzip_file_with_name)),
        Case("gzip_pyarrow", big, (2, 200, 128), GZIP, _per_chunk(pyarrow_gzip)),
        Case("gzip_header_fields", f32, (2, 16, 32), GZIP, _per_chunk(lambda r: _gzip_variants(r, "fields"))),
        Case("gzip_members", f32, (2, 16, 32), GZIP, _per_chunk(lambda r: _gzip_variants(r, "members"))),
        Case("gzip_nul_padding", f32, (2, 16, 32), GZIP, _per_chunk(lambda r: _gzip_variants(r, "padding"))),
        Case("zlib_trailing_bytes", f32, (2, 16, 32), ZLIB, _per_chunk(lambda r: zlib.compress(r) + b"junk")),
        Case("blosc_zlib_stored_streams", f32, (2, 16, 32), BLOSC_ZLIB, _blosc_zlib(4, 1024, store_streams=True)),
        Case("blosc_zlib_stored_frame", f32, (2, 16, 32), BLOSC_ZLIB, _stored_frame),
        Case("zlib_missing_chunks", f32, (2, 16, 32), ZLIB,
             lambda raw, key: None if key in ("0.0.1", "2.1.0") else zlib.compress(raw)),
        Case("gzip_missing_chunks", f32, (2, 16, 32), GZIP,
             lambda raw, key: None if key == "1.0.0" else gzip.compress(raw)),
        Case("blosc_zlib_missing_chunks", f32, (2, 16, 32), BLOSC_ZLIB, _blosc_zlib(4, 1024, missing=("1.0.0",))),
        Case("zlib_ragged_edges_window", f32, (2, 16, 32), ZLIB, _per_chunk(zlib.compress), b0=2, nb=3,
             window=(7, 29)),
        Case("gzip_band_depth_3_of_2", f32, (3, 16, 32), GZIP, _per_chunk(gzip.compress), b0=1, nb=2),
        Case("blosc_zlib_band_depth_3_of_4", f32, (3, 16, 32), BLOSC_ZLIB, _blosc_zlib(4, 1024), b0=1, nb=4),
        Case("blosc_zlib_tail_not_an_element", _values("uint8", (2, 11, 23), seed=64), (1, 5, 9), BLOSC_ZLIB,
             _blosc_zlib(4, 16)),
    ]
    for dt in (">f4", ">i2", ">f8", ">u4"):
        a = _values(np.dtype(dt).newbyteorder("="), (3, 21, 37), seed=65).astype(dt)
        isz = a.dtype.itemsize
        out.append(Case(f"zlib_big_endian_{dt[1:]}", a, (2, 8, 17), ZLIB, _per_chunk(zlib.compress)))
        out.append(Case(f"gzip_big_endian_{dt[1:]}", a, (2, 8, 17), GZIP, _per_chunk(gzip.compress)))
        out.append(Case(f"blosc_zlib_big_endian_{dt[1:]}", a, (2, 8, 17), BLOSC_ZLIB, _blosc_zlib(isz, 128 * isz)))
    cf = [("uint16", {"scale_factor": 0.01, "add_offset": -5.0, "_FillValue": 3, "missing_value": [8, 65535]}),
          ("int16", {"scale_factor": 2.5e-4, "add_offset": 1.25, "_FillValue": -32768}),
          ("float32", {"scale_factor": 3.0, "add_offset": 0.5, "_FillValue": "NaN", "missing_value": [3.0]})]
    for k, (dt, attrs) in enumerate(cf):
        isz = np.dtype(dt).itemsize
        a = _values(dt, (3, 21, 37), seed=66 + k)
        out.append(Case(f"zlib_cf_{k}_{dt}", a, (2, 8, 17), ZLIB,
                        lambda raw, key: None if key == "1.1.0" else zlib.compress(raw), attrs=attrs, b0=1, nb=2))
        out.append(Case(f"gzip_cf_{k}_{dt}", a, (2, 8, 17), GZIP, _per_chunk(gzip.compress), attrs=attrs))
        out.append(Case(f"blosc_zlib_cf_{k}_{dt}", a, (2, 8, 17), BLOSC_ZLIB, _blosc_zlib(isz, 128 * isz),
                        attrs=attrs))
    for name, make in HAND.items():
        raw, dec = make()
        arr = np.frombuffer(dec, np.uint8).reshape(1, -1)
        out.append(Case(name, arr, arr.shape, ZLIB, _hand(zlib_wrap(raw, dec))))
        out.append(Case(name.replace("hand_", "hand_gzip_"), arr, arr.shape, GZIP, _hand(gzip_member(raw, dec))))
    out += malformed_cases()
    return out


def _hand(data: bytes):
    return lambda raw, key: data


def _fixed(ops, last=True) -> tuple[bytes, bytes]:
    w, out = Bits(), bytearray()
    fixed_block(w, ops, out, last)
    return w.done(), bytes(out)


def _raw_fixed_symbols(syms) -> bytes:
    """A final fixed block of litlen symbols given as (symbol, [distance symbol]) without checks."""
    w = Bits()
    w.bits(1, 1)
    w.bits(1, 2)
    for s in syms:
        if isinstance(s, tuple):
            w.code(*FIXED_LIT[s[0]])
            w.code(*FIXED_DIST[s[1]])
        else:
            w.code(*FIXED_LIT[s])
    return w.done()


def _dynamic_header(hlit: int, hdist: int, cl_lengths, toks) -> Bits:
    """The start of a final dynamic block with the given fields (unchecked); code-length symbols from ``toks``."""
    w = Bits()
    w.bits(1, 1)
    w.bits(2, 2)
    w.bits(hlit - 257, 5)
    w.bits(hdist - 1, 5)
    w.bits(19 - 4, 4)
    for k in range(19):
        w.bits(cl_lengths[k], 3)
    cl = canonical([cl_lengths[CL_ORDER.index(s)] for s in range(19)])
    for sym, nb, val in toks:
        w.code(*cl[sym])
        w.bits(val, nb)
    return w


def malformed_cases() -> list[Case]:
    """One numcodecs zlib / gzip chunk of uint8 (1, n) each (or a Blosc-Zlib frame for header errors the host checks
    on the file itself), with the reason the device must report."""
    n = 40
    good, dec = _fixed([b"abcdefgh", (8, 8), _rand(24, 3)])
    assert len(dec) == n
    z, g = (lambda raw: zlib_wrap(raw, dec)), (lambda raw: gzip_member(raw, dec))
    lit = [0] * 257  # with a 258th length of 2: a complete litlen set of 'a', end of block and code 257
    lit[ord("a")], lit[256] = 1, 2
    bad = [
        # wrappers
        ("bad_zlib_adler", ZLIB, z(good)[:-1] + bytes([z(good)[-1] ^ 1]), CHECKSUM),
        ("bad_zlib_adler_missing", ZLIB, z(good)[:-2], INPUT_OVERRUN),
        ("bad_zlib_truncated", ZLIB, z(good)[:12], INPUT_OVERRUN),
        ("bad_gzip_crc", GZIP, g(good)[:-8] + bytes(4) + g(good)[-4:], CHECKSUM),
        ("bad_gzip_isize", GZIP, g(good)[:-4] + (n + 1).to_bytes(4, "little"), CHECKSUM),
        ("bad_gzip_trailer_missing", GZIP, g(good)[:-3], INPUT_OVERRUN),
        ("bad_gzip_trailing_junk", GZIP, g(good) + b"\x00abc", TRAILING_BYTES),
        ("bad_gzip_second_member_method", GZIP, g(good) + b"\x1f\x8b\x09" + bytes(7) + b"\x03\x00" + bytes(8),
         BAD_FRAME_HEADER),
        ("bad_gzip_second_member_truncated", GZIP, g(good) + b"\x1f\x8b\x08\x00", INPUT_OVERRUN),
        ("bad_gzip_name_unterminated", GZIP, b"\x1f\x8b\x08\x08" + bytes(6) + b"name" * 5, INPUT_OVERRUN),
        # sizes
        ("bad_short", ZLIB, zlib_wrap(*_fixed([dec[:n - 1]])), SHORT),
        ("bad_gzip_short_members", GZIP, gzip_member(*_fixed([dec[:20]])) + gzip_member(*_fixed([dec[20:39]])), SHORT),
        ("bad_literals_past_size", ZLIB, zlib_wrap(*_fixed([dec + b"!"])), LITERALS_OVERRUN),
        ("bad_stored_past_size", ZLIB, zlib_wrap(*_stored(dec + b"!")), LITERALS_OVERRUN),
        ("bad_match_past_size", ZLIB, zlib_wrap(*_fixed([dec[:36], (5, 4)])), MATCH_OVERRUN),
        ("bad_distance_before_start", ZLIB, zlib_wrap(*_fixed([b"abcd", (36, 5)])), OFFSET_BEFORE_START),
        ("bad_gzip_distance_into_previous_member", GZIP,
         gzip_member(*_fixed([dec[:20]])) + gzip_member(*_fixed([dec[20:24], (16, 8)])), OFFSET_BEFORE_START),
        ("bad_stored_past_input", ZLIB, zlib_wrap(*_stored(dec))[:30], INPUT_OVERRUN),
        # blocks
        ("bad_block_type_3", ZLIB, zlib_wrap(b"\x07\x00", dec), BAD_BLOCK),
        ("bad_stored_nlen", ZLIB, zlib_wrap(b"\x01" + n.to_bytes(2, "little") + n.to_bytes(2, "little") + dec, dec),
         BAD_BLOCK),
        # code descriptions
        ("bad_hlit_287", ZLIB, zlib_wrap(_dynamic_header(287, 1, [4] * 13 + [5] * 6, []).done(), dec), BAD_CODES),
        ("bad_hdist_31", ZLIB, zlib_wrap(_dynamic_header(257, 31, [4] * 13 + [5] * 6, []).done(), dec), BAD_CODES),
        ("bad_code_lengths_incomplete", ZLIB, zlib_wrap(_dynamic_header(257, 1, [4] * 12 + [0] + [5] * 6, []).done()
                                                         + bytes(8), dec), BAD_CODES),
        ("bad_code_lengths_oversubscribed", ZLIB, zlib_wrap(_dynamic_header(257, 1, [4] * 19, []).done() + bytes(8),
                                                            dec), BAD_CODES),
        ("bad_repeat_without_previous", ZLIB, zlib_wrap(_lengths_stream([(16, 2, 0)]), dec), BAD_CODES),
        ("bad_repeat_past_the_end", ZLIB, zlib_wrap(_lengths_stream(tokens([0] * 250) + [(18, 7, 127)]), dec),
         BAD_CODES),
        ("bad_no_end_of_block", ZLIB, zlib_wrap(_lengths_stream(tokens([1, 1] + [0] * 255 + [1])), dec), BAD_CODES),
        ("bad_litlen_oversubscribed", ZLIB, zlib_wrap(_lengths_stream(tokens([1] * 3 + [0] * 253 + [1, 1])), dec),
         BAD_CODES),
        ("bad_litlen_incomplete", ZLIB, zlib_wrap(_lengths_stream(tokens([2] * 2 + [0] * 254 + [2, 0])), dec),
         BAD_CODES),
        ("bad_distance_incomplete", ZLIB, zlib_wrap(_dynamic_header(258, 3, [4] * 13 + [5] * 6, tokens(
            lit + [2, 2, 2, 2])).done() + bytes(16), dec), BAD_CODES),
        # symbols
        ("bad_litlen_286", ZLIB, zlib_wrap(_raw_fixed_symbols([97, 286]), dec), BAD_SYMBOL),
        ("bad_litlen_287", ZLIB, zlib_wrap(_raw_fixed_symbols([97, 287]), dec), BAD_SYMBOL),
        ("bad_distance_30", ZLIB, zlib_wrap(_raw_fixed_symbols([97, 98, (257, 30)]), dec), BAD_SYMBOL),
        ("bad_distance_31", GZIP, gzip_member(_raw_fixed_symbols([97, 98, (257, 31)]), dec), BAD_SYMBOL),
        ("bad_distance_hole", ZLIB, zlib_wrap(_hole_stream(), dec), BAD_SYMBOL),
        ("bad_litlen_hole", ZLIB, zlib_wrap(_litlen_hole_stream(), dec), BAD_SYMBOL),
        ("bad_no_distance_codes_used", ZLIB, zlib_wrap(_empty_distance_stream(), dec), BAD_SYMBOL),
    ]
    out = [Case(name, np.zeros((1, n), np.uint8), (1, n), comp, _hand(data), error=reason)
           for name, comp, data, reason in bad]

    # a Blosc-Zlib stream whose zlib header is wrong (the file's own header passes the host's checks)
    def stream_header(fix):
        def encode(raw, key):
            f = bytearray(_blosc_frame(raw, 1, len(raw), False, "zlib"))
            pos = int.from_bytes(f[16:20], "little") + 4
            f[pos:pos + 2] = fix(bytes(f[pos:pos + 2]))
            return bytes(f)
        return encode

    a = _values("uint8", (1, 16, 32), seed=67)
    for name, fix in (("bad_blosc_zlib_fcheck", lambda h: bytes([h[0], h[1] ^ 1])),
                      ("bad_blosc_zlib_method", lambda h: bytes([0x79, 0x01 + (31 - ((0x79 << 8) + 1) % 31) % 31])),
                      ("bad_blosc_zlib_fdict", lambda h: bytes([0x78, 0x20 + (31 - ((0x78 << 8) + 0x20) % 31) % 31]))):
        out.append(Case(name, a, (1, 16, 32), dict(BLOSC_ZLIB, shuffle=0), stream_header(fix),
                        error=BAD_FRAME_HEADER))
    return out


def _stored(data: bytes) -> tuple[bytes, bytes]:
    w, out = Bits(), bytearray()
    stored_block(w, data, out, True)
    return w.done(), bytes(out)


def _lengths_stream(toks) -> bytes:
    """A final dynamic block of 258 litlen and 1 distance lengths given by ``toks``, then zero bits."""
    return _dynamic_header(258, 1, [4] * 13 + [5] * 6, toks).done() + bytes(16)


def _hole_stream() -> bytes:
    """A single distance code of length 1 (code 0): the block decodes the other code, 1."""
    lit = [0] * 258
    lit[ord("a")], lit[256], lit[257] = 1, 2, 2
    w = _dynamic_header(258, 1, [4] * 13 + [5] * 6, tokens(lit + [1]))
    codes = canonical(lit)
    for _ in range(8):
        w.code(*codes[ord("a")])
    w.code(*codes[257])
    w.bits(1, 1)  # distance code "1": not assigned
    return w.done() + bytes(4)


def _litlen_hole_stream() -> bytes:
    """A single litlen code of length 1 (the end-of-block code 0): the block decodes the code 1."""
    lit = [0] * 257
    lit[256] = 1
    w = _dynamic_header(257, 1, [4] * 13 + [5] * 6, tokens(lit + [1]))
    w.bits(1, 1)
    return w.done() + bytes(4)


def _empty_distance_stream() -> bytes:
    """No distance codes, yet a length symbol follows."""
    lit = [0] * 258
    lit[ord("a")], lit[256], lit[257] = 1, 2, 2
    w = _dynamic_header(258, 1, [4] * 13 + [5] * 6, tokens(lit + [0]))
    codes = canonical(lit)
    w.code(*codes[ord("a")])
    w.code(*codes[257])
    return w.done() + bytes(4)
