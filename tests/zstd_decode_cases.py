"""Case table of the device decode of Zstd-compressed Zarr chunks (numcodecs ``zstd`` and Blosc-Zstd; csrc/decode.cu,
``k_zstd_decode``), shared by the host build (test_host_zstd_decode.py) and the GPU (test_zstd_decode_gpu.py).

Cases are :class:`zarr_decode_cases.Case`.  Frames come from pyarrow's ``zstd`` codec at levels -5, 1, 3, 9 and 19,
and from the system libzstd through ctypes for what pyarrow cannot set: the content checksum, frames without a
content size and small window logs (a window descriptor, blocks of the window's size).  Blosc-Zstd frames come from
test_host_io's assembler.  Frames with header variants, RLE / raw / Huffman literals and hand-written sequences are
assembled here from RFC 8878; the sequences use RLE tables, so their bitstream holds only the extra bits.  Malformed
files name the reason ``xrs_zarr_decode`` must report (``include/xrs.h``, enum xrs_decode_error); the host path
rejects each of them too.  :func:`walk` reads a frame's block, literals and sequence-table types from the headers
alone, to show what the corpus exercises."""

from __future__ import annotations

import ctypes
import functools

import numpy as np

from .test_host_io import _blosc_frame
from .zarr_decode_cases import Case, _values

(OFFSET_ZERO, OFFSET_BEFORE_START, LITERALS_OVERRUN, MATCH_OVERRUN, INPUT_OVERRUN, SHORT, BAD_FRAME_HEADER, BAD_BLOCK,
 BAD_LITERALS, BAD_HUFFMAN, BAD_FSE, BAD_SEQUENCES, TRAILING_BYTES, CHECKSUM) = range(2, 16)

ZSTD = {"id": "zstd", "level": 3}
BLOSC_ZSTD = {"id": "blosc", "cname": "zstd", "clevel": 5, "shuffle": 1, "blocksize": 0}
MAGIC = b"\x28\xb5\x2f\xfd"
LEVELS = (-5, 1, 3, 9, 19)


def pyarrow_zstd(raw: bytes, level: int = 3) -> bytes:
    import pyarrow as pa

    return pa.Codec("zstd", compression_level=level).compress(raw).to_pybytes()


@functools.lru_cache(maxsize=1)
def libzstd():
    """The system libzstd (``None`` if this machine has none)."""
    try:
        lib = ctypes.CDLL("libzstd.so.1")
    except OSError:
        return None
    lib.ZSTD_createCCtx.restype = ctypes.c_void_p
    lib.ZSTD_freeCCtx.argtypes = [ctypes.c_void_p]
    lib.ZSTD_CCtx_setParameter.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    lib.ZSTD_CCtx_setParameter.restype = ctypes.c_size_t
    lib.ZSTD_compress2.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t]
    lib.ZSTD_compress2.restype = ctypes.c_size_t
    lib.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    lib.ZSTD_compressBound.restype = ctypes.c_size_t
    lib.ZSTD_isError.argtypes = [ctypes.c_size_t]
    return lib


LIBZSTD_MISSING = "libzstd.so.1 cannot be loaded through ctypes on this machine: its cases are skipped"


def libzstd_frame(raw: bytes, level: int = 3, checksum: bool = False, content_size: bool = True,
                  window_log: int | None = None) -> bytes:
    """One frame from libzstd's ZSTD_compress2 with the given parameters (ZSTD_c_* of zstd.h)."""
    lib = libzstd()
    cctx = lib.ZSTD_createCCtx()
    try:
        for param, value in ((100, level), (200, int(content_size)), (201, int(checksum))) + \
                ((((101, window_log),) if window_log else ())):
            assert not lib.ZSTD_isError(lib.ZSTD_CCtx_setParameter(cctx, param, value))
        cap = lib.ZSTD_compressBound(len(raw))
        dst = ctypes.create_string_buffer(cap)
        n = lib.ZSTD_compress2(cctx, dst, cap, raw, len(raw))
        assert not lib.ZSTD_isError(n)
        return dst.raw[:n]
    finally:
        lib.ZSTD_freeCCtx(cctx)


# ---- hand assembly (RFC 8878) ----

def frame(blocks: list[bytes], size: int | None, fcs_bytes: int = 1, window: int | None = None, dict_id: bytes = b"",
          checksum: bool = False, fhd_or: int = 0) -> bytes:
    """A frame header (single segment unless ``window`` gives a window descriptor; ``size`` None: no content
    size) followed by ``blocks`` and, with ``checksum``, a placeholder the caller fills."""
    single = window is None
    fcs_flag = {None: 0, 1: 0, 2: 1, 4: 2, 8: 3}[None if size is None else fcs_bytes]
    fhd = (fcs_flag << 6) | (single << 5) | (checksum << 2) | {0: 0, 1: 1, 2: 2, 4: 3}[len(dict_id)] | fhd_or
    out = MAGIC + bytes([fhd]) + (b"" if single else bytes([window])) + dict_id
    if size is not None:
        out += (size - 256 if fcs_bytes == 2 else size).to_bytes(fcs_bytes, "little")
    return out + b"".join(blocks)


def block(kind: int, content: bytes, last: bool, size: int | None = None) -> bytes:
    """A block header (kind 0 raw, 1 RLE, 2 compressed; ``size`` defaults to the content's) and its content."""
    n = len(content) if size is None else size
    return ((n << 3) | (kind << 1) | int(last)).to_bytes(3, "little") + content


def _lit_header(kind: int, n: int) -> bytes:
    if n < 32:
        return bytes([(n << 3) | kind])
    if n < 4096:
        return ((n << 4) | (1 << 2) | kind).to_bytes(2, "little")
    return ((n << 4) | (3 << 2) | kind).to_bytes(3, "little")


def raw_literals(lit: bytes) -> bytes:
    return _lit_header(0, len(lit)) + lit


def rle_literals(byte: int, n: int) -> bytes:
    return _lit_header(1, n) + bytes([byte])


def backward(fields) -> bytes:
    """A backward bitstream whose first read field is the first of ``fields`` ((bits, value) pairs), end mark set."""
    acc, nbits = 0, 0
    for nb, v in fields:
        assert 0 <= v < (1 << nb) or nb == v == 0
        acc, nbits = (acc << nb) | v, nbits + nb
    return ((1 << nbits) | acc).to_bytes(nbits // 8 + 1, "little")


# a two-symbol Huffman tree given directly: one weight (1) for byte 0, the last (1) implied for byte 1: 1-bit codes
HUF_TREE_01 = bytes([128, 0x10])


def huffman_literals(lit: bytes, streams: int, treeless: bool = False, tree: bytes = HUF_TREE_01,
                     spare_bits: int = 0) -> bytes:
    """Compressed (or treeless) literals of bytes 0 / 1 under the tree above, in 1 or 4 streams; ``spare_bits``
    extra bits in the last stream make it malformed."""
    assert set(lit) <= {0, 1}
    if streams == 1:
        parts = [lit]
    else:
        seg = (len(lit) + 3) // 4
        parts = [lit[:seg], lit[seg:2 * seg], lit[2 * seg:3 * seg], lit[3 * seg:]]
    enc = [backward([(1, b) for b in p] + ([(spare_bits, 0)] if spare_bits and k == len(parts) - 1 else []))
           for k, p in enumerate(parts)]
    body = (b"" if treeless else tree) + (b"".join(len(e).to_bytes(2, "little") for e in enc[:3]) if streams == 4
                                          else b"") + b"".join(enc)
    kind, sf = (3 if treeless else 2), (0 if streams == 1 else 1)
    h = kind | (sf << 2) | (len(lit) << 4) | (len(body) << 14)
    return h.to_bytes(3, "little") + body


_LL_BITS = [0] * 16 + [1, 1, 1, 1, 2, 2, 3, 3, 4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16]
_ML_BITS = [0] * 32 + [1, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16]


def rle_sequences(codes, seqs, spare_bits: int = 0, modes: int | None = None) -> bytes:
    """A sequences section with RLE tables of (LL, OF, ML) ``codes``; ``seqs`` of (LL extra, OF extra, ML extra)
    values.  States read no bits, so the bitstream is the extra bits: offset, match length, literal length."""
    llc, ofc, mlc = codes
    fields = []
    for lle, ofe, mle in seqs:
        fields += [(ofc, ofe), (_ML_BITS[mlc], mle), (_LL_BITS[llc], lle)]
    fields += [(spare_bits, 0)] if spare_bits else []
    n = len(seqs)
    head = bytes([n]) if n < 128 else bytes([128 + (n >> 8), n & 255])
    return head + bytes([0x54 if modes is None else modes, llc, ofc, mlc]) + backward(fields)


# ---- header-level walker ----

def walk(data: bytes) -> list[dict]:
    """The blocks of the zstd frame ``data`` (skippable frames after it are ignored): block type, and for compressed
    blocks the literals type, Huffman stream count and the LL / OF / ML table modes (0 predefined, 1 RLE, 2 FSE,
    3 repeat), read from the headers alone."""
    fhd = data[4]
    single, did, fcs_flag = (fhd >> 5) & 1, fhd & 3, fhd >> 6
    p = 5 + (not single) + (0, 1, 2, 4)[did] + ((1 if single else 0), 2, 4, 8)[fcs_flag]
    out = []
    while True:
        bh = int.from_bytes(data[p:p + 3], "little")
        p += 3
        last, kind, size = bh & 1, (bh >> 1) & 3, bh >> 3
        b = {"type": kind}
        if kind == 2:
            blk = data[p:p + size]
            lt, sf = blk[0] & 3, (blk[0] >> 2) & 3
            b["literals"] = lt
            if lt < 2:
                lh = {0: 1, 1: 2, 2: 1, 3: 3}[sf]
                h = int.from_bytes(blk[:lh], "little")
                n = h >> 3 if lh == 1 else h >> 4
                q = lh + (n if lt == 0 else 1)
            else:
                lh = 3 if sf < 2 else sf + 2
                bits = (10, 10, 14, 18)[sf]
                h = int.from_bytes(blk[:lh], "little")
                q = lh + ((h >> (4 + bits)) & ((1 << bits) - 1))
                b["streams"] = 1 if sf == 0 else 4
            c0 = blk[q]
            nseq = c0 if c0 < 128 else (((c0 - 128) << 8) + blk[q + 1] if c0 < 255 else
                                        blk[q + 1] + (blk[q + 2] << 8) + 0x7F00)
            if nseq:
                m = blk[q + (1 if c0 < 128 else 2 if c0 < 255 else 3)]
                b["modes"] = (m >> 6, (m >> 4) & 3, (m >> 2) & 3)
        p += 1 if kind == 1 else size
        out.append(b)
        if last:
            return out


# ---- the table ----

def _per_chunk(fn):
    return lambda raw, key: fn(raw)


def _blosc_zstd(typesize, blocksize, shuffle=True, dont_split=False, store_streams=False, missing=()):
    def encode(raw, key):
        if key in missing:
            return None
        return _blosc_frame(raw, typesize, blocksize, shuffle, "zstd", dont_split=dont_split,
                            store_streams=store_streams)
    return encode


def _blosc_restream(typesize, blocksize, enc):
    """A Blosc-Zstd frame whose streams ``enc`` compresses (test_host_io's assembler, streams stored, then
    re-encoded; a stream that does not shrink stays stored)."""
    def encode(raw, key):
        f = bytearray(_blosc_frame(raw, typesize, blocksize, True, "zstd", store_streams=True))
        nblocks = -(-len(raw) // blocksize)
        body = bytearray()
        starts = []
        head = 16 + 4 * nblocks
        for b in range(nblocks):
            pos = int.from_bytes(f[16 + 4 * b:20 + 4 * b], "little")
            end = int.from_bytes(f[20 + 4 * b:24 + 4 * b], "little") if b + 1 < nblocks else len(f)
            starts.append(head + len(body))
            while pos < end:
                n = int.from_bytes(f[pos:pos + 4], "little")
                part = bytes(f[pos + 4:pos + 4 + n])
                comp = enc(part)
                comp = comp if len(comp) < n else part
                body += len(comp).to_bytes(4, "little") + comp
                pos += 4 + n
        total = head + len(body)
        return bytes(f[:12]) + total.to_bytes(4, "little") + b"".join(s.to_bytes(4, "little") for s in starts) + \
            bytes(body)
    return encode


def _skippable(data: bytes, n: int = 5) -> bytes:
    return data + (0x184D2A53).to_bytes(4, "little") + n.to_bytes(4, "little") + bytes(range(n))


def _hand(data: bytes):
    return lambda raw, key: data


def cases() -> list[Case]:
    out = []
    nine = ("float32", "float64", "uint8", "int8", "uint16", "int16", "int32", "uint32", "int64")
    for k, dt in enumerate(nine):
        isz = np.dtype(dt).itemsize
        a = _values(dt, (3, 21, 37), seed=40 + isz)
        out.append(Case(f"{dt}_zstd_split", a, (2, 8, 17), BLOSC_ZSTD, _blosc_zstd(isz, 128 * isz), b0=1, nb=2,
                        window=(3, 19)))
        out.append(Case(f"{dt}_zstd_dont_split", a, (2, 8, 17), BLOSC_ZSTD, _blosc_zstd(isz, 128 * isz,
                                                                                       dont_split=True)))
        out.append(Case(f"{dt}_zstd_no_shuffle", a, (2, 8, 17), dict(BLOSC_ZSTD, shuffle=0),
                        _blosc_zstd(isz, 64 * isz, shuffle=False)))
        level = LEVELS[k % len(LEVELS)]
        out.append(Case(f"{dt}_zstd", a[0], (8, 16), dict(ZSTD, level=level),
                        _per_chunk(lambda raw, lv=level: pyarrow_zstd(raw, lv))))
    f32 = _values("float32", (5, 30, 45), seed=43)
    # one multi-block frame per level: 2 x 200 x 128 float32 = 200 KiB chunks, a smooth field with noise
    rng = np.random.default_rng(44)
    field = (np.sin(np.arange(400 * 128) / 300.0).reshape(4, 100, 128) * 1000).astype(np.float32)
    field += rng.integers(0, 4, field.shape).astype(np.float32)
    big = np.concatenate([field, field[::-1]], axis=1)  # (4, 200, 128)
    for level in LEVELS:
        out.append(Case(f"level_{level}_multi_block", big, (2, 200, 128), dict(ZSTD, level=level),
                        _per_chunk(lambda raw, lv=level: pyarrow_zstd(raw, lv))))
    out.append(Case("level_19_text_like", _values("uint8", (300, 700), seed=45), (150, 700), dict(ZSTD, level=19),
                    _per_chunk(lambda raw: pyarrow_zstd(raw, 19))))
    out += [
        Case("random_bytes_raw_blocks", np.random.default_rng(46).integers(0, 256, (2, 300, 600), dtype=np.uint8),
             (1, 300, 600), ZSTD, _per_chunk(pyarrow_zstd)),
        Case("constant_rle_blocks", np.full((2, 400, 500), 0x0707, np.int16), (1, 400, 500), ZSTD,
             _per_chunk(pyarrow_zstd)),
        Case("skippable_frames_after", f32, (2, 16, 32), ZSTD, _per_chunk(lambda r: _skippable(_skippable(
            pyarrow_zstd(r), 0), 9))),
        Case("blosc_zstd_stored_streams", f32, (2, 16, 32), BLOSC_ZSTD, _blosc_zstd(4, 1024, store_streams=True)),
        Case("blosc_zstd_skippable", f32, (2, 16, 32), BLOSC_ZSTD,
             _blosc_restream(4, 1024, lambda p: _skippable(pyarrow_zstd(p)))),
        Case("zstd_missing_chunks", f32, (2, 16, 32), ZSTD,
             lambda raw, key: None if key in ("0.0.1", "2.1.0") else pyarrow_zstd(raw)),
        Case("blosc_zstd_missing_chunks", f32, (2, 16, 32), BLOSC_ZSTD, _blosc_zstd(4, 1024, missing=("1.0.0",))),
        Case("zstd_ragged_edges_window", f32, (2, 16, 32), ZSTD, _per_chunk(pyarrow_zstd), b0=2, nb=3,
             window=(7, 29)),
        Case("zstd_band_depth_3_of_2", f32, (3, 16, 32), ZSTD, _per_chunk(pyarrow_zstd), b0=1, nb=2),
        Case("blosc_zstd_band_depth_3_of_4", f32, (3, 16, 32), BLOSC_ZSTD, _blosc_zstd(4, 1024), b0=1, nb=4),
        Case("blosc_zstd_tail_not_an_element", _values("uint8", (2, 11, 23), seed=47), (1, 5, 9), BLOSC_ZSTD,
             _blosc_zstd(4, 16)),
    ]
    for dt in (">f4", ">i2", ">f8", ">u4"):
        a = _values(np.dtype(dt).newbyteorder("="), (3, 21, 37), seed=48).astype(dt)
        isz = a.dtype.itemsize
        out.append(Case(f"zstd_big_endian_{dt[1:]}", a, (2, 8, 17), ZSTD, _per_chunk(pyarrow_zstd)))
        out.append(Case(f"blosc_zstd_big_endian_{dt[1:]}", a, (2, 8, 17), BLOSC_ZSTD,
                        _blosc_zstd(isz, 128 * isz)))
    cf = [("uint16", {"scale_factor": 0.01, "add_offset": -5.0, "_FillValue": 3, "missing_value": [8, 65535]}),
          ("int16", {"scale_factor": 2.5e-4, "add_offset": 1.25, "_FillValue": -32768}),
          ("float32", {"scale_factor": 3.0, "add_offset": 0.5, "_FillValue": "NaN", "missing_value": [3.0]})]
    for k, (dt, attrs) in enumerate(cf):
        isz = np.dtype(dt).itemsize
        a = _values(dt, (3, 21, 37), seed=50 + k)
        out.append(Case(f"zstd_cf_{k}_{dt}", a, (2, 8, 17), ZSTD,
                        lambda raw, key: None if key == "1.1.0" else pyarrow_zstd(raw), attrs=attrs, b0=1, nb=2))
        out.append(Case(f"blosc_zstd_cf_{k}_{dt}", a, (2, 8, 17), BLOSC_ZSTD, _blosc_zstd(isz, 128 * isz),
                        attrs=attrs))
    if libzstd() is not None:
        out += [
            Case("libzstd_checksum", big, (2, 200, 128), ZSTD, _per_chunk(lambda r: libzstd_frame(r, 3, True))),
            Case("libzstd_window_log_10", f32, (2, 16, 32), ZSTD,
                 _per_chunk(lambda r: libzstd_frame(r, 5, True, window_log=10))),
            Case("libzstd_window_log_12_multi_block", big, (2, 200, 128), ZSTD,
                 _per_chunk(lambda r: libzstd_frame(r, 19, window_log=12))),
            Case("blosc_libzstd_no_content_size", f32, (2, 16, 32), BLOSC_ZSTD,
                 _blosc_restream(4, 2048, lambda p: libzstd_frame(p, 3, True, content_size=False))),
            Case("blosc_libzstd_no_content_size_window_10", big, (2, 200, 128), BLOSC_ZSTD,
                 _blosc_restream(4, 1 << 16, lambda p: libzstd_frame(p, 9, False, False, window_log=10))),
        ]
    out += hand_cases()
    out += malformed_cases()
    return out


def _uint8(data: bytes) -> np.ndarray:
    return np.frombuffer(data, np.uint8).reshape(1, -1)


_LL_BASE = list(range(16)) + [16, 18, 20, 22, 24, 28, 32, 40, 48] + [1 << k for k in range(6, 17)]


def _offset(reps, llv, ofv):
    """The offset of an offset value and the repeat offsets after it (RFC 8878 3.1.2.5)."""
    if ofv > 3:
        return ofv - 3, [ofv - 3, reps[0], reps[1]]
    idx = ofv - (0 if llv == 0 else 1)
    off = reps[0] - 1 if idx == 3 else reps[idx]
    if idx == 0:
        return off, reps
    return off, ([off, reps[0], reps[2]] if idx == 1 else [off, reps[0], reps[1]])


def _continue(prev: bytes, lit: bytes, ops) -> bytes:
    """``prev`` followed by literals + (literal length, offset, match length) sequences, copied byte by byte."""
    out, lp = bytearray(prev), 0
    for ll, off, ml in ops:
        out += lit[lp:lp + ll]
        lp += ll
        for _ in range(ml):
            out.append(out[len(out) - off])
    return bytes(out + lit[lp:])


def hand_cases() -> list[Case]:
    rng = np.random.default_rng(60)
    lit = lambda n: rng.integers(0, 256, n, dtype=np.uint8).tobytes()  # noqa: E731
    out = []

    def add(name, dec, data):
        out.append(Case(name, _uint8(dec), (1, len(dec)), ZSTD, _hand(data)))

    def fcs(n):
        return 1 if n < 256 else 2

    a = lit(200)
    add("hand_fcs_1_raw", a, frame([block(0, a, True)], len(a)))
    b = bytes([9]) * 300 + lit(700)
    add("hand_fcs_2_rle_raw", b, frame([block(1, b[:1], False, 300), block(0, b[300:], True)], len(b), 2))
    c = lit(5000)  # window descriptor 0x10: 4 KiB, blocks up to 4 KiB
    add("hand_fcs_4_window", c, frame([block(0, c[:3000], False), block(0, c[3000:], True)], len(c), 4, window=0x10))
    d = lit(1000) + bytes(70000)  # window 0x38: 128 KiB
    add("hand_fcs_8_window", d, frame([block(0, d[:1000], False), block(1, b"\x00", True, 70000)], len(d), 8,
                                      window=0x38))
    # compressed blocks: RLE literals and raw literals (1-, 2- and 3-byte headers), RLE-table sequences.  Literal
    # length code 17 (18 + 1 bit), offset code 4 (values 16 ... 31: offsets 13 ... 28), match length code 0 (3)
    seq1 = rle_sequences((17, 4, 0), [(0, 3, 0), (1, 7, 0), (0, 0, 0)])
    ops1 = [(18, 16, 3), (19, 20, 3), (18, 13, 3)]
    e = _continue(b"", bytes([5]) * 60, ops1)
    add("hand_rle_literals", e, frame([block(2, rle_literals(5, 60) + seq1, True)], len(e)))
    la = lit(20)  # literal length code 10, offset code 2 (value 7: offset 4)
    f = _continue(b"", la, [(10, 4, 3)])
    # a compressed block may not exceed the window: these take a window descriptor (8 KiB)
    add("hand_raw_literals_20", f, frame([block(2, raw_literals(la) + rle_sequences((10, 2, 0), [(0, 3, 0)]), True)],
                                         len(f), 4, window=0x18))
    for n in (100, 5000):
        la = lit(n)
        f = _continue(b"", la, ops1)
        add(f"hand_raw_literals_{n}", f, frame([block(2, raw_literals(la) + seq1, True)], len(f), 4, window=0x18))
    # Huffman literals (bytes 0 / 1) in 1 and 4 streams, then treeless in 1 and 4 streams; literals only
    bits = lambda n: rng.integers(0, 2, n, dtype=np.uint8).tobytes()  # noqa: E731
    h1, h4, t1, t4 = bits(40), bits(300), bits(90), bits(1000)
    blocks = [block(2, huffman_literals(h1, 1) + b"\x00", False), block(2, huffman_literals(h4, 4) + b"\x00", False),
              block(2, huffman_literals(t1, 1, treeless=True) + b"\x00", False),
              block(2, huffman_literals(t4, 4, treeless=True) + b"\x00", True)]
    g = h1 + h4 + t1 + t4
    add("hand_huffman_streams", g, frame(blocks, len(g), 2))
    # repeat offsets, one sequences section per block (they carry across blocks): after literals, offset values
    # 1 / 2 / 3 select Repeat_Offset1 / 2 / 3; with no literals, 1 -> Repeat_Offset2, 2 -> Repeat_Offset3,
    # 3 -> Repeat_Offset1 - 1.  Offset code 0 gives value 1, code 1 values 2 and 3.
    sections = [
        ((20, 0, 0), [(0, 0, 0), (0, 0, 0)]),  # literal length code 20: 24 + 2 bits
        ((20, 1, 0), [(1, 0, 0), (2, 1, 0)]),
        ((0, 1, 0), [(0, 1, 0), (0, 0, 0)]),   # literal length 0
        ((0, 0, 0), [(0, 0, 0), (0, 0, 0)]),
        ((16, 5, 3), [(1, 5, 0), (0, 17, 0)]),  # new offsets 34 and 46, match length 6
    ]
    la = lit(400)
    reps, dec, lp, blocks = [1, 4, 8], b"", 0, []
    for k, ((llc, ofc, mlc), seqs) in enumerate(sections):
        ops = []
        for lle, ofe, _ in seqs:
            llv = _LL_BASE[llc] + lle
            off, reps = _offset(reps, llv, (1 << ofc) + ofe)
            assert 0 < off <= len(dec) + sum(o[0] + o[2] for o in ops) + llv
            ops.append((llv, off, mlc + 3))
        n_lit = sum(o[0] for o in ops) + 2
        bl = la[lp:lp + n_lit]
        lp += n_lit
        dec = _continue(dec, bl, ops)
        blocks.append(block(2, raw_literals(bl) + rle_sequences((llc, ofc, mlc), seqs), k == len(sections) - 1))
    add("hand_repeat_offsets", dec, frame(blocks, len(dec), fcs(len(dec))))
    return out


def malformed_cases() -> list[Case]:
    out = []
    rng = np.random.default_rng(70)
    n = 4000

    def add(name, data, reason, size=n):
        out.append(Case(name, np.zeros((1, size), np.uint8), (1, size), ZSTD, _hand(data), error=reason))

    good = pyarrow_zstd((np.sin(np.arange(n) / 7.0) * 50 + 100).astype(np.uint8).tobytes(), 3)
    blocks = walk(good)
    assert blocks[0]["type"] == 2 and blocks[0].get("modes")
    hs = _header_size(good)
    # truncations: after the frame header, inside the block header, inside the block, at the block's end
    add("bad_truncated_after_header", good[:hs], INPUT_OVERRUN)
    add("bad_truncated_block_header", good[:hs + 2], INPUT_OVERRUN)
    add("bad_truncated_block", good[:len(good) - 5], INPUT_OVERRUN)
    add("bad_trailing_garbage", good + b"\x01\x02\x03", TRAILING_BYTES)
    add("bad_trailing_short_skippable", good + (0x184D2A50).to_bytes(4, "little") + (9).to_bytes(4, "little") + b"x",
        TRAILING_BYTES)
    bad = bytearray(good)
    bad[4] |= 0x08
    add("bad_reserved_bit", bytes(bad), BAD_FRAME_HEADER)
    a = bytes(range(100))
    # hand frames of 100 bytes
    m = 100

    def add_hand(name, blocks_, reason, **kw):  # a 1 KiB window: blocks may be larger than the frame
        add(name, frame(blocks_, m, **dict(dict(fcs_bytes=4, window=0x00), **kw)), reason, size=m)

    add_hand("bad_dictionary_id", [block(0, a, True)], BAD_FRAME_HEADER, dict_id=b"\x07")
    add_hand("bad_reserved_block_type", [block(3, a, True)], BAD_BLOCK)
    # compressed blocks above the window (1 KiB) and above 128 KiB (window 256 KiB): literals only
    add("bad_block_above_window", frame([block(2, raw_literals(bytes(2000)) + b"\x00", True)], 2000, 2, window=0x00),
        BAD_BLOCK, size=2000)
    big = (128 << 10) + 1
    add("bad_block_above_128k", frame([block(2, raw_literals(bytes(big)) + b"\x00", True)], big, 4, window=0x40),
        BAD_BLOCK, size=big)
    add("bad_literals_above_window", frame([block(2, rle_literals(0, 1500) + b"\x00", True)], 1500, 2, window=0x00),
        BAD_LITERALS, size=1500)
    add_hand("bad_raw_block_past_size", [block(0, a + b"!", True)], LITERALS_OVERRUN)
    add_hand("bad_short", [block(0, a[:60], True)], SHORT)
    chk = frame([block(0, a, True)], m, checksum=True)
    add("bad_checksum", chk + b"\x00\x00\x00\x00", CHECKSUM, size=m)
    add("bad_truncated_checksum", chk + b"\x00\x00", INPUT_OVERRUN, size=m)
    # sequences: literal length code 17 (18 + 1 bit), offset code 4 (offsets 13 ... 28), match length code 0 (3)
    lit20 = a[:20]
    add_hand("bad_offset_before_start", [block(2, raw_literals(lit20) + rle_sequences((17, 4, 0), [(0, 15, 0)]),
                                               True)], OFFSET_BEFORE_START)
    add("bad_match_past_end", frame([block(2, raw_literals(lit20) + rle_sequences((17, 4, 47), [(0, 3, 2000)]),
                                           True)], 30), MATCH_OVERRUN, size=30)
    add_hand("bad_bits_left_over", [block(2, raw_literals(lit20) + rle_sequences((17, 4, 0), [(0, 3, 0)],
                                                                                spare_bits=3), True)], BAD_SEQUENCES)
    add_hand("bad_literals_past_section", [block(2, raw_literals(lit20) + rle_sequences((19, 4, 0), [(1, 3, 0)]),
                                                 True)], LITERALS_OVERRUN)
    add_hand("bad_repeat_offset_zero", [block(2, raw_literals(lit20) + rle_sequences((0, 1, 0), [(0, 1, 0)]),
                                              True)], OFFSET_ZERO)
    add_hand("bad_offset_code_out_of_range", [block(2, raw_literals(lit20) + rle_sequences((17, 32, 0),
                                                                                          [(0, 0, 0)]), True)],
             BAD_SEQUENCES)
    add_hand("bad_repeat_table_without_one", [block(2, raw_literals(lit20) + rle_sequences((17, 4, 0), [(0, 3, 0)],
                                                                                          modes=0xFC), True)],
             BAD_SEQUENCES)
    add_hand("bad_reserved_mode_bits", [block(2, raw_literals(lit20) + rle_sequences((17, 4, 0), [(0, 3, 0)],
                                                                                    modes=0x55), True)],
             BAD_SEQUENCES)
    add_hand("bad_no_sequences_then_bytes", [block(2, raw_literals(a) + b"\x00\x00", True)], BAD_SEQUENCES)
    # an FSE description with an accuracy log above the table's (LL: 9; low nibble 15 -> 20)
    fse = bytes([1]) + bytes([0x80]) + bytes([0x0F, 0xFF]) + b"\x01"
    add_hand("bad_fse_accuracy_log", [block(2, raw_literals(lit20) + fse, True)], BAD_FSE)
    # an FSE description that runs out of symbols before its probabilities sum (all 36 LL symbols at 1 of 64)
    add_hand("bad_fse_probabilities", [block(2, raw_literals(lit20) + bytes([1, 0x80]) + _fse_ones(36, 6) + b"\x01",
                                             True)], BAD_FSE)
    # a Huffman tree that does not form a tree: weights 2, 2, 1 (sum 5: 8 - 5 is not a power of 2)
    bad_tree = bytes([130, 0x22, 0x10])
    add_hand("bad_huffman_tree", [block(2, huffman_literals(bytes(100), 1, tree=bad_tree) + b"\x00", True)],
             BAD_HUFFMAN)
    add_hand("bad_huffman_truncated", [block(2, (2 | (100 << 4) | (1 << 14)).to_bytes(3, "little") + b"\xff", True)],
             BAD_HUFFMAN)  # a direct tree of 128 weights in a 1-byte section
    bits = rng.integers(0, 2, 100, dtype=np.uint8).tobytes()
    add_hand("bad_huffman_bits_left_over", [block(2, huffman_literals(bits, 4, spare_bits=5) + b"\x00", True)],
             BAD_LITERALS)
    add_hand("bad_treeless_first", [block(2, huffman_literals(bits, 1, treeless=True) + b"\x00", True)],
             BAD_LITERALS)
    add_hand("bad_literals_section_past_block", [block(2, _lit_header(0, 90) + a[:50], True)], BAD_LITERALS)
    # corrupted tables of a real frame: the first FSE description's accuracy log
    fse_at = _first_fse_description(good)
    if fse_at is not None:
        bad = bytearray(good)
        bad[fse_at] |= 0x0F
        add("bad_fse_in_libzstd_frame", bytes(bad), BAD_FSE)
    return out


def _fse_ones(n_sym: int, log: int) -> bytes:
    """The count bits of an FSE description with ``n_sym`` symbols of probability 1 (count field 2), accuracy log
    ``log`` in the header byte before it: they sum to n_sym, short of 2^log when n_sym < 2^log."""
    assert n_sym < (1 << log)
    bits, nbits = log - 5, 4
    remaining, threshold, nb = (1 << log) + 1, 1 << log, log + 1
    for _ in range(n_sym):
        mx = 2 * threshold - 1 - remaining
        v = 2
        if v < mx:
            bits |= v << nbits
            nbits += nb - 1
        else:
            bits |= (v if v < threshold else v + mx) << nbits
            nbits += nb
        remaining -= 1
        while remaining < threshold:
            nb -= 1
            threshold >>= 1
    return bits.to_bytes((nbits + 7) // 8, "little")


def _header_size(data: bytes) -> int:
    fhd = data[4]
    single, did, fcs_flag = (fhd >> 5) & 1, fhd & 3, fhd >> 6
    return 5 + (not single) + (0, 1, 2, 4)[did] + ((1 if single else 0), 2, 4, 8)[fcs_flag]


def _first_fse_description(data: bytes) -> int | None:
    """Offset of the first FSE table description of the frame's first block, None if it has none."""
    p = _header_size(data)
    blk = data[p + 3:]
    lt, sf = blk[0] & 3, (blk[0] >> 2) & 3
    if lt < 2:
        lh = {0: 1, 1: 2, 2: 1, 3: 3}[sf]
        h = int.from_bytes(blk[:lh], "little")
        n = h >> 3 if lh == 1 else h >> 4
        q = lh + (n if lt == 0 else 1)
    else:
        lh = 3 if sf < 2 else sf + 2
        bits = (10, 10, 14, 18)[sf]
        q = lh + ((int.from_bytes(blk[:lh], "little") >> (4 + bits)) & ((1 << bits) - 1))
    c0 = blk[q]
    q += 1 if c0 < 128 else 2 if c0 < 255 else 3
    modes = blk[q]
    q += 1
    for shift in (6, 4, 2):
        m = (modes >> shift) & 3
        if m == 2:
            return p + 3 + q
        q += 1 if m == 1 else 0
    return None
