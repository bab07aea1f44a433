// decode.cu -- Zarr chunks compressed with Blosc-LZ4 / Blosc-Zstd / Blosc-Zlib / LZ4 / Zstd / Zlib / GZip
// (numcodecs, and the Zarr v3 codecs that write the same streams) decoded on the device.
//
// The chunk files of a pipeline band chunk (Zarr v3: the inner chunks of a shard) cross PCIe as they are on disk;
// six kernels turn them into the pipeline's pitched (bands, win_h, wp) slot:
//   k_crc32c        one warp per file with a CRC-32C trailer (Zarr v3's crc32c codec): checks it, then drops it from
//                   the device copy of the chunk table (decode_crc32c.cuh);
//   k_zarr_index    one thread per Blosc block: walks the block's int32 stream-size prefixes and writes one
//                   descriptor per stream (source range, destination range in the scratch, stored or compressed);
//                   LZ4 streams come first in the descriptor array, Zstd streams after them, Deflate streams last;
//   k_lz4_decode    one warp per LZ4 stream: LZ4 block format into the scratch of decoded, still-shuffled blocks;
//   k_zstd_decode   one warp per Zstd stream: a Zstandard frame into the same scratch (decode_zstd.cuh);
//   k_inflate       one warp per Deflate stream: a zlib stream or gzip file into the same scratch (decode_deflate.cuh);
//   k_zarr_scatter  one thread per chunk element: gathers its bytes from the shuffled block, swaps big-endian
//                   values, applies CF mask-and-scale, and stores it at its true position in the slot.
// The container layout and the shuffle rule are those of io.blosc_decompress, which stays the reference.
// Chunk files are outside input: every read stays inside its file, every write inside its stream's range,
// and a stream that breaks the format sets the caller's error word instead.
#include <cstring>

#include "common.cuh"

namespace xrs {
namespace {

constexpr int kBloscMaxSplits = 16, kBloscMinBufferSize = 128;
constexpr int kMaxChunks = (1 << 24) - 1;  // the error word holds the chunk index in 24 bits
constexpr int kZstdBlockMax = 128 << 10;  // a zstd block's largest decoded size, and its literals'

// a stream of one Blosc block or of a numcodecs lz4 / zstd / zlib / gzip chunk (dsize 0: unused descriptor)
struct StreamDesc {
    int64_t src;    // byte offset in `data`
    int64_t dst;    // byte offset in the scratch
    int32_t csize;  // compressed bytes
    int32_t dsize;  // decoded bytes
    int32_t stored; // csize == dsize: the bytes are copied
    int32_t chunk;  // index in the chunk table (error reports)
};

struct BloscHeader {
    int flags, typesize;
    int64_t nbytes, blocksize, cbytes;
};

__host__ __device__ inline uint32_t le32(const uint8_t *p) {
    return uint32_t(p[0]) | (uint32_t(p[1]) << 8) | (uint32_t(p[2]) << 16) | (uint32_t(p[3]) << 24);
}

__host__ __device__ inline BloscHeader blosc_header(const uint8_t *h) {
    BloscHeader b;
    b.flags = h[2];
    b.typesize = h[3] > 0 ? h[3] : 1;
    b.nbytes = le32(h + 4);
    b.blocksize = le32(h + 8);
    b.cbytes = le32(h + 12);
    return b;
}

// streams per FULL block (io.blosc_decompress: the last, partial block is never split)
__host__ __device__ inline int blosc_full_streams(const BloscHeader &b) {
    const bool split = !(b.flags & 0x10) && b.typesize <= kBloscMaxSplits &&
                       b.blocksize / b.typesize >= kBloscMinBufferSize;
    return split ? b.typesize : 1;
}

// decoded bytes are still byte-shuffled (flag bit 0, typesize > 1; a frame stored whole is not)
__host__ __device__ inline bool blosc_shuffled(const BloscHeader &b) {
    return (b.flags & 0x1) && !(b.flags & 0x2) && b.typesize > 1;
}

__device__ inline void report(uint32_t *err, int chunk, int reason) {
    atomicCAS(err, 0u, (static_cast<uint32_t>(reason) << 24) | static_cast<uint32_t>(chunk + 1));
}

// descriptors of block b of chunk c (one thread)
__device__ inline void index_block(const uint8_t *data, const xrs_zarr_chunk *chunks, int c, int64_t b,
                                   int64_t chunk_bytes, StreamDesc *desc, uint32_t *err) {
    const xrs_zarr_chunk ch = chunks[c];
    StreamDesc d;
    d.chunk = c;
    d.stored = 0;
    if (ch.codec == XRS_CHUNK_LZ4) {  // numcodecs: int32 decoded size, then one LZ4 block
        if (b != 0) return;
        d.src = ch.offset + 4;
        d.csize = static_cast<int32_t>(ch.length - 4);
        d.dst = ch.scratch;
        d.dsize = static_cast<int32_t>(chunk_bytes);
        desc[ch.stream_base] = d;
        return;
    }
    if (ch.codec == XRS_CHUNK_ZSTD || ch.codec == XRS_CHUNK_ZLIB || ch.codec == XRS_CHUNK_GZIP) {  // the whole file
        if (b != 0) return;
        d.src = ch.offset;
        d.csize = static_cast<int32_t>(ch.length);
        d.dst = ch.scratch;
        d.dsize = static_cast<int32_t>(chunk_bytes);
        desc[ch.stream_base] = d;
        return;
    }
    if (ch.codec != XRS_CHUNK_BLOSC) return;
    const BloscHeader h = blosc_header(ch.header);
    if (h.flags & 0x2) {  // the frame is a plain copy of the chunk
        if (b != 0) return;
        d.src = ch.offset + 16;
        d.csize = d.dsize = static_cast<int32_t>(h.nbytes);
        d.dst = ch.scratch;
        d.stored = 1;
        desc[ch.stream_base] = d;
        return;
    }
    const int64_t nblocks = ceil_div(h.nbytes, h.blocksize);
    if (b >= nblocks) return;
    const int slots = blosc_full_streams(h);
    StreamDesc *out = desc + ch.stream_base + b * slots;
    for (int s = 0; s < slots; ++s) {
        StreamDesc e = {};
        e.chunk = c;
        out[s] = e;
    }
    const int64_t bsize = h.nbytes - b * h.blocksize < h.blocksize ? h.nbytes - b * h.blocksize : h.blocksize;
    const int ns = bsize == h.blocksize ? slots : 1;
    const int64_t neblock = bsize / ns;
    const uint8_t *file = data + ch.offset;
    const int64_t len = ch.length;
    if (16 + 4 * (b + 1) > len) {
        report(err, c, XRS_DECODE_BAD_LAYOUT);
        return;
    }
    int64_t pos = static_cast<int32_t>(le32(file + 16 + 4 * b));
    for (int s = 0; s < ns; ++s) {
        if (pos < 16 || pos + 4 > len) {
            report(err, c, XRS_DECODE_BAD_LAYOUT);
            return;
        }
        const int64_t csize = static_cast<int32_t>(le32(file + pos));
        pos += 4;
        if (csize < 0 || pos + csize > len) {
            report(err, c, XRS_DECODE_BAD_LAYOUT);
            return;
        }
        d.src = ch.offset + pos;
        d.csize = static_cast<int32_t>(csize);
        d.dst = ch.scratch + b * h.blocksize + s * neblock;
        d.dsize = static_cast<int32_t>(neblock);
        d.stored = csize == neblock;
        out[s] = d;
        pos += csize;
    }
}

// One thread per Blosc block: x walks the blocks of a chunk, y strides over the chunks (gridDim.y is capped at
// 65535, a call may carry up to 2^24 - 1 files).
__global__ void __launch_bounds__(128) k_zarr_index(const uint8_t *__restrict__ data,
                                                    const xrs_zarr_chunk *__restrict__ chunks, int64_t n_chunks,
                                                    int64_t chunk_bytes, StreamDesc *__restrict__ desc, uint32_t *err) {
    const int64_t b = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    for (int64_t c = blockIdx.y; c < n_chunks; c += gridDim.y)
        index_block(data, chunks, static_cast<int>(c), b, chunk_bytes, desc, err);
}

// adds the extension bytes of a literal or match length (a run of 255s and the byte that ends it); false when the
// input ends inside the run
__device__ inline bool extend(const uint8_t *in, int64_t &ip, int64_t iend, int64_t &len) {
    int x;
    do {
        if (ip >= iend) return false;
        x = __ldg(in + ip++);
        len += x;
    } while (x == 255);
    return true;
}

// One warp per stream.  Every lane parses the tokens itself (the same bytes: broadcast loads) and the warp copies
// literals and matches cooperatively.  Byte k of a match is out[op - off + k % off]: the periodic extension of the
// window the offset points at, so an overlapping match (off < length) needs no rounds -- every source byte was
// final before the match began.  One __syncwarp per sequence publishes the bytes before a match reads them.
__global__ void __launch_bounds__(128) k_lz4_decode(const uint8_t *__restrict__ data, const StreamDesc *__restrict__ desc,
                                                    int64_t n_streams, uint8_t *__restrict__ scratch, uint32_t *err) {
    const int64_t w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) / 32;
    const int lane = threadIdx.x % 32;
    if (w >= n_streams) return;
    const StreamDesc d = desc[w];
    if (d.dsize == 0) return;
    const uint8_t *in = data + d.src;
    uint8_t *out = scratch + d.dst;
    if (d.stored) {
        for (int64_t k = lane; k < d.dsize; k += 32) out[k] = __ldg(in + k);
        return;
    }
    const int64_t iend = d.csize, oend = d.dsize;
    int64_t ip = 0, op = 0;
    int reason = 0;
    while (true) {
        if (ip >= iend) {  // a block ends with a literals-only sequence, never after a match
            reason = XRS_DECODE_INPUT_OVERRUN;
            break;
        }
        const int token = __ldg(in + ip++);
        int64_t lit = token >> 4;
        if (lit == 15 && !extend(in, ip, iend, lit)) {
            reason = XRS_DECODE_INPUT_OVERRUN;
            break;
        }
        if (lit > oend - op || lit > iend - ip) {
            reason = XRS_DECODE_LITERALS_OVERRUN;
            break;
        }
        for (int64_t k = lane; k < lit; k += 32) out[op + k] = __ldg(in + ip + k);
        ip += lit;
        op += lit;
        if (ip == iend) {  // the last sequence: literals only
            if (op != oend) reason = XRS_DECODE_SHORT;
            break;
        }
        if (iend - ip < 2) {
            reason = XRS_DECODE_INPUT_OVERRUN;
            break;
        }
        const int64_t off = __ldg(in + ip) | (__ldg(in + ip + 1) << 8);
        ip += 2;
        if (off == 0) {
            reason = XRS_DECODE_OFFSET_ZERO;
            break;
        }
        if (off > op) {
            reason = XRS_DECODE_OFFSET_BEFORE_START;
            break;
        }
        int64_t ml = (token & 15) + 4;
        if ((token & 15) == 15 && !extend(in, ip, iend, ml)) {
            reason = XRS_DECODE_INPUT_OVERRUN;
            break;
        }
        if (ml > oend - op) {
            reason = XRS_DECODE_MATCH_OVERRUN;
            break;
        }
        __syncwarp();
        const uint8_t *from = out + op - off;
        for (int64_t k = lane; k < ml; k += 32) out[op + k] = from[k < off ? k : k % off];
        op += ml;
    }
    if (reason && lane == 0) report(err, d.chunk, reason);
}

// CRC arithmetic modulo a reflected polynomial (zlib's multmodp / x2nmodp): a * b, and x^(8n).  Poly 0xEDB88320 is
// CRC-32 (gzip members), 0x82F63B78 CRC-32C (the crc32c codec of Zarr v3).
template <uint32_t Poly>
__device__ inline uint32_t crc_mul(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (uint32_t m = 1u << 31; m != 0; m >>= 1) {
        if (a & m) {
            p ^= b;
            if ((a & (m - 1)) == 0) break;
        }
        b = b & 1 ? (b >> 1) ^ Poly : b >> 1;
    }
    return p;
}
template <uint32_t Poly>
__device__ inline uint32_t crc_shift(int64_t n) {
    uint32_t p = 1u << 31, x = 1u << 23;  // x^0, x^8
    for (; n; n >>= 1) {
        if (n & 1) p = crc_mul<Poly>(x, p);
        x = crc_mul<Poly>(x, x);
    }
    return p;
}

// The CRC of buf[0, n) by the whole warp: one contiguous segment a lane through a byte table, the segments' CRCs
// combined as zlib's crc32_combine does.  `table` (256 words) and `part` (32 words) are the warp's shared memory.
template <uint32_t Poly>
__device__ inline uint32_t warp_crc(const uint8_t *buf, int64_t n, uint32_t *table, uint32_t *part, int lane) {
    for (int i = lane; i < 256; i += 32) {
        uint32_t c = static_cast<uint32_t>(i);
        for (int k = 0; k < 8; ++k) c = c & 1 ? (c >> 1) ^ Poly : c >> 1;
        table[i] = c;
    }
    __syncwarp();
    const int64_t seg = (n + 31) / 32, lo = lane * seg < n ? lane * seg : n, hi = lo + seg < n ? lo + seg : n;
    uint32_t c = 0xffffffffu;
    for (int64_t k = lo; k < hi; ++k) c = table[(c ^ buf[k]) & 0xff] ^ (c >> 8);
    part[lane] = ~c;
    __syncwarp();
    uint32_t crc = 0, shift = crc_shift<Poly>(seg);
    for (int s = 0; s < 32; ++s) {
        const int64_t l = s * seg < n ? (s * seg + seg < n ? seg : n - s * seg) : 0;
        crc = crc_mul<Poly>(l == seg ? shift : crc_shift<Poly>(l), crc) ^ part[s];
    }
    __syncwarp();
    return crc;
}

// The CRC-32C check (k_crc32c, launch_crc32c) is compiled by nvcc; a host build of this file compiles it when it
// defines XRS_HOST_CRC32C and leaves it out otherwise (a chunk flagged XRS_CHUNK_CRC32C then fails the call).
#if defined(__CUDACC__) || defined(XRS_HOST_CRC32C)
#define XRS_CRC32C_CHECK 1
#include "decode_crc32c.cuh"
#endif

// The Zstd decoder (k_zstd_decode, launch_zstd) is compiled by nvcc; a host build of this file compiles it when it
// defines XRS_HOST_ZSTD and leaves it out otherwise (a Zstd stream then fails the call).
#if defined(__CUDACC__) || defined(XRS_HOST_ZSTD)
#define XRS_ZSTD_DECODER 1
#include "decode_zstd.cuh"
#endif

// The Deflate decoder (k_inflate, launch_inflate) likewise: a host build compiles it when it defines XRS_HOST_DEFLATE.
#if defined(__CUDACC__) || defined(XRS_HOST_DEFLATE)
#define XRS_DEFLATE_DECODER 1
#include "decode_deflate.cuh"
#endif

struct ScatterGeom {
    int64_t chunk_bytes, chunk_elems, cb, ch, cw;  // chunk shape (bands 1 for 2-D arrays)
    int64_t img_h, img_w, win_j0, win_j1, b0, nb;  // clip: image, slot rows, pipeline bands
    int64_t pitch, band_stride;                    // of the destination, in elements
    int64_t n_chunks;
    uint64_t fill_bits;                            // raw value of a missing chunk (native byte order)
    int32_t big_endian;
};

// chunk-local byte q -> its position in the decoded (still shuffled) chunk
__device__ inline int64_t shuffled_pos(int64_t q, const BloscHeader &h) {
    const int64_t b = q / h.blocksize;
    const int64_t r = q - b * h.blocksize;
    const int64_t rest = h.nbytes - b * h.blocksize;
    const int64_t n = (rest < h.blocksize ? rest : h.blocksize) / h.typesize;
    return r < n * h.typesize ? b * h.blocksize + (r % h.typesize) * n + r / h.typesize : q;
}

template <typename T>
__device__ inline T from_bits(uint64_t bits) {
    T v;
    memcpy(&v, &bits, sizeof(T));
    return v;
}

__device__ inline float quieted(float v) { return __int_as_float(__float_as_int(v) | 0x00400000); }
__device__ inline double quieted(double v) {
    return __longlong_as_double(__double_as_longlong(v) | 0x0008000000000000ll);
}
__device__ inline float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ inline double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ inline float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ inline double add_rn(double a, double b) { return __dadd_rn(a, b); }

// R: stored type (for CF = false only its size matters), D: type written to the slot
template <typename R, typename D, bool CF>
__global__ void __launch_bounds__(256) k_zarr_scatter(const uint8_t *__restrict__ scratch,
                                                      const xrs_zarr_chunk *__restrict__ chunks, ScatterGeom g,
                                                      xrs_zarr_cf cf, D *__restrict__ dst) {
    const int64_t total = g.n_chunks * g.chunk_elems;
    const int64_t plane = g.ch * g.cw;
    for (int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; e < total;
         e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const int64_t c = e / g.chunk_elems, r = e - c * g.chunk_elems;
        const int64_t lb = r / plane, lj = (r - lb * plane) / g.cw, li = r - lb * plane - lj * g.cw;
        const xrs_zarr_chunk &ch = chunks[c];
        const int64_t band = ch.band + lb, row = ch.row + lj, col = ch.col + li;
        if (band < g.b0 || band >= g.b0 + g.nb || row < g.win_j0 || row >= g.win_j1 || row >= g.img_h ||
            col >= g.img_w)
            continue;
        R raw;
        if (ch.codec == XRS_CHUNK_MISSING) {
            raw = from_bits<R>(g.fill_bits);
        } else {
            const BloscHeader h = blosc_header(ch.header);
            const bool shuffled = ch.codec == XRS_CHUNK_BLOSC && blosc_shuffled(h);
            const uint8_t *src = scratch + ch.scratch;
            uint8_t bytes[sizeof(R)];
            for (int k = 0; k < static_cast<int>(sizeof(R)); ++k) {
                const int64_t q = r * static_cast<int64_t>(sizeof(R)) + k;
                bytes[g.big_endian ? sizeof(R) - 1 - k : k] = src[shuffled ? shuffled_pos(q, h) : q];
            }
            memcpy(&raw, bytes, sizeof(R));
        }
        D v;
        if constexpr (CF) {
            v = static_cast<D>(raw);
            for (int k = 0; k < cf.n_fills; ++k)
                if (raw == from_bits<R>(cf.fills[k])) v = std::numeric_limits<D>::quiet_NaN();
            if (v == v) {
                if (cf.has_scale) v = mul_rn(v, static_cast<D>(cf.scale));
                if (cf.has_offset) v = add_rn(v, static_cast<D>(cf.offset));
            } else if (cf.has_scale || cf.has_offset) {
                v = quieted(v);  // x86 arithmetic returns its NaN operand quieted; the GPU's, a canonical NaN
            }
        } else {
            v = raw;
        }
        dst[(band - g.b0) * g.band_stride + (row - g.win_j0) * g.pitch + col] = v;
    }
}

template <typename R, typename D, bool CF>
int launch_scatter(const uint8_t *scratch, const xrs_zarr_chunk *chunks, const ScatterGeom &g, const xrs_zarr_cf &cf,
                   void *dst, cudaStream_t st) {
    const int64_t total = g.n_chunks * g.chunk_elems;
    if (total == 0) return 0;
    const unsigned blocks = static_cast<unsigned>(ceil_div(total, 256) < 148 * 32 ? ceil_div(total, 256) : 148 * 32);
    D *out = static_cast<D *>(dst);
    XRS_TIMED("zarr_scatter", st, k_zarr_scatter<R, D, CF><<<blocks, 256, 0, st>>>(scratch, chunks, g, cf, out));
    XRS_LAUNCH_CHECK("k_zarr_scatter");
    return 0;
}

template <typename R>
int dispatch_cf(const uint8_t *scratch, const xrs_zarr_chunk *chunks, const ScatterGeom &g, const xrs_zarr_cf &cf,
                void *dst, cudaStream_t st) {
    if (cf.out_dtype == XRS_F32) return launch_scatter<R, float, true>(scratch, chunks, g, cf, dst, st);
    if (cf.out_dtype == XRS_F64) return launch_scatter<R, double, true>(scratch, chunks, g, cf, dst, st);
    return fail("xrs_zarr_decode: the CF decoded dtype must be XRS_F32 or XRS_F64");
}

int element_size(int dtype) {
    switch (dtype) {
    case XRS_F64: case XRS_I64: return 8;
    case XRS_F32: case XRS_I32: case XRS_U32: return 4;
    case XRS_U16: case XRS_I16: return 2;
    case XRS_U8: case XRS_I8: return 1;
    default: return 0;
    }
}

// the codec of a table entry without the XRS_CHUNK_CRC32C flag
inline int base_codec(const xrs_zarr_chunk &ch) { return ch.codec & ~XRS_CHUNK_CRC32C; }

// Zstd streams: a numcodecs zstd chunk, or a Blosc frame with the Zstd inner codec that is not stored whole
inline bool zstd_chunk(const xrs_zarr_chunk &ch) {
    const int codec = base_codec(ch);
    return codec == XRS_CHUNK_ZSTD || (codec == XRS_CHUNK_BLOSC && !(ch.header[2] & 0x2) && (ch.header[2] >> 5) == 4);
}

// Deflate streams: a numcodecs zlib or gzip chunk, or a Blosc frame with the Zlib inner codec not stored whole
inline bool deflate_chunk(const xrs_zarr_chunk &ch) {
    const int codec = base_codec(ch);
    return codec == XRS_CHUNK_ZLIB || codec == XRS_CHUNK_GZIP ||
           (codec == XRS_CHUNK_BLOSC && !(ch.header[2] & 0x2) && (ch.header[2] >> 5) == 3);
}

struct StreamPlan {
    int64_t n;           // descriptors: [0, n_lz4) LZ4 or stored, then n_zstd Zstd, then Deflate up to n
    int64_t n_lz4, n_zstd;
    int64_t max_blocks;  // the most Blosc blocks of one chunk
    int64_t scratch;     // bytes: one decoded chunk per file present
    int64_t lit_stride;  // literal buffer of one Zstd stream: min(largest decoded Zstd stream, 128 KiB)
    int64_t n_crc;       // files flagged XRS_CHUNK_CRC32C
};

// Checks the table against the headers it carries and fills stream_base / n_streams / scratch; false on an error,
// reported through fail().
bool plan_streams(xrs_zarr_chunk *chunks, int64_t n_chunks, int64_t chunk_bytes, int64_t data_bytes, StreamPlan *plan) {
    if (n_chunks < 0 || n_chunks > kMaxChunks) return fail("xrs_zarr_decode: bad chunk count"), false;
    if (chunk_bytes <= 0 || chunk_bytes > INT32_MAX)
        return fail("xrs_zarr_decode: a chunk must hold 1 to 2^31 - 1 bytes"), false;
    int64_t n_zstd = 0, n_deflate = 0, largest = 0;
    *plan = StreamPlan{0, 0, 0, 1, 0, 0, 0};
    for (int64_t c = 0; c < n_chunks; ++c) {
        xrs_zarr_chunk &ch = chunks[c];
        const std::string where = "xrs_zarr_decode: chunk " + std::to_string(c) + ": ";
        ch.stream_base = plan->n_lz4;
        ch.n_streams = 0;
        ch.scratch = -1;
        if (ch.codec == XRS_CHUNK_MISSING) continue;
        if (ch.offset < 0 || ch.length < 0 || (data_bytes >= 0 && ch.offset + ch.length > data_bytes))
            return fail(where + "file bytes outside the data buffer"), false;
        // a CRC-32C trailer: the codec applies to the payload in front of it (k_crc32c checks and drops it)
        const int codec = base_codec(ch);
        const bool crc = ch.codec & XRS_CHUNK_CRC32C;
        if (crc && (codec == XRS_CHUNK_MISSING || ch.length < 4))
            return fail(where + "a CRC-32C flag on a missing chunk or on a file shorter than its 4-byte trailer"), false;
        const int64_t length = ch.length - (crc ? 4 : 0);
        plan->n_crc += crc;
        if (codec == XRS_CHUNK_LZ4) {
            if (length < 4 || length - 4 > INT32_MAX || static_cast<int32_t>(le32(ch.header)) != chunk_bytes)
                return fail(where + "numcodecs lz4 size prefix does not match the chunk size"), false;
            ch.n_streams = 1;
        } else if (codec == XRS_CHUNK_ZSTD) {
            if (length < 6 || length > INT32_MAX || le32(ch.header) != 0xFD2FB528u)
                return fail(where + "not a zstd frame"), false;
            ch.n_streams = 1;
            largest = chunk_bytes > largest ? chunk_bytes : largest;
        } else if (codec == XRS_CHUNK_ZLIB) {  // CMF, FLG, at least one byte of Deflate, Adler-32
            const int cmf = ch.header[0], flg = ch.header[1];
            if (length < 7 || length > INT32_MAX || (cmf & 15) != 8 || (cmf >> 4) > 7 ||
                (cmf * 256 + flg) % 31 || (flg & 0x20))
                return fail(where + "not a zlib stream without a preset dictionary"), false;
            ch.n_streams = 1;
        } else if (codec == XRS_CHUNK_GZIP) {  // a 10-byte header, at least one byte of Deflate, CRC-32, ISIZE
            if (length < 19 || length > INT32_MAX || ch.header[0] != 0x1f || ch.header[1] != 0x8b ||
                ch.header[2] != 8)
                return fail(where + "not a gzip member of method 8"), false;
            ch.n_streams = 1;
        } else if (codec == XRS_CHUNK_BLOSC) {
            const BloscHeader h = blosc_header(ch.header);
            if (length < 16 || ch.header[0] != 2 || h.nbytes != chunk_bytes || h.cbytes > length)
                return fail(where + "not a Blosc-1 frame of the chunk's size"), false;
            if (h.flags & 0x2) {
                if (16 + h.nbytes > length) return fail(where + "truncated Blosc frame"), false;
                ch.n_streams = 1;
            } else {
                if (h.flags & 0x4) return fail(where + "bit-shuffled Blosc frames are not decoded on the device"), false;
                if ((h.flags >> 5) != 1 && (h.flags >> 5) != 3 && (h.flags >> 5) != 4)
                    return fail(where + "the Blosc frame's inner codec is not LZ4, Zlib or Zstd"), false;
                if (h.blocksize <= 0) return fail(where + "Blosc block size 0"), false;
                const int64_t nblocks = ceil_div(h.nbytes, h.blocksize);
                ch.n_streams = static_cast<int32_t>(nblocks * blosc_full_streams(h));
                if (nblocks > plan->max_blocks) plan->max_blocks = nblocks;
                if ((h.flags >> 5) == 4) {  // a full block's streams, and the last, partial block (one stream)
                    const int64_t full = h.nbytes >= h.blocksize ? h.blocksize / blosc_full_streams(h) : 0;
                    const int64_t part = h.nbytes % h.blocksize;
                    largest = full > largest ? full : largest;
                    largest = part > largest ? part : largest;
                }
            }
        } else {
            return fail(where + "unknown codec " + std::to_string(ch.codec)), false;
        }
        int64_t &count = zstd_chunk(ch) ? n_zstd : deflate_chunk(ch) ? n_deflate : plan->n_lz4;
        ch.stream_base = count;
        count += ch.n_streams;
        ch.scratch = plan->scratch;
        plan->scratch += chunk_bytes;
    }
    for (int64_t c = 0; c < n_chunks; ++c) {
        xrs_zarr_chunk &ch = chunks[c];
        if (ch.codec == XRS_CHUNK_MISSING) continue;
        if (zstd_chunk(ch)) ch.stream_base += plan->n_lz4;
        else if (deflate_chunk(ch)) ch.stream_base += plan->n_lz4 + n_zstd;
    }
    plan->n_zstd = n_zstd;
    plan->n = plan->n_lz4 + n_zstd + n_deflate;
    plan->lit_stride = largest < kZstdBlockMax ? largest : kZstdBlockMax;
    if (ceil_div(plan->n_lz4, 4) > INT32_MAX) return fail("xrs_zarr_decode: more LZ4 streams than one launch can take"), false;
    if (n_zstd > INT32_MAX) return fail("xrs_zarr_decode: more Zstd streams than one launch can take"), false;
    if (n_deflate > INT32_MAX) return fail("xrs_zarr_decode: more Deflate streams than one launch can take"), false;
    return true;
}

int64_t align256(int64_t n) { return (n + 255) / 256 * 256; }

// workspace: the chunk table, the descriptors, the scratch and, with Zstd streams, their literal buffers
struct Workspace {
    int64_t table, desc, scratch, lits;
    Workspace(const StreamPlan &plan, int64_t n_chunks)
        : table(align256(n_chunks * static_cast<int64_t>(sizeof(xrs_zarr_chunk)))),
          desc(align256(plan.n * static_cast<int64_t>(sizeof(StreamDesc)))),
          scratch(plan.n_zstd > 0 ? align256(plan.scratch) : plan.scratch),
          lits(plan.n_zstd * plan.lit_stride) {}
    int64_t total() const { return table + desc + scratch + lits; }
};

}  // namespace
}  // namespace xrs

extern "C" {

int64_t xrs_zarr_decode_workspace_bytes(xrs_zarr_chunk *chunks_host, int64_t n_chunks, int64_t chunk_bands,
                                        int64_t chunk_h, int64_t chunk_w, int32_t dtype) {
    const int64_t chunk_bytes = chunk_bands * chunk_h * chunk_w * xrs::element_size(dtype);
    xrs::StreamPlan plan;
    if (!xrs::plan_streams(chunks_host, n_chunks, chunk_bytes, -1, &plan)) return -1;
    return xrs::Workspace(plan, n_chunks).total();
}

int xrs_zarr_decode(const void *data, int64_t data_bytes, xrs_zarr_chunk *chunks_host, int64_t n_chunks,
                    int64_t chunk_bands, int64_t chunk_h, int64_t chunk_w, int32_t dtype, int32_t big_endian,
                    uint64_t fill_bits, const xrs_zarr_cf *cf_host, int64_t img_h, int64_t img_w, void *dst,
                    int64_t dst_pitch, int64_t dst_band_stride, int64_t win_j0, int64_t win_j1, int64_t b0, int64_t nb,
                    void *workspace, int64_t workspace_bytes, uint32_t *error_word, void *stream) {
    using namespace xrs;
    const int isz = element_size(dtype);
    if (isz == 0) return fail("xrs_zarr_decode: unsupported dtype code " + std::to_string(dtype));
    if (chunk_bands <= 0 || chunk_h <= 0 || chunk_w <= 0) return fail("xrs_zarr_decode: bad chunk shape");
    if (!error_word || (n_chunks > 0 && (!data || !dst || !workspace)))
        return fail("xrs_zarr_decode: null buffer");
    const int64_t chunk_bytes = chunk_bands * chunk_h * chunk_w * isz;
    StreamPlan plan;
    if (!plan_streams(chunks_host, n_chunks, chunk_bytes, data_bytes, &plan)) return 1;
    const int64_t n_streams = plan.n, n_zstd = plan.n_zstd, n_deflate = plan.n - plan.n_lz4 - plan.n_zstd;
    const Workspace ws(plan, n_chunks);
    if (workspace_bytes < ws.total())
        return fail("xrs_zarr_decode: workspace smaller than xrs_zarr_decode_workspace_bytes");
    if (n_chunks == 0) return 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    auto *chunks = static_cast<xrs_zarr_chunk *>(workspace);
    auto *desc = reinterpret_cast<StreamDesc *>(static_cast<uint8_t *>(workspace) + ws.table);
    uint8_t *scratch = static_cast<uint8_t *>(workspace) + ws.table + ws.desc;
    const auto *bytes = static_cast<const uint8_t *>(data);
    XRS_CUDA(cudaMemcpyAsync(chunks, chunks_host, n_chunks * sizeof(xrs_zarr_chunk), cudaMemcpyHostToDevice, st));
    if (plan.n_crc > 0) {
#ifdef XRS_CRC32C_CHECK
        const int rc = launch_crc32c(bytes, chunks, n_chunks, error_word, st);
        if (rc) return rc;
#else
        return fail("xrs_zarr_decode: this build has no CRC-32C check");
#endif
    }
    if (n_streams > 0) {
        const dim3 grid(static_cast<unsigned>(ceil_div(plan.max_blocks, 128)),
                        static_cast<unsigned>(n_chunks < 65535 ? n_chunks : 65535));  // the kernel strides over y
        XRS_TIMED("zarr_index", st,
                  k_zarr_index<<<grid, 128, 0, st>>>(bytes, chunks, n_chunks, chunk_bytes, desc, error_word));
        XRS_LAUNCH_CHECK("k_zarr_index");
    }
    if (plan.n_lz4 > 0) {
        const unsigned warps4 = static_cast<unsigned>(ceil_div(plan.n_lz4, 4));  // 4 warps of 32 per block
        XRS_TIMED("zarr_lz4_decode", st,
                  k_lz4_decode<<<warps4, 128, 0, st>>>(bytes, desc, plan.n_lz4, scratch, error_word));
        XRS_LAUNCH_CHECK("k_lz4_decode");
    }
    if (n_zstd > 0) {
#ifdef XRS_ZSTD_DECODER
        const int rc = launch_zstd(bytes, desc + plan.n_lz4, n_zstd, scratch, scratch + ws.scratch, plan.lit_stride,
                                   error_word, st);
        if (rc) return rc;
#else
        return fail("xrs_zarr_decode: this build has no Zstd decoder");
#endif
    }
    if (n_deflate > 0) {
#ifdef XRS_DEFLATE_DECODER
        const int rc = launch_inflate(bytes, chunks, desc + plan.n_lz4 + n_zstd, n_deflate, scratch, error_word, st);
        if (rc) return rc;
#else
        return fail("xrs_zarr_decode: this build has no Deflate decoder");
#endif
    }
    ScatterGeom g;
    g.chunk_bytes = chunk_bytes;
    g.chunk_elems = chunk_bands * chunk_h * chunk_w;
    g.cb = chunk_bands;
    g.ch = chunk_h;
    g.cw = chunk_w;
    g.img_h = img_h;
    g.img_w = img_w;
    g.win_j0 = win_j0;
    g.win_j1 = win_j1;
    g.b0 = b0;
    g.nb = nb;
    g.pitch = dst_pitch;
    g.band_stride = dst_band_stride;
    g.n_chunks = n_chunks;
    g.fill_bits = fill_bits;
    g.big_endian = big_endian;
    xrs_zarr_cf cf = {};
    if (cf_host) {
        cf = *cf_host;
        if (cf.n_fills < 0 || cf.n_fills > XRS_ZARR_CF_MAX_FILLS) return fail("xrs_zarr_decode: bad CF fill count");
        XRS_DISPATCH_DTYPE(dtype, R, return dispatch_cf<R>(scratch, chunks, g, cf, dst, st));
    }
    switch (isz) {
    case 1: return launch_scatter<uint8_t, uint8_t, false>(scratch, chunks, g, cf, dst, st);
    case 2: return launch_scatter<uint16_t, uint16_t, false>(scratch, chunks, g, cf, dst, st);
    case 4: return launch_scatter<uint32_t, uint32_t, false>(scratch, chunks, g, cf, dst, st);
    default: return launch_scatter<uint64_t, uint64_t, false>(scratch, chunks, g, cf, dst, st);
    }
}

}  // extern "C"
