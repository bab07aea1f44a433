// decode_zstd.cuh -- Zstandard frames (RFC 8878, without dictionaries) decoded by one warp each; part of decode.cu.
//
// k_zstd_decode takes the Zstd descriptors k_zarr_index wrote (a numcodecs zstd chunk, or one stream of a
// Blosc-Zstd frame) and decodes each frame into its range of the scratch.  The whole decoded frame lies there, so the
// window is the frame itself and a match may not reach before its first byte.  Serial work -- table descriptions,
// decode tables, the FSE state walk of the sequences -- runs on lane 0 and is published through shared memory; the
// four Huffman streams of a literals section decode on lanes 0-3; the lanes copy raw blocks, literals and matches
// cooperatively.  A block's literals go to a per-stream literal buffer in the workspace (at most min(decoded size of
// the largest Zstd stream of the call, 128 KiB) a stream).  Every read stays inside the stream's bytes, every write
// inside its scratch range or literal buffer, every table index inside its table; a stream that breaks the format sets
// the caller's error word.  Every loop is bounded by the input or by counts checked against the decoded size.

// Counts repeat-offset events (a test hook: the host build of this file defines it; on the device it is nothing).
#ifndef XRS_ZSTD_COUNT
#define XRS_ZSTD_COUNT(event) ((void)0)
#endif

constexpr int kHufLogMax = 11, kLLLogMax = 9, kMLLogMax = 9, kOFLogMax = 8, kHwLogMax = 6;
constexpr int kLLMax = 35, kMLMax = 52, kOFMax = 31, kHwMax = 15;
constexpr int kZstdBatch = 32;  // sequences lane 0 decodes before the warp executes them

// FSE decode entry: symbol (bits 0-7), bits to read (8-15), base of the next state (16-31)
struct ZstdShared {
    uint32_t ll[1 << kLLLogMax], ml[1 << kMLLogMax], of[1 << kOFLogMax], hw[1 << kHwLogMax];
    uint16_t huf[1 << kHufLogMax];  // Huffman decode entry: symbol (bits 0-7), code length (8-15)
    int16_t norm[64];
    uint16_t next[64];
    uint8_t weights[256];
    int32_t op[kZstdBatch], lp[kZstdBatch], ll_len[kZstdBatch], ml_len[kZstdBatch], off[kZstdBatch];
    uint64_t acc[4];
    int32_t v[8];  // values lane 0 (or lanes 0-3) publish to the warp
};

__device__ inline int highbit32(uint32_t v) { return 31 - __clz(static_cast<int>(v)); }  // v > 0

__device__ inline uint32_t le_bytes(const uint8_t *p, int n) {  // n <= 4
    uint32_t v = 0;
    for (int k = 0; k < n; ++k) v |= static_cast<uint32_t>(__ldg(p + k)) << (8 * k);
    return v;
}

// A zstd bitstream read backwards (RFC 8878 4.1, 4.2.2): in[0, n), its last byte carries the end mark, the first bit
// read is the one below the mark.  Bits below the stream's start read as 0 and drive `pos` negative: the callers check.
struct RevBits {
    const uint8_t *in;
    int64_t pos;  // unread bits: [0, pos)
    int64_t wlo;  // `win` holds bits [wlo, wlo + 64)
    uint64_t win;

    __device__ bool init(const uint8_t *p, int64_t n) {
        in = p;
        if (n < 1 || __ldg(p + n - 1) == 0) return false;
        pos = 8 * (n - 1) + highbit32(__ldg(p + n - 1));
        refill();
        return true;
    }
    __device__ void refill() {
        const int64_t hi = (pos + 7) >> 3;  // bytes [hi - 8, hi) hold bits [pos - 57, pos) at least
        win = 0;
        for (int k = 0; k < 8; ++k) {
            const int64_t b = hi - 8 + k;
            if (b >= 0) win |= static_cast<uint64_t>(__ldg(in + b)) << (8 * k);
        }
        wlo = 8 * (hi - 8);
    }
    __device__ uint32_t peek(int k) {  // 1 <= k <= 32
        if (pos - k < wlo) refill();
        return static_cast<uint32_t>((win >> (pos - k - wlo)) & ((1ull << k) - 1));
    }
    __device__ uint32_t read(int k) {  // 0 <= k <= 32
        if (k == 0) return 0;
        const uint32_t v = peek(k);
        pos -= k;
        return v;
    }
};

// k bits (k <= 16) at bit `bit` of the forward little-endian bitstream in[0, n); bits past the end read as 0
__device__ inline uint32_t fwd_bits(const uint8_t *in, int64_t n, int64_t bit, int k) {
    uint32_t v = 0;
    for (int b = 0; b < 4; ++b) {
        const int64_t i = (bit >> 3) + b;
        if (i < n) v |= static_cast<uint32_t>(__ldg(in + i)) << (8 * b);
    }
    return (v >> (bit & 7)) & ((1u << k) - 1);
}

// FSE table description (RFC 8878 4.1.1) at in[0, n) into norm[]: returns the bytes it takes, -1 if malformed
__device__ inline int64_t fse_read_counts(const uint8_t *in, int64_t n, int max_log, int max_sym, int16_t *norm,
                                          int *log, int *n_sym) {
    if (n < 1) return -1;
    const int al = (__ldg(in) & 15) + 5;
    if (al > max_log) return -1;
    int64_t bit = 4;
    int remaining = (1 << al) + 1, threshold = 1 << al, nbits = al + 1, s = 0;
    bool prev0 = false;
    while (remaining > 1 && s <= max_sym) {
        if (prev0) {  // 2-bit repeat flags: more symbols of probability 0
            int n0 = s;
            while (true) {
                const int r = fwd_bits(in, n, bit, 2);
                bit += 2;
                n0 += r;
                if (r != 3 || n0 > max_sym) break;
            }
            if (n0 > max_sym) return -1;
            while (s < n0) norm[s++] = 0;
        }
        const int max = 2 * threshold - 1 - remaining;
        int count;
        if (static_cast<int>(fwd_bits(in, n, bit, nbits - 1)) < max) {
            count = fwd_bits(in, n, bit, nbits - 1);
            bit += nbits - 1;
        } else {
            count = fwd_bits(in, n, bit, nbits);
            if (count >= threshold) count -= max;
            bit += nbits;
        }
        --count;  // -1: "less than 1", one cell at the table's end
        remaining -= count < 0 ? -count : count;
        norm[s++] = static_cast<int16_t>(count);
        prev0 = count == 0;
        while (remaining < threshold) {
            --nbits;
            threshold >>= 1;
        }
        if (bit > 8 * n) return -1;
    }
    if (remaining != 1 || bit > 8 * n) return -1;
    *log = al;
    *n_sym = s;
    return (bit + 7) >> 3;
}

// FSE decode table from norm[0, n_sym) (RFC 8878 4.1.1, "FSE table"); false if the counts do not tile the table
__device__ inline bool fse_build(const int16_t *norm, int n_sym, int log, uint32_t *table, uint16_t *next) {
    const int size = 1 << log;
    int high = size - 1;
    for (int s = 0; s < n_sym; ++s) {
        if (norm[s] == -1) {
            if (high < 0) return false;
            table[high--] = static_cast<uint32_t>(s);
            next[s] = 1;
        } else {
            next[s] = static_cast<uint16_t>(norm[s] < 0 ? 0 : norm[s]);
        }
    }
    const int step = (size >> 1) + (size >> 3) + 3, mask = size - 1;
    int pos = 0;
    for (int s = 0; s < n_sym; ++s)
        for (int i = 0; i < norm[s]; ++i) {
            table[pos] = static_cast<uint32_t>(s);
            do pos = (pos + step) & mask;
            while (pos > high);
        }
    if (pos != 0) return false;
    for (int u = 0; u < size; ++u) {
        const int s = table[u] & 0xff;
        const uint32_t ns = next[s]++;
        const int nb = log - highbit32(ns);
        table[u] = static_cast<uint32_t>(s) | (static_cast<uint32_t>(nb) << 8) | (((ns << nb) - size) << 16);
    }
    return true;
}

// predefined distributions (RFC 8878 3.1.1.3.2.2): literal lengths (kind 0), match lengths (1), offsets (2)
__device__ inline int predefined_count(int kind, int s) {
    if (kind == 0)
        return s == 0 ? 4 : s == 1 ? 3 : s <= 12 ? 2 : s <= 15 ? 1 : s <= 24 ? 2 : s == 25 ? 3 : s == 26 ? 2
               : s <= 31 ? 1 : -1;
    if (kind == 1) return s == 0 ? 1 : s == 1 ? 4 : s == 2 ? 3 : s <= 8 ? 2 : s <= 45 ? 1 : -1;
    return s <= 5 ? 1 : s <= 8 ? 2 : s <= 23 ? 1 : -1;
}

// baselines and extra bits of literal-length and match-length codes (RFC 8878 3.1.1.3.2.1.1)
__device__ inline int ll_bits(int c) { return c < 16 ? 0 : c < 20 ? 1 : c < 22 ? 2 : c < 24 ? 3 : c == 24 ? 4 : c - 19; }
__device__ inline int ll_base(int c) {
    return c < 16 ? c : c < 20 ? 16 + 2 * (c - 16) : c < 22 ? 24 + 4 * (c - 20) : c < 24 ? 32 + 8 * (c - 22)
           : c == 24 ? 48 : 1 << (c - 19);
}
__device__ inline int ml_bits(int c) {
    return c < 32 ? 0 : c < 36 ? 1 : c < 38 ? 2 : c < 40 ? 3 : c < 42 ? 4 : c == 42 ? 5 : c - 36;
}
__device__ inline int ml_base(int c) {
    return c < 32 ? c + 3 : c < 36 ? 35 + 2 * (c - 32) : c < 38 ? 43 + 4 * (c - 36) : c < 40 ? 51 + 8 * (c - 38)
           : c < 42 ? 67 + 16 * (c - 40) : c == 42 ? 99 : (1 << (c - 36)) + 3;
}

// Huffman tree description (RFC 8878 4.2.1) at in[0, n) into sm.huf; returns the bytes it takes (-1: malformed) and
// the table's log in *max_bits.  Lane 0.
__device__ inline int64_t huf_read_table(const uint8_t *in, int64_t n, ZstdShared &sm, int *max_bits) {
    if (n < 1) return -1;
    const int hb = __ldg(in);
    int nw = 0;
    int64_t used;
    if (hb >= 128) {  // direct: 4-bit weights, two a byte
        nw = hb - 127;
        used = 1 + (nw + 1) / 2;
        if (used > n) return -1;
        for (int k = 0; k < nw; ++k) {
            const int b = __ldg(in + 1 + k / 2);
            sm.weights[k] = static_cast<uint8_t>(k % 2 ? b & 15 : b >> 4);
        }
    } else {  // FSE-compressed weights, two interleaved states
        used = 1 + hb;
        if (used > n) return -1;
        int log, n_sym;
        const int64_t desc = fse_read_counts(in + 1, hb, kHwLogMax, kHwMax, sm.norm, &log, &n_sym);
        if (desc < 0 || !fse_build(sm.norm, n_sym, log, sm.hw, sm.next)) return -1;
        RevBits br;
        if (!br.init(in + 1 + desc, hb - desc)) return -1;
        uint32_t s1 = br.read(log), s2 = br.read(log);
        while (true) {  // each state emits its symbol, then reads its next state; the stream ends by overflowing
            if (nw > 253) return -1;
            sm.weights[nw++] = static_cast<uint8_t>(sm.hw[s1] & 0xff);
            s1 = (sm.hw[s1] >> 16) + br.read((sm.hw[s1] >> 8) & 0xff);
            if (br.pos < 0) {
                sm.weights[nw++] = static_cast<uint8_t>(sm.hw[s2] & 0xff);
                break;
            }
            if (nw > 253) return -1;
            sm.weights[nw++] = static_cast<uint8_t>(sm.hw[s2] & 0xff);
            s2 = (sm.hw[s2] >> 16) + br.read((sm.hw[s2] >> 8) & 0xff);
            if (br.pos < 0) {
                sm.weights[nw++] = static_cast<uint8_t>(sm.hw[s1] & 0xff);
                break;
            }
        }
    }
    int rank[kHufLogMax + 2] = {};
    uint32_t total = 0;
    for (int k = 0; k < nw; ++k) {
        if (sm.weights[k] > kHufLogMax) return -1;
        ++rank[sm.weights[k]];
        total += sm.weights[k] ? 1u << (sm.weights[k] - 1) : 0u;
    }
    if (total == 0) return -1;
    const int mb = highbit32(total) + 1;
    if (mb > kHufLogMax) return -1;
    const uint32_t rest = (1u << mb) - total;
    if (rest & (rest - 1)) return -1;
    const int last = highbit32(rest) + 1;  // the implied weight of the last symbol
    sm.weights[nw] = static_cast<uint8_t>(last);
    ++rank[last];
    if (rank[1] < 2 || (rank[1] & 1)) return -1;
    int start[kHufLogMax + 2];
    for (int w = 1, p = 0; w <= mb; ++w) {
        start[w] = p;
        p += rank[w] << (w - 1);
    }
    for (int s = 0; s <= nw; ++s) {
        const int w = sm.weights[s];
        if (w == 0) continue;
        const uint16_t e = static_cast<uint16_t>(s | ((mb + 1 - w) << 8));
        for (int k = 0; k < (1 << (w - 1)); ++k) sm.huf[start[w] + k] = e;
        start[w] += 1 << (w - 1);
    }
    *max_bits = mb;
    return used;
}

// `count` literals of one Huffman stream in[0, n) into out; false unless the stream holds exactly them
__device__ inline bool huf_stream(const uint8_t *in, int64_t n, uint8_t *out, int64_t count, const uint16_t *table,
                                  int max_bits) {
    RevBits br;
    if (!br.init(in, n)) return false;
    for (int64_t k = 0; k < count; ++k) {
        const uint16_t e = table[br.peek(max_bits)];
        out[k] = static_cast<uint8_t>(e & 0xff);
        br.pos -= e >> 8;
        if (br.pos < 0) return false;
    }
    return br.pos == 0;
}

// one of the three sequence tables from its mode (RFC 8878 3.1.1.3.2.2) at in[*p, e); 0 or the reason.  Lane 0.
__device__ inline int seq_table(const uint8_t *in, int64_t *p, int64_t e, int mode, int kind, ZstdShared &sm,
                                uint32_t *table, int *log, bool *have) {
    const int max_sym = kind == 0 ? kLLMax : kind == 1 ? kMLMax : kOFMax;
    const int max_log = kind == 0 ? kLLLogMax : kind == 1 ? kMLLogMax : kOFLogMax;
    if (mode == 0) {  // predefined
        const int n_sym = max_sym + 1 - (kind == 2 ? kOFMax - 28 : 0);
        for (int s = 0; s < n_sym; ++s) sm.norm[s] = static_cast<int16_t>(predefined_count(kind, s));
        *log = kind == 2 ? 5 : 6;
        fse_build(sm.norm, n_sym, *log, table, sm.next);
    } else if (mode == 1) {  // RLE: one symbol, no bits
        if (*p >= e) return XRS_DECODE_BAD_SEQUENCES;
        const int s = __ldg(in + (*p)++);
        if (s > max_sym) return XRS_DECODE_BAD_SEQUENCES;
        table[0] = static_cast<uint32_t>(s);
        *log = 0;
    } else if (mode == 2) {  // FSE table description
        int n_sym;
        const int64_t used = fse_read_counts(in + *p, e - *p, max_log, max_sym, sm.norm, log, &n_sym);
        if (used < 0 || !fse_build(sm.norm, n_sym, *log, table, sm.next)) return XRS_DECODE_BAD_FSE;
        *p += used;
    } else if (!*have) {  // repeat: the previous block's table
        return XRS_DECODE_BAD_SEQUENCES;
    }
    *have = true;
    return 0;
}

// XXH64 (seed 0) of out[0, n): lanes 0-3 run the four accumulators over 32-byte stripes, lane 0 the rest
__device__ inline uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
constexpr uint64_t kP1 = 11400714785074694791ull, kP2 = 14029467366897019727ull, kP3 = 1609587929392839161ull,
                   kP4 = 9650029242287828579ull, kP5 = 2870177450012600261ull;
__device__ inline uint64_t xxh_round(uint64_t acc, uint64_t in) { return rotl64(acc + in * kP2, 31) * kP1; }
__device__ inline uint64_t le64(const uint8_t *p) {
    uint64_t v = 0;
    for (int k = 0; k < 8; ++k) v |= static_cast<uint64_t>(p[k]) << (8 * k);
    return v;
}
__device__ inline uint32_t xxh64_low32(const uint8_t *out, int64_t n, ZstdShared &sm, int lane) {
    const int64_t stripes = n / 32;
    if (lane < 4) {
        uint64_t v = lane == 0 ? kP1 + kP2 : lane == 1 ? kP2 : lane == 2 ? 0 : 0 - kP1;
        for (int64_t s = 0; s < stripes; ++s) v = xxh_round(v, le64(out + 32 * s + 8 * lane));
        sm.acc[lane] = v;
    }
    __syncwarp();
    uint64_t h;
    if (stripes > 0) {
        h = rotl64(sm.acc[0], 1) + rotl64(sm.acc[1], 7) + rotl64(sm.acc[2], 12) + rotl64(sm.acc[3], 18);
        for (int k = 0; k < 4; ++k) h = (h ^ xxh_round(0, sm.acc[k])) * kP1 + kP4;
    } else {
        h = kP5;
    }
    h += static_cast<uint64_t>(n);
    int64_t p = 32 * stripes;
    for (; p + 8 <= n; p += 8) h = rotl64(h ^ xxh_round(0, le64(out + p)), 27) * kP1 + kP4;
    if (p + 4 <= n) {
        uint64_t v = 0;
        for (int k = 0; k < 4; ++k) v |= static_cast<uint64_t>(out[p + k]) << (8 * k);
        h = rotl64(h ^ (v * kP1), 23) * kP2 + kP3;
        p += 4;
    }
    for (; p < n; ++p) h = rotl64(h ^ (out[p] * kP5), 11) * kP1;
    h ^= h >> 33;
    h *= kP2;
    h ^= h >> 29;
    h *= kP3;
    h ^= h >> 32;
    return static_cast<uint32_t>(h);
}

// The frame in[0, n) into out[0, dsize), by the whole warp (every branch below is taken by all lanes alike);
// returns 0 or the reason.
__device__ inline int zstd_frame(const uint8_t *in, int64_t n, uint8_t *out, int64_t dsize, uint8_t *lbuf,
                                 ZstdShared &sm, int lane) {
    // frame header (RFC 8878 3.1.1.1)
    if (n < 5) return XRS_DECODE_INPUT_OVERRUN;
    if (le_bytes(in, 4) != 0xFD2FB528u) return XRS_DECODE_BAD_FRAME_HEADER;
    const int fhd = __ldg(in + 4);
    const int fcs_flag = fhd >> 6, single = (fhd >> 5) & 1, checksum = (fhd >> 2) & 1, did_flag = fhd & 3;
    if (fhd & 0x8) return XRS_DECODE_BAD_FRAME_HEADER;
    const int did_bytes = did_flag == 3 ? 4 : did_flag, fcs_bytes = fcs_flag == 0 ? single : 1 << fcs_flag;
    int64_t p = 5 + !single + did_bytes + fcs_bytes;
    if (p > n) return XRS_DECODE_INPUT_OVERRUN;
    int64_t window = 0;
    if (!single) {
        const int wd = __ldg(in + 5), wlog = 10 + (wd >> 3);
        if (wlog > 31) return XRS_DECODE_BAD_FRAME_HEADER;
        window = (1ll << wlog) + ((1ll << wlog) >> 3) * (wd & 7);
    }
    if (le_bytes(in + 5 + !single, did_bytes) != 0) return XRS_DECODE_BAD_FRAME_HEADER;  // dictionaries: not here
    if (fcs_bytes) {
        const uint8_t *f = in + 5 + !single + did_bytes;
        uint64_t fcs = fcs_bytes == 8 ? le_bytes(f, 4) | (static_cast<uint64_t>(le_bytes(f + 4, 4)) << 32)
                                      : le_bytes(f, fcs_bytes) + (fcs_bytes == 2 ? 256 : 0);
        if (fcs != static_cast<uint64_t>(dsize)) return XRS_DECODE_BAD_FRAME_HEADER;
        if (single) window = dsize;
    }
    const int64_t block_max = window < kZstdBlockMax ? window : kZstdBlockMax;

    int64_t op = 0;
    bool have_huf = false, have[3] = {false, false, false};
    int huf_bits = 0, log_ll = 0, log_ml = 0, log_of = 0;
    uint32_t rep[3] = {1, 4, 8};  // lane 0's
    while (true) {  // blocks (RFC 8878 3.1.1.2)
        if (p + 3 > n) return XRS_DECODE_INPUT_OVERRUN;
        const uint32_t bh = le_bytes(in + p, 3);
        p += 3;
        const int last = bh & 1, type = (bh >> 1) & 3;
        const int64_t bsize = bh >> 3;
        // a compressed block may not exceed Block_Maximum_Size; raw and RLE blocks are bounded by the decoded size
        if (type == 3 || (type == 2 && bsize > block_max)) return XRS_DECODE_BAD_BLOCK;
        if (type == 1) {  // RLE: one byte, bsize times
            if (p + 1 > n) return XRS_DECODE_INPUT_OVERRUN;
            if (bsize > dsize - op) return XRS_DECODE_LITERALS_OVERRUN;
            const uint8_t b = __ldg(in + p);
            for (int64_t k = lane; k < bsize; k += 32) out[op + k] = b;
            p += 1;
            op += bsize;
        } else if (bsize > n - p) {
            return XRS_DECODE_INPUT_OVERRUN;
        } else if (type == 0) {  // raw
            if (bsize > dsize - op) return XRS_DECODE_LITERALS_OVERRUN;
            for (int64_t k = lane; k < bsize; k += 32) out[op + k] = __ldg(in + p + k);
            p += bsize;
            op += bsize;
        } else {  // compressed: literals section (3.1.1.3.1), then sequences section (3.1.1.3.2)
            const uint8_t *blk = in + p;
            const int64_t be = bsize;
            p += bsize;
            const int b0 = be > 0 ? __ldg(blk) : 0, ltype = b0 & 3, sf = (b0 >> 2) & 3;
            if (be < 1) return XRS_DECODE_BAD_LITERALS;
            int64_t lh, lsize, lcsize = 0;
            int streams = 1;
            if (ltype < 2) {
                lh = sf == 1 ? 2 : sf == 3 ? 3 : 1;
                if (lh > be) return XRS_DECODE_BAD_LITERALS;
                const uint32_t h = le_bytes(blk, static_cast<int>(lh));
                lsize = lh == 1 ? (h >> 3) : (h >> 4);
            } else {
                lh = sf < 2 ? 3 : sf + 2;
                if (lh > be) return XRS_DECODE_BAD_LITERALS;
                const int bits = sf < 2 ? 10 : sf == 2 ? 14 : 18;
                const uint64_t h = lh == 5 ? le_bytes(blk, 4) | (static_cast<uint64_t>(__ldg(blk + 4)) << 32)
                                           : le_bytes(blk, static_cast<int>(lh));
                lsize = static_cast<int64_t>((h >> 4) & ((1u << bits) - 1));
                lcsize = static_cast<int64_t>((h >> (4 + bits)) & ((1u << bits) - 1));
                streams = sf == 0 ? 1 : 4;
            }
            if (lsize > block_max || (streams == 4 && lsize < 6)) return XRS_DECODE_BAD_LITERALS;
            if (lsize > dsize - op) return XRS_DECODE_LITERALS_OVERRUN;
            const uint8_t *lit = lbuf;  // where the block's literals are read from
            int64_t q = lh;           // the sequences section's start in blk
            if (ltype == 0) {
                if (lsize > be - lh) return XRS_DECODE_BAD_LITERALS;
                lit = blk + lh;
                q = lh + lsize;
            } else if (ltype == 1) {
                if (lh + 1 > be) return XRS_DECODE_BAD_LITERALS;
                const uint8_t b = __ldg(blk + lh);
                for (int64_t k = lane; k < lsize; k += 32) lbuf[k] = b;
                q = lh + 1;
            } else {
                if (lcsize > be - lh) return XRS_DECODE_BAD_LITERALS;
                if (ltype == 3 && !have_huf) return XRS_DECODE_BAD_LITERALS;  // treeless without a previous tree
                int64_t tree = 0;
                if (ltype == 2) {
                    if (lane == 0) {
                        int mb = 0;
                        sm.v[0] = static_cast<int32_t>(huf_read_table(blk + lh, lcsize, sm, &mb));
                        sm.v[1] = mb;
                    }
                    __syncwarp();
                    tree = sm.v[0];
                    huf_bits = sm.v[1];
                    __syncwarp();
                    if (tree < 0) return XRS_DECODE_BAD_HUFFMAN;
                    have_huf = true;
                }
                const uint8_t *s0 = blk + lh + tree;
                const int64_t sbytes = lcsize - tree;
                bool ok = true;
                if (streams == 1) {
                    if (lane == 0) ok = huf_stream(s0, sbytes, lbuf, lsize, sm.huf, huf_bits);
                } else {
                    int64_t at = 6, size[4];
                    if (sbytes < 6) return XRS_DECODE_BAD_LITERALS;
                    for (int k = 0; k < 3; ++k) size[k] = le_bytes(s0 + 2 * k, 2);
                    size[3] = sbytes - 6 - size[0] - size[1] - size[2];
                    if (size[3] < 1) return XRS_DECODE_BAD_LITERALS;
                    const int64_t seg = (lsize + 3) / 4;
                    if (lane < 4) {
                        for (int k = 0; k < lane; ++k) at += size[k];
                        ok = huf_stream(s0 + at, size[lane], lbuf + seg * lane, lane < 3 ? seg : lsize - 3 * seg,
                                        sm.huf, huf_bits);
                    }
                }
                if (lane < 4) sm.v[lane] = ok;
                __syncwarp();
                const bool all = sm.v[0] && sm.v[1] && sm.v[2] && sm.v[3];
                __syncwarp();
                if (!all) return XRS_DECODE_BAD_LITERALS;
                q = lh + lcsize;
            }
            __syncwarp();  // the literal buffer is complete

            // sequences: lane 0 decodes batches of them into sm, the warp executes each batch
            int64_t lp = 0;
            int reason = 0;
            {
                RevBits br;
                uint32_t sll = 0, sof = 0, sml = 0;
                int64_t n_seq = 0, lop = op, llp = 0;
                if (lane == 0) {
                    int64_t s = q;
                    if (s >= be) {
                        reason = XRS_DECODE_BAD_SEQUENCES;
                    } else {
                        const int c0 = __ldg(blk + s);
                        if (c0 < 128) {
                            n_seq = c0;
                            s += 1;
                        } else if (c0 < 255) {
                            if (s + 2 > be) reason = XRS_DECODE_BAD_SEQUENCES;
                            else n_seq = ((c0 - 128) << 8) + __ldg(blk + s + 1);
                            s += 2;
                        } else {
                            if (s + 3 > be) reason = XRS_DECODE_BAD_SEQUENCES;
                            else n_seq = __ldg(blk + s + 1) + (__ldg(blk + s + 2) << 8) + 0x7F00;
                            s += 3;
                        }
                    }
                    if (!reason && n_seq == 0 && s != be) reason = XRS_DECODE_BAD_SEQUENCES;
                    if (!reason && n_seq > 0) {
                        if (s >= be) {
                            reason = XRS_DECODE_BAD_SEQUENCES;
                        } else {
                            const int modes = __ldg(blk + s++);
                            if (modes & 3) reason = XRS_DECODE_BAD_SEQUENCES;
                            if (!reason) reason = seq_table(blk, &s, be, modes >> 6, 0, sm, sm.ll, &log_ll, &have[0]);
                            if (!reason)
                                reason = seq_table(blk, &s, be, (modes >> 4) & 3, 2, sm, sm.of, &log_of, &have[2]);
                            if (!reason)
                                reason = seq_table(blk, &s, be, (modes >> 2) & 3, 1, sm, sm.ml, &log_ml, &have[1]);
                            if (!reason && !br.init(blk + s, be - s)) reason = XRS_DECODE_BAD_SEQUENCES;
                            if (!reason) {
                                sll = br.read(log_ll);
                                sof = br.read(log_of);
                                sml = br.read(log_ml);
                            }
                        }
                    }
                }
                while (true) {
                    int batch = 0, done = 0;
                    if (lane == 0) {
                        while (!reason && n_seq > 0 && batch < kZstdBatch) {
                            const uint32_t ell = sm.ll[sll], eof = sm.of[sof], eml = sm.ml[sml];
                            const int llc = ell & 0xff, ofc = eof & 0xff, mlc = eml & 0xff;
                            const int64_t ofv = (1ll << ofc) + br.read(ofc);
                            const int64_t mlv = ml_base(mlc) + br.read(ml_bits(mlc));
                            const int64_t llv = ll_base(llc) + br.read(ll_bits(llc));
                            int64_t off;
                            if (ofv > 3) {
                                off = ofv - 3;
                                rep[2] = rep[1];
                                rep[1] = rep[0];
                                rep[0] = static_cast<uint32_t>(off);
                            } else {  // repeat offsets (RFC 8878 3.1.2.5); literal length 0 shifts them by one
                                const int idx = static_cast<int>(ofv) - (llv == 0 ? 0 : 1);
                                XRS_ZSTD_COUNT(llv == 0 ? 3 + idx : idx);
                                off = idx == 3 ? static_cast<int64_t>(rep[0]) - 1 : rep[idx];
                                if (idx != 0) {
                                    if (idx != 1) rep[2] = rep[1];
                                    rep[1] = rep[0];
                                    rep[0] = static_cast<uint32_t>(off);
                                }
                            }
                            if (--n_seq > 0) {
                                sll = (ell >> 16) + br.read((ell >> 8) & 0xff);
                                sml = (eml >> 16) + br.read((eml >> 8) & 0xff);
                                sof = (eof >> 16) + br.read((eof >> 8) & 0xff);
                            }
                            if (br.pos < 0 || (n_seq == 0 && br.pos != 0)) reason = XRS_DECODE_BAD_SEQUENCES;
                            else if (llv > lsize - llp || llv > dsize - lop) reason = XRS_DECODE_LITERALS_OVERRUN;
                            else if (off == 0) reason = XRS_DECODE_OFFSET_ZERO;
                            else if (off > lop + llv) reason = XRS_DECODE_OFFSET_BEFORE_START;
                            else if (mlv > dsize - lop - llv) reason = XRS_DECODE_MATCH_OVERRUN;
                            if (reason) break;
                            sm.op[batch] = static_cast<int32_t>(lop);
                            sm.lp[batch] = static_cast<int32_t>(llp);
                            sm.ll_len[batch] = static_cast<int32_t>(llv);
                            sm.ml_len[batch] = static_cast<int32_t>(mlv);
                            sm.off[batch] = static_cast<int32_t>(off);
                            ++batch;
                            lop += llv + mlv;
                            llp += llv;
                        }
                        sm.v[0] = batch;
                        sm.v[1] = reason;
                        sm.v[2] = reason || n_seq == 0;
                        sm.v[3] = static_cast<int32_t>(lop);
                        sm.v[4] = static_cast<int32_t>(llp);
                    }
                    __syncwarp();
                    batch = sm.v[0];
                    reason = sm.v[1];
                    done = sm.v[2];
                    for (int i = 0; i < batch; ++i) {
                        const int64_t o = sm.op[i], l = sm.ll_len[i], m = sm.ml_len[i], f = sm.off[i];
                        const uint8_t *from_lit = lit + sm.lp[i];
                        for (int64_t k = lane; k < l; k += 32) out[o + k] = from_lit[k];
                        __syncwarp();
                        const uint8_t *from = out + o + l - f;
                        for (int64_t k = lane; k < m; k += 32) out[o + l + k] = from[k < f ? k : k % f];
                    }
                    op = sm.v[3];
                    lp = sm.v[4];
                    __syncwarp();  // lane 0 may overwrite the batch
                    if (done) break;
                }
            }
            if (reason) return reason;
            const int64_t rest = lsize - lp;  // the literals after the last sequence
            if (rest > dsize - op) return XRS_DECODE_LITERALS_OVERRUN;
            for (int64_t k = lane; k < rest; k += 32) out[op + k] = lit[lp + k];
            op += rest;
        }
        __syncwarp();
        if (last) break;
    }
    if (checksum && p + 4 > n) return XRS_DECODE_INPUT_OVERRUN;
    if (op != dsize) return XRS_DECODE_SHORT;
    if (checksum) {
        if (xxh64_low32(out, op, sm, lane) != le_bytes(in + p, 4)) return XRS_DECODE_CHECKSUM;
        p += 4;
    }
    while (p < n) {  // skippable frames (RFC 8878 3.1.2) may follow; nothing else may
        if (p + 8 > n || (le_bytes(in + p, 4) & 0xFFFFFFF0u) != 0x184D2A50u) return XRS_DECODE_TRAILING_BYTES;
        const int64_t skip = le_bytes(in + p + 4, 4);
        if (skip > n - p - 8) return XRS_DECODE_TRAILING_BYTES;
        p += 8 + skip;
    }
    return 0;
}

// One warp (one block of 32) per Zstd stream: descriptors [0, n_streams) of `desc`, literal buffer w at
// lits + w * lit_stride.
__global__ void __launch_bounds__(32) k_zstd_decode(const uint8_t *__restrict__ data, const StreamDesc *__restrict__ desc,
                                                    int64_t n_streams, uint8_t *__restrict__ scratch,
                                                    uint8_t *__restrict__ lits, int64_t lit_stride, uint32_t *err) {
    __shared__ ZstdShared sm;
    const int64_t w = blockIdx.x;
    const int lane = threadIdx.x;
    if (w >= n_streams) return;
    const StreamDesc d = desc[w];
    if (d.dsize == 0) return;
    const uint8_t *in = data + d.src;
    uint8_t *out = scratch + d.dst;
    if (d.stored) {
        for (int64_t k = lane; k < d.dsize; k += 32) out[k] = __ldg(in + k);
        return;
    }
    const int reason = zstd_frame(in, d.csize, out, d.dsize, lits + w * lit_stride, sm, lane);
    if (reason && lane == 0) report(err, d.chunk, reason);
    __syncwarp();  // `sm` is free for the next block of this SM
}

int launch_zstd(const uint8_t *data, const StreamDesc *desc, int64_t n_streams, uint8_t *scratch, uint8_t *lits,
                int64_t lit_stride, uint32_t *err, cudaStream_t st) {
    const unsigned warps = static_cast<unsigned>(n_streams);  // one warp of 32 per block
    XRS_TIMED("zarr_zstd_decode", st,
              k_zstd_decode<<<warps, 32, 0, st>>>(data, desc, n_streams, scratch, lits, lit_stride, err));
    XRS_LAUNCH_CHECK("k_zstd_decode");
    return 0;
}
