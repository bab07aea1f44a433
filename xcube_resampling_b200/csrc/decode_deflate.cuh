// decode_deflate.cuh -- Deflate streams (RFC 1951) in a zlib (RFC 1950) or gzip (RFC 1952) wrapper decoded by one
// warp each; part of decode.cu.
//
// k_inflate takes the Deflate descriptors k_zarr_index wrote (a numcodecs zlib or gzip chunk, or one stream of a
// Blosc-Zlib frame) and decodes each into its range of the scratch.  The whole decoded stream lies there, so a
// distance may reach back up to 32768 bytes but never before the first byte of the stream (of the member, for
// gzip).  Lane 0 reads the block headers, builds zlib-style Huffman tables in shared memory (a root table plus
// subtables) and decodes the symbols from a 64-bit bit buffer, writing literals straight to the output; it collects
// up to 32 matches whose sources lie before the batch's first destination, and the warp copies them together with
// the periodic-extension rule of k_lz4_decode.  Stored blocks are copied by the warp.  The Adler-32 / CRC-32 of the
// output is computed by the warp, one contiguous segment a lane.  Every read stays inside the stream's bytes, every
// write inside its scratch range, every table index inside its table; a stream that breaks the format sets the
// caller's error word.  Every loop is bounded by the input or by counts checked against the decoded size.

// Counts what the corpus exercises (a test hook: the host build of this file defines it; on the device it is nothing):
// 0-2 block types, 3-60 length codes 257-285 at their lowest (3 + 2c) and highest (4 + 2c) extra value, 61-120
// distance codes at both ends (61 + 2c, 62 + 2c), 121-123 repeat codes 16-18, 124 zlib, 125 gzip member, 126 length
// 258 from code 284, 127 a block with no distance codes.
#ifndef XRS_DEFLATE_COUNT
#define XRS_DEFLATE_COUNT(event) ((void)0)
#endif

constexpr int kInfLenRoot = 9, kInfDistRoot = 6, kInfCodeRoot = 7;  // root index bits, as zlib's inflate
constexpr int kInfLenTable = 852, kInfDistTable = 592;  // zlib's ENOUGH_LENS / ENOUGH_DISTS for those roots
constexpr int kInfBatch = 32;                            // matches lane 0 decodes before the warp copies them
constexpr uint32_t kInfInvalid = 64;

// Table entry: value (bits 0-15), bits (16-23), op (24-31): 0 a symbol of `bits` bits; 1-15 a link to a subtable of
// 2^op entries at `value`, indexed by the bits after the root's; kInfInvalid no code (an incomplete set).
struct InflateShared {
    uint32_t lcode[kInfLenTable], dcode[kInfDistTable];
    uint32_t crc[256];
    uint16_t work[288];
    uint8_t lens[320];
    int32_t m_dst[kInfBatch], m_dist[kInfBatch], m_cum[kInfBatch + 1];
    uint32_t part[64];
    int64_t v[8];  // values lane 0 publishes to the warp
};

// zlib's inflate_table over lens[0, n): a root table of 2^*root entries (fewer when no code is that long) and the
// subtables behind it, at most `cap` entries.  false for an over-subscribed or an incomplete set -- except that a
// length or distance set may be a single code of length 1, and a set without codes decodes to invalid entries.
__device__ inline bool inf_table(const uint8_t *lens, int n, bool code_lengths, uint32_t *table, int cap, int *root,
                                 uint16_t *work) {
    int count[16] = {}, offs[16];
    for (int s = 0; s < n; ++s) ++count[lens[s]];
    int max = 15;
    while (max >= 1 && count[max] == 0) --max;
    if (max == 0) {
        table[0] = table[1] = (kInfInvalid << 24) | (1u << 16);
        *root = 1;
        return true;
    }
    int min = 1;
    while (min < max && count[min] == 0) ++min;
    int rt = *root < max ? *root : max;
    if (rt < min) rt = min;
    int left = 1;
    for (int l = 1; l <= 15; ++l) {
        left = 2 * left - count[l];
        if (left < 0) return false;
    }
    if (left > 0 && (code_lengths || max != 1)) return false;
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + count[l];
    for (int s = 0; s < n; ++s)
        if (lens[s]) work[offs[lens[s]]++] = static_cast<uint16_t>(s);
    uint32_t huff = 0, low = 0xffffffffu, used = 1u << rt;
    const uint32_t mask = used - 1;
    int sym = 0, len = min, curr = rt, drop = 0, next = 0;
    if (used > static_cast<uint32_t>(cap)) return false;
    while (true) {  // the codes in canonical order; huff is the current code, bit-reversed
        const uint32_t here = work[sym] | (static_cast<uint32_t>(len - drop) << 16);
        const uint32_t size = 1u << curr;
        for (uint32_t fill = size, incr = 1u << (len - drop); fill != 0;) {
            fill -= incr;
            table[next + (huff >> drop) + fill] = here;
        }
        uint32_t incr = 1u << (len - 1);
        while (huff & incr) incr >>= 1;
        huff = incr ? (huff & (incr - 1)) + incr : 0;
        ++sym;
        if (--count[len] == 0) {
            if (len == max) break;
            len = lens[work[sym]];
        }
        if (len > rt && (huff & mask) != low) {  // a new subtable
            if (drop == 0) drop = rt;
            next += size;
            curr = len - drop;
            int room = 1 << curr;
            while (curr + drop < max) {
                room -= count[curr + drop];
                if (room <= 0) break;
                ++curr;
                room <<= 1;
            }
            used += 1u << curr;
            if (used > static_cast<uint32_t>(cap)) return false;
            low = huff & mask;
            table[low] = static_cast<uint32_t>(next) | (static_cast<uint32_t>(rt) << 16) |
                         (static_cast<uint32_t>(curr) << 24);
        }
    }
    if (huff != 0) table[next + huff] = (kInfInvalid << 24) | (static_cast<uint32_t>(len - drop) << 16);
    *root = rt;
    return true;
}

// LSB-first bit reader over in[0, n) (lane 0).  It never loads past in[n - 1]; a whole-word refill may put the
// bits of bytes it has not counted yet above `cnt` -- they are the stream's own and the next refill ORs them again.
struct InfBits {
    const uint8_t *in;
    int64_t n, ip;  // bytes [0, ip) are in `buf` or consumed
    uint64_t buf;
    int cnt;        // valid bits in buf

    __device__ void refill() {
        if (ip + 8 <= n) {
            uint64_t w = 0;
            for (int k = 0; k < 8; ++k) w |= static_cast<uint64_t>(__ldg(in + ip + k)) << (8 * k);
            buf |= w << cnt;
            const int take = (63 - cnt) >> 3;
            ip += take;
            cnt += 8 * take;
        } else {
            while (cnt <= 56 && ip < n) {
                buf |= static_cast<uint64_t>(__ldg(in + ip++)) << cnt;
                cnt += 8;
            }
        }
    }
    __device__ bool need(int k) {  // k <= 32
        if (cnt < k) refill();
        return cnt >= k;
    }
    __device__ uint32_t take(int k) {  // after need(k)
        const uint32_t v = static_cast<uint32_t>(buf & ((1ull << k) - 1));
        buf >>= k;
        cnt -= k;
        return v;
    }
    __device__ int64_t byte_pos() {  // drops the bits up to the next byte boundary
        buf >>= cnt & 7;
        cnt &= ~7;
        return ip - cnt / 8;
    }
    __device__ void seek(int64_t p) {
        ip = p;
        buf = 0;
        cnt = 0;
    }
};

// one symbol through `table`; -1 with *reason set if the input ends inside the code or the code is a hole
__device__ inline int inf_symbol(InfBits &br, const uint32_t *table, int root, int *reason) {
    if (br.cnt < 15) br.refill();
    uint32_t e = table[br.buf & ((1u << root) - 1)];
    int bits = 0;
    if ((e >> 24) != 0 && (e >> 24) < 16) {
        bits = root;
        e = table[(e & 0xffff) + ((br.buf >> root) & ((1u << (e >> 24)) - 1))];
    }
    bits += (e >> 16) & 0xff;
    if (bits > br.cnt) {
        *reason = XRS_DECODE_INPUT_OVERRUN;
        return -1;
    }
    if ((e >> 24) == kInfInvalid) {
        *reason = XRS_DECODE_BAD_DEFLATE_SYMBOL;
        return -1;
    }
    br.take(bits);
    return static_cast<int>(e & 0xffff);
}

// base and extra bits of length code c = symbol - 257 (0-28) and of distance code c (0-29), RFC 1951 3.2.5
__device__ inline int inf_len_extra(int c) { return c < 8 || c == 28 ? 0 : (c - 4) >> 2; }
__device__ inline int inf_len_base(int c) {
    return c < 8 ? c + 3 : c == 28 ? 258 : ((4 + (c & 3)) << inf_len_extra(c)) + 3;
}
__device__ inline int inf_dist_extra(int c) { return c < 4 ? 0 : (c >> 1) - 1; }
__device__ inline int inf_dist_base(int c) { return c < 4 ? c + 1 : ((2 + (c & 1)) << inf_dist_extra(c)) + 1; }

// the tables of a fixed-Huffman block (RFC 1951 3.2.6): 288 litlen codes, 32 distance codes of 5 bits
__device__ inline void inf_fixed(InflateShared &sm, int *lroot, int *droot) {
    for (int s = 0; s < 288; ++s) sm.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
    *lroot = kInfLenRoot;
    inf_table(sm.lens, 288, false, sm.lcode, kInfLenTable, lroot, sm.work);
    for (int s = 0; s < 32; ++s) sm.lens[s] = 5;
    *droot = kInfDistRoot;
    inf_table(sm.lens, 32, false, sm.dcode, kInfDistTable, droot, sm.work);
}

// the code description of a dynamic-Huffman block (RFC 1951 3.2.7) into the litlen and distance tables; 0 or the
// reason
__device__ inline int inf_dynamic(InfBits &br, InflateShared &sm, int *lroot, int *droot) {
    if (!br.need(14)) return XRS_DECODE_INPUT_OVERRUN;
    const int nlen = static_cast<int>(br.take(5)) + 257, ndist = static_cast<int>(br.take(5)) + 1;
    const int ncode = static_cast<int>(br.take(4)) + 4;
    if (nlen > 286 || ndist > 30) return XRS_DECODE_BAD_DEFLATE_CODES;
    const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    for (int k = 0; k < 19; ++k) sm.lens[k] = 0;
    for (int k = 0; k < ncode; ++k) {
        if (!br.need(3)) return XRS_DECODE_INPUT_OVERRUN;
        sm.lens[order[k]] = static_cast<uint8_t>(br.take(3));
    }
    int croot = kInfCodeRoot;  // the code-length code's table borrows the litlen table's space
    if (!inf_table(sm.lens, 19, true, sm.lcode, kInfLenTable, &croot, sm.work)) return XRS_DECODE_BAD_DEFLATE_CODES;
    for (int i = 0; i < nlen + ndist;) {
        int reason = 0;
        const int sym = inf_symbol(br, sm.lcode, croot, &reason);
        if (sym < 0) return reason == XRS_DECODE_BAD_DEFLATE_SYMBOL ? XRS_DECODE_BAD_DEFLATE_CODES : reason;
        if (sym < 16) {
            sm.lens[i++] = static_cast<uint8_t>(sym);
            continue;
        }
        XRS_DEFLATE_COUNT(121 + sym - 16);
        const int xb = sym == 16 ? 2 : sym == 17 ? 3 : 7;
        if (!br.need(xb)) return XRS_DECODE_INPUT_OVERRUN;
        const int rep = (sym == 18 ? 11 : 3) + static_cast<int>(br.take(xb));
        if (sym == 16 && i == 0) return XRS_DECODE_BAD_DEFLATE_CODES;  // no previous length
        if (rep > nlen + ndist - i) return XRS_DECODE_BAD_DEFLATE_CODES;
        const uint8_t val = sym == 16 ? sm.lens[i - 1] : 0;
        for (int k = 0; k < rep; ++k) sm.lens[i++] = val;  // may cross from the litlen to the distance lengths
    }
    if (sm.lens[256] == 0) return XRS_DECODE_BAD_DEFLATE_CODES;  // no end-of-block code
    *lroot = kInfLenRoot;
    if (!inf_table(sm.lens, nlen, false, sm.lcode, kInfLenTable, lroot, sm.work)) return XRS_DECODE_BAD_DEFLATE_CODES;
    *droot = kInfDistRoot;
    if (!inf_table(sm.lens + nlen, ndist, false, sm.dcode, kInfDistTable, droot, sm.work))
        return XRS_DECODE_BAD_DEFLATE_CODES;
    bool any = false;
    for (int k = 0; k < ndist; ++k) any = any || sm.lens[nlen + k];
    if (!any) XRS_DEFLATE_COUNT(127);
    return 0;
}

// The Deflate stream at in[*p, n) into out[*op, dsize), by the whole warp; `start` is the first output byte a
// distance may reach.  Returns 0 or the reason; on success *p is the first byte after the stream and *op the end of
// its output.
__device__ inline int inflate_stream(const uint8_t *in, int64_t n, int64_t *p, uint8_t *out, int64_t *op,
                                     int64_t start, int64_t dsize, InflateShared &sm, int lane) {
    InfBits br;  // lane 0's decoder state, kept across the rounds below
    br.in = in;
    br.n = n;
    br.seek(*p);
    int64_t o = *op;
    bool in_block = false, last = false, done = false, carry = false;
    int lroot = 0, droot = 0, c_len = 0, c_dist = 0;
    while (true) {
        if (lane == 0) {  // decode until the batch is full, a block ends, a stored block is read or an error
            int reason = 0, nb = 0, cum = 0;
            int64_t s_src = 0, s_dst = 0, s_len = 0;
            if (carry) {  // the match that ended the previous round: it reads what that round's matches wrote
                sm.m_dst[0] = static_cast<int32_t>(o - c_len);
                sm.m_dist[0] = c_dist;
                sm.m_cum[0] = 0;
                cum = c_len;
                nb = 1;
                carry = false;
            }
            while (!reason && !done) {
                if (!in_block) {
                    if (!br.need(3)) {
                        reason = XRS_DECODE_INPUT_OVERRUN;
                        break;
                    }
                    last = br.take(1);
                    const int type = static_cast<int>(br.take(2));
                    if (type == 3) {
                        reason = XRS_DECODE_BAD_DEFLATE_BLOCK;
                        break;
                    }
                    XRS_DEFLATE_COUNT(type);
                    if (type == 0) {  // stored: LEN, NLEN at the next byte boundary, then LEN bytes
                        int64_t q = br.byte_pos();
                        if (q + 4 > n) {
                            reason = XRS_DECODE_INPUT_OVERRUN;
                            break;
                        }
                        const int len = __ldg(in + q) | (__ldg(in + q + 1) << 8);
                        const int nlen = __ldg(in + q + 2) | (__ldg(in + q + 3) << 8);
                        q += 4;
                        if (len != (~nlen & 0xffff)) reason = XRS_DECODE_BAD_DEFLATE_BLOCK;
                        else if (len > n - q) reason = XRS_DECODE_INPUT_OVERRUN;
                        else if (len > dsize - o) reason = XRS_DECODE_LITERALS_OVERRUN;
                        if (reason) break;
                        s_src = q;
                        s_dst = o;
                        s_len = len;
                        o += len;
                        br.seek(q + len);
                        done = last;
                        break;
                    }
                    if (type == 1) {
                        inf_fixed(sm, &lroot, &droot);
                    } else {
                        reason = inf_dynamic(br, sm, &lroot, &droot);
                        if (reason) break;
                    }
                    in_block = true;
                }
                if (nb == kInfBatch) break;
                const int sym = inf_symbol(br, sm.lcode, lroot, &reason);
                if (sym < 0) break;
                if (sym < 256) {
                    if (o >= dsize) {
                        reason = XRS_DECODE_LITERALS_OVERRUN;
                        break;
                    }
                    out[o++] = static_cast<uint8_t>(sym);
                    continue;
                }
                if (sym == 256) {  // end of block: the warp copies the batch before the next block
                    in_block = false;
                    done = last;
                    break;
                }
                if (sym > 285) {
                    reason = XRS_DECODE_BAD_DEFLATE_SYMBOL;
                    break;
                }
                const int lc = sym - 257, lx = inf_len_extra(lc);
                if (!br.need(lx)) {
                    reason = XRS_DECODE_INPUT_OVERRUN;
                    break;
                }
                const int le = static_cast<int>(br.take(lx)), len = inf_len_base(lc) + le;
                if (le == 0) XRS_DEFLATE_COUNT(3 + 2 * lc);
                if (le == (1 << lx) - 1) XRS_DEFLATE_COUNT(4 + 2 * lc);
                if (lc == 27 && le == 31) XRS_DEFLATE_COUNT(126);
                const int dc = inf_symbol(br, sm.dcode, droot, &reason);
                if (dc < 0) break;
                if (dc > 29) {
                    reason = XRS_DECODE_BAD_DEFLATE_SYMBOL;
                    break;
                }
                const int dx = inf_dist_extra(dc);
                if (!br.need(dx)) {
                    reason = XRS_DECODE_INPUT_OVERRUN;
                    break;
                }
                const int de = static_cast<int>(br.take(dx)), dist = inf_dist_base(dc) + de;
                if (de == 0) XRS_DEFLATE_COUNT(61 + 2 * dc);
                if (de == (1 << dx) - 1) XRS_DEFLATE_COUNT(62 + 2 * dc);
                if (dist > o - start) {
                    reason = XRS_DECODE_OFFSET_BEFORE_START;
                    break;
                }
                if (len > dsize - o) {
                    reason = XRS_DECODE_MATCH_OVERRUN;
                    break;
                }
                o += len;
                // a match may join the batch when it reads nothing an earlier match of the batch writes
                if (nb > 0 && o - len - dist + (len < dist ? len : dist) > sm.m_dst[0]) {
                    carry = true;
                    c_len = len;
                    c_dist = dist;
                    break;
                }
                sm.m_dst[nb] = static_cast<int32_t>(o - len);
                sm.m_dist[nb] = dist;
                sm.m_cum[nb] = cum;
                cum += len;
                ++nb;
            }
            sm.m_cum[nb] = cum;
            sm.v[0] = nb;
            sm.v[1] = reason;
            sm.v[2] = done;
            sm.v[3] = s_src;
            sm.v[4] = s_dst;
            sm.v[5] = s_len;
            sm.v[6] = done ? br.byte_pos() : 0;
            sm.v[7] = o;
        }
        __syncwarp();
        const int nb = static_cast<int>(sm.v[0]), reason = static_cast<int>(sm.v[1]);
        if (reason) {
            __syncwarp();
            return reason;
        }
        // the batch's match bytes, flattened: every source byte is final, so four loads a lane go out before the
        // stores (byte k of a match is out[dst - dist + k % dist])
        const int total = sm.m_cum[nb];
        for (int base = 0, i = 0; base < total; base += 4 * 32) {
            uint8_t val[4];
            int64_t at[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int f = base + 32 * u + lane;
                at[u] = -1;
                if (f < total) {
                    while (sm.m_cum[i + 1] <= f) ++i;
                    const int k = f - sm.m_cum[i], d = sm.m_dist[i];
                    at[u] = sm.m_dst[i] + k;
                    val[u] = out[sm.m_dst[i] - d + (k < d ? k : k % d)];
                }
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (at[u] >= 0) out[at[u]] = val[u];
        }
        const int64_t s_src = sm.v[3], s_dst = sm.v[4], s_len = sm.v[5];
        for (int64_t k = lane; k < s_len; k += 32) out[s_dst + k] = __ldg(in + s_src + k);
        const bool fin = sm.v[2];
        if (fin) {
            *p = sm.v[6];
            *op = sm.v[7];
        }
        __syncwarp();  // lane 0 may overwrite the batch; the next round's matches read this one's bytes
        if (fin) return 0;
    }
}

// Adler-32 of buf[0, n), one segment a lane: a segment's sums (a, b) enter the whole as a and b + a * (bytes after it)
__device__ inline uint32_t inf_adler32(const uint8_t *buf, int64_t n, InflateShared &sm, int lane) {
    const int64_t seg = (n + 31) / 32, lo = lane * seg < n ? lane * seg : n, hi = lo + seg < n ? lo + seg : n;
    uint32_t a = 0, b = 0;
    for (int64_t k = lo; k < hi;) {
        const int64_t e = hi - k < 5552 ? hi : k + 5552;  // zlib's NMAX: no uint32 overflow before the reduction
        for (; k < e; ++k) {
            a += buf[k];
            b += a;
        }
        a %= 65521;
        b %= 65521;
    }
    sm.part[lane] = a;
    sm.part[32 + lane] = static_cast<uint32_t>((b + static_cast<uint64_t>(a) * ((n - hi) % 65521)) % 65521);
    __syncwarp();
    uint64_t sa = 1, sb = static_cast<uint64_t>(n % 65521);
    for (int s = 0; s < 32; ++s) {
        sa += sm.part[s];
        sb += sm.part[32 + s];
    }
    __syncwarp();
    return static_cast<uint32_t>(((sb % 65521) << 16) | (sa % 65521));
}

// The zlib stream or gzip file in[0, n) into out[0, dsize), by the whole warp; returns 0 or the reason.  Not inlined:
// inlined, it changes how nvcc compiles k_zstd_decode in the same file.
__device__ __noinline__ int inflate_file(const uint8_t *in, int64_t n, uint8_t *out, int64_t dsize, bool gzip,
                                   InflateShared &sm, int lane) {
    int64_t p = 0, op = 0;
    if (!gzip) {  // CMF, FLG; bytes after the Adler-32 are ignored, as zlib.decompress ignores them
        if (lane == 0) XRS_DEFLATE_COUNT(124);
        if (n < 2) return XRS_DECODE_INPUT_OVERRUN;
        const int cmf = __ldg(in), flg = __ldg(in + 1);
        if ((cmf & 15) != 8 || (cmf >> 4) > 7 || (cmf * 256 + flg) % 31 || (flg & 0x20))
            return XRS_DECODE_BAD_FRAME_HEADER;
        p = 2;
        const int reason = inflate_stream(in, n, &p, out, &op, 0, dsize, sm, lane);
        if (reason) return reason;
        if (p + 4 > n) return XRS_DECODE_INPUT_OVERRUN;
        if (op != dsize) return XRS_DECODE_SHORT;
        const uint32_t want = (static_cast<uint32_t>(__ldg(in + p)) << 24) | (__ldg(in + p + 1) << 16) |
                              (__ldg(in + p + 2) << 8) | __ldg(in + p + 3);
        return inf_adler32(out, op, sm, lane) == want ? 0 : XRS_DECODE_CHECKSUM;
    }
    for (bool first = true;; first = false) {  // gzip members, NUL bytes between and after them
        if (!first) {
            while (p < n && __ldg(in + p) == 0) ++p;
            if (p == n) break;
            if (n - p < 2 || __ldg(in + p) != 0x1f || __ldg(in + p + 1) != 0x8b) return XRS_DECODE_TRAILING_BYTES;
        }
        if (lane == 0) XRS_DEFLATE_COUNT(125);
        if (n - p < 10) return XRS_DECODE_INPUT_OVERRUN;
        if (__ldg(in + p) != 0x1f || __ldg(in + p + 1) != 0x8b || __ldg(in + p + 2) != 8)
            return XRS_DECODE_BAD_FRAME_HEADER;
        const int flg = __ldg(in + p + 3);  // MTIME, XFL, OS and the reserved flag bits are ignored
        p += 10;
        if (flg & 4) {  // FEXTRA
            if (n - p < 2) return XRS_DECODE_INPUT_OVERRUN;
            const int64_t xlen = __ldg(in + p) | (__ldg(in + p + 1) << 8);
            p += 2;
            if (xlen > n - p) return XRS_DECODE_INPUT_OVERRUN;
            p += xlen;
        }
        for (int f = 8; f <= 16; f += 8) {  // FNAME, FCOMMENT: zero-terminated
            if (!(flg & f)) continue;
            while (p < n && __ldg(in + p) != 0) ++p;
            if (p == n) return XRS_DECODE_INPUT_OVERRUN;
            ++p;
        }
        if (flg & 2) {  // FHCRC: skipped, not checked
            if (n - p < 2) return XRS_DECODE_INPUT_OVERRUN;
            p += 2;
        }
        const int64_t m0 = op;
        const int reason = inflate_stream(in, n, &p, out, &op, m0, dsize, sm, lane);
        if (reason) return reason;
        if (n - p < 8) return XRS_DECODE_INPUT_OVERRUN;
        if (warp_crc<0xEDB88320u>(out + m0, op - m0, sm.crc, sm.part, lane) != le32(in + p) ||
            le32(in + p + 4) != static_cast<uint32_t>(op - m0))
            return XRS_DECODE_CHECKSUM;
        p += 8;
    }
    return op == dsize ? 0 : XRS_DECODE_SHORT;
}

// One warp (one block of 32) per Deflate stream: descriptors [0, n_streams) of `desc`
__global__ void __launch_bounds__(32) k_inflate(const uint8_t *__restrict__ data,
                                                const xrs_zarr_chunk *__restrict__ chunks,
                                                const StreamDesc *__restrict__ desc, int64_t n_streams,
                                                uint8_t *__restrict__ scratch, uint32_t *err) {
    __shared__ InflateShared sm;
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
    const bool gzip = chunks[d.chunk].codec == XRS_CHUNK_GZIP;
    const int reason = inflate_file(in, d.csize, out, d.dsize, gzip, sm, lane);
    if (reason && lane == 0) report(err, d.chunk, reason);
    __syncwarp();  // `sm` is free for the next block of this SM
}

int launch_inflate(const uint8_t *data, const xrs_zarr_chunk *chunks, const StreamDesc *desc, int64_t n_streams,
                   uint8_t *scratch, uint32_t *err, cudaStream_t st) {
    const unsigned warps = static_cast<unsigned>(n_streams);  // one warp of 32 per block
    XRS_TIMED("zarr_inflate", st, k_inflate<<<warps, 32, 0, st>>>(data, chunks, desc, n_streams, scratch, err));
    XRS_LAUNCH_CHECK("k_inflate");
    return 0;
}
