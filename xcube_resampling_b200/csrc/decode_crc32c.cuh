// decode_crc32c.cuh -- the CRC-32C trailer of Zarr v3's crc32c codec checked on the device; part of decode.cu.
//
// A file flagged XRS_CHUNK_CRC32C holds its payload and then 4 bytes: the little-endian CRC-32C (Castagnoli, the
// reflected polynomial 0x82F63B78) of the payload.  k_crc32c runs before k_zarr_index, one warp per chunk of the
// table.  It checks the trailer of a flagged file and then drops the trailer and the flag from the DEVICE copy of the
// table, so k_zarr_index, the decoders and k_zarr_scatter see the payload alone, exactly as they see an unflagged file.
// Reads stay inside the file (plan_streams checked that it holds its trailer); every loop is bounded by its length.

constexpr uint32_t kCrc32cPoly = 0x82F63B78u;

// One warp (one block of 32) per chunk of the table: chunks that carry no flag are left as they are.
__global__ void __launch_bounds__(32) k_crc32c(const uint8_t *__restrict__ data, xrs_zarr_chunk *chunks,
                                               int64_t n_chunks, uint32_t *err) {
    __shared__ uint32_t table[256], part[32];
    const int64_t c = blockIdx.x;
    const int lane = threadIdx.x;
    if (c >= n_chunks) return;
    const xrs_zarr_chunk ch = chunks[c];
    if (!(ch.codec & XRS_CHUNK_CRC32C)) return;
    const int64_t n = ch.length - 4;
    const uint8_t *file = data + ch.offset;
    const uint32_t crc = warp_crc<kCrc32cPoly>(file, n, table, part, lane);  // every lane has read `ch` by now
    if (lane == 0) {
        if (crc != le32(file + n)) report(err, static_cast<int>(c), XRS_DECODE_CRC32C);
        chunks[c].codec = ch.codec & ~XRS_CHUNK_CRC32C;
        chunks[c].length = n;
    }
}

int launch_crc32c(const uint8_t *data, xrs_zarr_chunk *chunks, int64_t n_chunks, uint32_t *err, cudaStream_t st) {
    const unsigned warps = static_cast<unsigned>(n_chunks);  // one warp of 32 per block; n_chunks < 2^24
    XRS_TIMED("zarr_crc32c", st, k_crc32c<<<warps, 32, 0, st>>>(data, chunks, n_chunks, err));
    XRS_LAUNCH_CHECK("k_crc32c");
    return 0;
}
