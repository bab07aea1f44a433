// gather_dual.cu -- K2d: the same bands gathered with TWO interpolation methods in one launch.
//
//   xrs_gather_ij2   rectify.py:579-734 (_compute_var_image*), called by the reference once per
//                    output variable (rectify.py:159-174): when a call wants the same source bands
//                    with nearest AND with bilinear / triangular interpolation, both passes walk the
//                    same ij image and read the same source pixels.
//
// The nearest-neighbour sample of a target pixel is always ONE OF THE FOUR TAPS of its bilinear
// sample: both start from (i0, j0) = int(i), int(j) and the clamped neighbours (i1, j1)
// (rectify.py:689-692); nearest then picks i1 when u > 0.5 and j1 when v > 0.5 (rectify.py:693-698).
// So the staged box of source pixels, the four shared-memory reads and the ij values are shared and
// the second result costs three selects and one store per band and pixel instead of a second pass
// over ij and the source: 16*T + 4*B*S + 8*B*T bytes instead of 2 * (16*T + 4*B*S + 4*B*T).
//
// Same tiling as k2_gather_staged (gather.cu): one CTA per 32x32 target tile, the tile's source box of
// every band through 2-D TMA tensor copies into a 4-stage mbarrier ring, taps from shared memory;
// tiles whose box exceeds 64x48 read their taps from global memory inside the same kernel.
#include <algorithm>
#include <cstring>
#include <vector>

#include "gather_common.cuh"

namespace xrs {

template <typename T>
struct DualParams {
    CUtensorMap maps[K2_MAX_BANDS];
    const T *src[K2_MAX_BANDS];
    T *dst_interp[K2_MAX_BANDS];
    T *dst_near[K2_MAX_BANDS];
};

// the raw tap nearest interpolation picks: `right` = column i1 instead of i0, `lower` = row j1 instead of j0
template <typename T>
__device__ __forceinline__ T pick_tap(T r00, T r01, T r10, T r11, bool right, bool lower) {
    const T upper_v = right ? r01 : r00;
    const T lower_v = right ? r11 : r10;
    return lower ? lower_v : upper_v;
}

template <typename T, int METHOD>
__global__ void __launch_bounds__(K2S_THREADS, 3)
k2_gather_dual(const __grid_constant__ DualParams<T> p, int n_bands, int64_t src_h, int64_t src_w, int64_t src_pitch,
               int64_t win_i0, int64_t win_j0, const double *__restrict__ ij, int64_t dst_h, int64_t dst_w,
               T fill_interp, T fill_near) {
    static_assert(METHOD == XRS_BILINEAR || METHOD == XRS_TRIANGULAR, "the second method is always nearest");
    extern __shared__ unsigned char k2d_smem_raw[];
    constexpr int STAGE_ELEMS = K2S_BOX_W * K2S_BOX_H;
    unsigned char *smem = k2d_smem_raw + ((128u - (smem_u32(k2d_smem_raw) & 127u)) & 127u);  // TMA: 128-byte aligned
    T *stages = reinterpret_cast<T *>(smem);
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + static_cast<size_t>(K2S_STAGES) * STAGE_ELEMS * sizeof(T));
    int(*red)[K2S_THREADS / 32] = reinterpret_cast<int(*)[K2S_THREADS / 32]>(full_bar + K2S_STAGES);

    const int tid = threadIdx.x;
    const int tx = tid % K2S_TW, ty = tid / K2S_TW;
    const int64_t c = static_cast<int64_t>(blockIdx.x) * K2S_TW + tx;
    const int64_t r_base = static_cast<int64_t>(blockIdx.y) * K2S_TH + ty;  // rows r_base + k * K2S_ROW_STEP
    const bool col_in = c < dst_w;

    // ---- this thread's pixels: the four taps, the fractions, and which tap nearest takes ----
    double fi[K2S_PX], fj[K2S_PX];
#pragma unroll
    for (int k = 0; k < K2S_PX; ++k) {
        const int64_t r = r_base + k * K2S_ROW_STEP;
        fi[k] = fj[k] = NAN;
        if (col_in && r < dst_h) {
            const int64_t o = r * dst_w + c;
            fi[k] = ld_stream(ij + o);
            fj[k] = ld_stream(ij + dst_h * dst_w + o);
        }
    }
    Taps t[K2S_PX];
    uint32_t near_sel = 0;  // bits 2k, 2k+1: pixel k takes column i1 / row j1 (rectify.py:693-698)
    int i_lo = INT32_MAX, i_hi = -1, j_lo = INT32_MAX, j_hi = -1;
#pragma unroll
    for (int k = 0; k < K2S_PX; ++k) {
        t[k] = make_taps<METHOD>(fi[k], fj[k], src_w, src_h);
        if (t[k].valid) {
            i_lo = min(i_lo, t[k].i0); i_hi = max(i_hi, t[k].i1);
            j_lo = min(j_lo, t[k].j0); j_hi = max(j_hi, t[k].j1);
            near_sel |= (t[k].u > 0.5 ? 1u : 0u) << (2 * k);
            near_sel |= (t[k].v > 0.5 ? 2u : 0u) << (2 * k);
        }
    }
    // ---- CTA-wide bounding box of the source pixels ------------------------------------
    i_lo = __reduce_min_sync(0xffffffffu, i_lo); i_hi = __reduce_max_sync(0xffffffffu, i_hi);
    j_lo = __reduce_min_sync(0xffffffffu, j_lo); j_hi = __reduce_max_sync(0xffffffffu, j_hi);
    if ((tid & 31) == 0) {
        red[0][tid >> 5] = i_lo; red[1][tid >> 5] = i_hi; red[2][tid >> 5] = j_lo; red[3][tid >> 5] = j_hi;
    }
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < K2S_STAGES; ++s) mbar_init(&full_bar[s], 1);
        mbar_fence_init();
    }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < K2S_THREADS / 32; ++w) {
        i_lo = min(i_lo, red[0][w]); i_hi = max(i_hi, red[1][w]);
        j_lo = min(j_lo, red[2][w]); j_hi = max(j_hi, red[3][w]);
    }
    if (i_hi < 0) {  // CTA-uniform early out: no target pixel of this tile has a source
        if (col_in)
            for (int b = 0; b < n_bands; ++b)
#pragma unroll
                for (int k = 0; k < K2S_PX; ++k) {
                    const int64_t r = r_base + k * K2S_ROW_STEP;
                    if (r < dst_h) {
                        st_stream(p.dst_interp[b] + r * dst_w + c, fill_interp);
                        st_stream(p.dst_near[b] + r * dst_w + c, fill_near);
                    }
                }
        return;
    }
    // TMA wants the box to start on a 16-byte boundary of the innermost dimension
    constexpr int ALIGN_ELEMS = 16 / sizeof(T) > 0 ? 16 / sizeof(T) : 1;
    const int box_x = ((i_lo - static_cast<int>(win_i0)) / ALIGN_ELEMS) * ALIGN_ELEMS;
    const int box_y = j_lo - static_cast<int>(win_j0);
    i_lo = box_x + static_cast<int>(win_i0);  // first source column held by the staged box
    const bool staged = (i_hi - i_lo + 1 <= K2S_BOX_W) && (j_hi - j_lo + 1 <= K2S_BOX_H);

    if (staged) {
        // Band-independent state, computed once: the four tap addresses of each pixel inside stage 0
        // (the ring is unrolled, the other stages are immediates), output offsets, store predicates.
        // Pixels without a source tap element (0, 0) with u = v = 0 and are overwritten by the fills.
        const T *t00[K2S_PX], *t01[K2S_PX], *t10[K2S_PX], *t11[K2S_PX];
        uint32_t o32[K2S_PX];
        uint32_t st_mask = 0;  // bit k: pixel k lies inside the target image (is stored)
#pragma unroll
        for (int k = 0; k < K2S_PX; ++k) {
            const int off = t[k].valid ? (t[k].j0 - j_lo) * K2S_BOX_W + (t[k].i0 - i_lo) : 0;
            const int di = t[k].valid ? t[k].i1 - t[k].i0 : 0;
            const int dj = t[k].valid ? (t[k].j1 - t[k].j0) * K2S_BOX_W : 0;
            t00[k] = stages + off;
            t01[k] = t00[k] + di;
            t10[k] = t00[k] + dj;
            t11[k] = t10[k] + di;
            const int64_t r = r_base + k * K2S_ROW_STEP;
            st_mask |= (col_in && r < dst_h) ? (1u << k) : 0u;
            o32[k] = static_cast<uint32_t>(r * dst_w + c);
            if (!t[k].valid) t[k].u = t[k].v = 0.0;
        }
        asm volatile("" : "+r"(st_mask), "+r"(near_sel));  // opaque: one bit test per use in the band loop
        constexpr uint32_t STAGE_BYTES = STAGE_ELEMS * sizeof(T);
        if (tid == 0) {
            for (int s = 0; s < K2S_STAGES && s < n_bands; ++s) {
                mbar_arrive_expect_tx(&full_bar[s], STAGE_BYTES);
                tma_load_2d(stages + s * STAGE_ELEMS, &p.maps[s], box_x, box_y, &full_bar[s]);
            }
        }
        for (int b0 = 0; b0 < n_bands; b0 += K2S_STAGES) {
            const uint32_t parity = (b0 / K2S_STAGES) & 1;
#pragma unroll
            for (int s = 0; s < K2S_STAGES; ++s) {
                const int b = b0 + s;
                if (b >= n_bands) break;
                mbar_wait(&full_bar[s], parity);
                T out_i[K2S_PX], out_n[K2S_PX];
#pragma unroll
                for (int k = 0; k < K2S_PX; ++k) {
                    const T r00 = t00[k][s * STAGE_ELEMS], r01 = t01[k][s * STAGE_ELEMS];
                    const T r10 = t10[k][s * STAGE_ELEMS], r11 = t11[k][s * STAGE_ELEMS];
                    const T near = nearest_value(pick_tap(r00, r01, r10, r11, (near_sel >> (2 * k)) & 1u, (near_sel >> (2 * k + 1)) & 1u));
                    const T val = cast_like_numpy<T>(interp_value<METHOD>(
                        static_cast<double>(r00), static_cast<double>(r01), static_cast<double>(r10),
                        static_cast<double>(r11), t[k].u, t[k].v));
                    out_i[k] = t[k].valid ? val : fill_interp;
                    out_n[k] = t[k].valid ? near : fill_near;
                }
                T *di = p.dst_interp[b], *dn = p.dst_near[b];
#pragma unroll
                for (int k = 0; k < K2S_PX; ++k)
                    if (st_mask & (1u << k)) {
                        st_stream(elem_ptr(dn, o32[k]), out_n[k]);
                        st_stream(elem_ptr(di, o32[k]), out_i[k]);
                    }
                __syncthreads();  // every thread is done with stage s
                if (tid == 0 && b + K2S_STAGES < n_bands) {
                    fence_proxy_async();
                    mbar_arrive_expect_tx(&full_bar[s], STAGE_BYTES);
                    tma_load_2d(stages + s * STAGE_ELEMS, &p.maps[b + K2S_STAGES], box_x, box_y, &full_bar[s]);
                }
            }
        }
        return;
    }

    // ---- box too large for the staging buffers: the four taps straight from global memory ----
    if (!col_in) return;
    int64_t o00[K2S_PX], od[K2S_PX], oj[K2S_PX];
#pragma unroll
    for (int k = 0; k < K2S_PX; ++k) {
        o00[k] = (t[k].j0 - win_j0) * src_pitch + (t[k].i0 - win_i0);
        od[k] = t[k].i1 - t[k].i0;
        oj[k] = (t[k].j1 - t[k].j0) * src_pitch;
    }
    for (int b = 0; b < n_bands; ++b) {
        const T *sp = p.src[b];
        T out_i[K2S_PX], out_n[K2S_PX];
#pragma unroll
        for (int k = 0; k < K2S_PX; ++k) {
            out_i[k] = fill_interp;
            out_n[k] = fill_near;
            if (t[k].valid) {
                const T r00 = __ldg(sp + o00[k]), r01 = __ldg(sp + o00[k] + od[k]);
                const T r10 = __ldg(sp + o00[k] + oj[k]), r11 = __ldg(sp + o00[k] + oj[k] + od[k]);
                out_n[k] = nearest_value(pick_tap(r00, r01, r10, r11, (near_sel >> (2 * k)) & 1u, (near_sel >> (2 * k + 1)) & 1u));
                out_i[k] = cast_like_numpy<T>(interp_value<METHOD>(
                    static_cast<double>(r00), static_cast<double>(r01), static_cast<double>(r10),
                    static_cast<double>(r11), t[k].u, t[k].v));
            }
        }
#pragma unroll
        for (int k = 0; k < K2S_PX; ++k) {
            const int64_t r = r_base + k * K2S_ROW_STEP;
            if (r < dst_h) {
                st_stream(p.dst_near[b] + r * dst_w + c, out_n[k]);
                st_stream(p.dst_interp[b] + r * dst_w + c, out_i[k]);
            }
        }
    }
}

// -1: the source cannot be described to TMA (pitch / alignment / size) -- the caller runs two
// single-method gathers instead; 0: enqueued; > 0: error.
template <typename T>
static int launch_dual(const void *const *src_planes, void *const *dst_interp, void *const *dst_near, int n_bands,
                       int64_t src_h, int64_t src_w, int64_t src_pitch, int64_t win_i0, int64_t win_j0, int64_t win_w,
                       int64_t win_h, const double *ij, int64_t dst_h, int64_t dst_w, int method, double fill_interp,
                       double fill_near, cudaStream_t st) {
    bool tma_ok = (src_pitch * sizeof(T)) % 16 == 0 && win_w < (1ll << 31) && win_h < (1ll << 31) &&
                  ceil_div(dst_h, K2S_TH) <= 65535 && dst_h * dst_w < (1ll << 32) && tma_available();
    for (int b = 0; b < n_bands && tma_ok; ++b) tma_ok = (reinterpret_cast<uintptr_t>(src_planes[b]) & 15) == 0;
    if (!tma_ok) return -1;
    const size_t smem = static_cast<size_t>(K2S_STAGES) * K2S_BOX_W * K2S_BOX_H * sizeof(T) +
                        K2S_STAGES * sizeof(uint64_t) + 4 * (K2S_THREADS / 32) * sizeof(int) + 128;
    const dim3 grid(static_cast<unsigned>(ceil_div(dst_w, K2S_TW)), static_cast<unsigned>(ceil_div(dst_h, K2S_TH)));
    const T fi = cast_fill<T>(fill_interp), fn = cast_fill<T>(fill_near);
    // every chunk's tensor maps first: nothing is enqueued if one of them cannot be encoded
    const int n_chunks = static_cast<int>(ceil_div(n_bands, K2_MAX_BANDS));
    std::vector<DualParams<T>> params(n_chunks);
    for (int ch = 0; ch < n_chunks; ++ch) {
        DualParams<T> &dp = params[ch];
        memset(&dp, 0, sizeof(dp));
        const int b0 = ch * K2_MAX_BANDS, nb = std::min(K2_MAX_BANDS, n_bands - b0);
        for (int b = 0; b < nb; ++b) {
            dp.src[b] = static_cast<const T *>(src_planes[b0 + b]);
            dp.dst_interp[b] = static_cast<T *>(dst_interp[b0 + b]);
            dp.dst_near[b] = static_cast<T *>(dst_near[b0 + b]);
            if (!tma_encode_2d(&dp.maps[b], sizeof(T), src_planes[b0 + b], static_cast<uint64_t>(win_w),
                               static_cast<uint64_t>(win_h), static_cast<uint64_t>(src_pitch) * sizeof(T), K2S_BOX_W,
                               K2S_BOX_H))
                return -1;
        }
    }
    for (int ch = 0; ch < n_chunks; ++ch) {
        const int nb = std::min(K2_MAX_BANDS, n_bands - ch * K2_MAX_BANDS);
        if (method == XRS_BILINEAR) {
            XRS_CUDA(cudaFuncSetAttribute(k2_gather_dual<T, XRS_BILINEAR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          static_cast<int>(smem)));
            XRS_TIMED("k2_gather_dual<nearest+bilinear>", st,
                      k2_gather_dual<T, XRS_BILINEAR><<<grid, K2S_THREADS, smem, st>>>(
                          params[ch], nb, src_h, src_w, src_pitch, win_i0, win_j0, ij, dst_h, dst_w, fi, fn));
        } else {
            XRS_CUDA(cudaFuncSetAttribute(k2_gather_dual<T, XRS_TRIANGULAR>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          static_cast<int>(smem)));
            XRS_TIMED("k2_gather_dual<nearest+triangular>", st,
                      k2_gather_dual<T, XRS_TRIANGULAR><<<grid, K2S_THREADS, smem, st>>>(
                          params[ch], nb, src_h, src_w, src_pitch, win_i0, win_j0, ij, dst_h, dst_w, fi, fn));
        }
        XRS_LAUNCH_CHECK("k2_gather_dual");
    }
    return 0;
}

}  // namespace xrs

using namespace xrs;

extern "C" {

int xrs_gather_ij2(const void *const *src_planes_host, void *const *dst_interp_planes_host,
                   void *const *dst_nearest_planes_host, int32_t n_bands, int32_t dtype, int64_t src_h, int64_t src_w,
                   int64_t src_pitch, int64_t win_i0, int64_t win_j0, int64_t win_w, int64_t win_h, const double *ij,
                   int64_t dst_h, int64_t dst_w, int32_t method, double fill_interp, double fill_nearest, void *stream) {
    if (!src_planes_host || !dst_interp_planes_host || !dst_nearest_planes_host || !ij)
        return fail("xrs_gather_ij2: null pointer");
    if (n_bands < 1) return fail("xrs_gather_ij2: n_bands must be >= 1");
    if (method != XRS_BILINEAR && method != XRS_TRIANGULAR)
        return fail("xrs_gather_ij2: method (the one beside nearest) must be 'bilinear' or 'triangular'");
    if (src_h < 1 || src_w < 1 || src_pitch < 1 || dst_h < 1 || dst_w < 1) return fail("xrs_gather_ij2: bad shape");
    if (src_w > INT32_MAX || src_h > INT32_MAX) return fail("xrs_gather_ij2: source too large");
    if (win_i0 < 0 || win_j0 < 0 || win_w < 1 || win_h < 1 || win_i0 + win_w > src_w || win_j0 + win_h > src_h ||
        src_pitch < win_w)
        return fail("xrs_gather_ij2: bad source window");
    for (int b = 0; b < n_bands; ++b)
        if (!src_planes_host[b] || !dst_interp_planes_host[b] || !dst_nearest_planes_host[b])
            return fail("xrs_gather_ij2: null plane pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = -1;
    XRS_DISPATCH_DTYPE(dtype, T, rc = launch_dual<T>(src_planes_host, dst_interp_planes_host, dst_nearest_planes_host, n_bands, src_h, src_w, src_pitch, win_i0, win_j0, win_w, win_h, ij, dst_h, dst_w, method, fill_interp, fill_nearest, st));
    if (rc >= 0) return rc;
    // no TMA for this source: two single-method passes (same results)
    rc = xrs_gather_ij(src_planes_host, dst_nearest_planes_host, n_bands, dtype, src_h, src_w, src_pitch, win_i0, win_j0,
                       win_w, win_h, ij, dst_h, dst_w, XRS_NEAREST, fill_nearest, stream);
    if (rc) return rc;
    return xrs_gather_ij(src_planes_host, dst_interp_planes_host, n_bands, dtype, src_h, src_w, src_pitch, win_i0, win_j0,
                         win_w, win_h, ij, dst_h, dst_w, method, fill_interp, stream);
}

}  // extern "C"
