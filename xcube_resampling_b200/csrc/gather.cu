// gather.cu -- K2: gather of all bands through the source-index (ij) image.
//
//   xrs_gather_ij   rectify.py:579-734 (_compute_var_image* / _for_dest_line)
//
// Two kernels share the per-pixel arithmetic (fp64, no FMA contraction, one cast with x86's results,
// xrs_casts.h):
//   * k2_gather_staged: one CTA per 32x32 target tile.  The CTA reduces the bounding box of the
//     source pixels its ij values reach and pulls that box of every band into shared memory with
//     TMA tensor copies (cp.async.bulk.tensor.2d, one 64x48 box per band, 4-stage mbarrier ring),
//     so the irregular 1/4-tap reads hit shared memory instead of issuing ~7 L1 wavefronts each.
//     Needs a 16-byte aligned source pitch (TMA global strides); tiles whose box exceeds 64x48
//     take the direct path inside the same kernel.
//   * k2_gather_direct: plain per-pixel global loads, for sources whose pitch TMA cannot describe.
#include "gather_common.cuh"

namespace xrs {

// Where a gather kernel gets the fractional source index of a target pixel from: the ij image of
// xrs_rectify_ij, or -- fused mode (xrs_rectify_gather) -- straight from K1's claim words, running
// the resolve step (rectify_common.cuh) in registers so that the 16 bytes per pixel of ij are neither
// written nor read back.
struct IjSource {
    const double *ij;  // (2, dst_h, dst_w), or nullptr in fused mode
    IjGeom geom;       // fused mode: claims, source coordinates, tile windows, target grid
};

template <bool FUSED>
__device__ __forceinline__ void load_ij(const IjSource &s, int64_t r, int64_t c, int64_t dst_h, int64_t dst_w,
                                        double &fi, double &fj) {
    const int64_t o = r * dst_w + c;
    if (!FUSED) {
        fi = ld_stream(s.ij + o);
        fj = ld_stream(s.ij + dst_h * dst_w + o);
    } else {
        resolve_pixel(s.geom, s.geom.row_begin + r, c, __ldcs(s.geom.claims + o), fi, fj);
    }
}

// ---------------------------------------------------------------------------
// direct kernel
// ---------------------------------------------------------------------------
constexpr int K2_BX = 32, K2_BY = 8;

template <typename T>
struct PlaneTable {
    const T *src[K2_MAX_BANDS];
    T *dst[K2_MAX_BANDS];
};

template <typename T, int METHOD, bool FUSED>
__global__ void __launch_bounds__(K2_BX *K2_BY)
k2_gather_direct(PlaneTable<T> planes, int n_bands, int64_t src_h, int64_t src_w, int64_t src_pitch, int64_t win_i0,
                 int64_t win_j0, const __grid_constant__ IjSource ijs, int64_t dst_h, int64_t dst_w, T fill) {
    const int64_t c = static_cast<int64_t>(blockIdx.x) * K2_BX + threadIdx.x;
    const int64_t r = static_cast<int64_t>(blockIdx.y) * K2_BY + threadIdx.y;
    if (c >= dst_w || r >= dst_h) return;
    const int64_t o = r * dst_w + c;
    double fi_, fj_;
    load_ij<FUSED>(ijs, r, c, dst_h, dst_w, fi_, fj_);
    const Taps t = make_taps<METHOD>(fi_, fj_, src_w, src_h);
    if (!t.valid) {
        for (int b = 0; b < n_bands; ++b) st_stream(planes.dst[b] + o, fill);
        return;
    }
    const int64_t o00 = (t.j0 - win_j0) * src_pitch + (t.i0 - win_i0), o01 = o00 + (t.i1 - t.i0);
    const int64_t o10 = o00 + (t.j1 - t.j0) * src_pitch, o11 = o10 + (t.i1 - t.i0);
    if (METHOD == XRS_NEAREST) {
#pragma unroll 8
        for (int b = 0; b < n_bands; ++b) st_stream(planes.dst[b] + o, nearest_value(__ldg(planes.src[b] + o00)));
        return;
    }
#pragma unroll 4
    for (int b = 0; b < n_bands; ++b) {
        const T *sp = planes.src[b];
        const double val = interp_value<METHOD>(ld_f64(sp + o00), ld_f64(sp + o01), ld_f64(sp + o10), ld_f64(sp + o11),
                                                t.u, t.v);
        st_stream(planes.dst[b] + o, cast_like_numpy<T>(val));
    }
}

// ---------------------------------------------------------------------------
// staged kernel (TMA tensor tiles -> shared memory)
// ---------------------------------------------------------------------------
// tile constants: gather_common.cuh

template <typename T>
struct StagedParams {
    CUtensorMap maps[K2_MAX_BANDS];
    const T *src[K2_MAX_BANDS];
    T *dst[K2_MAX_BANDS];
};

template <typename T, int METHOD, bool FUSED>
__global__ void __launch_bounds__(K2S_THREADS, (!FUSED && METHOD == XRS_NEAREST) ? 4 : 3)
k2_gather_staged(const __grid_constant__ StagedParams<T> p, int n_bands, int64_t src_h, int64_t src_w,
                 int64_t src_pitch, int64_t win_i0, int64_t win_j0, const __grid_constant__ IjSource ijs, int64_t dst_h,
                 int64_t dst_w, T fill) {
    // TMA tensor copies need a 128-byte aligned shared-memory destination; static __shared__
    // variables would shift the dynamic segment, so everything lives in it behind an aligned base.
    extern __shared__ unsigned char k2s_smem_raw[];
    constexpr int STAGE_ELEMS = K2S_BOX_W * K2S_BOX_H;
    unsigned char *k2s_smem = k2s_smem_raw + ((128u - (smem_u32(k2s_smem_raw) & 127u)) & 127u);
    T *stages = reinterpret_cast<T *>(k2s_smem);
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(k2s_smem + static_cast<size_t>(K2S_STAGES) * STAGE_ELEMS * sizeof(T));
    int(*red)[K2S_THREADS / 32] = reinterpret_cast<int(*)[K2S_THREADS / 32]>(full_bar + K2S_STAGES);

    const int tid = threadIdx.x;
    const int tx = tid % K2S_TW, ty = tid / K2S_TW;
    const int64_t c = static_cast<int64_t>(blockIdx.x) * K2S_TW + tx;
    const int64_t r_base = static_cast<int64_t>(blockIdx.y) * K2S_TH + ty;  // rows r_base + k * K2S_ROW_STEP
    const bool col_in = c < dst_w;

    // ---- this thread's pixels: source taps and fractions --------------------------------
    double fi[K2S_PX], fj[K2S_PX];
#pragma unroll
    for (int k = 0; k < K2S_PX; ++k) {
        const int64_t r = r_base + k * K2S_ROW_STEP;
        const bool in = col_in && r < dst_h;
        fi[k] = fj[k] = NAN;
        if (in) load_ij<FUSED>(ijs, r, c, dst_h, dst_w, fi[k], fj[k]);
    }
    Taps t[K2S_PX];
    int i_lo = INT32_MAX, i_hi = -1, j_lo = INT32_MAX, j_hi = -1;
#pragma unroll
    for (int k = 0; k < K2S_PX; ++k) {
        t[k] = make_taps<METHOD>(fi[k], fj[k], src_w, src_h);
        if (t[k].valid) {
            i_lo = min(i_lo, t[k].i0); i_hi = max(i_hi, t[k].i1);
            j_lo = min(j_lo, t[k].j0); j_hi = max(j_hi, t[k].j1);
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
                    if (r < dst_h) st_stream(p.dst[b] + r * dst_w + c, fill);
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
        // Everything that does not depend on the band is computed once: the four tap addresses of each
        // pixel inside stage 0 (the other stages are compile-time offsets from them -- the band loop is
        // unrolled over the ring), the output element offsets and the store predicates.  Pixels
        // without a source read tap (0, 0) with u = v = 0 and are overwritten by `fill` with one
        // select, so the band loop is branch-free.
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
        // opaque to the compiler, so that the band loop tests one bit instead of re-deriving the 64-bit
        // row / column comparisons for every band and pixel
        asm volatile("" : "+r"(st_mask));
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
                T out[K2S_PX];
#pragma unroll
                for (int k = 0; k < K2S_PX; ++k) {
                    if (METHOD == XRS_NEAREST) {
                        out[k] = nearest_value(t00[k][s * STAGE_ELEMS]);
                    } else {
                        const double v00 = static_cast<double>(t00[k][s * STAGE_ELEMS]);
                        const double v01 = static_cast<double>(t01[k][s * STAGE_ELEMS]);
                        const double v10 = static_cast<double>(t10[k][s * STAGE_ELEMS]);
                        const double v11 = static_cast<double>(t11[k][s * STAGE_ELEMS]);
                        out[k] = cast_like_numpy<T>(interp_value<METHOD>(v00, v01, v10, v11, t[k].u, t[k].v));
                    }
                    out[k] = t[k].valid ? out[k] : fill;
                }
                T *dp = p.dst[b];
#pragma unroll
                for (int k = 0; k < K2S_PX; ++k)
                    if (st_mask & (1u << k)) st_stream(elem_ptr(dp, o32[k]), out[k]);
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

    // ---- box too large for the staging buffers: direct global taps ----------------------
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
        T out[K2S_PX];
#pragma unroll
        for (int k = 0; k < K2S_PX; ++k) {
            if (!t[k].valid) {
                out[k] = fill;
            } else if (METHOD == XRS_NEAREST) {
                out[k] = nearest_value(__ldg(sp + o00[k]));
            } else {
                out[k] = cast_like_numpy<T>(interp_value<METHOD>(ld_f64(sp + o00[k]), ld_f64(sp + o00[k] + od[k]),
                                                                ld_f64(sp + o00[k] + oj[k]),
                                                                ld_f64(sp + o00[k] + oj[k] + od[k]), t[k].u, t[k].v));
            }
        }
#pragma unroll
        for (int k = 0; k < K2S_PX; ++k) {
            const int64_t r = r_base + k * K2S_ROW_STEP;
            if (r < dst_h) st_stream(p.dst[b] + r * dst_w + c, out[k]);
        }
    }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
        else
            cudaGetLastError();
    }
    return fn;
}

bool tma_available() { return get_encode_tiled() != nullptr; }

// 2-D tensor map over a (height, width) plane of `elem_size`-byte elements with row pitch `pitch_bytes`
// (a multiple of 16) and a (box_h, box_w) box; out-of-bounds elements read as zero.
bool tma_encode_2d(CUtensorMap *map, int elem_size, const void *base, uint64_t width, uint64_t height,
                   uint64_t pitch_bytes, uint32_t box_w, uint32_t box_h) {
    EncodeTiledFn fn = get_encode_tiled();
    if (!fn) return false;
    const CUtensorMapDataType dt = elem_size == 1   ? CU_TENSOR_MAP_DATA_TYPE_UINT8
                                   : elem_size == 2 ? CU_TENSOR_MAP_DATA_TYPE_UINT16
                                   : elem_size == 4 ? CU_TENSOR_MAP_DATA_TYPE_UINT32
                                                    : CU_TENSOR_MAP_DATA_TYPE_UINT64;
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(width), static_cast<cuuint64_t>(height)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(pitch_bytes)};
    const cuuint32_t box[2] = {box_w, box_h};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, dt, 2, const_cast<void *>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <typename T, int METHOD, bool FUSED>
static int launch_staged(const StagedParams<T> &sp, int nb, int64_t src_h, int64_t src_w, int64_t src_pitch,
                         int64_t win_i0, int64_t win_j0, const IjSource &ij, int64_t dst_h, int64_t dst_w, T fill,
                         cudaStream_t st) {
    const size_t smem = static_cast<size_t>(K2S_STAGES) * K2S_BOX_W * K2S_BOX_H * sizeof(T) +
                        K2S_STAGES * sizeof(uint64_t) + 4 * (K2S_THREADS / 32) * sizeof(int) + 128;
    XRS_CUDA(cudaFuncSetAttribute(k2_gather_staged<T, METHOD, FUSED>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(smem)));
    const dim3 grid(static_cast<unsigned>(ceil_div(dst_w, K2S_TW)), static_cast<unsigned>(ceil_div(dst_h, K2S_TH)));
    XRS_TIMED(METHOD == XRS_NEAREST ? "k2_gather_staged<nearest>" : METHOD == XRS_BILINEAR ? "k2_gather_staged<bilinear>" : "k2_gather_staged<triangular>", st, k2_gather_staged<T, METHOD, FUSED><<<grid, K2S_THREADS, smem, st>>>(sp, nb, src_h, src_w, src_pitch, win_i0, win_j0, ij,
                                                                 dst_h, dst_w, fill));
    XRS_LAUNCH_CHECK("k2_gather_staged");
    return 0;
}

template <typename T, bool FUSED>
static int launch_gather(const void *const *src_planes, void *const *dst_planes, int n_bands, int64_t src_h,
                         int64_t src_w, int64_t src_pitch, int64_t win_i0, int64_t win_j0, int64_t win_w,
                         int64_t win_h, const IjSource &ij, int64_t dst_h, int64_t dst_w, int method, double fill,
                         cudaStream_t st) {
    const T fill_t = cast_fill<T>(fill);
    // TMA needs 16-byte aligned plane bases and row strides
    bool tma_ok = (src_pitch * sizeof(T)) % 16 == 0 && win_w < (1ll << 31) && win_h < (1ll << 31) &&
                  ceil_div(dst_h, K2S_TH) <= 65535 && dst_h * dst_w < (1ll << 32) && tma_available();
    for (int b = 0; b < n_bands && tma_ok; ++b)
        tma_ok = (reinterpret_cast<uintptr_t>(src_planes[b]) & 15) == 0;

    for (int b0 = 0; b0 < n_bands; b0 += K2_MAX_BANDS) {
        const int nb = std::min(K2_MAX_BANDS, n_bands - b0);
        if (tma_ok) {
            StagedParams<T> sp;
            memset(&sp, 0, sizeof(sp));
            bool ok = true;
            for (int b = 0; b < nb && ok; ++b) {
                sp.src[b] = static_cast<const T *>(src_planes[b0 + b]);
                sp.dst[b] = static_cast<T *>(dst_planes[b0 + b]);
                ok = tma_encode_2d(&sp.maps[b], sizeof(T), src_planes[b0 + b], static_cast<uint64_t>(win_w),
                                   static_cast<uint64_t>(win_h), static_cast<uint64_t>(src_pitch) * sizeof(T), K2S_BOX_W,
                                   K2S_BOX_H);
            }
            if (ok) {
                int rc;
                switch (method) {
                case XRS_NEAREST:
                    rc = launch_staged<T, XRS_NEAREST, FUSED>(sp, nb, src_h, src_w, src_pitch, win_i0, win_j0, ij, dst_h, dst_w, fill_t, st);
                    break;
                case XRS_BILINEAR:
                    rc = launch_staged<T, XRS_BILINEAR, FUSED>(sp, nb, src_h, src_w, src_pitch, win_i0, win_j0, ij, dst_h, dst_w, fill_t, st);
                    break;
                default:
                    rc = launch_staged<T, XRS_TRIANGULAR, FUSED>(sp, nb, src_h, src_w, src_pitch, win_i0, win_j0, ij, dst_h, dst_w, fill_t, st);
                    break;
                }
                if (rc) return rc;
                continue;
            }
        }
        if (ceil_div(dst_h, K2_BY) > 65535) return fail("xrs_gather_ij: target too tall for one launch");
        PlaneTable<T> pt;
        for (int b = 0; b < K2_MAX_BANDS; ++b) {
            pt.src[b] = b < nb ? static_cast<const T *>(src_planes[b0 + b]) : nullptr;
            pt.dst[b] = b < nb ? static_cast<T *>(dst_planes[b0 + b]) : nullptr;
        }
        const dim3 block(K2_BX, K2_BY);
        const dim3 grid(static_cast<unsigned>(ceil_div(dst_w, K2_BX)), static_cast<unsigned>(ceil_div(dst_h, K2_BY)));
        switch (method) {
        case XRS_NEAREST:
            XRS_TIMED("k2_gather_direct", st, k2_gather_direct<T, XRS_NEAREST, FUSED><<<grid, block, 0, st>>>(pt, nb, src_h, src_w, src_pitch, win_i0, win_j0, ij, dst_h, dst_w, fill_t));
            break;
        case XRS_BILINEAR:
            XRS_TIMED("k2_gather_direct", st, k2_gather_direct<T, XRS_BILINEAR, FUSED><<<grid, block, 0, st>>>(pt, nb, src_h, src_w, src_pitch, win_i0, win_j0, ij, dst_h, dst_w, fill_t));
            break;
        default:
            XRS_TIMED("k2_gather_direct", st, k2_gather_direct<T, XRS_TRIANGULAR, FUSED><<<grid, block, 0, st>>>(pt, nb, src_h, src_w, src_pitch, win_i0, win_j0, ij, dst_h, dst_w, fill_t));
            break;
        }
        XRS_LAUNCH_CHECK("k2_gather_direct");
    }
    return 0;
}

}  // namespace xrs

using namespace xrs;

extern "C" {

int xrs_gather_ij(const void *const *src_planes_host, void *const *dst_planes_host, int32_t n_bands, int32_t dtype,
                  int64_t src_h, int64_t src_w, int64_t src_pitch, int64_t win_i0, int64_t win_j0, int64_t win_w,
                  int64_t win_h, const double *ij, int64_t dst_h, int64_t dst_w, int32_t method, double fill,
                  void *stream) {
    if (!src_planes_host || !dst_planes_host || !ij) return fail("xrs_gather_ij: null pointer");
    if (n_bands < 1) return fail("xrs_gather_ij: n_bands must be >= 1");
    if (method != XRS_NEAREST && method != XRS_BILINEAR && method != XRS_TRIANGULAR)
        return fail("interp_methods must be one of 0, 1, 'nearest', 'bilinear', 'triangular'");
    if (src_h < 1 || src_w < 1 || src_pitch < 1 || dst_h < 1 || dst_w < 1) return fail("xrs_gather_ij: bad shape");
    if (src_w > INT32_MAX || src_h > INT32_MAX) return fail("xrs_gather_ij: source too large");
    if (win_i0 < 0 || win_j0 < 0 || win_w < 1 || win_h < 1 || win_i0 + win_w > src_w || win_j0 + win_h > src_h ||
        src_pitch < win_w)
        return fail("xrs_gather_ij: bad source window");
    for (int b = 0; b < n_bands; ++b)
        if (!src_planes_host[b] || !dst_planes_host[b]) return fail("xrs_gather_ij: null plane pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    IjSource ijs;
    memset(&ijs, 0, sizeof(ijs));
    ijs.ij = ij;
    XRS_DISPATCH_DTYPE(dtype, T, return launch_gather<T, false>(src_planes_host, dst_planes_host, n_bands, src_h, src_w, src_pitch, win_i0, win_j0, win_w, win_h, ijs, dst_h, dst_w, method, fill, st));
    return 0;
}

int xrs_rectify_gather(const double *x, const double *y, int64_t src_h, int64_t src_w, int64_t src_pitch,
                       const int64_t *tile_boxes, int64_t dst_h, int64_t dst_w, int32_t tile_h, int32_t tile_w,
                       double x_min, double y_min, double y_max, double x_res, double y_res, int32_t is_j_axis_up,
                       double uv_delta, int64_t row_begin, int64_t row_end, const int32_t *src_col_ranges,
                       void *workspace, const void *const *src_planes_host, void *const *dst_planes_host, int32_t n_bands, int32_t dtype,
                       int64_t data_pitch, int64_t win_i0, int64_t win_j0, int64_t win_w, int64_t win_h, int32_t method,
                       double fill, void *stream) {
    if (!src_planes_host || !dst_planes_host) return fail("xrs_rectify_gather: null pointer");
    if (n_bands < 1) return fail("xrs_rectify_gather: n_bands must be >= 1");
    if (method != XRS_NEAREST && method != XRS_BILINEAR && method != XRS_TRIANGULAR)
        return fail("interp_methods must be one of 0, 1, 'nearest', 'bilinear', 'triangular'");
    if (src_w > INT32_MAX || src_h > INT32_MAX) return fail("xrs_rectify_gather: source too large");
    if (win_i0 < 0 || win_j0 < 0 || win_w < 1 || win_h < 1 || win_i0 + win_w > src_w || win_j0 + win_h > src_h ||
        data_pitch < win_w)
        return fail("xrs_rectify_gather: bad source window");
    for (int b = 0; b < n_bands; ++b)
        if (!src_planes_host[b] || !dst_planes_host[b]) return fail("xrs_rectify_gather: null plane pointer");
    IjSource ijs;
    memset(&ijs, 0, sizeof(ijs));
    if (int rc = k1_make_geom("xrs_rectify_gather", x, y, src_h, src_w, src_pitch, tile_boxes, dst_h, dst_w, tile_h, tile_w,
                              x_min, y_min, y_max, x_res, y_res, is_j_axis_up, uv_delta, row_begin, row_end, workspace,
                              &ijs.geom))
        return rc;
    ijs.geom.fp_cols = src_col_ranges;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (int rc = k1_enqueue_claims(ijs.geom, st)) return rc;
    const int64_t n_rows = row_end - row_begin;
    XRS_DISPATCH_DTYPE(dtype, T, return launch_gather<T, true>(src_planes_host, dst_planes_host, n_bands, src_h, src_w, data_pitch, win_i0, win_j0, win_w, win_h, ijs, n_rows, dst_w, method, fill, st));
    return 0;
}

}  // extern "C"
