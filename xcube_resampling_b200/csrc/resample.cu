// resample.cu -- K4 + K5: affine resampling (order 0 / 1) fused with block aggregation.
//
//   xrs_affine    affine.py:243-362 (_resample_array / _downscale / _upscale), i.e. what
//                 scipy.ndimage.affine_transform(order<=1, mode="constant", cval) computes per
//                 output sample, followed by the coarsen reducers of coarsen.py:50-155 /
//                 constants.py:51-65 on f_j x f_i windows of those samples
//   xrs_coarsen   plain block aggregation (dask.array.coarsen with the same reducers)
//
// scipy semantics restated (ni_interpolation.c, NI_GeometricTransform; pinned bit-for-bit against
// scipy 1.18 by tests/test_resample_gpu.py):
//   * source coordinate c = out_index * scale + offset (one product, one sum, double);
//   * c < 0 or c > len-1 -> cval, no tolerance;
//   * order 0: index floor(c + 0.5);
//   * order 1: taps floor(c), floor(c)+1 (tap len mirrored to len-2), weights w0 = 1 - t,
//     w1 = 1 - w0; value = sum over taps of v * w_j * w_i accumulated from 0.0 in tap order, so a
//     NaN / inf neighbour contaminates even with weight 0;
//   * for (time, y, x) arrays the order-1 filter also reads slice t+1 (mirrored for the last one)
//     with weight 0: non-finite values there turn the sample into NaN ("slice_blend");
//   * result -> dtype: floats by cast, signed ints round half away from zero, unsigned ints
//     floor(t + 0.5) clipped at 0, both saturating.
// Reducer semantics restated from numpy (nan-reducers for floats, float32 accumulation in numpy's
// pairwise-by-row order so that means are bit-identical for the usual factors).
#include "resample_common.cuh"

namespace xrs {

// One intermediate sample of slice `sl` at intermediate index (J, I); `nx` = slice whose taps
// contaminate with weight zero (nullptr: none).
template <typename T>
__device__ __forceinline__ T affine_sample(const T *__restrict__ sl, const T *__restrict__ nx, int64_t J, int64_t I,
                                           const AffineGeom &g) {
    const double cj = dadd(dmul(static_cast<double>(J), g.j_scale), g.j_off);
    const double ci = dadd(dmul(static_cast<double>(I), g.i_scale), g.i_off);
    if (g.order == 0) {
        if (cj < 0.0 || cj > static_cast<double>(g.src_h - 1) || ci < 0.0 || ci > static_cast<double>(g.src_w - 1))
            return scipy_cast<T>(g.cval);
        const int64_t j = static_cast<int64_t>(floor(dadd(cj, 0.5))), i = static_cast<int64_t>(floor(dadd(ci, 0.5)));
        const T v = __ldg(sl + j * g.src_pitch + i);
        if constexpr (std::is_floating_point<T>::value || sizeof(T) == 8) {
            // scipy adds every sample as a double to 0.0: -0.0 becomes +0.0, int64 beyond 2^53 is rounded
            if (!g.exact_samples) return scipy_cast<T>(dadd(0.0, static_cast<double>(v)));
        }
        return v;
    }
    const Axis1 aj = axis_order1(cj, g.src_h), ai = axis_order1(ci, g.src_w);
    if (!aj.inside || !ai.inside) return scipy_cast<T>(g.cval);
    const T v00 = __ldg(sl + aj.k0 * g.src_pitch + ai.k0), v01 = __ldg(sl + aj.k0 * g.src_pitch + ai.k1);
    const T v10 = __ldg(sl + aj.k1 * g.src_pitch + ai.k0), v11 = __ldg(sl + aj.k1 * g.src_pitch + ai.k1);
    double t = 0.0;
    t = dadd(t, dmul(dmul(static_cast<double>(v00), aj.w0), ai.w0));
    t = dadd(t, dmul(dmul(static_cast<double>(v01), aj.w0), ai.w1));
    t = dadd(t, dmul(dmul(static_cast<double>(v10), aj.w1), ai.w0));
    t = dadd(t, dmul(dmul(static_cast<double>(v11), aj.w1), ai.w1));
    if (nx != nullptr) {
        if (non_finite(__ldg(nx + aj.k0 * g.src_pitch + ai.k0)) || non_finite(__ldg(nx + aj.k0 * g.src_pitch + ai.k1)) ||
            non_finite(__ldg(nx + aj.k1 * g.src_pitch + ai.k0)) || non_finite(__ldg(nx + aj.k1 * g.src_pitch + ai.k1)))
            t = NAN;
    }
    return scipy_cast<T>(t);
}

template <typename T>
__device__ __forceinline__ void insertion_sort(T *w, int n) {
    for (int a = 1; a < n; ++a) {
        const T v = w[a];
        int b = a - 1;
        while (b >= 0 && w[b] > v) { w[b + 1] = w[b]; --b; }
        w[b + 1] = v;
    }
}

// Reduce a window to one value.  OutT is T, or int64 for mode / count / integer sum, prod.
template <typename T, typename OutT>
__device__ __forceinline__ OutT reduce_window(T *w, int f_j, int f_i, int agg) {
    const int n = f_j * f_i;
    constexpr bool FLT = std::is_floating_point<T>::value;
    switch (agg) {
    case XRS_AGG_FIRST: return static_cast<OutT>(w[0]);
    case XRS_AGG_LAST: return static_cast<OutT>(w[n - 1]);
    case XRS_AGG_CENTER: return static_cast<OutT>(w[(f_j / 2) * f_i + f_i / 2]);
    case XRS_AGG_COUNT: {  // np.count_nonzero (NaN is non-zero)
        long long c = 0;
        for (int k = 0; k < n; ++k) c += (w[k] != T(0)) ? 1 : 0;
        return static_cast<OutT>(c);
    }
    case XRS_AGG_MAX:
    case XRS_AGG_MIN: {  // np.nanmax / np.nanmin (fmax / fmin reductions)
        bool any = false;
        T m = T(0);
        for (int k = 0; k < n; ++k) {
            if (is_nan(w[k])) continue;
            if (!any) { m = w[k]; any = true; }
            else if (agg == XRS_AGG_MAX ? (w[k] > m) : (w[k] < m)) m = w[k];
        }
        if (!any) {
            if constexpr (FLT) return static_cast<OutT>(NAN);
        }
        return static_cast<OutT>(m);
    }
    case XRS_AGG_SUM:
    case XRS_AGG_MEAN: {
        if constexpr (FLT) {  // np.nansum / np.nanmean: NaN -> 0, accumulate in T, divide by the count in double
            const T s = numpy_window_sum<T>(f_j, f_i, [&](int k) { return is_nan(w[k]) ? T(0) : w[k]; });
            if (agg == XRS_AGG_SUM) return static_cast<OutT>(s);
            long long c = 0;
            for (int k = 0; k < n; ++k) c += is_nan(w[k]) ? 0 : 1;
            return static_cast<OutT>(static_cast<T>(static_cast<double>(s) / static_cast<double>(c)));
        } else {
            if (agg == XRS_AGG_SUM) {  // np.nansum on integers: exact 64-bit sum
                long long s = 0;
                for (int k = 0; k < n; ++k) s += static_cast<long long>(w[k]);
                return static_cast<OutT>(s);
            }
            // np.mean in float64, then np.rint(...).astype(dtype) (coarsen.py:104-111)
            const double s = numpy_window_sum<double>(f_j, f_i, [&](int k) { return static_cast<double>(w[k]); });
            return static_cast<OutT>(static_cast<long long>(rint(s / static_cast<double>(n))));
        }
    }
    case XRS_AGG_PROD: {  // np.nanprod: NaN -> 1, sequential products
        if constexpr (FLT) {
            T p = T(1);
            for (int k = 0; k < n; ++k) p = p * (is_nan(w[k]) ? T(1) : w[k]);
            return static_cast<OutT>(p);
        } else {
            long long p = 1;
            for (int k = 0; k < n; ++k) p *= static_cast<long long>(w[k]);
            return static_cast<OutT>(p);
        }
    }
    case XRS_AGG_STD:
    case XRS_AGG_VAR: {
        if constexpr (FLT) {  // np.nanvar / np.nanstd in T (numpy/lib/_nanfunctions_impl.py)
            long long c = 0;
            for (int k = 0; k < n; ++k) c += is_nan(w[k]) ? 0 : 1;
            const T s = numpy_window_sum<T>(f_j, f_i, [&](int k) { return is_nan(w[k]) ? T(0) : w[k]; });
            const T avg = static_cast<T>(static_cast<double>(s) / static_cast<double>(c));
            const T sq = numpy_window_sum<T>(f_j, f_i, [&](int k) {
                if (is_nan(w[k])) return T(0);
                const T d = w[k] - avg;
                return static_cast<T>(d * d);
            });
            if (c <= 0) return static_cast<OutT>(NAN);
            const T var = static_cast<T>(static_cast<double>(sq) / static_cast<double>(c));
            return static_cast<OutT>(agg == XRS_AGG_VAR ? var : static_cast<T>(sqrt(static_cast<double>(var))));
        } else {  // np.var / np.std in float64, then rint and cast back
            const double s = numpy_window_sum<double>(f_j, f_i, [&](int k) { return static_cast<double>(w[k]); });
            const double avg = s / static_cast<double>(n);
            const double sq = numpy_window_sum<double>(f_j, f_i, [&](int k) {
                const double d = static_cast<double>(w[k]) - avg;
                return d * d;
            });
            const double var = sq / static_cast<double>(n);
            return static_cast<OutT>(static_cast<long long>(rint(agg == XRS_AGG_VAR ? var : sqrt(var))));
        }
    }
    case XRS_AGG_MEDIAN: {
        int m = 0;  // compact the non-NaN values to the front
        for (int k = 0; k < n; ++k)
            if (!is_nan(w[k])) w[m++] = w[k];
        if (m == 0) {
            if constexpr (FLT) return static_cast<OutT>(NAN);
            return OutT(0);
        }
        insertion_sort(w, m);
        const T b = w[m / 2], a = (m & 1) ? b : w[m / 2 - 1];
        if constexpr (FLT) {  // np.nanmedian of small windows (np.ma.median): (low + high) / 2 in T, summed from +0.0
            return static_cast<OutT>(static_cast<T>(static_cast<T>(static_cast<T>(a + b) + T(0)) * T(0.5)));
        } else {  // float64 mean (np.median: of the middle value alone for odd counts), then rint (half to even), cast
            if (m & 1) return static_cast<OutT>(static_cast<long long>(rint(static_cast<double>(b))));
            return static_cast<OutT>(static_cast<long long>(rint((static_cast<double>(a) + static_cast<double>(b)) / 2.0)));
        }
    }
    case XRS_AGG_MODE: {  // coarsen.py:138-155: most frequent value, lowest value wins ties
        insertion_sort(w, n);
        T best = w[0];
        int best_n = 0, run = 0;
        for (int k = 0; k < n; ++k) {
            run = (k > 0 && w[k] == w[k - 1]) ? run + 1 : 1;
            if (run > best_n) { best_n = run; best = w[k]; }
        }
        return static_cast<OutT>(best);
    }
    default: return OutT(0);
    }
}

// NaN recovery (affine.py:344-360): the zero-filled image and the validity mask go through the same
// order-1 filter; the sample is their quotient, NaN where the mask weight is ~0.  scipy returns the
// filtered image in the array's dtype and the filtered mask in float64, numpy divides in float64.
template <typename T>
__device__ __forceinline__ double affine_sample_recover(const T *__restrict__ sl, const T *__restrict__ nx, int64_t J,
                                                        int64_t I, const AffineGeom &g) {
    const double cj = dadd(dmul(static_cast<double>(J), g.j_scale), g.j_off);
    const double ci = dadd(dmul(static_cast<double>(I), g.i_scale), g.i_off);
    const Axis1 aj = axis_order1(cj, g.src_h), ai = axis_order1(ci, g.src_w);
    double im, norm;
    if (!aj.inside || !ai.inside) {
        im = static_cast<double>(scipy_cast<T>(g.cval));
        norm = g.cval;
    } else {
        const T v[4] = {__ldg(sl + aj.k0 * g.src_pitch + ai.k0), __ldg(sl + aj.k0 * g.src_pitch + ai.k1),
                        __ldg(sl + aj.k1 * g.src_pitch + ai.k0), __ldg(sl + aj.k1 * g.src_pitch + ai.k1)};
        const double wj[4] = {aj.w0, aj.w0, aj.w1, aj.w1}, wi[4] = {ai.w0, ai.w1, ai.w0, ai.w1};
        double t = 0.0, n = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool nan = v[k] != v[k];
            t = dadd(t, dmul(dmul(nan ? 0.0 : static_cast<double>(v[k]), wj[k]), wi[k]));
            n = dadd(n, dmul(dmul(nan ? 0.0 : 1.0, wj[k]), wi[k]));
        }
        if (nx != nullptr) {  // zero-weight taps of the next slice: only +-inf survives the zero filling
            const T u[4] = {__ldg(nx + aj.k0 * g.src_pitch + ai.k0), __ldg(nx + aj.k0 * g.src_pitch + ai.k1),
                            __ldg(nx + aj.k1 * g.src_pitch + ai.k0), __ldg(nx + aj.k1 * g.src_pitch + ai.k1)};
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (u[k] == u[k] && non_finite(u[k])) t = NAN;
        }
        im = static_cast<double>(scipy_cast<T>(t));
        norm = n;
    }
    if (fabs(norm) <= 1e-8) return NAN;  // np.isclose(scaled_norm, 0.0)
    return ddiv(im, norm);
}

// ---------------------------------------------------------------------------
// generic kernel: one thread per output pixel and slice
// ---------------------------------------------------------------------------
template <typename T, typename OutT>
__global__ void __launch_bounds__(256) k4_affine_generic(const T *__restrict__ src, OutT *__restrict__ dst, AffineGeom g) {
    const int64_t oi = static_cast<int64_t>(blockIdx.x) * 32 + threadIdx.x;
    const int64_t oj = static_cast<int64_t>(blockIdx.y) * 8 + threadIdx.y;
    const int64_t sl = blockIdx.z;
    if (oi >= g.dst_w || oj >= g.dst_h) return;
    const T *cur = src + sl * g.src_slice_stride;
    const T *nx = nullptr;
    if (g.slice_blend && g.order == 1 && std::is_floating_point<T>::value) {
        int64_t nsl = sl + 1;
        if (nsl >= g.n_slices) nsl = g.n_slices > 2 ? g.n_slices - 2 : 0;  // mirrored tap; one slice: itself
        nx = src + nsl * g.src_slice_stride;
    }
    OutT *out = dst + (sl * g.dst_h + oj) * g.dst_w + oi;
    const int n = g.f_j * g.f_i;
    if (n == 1) {
        *out = static_cast<OutT>(affine_sample<T>(cur, nx, oj, oi, g));
        return;
    }
    T w[RS_MAX_WINDOW];
    for (int a = 0; a < g.f_j; ++a)
        for (int b = 0; b < g.f_i; ++b) w[a * g.f_i + b] = affine_sample<T>(cur, nx, oj * g.f_j + a, oi * g.f_i + b, g);
    *out = reduce_window<T, OutT>(w, g.f_j, g.f_i, g.agg);
}

template <typename T>
__global__ void __launch_bounds__(256) k4_affine_recover(const T *__restrict__ src, double *__restrict__ dst, AffineGeom g) {
    const int64_t oi = static_cast<int64_t>(blockIdx.x) * 32 + threadIdx.x;
    const int64_t oj = static_cast<int64_t>(blockIdx.y) * 8 + threadIdx.y;
    const int64_t sl = blockIdx.z;
    if (oi >= g.dst_w || oj >= g.dst_h) return;
    const T *cur = src + sl * g.src_slice_stride;
    const T *nx = nullptr;
    if (g.slice_blend) {
        int64_t nsl = sl + 1;
        if (nsl >= g.n_slices) nsl = g.n_slices > 2 ? g.n_slices - 2 : 0;
        nx = src + nsl * g.src_slice_stride;
    }
    double *out = dst + (sl * g.dst_h + oj) * g.dst_w + oi;
    const int n = g.f_j * g.f_i;
    if (n == 1) {
        *out = affine_sample_recover<T>(cur, nx, oj, oi, g);
        return;
    }
    double w[RS_MAX_WINDOW];
    for (int a = 0; a < g.f_j; ++a)
        for (int b = 0; b < g.f_i; ++b) w[a * g.f_i + b] = affine_sample_recover<T>(cur, nx, oj * g.f_j + a, oi * g.f_i + b, g);
    *out = reduce_window<double, double>(w, g.f_j, g.f_i, g.agg);
}

__global__ void __launch_bounds__(256) k4_has_nan_f32(const float *__restrict__ p, int64_t h, int64_t w, int64_t pitch,
                                                      int64_t slice_stride, int32_t *flag) {
    const float *base = p + blockIdx.z * slice_stride;
    bool any = false;
    for (int64_t r = blockIdx.y; r < h; r += gridDim.y)
        for (int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; c < w;
             c += static_cast<int64_t>(gridDim.x) * blockDim.x) {
            const float v = __ldg(base + r * pitch + c);
            any = any || (v != v);
        }
    if (__any_sync(0xffffffffu, any) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}
__global__ void __launch_bounds__(256) k4_has_nan_f64(const double *__restrict__ p, int64_t h, int64_t w, int64_t pitch,
                                                      int64_t slice_stride, int32_t *flag) {
    const double *base = p + blockIdx.z * slice_stride;
    bool any = false;
    for (int64_t r = blockIdx.y; r < h; r += gridDim.y)
        for (int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; c < w;
             c += static_cast<int64_t>(gridDim.x) * blockDim.x) {
            const double v = __ldg(base + r * pitch + c);
            any = any || (v != v);
        }
    if (__any_sync(0xffffffffu, any) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

static bool agg_outputs_int64(int agg, bool is_float) {
    if (agg == XRS_AGG_MODE || agg == XRS_AGG_COUNT) return true;
    if (!is_float && (agg == XRS_AGG_SUM || agg == XRS_AGG_PROD)) return true;
    return false;
}

template <typename T>
static int launch_affine(const void *src, void *dst, const AffineGeom &g, cudaStream_t st) {
    const bool i64 = g.f_j * g.f_i > 1 && agg_outputs_int64(g.agg, std::is_floating_point<T>::value);
    if (g.n_slices > 65535 || ceil_div(g.dst_h, 8) > 65535) return fail("xrs_affine: too many slices or rows for one launch");
    const dim3 block(32, 8);
    const dim3 grid(static_cast<unsigned>(ceil_div(g.dst_w, 32)), static_cast<unsigned>(ceil_div(g.dst_h, 8)),
                    static_cast<unsigned>(g.n_slices));
    if (i64)
        XRS_TIMED("k4_affine_generic", st, k4_affine_generic<T, int64_t><<<grid, block, 0, st>>>(static_cast<const T *>(src), static_cast<int64_t *>(dst), g));
    else
        XRS_TIMED("k4_affine_generic", st, k4_affine_generic<T, T><<<grid, block, 0, st>>>(static_cast<const T *>(src), static_cast<T *>(dst), g));
    XRS_LAUNCH_CHECK("k4_affine_generic");
    return 0;
}

static int affine_entry(const void *src, void *dst, int32_t dtype, int64_t n_slices, int64_t src_h, int64_t src_w,
                        int64_t src_pitch, int64_t src_slice_stride, int64_t dst_h, int64_t dst_w, double j_scale,
                        double j_off, double i_scale, double i_off, int32_t order, double cval, int32_t agg, int32_t f_j,
                        int32_t f_i, int32_t slice_blend, int exact_samples, void *stream) {
    if (!src || !dst) return fail("xrs_affine: null pointer");
    if (order != 0 && order != 1)
        return fail("interp_methods must be one of 0, 1, 'nearest', 'bilinear'. Higher order is not supported for 3D "
                    "arrays in affine transforms, as it causes unintended blending across the non-spatial (e.g., time) "
                    "dimension.");
    if (n_slices < 1 || src_h < 1 || src_w < 1 || src_pitch < src_w || dst_h < 1 || dst_w < 1) return fail("xrs_affine: bad shape");
    if (f_j < 1 || f_i < 1) return fail("xrs_affine: aggregation factors must be >= 1");
    if (f_j * f_i > 1) {
        if (agg < XRS_AGG_CENTER || agg > XRS_AGG_VAR) return fail("xrs_affine: unknown aggregation method");
        if (static_cast<int64_t>(f_j) * f_i > RS_MAX_WINDOW) return fail("xrs_affine: aggregation window larger than 256 samples");
        if (f_i > 128) return fail("xrs_affine: aggregation factor along x larger than 128");
        if (agg == XRS_AGG_MODE && (dtype == XRS_F32 || dtype == XRS_F64))
            return fail("xrs_affine: mode aggregation is implemented for integer data types only");
    }
    AffineGeom g;
    g.n_slices = n_slices; g.src_h = src_h; g.src_w = src_w; g.src_pitch = src_pitch; g.src_slice_stride = src_slice_stride;
    g.dst_h = dst_h; g.dst_w = dst_w;
    g.j_scale = j_scale; g.j_off = j_off; g.i_scale = i_scale; g.i_off = i_off; g.cval = cval;
    g.order = order; g.agg = agg; g.f_j = f_j; g.f_i = f_i; g.slice_blend = slice_blend;
    g.exact_samples = exact_samples;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (f_j * f_i > 1) {  // aligned integer-factor windows: streaming kernels (resample_fast.cu)
        bool handled = false;
        const int rc = launch_affine_fast(src, dst, dtype, g, st, &handled);
        if (rc || handled) return rc;
    }
    XRS_DISPATCH_DTYPE(dtype, T, return launch_affine<T>(src, dst, g, st));
    return 0;
}

}  // namespace xrs

using namespace xrs;

extern "C" {

int xrs_affine(const void *src, void *dst, int32_t dtype, int64_t n_slices, int64_t src_h, int64_t src_w,
               int64_t src_pitch, int64_t src_slice_stride, int64_t dst_h, int64_t dst_w, double j_scale, double j_off,
               double i_scale, double i_off, int32_t order, double cval, int32_t agg, int32_t f_j, int32_t f_i,
               int32_t slice_blend, void *stream) {
    return affine_entry(src, dst, dtype, n_slices, src_h, src_w, src_pitch, src_slice_stride, dst_h, dst_w, j_scale, j_off,
                        i_scale, i_off, order, cval, agg, f_j, f_i, slice_blend, 0, stream);
}

int xrs_coarsen(const void *src, void *dst, int32_t dtype, int64_t n_slices, int64_t src_h, int64_t src_w,
                int64_t src_pitch, int64_t src_slice_stride, int32_t agg, int32_t f_j, int32_t f_i, void *stream) {
    if (f_j < 1 || f_i < 1 || src_h % f_j || src_w % f_i) return fail("xrs_coarsen: factors must divide the image size");
    // identity nearest-neighbour "resample" of the values as stored + aggregation == dask.array.coarsen
    return affine_entry(src, dst, dtype, n_slices, src_h, src_w, src_pitch, src_slice_stride, src_h / f_j, src_w / f_i, 1.0,
                        0.0, 1.0, 0.0, 0, 0.0, agg, f_j, f_i, 0, 1, stream);
}

int xrs_has_nan(const void *src, int32_t dtype, int64_t n_slices, int64_t src_h, int64_t src_w, int64_t src_pitch,
                int64_t src_slice_stride, int32_t *flag, void *stream) {
    if (!src || !flag) return fail("xrs_has_nan: null pointer");
    if (n_slices < 1 || src_h < 1 || src_w < 1 || src_pitch < src_w || n_slices > 65535) return fail("xrs_has_nan: bad shape");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    XRS_CUDA(cudaMemsetAsync(flag, 0, sizeof(int32_t), st));
    if (dtype != XRS_F32 && dtype != XRS_F64) return 0;  // integers hold no NaN
    const dim3 grid(static_cast<unsigned>(std::min<int64_t>(ceil_div(src_w, 256), 64)),
                    static_cast<unsigned>(std::min<int64_t>(src_h, 1024)), static_cast<unsigned>(n_slices));
    if (dtype == XRS_F32)
        XRS_TIMED("k4_has_nan", st, k4_has_nan_f32<<<grid, 256, 0, st>>>(static_cast<const float *>(src), src_h, src_w, src_pitch, src_slice_stride, flag));
    else
        XRS_TIMED("k4_has_nan", st, k4_has_nan_f64<<<grid, 256, 0, st>>>(static_cast<const double *>(src), src_h, src_w, src_pitch, src_slice_stride, flag));
    XRS_LAUNCH_CHECK("k4_has_nan");
    return 0;
}

int xrs_affine_recover(const void *src, double *dst, int32_t dtype, int64_t n_slices, int64_t src_h, int64_t src_w,
                       int64_t src_pitch, int64_t src_slice_stride, int64_t dst_h, int64_t dst_w, double j_scale,
                       double j_off, double i_scale, double i_off, double cval, int32_t agg, int32_t f_j, int32_t f_i,
                       int32_t slice_blend, void *stream) {
    if (!src || !dst) return fail("xrs_affine_recover: null pointer");
    if (dtype != XRS_F32 && dtype != XRS_F64) return fail("xrs_affine_recover: floating-point data only");
    if (n_slices < 1 || src_h < 1 || src_w < 1 || src_pitch < src_w || dst_h < 1 || dst_w < 1) return fail("xrs_affine_recover: bad shape");
    if (f_j < 1 || f_i < 1 || static_cast<int64_t>(f_j) * f_i > RS_MAX_WINDOW || f_i > 128) return fail("xrs_affine_recover: bad aggregation factors");
    if (f_j * f_i > 1 && (agg < XRS_AGG_CENTER || agg > XRS_AGG_VAR || agg == XRS_AGG_MODE || agg == XRS_AGG_COUNT))
        return fail("xrs_affine_recover: aggregation method not available for floating-point NaN recovery");
    if (n_slices > 65535 || ceil_div(dst_h, 8) > 65535) return fail("xrs_affine_recover: too many slices or rows for one launch");
    AffineGeom g;
    g.n_slices = n_slices; g.src_h = src_h; g.src_w = src_w; g.src_pitch = src_pitch; g.src_slice_stride = src_slice_stride;
    g.dst_h = dst_h; g.dst_w = dst_w;
    g.j_scale = j_scale; g.j_off = j_off; g.i_scale = i_scale; g.i_off = i_off; g.cval = cval;
    g.order = 1; g.agg = agg; g.f_j = f_j; g.f_i = f_i; g.slice_blend = slice_blend;
    g.exact_samples = 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const dim3 block(32, 8);
    const dim3 grid(static_cast<unsigned>(ceil_div(dst_w, 32)), static_cast<unsigned>(ceil_div(dst_h, 8)), static_cast<unsigned>(n_slices));
    if (dtype == XRS_F32)
        XRS_TIMED("k4_affine_recover", st, k4_affine_recover<float><<<grid, block, 0, st>>>(static_cast<const float *>(src), dst, g));
    else
        XRS_TIMED("k4_affine_recover", st, k4_affine_recover<double><<<grid, block, 0, st>>>(static_cast<const double *>(src), dst, g));
    XRS_LAUNCH_CHECK("k4_affine_recover");
    return 0;
}

}  // extern "C"
