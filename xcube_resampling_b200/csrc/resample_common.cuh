// resample_common.cuh -- pieces shared by the generic (resample.cu) and the streaming
// (resample_fast.cu) affine / coarsen kernels: geometry, scipy's output conversion, numpy's
// summation order.
#pragma once

#include "common.cuh"

namespace xrs {


constexpr int RS_MAX_WINDOW = 256;  // f_j * f_i samples buffered per output pixel (generic kernel)

struct AffineGeom {
    int64_t n_slices, src_h, src_w, src_pitch, src_slice_stride;
    int64_t dst_h, dst_w;
    double j_scale, j_off, i_scale, i_off;
    double cval;
    int order, agg, f_j, f_i, slice_blend;
    // order-0 samples are the source values as stored (xrs_coarsen: dask's coarsen never converts); otherwise
    // they take scipy's float64 round trip, which only 64-bit integers above 2^53 notice
    int exact_samples;
};

// ---------------------------------------------------------------------------
// scipy output conversion (CASE_INTERP_OUT*) with the results scipy gets on x86 where C leaves the
// conversion undefined: NaN -> INT32_MIN / INT64_MIN for 32- / 64-bit signed outputs (0 for narrower and
// unsigned ones, whose conversion goes through a wider integer); 2^63 after the +0.5 -> INT64_MIN;
// anything above -> INT64_MAX.  Written out so that the device and the host build agree.
// ---------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T scipy_cast(double t) {
    if constexpr (std::is_floating_point<T>::value) {
        return static_cast<T>(t);
    } else if constexpr (std::is_unsigned<T>::value) {
        t = t > 0 ? t + 0.5 : 0.0;
        const double mx = static_cast<double>(std::numeric_limits<T>::max());
        t = t > mx ? mx : t;
        t = t < 0 ? 0.0 : t;
        return static_cast<T>(static_cast<unsigned long long>(t));
    } else {
        t = t > 0 ? t + 0.5 : t - 0.5;
        if (t != t) return sizeof(T) >= 4 ? std::numeric_limits<T>::min() : T(0);
        const double mx = static_cast<double>(std::numeric_limits<T>::max());
        const double mn = static_cast<double>(std::numeric_limits<T>::min());
        if (t > mx) return std::numeric_limits<T>::max();
        if (t < mn) return std::numeric_limits<T>::min();
        if constexpr (sizeof(T) == 8) {
            if (t == mx) return std::numeric_limits<T>::min();  // double(INT64_MAX) is 2^63
        }
        return static_cast<T>(static_cast<long long>(t));
    }
}

template <typename T>
__device__ __forceinline__ bool non_finite(T v) {
    if constexpr (std::is_floating_point<T>::value) return !isfinite(static_cast<double>(v));
    return false;
}

// one axis of the order-1 filter: taps and weights, or outside
struct Axis1 {
    int64_t k0, k1;
    double w0, w1;
    bool inside;
};
__device__ __forceinline__ Axis1 axis_order1(double c, int64_t len) {
    Axis1 a;
    a.inside = !(c < 0.0 || c > static_cast<double>(len - 1));  // NaN coordinate -> treated as inside by scipy; cannot occur
    const double f = floor(c);
    a.k0 = static_cast<int64_t>(f);
    a.k1 = a.k0 + 1;
    if (a.k1 >= len) a.k1 = len > 2 ? len - 2 : 0;  // mirror (ni_interpolation.c edge handling)
    const double t = dsub(c, f);
    a.w0 = dsub(1.0, t);
    a.w1 = dsub(1.0, a.w0);
    return a;
}

// ---------------------------------------------------------------------------
// reducers over a window w[0 .. f_j*f_i) stored row-major
// ---------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ bool is_nan(T v) {
    if constexpr (std::is_floating_point<T>::value) return v != v;
    return false;
}

// numpy's pairwise_sum for one contiguous run of n <= 128 elements (umath loops, used for the
// innermost reduction axis); `get(k)` yields element k with NaN already replaced.
template <typename A, typename Get>
__device__ __forceinline__ A numpy_row_sum(int n, Get get) {
    if (n < 8) {
        A res = A(0);
        for (int k = 0; k < n; ++k) res = res + get(k);
        return res;
    }
    A r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = get(k);
    int i = 8;
    for (; i < n - (n % 8); i += 8) {
#pragma unroll
        for (int k = 0; k < 8; ++k) r[k] = r[k] + get(i + k);
    }
    A res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
    for (; i < n; ++i) res = res + get(i);
    return res;
}

// np.sum over the two window axes of the (h, f_j, w, f_i) view: innermost axis pairwise, rows
// accumulated sequentially into the output element (starting from the identity 0).
template <typename A, typename Get>
__device__ __forceinline__ A numpy_window_sum(int f_j, int f_i, Get get) {
    A s = A(0);
    for (int a = 0; a < f_j; ++a) s = s + numpy_row_sum<A>(f_i, [&](int k) { return get(a * f_i + k); });
    return s;
}


// resample_fast.cu: streaming kernels for the aligned integer-factor cases.  Sets *handled when it
// launched; otherwise the caller runs the generic kernel.
int launch_affine_fast(const void *src, void *dst, int dtype, const AffineGeom &g, cudaStream_t st, bool *handled);

}  // namespace xrs
