// resample_fast.cu -- K5 streaming kernels: block aggregation (and the aligned integer-factor case
// of affine down-scaling) at HBM speed.
//
//   xrs_coarsen / xrs_affine when the intermediate samples fall exactly on source pixels
//   (scale 1, non-negative integer offsets, every sample inside the source) and the window is
//   2x2, 4x4 or 8x8 -- i.e. dask.array.coarsen(agg, ...) of coarsen.py:50-155 and the down-scaling
//   branch of affine.py:277-313 for aligned grids (BASELINE configs C1 and C4).
//
// One thread owns one output pixel: it pulls the F rows of its F x F window with 4..16-byte vector
// loads (a warp reads F contiguous row segments -> fully coalesced, F*F/4 independent requests in
// flight per thread), keeps the window in registers and reduces it with numpy's exact semantics
// (resample_common.cuh).  Median and mode sort the window with a fully unrolled bitonic network
// (static register indexing, no local memory) -- 4x4 in 80 and 8x8 in 672 compare-exchanges.
//
// Order-1 resampling at integer coordinates has weights (1, 0): the value is the source pixel, but
// scipy still multiplies the right / lower neighbours by zero, so a non-finite neighbour turns the
// sample into NaN (and -0.0 becomes +0.0).  MODE_BLEND reproduces that from one extra row and
// column (mirrored at the image edge like scipy's tap `len` -> `len - 2`).
#include "resample_common.cuh"

namespace xrs {

constexpr int MODE_PLAIN = 0;  // sample == source pixel
constexpr int MODE_BLEND = 1;  // order-1 taps with zero weight contaminate (floats only)

constexpr int CLASS_SIMPLE = 0;  // everything except median / mode
constexpr int CLASS_SORT = 1;    // median, mode

struct FastGeom {
    int64_t n_slices, src_h, src_w, src_pitch, src_slice_stride, dst_h, dst_w;
    int64_t j_off, i_off;
    int agg;
    int vec;  // 1: rows may be read with vector loads
};

// ---- loading F consecutive elements --------------------------------------------------------
template <typename T, int F>
__device__ __forceinline__ void load_row(const T *__restrict__ p, T (&out)[F], bool vec) {
    constexpr int BYTES = F * static_cast<int>(sizeof(T));
    if (vec) {
        if constexpr (BYTES >= 16) {
            const uint4 *q = reinterpret_cast<const uint4 *>(p);
            uint4 *o = reinterpret_cast<uint4 *>(out);
#pragma unroll
            for (int k = 0; k < BYTES / 16; ++k) o[k] = __ldcs(q + k);
            return;
        } else if constexpr (BYTES == 8) {
            *reinterpret_cast<uint2 *>(out) = __ldcs(reinterpret_cast<const uint2 *>(p));
            return;
        } else if constexpr (BYTES == 4) {
            *reinterpret_cast<uint32_t *>(out) = __ldcs(reinterpret_cast<const uint32_t *>(p));
            return;
        } else if constexpr (BYTES == 2) {
            *reinterpret_cast<uint16_t *>(out) = __ldcs(reinterpret_cast<const uint16_t *>(p));
            return;
        }
    }
#pragma unroll
    for (int k = 0; k < F; ++k) out[k] = __ldg(p + k);
}

// ---- sorting network ---------------------------------------------------------------------------
// NaNs never reach the network (mapped to +inf before sorting), so the IEEE min / max instructions
// order the values exactly like the comparison-based exchange; +0 and -0 compare equal in numpy's
// sort as well, so which of them ends up first is immaterial to the reducers.
__device__ __forceinline__ float sort_min(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ float sort_max(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double sort_min(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ double sort_max(double a, double b) { return fmax(a, b); }
template <typename T>
__device__ __forceinline__ T sort_min(T a, T b) { return a < b ? a : b; }
template <typename T>
__device__ __forceinline__ T sort_max(T a, T b) { return a < b ? b : a; }
template <int N, typename T>
__device__ __forceinline__ void bitonic_sort(T (&a)[N]) {
#pragma unroll
    for (int k = 2; k <= N; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const int l = i ^ j;
                if (l > i) {  // compare-exchange as a min / max pair (FMNMX / VIMNMX: 2 instructions)
                    const bool up = (i & k) == 0;
                    const T x = a[i], y = a[l];
                    const T lo = sort_min(x, y), hi = sort_max(x, y);
                    a[i] = up ? lo : hi;
                    a[l] = up ? hi : lo;
                }
            }
        }
    }
}

template <int N, typename T>
__device__ __forceinline__ T pick(const T (&a)[N], int idx) {
    T v = a[0];
#pragma unroll
    for (int k = 1; k < N; ++k) v = (k == idx) ? a[k] : v;
    return v;
}

// ---- reducers on a register window w[F*F] (row-major), numpy semantics as in resample.cu ------
template <typename T, typename OutT, int F>
__device__ __forceinline__ OutT reduce_simple(const T (&w)[F * F], int agg) {
    constexpr int N = F * F;
    constexpr bool FLT = std::is_floating_point<T>::value;
    switch (agg) {
    case XRS_AGG_FIRST: return static_cast<OutT>(w[0]);
    case XRS_AGG_LAST: return static_cast<OutT>(w[N - 1]);
    case XRS_AGG_CENTER: return static_cast<OutT>(w[(F / 2) * F + F / 2]);
    case XRS_AGG_COUNT: {
        long long c = 0;
#pragma unroll
        for (int k = 0; k < N; ++k) c += (w[k] != T(0)) ? 1 : 0;
        return static_cast<OutT>(c);
    }
    case XRS_AGG_MAX:
    case XRS_AGG_MIN: {
        bool any = false;
        T m = T(0);
        const bool mx = agg == XRS_AGG_MAX;
#pragma unroll
        for (int k = 0; k < N; ++k) {
            const bool nan = is_nan(w[k]);
            const bool better = !nan && (!any || (mx ? (w[k] > m) : (w[k] < m)));
            m = better ? w[k] : m;
            any = any || !nan;
        }
        if constexpr (FLT) {
            if (!any) return static_cast<OutT>(NAN);
        }
        return static_cast<OutT>(m);
    }
    case XRS_AGG_SUM:
    case XRS_AGG_MEAN: {
        if constexpr (FLT) {
            const T s = numpy_window_sum<T>(F, F, [&](int k) { return is_nan(w[k]) ? T(0) : w[k]; });
            if (agg == XRS_AGG_SUM) return static_cast<OutT>(s);
            long long c = 0;
#pragma unroll
            for (int k = 0; k < N; ++k) c += is_nan(w[k]) ? 0 : 1;
            return static_cast<OutT>(static_cast<T>(static_cast<double>(s) / static_cast<double>(c)));
        } else {
            if (agg == XRS_AGG_SUM) {
                long long s = 0;
#pragma unroll
                for (int k = 0; k < N; ++k) s += static_cast<long long>(w[k]);
                return static_cast<OutT>(s);
            }
            const double s = numpy_window_sum<double>(F, F, [&](int k) { return static_cast<double>(w[k]); });
            return static_cast<OutT>(static_cast<long long>(rint(s / static_cast<double>(N))));
        }
    }
    case XRS_AGG_PROD: {
        if constexpr (FLT) {
            T p = T(1);
#pragma unroll
            for (int k = 0; k < N; ++k) p = p * (is_nan(w[k]) ? T(1) : w[k]);
            return static_cast<OutT>(p);
        } else {
            long long p = 1;
#pragma unroll
            for (int k = 0; k < N; ++k) p *= static_cast<long long>(w[k]);
            return static_cast<OutT>(p);
        }
    }
    case XRS_AGG_STD:
    case XRS_AGG_VAR: {
        if constexpr (FLT) {
            long long c = 0;
#pragma unroll
            for (int k = 0; k < N; ++k) c += is_nan(w[k]) ? 0 : 1;
            const T s = numpy_window_sum<T>(F, F, [&](int k) { return is_nan(w[k]) ? T(0) : w[k]; });
            const T avg = static_cast<T>(static_cast<double>(s) / static_cast<double>(c));
            const T sq = numpy_window_sum<T>(F, F, [&](int k) {
                if (is_nan(w[k])) return T(0);
                const T d = w[k] - avg;
                return static_cast<T>(d * d);
            });
            if (c <= 0) return static_cast<OutT>(NAN);
            const T var = static_cast<T>(static_cast<double>(sq) / static_cast<double>(c));
            return static_cast<OutT>(agg == XRS_AGG_VAR ? var : static_cast<T>(sqrt(static_cast<double>(var))));
        } else {
            const double s = numpy_window_sum<double>(F, F, [&](int k) { return static_cast<double>(w[k]); });
            const double avg = s / static_cast<double>(N);
            const double sq = numpy_window_sum<double>(F, F, [&](int k) {
                const double d = static_cast<double>(w[k]) - avg;
                return d * d;
            });
            const double var = sq / static_cast<double>(N);
            return static_cast<OutT>(static_cast<long long>(rint(agg == XRS_AGG_VAR ? var : sqrt(var))));
        }
    }
    default: return OutT(0);
    }
}

template <typename T, typename OutT, int F>
__device__ __forceinline__ OutT reduce_sort(T (&w)[F * F], int agg) {
    constexpr int N = F * F;
    constexpr bool FLT = std::is_floating_point<T>::value;
    if (agg == XRS_AGG_MEDIAN) {  // np.nanmedian / np.median
        int m = N;
        if constexpr (FLT) {
            m = 0;
#pragma unroll
            for (int k = 0; k < N; ++k) {
                const bool nan = is_nan(w[k]);
                m += nan ? 0 : 1;
                w[k] = nan ? static_cast<T>(INFINITY) : w[k];  // NaNs sort to the end
            }
            if (m == 0) return static_cast<OutT>(NAN);
        }
        bitonic_sort<N>(w);
        T a, b;
        if (m == N) {
            a = w[N / 2 - 1];
            b = w[N / 2];
        } else {  // some NaNs: the middle of the first m sorted values
            a = pick<N>(w, (m - 1) / 2);
            b = pick<N>(w, m / 2);
        }
        if constexpr (FLT) {  // np.nanmedian of small windows (np.ma.median): (low + high) / 2 in T, summed from +0.0
            if (m & 1) a = b;
            return static_cast<OutT>(static_cast<T>(static_cast<T>(static_cast<T>(a + b) + T(0)) * T(0.5)));
        }
        if (m & 1) return static_cast<OutT>(b);
        return static_cast<OutT>(static_cast<long long>(rint((static_cast<double>(a) + static_cast<double>(b)) / 2.0)));
    }
    // mode (coarsen.py:138-155): most frequent value, lowest value wins ties
    bitonic_sort<N>(w);
    T best = w[0];
    int best_n = 0, run = 0;
#pragma unroll
    for (int k = 0; k < N; ++k) {
        run = (k > 0 && w[k] == w[k > 0 ? k - 1 : 0]) ? run + 1 : 1;
        const bool better = run > best_n;
        best_n = better ? run : best_n;
        best = better ? w[k] : best;
    }
    return static_cast<OutT>(best);
}

// tap k+1 of scipy's order-1 filter with its edge mirror (ni_interpolation.c)
__device__ __forceinline__ int64_t next_tap(int64_t k, int64_t len) {
    return (k + 1 < len) ? k + 1 : (len > 2 ? len - 2 : 0);
}

template <typename T, typename OutT, int F, int MODE, int CLASS>
__global__ void __launch_bounds__(256) k5_window_reduce(const T *__restrict__ src, OutT *__restrict__ dst, FastGeom g) {
    const int64_t oi = static_cast<int64_t>(blockIdx.x) * 32 + threadIdx.x;
    const int64_t oj = static_cast<int64_t>(blockIdx.y) * 8 + threadIdx.y;
    const int64_t sl = blockIdx.z;
    if (oi >= g.dst_w || oj >= g.dst_h) return;
    const T *base = src + sl * g.src_slice_stride;
    const int64_t j0 = oj * F + g.j_off, i0 = oi * F + g.i_off;
    T w[F * F];
#pragma unroll
    for (int a = 0; a < F; ++a) {
        T row[F];
        load_row<T, F>(base + (j0 + a) * g.src_pitch + i0, row, g.vec != 0);
#pragma unroll
        for (int b = 0; b < F; ++b) w[a * F + b] = row[b];
    }
    if constexpr (MODE == MODE_BLEND) {
        // non-finite flags of the (F+1) x (F+1) neighbourhood: own window + next column + next row
        bool nf_col[F + 1];   // column F (right neighbours), rows 0..F
        bool nf_row[F];       // row F (lower neighbours), columns 0..F-1
        const int64_t ic = next_tap(i0 + F - 1, g.src_w), jr = next_tap(j0 + F - 1, g.src_h);
#pragma unroll
        for (int a = 0; a < F; ++a) nf_col[a] = non_finite(__ldg(base + (j0 + a) * g.src_pitch + ic));
        nf_col[F] = non_finite(__ldg(base + jr * g.src_pitch + ic));
        {
            T row[F];
            load_row<T, F>(base + jr * g.src_pitch + i0, row, g.vec != 0);
#pragma unroll
            for (int b = 0; b < F; ++b) nf_row[b] = non_finite(row[b]);
        }
        bool nf[F * F];
#pragma unroll
        for (int k = 0; k < F * F; ++k) nf[k] = non_finite(w[k]);
#pragma unroll
        for (int a = 0; a < F; ++a) {
#pragma unroll
            for (int b = 0; b < F; ++b) {
                // taps (a, b+1), (a+1, b), (a+1, b+1)
                const bool right = (b + 1 < F) ? nf[a * F + (b + 1 < F ? b + 1 : b)] : nf_col[a];
                const bool below = (a + 1 < F) ? nf[(a + 1 < F ? a + 1 : a) * F + b] : nf_row[b];
                const bool diag = (a + 1 < F) ? ((b + 1 < F) ? nf[(a + 1 < F ? a + 1 : a) * F + (b + 1 < F ? b + 1 : b)]
                                                              : nf_col[a + 1 < F ? a + 1 : a])
                                              : ((b + 1 < F) ? nf_row[b + 1 < F ? b + 1 : b] : nf_col[F]);
                T v = w[a * F + b];
                v = (v == T(0)) ? T(0) : v;  // 0.0 + (-0.0) = +0.0 in scipy's accumulation
                w[a * F + b] = (right || below || diag) ? static_cast<T>(NAN) : v;
            }
        }
    }
    OutT r;
    if constexpr (CLASS == CLASS_SORT) r = reduce_sort<T, OutT, F>(w, g.agg);
    else r = reduce_simple<T, OutT, F>(w, g.agg);
    dst[(sl * g.dst_h + oj) * g.dst_w + oi] = r;
}

// ---------------------------------------------------------------------------
// 2x2 windows of order-1 samples (the 2x bilinear down-scaling of affine.py:277-313 on aligned
// grids, BASELINE config C1): four adjacent output pixels per thread.  The 3 x 9 neighbourhood
// (two window rows + the lower tap row, eight window columns + the right tap column) comes in with
// six 16-byte loads and three scalar ones, instead of six loads per single window.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k5_blend2_x4(const T *__restrict__ src, T *__restrict__ dst, FastGeom g) {
    const int64_t og = static_cast<int64_t>(blockIdx.x) * 32 + threadIdx.x;  // group of 4 output columns
    const int64_t oj = static_cast<int64_t>(blockIdx.y) * 8 + threadIdx.y;
    const int64_t sl = blockIdx.z;
    const int64_t oi = og * 4;
    if (oi >= g.dst_w || oj >= g.dst_h) return;
    const T *base = src + sl * g.src_slice_stride;
    const int64_t j0 = oj * 2 + g.j_off, i0 = oi * 2 + g.i_off;
    const int64_t jr = next_tap(j0 + 1, g.src_h), ic = next_tap(i0 + 7, g.src_w);
    const int64_t rows[3] = {j0, j0 + 1, jr};
    T v[3][9];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const T *p = base + rows[a] * g.src_pitch + i0;
        T seg[8];
        load_row<T, 8>(p, seg, true);
#pragma unroll
        for (int b = 0; b < 8; ++b) v[a][b] = seg[b];
        v[a][8] = __ldg(base + rows[a] * g.src_pitch + ic);
    }
    bool nf[3][9];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 9; ++b) nf[a][b] = non_finite(v[a][b]);
    T out[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        T w[4];
#pragma unroll
        for (int a = 0; a < 2; ++a)
#pragma unroll
            for (int b = 0; b < 2; ++b) {
                const int c = 2 * k + b;
                T x = v[a][c];
                x = (x == T(0)) ? T(0) : x;  // 0.0 + (-0.0) = +0.0 in scipy's accumulation
                w[a * 2 + b] = (nf[a][c + 1] || nf[a + 1][c] || nf[a + 1][c + 1]) ? static_cast<T>(NAN) : x;
            }
        out[k] = reduce_simple<T, T, 2>(w, g.agg);
    }
    T *q = dst + (sl * g.dst_h + oj) * g.dst_w + oi;
    if constexpr (sizeof(T) == 4) {
        *reinterpret_cast<uint4 *>(q) = *reinterpret_cast<const uint4 *>(out);
    } else {
        reinterpret_cast<uint4 *>(q)[0] = reinterpret_cast<const uint4 *>(out)[0];
        reinterpret_cast<uint4 *>(q)[1] = reinterpret_cast<const uint4 *>(out)[1];
    }
}

template <typename T>
static bool blend2_x4_applicable(const void *src, const void *dst, const FastGeom &g, int agg_class) {
    if (agg_class != CLASS_SIMPLE || g.agg == XRS_AGG_COUNT) return false;  // count writes int64
    if (g.dst_w % 4 != 0) return false;
    const uintptr_t p = reinterpret_cast<uintptr_t>(src);
    const int64_t es = sizeof(T);
    if (p % 16 || (g.src_pitch * es) % 16 || (g.src_slice_stride * es) % 16 || (g.i_off * es) % 16) return false;
    return reinterpret_cast<uintptr_t>(dst) % 16 == 0;
}

// ---------------------------------------------------------------------------
// uint8 rasters (class maps, masks): four horizontally adjacent windows per thread, SIMD-in-a-word.
//
// A thread reads 4*F bytes per window row with one or two 16-byte loads and transposes them with
// byte permutes into N = F*F registers t[p], byte lane k of t[p] = pixel p of window k.  min / max,
// the sorting network of median and mode (vminu4 / vmaxu4), run-length counting (vcmpeq4 / vadd4 /
// vcmpgtu4) and the pick reducers then work on four windows per instruction; sums use dp4a on the
// untransposed rows.  Results: 4 bytes, or 4 int64 for mode / count / sum, per thread.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void transpose4x4(uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t &r0, uint32_t &r1,
                                             uint32_t &r2, uint32_t &r3) {
    const uint32_t t0 = __byte_perm(a, b, 0x5140), t1 = __byte_perm(a, b, 0x7362);
    const uint32_t t2 = __byte_perm(c, d, 0x5140), t3 = __byte_perm(c, d, 0x7362);
    r0 = __byte_perm(t0, t2, 0x5410); r1 = __byte_perm(t0, t2, 0x7632);
    r2 = __byte_perm(t1, t3, 0x5410); r3 = __byte_perm(t1, t3, 0x7632);
}

template <int N>
__device__ __forceinline__ void bitonic_sort_u8x4(uint32_t (&a)[N]) {
#pragma unroll
    for (int k = 2; k <= N; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const int l = i ^ j;
                if (l > i) {
                    const bool up = (i & k) == 0;
                    const uint32_t lo = __vminu4(a[i], a[l]), hi = __vmaxu4(a[i], a[l]);
                    a[i] = up ? lo : hi;
                    a[l] = up ? hi : lo;
                }
            }
        }
    }
}

// rint(sum / N) for N = 4, 16, 64 (np.mean in float64 is exact here, np.rint rounds half to even)
template <int N>
__device__ __forceinline__ uint32_t mean_half_even(uint32_t sum) {
    const uint32_t q = sum / N, rem = sum % N;
    return q + ((rem > N / 2 || (rem == N / 2 && (q & 1u))) ? 1u : 0u);
}

template <int F>
__global__ void __launch_bounds__(256) k5_u8x4_reduce(const uint8_t *__restrict__ src, void *__restrict__ dst, FastGeom g) {
    constexpr int N = F * F;
    constexpr int WORDS = F;  // 32-bit words per loaded row (4 windows x F bytes)
    const int64_t og = static_cast<int64_t>(blockIdx.x) * 32 + threadIdx.x;  // group of 4 output columns
    const int64_t oj = static_cast<int64_t>(blockIdx.y) * 8 + threadIdx.y;
    const int64_t sl = blockIdx.z;
    const int64_t oi = og * 4;
    if (oi >= g.dst_w || oj >= g.dst_h) return;
    const uint8_t *base = src + sl * g.src_slice_stride + (oj * F + g.j_off) * g.src_pitch + oi * F + g.i_off;
    uint32_t rows[F][WORDS];
#pragma unroll
    for (int a = 0; a < F; ++a) {
        const uint8_t *p = base + a * g.src_pitch;
        if constexpr (F == 2) {
            const uint2 v = __ldcs(reinterpret_cast<const uint2 *>(p));
            rows[a][0] = v.x; rows[a][1] = v.y;
        } else {
#pragma unroll
            for (int q = 0; q < WORDS / 4; ++q) {
                const uint4 v = __ldcs(reinterpret_cast<const uint4 *>(p) + q);
                rows[a][4 * q + 0] = v.x; rows[a][4 * q + 1] = v.y; rows[a][4 * q + 2] = v.z; rows[a][4 * q + 3] = v.w;
            }
        }
    }
    const int agg = g.agg;
    const int64_t o = (sl * g.dst_h + oj) * g.dst_w + oi;
    // ---- sums on the untransposed rows: window k owns F consecutive bytes of every row ----------
    if (agg == XRS_AGG_SUM || agg == XRS_AGG_MEAN) {
        uint32_t sum[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int a = 0; a < F; ++a) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if constexpr (F == 2) {
                    const uint32_t w = rows[a][k >> 1];
                    sum[k] += (k & 1) ? ((w >> 16) & 0xffu) + (w >> 24) : (w & 0xffu) + ((w >> 8) & 0xffu);
                } else {
#pragma unroll
                    for (int q = 0; q < F / 4; ++q) sum[k] = __dp4a(rows[a][k * (F / 4) + q], 0x01010101u, sum[k]);
                }
            }
        }
        if (agg == XRS_AGG_SUM) {
            int64_t *out = static_cast<int64_t *>(dst) + o;
#pragma unroll
            for (int k = 0; k < 4; ++k) out[k] = sum[k];
        } else {
            const uint32_t r = mean_half_even<N>(sum[0]) | (mean_half_even<N>(sum[1]) << 8) |
                               (mean_half_even<N>(sum[2]) << 16) | (mean_half_even<N>(sum[3]) << 24);
            *reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(dst) + o) = r;
        }
        return;
    }
    // ---- transposed registers: t[p], byte lane k = pixel p (row-major in the window) of window k ---
    uint32_t t[N];
#pragma unroll
    for (int a = 0; a < F; ++a) {
        if constexpr (F == 2) {
            t[2 * a + 0] = __byte_perm(rows[a][0], rows[a][1], 0x6420);
            t[2 * a + 1] = __byte_perm(rows[a][0], rows[a][1], 0x7531);
        } else {
#pragma unroll
            for (int h = 0; h < F / 4; ++h)
                transpose4x4(rows[a][0 * (F / 4) + h], rows[a][1 * (F / 4) + h], rows[a][2 * (F / 4) + h],
                             rows[a][3 * (F / 4) + h], t[F * a + 4 * h + 0], t[F * a + 4 * h + 1], t[F * a + 4 * h + 2],
                             t[F * a + 4 * h + 3]);
        }
    }
    uint32_t r = 0;       // 4 uint8 results
    uint32_t cnt = 0;     // 4 byte-sized counts (count reducer)
    bool wide = false;    // results are int64 (mode, count)
    switch (agg) {
    case XRS_AGG_FIRST: r = t[0]; break;
    case XRS_AGG_LAST: r = t[N - 1]; break;
    case XRS_AGG_CENTER: r = t[(F / 2) * F + F / 2]; break;
    case XRS_AGG_MIN:
        r = t[0];
#pragma unroll
        for (int k = 1; k < N; ++k) r = __vminu4(r, t[k]);
        break;
    case XRS_AGG_MAX:
        r = t[0];
#pragma unroll
        for (int k = 1; k < N; ++k) r = __vmaxu4(r, t[k]);
        break;
    case XRS_AGG_COUNT:  // np.count_nonzero
#pragma unroll
        for (int k = 0; k < N; ++k) cnt = __vadd4(cnt, __vcmpne4(t[k], 0u) & 0x01010101u);
        r = cnt;
        wide = true;
        break;
    case XRS_AGG_MEDIAN: {  // mean of the two middle values in float64, np.rint (half to even)
        bitonic_sort_u8x4<N>(t);
        const uint32_t a = t[N / 2 - 1], b = t[N / 2];
        const uint32_t q = __vhaddu4(a, b);  // floor((a + b) / 2)
        r = __vadd4(q, (a ^ b) & q & 0x01010101u);
        break;
    }
    default: {  // mode (coarsen.py:138-155): most frequent value, lowest value wins ties
        bitonic_sort_u8x4<N>(t);
        uint32_t run = 0x01010101u, best_n = 0x01010101u, best = t[0];
#pragma unroll
        for (int k = 1; k < N; ++k) {
            const uint32_t eq = __vcmpeq4(t[k], t[k - 1]);
            run = __vadd4(run & eq, 0x01010101u);
            const uint32_t better = __vcmpgtu4(run, best_n);
            best_n = (run & better) | (best_n & ~better);
            best = (t[k] & better) | (best & ~better);
        }
        r = best;
        wide = true;
        break;
    }
    }
    if (wide) {
        int64_t *out = static_cast<int64_t *>(dst) + o;
#pragma unroll
        for (int k = 0; k < 4; ++k) out[k] = (r >> (8 * k)) & 0xffu;
    } else {
        *reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(dst) + o) = r;
    }
}

// Median and mode of uint8 windows: two windows per thread as 16-bit lanes (u16x2), because the
// packed 16-bit min / max are single instructions on sm_100a (VIMNMX.U16x2) while the byte-wise
// vminu4 / vmaxu4 are emulated with ~6 logic operations each.
template <int N>
__device__ __forceinline__ void bitonic_sort_u16x2(uint32_t (&a)[N]) {
#pragma unroll
    for (int k = 2; k <= N; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const int l = i ^ j;
                if (l > i) {
                    const bool up = (i & k) == 0;
                    const uint32_t lo = __vminu2(a[i], a[l]), hi = __vmaxu2(a[i], a[l]);
                    a[i] = up ? lo : hi;
                    a[l] = up ? hi : lo;
                }
            }
        }
    }
}

template <int F>
__global__ void __launch_bounds__(256) k5_u8x2_sort(const uint8_t *__restrict__ src, void *__restrict__ dst, FastGeom g) {
    constexpr int N = F * F;
    const int64_t og = static_cast<int64_t>(blockIdx.x) * 32 + threadIdx.x;  // pair of output columns
    const int64_t oj = static_cast<int64_t>(blockIdx.y) * 8 + threadIdx.y;
    const int64_t sl = blockIdx.z;
    const int64_t oi = og * 2;
    if (oi >= g.dst_w || oj >= g.dst_h) return;
    const uint8_t *base = src + sl * g.src_slice_stride + (oj * F + g.j_off) * g.src_pitch + oi * F + g.i_off;
    // u[p]: low half-word = pixel p of window 0, high half-word = pixel p of window 1
    uint32_t u[N];
#pragma unroll
    for (int a = 0; a < F; ++a) {
        const uint8_t *p = base + a * g.src_pitch;
        if constexpr (F == 2) {
            const uint32_t w = __ldcs(reinterpret_cast<const uint32_t *>(p));
            u[2 * a + 0] = __byte_perm(w, w, 0x2200) & 0x00ff00ffu;
            u[2 * a + 1] = __byte_perm(w, w, 0x3311) & 0x00ff00ffu;
        } else if constexpr (F == 4) {
            const uint2 w = __ldcs(reinterpret_cast<const uint2 *>(p));
            u[4 * a + 0] = __byte_perm(w.x, w.y, 0x4400) & 0x00ff00ffu;
            u[4 * a + 1] = __byte_perm(w.x, w.y, 0x5511) & 0x00ff00ffu;
            u[4 * a + 2] = __byte_perm(w.x, w.y, 0x6622) & 0x00ff00ffu;
            u[4 * a + 3] = __byte_perm(w.x, w.y, 0x7733) & 0x00ff00ffu;
        } else {
            const uint4 w = __ldcs(reinterpret_cast<const uint4 *>(p));
            u[8 * a + 0] = __byte_perm(w.x, w.z, 0x4400) & 0x00ff00ffu;
            u[8 * a + 1] = __byte_perm(w.x, w.z, 0x5511) & 0x00ff00ffu;
            u[8 * a + 2] = __byte_perm(w.x, w.z, 0x6622) & 0x00ff00ffu;
            u[8 * a + 3] = __byte_perm(w.x, w.z, 0x7733) & 0x00ff00ffu;
            u[8 * a + 4] = __byte_perm(w.y, w.w, 0x4400) & 0x00ff00ffu;
            u[8 * a + 5] = __byte_perm(w.y, w.w, 0x5511) & 0x00ff00ffu;
            u[8 * a + 6] = __byte_perm(w.y, w.w, 0x6622) & 0x00ff00ffu;
            u[8 * a + 7] = __byte_perm(w.y, w.w, 0x7733) & 0x00ff00ffu;
        }
    }
    bitonic_sort_u16x2<N>(u);
    const int64_t o = (sl * g.dst_h + oj) * g.dst_w + oi;
    if (g.agg == XRS_AGG_MEDIAN) {  // float64 mean of the two middle values, np.rint (half to even)
        const uint32_t sum = u[N / 2 - 1] + u[N / 2];  // lanes <= 510: no carry between them
        const uint32_t q = (sum >> 1) & 0x7fff7fffu;
        const uint32_t r = q + (sum & q & 0x00010001u);
        *reinterpret_cast<uint16_t *>(static_cast<uint8_t *>(dst) + o) =
            static_cast<uint16_t>((r & 0xffu) | ((r >> 8) & 0xff00u));
        return;
    }
    // mode (coarsen.py:138-155): most frequent value, lowest value wins ties.  Per lane the key
    // (run length << 8) | (255 - value) is maximal for the longest run and, among equal runs, for the
    // smallest value, so one packed max per element tracks the winner.
    uint32_t run = 0x00010001u;
    uint32_t best = 0x01000100u | (0x00ff00ffu - u[0]);
#pragma unroll
    for (int k = 1; k < N; ++k) {
        const uint32_t x = u[k] ^ u[k - 1];
        const uint32_t differs = ((x + 0x7fff7fffu) >> 15) & 0x00010001u;  // 1 per lane whose value changed
        const uint32_t same_mask = (differs ^ 0x00010001u) * 0xffffu;
        run = (run & same_mask) + 0x00010001u;
        best = __vmaxu2(best, (run << 8) | (0x00ff00ffu - u[k]));
    }
    int64_t *out = static_cast<int64_t *>(dst) + o;
    out[0] = 255 - static_cast<int64_t>(best & 0xffu);
    out[1] = 255 - static_cast<int64_t>((best >> 16) & 0xffu);
}

template <int F>
static int launch_u8x2_sort(const void *src, void *dst, const FastGeom &g, cudaStream_t st) {
    const dim3 block(32, 8);
    const dim3 grid(static_cast<unsigned>(ceil_div(g.dst_w / 2, 32)), static_cast<unsigned>(ceil_div(g.dst_h, 8)),
                    static_cast<unsigned>(g.n_slices));
    XRS_TIMED("k5_u8x2_sort", st, k5_u8x2_sort<F><<<grid, block, 0, st>>>(static_cast<const uint8_t *>(src), dst, g));
    XRS_LAUNCH_CHECK("k5_u8x2_sort");
    return 0;
}

static bool u8x2_sort_applicable(const void *src, const void *dst, const FastGeom &g, int F) {
    if (g.agg != XRS_AGG_MEDIAN && g.agg != XRS_AGG_MODE) return false;
    if (g.dst_w % 2 != 0) return false;
    const int64_t align = 2 * F;  // bytes per row segment of a thread
    const uintptr_t p = reinterpret_cast<uintptr_t>(src);
    if (p % align || g.src_pitch % align || g.src_slice_stride % align || g.i_off % align) return false;
    return reinterpret_cast<uintptr_t>(dst) % (g.agg == XRS_AGG_MODE ? 8 : 2) == 0;
}

template <int F>
static int launch_u8x4(const void *src, void *dst, const FastGeom &g, cudaStream_t st) {
    const dim3 block(32, 8);
    const dim3 grid(static_cast<unsigned>(ceil_div(g.dst_w / 4, 32)), static_cast<unsigned>(ceil_div(g.dst_h, 8)),
                    static_cast<unsigned>(g.n_slices));
    XRS_TIMED("k5_u8x4_reduce", st, k5_u8x4_reduce<F><<<grid, block, 0, st>>>(static_cast<const uint8_t *>(src), dst, g));
    XRS_LAUNCH_CHECK("k5_u8x4_reduce");
    return 0;
}

// the packed path needs 4 whole windows per thread, 16-byte (8 for F = 2) aligned row segments and
// a 4-byte aligned output row
static bool u8x4_applicable(const void *src, const void *dst, const FastGeom &g, int F) {
    const int agg = g.agg;
    if (agg == XRS_AGG_PROD || agg == XRS_AGG_STD || agg == XRS_AGG_VAR) return false;
    if (g.dst_w % 4 != 0) return false;
    const int64_t align = F == 2 ? 8 : 16;
    const uintptr_t p = reinterpret_cast<uintptr_t>(src);
    if (p % align || g.src_pitch % align || g.src_slice_stride % align || g.i_off % align) return false;
    const bool wide = agg == XRS_AGG_MODE || agg == XRS_AGG_COUNT || agg == XRS_AGG_SUM;
    return reinterpret_cast<uintptr_t>(dst) % (wide ? 8 : 4) == 0;
}

static bool fast_outputs_int64(int agg, bool is_float) {
    if (agg == XRS_AGG_MODE || agg == XRS_AGG_COUNT) return true;
    return !is_float && (agg == XRS_AGG_SUM || agg == XRS_AGG_PROD);
}

template <typename T, int F, int MODE, int CLASS>
static int launch_one(const void *src, void *dst, const FastGeom &g, cudaStream_t st) {
    const dim3 block(32, 8);
    const dim3 grid(static_cast<unsigned>(ceil_div(g.dst_w, 32)), static_cast<unsigned>(ceil_div(g.dst_h, 8)),
                    static_cast<unsigned>(g.n_slices));
    const bool i64 = fast_outputs_int64(g.agg, std::is_floating_point<T>::value);
    const char *name = CLASS == CLASS_SORT ? "k5_window_reduce<sort>" : "k5_window_reduce<simple>";
    if (i64)
        XRS_TIMED(name, st, k5_window_reduce<T, int64_t, F, MODE, CLASS><<<grid, block, 0, st>>>(
                                static_cast<const T *>(src), static_cast<int64_t *>(dst), g));
    else
        XRS_TIMED(name, st, k5_window_reduce<T, T, F, MODE, CLASS><<<grid, block, 0, st>>>(
                                static_cast<const T *>(src), static_cast<T *>(dst), g));
    XRS_LAUNCH_CHECK("k5_window_reduce");
    return 0;
}

template <typename T, int F>
static int launch_f(const void *src, void *dst, const FastGeom &g, int mode, int cls, cudaStream_t st, bool *handled) {
    constexpr bool FLT = std::is_floating_point<T>::value;
    constexpr bool SORTABLE = std::is_same<T, float>::value || std::is_same<T, double>::value ||
                              std::is_same<T, uint8_t>::value || std::is_same<T, int16_t>::value ||
                              std::is_same<T, uint16_t>::value || std::is_same<T, int32_t>::value;
    if (cls == CLASS_SORT) {
        if constexpr (SORTABLE) {
            *handled = true;
            if constexpr (FLT) {
                if (mode == MODE_BLEND) return launch_one<T, F, MODE_BLEND, CLASS_SORT>(src, dst, g, st);
            }
            return launch_one<T, F, MODE_PLAIN, CLASS_SORT>(src, dst, g, st);
        }
        return 0;  // not handled
    }
    *handled = true;
    if constexpr (FLT) {
        if (mode == MODE_BLEND) {
            if constexpr (F == 2) {
                if (blend2_x4_applicable<T>(src, dst, g, cls)) {
                    const dim3 block(32, 8);
                    const dim3 grid(static_cast<unsigned>(ceil_div(g.dst_w / 4, 32)),
                                    static_cast<unsigned>(ceil_div(g.dst_h, 8)), static_cast<unsigned>(g.n_slices));
                    XRS_TIMED("k5_blend2_x4", st, k5_blend2_x4<T><<<grid, block, 0, st>>>(
                                  static_cast<const T *>(src), static_cast<T *>(dst), g));
                    XRS_LAUNCH_CHECK("k5_blend2_x4");
                    return 0;
                }
            }
            return launch_one<T, F, MODE_BLEND, CLASS_SIMPLE>(src, dst, g, st);
        }
    }
    return launch_one<T, F, MODE_PLAIN, CLASS_SIMPLE>(src, dst, g, st);
}

template <typename T>
static int launch_t(const void *src, void *dst, const AffineGeom &a, cudaStream_t st, bool *handled) {
    constexpr bool FLT = std::is_floating_point<T>::value;
    const int F = a.f_j;
    FastGeom g;
    g.n_slices = a.n_slices; g.src_h = a.src_h; g.src_w = a.src_w; g.src_pitch = a.src_pitch;
    g.src_slice_stride = a.src_slice_stride; g.dst_h = a.dst_h; g.dst_w = a.dst_w;
    g.j_off = static_cast<int64_t>(a.j_off); g.i_off = static_cast<int64_t>(a.i_off);
    g.agg = a.agg;
    // vector loads need every window row start aligned to its own size (capped at 16 bytes)
    const int64_t row_bytes = static_cast<int64_t>(F) * sizeof(T);
    const int64_t align = row_bytes < 16 ? row_bytes : 16;
    const uintptr_t p = reinterpret_cast<uintptr_t>(src);
    g.vec = (p % align == 0 && (a.src_pitch * sizeof(T)) % align == 0 && (a.src_slice_stride * sizeof(T)) % align == 0 &&
             (g.i_off * sizeof(T)) % align == 0) ? 1 : 0;
    if constexpr (std::is_same<T, uint8_t>::value) {
        if (u8x2_sort_applicable(src, dst, g, F)) {
            *handled = true;
            switch (F) {
            case 2: return launch_u8x2_sort<2>(src, dst, g, st);
            case 4: return launch_u8x2_sort<4>(src, dst, g, st);
            default: return launch_u8x2_sort<8>(src, dst, g, st);
            }
        }
        if (u8x4_applicable(src, dst, g, F)) {
            *handled = true;
            switch (F) {
            case 2: return launch_u8x4<2>(src, dst, g, st);
            case 4: return launch_u8x4<4>(src, dst, g, st);
            default: return launch_u8x4<8>(src, dst, g, st);
            }
        }
    }
    const int mode = (a.order == 1 && FLT) ? MODE_BLEND : MODE_PLAIN;
    const int cls = (a.agg == XRS_AGG_MEDIAN || a.agg == XRS_AGG_MODE) ? CLASS_SORT : CLASS_SIMPLE;
    switch (F) {
    case 2: return launch_f<T, 2>(src, dst, g, mode, cls, st, handled);
    case 4: return launch_f<T, 4>(src, dst, g, mode, cls, st, handled);
    case 8: return launch_f<T, 8>(src, dst, g, mode, cls, st, handled);
    default: return 0;
    }
}

int launch_affine_fast(const void *src, void *dst, int dtype, const AffineGeom &a, cudaStream_t st, bool *handled) {
    *handled = false;
    if (a.f_j != a.f_i || (a.f_j != 2 && a.f_j != 4 && a.f_j != 8)) return 0;
    if (a.j_scale != 1.0 || a.i_scale != 1.0) return 0;
    if (!(a.j_off >= 0.0 && a.i_off >= 0.0 && a.j_off < 1e15 && a.i_off < 1e15)) return 0;
    if (a.j_off != floor(a.j_off) || a.i_off != floor(a.i_off)) return 0;
    // every sample must lie inside the source (no cval), cf. ni_interpolation.c bounds test
    if (static_cast<int64_t>(a.j_off) + a.dst_h * a.f_j > a.src_h || static_cast<int64_t>(a.i_off) + a.dst_w * a.f_i > a.src_w)
        return 0;
    const bool is_float = dtype == XRS_F32 || dtype == XRS_F64;
    if (a.order == 1 && is_float && a.slice_blend) return 0;  // next-slice taps (one slice: its own): generic kernel
    // samples scipy changes on the way through float64 -- int64 beyond 2^53 at order 0 and 1, -0.0 at order 0 --
    // unless they come from xrs_coarsen: generic kernel
    if (a.order == 0 && !a.exact_samples && (is_float || dtype == XRS_I64)) return 0;
    if (a.order == 1 && dtype == XRS_I64) return 0;
    if (a.n_slices > 65535 || ceil_div(a.dst_h, 8) > 65535) return 0;
    XRS_DISPATCH_DTYPE(dtype, T, return launch_t<T>(src, dst, a, st, handled));
    return 0;
}

}  // namespace xrs
