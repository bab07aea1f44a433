// gather_common.cuh -- per-pixel arithmetic and tile constants shared by the K2 gather kernels
// (gather.cu: one interpolation method per launch; gather_dual.cu: nearest + bilinear / triangular
// of the same bands in one launch).  rectify.py:689-734 of the reference.
#pragma once

#include "rectify_common.cuh"
#include "tma.cuh"

namespace xrs {

constexpr int K2_MAX_BANDS = 24;

// ---------------------------------------------------------------------------
// per-pixel arithmetic shared by both kernels
// ---------------------------------------------------------------------------
template <int METHOD>
__device__ __forceinline__ double interp_value(double v00, double v01, double v10, double v11, double u, double v) {
    if (METHOD == XRS_BILINEAR) {  // rectify.py:718-727
        const double a = dadd(v00, dmul(u, dsub(v01, v00)));
        const double b = dadd(v10, dmul(u, dsub(v11, v10)));
        return dadd(a, dmul(v, dsub(b, a)));
    }
    // triangular, rectify.py:699-717
    if (dadd(u, v) < 1.0) return dadd(dadd(v00, dmul(u, dsub(v01, v00))), dmul(v, dsub(v10, v00)));
    return dadd(dadd(v11, dmul(dsub(1.0, u), dsub(v10, v11))), dmul(dsub(1.0, v), dsub(v01, v11)));
}

// Source taps of one target pixel: (i0, j0) and the clamped neighbours (i1, j1), fractions u, v.
// For nearest the single tap is already moved to the nearer pixel (ties keep the lower index).
struct Taps {
    int i0, j0, i1, j1;
    double u, v;
    bool valid;
};

template <int METHOD>
__device__ __forceinline__ Taps make_taps(double fi, double fj, int64_t src_w, int64_t src_h) {
    Taps t;
    t.valid = (fi == fi) && (fj == fj);
    t.i0 = t.j0 = t.i1 = t.j1 = 0;
    t.u = t.v = 0.0;
    if (!t.valid) return t;
    // rectify.py:689-692: int() truncation of non-negative values
    const int64_t i0 = static_cast<int64_t>(fi), j0 = static_cast<int64_t>(fj);
    t.u = dsub(fi, static_cast<double>(i0));
    t.v = dsub(fj, static_cast<double>(j0));
    const int64_t i1 = min(max(i0 + 1, int64_t(0)), src_w - 1), j1 = min(max(j0 + 1, int64_t(0)), src_h - 1);
    if (METHOD == XRS_NEAREST) {  // rectify.py:693-698
        t.i0 = t.i1 = static_cast<int>(t.u > 0.5 ? i1 : i0);
        t.j0 = t.j1 = static_cast<int>(t.v > 0.5 ? j1 : j0);
    } else {
        t.i0 = static_cast<int>(i0); t.j0 = static_cast<int>(j0);
        t.i1 = static_cast<int>(i1); t.j1 = static_cast<int>(j1);
    }
    return t;
}

template <typename T>
__device__ __forceinline__ double ld_f64(const T *p) { return static_cast<double>(__ldg(p)); }

// staged kernels (TMA tensor tiles -> shared memory): target tile, threads, source box, ring depth
constexpr int K2S_TW = 32, K2S_TH = 32;   // target tile
constexpr int K2S_THREADS = 256;
constexpr int K2S_PX = 4;                  // pixels per thread: same column, rows 8 apart, so that a warp
                                           // reads 32 neighbouring source pixels (bank-conflict free)
constexpr int K2S_ROW_STEP = K2S_THREADS / K2S_TW;
constexpr int K2S_BOX_W = 64, K2S_BOX_H = 48;
constexpr int K2S_STAGES = 4;

// A nearest sample as the reference stores it: it casts the source window to float64 (rectify.py:628-630) and
// assigns the float64 value back (rectify.py:734).  The round trip is the identity for every type but int64,
// whose values beyond 2^53 it rounds (and INT64_MAX, rounded up to 2^63, turns into INT64_MIN).
template <typename T>
__device__ __forceinline__ T nearest_value(T v) {
    if constexpr (std::is_same<T, int64_t>::value) return cast_like_numpy<T>(static_cast<double>(v));
    else return v;
}

}  // namespace xrs
