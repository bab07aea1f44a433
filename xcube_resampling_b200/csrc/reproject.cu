// reproject.cu -- K3: CRS transform of target pixel centres fused with the gather of all bands.
//
//   xrs_transform_points   pyproj.Transformer.transform call sites: reproject.py:472-496
//                          (_transform_gridpoints), rectify.py:182-231 (_transform_coords),
//                          and, through the host, transform_bounds (reproject.py:347,398)
//   xrs_reproject          reproject.py:472-496 + 268-335 (_transform_gridpoints + _reproject_block)
//                          reading the source in place of the padded / re-tiled copy of
//                          reproject.py:499-530 (_reorganize_data_array_slice)
//
// The projection math (proj.cuh) is compiled with FMA contraction; everything the reference
// computes with numpy after the transform -- fractional index, rounding, tap differences in the
// source dtype, the lerps in float64 -- uses explicit round-to-nearest intrinsics in the
// reference's operation order.
#include <cmath>
#include <cstdlib>
#include <cstring>

#include "proj.cuh"
#include "tma.cuh"

namespace xrs {

// ---------------------------------------------------------------------------
// host: projection constants
// ---------------------------------------------------------------------------
namespace {

typedef long double ld;
const ld LD_PI = 3.14159265358979323846264338327950288L;

ld taup_ld(ld tau, ld e) {
    const ld s1 = sqrtl(1 + tau * tau);
    const ld sigma = sinhl(e * atanhl(e * tau / s1));
    return tau * sqrtl(1 + sigma * sigma) - sigma * s1;
}

// geodetic tangent from conformal tangent (Karney 2011 eqs. 19-21)
ld tau_from_taup_ld(ld taup, ld e) {
    const ld e2m = 1 - e * e;
    ld tau = taup / e2m;
    for (int it = 0; it < 16; ++it) {
        const ld tp = taup_ld(tau, e);
        tau += (taup - tp) / sqrtl(1 + tp * tp) * (1 + e2m * tau * tau) / (e2m * sqrtl(1 + tau * tau));
    }
    return tau;
}

ld q_ld(ld s, ld e) {
    const ld es = e * s;
    return (1 - e * e) * (s / (1 - es * es) - (0.5L / e) * logl((1 - es) / (1 + es)));
}

// geodetic latitude from authalic latitude: Newton on q(phi) (Snyder eq. 3-16)
ld phi_from_beta_ld(ld beta, ld e) {
    const ld q = q_ld(1, e) * sinl(beta);
    ld phi = asinl(q / 2);
    for (int it = 0; it < 40; ++it) {
        const ld s = sinl(phi), c = cosl(phi), es = e * s;
        phi += (1 - es * es) * (1 - es * es) / (2 * c) *
               (q / (1 - e * e) - s / (1 - es * es) + (0.5L / e) * logl((1 - es) / (1 + es)));
    }
    return phi;
}

// Sine-series coefficients c_k, k = 1..6, of the odd pi-periodic function g(t) = f(t) - t:
// midpoint rule on (0, pi/2), exact up to rounding because the series decays like n^k.
template <typename F>
void sine_series(F f, double *out) {
    const int M = 64;
    ld acc[PROJ_TERMS] = {0, 0, 0, 0, 0, 0};
    for (int m = 0; m < M; ++m) {
        const ld t = (LD_PI / 2) * (m + 0.5L) / M;
        const ld g = f(t) - t;
        for (int k = 1; k <= PROJ_TERMS; ++k) acc[k - 1] += g * sinl(2 * k * t);
    }
    for (int k = 0; k < PROJ_TERMS; ++k) out[k] = static_cast<double>(acc[k] * 2 / M);
}

}  // namespace

int make_proj_consts(const xrs_proj *p, ProjC *c) {
    if (!p) return fail("projection descriptor is null");
    ProjC z = {};
    *c = z;
    c->kind = p->kind;
    if (p->kind < XRS_PROJ_GEOGRAPHIC || p->kind > XRS_PROJ_LAEA)
        return fail("unknown projection kind " + std::to_string(p->kind));
    if (!(p->a > 0.0)) return fail("projection: semi-major axis must be positive");
    const double f = p->inv_f != 0.0 ? 1.0 / p->inv_f : 0.0;
    c->a = p->a;
    c->es = f * (2.0 - f);
    c->e = std::sqrt(c->es);
    c->one_es = 1.0 - c->es;
    c->lon0 = p->lon0 * PROJ_DEG2RAD;
    c->lat0 = p->lat0 * PROJ_DEG2RAD;
    c->fe = p->fe;
    c->fn = p->fn;
    if (p->kind == XRS_PROJ_GEOGRAPHIC || p->kind == XRS_PROJ_WEBMERC) return 0;
    if (f == 0.0) return fail("spherical tmerc / laea are not supported (inverse flattening must be non-zero)");
    const ld e = sqrtl(static_cast<ld>(f) * (2 - static_cast<ld>(f)));
    if (p->kind == XRS_PROJ_TMERC) {
        const double n = f / (2.0 - f), n2 = n * n, n3 = n2 * n, n4 = n3 * n, n5 = n4 * n, n6 = n5 * n;
        // Karney (2011) eqs. 35, 36
        const double al[PROJ_TERMS] = {
            n / 2 - 2 * n2 / 3 + 5 * n3 / 16 + 41 * n4 / 180 - 127 * n5 / 288 + 7891 * n6 / 37800,
            13 * n2 / 48 - 3 * n3 / 5 + 557 * n4 / 1440 + 281 * n5 / 630 - 1983433 * n6 / 1935360,
            61 * n3 / 240 - 103 * n4 / 140 + 15061 * n5 / 26880 + 167603 * n6 / 181440,
            49561 * n4 / 161280 - 179 * n5 / 168 + 6601661 * n6 / 7257600,
            34729 * n5 / 80640 - 3418889 * n6 / 1995840,
            212378941 * n6 / 319334400};
        const double be[PROJ_TERMS] = {
            n / 2 - 2 * n2 / 3 + 37 * n3 / 96 - n4 / 360 - 81 * n5 / 512 + 96199 * n6 / 604800,
            n2 / 48 + n3 / 15 - 437 * n4 / 1440 + 46 * n5 / 105 - 1118711 * n6 / 3870720,
            17 * n3 / 480 - 37 * n4 / 840 - 209 * n5 / 4480 + 5569 * n6 / 90720,
            4397 * n4 / 161280 - 11 * n5 / 504 - 830251 * n6 / 7257600,
            4583 * n5 / 161280 - 108847 * n6 / 3991680,
            20648693 * n6 / 638668800};
        for (int k = 0; k < PROJ_TERMS; ++k) {
            c->alpha[k] = al[k];
            c->beta[k] = be[k];
        }
        c->Qn = p->k0 * p->a * (1 + n2 / 4 + n4 / 64 + n6 / 256) / (1 + n);
        sine_series([e](ld t) { return atanl(taup_ld(tanl(t), e)); }, c->cbg);
        sine_series([e](ld t) { return atanl(tau_from_taup_ld(tanl(t), e)); }, c->cgb);
        c->xi0 = 0.0;
        if (p->lat0 != 0.0) {
            const ld xip = atanl(taup_ld(tanl(static_cast<ld>(p->lat0) * LD_PI / 180), e));
            ld xi = xip;
            for (int k = 1; k <= PROJ_TERMS; ++k) xi += al[k - 1] * sinl(2 * k * xip);
            c->xi0 = static_cast<double>(xi);
        }
        return 0;
    }
    // LAEA, oblique or equatorial aspect
    if (std::fabs(std::fabs(p->lat0) - 90.0) < 1e-9) return fail("polar LAEA is not supported");
    const ld phi1 = static_cast<ld>(p->lat0) * LD_PI / 180;
    const ld qp = q_ld(1, e), q1 = q_ld(sinl(phi1), e);
    const ld sinb1 = q1 / qp, cosb1 = sqrtl(1 - sinb1 * sinb1);
    const ld rq = p->a * sqrtl(qp / 2);
    const ld m1 = cosl(phi1) / sqrtl(1 - e * e * sinl(phi1) * sinl(phi1));
    c->qp = static_cast<double>(qp);
    c->rq = static_cast<double>(rq);
    c->dd = static_cast<double>(p->a * m1 / (rq * cosb1));
    c->sinb1 = static_cast<double>(sinb1);
    c->cosb1 = static_cast<double>(cosb1);
    sine_series([e](ld t) { return phi_from_beta_ld(t, e); }, c->apa);
    return 0;
}

// ---------------------------------------------------------------------------
// K3a: point transform
// ---------------------------------------------------------------------------
__device__ __noinline__ void transform_point(const ProjC &from, const ProjC &to, double x, double y, double &ox,
                                             double &oy) {
    proj_transform(from, to, x, y, ox, oy);
}

__global__ void __launch_bounds__(256)
k3_transform_points(const __grid_constant__ ProjC from, const __grid_constant__ ProjC to, const double *__restrict__ x,
                    const double *__restrict__ y, double *__restrict__ ox, double *__restrict__ oy, int64_t n) {
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        double tx, ty;
        transform_point(from, to, x[i], y[i], tx, ty);
        ox[i] = tx;
        oy[i] = ty;
    }
}

// ---------------------------------------------------------------------------
// K3: fused transform + gather
// ---------------------------------------------------------------------------
constexpr int K3_MAX_BANDS = 24;

template <typename T, typename OUT>
struct K3Planes {
    const T *src[K3_MAX_BANDS];
    OUT *dst[K3_MAX_BANDS];
};

struct K3Geom {
    ProjC from, to;  // target CRS -> source CRS
    const double *dst_x, *dst_y;
    int64_t dst_h, dst_w, row_begin, row_end;
    int64_t row_tile0;  // row_begin rounded down to the CTA tile height: tiles (and with them the lattice
                        // of the transform) sit at the same rows whatever row band a call computes
    int tile_h, tile_w, ntx;
    const double *tile_x0, *tile_y0;  // float32 window origins (widened), reproject.py:427-450
    const int32_t *tile_i0, *tile_j0; // window start in source index space (may be negative)
    int tile_win_w, tile_win_h;
    double x_res, y_res;              // source resolution
    double inv_x_res, inv_y_res;      // 1 / x_res, 1 / y_res (lattice path only, see k3_reproject)
    const double *lat_nodes;          // lattice of the transform, 34 doubles per CTA tile (k3_lattice_nodes), or null
    int64_t src_h, src_w, src_pitch, win_i0, win_j0, win_w, win_h;
};

// numpy index semantics inside the reference window: negative indices count from the end
// (reproject.py:284,295-298,321-324).  Anything still outside raises IndexError there; here it
// reads as "no data".
__device__ __forceinline__ bool window_index(int64_t &k, int n) {
    if (k < 0) k += n;
    return k >= 0 && k < n;
}

// a - b in the array's own dtype (numpy: value_01 - value_00 before the float64 promotion)
template <typename T>
__device__ __forceinline__ double diff_as_f64(T a, T b) {
    if constexpr (std::is_same<T, float>::value) {
        return static_cast<double>(__fsub_rn(a, b));
    } else if constexpr (std::is_same<T, double>::value) {
        return dsub(a, b);
    } else if constexpr (sizeof(T) == 8) {
        return static_cast<double>(static_cast<T>(static_cast<uint64_t>(a) - static_cast<uint64_t>(b)));
    } else {
        return static_cast<double>(static_cast<T>(static_cast<uint32_t>(a) - static_cast<uint32_t>(b)));
    }
}

// (reproject.py:299-300 assigns the float64 results into an array of the source dtype: cast_like_numpy,
// xrs_casts.h)
template <typename T, typename OUT>
__device__ __forceinline__ OUT k3_store_cast(double v) {
    if constexpr (std::is_same<OUT, double>::value) return v;
    else return cast_like_numpy<OUT>(v);
}

// reproject.py:301-328: the blend of the four taps.  Differences are taken in the array's own dtype
// (numpy subtracts before the float64 promotion), the lerps in float64 without contraction.
template <typename T, typename OUT, int METHOD>
__device__ __forceinline__ OUT k3_blend(T v00, T v01, T v10, T v11, double u, double v) {
    double val;
    if (METHOD == XRS_BILINEAR) {  // reproject.py:325-327
        const double a = dadd(static_cast<double>(v00), dmul(u, diff_as_f64(v01, v00)));
        const double bb = dadd(static_cast<double>(v10), dmul(u, diff_as_f64(v11, v10)));
        val = dadd(a, dmul(v, dsub(bb, a)));
    } else if (dadd(u, v) < 1.0) {  // reproject.py:301-307
        val = dadd(dadd(static_cast<double>(v00), dmul(u, diff_as_f64(v01, v00))), dmul(v, diff_as_f64(v10, v00)));
    } else {                        // reproject.py:309-313
        val = dadd(dadd(static_cast<double>(v11), dmul(dsub(1.0, u), diff_as_f64(v10, v11))),
                   dmul(dsub(1.0, v), diff_as_f64(v01, v11)));
    }
    return k3_store_cast<T, OUT>(val);
}

// A source tap.  XRS_K3_LD256: 4-byte taps ask L2 to fetch the 256-byte pair of lines on a miss (the
// CTA to the right reads the next 128 bytes of the same source rows).
#ifndef XRS_K3_TAPS_PIPE
#define XRS_K3_TAPS_PIPE 0  // bands per register buffer of the pipelined tap loop (0 = chunked loop)
#endif
#ifndef XRS_K3_LD256
#define XRS_K3_LD256 1
#endif
template <typename T>
__device__ __forceinline__ T ld_tap(const T *p) {
    if constexpr (XRS_K3_LD256 && sizeof(T) == 4) {
        uint32_t v;
        asm("ld.global.nc.L2::256B.b32 %0, [%1];" : "=r"(v) : "l"(p));
        T out;
        memcpy(&out, &v, 4);
        return out;
    } else {
        return __ldg(p);
    }
}

// ---- band loops of a pixel whose taps all lie inside the resident source ----------------------
constexpr int K3_CHUNK = 4;  // bands whose taps are loaded before any of them is consumed
constexpr int K3_SEP_CHUNK = 4;  // ... in the separable kernel
#ifndef XRS_K3_COPY_CHUNK
#define XRS_K3_COPY_CHUNK 8
#endif
constexpr int K3_COPY_CHUNK = XRS_K3_COPY_CHUNK;  // nearest: one tap per band, so twice as many bands in flight

template <typename T, typename OUT, int CHUNK = K3_COPY_CHUNK>
__device__ __forceinline__ void k3_copy_tap(const K3Planes<T, OUT> &planes, int n_bands, int64_t o, int off) {
    for (int b = 0; b < n_bands; b += CHUNK) {  // (the last group is predicated, not a band-by-band tail)
        T v[CHUNK];
#pragma unroll
        for (int q = 0; q < CHUNK; ++q)
            if (b + q < n_bands) v[q] = ld_tap(planes.src[b + q] + off);
#pragma unroll
        for (int q = 0; q < CHUNK; ++q)
            if (b + q < n_bands) st_stream(planes.dst[b + q] + o, static_cast<OUT>(v[q]));
    }
}

// o00: element offset of tap (0, 0); d01 in {0, 1}: the right-hand tap is the next element or the same;
// d10 in {0, pitch}: likewise for the lower taps.  Bands [b_begin, n_bands).
template <typename T, typename OUT, int METHOD, int CHUNK = K3_CHUNK>
__device__ __forceinline__ void k3_blend_taps(const K3Planes<T, OUT> &planes, int n_bands, int64_t o, int o00, int d01,
                                              int d10, int pitch, double u, double v, int b_begin = 0) {
    const int d11 = d10 + d01;
#if XRS_K3_TAPS_PIPE
    if (d01 == 1 && d10 != 0 && b_begin == 0) {
        // Software-pipelined over groups of HALF bands with two register buffers: the taps of the next group
        // are requested before the current group is blended, so a warp always has loads in flight while
        // it computes instead of draining its loads, computing, and starting over.
        constexpr int HALF = XRS_K3_TAPS_PIPE;
        T wa[HALF][4], wb[HALF][4];
        auto request = [&](T (&w)[HALF][4], int b) {
#pragma unroll
            for (int q = 0; q < HALF; ++q)
                if (b + q < n_bands) {
                    const T *p0 = planes.src[b + q] + o00;
                    const T *p1 = p0 + pitch;
                    w[q][0] = ld_tap(p0); w[q][1] = ld_tap(p0 + 1); w[q][2] = ld_tap(p1); w[q][3] = ld_tap(p1 + 1);
                }
        };
        auto blend = [&](T (&w)[HALF][4], int b) {
#pragma unroll
            for (int q = 0; q < HALF; ++q)
                if (b + q < n_bands)
                    st_stream(planes.dst[b + q] + o, k3_blend<T, OUT, METHOD>(w[q][0], w[q][1], w[q][2], w[q][3], u, v));
        };
        request(wa, 0);
#pragma unroll 1
        for (int b = 0; b < n_bands; b += 2 * HALF) {
            request(wb, b + HALF);
            blend(wa, b);
            request(wa, b + 2 * HALF);
            blend(wb, b + HALF);
        }
        return;
    }
#endif
    if (d01 == 1 && d10 != 0) {
        // generic position: the right-hand taps are the next element, so they are addressed with an
        // immediate offset from the two row pointers (2 address computations per band instead of 4)
        int b = b_begin;
        for (; b + CHUNK <= n_bands; b += CHUNK) {
            T w[CHUNK][4];
#pragma unroll
            for (int q = 0; q < CHUNK; ++q) {
                const T *p0 = planes.src[b + q] + o00;
                const T *p1 = p0 + pitch;
                w[q][0] = ld_tap(p0); w[q][1] = ld_tap(p0 + 1); w[q][2] = ld_tap(p1); w[q][3] = ld_tap(p1 + 1);
            }
#pragma unroll
            for (int q = 0; q < CHUNK; ++q)
                st_stream(planes.dst[b + q] + o, k3_blend<T, OUT, METHOD>(w[q][0], w[q][1], w[q][2], w[q][3], u, v));
        }
        for (; b < n_bands; ++b) {
            const T *p0 = planes.src[b] + o00;
            const T *p1 = p0 + pitch;
            st_stream(planes.dst[b] + o, k3_blend<T, OUT, METHOD>(ld_tap(p0), ld_tap(p0 + 1), ld_tap(p1), ld_tap(p1 + 1), u, v));
        }
        return;
    }
    for (int b = b_begin; b < n_bands; ++b) {  // a coordinate exactly on a pixel centre: ceil == floor
        const T *sp = planes.src[b] + o00;
        st_stream(planes.dst[b] + o, k3_blend<T, OUT, METHOD>(ld_tap(sp), ld_tap(sp + d01), ld_tap(sp + d10), ld_tap(sp + d11), u, v));
    }
}

// ---- per-pixel gather (reproject.py:268-335) given the source-CRS coordinates (sx, sy) --------
// The window origin of the pixel's reference tile (float32, widened) and the window's first source index.
struct K3Tile {
    double x0, y0;
    int i0, j0;
};
__device__ __forceinline__ K3Tile k3_load_tile(const K3Geom &g, int t) {
    K3Tile tl;
    tl.x0 = __ldg(g.tile_x0 + t); tl.y0 = __ldg(g.tile_y0 + t);
    tl.i0 = __ldg(g.tile_i0 + t); tl.j0 = __ldg(g.tile_j0 + t);
    return tl;
}

// RCP: the fractional index is formed with the reciprocal resolution instead of a division.  Only the
// lattice path uses it: its coordinates are interpolated (error bound ~1e-8 px, see k3_reproject), so
// the last-bit agreement with numpy's division that the exact paths keep has no meaning there.
template <typename T, typename OUT, int METHOD, bool RCP = false>
__device__ __forceinline__ void k3_gather_pixel(const K3Geom &g, const K3Planes<T, OUT> &planes, int n_bands, T fill,
                                                int64_t o, const K3Tile &tl, double sx, double sy) {
    // reproject.py:278-279
    const double fx = RCP ? dmul(dsub(sx, tl.x0), g.inv_x_res) : ddiv(dsub(sx, tl.x0), g.x_res);
    const double fy = RCP ? dmul(dsub(tl.y0, sy), g.inv_y_res) : ddiv(dsub(sy, tl.y0), -g.y_res);
    const int i_base = tl.i0, j_base = tl.j0;
    const OUT fill_out = static_cast<OUT>(fill);
    if (!(fabs(fx) < 1e9 && fabs(fy) < 1e9)) {  // NaN / inf / absurdly far: no data
        for (int b = 0; b < n_bands; ++b) st_stream(planes.dst[b] + o, fill_out);
        return;
    }
    const int ww = g.tile_win_w, wh = g.tile_win_h;
    // resident window expressed in source indices
    const int res_i0 = static_cast<int>(g.win_i0), res_j0 = static_cast<int>(g.win_j0);
    const int res_i1 = res_i0 + static_cast<int>(g.win_w), res_j1 = res_j0 + static_cast<int>(g.win_h);
    const int pitch = static_cast<int>(g.src_pitch);

    // element offset of window index (wy, wx) inside a resident plane, or -1 for the constant
    // padding (reproject.py:507 da.pad(..., constant_values=fill_value)); `ok` turns false where
    // numpy would raise IndexError.  Negative window indices count from the end, as in numpy.
    auto tap = [&](int wy, int wx, bool &ok) -> int {
        if (wx < 0) wx += ww;
        if (wy < 0) wy += wh;
        ok = ok && wx >= 0 && wx < ww && wy >= 0 && wy < wh;
        const int si = i_base + wx, sj = j_base + wy;
        if (si < res_i0 || sj < res_j0 || si >= res_i1 || sj >= res_j1) return -1;  // padding (or not resident)
        return (sj - res_j0) * pitch + (si - res_i0);
    };

    if (METHOD == XRS_NEAREST) {
        bool ok = true;
        int off = tap(__double2int_rn(fy), __double2int_rn(fx), ok);
        if (!ok) off = -1;
        if (off >= 0) {
            k3_copy_tap<T, OUT>(planes, n_bands, o, off);
        } else {
            for (int b = 0; b < n_bands; ++b) st_stream(planes.dst[b] + o, fill_out);
        }
        return;
    }
    const double fx0 = floor(fx), fy0 = floor(fy);
    const double u = dsub(fx, fx0), v = dsub(fy, fy0);
    const int ix0 = __double2int_rd(fx), ix1 = __double2int_ru(fx);
    const int iy0 = __double2int_rd(fy), iy1 = __double2int_ru(fy);
    auto blend = [&](T v00, T v01, T v10, T v11) -> OUT { return k3_blend<T, OUT, METHOD>(v00, v01, v10, v11, u, v); };
    // common case: the 2 x 2 taps lie inside the tile window and inside the resident source
    const int si0 = i_base + ix0, sj0 = j_base + iy0, si1 = i_base + ix1, sj1 = j_base + iy1;
    if (ix0 >= 0 && iy0 >= 0 && ix1 < ww && iy1 < wh && si0 >= res_i0 && sj0 >= res_j0 && si1 < res_i1 && sj1 < res_j1) {
        k3_blend_taps<T, OUT, METHOD>(planes, n_bands, o, (sj0 - res_j0) * pitch + (si0 - res_i0), ix1 - ix0,
                                      (iy1 - iy0) * pitch, pitch, u, v);
        return;
    }
    bool ok = true;
    const int o00 = tap(iy0, ix0, ok), o01 = tap(iy0, ix1, ok), o10 = tap(iy1, ix0, ok), o11 = tap(iy1, ix1, ok);
    if (!ok) {
        for (int b = 0; b < n_bands; ++b) st_stream(planes.dst[b] + o, fill_out);
        return;
    }
    for (int b = 0; b < n_bands; ++b) {
        const T *sp = planes.src[b];
        const T v00 = o00 >= 0 ? __ldg(sp + o00) : fill, v01 = o01 >= 0 ? __ldg(sp + o01) : fill;
        const T v10 = o10 >= 0 ? __ldg(sp + o10) : fill, v11 = o11 >= 0 ? __ldg(sp + o11) : fill;
        st_stream(planes.dst[b] + o, blend(v00, v01, v10, v11));
    }
}
template <typename T, typename OUT, int METHOD>
__device__ __forceinline__ void k3_gather_pixel(const K3Geom &g, const K3Planes<T, OUT> &planes, int n_bands, T fill,
                                                int64_t o, int t, double sx, double sy) {
    k3_gather_pixel<T, OUT, METHOD, false>(g, planes, n_bands, fill, o, k3_load_tile(g, t), sx, sy);
}

// ---- how the target -> source transform of a tile is evaluated --------------------------------
enum K3Plan {
    K3_PLAN_GENERIC = 0,    // per pixel, full formulas (target CRS = LAEA)
    K3_PLAN_IDENTITY = 1,   // both CRSs geographic: coordinates pass through untouched
    K3_PLAN_SEPARABLE = 2,  // target CRS geographic / web Mercator: lon by column, lat by row
    K3_PLAN_TMERC_INV = 3,  // target CRS transverse Mercator: xi by row, eta by column
    K3_PLAN_MASK = 0xff,
    K3_PLAN_EXACT_ONLY = 0x100  // flag: no lattice interpolation of the transform (XRS_K3_EXACT=1, tests)
};

__device__ __noinline__ void forward_point(const ProjC &to, double lam, double phi, double &ox, double &oy) {
    if (!proj_forward(to, lam, phi, ox, oy)) ox = oy = NAN;
}

// Source-CRS coordinates of target pixel (r, c) from its row / column terms.
__device__ __forceinline__ void k3_pixel_source_xy(const K3Geom &g, int plan, const Terms4 &rt, const Terms4 &ct,
                                                   int64_t c, int64_t r, double &sx, double &sy) {
    if (plan == K3_PLAN_TMERC_INV) {
        double lam, phi;
        if (tmerc_inv_tail(g.from, rt, ct, lam, phi)) {
            if (g.to.kind == XRS_PROJ_GEOGRAPHIC) {
                sx = lam * PROJ_RAD2DEG;
                sy = phi * PROJ_RAD2DEG;
            } else {
                forward_point(g.to, lam, phi, sx, sy);
            }
        } else {
            transform_point(g.from, g.to, __ldg(g.dst_x + c), __ldg(g.dst_y + r), sx, sy);
        }
    } else if (plan == K3_PLAN_SEPARABLE) {
        fwd_tail(g.to, rt, ct, sx, sy);
    } else if (plan == K3_PLAN_IDENTITY) {
        sx = ct.a;
        sy = rt.a;
    } else {
        transform_point(g.from, g.to, ct.a, rt.a, sx, sy);
    }
}

// Row-only / column-only terms of the target -> source transform (one sincos / exp per tile row or
// column instead of one per pixel).
__device__ __forceinline__ Terms4 k3_row_terms(const K3Geom &g, int plan, double y) {
    Terms4 t;
    t.a = y; t.b = t.c = t.d = 0.0;
    if (plan == K3_PLAN_TMERC_INV) {
        t = tmerc_inv_row_terms(g.from, y);
    } else if (plan == K3_PLAN_SEPARABLE) {
        double phi;
        bool ok = true;
        if (g.from.kind == XRS_PROJ_GEOGRAPHIC) {
            phi = y * PROJ_DEG2RAD;
            ok = fabs(y) <= 90.0;
        } else {
            phi = atan(sinh((y - g.from.fn) / g.from.a));
        }
        t = fwd_row_terms(g.to, phi, ok);
    }
    return t;
}
__device__ __forceinline__ Terms4 k3_col_terms(const K3Geom &g, int plan, double x) {
    Terms4 t;
    t.a = x; t.b = t.c = t.d = 0.0;
    if (plan == K3_PLAN_TMERC_INV) {
        t = tmerc_inv_col_terms(g.from, x);
    } else if (plan == K3_PLAN_SEPARABLE) {
        const double lam = g.from.kind == XRS_PROJ_GEOGRAPHIC ? x * PROJ_DEG2RAD
                                                               : wrap_pi(g.from.lon0 + (x - g.from.fe) / g.from.a);
        t = fwd_col_terms(g.to, lam);
    }
    return t;
}

// One axis of a pixel's taps (separable transforms): source index of tap 0, whether tap 1 is the next
// element (flags bit 0), whether both taps lie inside the tile window and the resident source
// (bit 1), and the interpolation fraction.  Same arithmetic as k3_gather_pixel, per axis.
struct AxisTap {
    double frac;
    int idx, flags;
};
template <int METHOD>
__device__ __forceinline__ void axis_tap(double f, int base, int win_n, int res_lo, int res_hi, AxisTap &a) {
    if (!(fabs(f) < 1e9)) return;  // NaN / inf / absurdly far: the general path writes the fill value
    int w0, w1;
    if (METHOD == XRS_NEAREST) {
        w0 = w1 = __double2int_rn(f);
    } else {
        w0 = __double2int_rd(f);
        w1 = __double2int_ru(f);
        a.frac = dsub(f, floor(f));
    }
    a.idx = base + w0;
    const bool ok = w0 >= 0 && w1 < win_n && base + w0 >= res_lo && base + w1 < res_hi;
    a.flags = (w1 - w0) | (ok ? 2 : 0);
}

// ---- lattice form of a non-separable transform -----------------------------------------------
// The target -> source transform is smooth at the scale of a CTA tile (64 x 32 pixels against the
// radius of the Earth), so it does not have to be evaluated per pixel: the CTA evaluates the full
// formulas at a 4 x 4 lattice spanning its tile plus the tile centre, and every pixel interpolates
// the source coordinates with the bicubic Lagrange polynomial through the lattice (collapsed per row
// in shared memory: 8 fused multiply-adds per pixel instead of ~400 instructions of series and
// arctangents).  The truncation error is |d4f/dx4| L^4 / 1944 per axis -- (L / R)^4 ~ 1e-16 of the
// coordinate for a 640 m tile -- and it is CHECKED, not assumed: the interpolant must reproduce the
// exactly transformed tile centre within K3L_TOL_PX source pixels on both axes, all 17 points must be
// finite, and the target coordinates must be equidistant; otherwise (coarse grids, projection
// singularities, the antimeridian inside the tile, domain limits) the CTA takes the exact per-pixel
// path.  1e-8 px is a hundredth of the 1e-6 px the ij image may differ from the reference.
#ifndef XRS_K3_LATTICE
#define XRS_K3_LATTICE 1
#endif
#ifndef XRS_K3_PREFETCH
#define XRS_K3_PREFETCH 1
#endif
constexpr double K3L_TOL_PX = 1e-8;
#ifndef XRS_K3_SEP_ROWBLOCK
#define XRS_K3_SEP_ROWBLOCK 1
#endif
#ifndef XRS_K3_SEP_PIPE
#define XRS_K3_SEP_PIPE 1
#endif
constexpr int K3W_NR = 10;  // source rows the 8 target rows of a thread may span in the row-block form

// cubic Lagrange basis on the nodes t = 0, 1, 2, 3
__device__ __forceinline__ void lagrange4(double t, double &w0, double &w1, double &w2, double &w3) {
    const double b = t - 1.0, c = t - 2.0, d = t - 3.0;
    w0 = b * c * d * (-1.0 / 6.0);
    w1 = t * c * d * 0.5;
    w2 = t * b * d * -0.5;
    w3 = t * b * c * (1.0 / 6.0);
}

// L2 prefetch of the source box [rj_lo, rj_hi] x [ci_lo, ci_hi] (element indices inside the resident
// planes) of every band: lane -> (row lane / 4, 128-byte line lane % 4), one instruction per band and
// 8 box rows.  The warp's demand loads of the following pixel rows then find their lines in L2 (or
// on the way) instead of paying the DRAM latency one pixel row at a time.
template <typename T, typename OUT>
__device__ __forceinline__ void k3_prefetch_box(const K3Planes<T, OUT> &planes, int n_bands, int pitch, int win_w,
                                                int win_h, int ci_lo, int ci_hi, int rj_lo, int rj_hi, int lane) {
    constexpr int LINE = 128 / static_cast<int>(sizeof(T));
    ci_lo = max(ci_lo, 0); ci_hi = min(ci_hi, win_w - 1);
    rj_lo = max(rj_lo, 0); rj_hi = min(rj_hi, win_h - 1);
    if (ci_lo > ci_hi || rj_lo > rj_hi) return;
    const int q = lane & 3;
    const bool col_on = q == 0 || ci_lo + (q - 1) * LINE < ci_hi;
    const int ce = min(ci_lo + q * LINE, ci_hi);
#pragma unroll 1
    for (int rb = rj_lo; rb <= rj_hi && rb < rj_lo + 16; rb += 8) {
        const int rj = rb + (lane >> 2);
        if (col_on && rj <= rj_hi) {
            const int off = rj * pitch + ce;
            for (int b = 0; b < n_bands; ++b)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(planes.src[b] + off));
        }
    }
}

#ifndef XRS_K3_TILE_COLS
#define XRS_K3_TILE_COLS 64
#endif
// CTA tile: K3T_COLS x K3T_ROWS target pixels, 8 warps of 32 columns x K3T_RPT rows (COLS * ROWS = 2048)
constexpr int K3T_COLS = XRS_K3_TILE_COLS, K3T_ROWS = 2048 / XRS_K3_TILE_COLS, K3T_THREADS = 256;
static_assert(K3T_COLS % 32 == 0 && K3T_COLS * K3T_ROWS == 2048 && K3T_COLS <= 256, "tile shape");
constexpr int K3T_RPT = K3T_ROWS / (K3T_THREADS / 32 / (K3T_COLS / 32));  // rows per thread (8)

// Row-block form of the separable bilinear kernel (see k3_reproject): the bands of one thread's 8 pixels.
// NR source rows starting at element offset o_src are lerped horizontally into the thread's slots of
// s_h; slot[i] holds the byte offsets (two 16-bit halves) of the slots pixel i blends vertically.
// Software-pipelined over the bands: the loads of band b + 1 are in flight while band b is blended.
template <typename T, typename OUT, int NR>
__device__ __forceinline__ void k3_rowblock_bands(const K3Planes<T, OUT> &planes, int n_bands, int o_src, int pitch,
                                                  double u, double *s_h, int tid, const uint32_t (&slot)[K3T_RPT],
                                                  const AxisTap *rt, int64_t o_first, int64_t dst_w) {
    T t0[NR], t1[NR];
    auto request = [&](int b) {
        const T *sp = planes.src[b] + o_src;
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            t0[k] = ld_tap(sp);
            t1[k] = ld_tap(sp + 1);
            sp += pitch;
        }
    };
    const char *hb = reinterpret_cast<const char *>(s_h);
    request(0);
#pragma unroll 1
    for (int b = 0; b < n_bands; ++b) {
#pragma unroll
        for (int k = 0; k < NR; ++k)
            s_h[k * K3T_THREADS + tid] = dadd(static_cast<double>(t0[k]), dmul(u, diff_as_f64(t1[k], t0[k])));
        if (XRS_K3_SEP_PIPE && b + 1 < n_bands) request(b + 1);
        OUT *dp = planes.dst[b] + o_first;
#pragma unroll
        for (int i = 0; i < K3T_RPT; ++i) {
            const double a = *reinterpret_cast<const double *>(hb + (slot[i] & 0xffffu));
            const double bb = *reinterpret_cast<const double *>(hb + (slot[i] >> 16));
            st_stream(dp, k3_store_cast<T, OUT>(dadd(a, dmul(rt[2 * i].frac, dsub(bb, a)))));
            dp += dst_w;
        }
        if (!XRS_K3_SEP_PIPE && b + 1 < n_bands) request(b + 1);
    }
}

// Lattice set-up of one CTA tile (see above).  On success s_rxy[rl] holds, for tile row rl, the four
// column-node values of the row-collapsed interpolant of x (entries 0-3) and y (4-7); xa / hx give the
// column parameter t = (x - xa) / hx of a pixel.  (The cubic Lagrange weights are bounded by 1 on the
// tile, so summing absolute coordinates costs a few ulp of the coordinate: ~1e-9 px at worst.)
// Target coordinates of lattice point `node` (0-15: the 4 x 4 nodes, row-major; 16: the centre) of the
// CTA tile whose first pixel is (c0, r0), and the node spacings.
__device__ __forceinline__ void k3_lattice_point(const K3Geom &g, int64_t c0, int64_t r0, int node, double &xa,
                                                 double &ya, double &hx, double &hy, double &step_x, double &step_y,
                                                 double &x, double &y) {
    xa = __ldg(g.dst_x + c0);
    ya = __ldg(g.dst_y + r0);
    step_x = (__ldg(g.dst_x + g.dst_w - 1) - __ldg(g.dst_x)) / static_cast<double>(g.dst_w - 1);
    step_y = (__ldg(g.dst_y + g.dst_h - 1) - __ldg(g.dst_y)) / static_cast<double>(g.dst_h - 1);
    hx = step_x * ((K3T_COLS - 1) / 3.0);
    hy = step_y * ((K3T_ROWS - 1) / 3.0);
    const double ti = node < 16 ? static_cast<double>(node & 3) : 1.5;
    const double tj = node < 16 ? static_cast<double>(node >> 2) : 1.5;
    x = xa + ti * hx;
    y = ya + tj * hy;
}

// The lattice of every CTA tile of a launch, evaluated ahead of the gather kernel (one thread per
// point, full formulas) so that the gather's CTAs start with a table read instead of a ~3 us serial
// chain of series and arctangents in 17 of their 256 threads.  34 doubles per tile: x of the 17
// points, then y.
__global__ void __launch_bounds__(256)
k3_lattice_nodes(const __grid_constant__ K3Geom g, double *__restrict__ nodes, int ntx, int n_tiles) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int tile = idx >> 5, node = idx & 31;
    if (tile >= n_tiles || node >= 17) return;
    const int64_t c0 = static_cast<int64_t>(tile % ntx) * K3T_COLS;
    const int64_t r0 = g.row_tile0 + static_cast<int64_t>(tile / ntx) * K3T_ROWS;
    double xa, ya, hx, hy, step_x, step_y, x, y, ox, oy;
    k3_lattice_point(g, c0, r0, node, xa, ya, hx, hy, step_x, step_y, x, y);
    transform_point(g.from, g.to, x, y, ox, oy);
    nodes[static_cast<size_t>(tile) * 34 + node] = ox;
    nodes[static_cast<size_t>(tile) * 34 + 17 + node] = oy;
}

__device__ __forceinline__ bool k3_lattice_setup(const K3Geom &g, int64_t c0, int64_t r0, int tid, double (*s_node)[17],
                                                 double (*s_rxy)[8], double &xa, double &hx) {
    double ya, hy, step_x, step_y, x, y;
    k3_lattice_point(g, c0, r0, tid < 17 ? tid : 0, xa, ya, hx, hy, step_x, step_y, x, y);
    bool ok = fabs(hx) > 0.0 && fabs(hy) > 0.0 && fabs(hx) < 1e300 && fabs(hy) < 1e300;
    if (tid < 17) {  // the 4 x 4 nodes (row-major) and the tile centre
        double ox, oy;
        if (g.lat_nodes) {
            const double *p = g.lat_nodes + (static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x) * 34;
            ox = __ldg(p + tid);
            oy = __ldg(p + 17 + tid);
        } else {
            transform_point(g.from, g.to, x, y, ox, oy);
        }
        s_node[0][tid] = ox;
        s_node[1][tid] = oy;
        ok = ok && fabs(ox) < 1e300 && fabs(oy) < 1e300;
    } else if (tid == 32) {  // equidistant target coordinates: the last column / row of the tile, where it exists
        const int64_t c = c0 + K3T_COLS - 1;
        if (c < g.dst_w) ok = ok && fabs(__ldg(g.dst_x + c) - (xa + 3.0 * hx)) <= 1e-6 * fabs(step_x);
    } else if (tid == 33) {
        const int64_t r = r0 + K3T_ROWS - 1;
        if (r < g.dst_h) ok = ok && fabs(__ldg(g.dst_y + r) - (ya + 3.0 * hy)) <= 1e-6 * fabs(step_y);
    }
    if (!__syncthreads_and(ok)) return false;
    for (int item = tid; item < K3T_ROWS * 8; item += K3T_THREADS) {  // rows x 4 column nodes x {x, y}
        const int rl = item >> 3, i = (item >> 1) & 3, cd = item & 1;
        double v = 0.0;
        if (r0 + rl < g.row_end) {
            double w0, w1, w2, w3;
            lagrange4((__ldg(g.dst_y + r0 + rl) - ya) / hy, w0, w1, w2, w3);
            v = w0 * s_node[cd][i] + w1 * s_node[cd][4 + i] + w2 * s_node[cd][8 + i] + w3 * s_node[cd][12 + i];
        }
        s_rxy[rl][cd * 4 + i] = v;
    }
    const int cd = tid & 1;
    bool ok2 = true;
    if (tid < 2) {  // the interpolant at the tile centre (t = 1.5 on both axes) against the exact transform
        const double w[4] = {-0.0625, 0.5625, 0.5625, -0.0625};
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc += w[j] * w[k] * s_node[cd][4 * j + k];
        ok2 = fabs(acc - s_node[cd][16]) <= K3L_TOL_PX * (cd == 0 ? g.x_res : g.y_res);
    }
    return __syncthreads_and(ok2);
}

// One CTA per 64 x 32 target tile; a warp owns 32 columns x 8 rows.  How a pixel gets its source
// coordinates depends on the transform:
//   separable (SEP)  lon / lat by column / row: the whole index arithmetic is per tile row / column
//   lattice          bicubic interpolation of the exact transform at 4 x 4 points of the tile (checked)
//   exact            32 + 64 threads evaluate the row-only and column-only parts of the transform (one
//                    sincos / exp each) into shared memory, each lane finishes the transform per pixel
// and then gathers all bands.
#ifndef XRS_K3_MINBLOCKS
#define XRS_K3_MINBLOCKS 4  // 64 registers; 2 and 3 CTAs per SM measured slower (profiles/README.md)
#endif
#ifndef XRS_K3_MINBLOCKS_NEAREST
#define XRS_K3_MINBLOCKS_NEAREST 5  // nearest keeps one tap per band: 5 CTAs (51 registers) measured 6 % faster on C3;
#endif                              // the blends spill at 5 and lose 25 %
template <typename T, typename OUT, int METHOD, bool SEP>
__global__ void __launch_bounds__(K3T_THREADS, METHOD == XRS_NEAREST ? XRS_K3_MINBLOCKS_NEAREST : XRS_K3_MINBLOCKS)
k3_reproject(const __grid_constant__ K3Geom g, const __grid_constant__ K3Planes<T, OUT> planes, int n_bands, T fill,
             int plan) {
    __shared__ Terms4 s_row[K3T_ROWS];
    __shared__ Terms4 s_col[K3T_COLS];
    __shared__ int s_ty[K3T_ROWS];
    __shared__ int s_tx[K3T_COLS];
    __shared__ AxisTap s_rowtap[SEP ? K3T_ROWS : 1][2];
    __shared__ AxisTap s_coltap[SEP ? K3T_COLS : 1][2];
    __shared__ double s_h[(SEP && METHOD == XRS_BILINEAR && XRS_K3_SEP_ROWBLOCK) ? K3W_NR : 1][K3T_THREADS];
    __shared__ double s_node[SEP ? 1 : 2][17];
    __shared__ __align__(16) double s_rxy[SEP ? 1 : K3T_ROWS][8];
    const int tid = threadIdx.x;
    const int64_t c0 = static_cast<int64_t>(blockIdx.x) * K3T_COLS;
    const int64_t r0 = g.row_tile0 + static_cast<int64_t>(blockIdx.y) * K3T_ROWS;
    // reference tile of every row / column of the CTA tile
    for (int k = tid; k < K3T_ROWS + K3T_COLS; k += K3T_THREADS) {
        if (k < K3T_ROWS) {
            const int64_t r = r0 + k;
            if (r < g.row_end) s_ty[k] = static_cast<int>(r / g.tile_h);
        } else {
            const int64_t c = c0 + (k - K3T_ROWS);
            if (c < g.dst_w) s_tx[k - K3T_ROWS] = static_cast<int>(c / g.tile_w);
        }
    }
    bool lattice = false;
    double lat_xa = 0.0, lat_hx = 1.0;
    const bool lattice_allowed = !(plan & K3_PLAN_EXACT_ONLY);
    plan &= K3_PLAN_MASK;
    if constexpr (!SEP) {
        if (XRS_K3_LATTICE && lattice_allowed && plan != K3_PLAN_IDENTITY && g.dst_w > 1 && g.dst_h > 1)
            lattice = k3_lattice_setup(g, c0, r0, tid, s_node, s_rxy, lat_xa, lat_hx);
    }
    if (!lattice) {
        for (int k = tid; k < K3T_ROWS + K3T_COLS; k += K3T_THREADS) {
            if (k < K3T_ROWS) {
                const int64_t r = r0 + k;
                if (r < g.row_end) s_row[k] = k3_row_terms(g, plan, __ldg(g.dst_y + r));
            } else {
                const int64_t c = c0 + (k - K3T_ROWS);
                if (c < g.dst_w) s_col[k - K3T_ROWS] = k3_col_terms(g, plan, __ldg(g.dst_x + c));
            }
        }
        __syncthreads();
    }
    // Separable transforms (geographic <-> web Mercator, identity): the source x of a pixel depends on
    // its column only and the source y on its row only, so the whole index arithmetic of
    // reproject.py:278-300 -- the two divisions, floor / ceil, the fractions, the window and residency
    // tests -- is done once per tile column and tile row instead of once per pixel.  The window
    // origins belong to the reference tile, and a CTA tile can straddle a reference-tile border, so
    // every column gets one entry per reference-tile ROW the CTA touches (at most two) and vice versa.
    const int ty_a = static_cast<int>(r0 / g.tile_h), tx_a = static_cast<int>(c0 / g.tile_w);
    const int ty_b = static_cast<int>(min(r0 + K3T_ROWS, g.row_end) - 1) / g.tile_h;
    const int tx_b = static_cast<int>(min(c0 + K3T_COLS, g.dst_w) - 1) / g.tile_w;
    // (SEP kernels are launched only for transforms whose source x / y depend on the target column / row
    // alone: both CRSs geographic or web Mercator)
    const bool sep = SEP && ty_b - ty_a <= 1 && tx_b - tx_a <= 1;
    if (sep) {
        const int res_i0 = static_cast<int>(g.win_i0), res_j0 = static_cast<int>(g.win_j0);
        const int res_i1 = res_i0 + static_cast<int>(g.win_w), res_j1 = res_j0 + static_cast<int>(g.win_h);
        for (int k = tid; k < 2 * K3T_ROWS + 2 * K3T_COLS; k += K3T_THREADS) {
            AxisTap a;
            a.frac = 0.0; a.idx = 0; a.flags = 0;
            const int q = k & 1;
            if (k < 2 * K3T_ROWS) {  // rows: entry [rl][q] for reference-tile column tx_a + q
                const int rl = k >> 1;
                if (r0 + rl < g.row_end && tx_a + q <= tx_b) {
                    const int t = s_ty[rl] * g.ntx + tx_a + q;
                    const double f = ddiv(dsub(s_row[rl].a, __ldg(g.tile_y0 + t)), -g.y_res);
                    axis_tap<METHOD>(f, __ldg(g.tile_j0 + t), g.tile_win_h, res_j0, res_j1, a);
                }
                s_rowtap[rl][q] = a;
            } else {  // columns: entry [cl][q] for reference-tile row ty_a + q
                const int cl = (k - 2 * K3T_ROWS) >> 1;
                if (c0 + cl < g.dst_w && ty_a + q <= ty_b) {
                    const int t = (ty_a + q) * g.ntx + s_tx[cl];
                    const double f = ddiv(dsub(s_col[cl].a, __ldg(g.tile_x0 + t)), g.x_res);
                    axis_tap<METHOD>(f, __ldg(g.tile_i0 + t), g.tile_win_w, res_i0, res_i1, a);
                }
                s_coltap[cl][q] = a;
            }
        }
        __syncthreads();
    }
    const int warp = tid >> 5, lane = tid & 31;
    const int col_l = (warp % (K3T_COLS / 32)) * 32 + lane;
    const int row_l0 = (warp / (K3T_COLS / 32)) * K3T_RPT;
    const int64_t c = c0 + col_l;
    // the warp's rows inside the requested band [row_begin, row_end) (warp-uniform)
    const int row_first = static_cast<int>(max(static_cast<int64_t>(row_l0), g.row_begin - r0));
    const int row_last = static_cast<int>(min(static_cast<int64_t>(row_l0 + K3T_RPT), g.row_end - r0)) - 1;
    if (row_first > row_last) return;
    const bool col_in = c < g.dst_w;
    if (sep) {
        const int pitch = static_cast<int>(g.src_pitch);
        const int res_i0 = static_cast<int>(g.win_i0), res_j0 = static_cast<int>(g.win_j0);
        AxisTap ca0, ca1;
        ca0.frac = ca1.frac = 0.0; ca0.idx = ca1.idx = 0; ca0.flags = ca1.flags = 0;
        int tx = tx_a;
        if (col_in) {
            ca0 = s_coltap[col_l][0]; ca1 = s_coltap[col_l][1];
            tx = s_tx[col_l];
        }
        if (XRS_K3_PREFETCH) {  // the source box of the warp's 32 x 8 pixels
            const AxisTap ra = s_rowtap[row_first][tx - tx_a], rb = s_rowtap[row_last][tx - tx_a];
            int ci_lo = INT32_MAX, ci_hi = INT32_MIN, rj_lo = INT32_MAX, rj_hi = INT32_MIN;
            const AxisTap &ca = (s_ty[row_first] == ty_a) ? ca0 : ca1;
            if (col_in && (ca.flags & ra.flags & rb.flags & 2)) {
                ci_lo = ca.idx - res_i0; ci_hi = ci_lo + 1;
                rj_lo = min(ra.idx, rb.idx) - res_j0; rj_hi = max(ra.idx, rb.idx) - res_j0 + 1;
            }
            ci_lo = __reduce_min_sync(0xffffffffu, ci_lo); ci_hi = __reduce_max_sync(0xffffffffu, ci_hi);
            rj_lo = __reduce_min_sync(0xffffffffu, rj_lo); rj_hi = __reduce_max_sync(0xffffffffu, rj_hi);
            k3_prefetch_box<T, OUT>(planes, n_bands, pitch, static_cast<int>(g.win_w), static_cast<int>(g.win_h), ci_lo,
                                    ci_hi, rj_lo, rj_hi, lane);
        }
        if (!col_in) return;
        if constexpr (SEP && METHOD == XRS_BILINEAR && XRS_K3_SEP_ROWBLOCK) {
            // Row-block form.  Along a target column the horizontal part of the blend -- the two taps of a
            // source row, their difference in the source dtype, the widening to float64 and the lerp with
            // the column's fraction (reproject.py:325-326) -- depends on the SOURCE row only, and the
            // thread's 8 target rows share their source rows (lower taps of one pixel = upper taps of the
            // next; when upsampling several pixels sit between the same two rows).  So per band the thread
            // loads and lerps every source row of its span ONCE into its own shared-memory slots (all loads
            // of a band in flight together) and each pixel is one vertical lerp of two slots
            // (reproject.py:327): the same operations on the same operands as the per-pixel form, bit for
            // bit, with about half the loads, conversions and float64 operations.
            const int q = tx - tx_a;
            const int ty = s_ty[row_first];
            const AxisTap ca = (ty == ty_a) ? ca0 : ca1;
            // (a column exactly on a source pixel centre -- both taps the same element -- takes the per-pixel form)
            bool block = ty == s_ty[row_last] && (ca.flags & 3) == 3 && row_last - row_first == K3T_RPT - 1;
            int j_lo = INT32_MAX, j_hi = INT32_MIN;
#pragma unroll
            for (int i = 0; i < K3T_RPT; ++i) {
                const AxisTap ra = s_rowtap[min(row_first + i, row_last)][q];
                block = block && (ra.flags & 2);
                j_lo = min(j_lo, ra.idx);
                j_hi = max(j_hi, ra.idx + (ra.flags & 1));
            }
            const int n_src = j_hi - j_lo + 1;
            // number of source rows staged: the smallest of 4 / 7 / 10 that holds the span of every lane
            // (no per-row predicates in the band loop); they must all lie inside the resident source
            const int n_max = __reduce_max_sync(__activemask(), block ? n_src : K3W_NR + 1);
            const int nr = n_max <= 4 ? 4 : n_max <= 7 ? 7 : K3W_NR;
            block = block && n_max <= K3W_NR && (j_lo - res_j0) + nr <= static_cast<int>(g.win_h);
            if (block) {
                // byte offsets of each pixel's two slots inside s_h, packed as two 16-bit halves
                uint32_t slot[K3T_RPT];
#pragma unroll
                for (int i = 0; i < K3T_RPT; ++i) {
                    const AxisTap ra = s_rowtap[row_first + i][q];
                    const uint32_t k0 = static_cast<uint32_t>(ra.idx - j_lo), k1 = k0 + (ra.flags & 1);
                    slot[i] = (k0 * (K3T_THREADS * 8) + tid * 8) | ((k1 * (K3T_THREADS * 8) + tid * 8) << 16);
                }
                const int o_src = (j_lo - res_j0) * pitch + (ca.idx - res_i0);
                const int64_t o_first = (r0 + row_first - g.row_begin) * g.dst_w + c;
                const AxisTap *rt = &s_rowtap[row_first][q];
                if (nr == 4) k3_rowblock_bands<T, OUT, 4>(planes, n_bands, o_src, pitch, ca.frac, &s_h[0][0], tid, slot, rt, o_first, g.dst_w);
                else if (nr == 7) k3_rowblock_bands<T, OUT, 7>(planes, n_bands, o_src, pitch, ca.frac, &s_h[0][0], tid, slot, rt, o_first, g.dst_w);
                else k3_rowblock_bands<T, OUT, K3W_NR>(planes, n_bands, o_src, pitch, ca.frac, &s_h[0][0], tid, slot, rt, o_first, g.dst_w);
                return;
            }
        }
#pragma unroll 1
        for (int rl = row_first; rl <= row_last; ++rl) {
            const int64_t r = r0 + rl;
            const int ty = s_ty[rl];
            const AxisTap ca = (ty == ty_a) ? ca0 : ca1;
            const AxisTap ra = s_rowtap[rl][tx - tx_a];
            const int64_t o = (r - g.row_begin) * g.dst_w + c;
            if (ca.flags & ra.flags & 2) {  // every tap inside the tile window and the resident source
                const int o00 = (ra.idx - res_j0) * pitch + (ca.idx - res_i0);
                // (nothing but these loads stands between a pixel and its stores: more of them in flight)
                if (METHOD == XRS_NEAREST) k3_copy_tap<T, OUT>(planes, n_bands, o, o00);
                else k3_blend_taps<T, OUT, METHOD, K3_SEP_CHUNK>(planes, n_bands, o, o00, ca.flags & 1,
                                                                 (ra.flags & 1) * pitch, pitch, ca.frac, ra.frac);
            } else {  // source border, padding, untransformable: the general per-pixel path
                k3_gather_pixel<T, OUT, METHOD>(g, planes, n_bands, fill, o, ty * g.ntx + tx, s_col[col_l].a, s_row[rl].a);
            }
        }
        return;
    }
    if constexpr (!SEP) {
        if (lattice) {
            double wc0 = 0.0, wc1 = 0.0, wc2 = 0.0, wc3 = 0.0;
            int tx = 0;
            if (col_in) {
                lagrange4((__ldg(g.dst_x + c) - lat_xa) / lat_hx, wc0, wc1, wc2, wc3);
                tx = s_tx[col_l];
            }
            // source coordinates of the pixel in tile row rl: 4 broadcast reads + 8 multiply-adds
            auto source_xy = [&](int rl, double &sx, double &sy) {
                const double2 *p = reinterpret_cast<const double2 *>(s_rxy[rl]);
                const double2 x01 = p[0], x23 = p[1], y01 = p[2], y23 = p[3];
                sx = wc0 * x01.x + wc1 * x01.y + wc2 * x23.x + wc3 * x23.y;
                sy = wc0 * y01.x + wc1 * y01.y + wc2 * y23.x + wc3 * y23.y;
            };
            if (XRS_K3_PREFETCH) {  // the source box of the warp's 32 x 8 pixels from its first and last row
                int ci_lo = INT32_MAX, ci_hi = INT32_MIN, rj_lo = INT32_MAX, rj_hi = INT32_MIN;
                if (col_in) {
#pragma unroll 1
                    for (int e = 0; e < 2; ++e) {
                        const int rl = e ? row_last : row_first;
                        double sx, sy;
                        source_xy(rl, sx, sy);
                        const K3Tile tl = k3_load_tile(g, s_ty[rl] * g.ntx + tx);
                        const double fx = (sx - tl.x0) * g.inv_x_res, fy = (tl.y0 - sy) * g.inv_y_res;
                        if (fabs(fx) < 1e9 && fabs(fy) < 1e9) {
                            const int ci = tl.i0 + __double2int_rd(fx) - static_cast<int>(g.win_i0);
                            const int rj = tl.j0 + __double2int_rd(fy) - static_cast<int>(g.win_j0);
                            ci_lo = min(ci_lo, ci); ci_hi = max(ci_hi, ci + 1);
                            rj_lo = min(rj_lo, rj); rj_hi = max(rj_hi, rj + 1);
                        }
                    }
                }
                ci_lo = __reduce_min_sync(0xffffffffu, ci_lo); ci_hi = __reduce_max_sync(0xffffffffu, ci_hi);
                rj_lo = __reduce_min_sync(0xffffffffu, rj_lo); rj_hi = __reduce_max_sync(0xffffffffu, rj_hi);
                k3_prefetch_box<T, OUT>(planes, n_bands, static_cast<int>(g.src_pitch), static_cast<int>(g.win_w),
                                        static_cast<int>(g.win_h), ci_lo, ci_hi, rj_lo, rj_hi, lane);
            }
            if (!col_in) return;
#pragma unroll 1
            for (int rl = row_first; rl <= row_last; ++rl) {
                const int64_t r = r0 + rl;
                double sx, sy;
                source_xy(rl, sx, sy);
                k3_gather_pixel<T, OUT, METHOD, true>(g, planes, n_bands, fill, (r - g.row_begin) * g.dst_w + c,
                                                      k3_load_tile(g, s_ty[rl] * g.ntx + tx), sx, sy);
            }
            return;
        }
    }
    if (!col_in) return;
    const Terms4 ct = s_col[col_l];
    const int tx = s_tx[col_l];
    // (Tried and measured slower on config C3, 13 bands: requesting the first bands' taps of pixel k before
    // transforming pixel k + 1 -- 6.9 ms against 4.9 ms, the extra live registers halve the occupancy; and
    // eight instead of four bands in flight in the separable kernel -- 2.99 against 2.92 ms on config C5.)
#pragma unroll 1
    for (int rl = row_first; rl <= row_last; ++rl) {
        const int64_t r = r0 + rl;
        const Terms4 rt = s_row[rl];
        double sx, sy;
        k3_pixel_source_xy(g, plan, rt, ct, c, r, sx, sy);
        k3_gather_pixel<T, OUT, METHOD>(g, planes, n_bands, fill, (r - g.row_begin) * g.dst_w + c,
                                        s_ty[rl] * g.ntx + tx, sx, sy);
    }
}

#ifdef XRS_K3_STAGED_EXPERIMENT
// ---------------------------------------------------------------------------
// K3, staged form: the gather of K2 (gather.cu) under the reprojection's index arithmetic.
//
// One CTA per 32 x 32 target tile, 4 pixels per thread (same column, rows 8 apart).  Every thread
// finishes the transform of its pixels and derives their taps; the CTA reduces the bounding box of
// the source pixels the tile reaches and pulls that box of every band into shared memory with 2-D TMA
// tensor copies (4-stage mbarrier ring), so that the 2 x 2 taps are shared-memory reads and each
// source pixel crosses L2 -> SM once per tile instead of once per tap.  Tiles that touch the source
// border (padding, numpy's negative-index wrap), whose box does not fit, or whose source pitch TMA
// cannot describe take the direct per-pixel path (k3_gather_pixel) -- same arithmetic.
//
// MEASURED SLOWER than the direct kernel on B200 (config C3, 13 bands: 5.8 vs 4.9 ms; 32 bands: 12.3 vs
// 10.8 ms; config C5, 8 variables: 4.4 vs 3.2 ms): the reprojection's taps of neighbouring pixels
// are neighbours in the source, so L1 / L2 already serve them, while the staging adds a box
// reduction, a TMA round trip per tile and a barrier per band, at half the occupancy.  Kept as a
// documented experiment: compiled only with -DXRS_K3_STAGED_EXPERIMENT, selected with XRS_K3_STAGED=1.
// ---------------------------------------------------------------------------
constexpr int K3S_TW = 32, K3S_TH = 32, K3S_THREADS = 256, K3S_PX = 4;
constexpr int K3S_ROW_STEP = K3S_THREADS / K3S_TW;
constexpr int K3S_BOX_W = 48, K3S_BOX_H = 40, K3S_STAGES = 4;

template <typename T, typename OUT>
struct K3StagedParams {
    CUtensorMap maps[K3_MAX_BANDS];
    K3Planes<T, OUT> planes;
};

template <typename T, typename OUT, int METHOD>
__global__ void __launch_bounds__(K3S_THREADS, 2)
k3_reproject_staged(const __grid_constant__ K3Geom g, const __grid_constant__ K3StagedParams<T, OUT> p, int n_bands,
                    T fill, int plan) {
    extern __shared__ unsigned char k3s_smem_raw[];
    constexpr int STAGE_ELEMS = K3S_BOX_W * K3S_BOX_H;
    unsigned char *base = k3s_smem_raw + ((128u - (smem_u32(k3s_smem_raw) & 127u)) & 127u);
    T *stages = reinterpret_cast<T *>(base);
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(base + static_cast<size_t>(K3S_STAGES) * STAGE_ELEMS * sizeof(T));
    Terms4 *s_row = reinterpret_cast<Terms4 *>(full_bar + K3S_STAGES);
    Terms4 *s_col = s_row + K3S_TH;
    int *s_ty = reinterpret_cast<int *>(s_col + K3S_TW);
    int *s_tx = s_ty + K3S_TH;
    int(*red)[K3S_THREADS / 32] = reinterpret_cast<int(*)[K3S_THREADS / 32]>(s_tx + K3S_TW);  // [5][8]

    const int tid = threadIdx.x;
    const int64_t c0 = static_cast<int64_t>(blockIdx.x) * K3S_TW;
    const int64_t r0 = g.row_begin + static_cast<int64_t>(blockIdx.y) * K3S_TH;
    if (tid < K3S_TH) {
        const int64_t r = r0 + tid;
        if (r < g.row_end) {
            s_row[tid] = k3_row_terms(g, plan, __ldg(g.dst_y + r));
            s_ty[tid] = static_cast<int>(r / g.tile_h);
        }
    } else if (tid < K3S_TH + K3S_TW) {
        const int k = tid - K3S_TH;
        const int64_t c = c0 + k;
        if (c < g.dst_w) {
            s_col[k] = k3_col_terms(g, plan, __ldg(g.dst_x + c));
            s_tx[k] = static_cast<int>(c / g.tile_w);
        }
    }
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < K3S_STAGES; ++s) mbar_init(&full_bar[s], 1);
        mbar_fence_init();
    }
    __syncthreads();

    const int lx = tid % K3S_TW, ly = tid / K3S_TW;
    const int64_t c = c0 + lx;
    const bool col_in = c < g.dst_w;
    const int res_i0 = static_cast<int>(g.win_i0), res_j0 = static_cast<int>(g.win_j0);
    const int res_i1 = res_i0 + static_cast<int>(g.win_w), res_j1 = res_j0 + static_cast<int>(g.win_h);
    const int ww = g.tile_win_w, wh = g.tile_win_h;

    // ---- this thread's pixels: transform, taps, fractions ----------------------------------
    double us[K3S_PX], vs[K3S_PX];
    int si0[K3S_PX], sj0[K3S_PX];
    uint32_t in_mask = 0, fast_mask = 0, d01_mask = 0, d10_mask = 0;  // bit k: pixel k / its right / lower tap is one further
    int i_lo = INT32_MAX, i_hi = -1, j_lo = INT32_MAX, j_hi = -1;
    Terms4 ct;
    int tx_tile = 0;
    if (col_in) {
        ct = s_col[lx];
        tx_tile = s_tx[lx];
    }
#pragma unroll
    for (int k = 0; k < K3S_PX; ++k) {
        us[k] = vs[k] = 0.0;
        si0[k] = sj0[k] = 0;
    }
    // (the transform code appears once: the loop is not unrolled and its results are moved into the
    // statically indexed per-pixel registers by predicated copies)
#pragma unroll 1
    for (int k = 0; k < K3S_PX; ++k) {
        const int rl = ly + k * K3S_ROW_STEP;
        const int64_t r = r0 + rl;
        if (!(col_in && r < g.row_end)) continue;
        double sx, sy, u = 0.0, v = 0.0;
        int a0 = 0, b0 = 0, da = 0, db = 0;
        bool fast = false;
        k3_pixel_source_xy(g, plan, s_row[rl], ct, c, r, sx, sy);
        const int t = s_ty[rl] * g.ntx + tx_tile;
        // reproject.py:278-279
        const double fx = ddiv(dsub(sx, __ldg(g.tile_x0 + t)), g.x_res);
        const double fy = ddiv(dsub(sy, __ldg(g.tile_y0 + t)), -g.y_res);
        if (fabs(fx) < 1e9 && fabs(fy) < 1e9) {
            const int i_base = __ldg(g.tile_i0 + t), j_base = __ldg(g.tile_j0 + t);
            int wx0, wx1, wy0, wy1;
            if (METHOD == XRS_NEAREST) {
                wx0 = wx1 = __double2int_rn(fx);
                wy0 = wy1 = __double2int_rn(fy);
            } else {
                wx0 = __double2int_rd(fx); wx1 = __double2int_ru(fx);
                wy0 = __double2int_rd(fy); wy1 = __double2int_ru(fy);
                u = dsub(fx, floor(fx));
                v = dsub(fy, floor(fy));
            }
            a0 = i_base + wx0; b0 = j_base + wy0;
            const int a1 = i_base + wx1, b1 = j_base + wy1;
            da = a1 - a0; db = b1 - b0;
            // all taps inside the tile window (no negative-index wrap, no IndexError) and inside the resident source
            fast = wx0 >= 0 && wy0 >= 0 && wx1 < ww && wy1 < wh && a0 >= res_i0 && b0 >= res_j0 && a1 < res_i1 && b1 < res_j1;
            if (fast) {
                i_lo = min(i_lo, a0); i_hi = max(i_hi, a1);
                j_lo = min(j_lo, b0); j_hi = max(j_hi, b1);
            }
        }
        in_mask |= 1u << k;
        fast_mask |= fast ? (1u << k) : 0u;
        d01_mask |= (fast && da) ? (1u << k) : 0u;
        d10_mask |= (fast && db) ? (1u << k) : 0u;
#pragma unroll
        for (int q = 0; q < K3S_PX; ++q)
            if (q == k) {
                us[q] = u; vs[q] = v;
                si0[q] = a0; sj0[q] = b0;
            }
    }
    // ---- CTA-wide: are all pixels on the fast path, and which source box do they reach? ----------
    int all_fast = (fast_mask == in_mask) ? 1 : 0;
    all_fast = __reduce_min_sync(0xffffffffu, all_fast);
    i_lo = __reduce_min_sync(0xffffffffu, i_lo); i_hi = __reduce_max_sync(0xffffffffu, i_hi);
    j_lo = __reduce_min_sync(0xffffffffu, j_lo); j_hi = __reduce_max_sync(0xffffffffu, j_hi);
    if ((tid & 31) == 0) {
        red[0][tid >> 5] = i_lo; red[1][tid >> 5] = i_hi; red[2][tid >> 5] = j_lo; red[3][tid >> 5] = j_hi;
        red[4][tid >> 5] = all_fast;
    }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < K3S_THREADS / 32; ++w) {
        i_lo = min(i_lo, red[0][w]); i_hi = max(i_hi, red[1][w]);
        j_lo = min(j_lo, red[2][w]); j_hi = max(j_hi, red[3][w]);
        all_fast = min(all_fast, red[4][w]);
    }
    constexpr int ALIGN_ELEMS = 16 / sizeof(T) > 0 ? 16 / sizeof(T) : 1;
    const int box_x = i_hi >= 0 ? ((i_lo - res_i0) / ALIGN_ELEMS) * ALIGN_ELEMS : 0;
    const int box_y = i_hi >= 0 ? j_lo - res_j0 : 0;
    const int box_i0 = box_x + res_i0;  // first source column held by the staged box
    const bool staged = all_fast && i_hi >= 0 && (i_hi - box_i0 + 1 <= K3S_BOX_W) && (j_hi - j_lo + 1 <= K3S_BOX_H);

    if (!staged) {  // CTA-uniform and rare: the direct per-pixel path, same arithmetic (transform redone)
#pragma unroll 1
        for (int k = 0; k < K3S_PX; ++k) {
            if (!(in_mask & (1u << k))) continue;
            const int rl = ly + k * K3S_ROW_STEP;
            const int64_t r = r0 + rl;
            double sx, sy;
            k3_pixel_source_xy(g, plan, s_row[rl], ct, c, r, sx, sy);
            k3_gather_pixel<T, OUT, METHOD>(g, p.planes, n_bands, fill, (r - g.row_begin) * g.dst_w + c,
                                            s_ty[rl] * g.ntx + tx_tile, sx, sy);
        }
        return;
    }

    const T *t00[K3S_PX], *t01[K3S_PX], *t10[K3S_PX], *t11[K3S_PX];
    uint32_t o32[K3S_PX];
#pragma unroll
    for (int k = 0; k < K3S_PX; ++k) {
        const bool on = in_mask & (1u << k);
        const int off = on ? (sj0[k] - j_lo) * K3S_BOX_W + (si0[k] - box_i0) : 0;
        const int d01 = (d01_mask >> k) & 1u, d10 = ((d10_mask >> k) & 1u) * K3S_BOX_W;
        t00[k] = stages + off;
        t01[k] = t00[k] + d01;
        t10[k] = t00[k] + d10;
        t11[k] = t10[k] + d01;
        const int64_t r = r0 + ly + k * K3S_ROW_STEP;
        o32[k] = static_cast<uint32_t>((r - g.row_begin) * g.dst_w + c);
    }
    asm volatile("" : "+r"(in_mask));  // keep the store predicate a one-bit test inside the band loop
    constexpr uint32_t STAGE_BYTES = STAGE_ELEMS * sizeof(T);
    if (tid == 0) {
        for (int s = 0; s < K3S_STAGES && s < n_bands; ++s) {
            mbar_arrive_expect_tx(&full_bar[s], STAGE_BYTES);
            tma_load_2d(stages + s * STAGE_ELEMS, &p.maps[s], box_x, box_y, &full_bar[s]);
        }
    }
    for (int b0 = 0; b0 < n_bands; b0 += K3S_STAGES) {
        const uint32_t parity = (b0 / K3S_STAGES) & 1;
#pragma unroll
        for (int s = 0; s < K3S_STAGES; ++s) {
            const int b = b0 + s;
            if (b >= n_bands) break;
            mbar_wait(&full_bar[s], parity);
            OUT out[K3S_PX];
#pragma unroll
            for (int k = 0; k < K3S_PX; ++k) {
                if (METHOD == XRS_NEAREST) {
                    out[k] = static_cast<OUT>(t00[k][s * STAGE_ELEMS]);
                } else {
                    out[k] = k3_blend<T, OUT, METHOD>(t00[k][s * STAGE_ELEMS], t01[k][s * STAGE_ELEMS],
                                                      t10[k][s * STAGE_ELEMS], t11[k][s * STAGE_ELEMS], us[k], vs[k]);
                }
            }
            OUT *dp = p.planes.dst[b];
#pragma unroll
            for (int k = 0; k < K3S_PX; ++k)
                if (in_mask & (1u << k)) st_stream(elem_ptr(dp, o32[k]), out[k]);
            __syncthreads();  // every thread is done with stage s
            if (tid == 0 && b + K3S_STAGES < n_bands) {
                fence_proxy_async();
                mbar_arrive_expect_tx(&full_bar[s], STAGE_BYTES);
                tma_load_2d(stages + s * STAGE_ELEMS, &p.maps[b + K3S_STAGES], box_x, box_y, &full_bar[s]);
            }
        }
    }
}

#endif  // XRS_K3_STAGED_EXPERIMENT

static int choose_plan(const ProjC &from, const ProjC &to) {
    if (from.kind == XRS_PROJ_GEOGRAPHIC && to.kind == XRS_PROJ_GEOGRAPHIC) return K3_PLAN_IDENTITY;
    if (from.kind == XRS_PROJ_GEOGRAPHIC || from.kind == XRS_PROJ_WEBMERC) return K3_PLAN_SEPARABLE;
    if (from.kind == XRS_PROJ_TMERC) return K3_PLAN_TMERC_INV;
    return K3_PLAN_GENERIC;
}

// The scratch of k3_lattice_nodes comes from the device's default stream-ordered pool; by default the
// pool gives freed memory back to the driver at the next synchronisation and every call would pay
// a fresh allocation (measured: +1.4 ... 3.6 ms per call on C3).  Keep what was allocated once.
static void retain_default_pool() {
    static bool done[64] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || done[dev]) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t keep = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    (void)cudaGetLastError();
    done[dev] = true;
}

template <typename T, typename OUT, int METHOD>
int launch_reproject(const K3Geom &g_in, const void *const *src_planes, void *const *dst_planes, int n_bands, double fill,
                     cudaStream_t st) {
    K3Geom g = g_in;
    g.lat_nodes = nullptr;
    const int64_t rows = g.row_end - g.row_begin;
    const dim3 grid(static_cast<unsigned>(ceil_div(g.dst_w, K3T_COLS)),
                    static_cast<unsigned>(ceil_div(g.row_end - g.row_tile0, K3T_ROWS)));
    if (grid.y > 65535) return fail("xrs_reproject: more than 2097120 target rows per call");
    const T fill_t = cast_fill<T>(fill);
    // XRS_K3_EXACT=1 makes every pixel evaluate the full projection formulas (the tests compare the
    // lattice form with it)
    const char *exact_env = getenv("XRS_K3_EXACT");
    const int plan = choose_plan(g.from, g.to) | ((exact_env && exact_env[0] == '1') ? K3_PLAN_EXACT_ONLY : 0);
    // TMA needs 16-byte aligned plane bases and row strides; 32-bit output offsets need < 2^32 elements
#ifdef XRS_K3_STAGED_EXPERIMENT
    const char *staged_env = getenv("XRS_K3_STAGED");
    bool tma_ok = staged_env && staged_env[0] == '1' && tma_available() && (g.src_pitch * sizeof(T)) % 16 == 0 &&
                  rows * g.dst_w < (int64_t(1) << 32) && ceil_div(rows, K3S_TH) <= 65535;
    for (int b = 0; b < n_bands && tma_ok; ++b) tma_ok = (reinterpret_cast<uintptr_t>(src_planes[b]) & 15) == 0;
#endif
    const bool axis_only_crs = (g.from.kind == XRS_PROJ_GEOGRAPHIC || g.from.kind == XRS_PROJ_WEBMERC) &&
                               (g.to.kind == XRS_PROJ_GEOGRAPHIC || g.to.kind == XRS_PROJ_WEBMERC);
    double *nodes = nullptr;
    if (XRS_K3_LATTICE && !axis_only_crs && !(plan & K3_PLAN_EXACT_ONLY) && g.dst_w > 1 && g.dst_h > 1) {
        // the transform's lattice for every CTA tile (stream-ordered scratch; without it the gather's CTAs
        // evaluate their own lattice)
        const int n_tiles = static_cast<int>(grid.x * grid.y);
        retain_default_pool();
        if (cudaMallocAsync(reinterpret_cast<void **>(&nodes), static_cast<size_t>(n_tiles) * 34 * sizeof(double), st) ==
            cudaSuccess) {
            XRS_TIMED("k3_lattice_nodes", st, k3_lattice_nodes<<<static_cast<unsigned>(ceil_div(static_cast<int64_t>(n_tiles) * 32, 256)), 256, 0, st>>>(g, nodes, static_cast<int>(grid.x), n_tiles));
            XRS_LAUNCH_CHECK("k3_lattice_nodes");
            g.lat_nodes = nodes;
        } else {
            (void)cudaGetLastError();
            nodes = nullptr;
        }
    }
    struct NodesGuard {
        double *p;
        cudaStream_t st;
        ~NodesGuard() { if (p) cudaFreeAsync(p, st); }
    } nodes_guard{nodes, st};
    for (int b0 = 0; b0 < n_bands; b0 += K3_MAX_BANDS) {
        const int nb = std::min(K3_MAX_BANDS, n_bands - b0);
        K3Planes<T, OUT> planes = {};
        for (int b = 0; b < nb; ++b) {
            planes.src[b] = static_cast<const T *>(src_planes[b0 + b]);
            planes.dst[b] = static_cast<OUT *>(dst_planes[b0 + b]);
        }
#ifdef XRS_K3_STAGED_EXPERIMENT
        if (tma_ok) {
            K3StagedParams<T, OUT> sp;
            memset(&sp, 0, sizeof(sp));
            sp.planes = planes;
            bool ok = true;
            for (int b = 0; b < nb && ok; ++b)
                ok = tma_encode_2d(&sp.maps[b], sizeof(T), src_planes[b0 + b], static_cast<uint64_t>(g.win_w),
                                   static_cast<uint64_t>(g.win_h), static_cast<uint64_t>(g.src_pitch) * sizeof(T),
                                   K3S_BOX_W, K3S_BOX_H);
            if (ok) {
                const size_t smem = static_cast<size_t>(K3S_STAGES) * K3S_BOX_W * K3S_BOX_H * sizeof(T) +
                                    K3S_STAGES * sizeof(uint64_t) + (K3S_TH + K3S_TW) * (sizeof(Terms4) + sizeof(int)) +
                                    5 * (K3S_THREADS / 32) * sizeof(int) + 128;
                XRS_CUDA(cudaFuncSetAttribute(k3_reproject_staged<T, OUT, METHOD>,
                                              cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
                const dim3 sgrid(static_cast<unsigned>(ceil_div(g.dst_w, K3S_TW)), static_cast<unsigned>(ceil_div(rows, K3S_TH)));
                XRS_TIMED(METHOD == XRS_NEAREST ? "k3_reproject_staged<nearest>" : METHOD == XRS_BILINEAR ? "k3_reproject_staged<bilinear>" : "k3_reproject_staged<triangular>", st, k3_reproject_staged<T, OUT, METHOD><<<sgrid, K3S_THREADS, smem, st>>>(g, sp, nb, fill_t, plan & K3_PLAN_MASK));
                XRS_LAUNCH_CHECK("k3_reproject_staged");
                continue;
            }
        }
#endif
        const bool axis_only = (g.from.kind == XRS_PROJ_GEOGRAPHIC || g.from.kind == XRS_PROJ_WEBMERC) &&
                               (g.to.kind == XRS_PROJ_GEOGRAPHIC || g.to.kind == XRS_PROJ_WEBMERC);
        if (axis_only) {
            XRS_TIMED(METHOD == XRS_NEAREST ? "k3_reproject_sep<nearest>" : METHOD == XRS_BILINEAR ? "k3_reproject_sep<bilinear>" : "k3_reproject_sep<triangular>", st, k3_reproject<T, OUT, METHOD, true><<<grid, K3T_THREADS, 0, st>>>(g, planes, nb, fill_t, plan));
        } else {
            XRS_TIMED(METHOD == XRS_NEAREST ? "k3_reproject<nearest>" : METHOD == XRS_BILINEAR ? "k3_reproject<bilinear>" : "k3_reproject<triangular>", st, k3_reproject<T, OUT, METHOD, false><<<grid, K3T_THREADS, 0, st>>>(g, planes, nb, fill_t, plan));
        }
        XRS_LAUNCH_CHECK("k3_reproject");
    }
    return 0;
}

template <typename T>
int dispatch_reproject(const K3Geom &g, const void *const *src_planes, void *const *dst_planes, int n_bands,
                       int out_is_f64, int method, double fill, cudaStream_t st) {
    constexpr bool t_is_f64 = std::is_same<T, double>::value;
    switch (method) {
    case XRS_NEAREST:
        if (out_is_f64 && !t_is_f64) return fail("xrs_reproject: nearest writes the source dtype");
        return launch_reproject<T, T, XRS_NEAREST>(g, src_planes, dst_planes, n_bands, fill, st);
    case XRS_TRIANGULAR:
        if (out_is_f64 && !t_is_f64) return fail("xrs_reproject: triangular writes the source dtype");
        return launch_reproject<T, T, XRS_TRIANGULAR>(g, src_planes, dst_planes, n_bands, fill, st);
    case XRS_BILINEAR:
        if (out_is_f64 && !t_is_f64)
            return launch_reproject<T, double, XRS_BILINEAR>(g, src_planes, dst_planes, n_bands, fill, st);
        return launch_reproject<T, T, XRS_BILINEAR>(g, src_planes, dst_planes, n_bands, fill, st);
    default:
        return fail("interp_methods must be one of 0, 1, 'nearest', 'bilinear', 'triangular', was code " +
                    std::to_string(method));
    }
}

}  // namespace xrs

using namespace xrs;

extern "C" {

int xrs_transform_points(const xrs_proj *from_crs, const xrs_proj *to_crs, const double *x_in, const double *y_in,
                         double *x_out, double *y_out, int64_t n, void *stream) {
    if (n < 0) return fail("xrs_transform_points: negative count");
    if (n == 0) return 0;
    if (!x_in || !y_in || !x_out || !y_out) return fail("xrs_transform_points: null pointer");
    ProjC from, to;
    if (int rc = make_proj_consts(from_crs, &from)) return rc;
    if (int rc = make_proj_consts(to_crs, &to)) return rc;
    const unsigned blocks = static_cast<unsigned>(std::min<int64_t>(ceil_div(n, 256), 148 * 16));
    XRS_TIMED("k3_transform_points", static_cast<cudaStream_t>(stream), k3_transform_points<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(from, to, x_in, y_in, x_out, y_out, n));
    XRS_LAUNCH_CHECK("k3_transform_points");
    return 0;
}

int xrs_reproject(const void *const *src_planes_host, void *const *dst_planes_host, int32_t n_bands, int32_t dtype,
                  int32_t out_dtype, int64_t src_h, int64_t src_w, int64_t src_pitch, int64_t win_i0, int64_t win_j0,
                  int64_t win_w, int64_t win_h, const xrs_proj *src_crs, const xrs_proj *dst_crs, const double *dst_x,
                  const double *dst_y, int64_t dst_h, int64_t dst_w, int32_t tile_h, int32_t tile_w,
                  const double *tile_x0, const double *tile_y0, const int32_t *tile_i0, const int32_t *tile_j0,
                  int32_t tile_win_w, int32_t tile_win_h, double src_x_res, double src_y_res, int32_t method,
                  double fill, int64_t row_begin, int64_t row_end, void *stream) {
    if (!src_planes_host || !dst_planes_host || !dst_x || !dst_y || !tile_x0 || !tile_y0 || !tile_i0 || !tile_j0)
        return fail("xrs_reproject: null pointer");
    if (n_bands < 1) return fail("xrs_reproject: n_bands must be >= 1");
    if (src_h < 1 || src_w < 1 || src_pitch < win_w || dst_h < 1 || dst_w < 1 || tile_h < 1 || tile_w < 1)
        return fail("xrs_reproject: bad image shape");
    if (win_i0 < 0 || win_j0 < 0 || win_w < 1 || win_h < 1 || win_i0 + win_w > src_w || win_j0 + win_h > src_h)
        return fail("xrs_reproject: resident window outside the source image");
    if (row_begin < 0 || row_end > dst_h || row_begin >= row_end) return fail("xrs_reproject: bad row range");
    if (tile_win_w < 1 || tile_win_h < 1) return fail("xrs_reproject: bad tile window size");
    if (win_h * src_pitch >= (int64_t(1) << 31) || src_w >= (int64_t(1) << 30) || src_h >= (int64_t(1) << 30))
        return fail("xrs_reproject: resident source window has 2^31 or more elements per band; split the target "
                    "into row bands");
    if (!(src_x_res > 0.0) || !(src_y_res > 0.0)) return fail("xrs_reproject: resolution must be positive");
    if (out_dtype != dtype && out_dtype != XRS_F64) return fail("xrs_reproject: out_dtype must be dtype or float64");
    for (int b = 0; b < n_bands; ++b)
        if (!src_planes_host[b] || !dst_planes_host[b]) return fail("xrs_reproject: null plane pointer");
    K3Geom g;
    g.lat_nodes = nullptr;
    if (int rc = make_proj_consts(dst_crs, &g.from)) return rc;
    if (int rc = make_proj_consts(src_crs, &g.to)) return rc;
    g.dst_x = dst_x; g.dst_y = dst_y; g.dst_h = dst_h; g.dst_w = dst_w;
    g.row_begin = row_begin; g.row_end = row_end;
    g.row_tile0 = row_begin - row_begin % K3T_ROWS;
    g.tile_h = static_cast<int>(std::min<int64_t>(tile_h, dst_h));
    g.tile_w = static_cast<int>(std::min<int64_t>(tile_w, dst_w));
    g.ntx = static_cast<int>(ceil_div(dst_w, g.tile_w));
    g.tile_x0 = tile_x0; g.tile_y0 = tile_y0; g.tile_i0 = tile_i0; g.tile_j0 = tile_j0;
    g.tile_win_w = tile_win_w; g.tile_win_h = tile_win_h;
    g.x_res = src_x_res; g.y_res = src_y_res;
    g.inv_x_res = 1.0 / src_x_res; g.inv_y_res = 1.0 / src_y_res;
    g.src_h = src_h; g.src_w = src_w; g.src_pitch = src_pitch;
    g.win_i0 = win_i0; g.win_j0 = win_j0; g.win_w = win_w; g.win_h = win_h;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int out_is_f64 = out_dtype == XRS_F64;
    XRS_DISPATCH_DTYPE(dtype, T,
                       return dispatch_reproject<T>(g, src_planes_host, dst_planes_host, n_bands, out_is_f64, method,
                                                    fill, st));
    return 0;
}

}  // extern "C"
