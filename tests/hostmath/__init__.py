"""The projection math of the CUDA kernels, compiled for the HOST (test infrastructure, no GPU needed).

``csrc/proj.cuh`` holds the fp64 formulas the reprojection kernels evaluate on the device (``proj_forward``,
``proj_inverse``, ``proj_transform``).  They are plain C++ apart from the ``__device__`` qualifiers, so the
very same text can be compiled by g++: :func:`build` writes a translation unit that defines the CUDA
qualifiers away, includes the text of proj.cuh and exports one C function, and links it against
``libxrs.so`` for ``make_proj_consts`` (the host routine that derives the series coefficients).  CPU tests can
then hold the product's own formulas -- not a restatement -- against published known-answer vectors and
against the oracle, for any ellipsoid and projection parameters.  Differences to the device build are
confined to libm vs CUDA math-library rounding and FMA contraction (~1e-9 m).
"""

import ctypes
import os
import re
import shutil
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
CSRC = os.path.join(ROOT, "xcube_resampling_b200", "csrc")

SHIM = r"""
#define _GNU_SOURCE 1
#include <cmath>
#include <cstdint>
#include <math.h>
#include "xrs.h"
#define __device__
#define __host__
#define __forceinline__ inline
#define __constant__ const
using std::fabs; using std::sqrt; using std::sin; using std::cos; using std::tan; using std::atan; using std::atan2;
using std::asin; using std::sinh; using std::asinh; using std::exp; using std::log; using std::rint; using std::fmin;
using std::fmax;
"""

EXPORT = r"""
extern "C" int xrsh_transform_points(const xrs_proj *from, const xrs_proj *to, const double *x, const double *y,
                                     double *ox, double *oy, long n) {
    xrs::ProjC f, t;
    if (int rc = xrs::make_proj_consts(from, &f)) return rc;
    if (int rc = xrs::make_proj_consts(to, &t)) return rc;
    for (long i = 0; i < n; ++i) xrs::proj_transform(f, t, x[i], y[i], ox[i], oy[i]);
    return 0;
}

// The separable forms the reprojection kernel uses on regular grids: row-only and column-only terms once
// per row / column, a tail per pixel, the exact per-pixel path where the tail declines (as the kernel does).
extern "C" int xrsh_tmerc_inverse_grid(const xrs_proj *crs, const double *xs, long nx, const double *ys, long ny,
                                       double *lam, double *phi, unsigned char *declined) {
    xrs::ProjC P;
    if (int rc = xrs::make_proj_consts(crs, &P)) return rc;
    for (long j = 0; j < ny; ++j) {
        const xrs::Terms4 r = xrs::tmerc_inv_row_terms(P, ys[j]);
        for (long i = 0; i < nx; ++i) {
            const xrs::Terms4 c = xrs::tmerc_inv_col_terms(P, xs[i]);
            double l, p;
            const bool ok = xrs::tmerc_inv_tail(P, r, c, l, p);
            declined[j * nx + i] = ok ? 0 : 1;
            if (!ok && !xrs::proj_inverse(P, xs[i], ys[j], l, p)) l = p = NAN;
            lam[j * nx + i] = l;
            phi[j * nx + i] = p;
        }
    }
    return 0;
}

extern "C" int xrsh_forward_grid(const xrs_proj *crs, const double *lam, long nx, const double *phi, long ny, double *x,
                                 double *y) {
    xrs::ProjC P;
    if (int rc = xrs::make_proj_consts(crs, &P)) return rc;
    for (long j = 0; j < ny; ++j) {
        const xrs::Terms4 r = xrs::fwd_row_terms(P, phi[j], true);
        for (long i = 0; i < nx; ++i) xrs::fwd_tail(P, r, xrs::fwd_col_terms(P, lam[i]), x[j * nx + i], y[j * nx + i]);
    }
    return 0;
}

extern "C" int xrsh_inverse_points(const xrs_proj *crs, const double *x, const double *y, double *lam, double *phi, long n) {
    xrs::ProjC P;
    if (int rc = xrs::make_proj_consts(crs, &P)) return rc;
    for (long i = 0; i < n; ++i)
        if (!xrs::proj_inverse(P, x[i], y[i], lam[i], phi[i])) lam[i] = phi[i] = NAN;
    return 0;
}

extern "C" int xrsh_forward_points(const xrs_proj *crs, const double *lam, const double *phi, double *x, double *y, long n) {
    xrs::ProjC P;
    if (int rc = xrs::make_proj_consts(crs, &P)) return rc;
    for (long i = 0; i < n; ++i)
        if (!xrs::proj_forward(P, lam[i], phi[i], x[i], y[i])) x[i] = y[i] = NAN;
    return 0;
}
"""


class XrsProj(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int32), ("_pad", ctypes.c_int32), ("a", ctypes.c_double), ("inv_f", ctypes.c_double),
                ("lon0", ctypes.c_double), ("lat0", ctypes.c_double), ("k0", ctypes.c_double), ("fe", ctypes.c_double),
                ("fn", ctypes.c_double)]


def build(out_dir: str, lib_path: str) -> str:
    """Compile the host build of proj.cuh into ``out_dir`` and return the path of the shared object."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    text = open(os.path.join(CSRC, "proj.cuh")).read()
    text, n = re.subn(r'#include "common.cuh"\n', "", text)
    assert n == 1, "proj.cuh no longer includes common.cuh exactly once"
    text = text.replace("#pragma once\n", "").replace("#pragma unroll\n", "")
    src = os.path.join(out_dir, "proj_host.cpp")
    with open(src, "w") as fh:
        fh.write(SHIM + text + EXPORT)
    so = os.path.join(out_dir, "libxrs_projhost.so")
    lib_dir = os.path.dirname(lib_path)
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", f"-I{os.path.join(ROOT, 'include')}", src,
           "-o", so, f"-L{lib_dir}", f"-l:{os.path.basename(lib_path)}", f"-Wl,-rpath,{lib_dir}"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of proj.cuh failed:\n" + res.stderr[-3000:])
    return so


class HostProj:
    """``transform(from, to, x, y)`` through the product's formulas on the CPU; CRSs as (kind, a, inv_f,
    lon0, lat0, k0, fe, fn) tuples -- what ``CRS.proj_params()`` returns."""

    def __init__(self, so_path: str):
        self.lib = ctypes.CDLL(so_path)
        self.lib.xrsh_transform_points.restype = ctypes.c_int
        self.lib.xrsh_transform_points.argtypes = [ctypes.c_void_p] * 6 + [ctypes.c_long]

    @staticmethod
    def _proj(params) -> XrsProj:
        kind, a, inv_f, lon0, lat0, k0, fe, fn = params
        return XrsProj(int(kind), 0, a, inv_f, lon0, lat0, k0, fe, fn)

    def transform(self, src, dst, x, y):
        x = np.ascontiguousarray(np.atleast_1d(x), dtype=np.float64)
        y = np.ascontiguousarray(np.atleast_1d(y), dtype=np.float64)
        ox, oy = np.empty_like(x), np.empty_like(y)
        f, t = self._proj(src), self._proj(dst)
        rc = self.lib.xrsh_transform_points(ctypes.byref(f), ctypes.byref(t), x.ctypes.data, y.ctypes.data,
                                            ox.ctypes.data, oy.ctypes.data, x.size)
        if rc:
            raise RuntimeError(f"xrsh_transform_points failed ({rc})")
        return ox, oy

    def _call(self, name, *args):
        fn = getattr(self.lib, name)
        fn.restype = ctypes.c_int
        rc = fn(*args)
        if rc:
            raise RuntimeError(f"{name} failed ({rc})")

    def tmerc_inverse_grid(self, crs, xs, ys):
        """(lam, phi) in radians on the grid ys x xs through the separable row / column terms + tail, and the
        mask of pixels where the tail declined (the exact per-pixel inverse was used instead)."""
        xs = np.ascontiguousarray(xs, dtype=np.float64)
        ys = np.ascontiguousarray(ys, dtype=np.float64)
        lam, phi = np.empty((ys.size, xs.size)), np.empty((ys.size, xs.size))
        declined = np.zeros((ys.size, xs.size), dtype=np.uint8)
        p = self._proj(crs)
        self._call("xrsh_tmerc_inverse_grid", ctypes.byref(p), ctypes.c_void_p(xs.ctypes.data), ctypes.c_long(xs.size),
                   ctypes.c_void_p(ys.ctypes.data), ctypes.c_long(ys.size), ctypes.c_void_p(lam.ctypes.data),
                   ctypes.c_void_p(phi.ctypes.data), ctypes.c_void_p(declined.ctypes.data))
        return lam, phi, declined.astype(bool)

    def forward_grid(self, crs, lam, phi):
        """CRS coordinates on the grid phi (rows) x lam (columns), radians in, through the separable forms."""
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        phi = np.ascontiguousarray(phi, dtype=np.float64)
        x, y = np.empty((phi.size, lam.size)), np.empty((phi.size, lam.size))
        p = self._proj(crs)
        self._call("xrsh_forward_grid", ctypes.byref(p), ctypes.c_void_p(lam.ctypes.data), ctypes.c_long(lam.size),
                   ctypes.c_void_p(phi.ctypes.data), ctypes.c_long(phi.size), ctypes.c_void_p(x.ctypes.data),
                   ctypes.c_void_p(y.ctypes.data))
        return x, y

    def _points(self, name, crs, a, b):
        a = np.ascontiguousarray(a, dtype=np.float64).ravel()
        b = np.ascontiguousarray(b, dtype=np.float64).ravel()
        oa, ob = np.empty_like(a), np.empty_like(b)
        p = self._proj(crs)
        self._call(name, ctypes.byref(p), ctypes.c_void_p(a.ctypes.data), ctypes.c_void_p(b.ctypes.data),
                   ctypes.c_void_p(oa.ctypes.data), ctypes.c_void_p(ob.ctypes.data), ctypes.c_long(a.size))
        return oa, ob

    def inverse_points(self, crs, x, y):
        return self._points("xrsh_inverse_points", crs, x, y)

    def forward_points(self, crs, lam, phi):
        return self._points("xrsh_forward_points", crs, lam, phi)


# ---------------------------------------------------------------------------
# K1's resolve step (csrc/rectify_common.cuh: resolve_row / resolve_pixel, div_magic)
# ---------------------------------------------------------------------------
RESOLVE_SHIM = r"""
#include <climits>
#include <cmath>
#include <cstdint>
#include "xrs.h"
#define __device__
#define __host__
#define __forceinline__ inline
typedef void *cudaStream_t;
namespace xrs {
// common.cuh's _rn wrappers: plain IEEE operations (this unit is compiled with -ffp-contract=off)
static inline double dadd(double a, double b) { return a + b; }
static inline double dsub(double a, double b) { return a - b; }
static inline double dmul(double a, double b) { return a * b; }
static inline double ddiv(double a, double b) { return a / b; }
}
template <typename T> static inline T __ldg(const T *p) { return *p; }
static inline unsigned long long __umul64hi(unsigned long long a, unsigned long long b) {
    return static_cast<unsigned long long>((static_cast<unsigned __int128>(a) * b) >> 64);
}
"""

RESOLVE_EXPORT = r"""
extern "C" void xrsh_resolve(const double *x, const double *y, long src_h, long src_w, long src_pitch,
                             const int64_t *tile_boxes, const uint32_t *claims, double *ij, long dst_h, long dst_w,
                             int tile_h, int tile_w, double x_min, double y_min, double y_max, double x_res,
                             double y_res, int j_up) {
    xrs::IjGeom g = {};
    g.x = x; g.y = y; g.src_h = src_h; g.src_w = src_w; g.src_pitch = src_pitch;
    g.tile_boxes = tile_boxes; g.ij = ij; g.claims = const_cast<uint32_t *>(claims);
    g.dst_h = dst_h; g.dst_w = dst_w;
    g.tile_h = tile_h < dst_h ? tile_h : static_cast<int>(dst_h);   // as k1_make_geom
    g.tile_w = tile_w < dst_w ? tile_w : static_cast<int>(dst_w);
    g.ntx = static_cast<int>((dst_w + g.tile_w - 1) / g.tile_w);
    g.nty = static_cast<int>((dst_h + g.tile_h - 1) / g.tile_h);
    g.x_min = x_min; g.y_min = y_min; g.y_max = y_max; g.x_res = x_res; g.y_res = y_res;
    g.j_up = j_up ? 1 : 0;
    g.row_begin = 0; g.row_end = dst_h;
    g.magic_nqi = xrs::div_magic_of(static_cast<uint64_t>(src_w - 1));
    g.magic_tw = xrs::div_magic_of(static_cast<uint64_t>(g.tile_w));
    g.magic_th = xrs::div_magic_of(static_cast<uint64_t>(g.tile_h));
    for (long r = 0; r < dst_h; ++r) {
        const xrs::ResolveRow row = xrs::resolve_row(g, r);
        for (long c = 0; c < dst_w; ++c)
            xrs::resolve_pixel(g, row, c, claims[r * dst_w + c], ij[r * dst_w + c], ij[dst_h * dst_w + r * dst_w + c]);
    }
}
"""


def build_resolve(out_dir: str) -> str:
    """Host build of rectify_common.cuh (K1's resolve step); no library needed."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    text = open(os.path.join(CSRC, "rectify_common.cuh")).read()
    text, n = re.subn(r'#include "common.cuh"\n', "", text)
    assert n == 1, "rectify_common.cuh no longer includes common.cuh exactly once"
    text = text.replace("#pragma once\n", "")
    src = os.path.join(out_dir, "resolve_host.cpp")
    with open(src, "w") as fh:
        fh.write(RESOLVE_SHIM + text + RESOLVE_EXPORT)
    so = os.path.join(out_dir, "libxrs_resolvehost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", f"-I{os.path.join(ROOT, 'include')}", src,
           "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of rectify_common.cuh failed:\n" + res.stderr[-3000:])
    return so


def resolve(so_path: str, x, y, tile_boxes, claims, g) -> np.ndarray:
    """(2, H, W) ij image from claim words through the product's resolve_pixel; ``g``: oracle RegularGrid."""
    lib = ctypes.CDLL(so_path)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    boxes = np.ascontiguousarray(tile_boxes, dtype=np.int64)
    claims = np.ascontiguousarray(claims, dtype=np.uint32)
    ij = np.empty((2, g.height, g.width), dtype=np.float64)
    h, w = x.shape
    c_d, c_l, c_i, c_p = ctypes.c_double, ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_resolve.restype = None
    lib.xrsh_resolve.argtypes = [c_p, c_p, c_l, c_l, c_l, c_p, c_p, c_p, c_l, c_l, c_i, c_i, c_d, c_d, c_d, c_d, c_d, c_i]
    lib.xrsh_resolve(x.ctypes.data, y.ctypes.data, h, w, w, boxes.ctypes.data, claims.ctypes.data, ij.ctypes.data,
                     g.height, g.width, g.tile_h, g.tile_w, float(g.x_min), float(g.y_min), float(g.y_max),
                     float(g.x_res), float(g.y_res), int(g.is_j_axis_up))
    return ij


# ---------------------------------------------------------------------------
# K2's per-pixel arithmetic (csrc/gather_common.cuh: make_taps / interp_value)
# ---------------------------------------------------------------------------
# cast_like_numpy / cast_fill come with "xrs.h" (include/xrs_casts.h), which every shim includes
GATHER_SHIM = r"""
#include <algorithm>
#include <type_traits>
using std::min; using std::max;
"""

GATHER_EXPORT = r"""
template <typename T, int METHOD>
static void gather_one(const T *src, long n_bands, long src_h, long src_w, const double *ij, T *dst, long dst_h, long dst_w,
                       T fill) {
    for (long r = 0; r < dst_h; ++r)
        for (long c = 0; c < dst_w; ++c) {
            const long o = r * dst_w + c;
            const xrs::Taps t = xrs::make_taps<METHOD>(ij[o], ij[dst_h * dst_w + o], src_w, src_h);
            for (long b = 0; b < n_bands; ++b) {
                const T *sp = src + b * src_h * src_w;
                T out = fill;
                if (t.valid) {
                    if (METHOD == XRS_NEAREST) out = xrs::nearest_value(sp[t.j0 * src_w + t.i0]);
                    else out = xrs::cast_like_numpy<T>(xrs::interp_value<METHOD>(
                        static_cast<double>(sp[t.j0 * src_w + t.i0]), static_cast<double>(sp[t.j0 * src_w + t.i1]),
                        static_cast<double>(sp[t.j1 * src_w + t.i0]), static_cast<double>(sp[t.j1 * src_w + t.i1]), t.u, t.v));
                }
                dst[b * dst_h * dst_w + o] = out;
            }
        }
}
template <typename T>
static int gather_t(const void *src, long n_bands, long src_h, long src_w, const double *ij, void *dst, long dst_h,
                    long dst_w, int method, double fill) {
    const T f = xrs::cast_fill<T>(fill);
    const T *s = static_cast<const T *>(src);
    T *d = static_cast<T *>(dst);
    switch (method) {
    case XRS_NEAREST: gather_one<T, XRS_NEAREST>(s, n_bands, src_h, src_w, ij, d, dst_h, dst_w, f); return 0;
    case XRS_BILINEAR: gather_one<T, XRS_BILINEAR>(s, n_bands, src_h, src_w, ij, d, dst_h, dst_w, f); return 0;
    case XRS_TRIANGULAR: gather_one<T, XRS_TRIANGULAR>(s, n_bands, src_h, src_w, ij, d, dst_h, dst_w, f); return 0;
    }
    return 1;
}
extern "C" int xrsh_gather(const void *src, int dtype, long n_bands, long src_h, long src_w, const double *ij, void *dst,
                           long dst_h, long dst_w, int method, double fill) {
    switch (dtype) {
    case XRS_F32: return gather_t<float>(src, n_bands, src_h, src_w, ij, dst, dst_h, dst_w, method, fill);
    case XRS_F64: return gather_t<double>(src, n_bands, src_h, src_w, ij, dst, dst_h, dst_w, method, fill);
    case XRS_U8: return gather_t<uint8_t>(src, n_bands, src_h, src_w, ij, dst, dst_h, dst_w, method, fill);
    case XRS_I16: return gather_t<int16_t>(src, n_bands, src_h, src_w, ij, dst, dst_h, dst_w, method, fill);
    case XRS_U16: return gather_t<uint16_t>(src, n_bands, src_h, src_w, ij, dst, dst_h, dst_w, method, fill);
    case XRS_I32: return gather_t<int32_t>(src, n_bands, src_h, src_w, ij, dst, dst_h, dst_w, method, fill);
    case XRS_I64: return gather_t<int64_t>(src, n_bands, src_h, src_w, ij, dst, dst_h, dst_w, method, fill);
    case XRS_I8: return gather_t<int8_t>(src, n_bands, src_h, src_w, ij, dst, dst_h, dst_w, method, fill);
    case XRS_U32: return gather_t<uint32_t>(src, n_bands, src_h, src_w, ij, dst, dst_h, dst_w, method, fill);
    }
    return 2;
}
"""


def build_gather(out_dir: str) -> str:
    """Host build of gather_common.cuh (on top of rectify_common.cuh, which it includes)."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    rc = open(os.path.join(CSRC, "rectify_common.cuh")).read()
    rc, n = re.subn(r'#include "common.cuh"\n', "", rc)
    assert n == 1
    gc = open(os.path.join(CSRC, "gather_common.cuh")).read()
    gc, n = re.subn(r'#include "rectify_common.cuh"\n#include "tma.cuh"\n', "", gc)
    assert n == 1, "gather_common.cuh no longer includes rectify_common.cuh and tma.cuh"
    text = (rc + gc).replace("#pragma once\n", "")
    src = os.path.join(out_dir, "gather_host.cpp")
    with open(src, "w") as fh:
        fh.write(RESOLVE_SHIM + GATHER_SHIM + text + GATHER_EXPORT)
    so = os.path.join(out_dir, "libxrs_gatherhost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", f"-I{os.path.join(ROOT, 'include')}", src,
           "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of gather_common.cuh failed:\n" + res.stderr[-3000:])
    return so


def gather(so_path: str, src, ij, method: str, fill) -> np.ndarray:
    """``_compute_var_image`` through the product's make_taps / interp_value on the CPU."""
    from xcube_resampling_b200.constants import DTYPE_CODES, INTERP_CODES

    lib = ctypes.CDLL(so_path)
    src = np.asarray(src)
    squeeze = src.ndim == 2
    src3 = np.ascontiguousarray(src[None] if squeeze else src)
    ij = np.ascontiguousarray(ij, dtype=np.float64)
    bands, sh, sw = src3.shape
    _, dh, dw = ij.shape
    out = np.empty((bands, dh, dw), dtype=src3.dtype)
    c_l, c_i, c_p = ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_gather.restype = c_i
    lib.xrsh_gather.argtypes = [c_p, c_i, c_l, c_l, c_l, c_p, c_p, c_l, c_l, c_i, ctypes.c_double]
    rc = lib.xrsh_gather(src3.ctypes.data, DTYPE_CODES[src3.dtype], bands, sh, sw, ij.ctypes.data, out.ctypes.data, dh,
                         dw, INTERP_CODES[method], float(fill))
    if rc:
        raise RuntimeError(f"xrsh_gather failed ({rc})")
    return out[0] if squeeze else out


# ---------------------------------------------------------------------------
# K4 / K5 shared pieces (csrc/resample_common.cuh: numpy's summation order, scipy's output cast, order-1 taps)
# ---------------------------------------------------------------------------
RESAMPLE_SHIM = r"""
#include <limits>
#include <type_traits>
using std::isfinite; using std::floor;
"""

RESAMPLE_EXPORT = r"""
template <typename A>
static void window_sums(const A *win, int f_j, int f_i, long n, A *out) {
    for (long k = 0; k < n; ++k) {
        const A *w = win + k * f_j * f_i;
        out[k] = xrs::numpy_window_sum<A>(f_j, f_i, [&](int i) { return w[i]; });
    }
}
extern "C" void xrsh_window_sums_f32(const float *win, int f_j, int f_i, long n, float *out) { window_sums<float>(win, f_j, f_i, n, out); }
extern "C" void xrsh_window_sums_f64(const double *win, int f_j, int f_i, long n, double *out) { window_sums<double>(win, f_j, f_i, n, out); }
// out: 9 rows of n values, in the order float32, float64, uint8, int8, uint16, int16, int32, uint32, int64
extern "C" void xrsh_scipy_cast(const double *v, long n, void *out) {
    char *o = static_cast<char *>(out);
    for (long k = 0; k < n; ++k) {
        reinterpret_cast<float *>(o)[k] = xrs::scipy_cast<float>(v[k]);
        reinterpret_cast<double *>(o + 4 * n)[k] = xrs::scipy_cast<double>(v[k]);
        reinterpret_cast<uint8_t *>(o + 12 * n)[k] = xrs::scipy_cast<uint8_t>(v[k]);
        reinterpret_cast<int8_t *>(o + 13 * n)[k] = xrs::scipy_cast<int8_t>(v[k]);
        reinterpret_cast<uint16_t *>(o + 14 * n)[k] = xrs::scipy_cast<uint16_t>(v[k]);
        reinterpret_cast<int16_t *>(o + 16 * n)[k] = xrs::scipy_cast<int16_t>(v[k]);
        reinterpret_cast<int32_t *>(o + 18 * n)[k] = xrs::scipy_cast<int32_t>(v[k]);
        reinterpret_cast<uint32_t *>(o + 22 * n)[k] = xrs::scipy_cast<uint32_t>(v[k]);
        reinterpret_cast<int64_t *>(o + 26 * n)[k] = xrs::scipy_cast<int64_t>(v[k]);
    }
}
extern "C" void xrsh_axis_order1(const double *c, long n, long len, long *k0, long *k1, double *w0, double *w1,
                                 unsigned char *inside) {
    for (long k = 0; k < n; ++k) {
        const xrs::Axis1 a = xrs::axis_order1(c[k], len);
        k0[k] = a.k0; k1[k] = a.k1; w0[k] = a.w0; w1[k] = a.w1; inside[k] = a.inside ? 1 : 0;
    }
}
"""


def build_resample(out_dir: str) -> str:
    """Host build of resample_common.cuh."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    text = open(os.path.join(CSRC, "resample_common.cuh")).read()
    text, n = re.subn(r'#include "common.cuh"\n', "", text)
    assert n == 1
    text = text.replace("#pragma once\n", "").replace("#pragma unroll\n", "")
    src = os.path.join(out_dir, "resample_host.cpp")
    with open(src, "w") as fh:
        fh.write(RESOLVE_SHIM + RESAMPLE_SHIM + text + RESAMPLE_EXPORT)
    so = os.path.join(out_dir, "libxrs_resamplehost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", f"-I{os.path.join(ROOT, 'include')}", src,
           "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of resample_common.cuh failed:\n" + res.stderr[-3000:])
    return so


# ---------------------------------------------------------------------------
# K4: scipy's affine sample + the 13 numpy reducers (csrc/resample.cu, everything above the kernels)
# ---------------------------------------------------------------------------
K4_EXPORT = r"""
// what k4_affine_generic does per output pixel, as a loop nest (one slice)
template <typename T, typename OutT>
static void affine_host(const T *src, OutT *dst, const xrs::AffineGeom &g) {
    const int n = g.f_j * g.f_i;
    for (int64_t oj = 0; oj < g.dst_h; ++oj)
        for (int64_t oi = 0; oi < g.dst_w; ++oi) {
            OutT *out = dst + oj * g.dst_w + oi;
            if (n == 1) {
                *out = static_cast<OutT>(xrs::affine_sample<T>(src, nullptr, oj, oi, g));
                continue;
            }
            T w[xrs::RS_MAX_WINDOW];
            for (int a = 0; a < g.f_j; ++a)
                for (int b = 0; b < g.f_i; ++b)
                    w[a * g.f_i + b] = xrs::affine_sample<T>(src, nullptr, oj * g.f_j + a, oi * g.f_i + b, g);
            *out = xrs::reduce_window<T, OutT>(w, g.f_j, g.f_i, g.agg);
        }
}
template <typename T>
static int affine_t(const void *src, void *dst, const xrs::AffineGeom &g, int out_i64) {
    if (out_i64) affine_host<T, int64_t>(static_cast<const T *>(src), static_cast<int64_t *>(dst), g);
    else affine_host<T, T>(static_cast<const T *>(src), static_cast<T *>(dst), g);
    return 0;
}
extern "C" int xrsh_affine(const void *src, void *dst, int dtype, long src_h, long src_w, long dst_h, long dst_w,
                           double j_scale, double j_off, double i_scale, double i_off, int order, double cval, int agg,
                           int f_j, int f_i, int out_i64) {
    if (f_j * f_i > xrs::RS_MAX_WINDOW) return 3;
    xrs::AffineGeom g = {};
    g.n_slices = 1; g.src_h = src_h; g.src_w = src_w; g.src_pitch = src_w; g.src_slice_stride = src_h * src_w;
    g.dst_h = dst_h; g.dst_w = dst_w; g.j_scale = j_scale; g.j_off = j_off; g.i_scale = i_scale; g.i_off = i_off;
    g.cval = cval; g.order = order; g.agg = agg; g.f_j = f_j; g.f_i = f_i; g.slice_blend = 0;
    switch (dtype) {
    case XRS_F32: return affine_t<float>(src, dst, g, out_i64);
    case XRS_F64: return affine_t<double>(src, dst, g, out_i64);
    case XRS_U8: return affine_t<uint8_t>(src, dst, g, out_i64);
    case XRS_I16: return affine_t<int16_t>(src, dst, g, out_i64);
    case XRS_U16: return affine_t<uint16_t>(src, dst, g, out_i64);
    case XRS_I32: return affine_t<int32_t>(src, dst, g, out_i64);
    }
    return 2;
}
"""


def build_k4(out_dir: str) -> str:
    """Host build of resample_common.cuh + the device helpers of resample.cu (affine_sample, reduce_window)."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    common = open(os.path.join(CSRC, "resample_common.cuh")).read()
    common, n = re.subn(r'#include "common.cuh"\n', "", common)
    assert n == 1
    cu = open(os.path.join(CSRC, "resample.cu")).read()
    start = cu.index('#include "resample_common.cuh"\n') + len('#include "resample_common.cuh"\n')
    end = cu.index("// generic kernel: one thread per output pixel and slice")
    end = cu.rindex("// ----", 0, end)  # the rule above the section title
    helpers = cu[start:end] + "\n}  // namespace xrs\n"
    text = (common + helpers).replace("#pragma once\n", "").replace("#pragma unroll\n", "").replace("__restrict__", "")
    src = os.path.join(out_dir, "k4_host.cpp")
    with open(src, "w") as fh:
        fh.write(RESOLVE_SHIM + RESAMPLE_SHIM + "using std::fabs; using std::sqrt; using std::rint;\n" + text + K4_EXPORT)
    so = os.path.join(out_dir, "libxrs_k4host.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", f"-I{os.path.join(ROOT, 'include')}", src,
           "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of resample.cu's helpers failed:\n" + res.stderr[-4000:])
    return so


def affine(so_path: str, src, out_hw, scale_ji=(1.0, 1.0), offset_ji=(0.0, 0.0), order=0, cval=0.0, agg="mean",
           factors=(1, 1)) -> np.ndarray:
    """One (h, w) image through the product's affine_sample + reduce_window on the CPU (the loop nest of
    k4_affine_generic); output dtype as the library chooses it (int64 for mode / count / integer sum, prod)."""
    from xcube_resampling_b200.constants import AGG_CODES, DTYPE_CODES

    lib = ctypes.CDLL(so_path)
    src = np.ascontiguousarray(src)
    is_float = src.dtype.kind == "f"
    f_j, f_i = int(factors[0]), int(factors[1])
    i64 = f_j * f_i > 1 and (agg in ("mode", "count") or (not is_float and agg in ("sum", "prod")))
    out = np.empty((int(out_hw[0]), int(out_hw[1])), dtype=np.int64 if i64 else src.dtype)
    c_d, c_l, c_i, c_p = ctypes.c_double, ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_affine.restype = c_i
    lib.xrsh_affine.argtypes = [c_p, c_p, c_i, c_l, c_l, c_l, c_l, c_d, c_d, c_d, c_d, c_i, c_d, c_i, c_i, c_i, c_i]
    rc = lib.xrsh_affine(src.ctypes.data, out.ctypes.data, DTYPE_CODES[src.dtype], src.shape[0], src.shape[1], out.shape[0],
                         out.shape[1], float(scale_ji[0]), float(offset_ji[0]), float(scale_ji[1]), float(offset_ji[1]),
                         int(order), float(cval), AGG_CODES[agg], f_j, f_i, int(i64))
    if rc:
        raise RuntimeError(f"xrsh_affine failed ({rc})")
    return out


# ---------------------------------------------------------------------------
# K5: the reducers of the streaming kernels on register windows (csrc/resample_fast.cu: bitonic network,
# reduce_simple, reduce_sort)
# ---------------------------------------------------------------------------
K5_EXPORT = r"""
template <typename T, typename OutT, int F>
static void fast_host(const T *src, long src_w, OutT *dst, long dst_h, long dst_w, int agg) {
    const bool sort = agg == XRS_AGG_MEDIAN || agg == XRS_AGG_MODE;   // CLASS_SORT of k5_window_reduce
    for (long oj = 0; oj < dst_h; ++oj)
        for (long oi = 0; oi < dst_w; ++oi) {
            T w[F * F];
            for (int a = 0; a < F; ++a)
                for (int b = 0; b < F; ++b) w[a * F + b] = src[(oj * F + a) * src_w + oi * F + b];
            dst[oj * dst_w + oi] = sort ? xrs::reduce_sort<T, OutT, F>(w, agg) : xrs::reduce_simple<T, OutT, F>(w, agg);
        }
}
template <typename T, int F>
static void fast_f(const void *src, long src_w, void *dst, long dst_h, long dst_w, int agg, int out_i64) {
    if (out_i64) fast_host<T, int64_t, F>(static_cast<const T *>(src), src_w, static_cast<int64_t *>(dst), dst_h, dst_w, agg);
    else fast_host<T, T, F>(static_cast<const T *>(src), src_w, static_cast<T *>(dst), dst_h, dst_w, agg);
}
template <typename T>
static int fast_t(const void *src, long src_w, void *dst, long dst_h, long dst_w, int f, int agg, int out_i64) {
    switch (f) {
    case 2: fast_f<T, 2>(src, src_w, dst, dst_h, dst_w, agg, out_i64); return 0;
    case 4: fast_f<T, 4>(src, src_w, dst, dst_h, dst_w, agg, out_i64); return 0;
    case 8: fast_f<T, 8>(src, src_w, dst, dst_h, dst_w, agg, out_i64); return 0;
    }
    return 3;
}
extern "C" int xrsh_fast_reduce(const void *src, int dtype, long src_w, void *dst, long dst_h, long dst_w, int f, int agg,
                                int out_i64) {
    switch (dtype) {
    case XRS_F32: return fast_t<float>(src, src_w, dst, dst_h, dst_w, f, agg, out_i64);
    case XRS_F64: return fast_t<double>(src, src_w, dst, dst_h, dst_w, f, agg, out_i64);
    case XRS_U8: return fast_t<uint8_t>(src, src_w, dst, dst_h, dst_w, f, agg, out_i64);
    case XRS_I16: return fast_t<int16_t>(src, src_w, dst, dst_h, dst_w, f, agg, out_i64);
    case XRS_U16: return fast_t<uint16_t>(src, src_w, dst, dst_h, dst_w, f, agg, out_i64);
    case XRS_I32: return fast_t<int32_t>(src, src_w, dst, dst_h, dst_w, f, agg, out_i64);
    }
    return 2;
}
"""


def build_k5(out_dir: str) -> str:
    """Host build of resample_common.cuh + the register-window reducers of resample_fast.cu."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    common = open(os.path.join(CSRC, "resample_common.cuh")).read()
    common, n = re.subn(r'#include "common.cuh"\n', "", common)
    assert n == 1
    cu = open(os.path.join(CSRC, "resample_fast.cu")).read()
    start = cu.index("// ---- sorting network")
    end = cu.index("// tap k+1 of scipy's order-1 filter")
    helpers = "namespace xrs {\n" + cu[start:end] + "\n}  // namespace xrs\n"
    text = (common + helpers).replace("#pragma once\n", "").replace("#pragma unroll\n", "")
    src = os.path.join(out_dir, "k5_host.cpp")
    with open(src, "w") as fh:
        fh.write(RESOLVE_SHIM + RESAMPLE_SHIM + "using std::fabs; using std::sqrt; using std::rint;\n" + text + K5_EXPORT)
    so = os.path.join(out_dir, "libxrs_k5host.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", f"-I{os.path.join(ROOT, 'include')}", src,
           "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of resample_fast.cu's reducers failed:\n" + res.stderr[-4000:])
    return so


def fast_reduce(so_path: str, src, f: int, agg: str) -> np.ndarray:
    """Block aggregation of one (h, w) image by f x f through the streaming kernels' reducers on the CPU."""
    from xcube_resampling_b200.constants import AGG_CODES, DTYPE_CODES

    lib = ctypes.CDLL(so_path)
    src = np.ascontiguousarray(src)
    is_float = src.dtype.kind == "f"
    i64 = agg in ("mode", "count") or (not is_float and agg in ("sum", "prod"))
    out = np.empty((src.shape[0] // f, src.shape[1] // f), dtype=np.int64 if i64 else src.dtype)
    c_l, c_i, c_p = ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_fast_reduce.restype = c_i
    lib.xrsh_fast_reduce.argtypes = [c_p, c_i, c_l, c_p, c_l, c_l, c_i, c_i, c_i]
    rc = lib.xrsh_fast_reduce(src.ctypes.data, DTYPE_CODES[src.dtype], src.shape[1], out.ctypes.data, out.shape[0],
                              out.shape[1], int(f), AGG_CODES[agg], int(i64))
    if rc:
        raise RuntimeError(f"xrsh_fast_reduce failed ({rc})")
    return out


# ---------------------------------------------------------------------------
# K3: numpy's dtype semantics in the blend of _reproject_block (csrc/reproject.cu: window_index,
# diff_as_f64, cast_like_numpy, k3_blend)
# ---------------------------------------------------------------------------
K3_SHIM = r"""
#include <type_traits>
static inline float __fsub_rn(float a, float b) { return a - b; }
"""

K3_EXPORT = r"""
template <typename T, typename OUT>
static void blend_host(int method, long n, const T *v00, const T *v01, const T *v10, const T *v11, const double *u,
                       const double *v, OUT *out) {
    for (long k = 0; k < n; ++k)
        out[k] = method == XRS_BILINEAR ? xrs::k3_blend<T, OUT, XRS_BILINEAR>(v00[k], v01[k], v10[k], v11[k], u[k], v[k])
                                        : xrs::k3_blend<T, OUT, XRS_TRIANGULAR>(v00[k], v01[k], v10[k], v11[k], u[k], v[k]);
}
template <typename T>
static int blend_t(int out_f64, int method, long n, const void *a, const void *b, const void *c, const void *d,
                   const double *u, const double *v, void *out) {
    const T *p = static_cast<const T *>(a), *q = static_cast<const T *>(b), *r = static_cast<const T *>(c),
            *s = static_cast<const T *>(d);
    if (out_f64) blend_host<T, double>(method, n, p, q, r, s, u, v, static_cast<double *>(out));
    else blend_host<T, T>(method, n, p, q, r, s, u, v, static_cast<T *>(out));
    return 0;
}
extern "C" int xrsh_k3_blend(int dtype, int out_f64, int method, long n, const void *v00, const void *v01, const void *v10,
                             const void *v11, const double *u, const double *v, void *out) {
    switch (dtype) {
    case XRS_F32: return blend_t<float>(out_f64, method, n, v00, v01, v10, v11, u, v, out);
    case XRS_F64: return blend_t<double>(out_f64, method, n, v00, v01, v10, v11, u, v, out);
    case XRS_U8: return blend_t<uint8_t>(out_f64, method, n, v00, v01, v10, v11, u, v, out);
    case XRS_I8: return blend_t<int8_t>(out_f64, method, n, v00, v01, v10, v11, u, v, out);
    case XRS_U16: return blend_t<uint16_t>(out_f64, method, n, v00, v01, v10, v11, u, v, out);
    case XRS_I16: return blend_t<int16_t>(out_f64, method, n, v00, v01, v10, v11, u, v, out);
    case XRS_I32: return blend_t<int32_t>(out_f64, method, n, v00, v01, v10, v11, u, v, out);
    case XRS_U32: return blend_t<uint32_t>(out_f64, method, n, v00, v01, v10, v11, u, v, out);
    case XRS_I64: return blend_t<int64_t>(out_f64, method, n, v00, v01, v10, v11, u, v, out);
    }
    return 2;
}
extern "C" int xrsh_window_index(long k, int n, long *out) {
    int64_t kk = k;
    const bool ok = xrs::window_index(kk, n);
    *out = kk;
    return ok ? 1 : 0;
}
"""


def build_k3_blend(out_dir: str) -> str:
    """Host build of the blend helpers of reproject.cu."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    cu = open(os.path.join(CSRC, "reproject.cu")).read()
    start = cu.index("// numpy index semantics inside the reference window")
    end = cu.index("// A source tap.")
    helpers = "namespace xrs {\n" + cu[start:end] + "\n}  // namespace xrs\n"
    src = os.path.join(out_dir, "k3_blend_host.cpp")
    with open(src, "w") as fh:
        fh.write(RESOLVE_SHIM + K3_SHIM + helpers + K3_EXPORT)
    so = os.path.join(out_dir, "libxrs_k3blendhost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", f"-I{os.path.join(ROOT, 'include')}", src,
           "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of reproject.cu's blend helpers failed:\n" + res.stderr[-4000:])
    return so


def k3_blend(so_path: str, v00, v01, v10, v11, u, v, method: str, out_f64: bool) -> np.ndarray:
    from xcube_resampling_b200.constants import DTYPE_CODES, INTERP_CODES

    lib = ctypes.CDLL(so_path)
    taps = [np.ascontiguousarray(t) for t in (v00, v01, v10, v11)]
    dt = taps[0].dtype
    u = np.ascontiguousarray(u, dtype=np.float64)
    v = np.ascontiguousarray(v, dtype=np.float64)
    out = np.empty(u.shape, dtype=np.float64 if out_f64 else dt)
    c_l, c_i, c_p = ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_k3_blend.restype = c_i
    lib.xrsh_k3_blend.argtypes = [c_i, c_i, c_i, c_l] + [c_p] * 7
    rc = lib.xrsh_k3_blend(DTYPE_CODES[dt], int(out_f64), INTERP_CODES[method], u.size, *(t.ctypes.data for t in taps),
                           u.ctypes.data, v.ctypes.data, out.ctypes.data)
    if rc:
        raise RuntimeError(f"xrsh_k3_blend failed ({rc})")
    return out


# ---------------------------------------------------------------------------
# K1 as a whole (csrc/rectify_ij.cu: k1_init_claims, k1_scatter, k1_scatter_slow, k1_resolve)
# ---------------------------------------------------------------------------
# The kernels' text is compiled unchanged.  CUDA's execution model is supplied by the shim: threadIdx /
# blockIdx are thread-local variables, a WARP is 32 host threads that run the kernel body for the same
# (block, warp) in lock step -- __shfl_down_sync / __shfl_sync / __ballot_sync exchange through a shared
# array between two barrier waits -- and atomics are GCC atomics.  k1_scatter's early returns are
# warp-uniform, so every lane meets the same sequence of collectives.
K1_SHIM = r"""
#include <pthread.h>
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
#include "xrs.h"
#define __device__
#define __host__
#define __global__
#define __forceinline__ inline
#define __launch_bounds__(...)
#define __grid_constant__
typedef void *cudaStream_t;
using std::min; using std::max; using std::isfinite;
struct xrsh_dim3 { unsigned x = 0, y = 0, z = 0; };
static thread_local xrsh_dim3 threadIdx, blockIdx, blockDim, gridDim;
namespace xrs {
static inline double dadd(double a, double b) { return a + b; }
static inline double dsub(double a, double b) { return a - b; }
static inline double dmul(double a, double b) { return a * b; }
static inline double ddiv(double a, double b) { return a / b; }
template <typename T> static inline void st_stream(T *p, T v) { *p = v; }
}
template <typename T> static inline T __ldg(const T *p) { return *p; }
template <typename T> static inline T __ldcs(const T *p) { return *p; }
static inline unsigned long long __umul64hi(unsigned long long a, unsigned long long b) {
    return static_cast<unsigned long long>((static_cast<unsigned __int128>(a) * b) >> 64);
}
static inline int __double2hiint(double d) { uint64_t b; std::memcpy(&b, &d, 8); return static_cast<int>(static_cast<uint32_t>(b >> 32)); }
static inline int __double2int_rd(double d) { return static_cast<int>(std::floor(d)); }
static inline int __popc(unsigned v) { return __builtin_popcount(v); }
static inline void __syncthreads() {}
struct uint4 { unsigned x, y, z, w; };
static inline uint4 make_uint4(unsigned x, unsigned y, unsigned z, unsigned w) { return uint4{x, y, z, w}; }
template <typename T> static inline T atomicMin(T *p, T v) {
    T old = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (v < old && !__atomic_compare_exchange_n(p, &old, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
    return old;
}
template <typename T> static inline T atomicMax(T *p, T v) {
    T old = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (v > old && !__atomic_compare_exchange_n(p, &old, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
    return old;
}
static inline unsigned atomicAdd(unsigned *p, unsigned v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
// one warp = 32 host threads in lock step
struct XrshWarp { pthread_barrier_t bar; double d[32]; long long i[32]; };
static XrshWarp xrsh_warp;
static thread_local int xrsh_lane = 0;
static thread_local bool xrsh_in_warp = false;
static inline void xrsh_sync() { pthread_barrier_wait(&xrsh_warp.bar); }
static inline double __shfl_down_sync(unsigned, double v, int delta) {
    xrsh_warp.d[xrsh_lane] = v; xrsh_sync();
    const double r = xrsh_lane + delta < 32 ? xrsh_warp.d[xrsh_lane + delta] : v; xrsh_sync();
    return r;
}
static inline int __shfl_down_sync(unsigned, int v, int delta) {
    xrsh_warp.i[xrsh_lane] = v; xrsh_sync();
    const int r = xrsh_lane + delta < 32 ? static_cast<int>(xrsh_warp.i[xrsh_lane + delta]) : v; xrsh_sync();
    return r;
}
static inline unsigned __shfl_sync(unsigned, unsigned v, int src) {
    xrsh_warp.i[xrsh_lane] = v; xrsh_sync();
    const unsigned r = static_cast<unsigned>(xrsh_warp.i[src]); xrsh_sync();
    return r;
}
static inline unsigned __ballot_sync(unsigned, bool p) {
    xrsh_warp.i[xrsh_lane] = p ? 1 : 0; xrsh_sync();
    unsigned m = 0;
    for (int k = 0; k < 32; ++k) m |= static_cast<unsigned>(xrsh_warp.i[k]) << k;
    xrsh_sync();
    return m;
}
"""

K1_EXPORT = r"""
namespace {
struct XrshJob { xrs::IjGeom g; unsigned gx, gy; };
struct XrshLane { int lane; const XrshJob *job; };
void *xrsh_lane_main(void *p) {
    const XrshLane *a = static_cast<const XrshLane *>(p);
    xrsh_lane = a->lane;
    blockDim.x = xrs::K1S_WARPS * 32; blockDim.y = blockDim.z = 1;
    gridDim.x = a->job->gx; gridDim.y = a->job->gy; gridDim.z = 1;
    for (unsigned by = 0; by < a->job->gy; ++by)
        for (unsigned bx = 0; bx < a->job->gx; ++bx)
            for (int w = 0; w < xrs::K1S_WARPS; ++w) {
                blockIdx.x = bx; blockIdx.y = by; threadIdx.x = static_cast<unsigned>(w * 32 + a->lane);
                xrs::k1_scatter(a->job->g);
            }
    return nullptr;
}
}

// xrs_rectify_ij (csrc/rectify_ij.cu) on the host: the geometry of k1_make_geom, then the four kernels in
// launch order with the launch shapes of k1_enqueue_claims / xrs_rectify_ij.  ij: (2, row_end - row_begin, dst_w);
// claims_out: (row_end - row_begin, dst_w); counts: [queued quads]
extern "C" int xrsh_k1(const double *x, const double *y, long src_h, long src_w, long src_pitch, const int64_t *tile_boxes,
                       double *ij, long dst_h, long dst_w, int tile_h, int tile_w, double x_min, double y_min,
                       double y_max, double x_res, double y_res, int j_up, double uv_delta, long row_begin, long row_end,
                       const int32_t *fp_cols, uint32_t *claims_out, unsigned *counts) {
    using namespace xrs;
    const long n_rows = row_end - row_begin, n_quads = (src_h - 1) * (src_w - 1);
    const long n_rb = (src_h - 1 + K1S_ROWS - 1) / K1S_ROWS;
    std::vector<uint32_t> claims(static_cast<size_t>(n_rows * dst_w), K1_NOCLAIM);
    std::vector<uint32_t> queue(static_cast<size_t>(n_quads + 4 + 2 * n_rb), 0u);
    IjGeom g = {};
    g.x = x; g.y = y; g.src_h = src_h; g.src_w = src_w; g.src_pitch = src_pitch;
    g.tile_boxes = tile_boxes; g.ij = ij; g.claims = claims.data();
    g.dst_h = dst_h; g.dst_w = dst_w;
    g.tile_h = tile_h < dst_h ? tile_h : static_cast<int>(dst_h);
    g.tile_w = tile_w < dst_w ? tile_w : static_cast<int>(dst_w);
    g.ntx = static_cast<int>((dst_w + g.tile_w - 1) / g.tile_w);
    g.nty = static_cast<int>((dst_h + g.tile_h - 1) / g.tile_h);
    g.x_min = x_min; g.y_min = y_min; g.y_max = y_max; g.x_res = x_res; g.y_res = y_res;
    g.j_up = j_up ? 1 : 0; g.uv_delta = uv_delta;
    g.row_begin = row_begin; g.row_end = row_end;
    g.fp_cols = fp_cols;
    g.magic_nqi = div_magic_of(static_cast<uint64_t>(src_w - 1));
    g.magic_tw = div_magic_of(static_cast<uint64_t>(g.tile_w));
    g.magic_th = div_magic_of(static_cast<uint64_t>(g.tile_h));
    g.slow_list = queue.data();
    g.slow_count = queue.data() + n_quads;
    // k1_init_claims: the claim words are set above; block 0 (one thread) derives the quad row / column ranges
    blockIdx = xrsh_dim3(); threadIdx = xrsh_dim3(); blockDim = xrsh_dim3(); blockDim.x = 1; gridDim = xrsh_dim3(); gridDim.x = 1;
    k1_init_claims(reinterpret_cast<uint4 *>(claims.data()), 0, g.slow_count, g);
    // k1_scatter: 32 lanes in lock step over every (block, warp)
    XrshJob job{g, static_cast<unsigned>(((src_w - 1 + 30) / 31 + K1S_WARPS - 1) / K1S_WARPS), static_cast<unsigned>(n_rb)};
    pthread_barrier_init(&xrsh_warp.bar, nullptr, 32);
    pthread_t th[32];
    XrshLane lanes[32];
    for (int l = 0; l < 32; ++l) {
        lanes[l] = XrshLane{l, &job};
        if (pthread_create(&th[l], nullptr, xrsh_lane_main, &lanes[l]) != 0) return 1;
    }
    for (int l = 0; l < 32; ++l) pthread_join(th[l], nullptr);
    pthread_barrier_destroy(&xrsh_warp.bar);
    counts[0] = *g.slow_count;
    // k1_scatter_slow: one thread strides over the queue
    blockIdx = xrsh_dim3(); threadIdx = xrsh_dim3(); blockDim.x = 1; gridDim.x = 1;
    k1_scatter_slow(g);
    std::memcpy(claims_out, claims.data(), claims.size() * sizeof(uint32_t));
    // k1_resolve: grid (ceil(dst_w / (K1R_THREADS * K1R_PX)), n_rows) x K1R_THREADS
    blockDim.x = K1R_THREADS;
    gridDim.x = static_cast<unsigned>((dst_w + K1R_THREADS * K1R_PX - 1) / (K1R_THREADS * K1R_PX));
    gridDim.y = static_cast<unsigned>(n_rows);
    for (unsigned by = 0; by < gridDim.y; ++by)
        for (unsigned bx = 0; bx < gridDim.x; ++bx)
            for (unsigned t = 0; t < static_cast<unsigned>(K1R_THREADS); ++t) {
                blockIdx.x = bx; blockIdx.y = by; threadIdx.x = t;
                k1_resolve(g);
            }
    return 0;
}
"""


def build_k1(out_dir: str) -> str:
    """Host build of rectify_common.cuh + the kernels of rectify_ij.cu (everything above its host launch code)."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    common = open(os.path.join(CSRC, "rectify_common.cuh")).read()
    common, n = re.subn(r'#include "common.cuh"\n', "", common)
    assert n == 1, "rectify_common.cuh no longer includes common.cuh exactly once"
    common = common.replace("#pragma once\n", "")
    text = open(os.path.join(CSRC, "rectify_ij.cu")).read()
    text, n = re.subn(r'#include "rectify_common.cuh"\n', "", text)
    assert n == 1, "rectify_ij.cu no longer includes rectify_common.cuh exactly once"
    cut = text.find("static int64_t claims_bytes_of")
    assert cut > 0 and "<<<" not in text[:cut] and "k1_resolve(const" in text[:cut], "layout of rectify_ij.cu changed"
    kernels = text[:cut] + "\n}  // namespace xrs\n"
    src = os.path.join(out_dir, "k1_host.cpp")
    with open(src, "w") as fh:
        fh.write(K1_SHIM + common + kernels + K1_EXPORT)
    so = os.path.join(out_dir, "libxrs_k1host.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of rectify_ij.cu failed:\n" + res.stderr[-4000:])
    return so


def k1(so_path: str, x, y, tile_boxes, g, uv_delta: float = 1e-3, rows=None, fp_cols=None):
    """``xrs_rectify_ij`` through the host build: ``(ij (2, rows, W), claims (rows, W) uint32, queued quads)``;
    ``g``: oracle RegularGrid, ``rows``: target row range (default all)."""
    lib = ctypes.CDLL(so_path)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    boxes = np.ascontiguousarray(tile_boxes, dtype=np.int64)
    r0, r1 = rows if rows is not None else (0, g.height)
    ij = np.empty((2, r1 - r0, g.width), dtype=np.float64)
    claims = np.empty((r1 - r0, g.width), dtype=np.uint32)
    counts = np.zeros(1, dtype=np.uint32)
    fp = None if fp_cols is None else np.ascontiguousarray(fp_cols, dtype=np.int32)
    h, w = x.shape
    c_d, c_l, c_i, c_p = ctypes.c_double, ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_k1.restype = c_i
    lib.xrsh_k1.argtypes = [c_p, c_p, c_l, c_l, c_l, c_p, c_p, c_l, c_l, c_i, c_i, c_d, c_d, c_d, c_d, c_d, c_i, c_d, c_l,
                            c_l, c_p, c_p, c_p]
    rc = lib.xrsh_k1(x.ctypes.data, y.ctypes.data, h, w, w, boxes.ctypes.data, ij.ctypes.data, g.height, g.width,
                     g.tile_h, g.tile_w, float(g.x_min), float(g.y_min), float(g.y_max), float(g.x_res), float(g.y_res),
                     int(g.is_j_axis_up), float(uv_delta), r0, r1, None if fp is None else fp.ctypes.data,
                     claims.ctypes.data, counts.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"xrsh_k1 failed ({rc})")
    return ij, claims, int(counts[0])


# ---------------------------------------------------------------------------
# K0 (csrc/rectify.cu: k0_tile_windows in its three forms, k0_init_table, k0_finalize, k0_fold_minform,
# k0_finalize_minform)
# ---------------------------------------------------------------------------
# A thread BLOCK is K0_THREADS host threads: __syncthreads is a barrier over all of them, dynamic shared
# memory a static array, __match_any_sync a full-warp exchange (two barrier waits of the warp's 32 threads),
# and the __reduce_*_sync calls that only the lanes of a peer group execute are group collectives built on
# per-lane generation counters (a lane publishes its value under generation n, readers wait until every peer
# of the mask has reached n; values are double-buffered by the generation's parity, and a lane cannot get two
# generations ahead of a peer that is still reading).
K0_SHIM = r"""
#include <pthread.h>
#include <sched.h>
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
#include "xrs.h"
#define __device__
#define __host__
#define __global__
#define __forceinline__ inline
#define __launch_bounds__(...)
#define __shared__
#define __align__(n) __attribute__((aligned(n)))
typedef void *cudaStream_t;
using std::min; using std::max;
struct xrsh_dim3 { unsigned x = 0, y = 0, z = 0; };
static thread_local xrsh_dim3 threadIdx, blockIdx, blockDim, gridDim;
struct int4 { int x, y, z, w; };
static inline int4 make_int4(int x, int y, int z, int w) { return int4{x, y, z, w}; }
namespace xrs {
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
template <typename T> static inline T ld_stream(const T *p) { return *p; }
alignas(16) unsigned char k0_smem[1 << 18];
}
template <typename T> static inline T atomicMin(T *p, T v) {
    T old = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (v < old && !__atomic_compare_exchange_n(p, &old, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
    return old;
}
template <typename T> static inline T atomicMax(T *p, T v) {
    T old = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (v > old && !__atomic_compare_exchange_n(p, &old, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
    return old;
}
static inline int __ffs(unsigned v) { return __builtin_ffs(static_cast<int>(v)); }
constexpr int XRSH_MAX_WARPS = 32;
struct XrshWarp { pthread_barrier_t bar; unsigned long long u[32]; int val[2][32]; unsigned gen[32]; };
static XrshWarp xrsh_warps[XRSH_MAX_WARPS];
static pthread_barrier_t xrsh_block_bar;
static thread_local unsigned xrsh_gen = 0;
static inline XrshWarp &xrsh_w() { return xrsh_warps[threadIdx.x >> 5]; }
static inline int xrsh_l() { return static_cast<int>(threadIdx.x & 31); }
static inline void __syncthreads() { pthread_barrier_wait(&xrsh_block_bar); }
static inline unsigned __match_any_sync(unsigned, unsigned long long key) {
    XrshWarp &w = xrsh_w();
    const int l = xrsh_l();
    w.u[l] = key;
    pthread_barrier_wait(&w.bar);
    unsigned m = 0;
    for (int k = 0; k < 32; ++k) m |= (w.u[k] == key ? 1u : 0u) << k;
    __atomic_store_n(&w.gen[l], 0u, __ATOMIC_RELEASE);  // a new round of group collectives starts at generation 0
    xrsh_gen = 0;
    pthread_barrier_wait(&w.bar);
    return m;
}
template <typename Op> static inline int xrsh_group_reduce(unsigned mask, int v, Op op) {
    XrshWarp &w = xrsh_w();
    const int l = xrsh_l();
    const unsigned my = ++xrsh_gen;
    w.val[my & 1][l] = v;
    __atomic_store_n(&w.gen[l], my, __ATOMIC_RELEASE);
    int r = v;
    for (int k = 0; k < 32; ++k) {
        if (!((mask >> k) & 1u) || k == l) continue;
        while (__atomic_load_n(&w.gen[k], __ATOMIC_ACQUIRE) < my) sched_yield();
        r = op(r, w.val[my & 1][k]);
    }
    return r;
}
static inline int __reduce_min_sync(unsigned mask, int v) { return xrsh_group_reduce(mask, v, [](int a, int b) { return a < b ? a : b; }); }
static inline int __reduce_max_sync(unsigned mask, int v) { return xrsh_group_reduce(mask, v, [](int a, int b) { return a > b ? a : b; }); }
"""

K0_EXPORT = r"""
namespace {
struct XrshK0Job {
    const double *x, *y; int64_t h, w, pitch; const double *x_lo, *x_hi; int ntx; const double *y_lo, *y_hi; int nty;
    int4 *table; int j_offset, rows_per_block, form; unsigned blocks;
};
struct XrshK0Thread { unsigned tid; const XrshK0Job *job; };
void *xrsh_k0_thread(void *p) {
    const XrshK0Thread *a = static_cast<const XrshK0Thread *>(p);
    const XrshK0Job &j = *a->job;
    threadIdx.x = a->tid; blockDim.x = xrs::K0_THREADS; gridDim.x = j.blocks;
    for (unsigned b = 0; b < j.blocks; ++b) {
        blockIdx.x = b;
        if (j.form == 0) xrs::k0_tile_windows<true, false>(j.x, j.y, j.h, j.w, j.pitch, j.x_lo, j.x_hi, j.ntx, j.y_lo, j.y_hi, j.nty, j.table, j.j_offset, j.rows_per_block);
        else if (j.form == 1) xrs::k0_tile_windows<false, false>(j.x, j.y, j.h, j.w, j.pitch, j.x_lo, j.x_hi, j.ntx, j.y_lo, j.y_hi, j.nty, j.table, j.j_offset, j.rows_per_block);
        else xrs::k0_tile_windows<true, true>(j.x, j.y, j.h, j.w, j.pitch, j.x_lo, j.x_hi, j.ntx, j.y_lo, j.y_hi, j.nty, j.table, j.j_offset, j.rows_per_block);
        __syncthreads();  // the next block re-initialises the shared table
    }
    return nullptr;
}
template <typename F> void xrsh_per_thread(int n, F f) {  // <<<ceil(n / 256), 256>>> of a kernel without collectives
    blockDim.x = 256; gridDim.x = static_cast<unsigned>((n + 255) / 256);
    for (unsigned b = 0; b < gridDim.x; ++b)
        for (unsigned t = 0; t < 256; ++t) { blockIdx.x = b; threadIdx.x = t; f(); }
}
}

// form 0: xrs_tile_src_bboxes with the table in shared memory; 1: table in global memory; 2: the slab scan
// of xrs_tile_src_bboxes_partial (slabs of `slab_rows` rows straight into a min-form table) followed by
// xrs_tile_src_bboxes_finalize; 3: slabs through the global-table kernel + k0_fold_minform, then finalize
extern "C" int xrsh_k0(const double *x, const double *y, long h, long w, long pitch, const double *x_lo,
                       const double *x_hi, int ntx, const double *y_lo, const double *y_hi, int nty, int ij_border,
                       int form, long slab_rows, int64_t *out_boxes) {
    using namespace xrs;
    const int n_tiles = ntx * nty;
    std::vector<int4> table(static_cast<size_t>(n_tiles));
    std::vector<int32_t> minform(static_cast<size_t>(4 * n_tiles), INT32_MAX);
    pthread_barrier_init(&xrsh_block_bar, nullptr, K0_THREADS);
    for (int k = 0; k < K0_THREADS / 32; ++k) pthread_barrier_init(&xrsh_warps[k].bar, nullptr, 32);
    auto scan = [&](const double *sx, const double *sy, long sh, long joff, int kform, int4 *tab) {
        const int rows = sh >= 2048 ? K0_ROWS : 8;
        XrshK0Job job{sx, sy, sh, w, pitch, x_lo, x_hi, ntx, y_lo, y_hi, nty, tab, static_cast<int>(joff), rows, kform,
                      static_cast<unsigned>(ceil_div(w, K0_THREADS) * ceil_div(sh, rows))};
        std::vector<pthread_t> th(K0_THREADS);
        std::vector<XrshK0Thread> args(K0_THREADS);
        for (int t = 0; t < K0_THREADS; ++t) {
            args[t] = XrshK0Thread{static_cast<unsigned>(t), &job};
            pthread_create(&th[t], nullptr, xrsh_k0_thread, &args[t]);
        }
        for (int t = 0; t < K0_THREADS; ++t) pthread_join(th[t], nullptr);
    };
    if (form == 0 || form == 1) {
        int4 *tab = table.data();
        xrsh_per_thread(n_tiles, [&] { k0_init_table(tab, n_tiles); });
        scan(x, y, h, 0, form, tab);
        xrsh_per_thread(n_tiles, [&] { k0_finalize(tab, n_tiles, ij_border, w, h, out_boxes); });
    } else {
        for (long j0 = 0; j0 < h; j0 += slab_rows) {
            const long sh = std::min(slab_rows, h - j0);
            if (form == 2) {
                scan(x + j0 * pitch, y + j0 * pitch, sh, j0, 2, reinterpret_cast<int4 *>(minform.data()));
            } else {
                int4 *tab = table.data();
                xrsh_per_thread(n_tiles, [&] { k0_init_table(tab, n_tiles); });
                scan(x + j0 * pitch, y + j0 * pitch, sh, j0, 1, tab);
                int32_t *mf = minform.data();
                xrsh_per_thread(n_tiles, [&] { k0_fold_minform(tab, n_tiles, mf); });
            }
        }
        const int32_t *mf = minform.data();
        xrsh_per_thread(n_tiles, [&] { k0_finalize_minform(mf, n_tiles, ij_border, w, h, out_boxes); });
    }
    pthread_barrier_destroy(&xrsh_block_bar);
    for (int k = 0; k < K0_THREADS / 32; ++k) pthread_barrier_destroy(&xrsh_warps[k].bar);
    return 0;
}
"""


def build_k0(out_dir: str) -> str:
    """Host build of the kernels of rectify.cu (everything above its host launch code)."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    text = open(os.path.join(CSRC, "rectify.cu")).read()
    text, n = re.subn(r'#include "common.cuh"\n', "", text)
    assert n == 1, "rectify.cu no longer includes common.cuh exactly once"
    cut = text.find("using namespace xrs;")
    assert cut > 0 and "<<<" not in text[:cut] and "k0_finalize_minform(const" in text[:cut], "layout of rectify.cu changed"
    src = os.path.join(out_dir, "k0_host.cpp")
    with open(src, "w") as fh:
        fh.write(K0_SHIM + text[:cut] + K0_EXPORT)
    so = os.path.join(out_dir, "libxrs_k0host.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of rectify.cu failed:\n" + res.stderr[-4000:])
    return so


def k0(so_path: str, x, y, x_lo, x_hi, y_lo, y_hi, ij_border: int = 1, form: int = 0, slab_rows: int = 0) -> np.ndarray:
    """(n_tiles, 4) int64 source windows through the host build of K0; ``form`` as in ``xrsh_k0``."""
    lib = ctypes.CDLL(so_path)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    axes = [np.ascontiguousarray(a, dtype=np.float64) for a in (x_lo, x_hi, y_lo, y_hi)]
    ntx, nty = len(axes[0]), len(axes[2])
    out = np.empty((ntx * nty, 4), dtype=np.int64)
    h, w = x.shape
    c_l, c_i, c_p = ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_k0.restype = c_i
    lib.xrsh_k0.argtypes = [c_p, c_p, c_l, c_l, c_l, c_p, c_p, c_i, c_p, c_p, c_i, c_i, c_i, c_l, c_p]
    rc = lib.xrsh_k0(x.ctypes.data, y.ctypes.data, h, w, w, axes[0].ctypes.data, axes[1].ctypes.data, ntx,
                     axes[2].ctypes.data, axes[3].ctypes.data, nty, int(ij_border), int(form), int(slab_rows or h),
                     out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"xrsh_k0 failed ({rc})")
    return out


# ---------------------------------------------------------------------------
# KB (csrc/bands.cu: kb_fill_i32, kb_quad_footprints) -- the row bands' ragged quad footprints
# ---------------------------------------------------------------------------
KB_SHIM = K0_SHIM.replace("#define __shared__\n", "#define __shared__ static\n") + r"""
namespace xrs {
static inline double dadd(double a, double b) { return a + b; }
static inline double dsub(double a, double b) { return a - b; }
static inline double dmul(double a, double b) { return a * b; }
static inline double ddiv(double a, double b) { return a / b; }
}
template <typename T> static inline T __ldg(const T *p) { return *p; }
static inline unsigned long long __umul64hi(unsigned long long a, unsigned long long b) {
    return static_cast<unsigned long long>((static_cast<unsigned __int128>(a) * b) >> 64);
}
static inline int __ffsll(long long v) { return __builtin_ffsll(v); }
static inline int __clz(unsigned v) { return v ? __builtin_clz(v) : 32; }
static inline unsigned long long __shfl_xor_sync(unsigned, unsigned long long v, int lane_mask) {
    XrshWarp &w = xrsh_w();
    const int l = xrsh_l();
    w.u[l] = v;
    pthread_barrier_wait(&w.bar);
    const unsigned long long r = w.u[l ^ lane_mask];
    pthread_barrier_wait(&w.bar);
    return r;
}
static inline unsigned __ballot_sync(unsigned, bool p) {
    XrshWarp &w = xrsh_w();
    const int l = xrsh_l();
    w.u[l] = p ? 1ull : 0ull;
    pthread_barrier_wait(&w.bar);
    unsigned m = 0;
    for (int k = 0; k < 32; ++k) m |= static_cast<unsigned>(w.u[k]) << k;
    pthread_barrier_wait(&w.bar);
    return m;
}
"""
assert "#define __shared__ static\n" in KB_SHIM

KB_EXPORT = r"""
namespace {
struct XrshKbJob {
    const double *x, *y; int64_t slab_h, src_w, pitch, j_offset; xrs::BandGrid g; const int32_t *edges; int n_bands, n_groups;
    int32_t *fp; unsigned blocks;
};
struct XrshKbThread { unsigned tid; const XrshKbJob *job; };
void *xrsh_kb_thread(void *p) {
    const XrshKbThread *a = static_cast<const XrshKbThread *>(p);
    const XrshKbJob &j = *a->job;
    threadIdx.x = a->tid; blockDim.x = xrs::KB_THREADS; gridDim.x = j.blocks;
    for (unsigned b = 0; b < j.blocks; ++b) {
        blockIdx.x = b;
        xrs::kb_quad_footprints(j.x, j.y, j.slab_h, j.src_w, j.pitch, j.j_offset, j.g, j.edges, j.n_bands, j.n_groups, j.fp);
        __syncthreads();  // the next block re-initialises the shared tables
    }
    return nullptr;
}
}

extern "C" int xrsh_quad_row_group(void) { return xrs::K1S_ROWS; }

extern "C" void xrsh_minform_init(int32_t *table, long n) {  // xrs_minform_init
    blockDim.x = 256; gridDim.x = static_cast<unsigned>((n + 255) / 256);
    for (unsigned b = 0; b < gridDim.x; ++b)
        for (unsigned t = 0; t < 256; ++t) { blockIdx.x = b; threadIdx.x = t; xrs::kb_fill_i32(table, n, INT32_MAX); }
}

// xrs_band_quad_footprints on the host (same geometry set-up and launch shape)
extern "C" int xrsh_band_quad_footprints(const double *x, const double *y, long slab_h, long src_w, long pitch, long j_offset,
                                         long src_h, long dst_h, long dst_w, double x_min, double y_min, double y_max,
                                         double x_res, double y_res, int j_up, const int32_t *band_edges, int n_bands,
                                         int32_t *fp) {
    using namespace xrs;
    if (slab_h < 2 || src_w < 2 || j_offset % K1S_ROWS != 0 || j_offset + slab_h > src_h || n_bands < 1 || n_bands > KB_MAX_BANDS) return 1;
    BandGrid g;
    g.x_min = x_min; g.y_min = y_min; g.y_max = y_max; g.inv_xr = 1.0 / x_res; g.inv_yr = 1.0 / y_res;
    g.j_up = j_up ? 1 : 0; g.dst_w = dst_w; g.dst_h = dst_h;
    XrshKbJob job{x, y, slab_h, src_w, pitch, j_offset, g, band_edges, n_bands, static_cast<int>(ceil_div(src_h - 1, K1S_ROWS)), fp,
                  static_cast<unsigned>(ceil_div(src_w - 1, KB_COLS) * ceil_div(slab_h - 1, K1S_ROWS))};
    pthread_barrier_init(&xrsh_block_bar, nullptr, KB_THREADS);
    for (int k = 0; k < KB_THREADS / 32; ++k) pthread_barrier_init(&xrsh_warps[k].bar, nullptr, 32);
    std::vector<pthread_t> th(KB_THREADS);
    std::vector<XrshKbThread> args(KB_THREADS);
    for (int t = 0; t < KB_THREADS; ++t) {
        args[t] = XrshKbThread{static_cast<unsigned>(t), &job};
        pthread_create(&th[t], nullptr, xrsh_kb_thread, &args[t]);
    }
    for (int t = 0; t < KB_THREADS; ++t) pthread_join(th[t], nullptr);
    pthread_barrier_destroy(&xrsh_block_bar);
    for (int k = 0; k < KB_THREADS / 32; ++k) pthread_barrier_destroy(&xrsh_warps[k].bar);
    return 0;
}
"""


def build_kb(out_dir: str) -> str:
    """Host build of rectify_common.cuh + the kernels of bands.cu."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    common = open(os.path.join(CSRC, "rectify_common.cuh")).read()
    common, n = re.subn(r'#include "common.cuh"\n', "", common)
    assert n == 1, "rectify_common.cuh no longer includes common.cuh exactly once"
    common = common.replace("#pragma once\n", "")
    text = open(os.path.join(CSRC, "bands.cu")).read()
    text, n = re.subn(r'#include "rectify_common.cuh"\n', "", text)
    assert n == 1, "bands.cu no longer includes rectify_common.cuh exactly once"
    cut = text.find("using namespace xrs;")
    assert cut > 0 and "<<<" not in text[:cut] and "kb_quad_footprints(const" in text[:cut], "layout of bands.cu changed"
    src = os.path.join(out_dir, "kb_host.cpp")
    with open(src, "w") as fh:
        fh.write(KB_SHIM + common + text[:cut] + KB_EXPORT)
    so = os.path.join(out_dir, "libxrs_kbhost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of bands.cu failed:\n" + res.stderr[-4000:])
    return so


def band_quad_footprints(so_path: str, x, y, g, band_edges, slabs=None) -> np.ndarray:
    """(n_bands, n_groups, 2) int32 min-form footprints through the host build of ``kb_quad_footprints``:
    ``slabs`` = list of (first vertex row, end vertex row) scanned one after the other into the same table
    (what the participants' partial scans + the MIN exchange produce); default: the whole image at once."""
    lib = ctypes.CDLL(so_path)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    h, w = x.shape
    group = lib.xrsh_quad_row_group()
    edges = np.ascontiguousarray(band_edges, dtype=np.int32)
    n_bands, n_groups = len(edges) - 1, -(-(h - 1) // group)
    fp = np.empty((n_bands, n_groups, 2), dtype=np.int32)
    c_d, c_l, c_i, c_p = ctypes.c_double, ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_minform_init.restype = None
    lib.xrsh_minform_init.argtypes = [c_p, c_l]
    lib.xrsh_minform_init(fp.ctypes.data, fp.size)
    lib.xrsh_band_quad_footprints.restype = c_i
    lib.xrsh_band_quad_footprints.argtypes = [c_p, c_p, c_l, c_l, c_l, c_l, c_l, c_l, c_l, c_d, c_d, c_d, c_d, c_d, c_i,
                                              c_p, c_i, c_p]
    for j0, j1 in (slabs or [(0, h)]):
        assert j0 % group == 0
        rc = lib.xrsh_band_quad_footprints(x.ctypes.data + j0 * w * 8, y.ctypes.data + j0 * w * 8, j1 - j0, w, w, j0, h,
                                           g.height, g.width, float(g.x_min), float(g.y_min), float(g.y_max),
                                           float(g.x_res), float(g.y_res), int(g.is_j_axis_up), edges.ctypes.data, n_bands,
                                           fp.ctypes.data)
        if rc != 0:
            raise RuntimeError(f"xrsh_band_quad_footprints refused the slab ({j0}, {j1})")
    return fp


# ---------------------------------------------------------------------------
# KC (csrc/coords.cu: kc_stats_init, kc_coords_stats, kc_lon_360)
# ---------------------------------------------------------------------------
KC_SHIM = K0_SHIM.replace("#define __shared__\n", "#define __shared__ static\n") + r"""
namespace xrs {
static inline double dadd(double a, double b) { return a + b; }
static inline double dsub(double a, double b) { return a - b; }
static inline double dmul(double a, double b) { return a * b; }
}
static inline long long __double_as_longlong(double d) { long long b; std::memcpy(&b, &d, 8); return b; }
template <typename T> static inline T atomicOr(T *p, T v) { return __atomic_fetch_or(p, v, __ATOMIC_RELAXED); }
"""

KC_EXPORT = r"""
namespace {
struct XrshKcJob { const double *x, *y; int64_t h, w, pitch; int geographic; unsigned long long *out; unsigned blocks; };
struct XrshKcThread { unsigned tid; const XrshKcJob *job; };
void *xrsh_kc_thread(void *p) {
    const XrshKcThread *a = static_cast<const XrshKcThread *>(p);
    const XrshKcJob &j = *a->job;
    threadIdx.x = a->tid; blockDim.x = xrs::KC_THREADS; gridDim.x = j.blocks;
    for (unsigned b = 0; b < j.blocks; ++b) {
        blockIdx.x = b;
        xrs::kc_coords_stats(j.x, j.y, j.h, j.w, j.pitch, j.geographic, j.out);
        __syncthreads();
    }
    return nullptr;
}
}

// xrs_coords_stats with `blocks` thread blocks (the device launch takes min(ceil(h * w / 256), 148 * 8))
extern "C" int xrsh_coords_stats(const double *x, const double *y, long h, long w, long pitch, int geographic,
                                 unsigned long long *out4, int blocks) {
    using namespace xrs;
    kc_stats_init(out4);
    XrshKcJob job{x, y, h, w, pitch, geographic ? 1 : 0, out4, static_cast<unsigned>(blocks)};
    pthread_barrier_init(&xrsh_block_bar, nullptr, KC_THREADS);
    std::vector<pthread_t> th(KC_THREADS);
    std::vector<XrshKcThread> args(KC_THREADS);
    for (int t = 0; t < KC_THREADS; ++t) {
        args[t] = XrshKcThread{static_cast<unsigned>(t), &job};
        pthread_create(&th[t], nullptr, xrsh_kc_thread, &args[t]);
    }
    for (int t = 0; t < KC_THREADS; ++t) pthread_join(th[t], nullptr);
    pthread_barrier_destroy(&xrsh_block_bar);
    return 0;
}

extern "C" void xrsh_lon_360(double *x, long h, long w, long pitch, int blocks) {
    blockDim.x = 256; gridDim.x = static_cast<unsigned>(blocks);
    for (unsigned b = 0; b < gridDim.x; ++b)
        for (unsigned t = 0; t < 256; ++t) { blockIdx.x = b; threadIdx.x = t; xrs::kc_lon_360(x, h, w, pitch); }
}
"""


def build_kc(out_dir: str) -> str:
    """Host build of the kernels of coords.cu."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    text = open(os.path.join(CSRC, "coords.cu")).read()
    text, n = re.subn(r'#include "common.cuh"\n', "", text)
    assert n == 1, "coords.cu no longer includes common.cuh exactly once"
    cut = text.find("using namespace xrs;")
    assert cut > 0 and "<<<" not in text[:cut] and "kc_lon_360(double" in text[:cut], "layout of coords.cu changed"
    src = os.path.join(out_dir, "kc_host.cpp")
    with open(src, "w") as fh:
        fh.write(KC_SHIM + text[:cut] + KC_EXPORT)
    so = os.path.join(out_dir, "libxrs_kchost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of coords.cu failed:\n" + res.stderr[-4000:])
    return so


def coords_stats(so_path: str, x, y, geographic: bool, blocks: int = 3):
    """``(any(x > 180), smallest positive cell area, largest)`` through the host build of ``kc_coords_stats``
    (areas ``nan`` when no cell has a positive area)."""
    lib = ctypes.CDLL(so_path)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    h, w = x.shape
    out = np.zeros(4, dtype=np.uint64)
    c_l, c_i, c_p = ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_coords_stats.restype = c_i
    lib.xrsh_coords_stats.argtypes = [c_p, c_p, c_l, c_l, c_l, c_i, c_p, c_i]
    lib.xrsh_coords_stats(x.ctypes.data, y.ctypes.data, h, w, w, int(bool(geographic)), out.ctypes.data, int(blocks))
    areas = out[1:3].copy().view(np.float64)
    return (bool(out[0]), float(areas[0]) if out[1] != np.uint64(0xFFFFFFFFFFFFFFFF) else float("nan"),
            float(areas[1]) if out[2] != 0 else float("nan"))


def lon_360(so_path: str, x, blocks: int = 2) -> np.ndarray:
    lib = ctypes.CDLL(so_path)
    x = np.array(x, dtype=np.float64, order="C")
    lib.xrsh_lon_360.restype = None
    lib.xrsh_lon_360.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_long, ctypes.c_long, ctypes.c_int]
    lib.xrsh_lon_360(x.ctypes.data, x.shape[0], x.shape[1], x.shape[1], int(blocks))
    return x


# ---------------------------------------------------------------------------
# K2 as kernels (csrc/gather.cu: k2_gather_staged / k2_gather_direct; csrc/gather_dual.cu: k2_gather_dual)
# ---------------------------------------------------------------------------
# The kernels' text is compiled unchanged.  What the hardware supplies is written out in the shim: a
# CUtensorMap is a plain descriptor (base, extents, pitch, box), `tma_load_2d` copies the box into "shared
# memory" (elements outside the tensor read as zero, as the TMA unit fills them) and then completes the
# mbarrier's phase; an mbarrier is a counter of completed phases whose parity `mbar_wait` polls; the fences are
# no-ops; `elem_ptr` is pointer arithmetic.  A CTA is K2S_THREADS host threads.
XRSH_DISPATCH = r"""
// XRS_DISPATCH_DTYPE of common.cuh without its error path
#define XRSH_DISPATCH_DTYPE(dtype, T, ...)                         \
    switch (dtype) {                                               \
    case XRS_F32: { using T = float; __VA_ARGS__; break; }         \
    case XRS_F64: { using T = double; __VA_ARGS__; break; }        \
    case XRS_U8: { using T = uint8_t; __VA_ARGS__; break; }        \
    case XRS_I8: { using T = int8_t; __VA_ARGS__; break; }         \
    case XRS_U16: { using T = uint16_t; __VA_ARGS__; break; }      \
    case XRS_I16: { using T = int16_t; __VA_ARGS__; break; }       \
    case XRS_I32: { using T = int32_t; __VA_ARGS__; break; }       \
    case XRS_U32: { using T = uint32_t; __VA_ARGS__; break; }      \
    case XRS_I64: { using T = int64_t; __VA_ARGS__; break; }       \
    }
"""

K2_SHIM = XRSH_DISPATCH + K0_SHIM + GATHER_SHIM.replace("#include <algorithm>\n", "").replace("using std::min; using std::max;\n", "") + r"""
#include <functional>
#define __grid_constant__
namespace xrs {
static inline double dadd(double a, double b) { return a + b; }
static inline double dsub(double a, double b) { return a - b; }
static inline double dmul(double a, double b) { return a * b; }
static inline double ddiv(double a, double b) { return a / b; }
template <typename T> static inline void st_stream(T *p, T v) { *p = v; }
unsigned char k2s_smem_raw[1 << 18];
unsigned char k2d_smem_raw[1 << 18];
}
template <typename T> static inline T __ldg(const T *p) { return *p; }
template <typename T> static inline T __ldcs(const T *p) { return *p; }
static inline unsigned long long __umul64hi(unsigned long long a, unsigned long long b) {
    return static_cast<unsigned long long>((static_cast<unsigned __int128>(a) * b) >> 64);
}
struct CUtensorMap { const void *base; uint64_t width, height, pitch_bytes; uint32_t box_w, box_h; int elem_size; };
namespace xrs {
static inline uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(reinterpret_cast<uintptr_t>(p)); }
static inline void mbar_init(uint64_t *bar, uint32_t) { __atomic_store_n(bar, 0ull, __ATOMIC_RELEASE); }
static inline void mbar_fence_init() {}
static inline void fence_proxy_async() {}
static inline void mbar_arrive_expect_tx(uint64_t *, uint32_t) {}
static inline void mbar_wait(uint64_t *bar, uint32_t parity) {
    while ((__atomic_load_n(bar, __ATOMIC_ACQUIRE) & 1ull) == parity) sched_yield();
}
static long xrsh_tma_boxes = 0, xrsh_tma_oob = 0;  // statistics for the tests
static inline void tma_load_2d(void *dst_smem, const CUtensorMap *map, int x, int y, uint64_t *bar) {
    unsigned char *d = static_cast<unsigned char *>(dst_smem);
    const unsigned char *s = static_cast<const unsigned char *>(map->base);
    const int e = map->elem_size;
    bool oob = false;
    for (uint32_t r = 0; r < map->box_h; ++r)
        for (uint32_t c = 0; c < map->box_w; ++c) {
            const int64_t yy = static_cast<int64_t>(y) + r, xx = static_cast<int64_t>(x) + c;
            unsigned char *o = d + (static_cast<size_t>(r) * map->box_w + c) * e;
            if (yy >= 0 && xx >= 0 && yy < static_cast<int64_t>(map->height) && xx < static_cast<int64_t>(map->width))
                std::memcpy(o, s + yy * map->pitch_bytes + xx * e, e);
            else { std::memset(o, 0, e); oob = true; }
        }
    ++xrsh_tma_boxes;
    if (oob) ++xrsh_tma_oob;
    __atomic_fetch_add(bar, 1ull, __ATOMIC_RELEASE);  // the phase completes: its parity flips
}
template <typename T> static inline T *elem_ptr(T *base, uint32_t index) { return base + index; }
}
"""

K2_EXPORT = r"""
namespace {
struct XrshLaunch { unsigned gx, gy; int threads; bool block2d; const std::function<void()> *body; };
struct XrshLaunchThread { unsigned tid; const XrshLaunch *l; };
void *xrsh_launch_thread(void *p) {
    const XrshLaunchThread *a = static_cast<const XrshLaunchThread *>(p);
    const XrshLaunch &l = *a->l;
    if (l.block2d) { threadIdx.x = a->tid % 32; threadIdx.y = a->tid / 32; blockDim.x = 32; blockDim.y = l.threads / 32; }
    else { threadIdx.x = a->tid; threadIdx.y = 0; blockDim.x = l.threads; blockDim.y = 1; }
    gridDim.x = l.gx; gridDim.y = l.gy;
    for (unsigned by = 0; by < l.gy; ++by)
        for (unsigned bx = 0; bx < l.gx; ++bx) {
            blockIdx.x = bx; blockIdx.y = by;
            (*l.body)();
            __syncthreads();  // the next CTA reuses the staging buffers and the barriers
        }
    return nullptr;
}
void xrsh_launch(unsigned gx, unsigned gy, int threads, bool block2d, const std::function<void()> &body) {
    XrshLaunch l{gx, gy, threads, block2d, &body};
    pthread_barrier_init(&xrsh_block_bar, nullptr, threads);
    for (int k = 0; k < threads / 32; ++k) {
        pthread_barrier_init(&xrsh_warps[k].bar, nullptr, 32);
        std::memset(xrsh_warps[k].gen, 0, sizeof(xrsh_warps[k].gen));
    }
    std::vector<pthread_t> th(threads);
    std::vector<XrshLaunchThread> args(threads);
    for (int t = 0; t < threads; ++t) {
        args[t] = XrshLaunchThread{static_cast<unsigned>(t), &l};
        pthread_create(&th[t], nullptr, xrsh_launch_thread, &args[t]);
    }
    for (int t = 0; t < threads; ++t) pthread_join(th[t], nullptr);
    pthread_barrier_destroy(&xrsh_block_bar);
    for (int k = 0; k < threads / 32; ++k) pthread_barrier_destroy(&xrsh_warps[k].bar);
}
CUtensorMap xrsh_map(const void *base, int elem, int64_t win_w, int64_t win_h, int64_t pitch_elems) {
    return CUtensorMap{base, static_cast<uint64_t>(win_w), static_cast<uint64_t>(win_h), static_cast<uint64_t>(pitch_elems) * elem,
                       static_cast<uint32_t>(xrs::K2S_BOX_W), static_cast<uint32_t>(xrs::K2S_BOX_H), elem};
}

// launch_gather of gather.cu: bands in chunks of K2_MAX_BANDS, staged kernel when `staged`, else the direct one
template <typename T, int METHOD>
void xrsh_gather_tm(const T *src, int64_t band_stride, int n_bands, int64_t src_h, int64_t src_w, int64_t src_pitch,
                    int64_t win_i0, int64_t win_j0, int64_t win_w, int64_t win_h, const double *ij, T *dst, int64_t dst_h,
                    int64_t dst_w, double fill, bool staged) {
    using namespace xrs;
    const T fill_t = cast_fill<T>(fill);
    IjSource ijs = {};
    ijs.ij = ij;
    for (int b0 = 0; b0 < n_bands; b0 += K2_MAX_BANDS) {
        const int nb = std::min(K2_MAX_BANDS, n_bands - b0);
        if (staged) {
            StagedParams<T> sp;
            std::memset(static_cast<void *>(&sp), 0, sizeof(sp));
            for (int b = 0; b < nb; ++b) {
                sp.src[b] = src + (b0 + b) * band_stride;
                sp.dst[b] = dst + (b0 + b) * dst_h * dst_w;
                sp.maps[b] = xrsh_map(sp.src[b], sizeof(T), win_w, win_h, src_pitch);
            }
            xrsh_launch(static_cast<unsigned>(ceil_div(dst_w, K2S_TW)), static_cast<unsigned>(ceil_div(dst_h, K2S_TH)), K2S_THREADS,
                        false, [&] { k2_gather_staged<T, METHOD, false>(sp, nb, src_h, src_w, src_pitch, win_i0, win_j0, ijs, dst_h, dst_w, fill_t); });
        } else {
            PlaneTable<T> pt;
            for (int b = 0; b < K2_MAX_BANDS; ++b) {
                pt.src[b] = b < nb ? src + (b0 + b) * band_stride : nullptr;
                pt.dst[b] = b < nb ? dst + (b0 + b) * dst_h * dst_w : nullptr;
            }
            xrsh_launch(static_cast<unsigned>(ceil_div(dst_w, K2_BX)), static_cast<unsigned>(ceil_div(dst_h, K2_BY)), K2_BX * K2_BY, true,
                        [&] { k2_gather_direct<T, METHOD, false>(pt, nb, src_h, src_w, src_pitch, win_i0, win_j0, ijs, dst_h, dst_w, fill_t); });
        }
    }
}
template <typename T>
int xrsh_gather_t(const void *src, int64_t band_stride, int n_bands, int64_t src_h, int64_t src_w, int64_t src_pitch,
                  int64_t win_i0, int64_t win_j0, int64_t win_w, int64_t win_h, const double *ij, void *dst, int64_t dst_h,
                  int64_t dst_w, int method, double fill, bool staged) {
    const T *s = static_cast<const T *>(src);
    T *d = static_cast<T *>(dst);
    switch (method) {
    case XRS_NEAREST: xrsh_gather_tm<T, XRS_NEAREST>(s, band_stride, n_bands, src_h, src_w, src_pitch, win_i0, win_j0, win_w, win_h, ij, d, dst_h, dst_w, fill, staged); return 0;
    case XRS_BILINEAR: xrsh_gather_tm<T, XRS_BILINEAR>(s, band_stride, n_bands, src_h, src_w, src_pitch, win_i0, win_j0, win_w, win_h, ij, d, dst_h, dst_w, fill, staged); return 0;
    case XRS_TRIANGULAR: xrsh_gather_tm<T, XRS_TRIANGULAR>(s, band_stride, n_bands, src_h, src_w, src_pitch, win_i0, win_j0, win_w, win_h, ij, d, dst_h, dst_w, fill, staged); return 0;
    }
    return 1;
}

// launch_dual of gather_dual.cu
template <typename T, int METHOD>
void xrsh_dual_tm(const T *src, int64_t band_stride, int n_bands, int64_t src_h, int64_t src_w, int64_t src_pitch, int64_t win_i0,
                  int64_t win_j0, int64_t win_w, int64_t win_h, const double *ij, T *dst_interp, T *dst_near, int64_t dst_h,
                  int64_t dst_w, double fill_interp, double fill_near) {
    using namespace xrs;
    const T fi = cast_fill<T>(fill_interp), fn = cast_fill<T>(fill_near);
    for (int b0 = 0; b0 < n_bands; b0 += K2_MAX_BANDS) {
        const int nb = std::min(K2_MAX_BANDS, n_bands - b0);
        DualParams<T> dp;
        std::memset(static_cast<void *>(&dp), 0, sizeof(dp));
        for (int b = 0; b < nb; ++b) {
            dp.src[b] = src + (b0 + b) * band_stride;
            dp.dst_interp[b] = dst_interp + (b0 + b) * dst_h * dst_w;
            dp.dst_near[b] = dst_near + (b0 + b) * dst_h * dst_w;
            dp.maps[b] = xrsh_map(dp.src[b], sizeof(T), win_w, win_h, src_pitch);
        }
        xrsh_launch(static_cast<unsigned>(ceil_div(dst_w, K2S_TW)), static_cast<unsigned>(ceil_div(dst_h, K2S_TH)), K2S_THREADS, false,
                    [&] { k2_gather_dual<T, METHOD>(dp, nb, src_h, src_w, src_pitch, win_i0, win_j0, ij, dst_h, dst_w, fi, fn); });
    }
}
template <typename T>
int xrsh_dual_t(const void *src, int64_t band_stride, int n_bands, int64_t src_h, int64_t src_w, int64_t src_pitch, int64_t win_i0,
                int64_t win_j0, int64_t win_w, int64_t win_h, const double *ij, void *di, void *dn, int64_t dst_h, int64_t dst_w,
                int method, double fill_interp, double fill_near) {
    const T *s = static_cast<const T *>(src);
    if (method == XRS_BILINEAR) xrsh_dual_tm<T, XRS_BILINEAR>(s, band_stride, n_bands, src_h, src_w, src_pitch, win_i0, win_j0, win_w, win_h, ij, static_cast<T *>(di), static_cast<T *>(dn), dst_h, dst_w, fill_interp, fill_near);
    else if (method == XRS_TRIANGULAR) xrsh_dual_tm<T, XRS_TRIANGULAR>(s, band_stride, n_bands, src_h, src_w, src_pitch, win_i0, win_j0, win_w, win_h, ij, static_cast<T *>(di), static_cast<T *>(dn), dst_h, dst_w, fill_interp, fill_near);
    else return 1;
    return 0;
}
}

// src points at the window origin (win_i0, win_j0) of band 0; src_h / src_w are the FULL image's (tap clamping)
extern "C" int xrsh_k2_gather(const void *src, int dtype, long band_stride, int n_bands, long src_h, long src_w, long src_pitch,
                              long win_i0, long win_j0, long win_w, long win_h, const double *ij, void *dst, long dst_h, long dst_w,
                              int method, double fill, int staged, long *stats) {
    xrs::xrsh_tma_boxes = xrs::xrsh_tma_oob = 0;
    int rc = 2;
    XRSH_DISPATCH_DTYPE(dtype, T, rc = xrsh_gather_t<T>(src, band_stride, n_bands, src_h, src_w, src_pitch, win_i0, win_j0, win_w, win_h, ij, dst, dst_h, dst_w, method, fill, staged != 0));
    stats[0] = xrs::xrsh_tma_boxes; stats[1] = xrs::xrsh_tma_oob;
    return rc;
}
extern "C" int xrsh_k2_gather_dual(const void *src, int dtype, long band_stride, int n_bands, long src_h, long src_w, long src_pitch,
                                   long win_i0, long win_j0, long win_w, long win_h, const double *ij, void *dst_interp,
                                   void *dst_near, long dst_h, long dst_w, int method, double fill_interp, double fill_near,
                                   long *stats) {
    xrs::xrsh_tma_boxes = xrs::xrsh_tma_oob = 0;
    int rc = 2;
    XRSH_DISPATCH_DTYPE(dtype, T, rc = xrsh_dual_t<T>(src, band_stride, n_bands, src_h, src_w, src_pitch, win_i0, win_j0, win_w, win_h, ij, dst_interp, dst_near, dst_h, dst_w, method, fill_interp, fill_near));
    stats[0] = xrs::xrsh_tma_boxes; stats[1] = xrs::xrsh_tma_oob;
    return rc;
}
"""


K2_EXPORT_FUSED = r"""
// xrs_rectify_gather's second half: the staged gather in FUSED mode -- the fractional source index of a target
// pixel comes from K1's claim words through resolve_pixel, in registers, instead of the ij image
namespace {
template <typename T, int METHOD>
void xrsh_fused_tm(const T *src, int n_bands, const xrs::IjGeom &geom, T *dst, double fill) {
    using namespace xrs;
    const int64_t dst_h = geom.row_end - geom.row_begin, dst_w = geom.dst_w;
    IjSource ijs = {};
    ijs.ij = nullptr;
    ijs.geom = geom;
    StagedParams<T> sp;
    std::memset(static_cast<void *>(&sp), 0, sizeof(sp));
    for (int b = 0; b < n_bands; ++b) {
        sp.src[b] = src + b * geom.src_h * geom.src_w;
        sp.dst[b] = dst + b * dst_h * dst_w;
        sp.maps[b] = xrsh_map(sp.src[b], sizeof(T), geom.src_w, geom.src_h, geom.src_w);
    }
    const T fill_t = cast_fill<T>(fill);
    xrsh_launch(static_cast<unsigned>(ceil_div(dst_w, K2S_TW)), static_cast<unsigned>(ceil_div(dst_h, K2S_TH)), K2S_THREADS, false,
                [&] { k2_gather_staged<T, METHOD, true>(sp, n_bands, geom.src_h, geom.src_w, geom.src_w, 0, 0, ijs, dst_h, dst_w, fill_t); });
}
template <typename T>
int xrsh_fused_t(const void *src, int n_bands, const xrs::IjGeom &g, void *dst, int method, double fill) {
    const T *s = static_cast<const T *>(src);
    T *d = static_cast<T *>(dst);
    switch (method) {
    case XRS_NEAREST: xrsh_fused_tm<T, XRS_NEAREST>(s, n_bands, g, d, fill); return 0;
    case XRS_BILINEAR: xrsh_fused_tm<T, XRS_BILINEAR>(s, n_bands, g, d, fill); return 0;
    case XRS_TRIANGULAR: xrsh_fused_tm<T, XRS_TRIANGULAR>(s, n_bands, g, d, fill); return 0;
    }
    return 1;
}
}
extern "C" int xrsh_k2_gather_fused(const void *src, int dtype, int n_bands, const double *x, const double *y, long src_h, long src_w,
                                    const int64_t *tile_boxes, const uint32_t *claims, long dst_h, long dst_w, int tile_h,
                                    int tile_w, double x_min, double y_min, double y_max, double x_res, double y_res, int j_up,
                                    long row_begin, long row_end, int method, double fill, void *dst) {
    using namespace xrs;
    if (n_bands > K2_MAX_BANDS) return 3;
    IjGeom g = {};
    g.x = x; g.y = y; g.src_h = src_h; g.src_w = src_w; g.src_pitch = src_w;
    g.tile_boxes = tile_boxes; g.claims = const_cast<uint32_t *>(claims);
    g.dst_h = dst_h; g.dst_w = dst_w;
    g.tile_h = tile_h < dst_h ? tile_h : static_cast<int>(dst_h);
    g.tile_w = tile_w < dst_w ? tile_w : static_cast<int>(dst_w);
    g.ntx = static_cast<int>((dst_w + g.tile_w - 1) / g.tile_w);
    g.nty = static_cast<int>((dst_h + g.tile_h - 1) / g.tile_h);
    g.x_min = x_min; g.y_min = y_min; g.y_max = y_max; g.x_res = x_res; g.y_res = y_res;
    g.j_up = j_up ? 1 : 0;
    g.row_begin = row_begin; g.row_end = row_end;
    g.magic_nqi = div_magic_of(static_cast<uint64_t>(src_w - 1));
    g.magic_tw = div_magic_of(static_cast<uint64_t>(g.tile_w));
    g.magic_th = div_magic_of(static_cast<uint64_t>(g.tile_h));
    int rc = 2;
    XRSH_DISPATCH_DTYPE(dtype, T, rc = xrsh_fused_t<T>(src, n_bands, g, dst, method, fill));
    return rc;
}
"""


def _kernel_text(name: str, cut_marker: str, drop_includes) -> str:
    text = open(os.path.join(CSRC, name)).read()
    for inc in drop_includes:
        text, n = re.subn(r"#include " + re.escape(inc) + r"\n", "", text)
        assert n == 1, f"{name} no longer includes {inc} exactly once"
    text = text.replace("#pragma once\n", "")
    if cut_marker:
        cut = text.find(cut_marker)
        assert cut > 0 and "<<<" not in text[:cut], f"layout of {name} changed"
        text = text[:cut] + "\n}  // namespace xrs\n"
    return text


def build_k2(out_dir: str) -> str:
    """Host build of rectify_common.cuh + gather_common.cuh + the kernels of gather.cu and gather_dual.cu."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    parts = [
        _kernel_text("rectify_common.cuh", "", ['"common.cuh"']),
        _kernel_text("gather_common.cuh", "", ['"rectify_common.cuh"', '"tma.cuh"']),
        _kernel_text("gather.cu", "// ---------------------------------------------------------------------------\n// host side",
                     ['"gather_common.cuh"']),
        _kernel_text("gather_dual.cu", "template <typename T>\nstatic int launch_dual", ['"gather_common.cuh"']),
    ]
    src = os.path.join(out_dir, "k2_host.cpp")
    with open(src, "w") as fh:
        fh.write(K2_SHIM + "".join(parts) + K2_EXPORT + K2_EXPORT_FUSED)
    so = os.path.join(out_dir, "libxrs_k2host.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of gather.cu / gather_dual.cu failed:\n" + res.stderr[-6000:])
    return so


def _k2_codes():
    """dtype / method codes from include/xrs.h (the enums the C ABI uses)."""
    hdr = open(os.path.join(ROOT, "include", "xrs.h")).read()
    def code(name):
        m = re.search(r"\b" + name + r"\s*=\s*(\d+)", hdr)
        assert m, name
        return int(m.group(1))
    dt = {np.dtype(t): code(name) for t, name in (
        (np.float32, "XRS_F32"), (np.float64, "XRS_F64"), (np.uint8, "XRS_U8"), (np.int8, "XRS_I8"), (np.uint16, "XRS_U16"),
        (np.int16, "XRS_I16"), (np.int32, "XRS_I32"), (np.uint32, "XRS_U32"), (np.int64, "XRS_I64"))}
    me = {"nearest": code("XRS_NEAREST"), "bilinear": code("XRS_BILINEAR"), "triangular": code("XRS_TRIANGULAR")}
    return dt, me


def _k2_window(src, window):
    """(pointer to the window origin of band 0, band stride, pitch, win_i0, win_j0, win_w, win_h)."""
    nb, h, w = src.shape
    i0, j0, i1, j1 = window if window is not None else (0, 0, w, h)
    return src.ctypes.data + (j0 * w + i0) * src.itemsize, h * w, w, i0, j0, i1 - i0, j1 - j0


def k2_gather(so_path: str, src, ij, method: str, fill, staged: bool = True, window=None):
    """``xrs_gather_ij`` through the host build of ``k2_gather_staged`` (or ``k2_gather_direct``): ``(out, stats)``
    with stats = (boxes copied by the TMA stand-in, boxes that reached outside the tensor).  ``window`` =
    (i0, j0, i1, j1): only that part of the source is addressable (the kernels get a pointer to its origin)."""
    lib = ctypes.CDLL(so_path)
    dt, me = _k2_codes()
    src = np.ascontiguousarray(src)
    ij = np.ascontiguousarray(ij, dtype=np.float64)
    nb, h, w = src.shape
    _, dh, dw = ij.shape
    out = np.empty((nb, dh, dw), dtype=src.dtype)
    stats = np.zeros(2, dtype=np.int64)
    base, bstride, pitch, i0, j0, ww, wh = _k2_window(src, window)
    c_d, c_l, c_i, c_p = ctypes.c_double, ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_k2_gather.restype = c_i
    lib.xrsh_k2_gather.argtypes = [c_p, c_i, c_l, c_i, c_l, c_l, c_l, c_l, c_l, c_l, c_l, c_p, c_p, c_l, c_l, c_i, c_d, c_i, c_p]
    rc = lib.xrsh_k2_gather(base, dt[src.dtype], bstride, nb, h, w, pitch, i0, j0, ww, wh, ij.ctypes.data, out.ctypes.data, dh,
                            dw, me[method], float(fill), int(staged), stats.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"xrsh_k2_gather failed ({rc})")
    return out, (int(stats[0]), int(stats[1]))


def k2_gather_dual(so_path: str, src, ij, method: str, fill_interp, fill_near, window=None):
    """``xrs_gather_ij2`` through the host build of ``k2_gather_dual``: ``(interp, nearest, stats)``."""
    lib = ctypes.CDLL(so_path)
    dt, me = _k2_codes()
    src = np.ascontiguousarray(src)
    ij = np.ascontiguousarray(ij, dtype=np.float64)
    nb, h, w = src.shape
    _, dh, dw = ij.shape
    out_i = np.empty((nb, dh, dw), dtype=src.dtype)
    out_n = np.empty((nb, dh, dw), dtype=src.dtype)
    stats = np.zeros(2, dtype=np.int64)
    base, bstride, pitch, i0, j0, ww, wh = _k2_window(src, window)
    c_d, c_l, c_i, c_p = ctypes.c_double, ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_k2_gather_dual.restype = c_i
    lib.xrsh_k2_gather_dual.argtypes = [c_p, c_i, c_l, c_i, c_l, c_l, c_l, c_l, c_l, c_l, c_l, c_p, c_p, c_p, c_l, c_l, c_i, c_d,
                                        c_d, c_p]
    rc = lib.xrsh_k2_gather_dual(base, dt[src.dtype], bstride, nb, h, w, pitch, i0, j0, ww, wh, ij.ctypes.data,
                                 out_i.ctypes.data, out_n.ctypes.data, dh, dw, me[method], float(fill_interp), float(fill_near),
                                 stats.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"xrsh_k2_gather_dual failed ({rc})")
    return out_i, out_n, (int(stats[0]), int(stats[1]))


def k2_gather_fused(so_path: str, src, x, y, tile_boxes, claims, g, method: str, fill, rows=None) -> np.ndarray:
    """The gather half of ``xrs_rectify_gather`` (``k2_gather_staged<T, METHOD, FUSED = true>``): the bands through K1's
    claim words (``claims``: (rows, W) uint32 of the row range ``rows``); ``g``: oracle RegularGrid."""
    lib = ctypes.CDLL(so_path)
    dt, me = _k2_codes()
    src = np.ascontiguousarray(src)
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    boxes = np.ascontiguousarray(tile_boxes, dtype=np.int64)
    claims = np.ascontiguousarray(claims, dtype=np.uint32)
    r0, r1 = rows if rows is not None else (0, g.height)
    nb, h, w = src.shape
    out = np.empty((nb, r1 - r0, g.width), dtype=src.dtype)
    c_d, c_l, c_i, c_p = ctypes.c_double, ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_k2_gather_fused.restype = c_i
    lib.xrsh_k2_gather_fused.argtypes = [c_p, c_i, c_i, c_p, c_p, c_l, c_l, c_p, c_p, c_l, c_l, c_i, c_i, c_d, c_d, c_d, c_d, c_d, c_i,
                                         c_l, c_l, c_i, c_d, c_p]
    rc = lib.xrsh_k2_gather_fused(src.ctypes.data, dt[src.dtype], nb, x.ctypes.data, y.ctypes.data, h, w, boxes.ctypes.data, claims.ctypes.data,
                                  g.height, g.width, g.tile_h, g.tile_w, float(g.x_min), float(g.y_min), float(g.y_max),
                                  float(g.x_res), float(g.y_res), int(g.is_j_axis_up), r0, r1, me[method], float(fill),
                                  out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"xrsh_k2_gather_fused failed ({rc})")
    return out


# ---------------------------------------------------------------------------
# K3 as kernels (csrc/reproject.cu: k3_lattice_nodes, k3_reproject<T, OUT, METHOD, SEP>) on top of proj.cuh
# ---------------------------------------------------------------------------
# Compiled with XRS_K3_LD256=0 (the tap loads are plain loads instead of the 256-byte L2 hint) and with the one
# `prefetch.global.L2` instruction replaced by a no-op -- memory hints, no arithmetic.  make_proj_consts, the
# lattice pre-kernel, the tile logic, the separable / row-block / lattice / exact forms and the per-pixel blend
# are the product's text.  Differences to the device build: libm instead of CUDA's math library and no FMA
# contraction in proj.cuh (~1e-9 m in the source coordinates).
K3K_SHIM = "#define _GNU_SOURCE 1\n#define XRS_K3_LD256 0\n" + XRSH_DISPATCH + K0_SHIM.replace("#define __shared__\n", "#define __shared__ static\n") + r"""
#include <string>
#include <type_traits>
#include <math.h>
#define __grid_constant__
#define __noinline__
#define __constant__ const
using std::fabs; using std::sqrt; using std::sin; using std::cos; using std::tan; using std::atan; using std::atan2;
using std::asin; using std::sinh; using std::asinh; using std::exp; using std::log; using std::rint; using std::fmin;
using std::fmax; using std::floor; using std::ceil;
struct double2 { double x, y; };
namespace xrs {
static inline int fail(const std::string &) { return 1; }
static inline double dadd(double a, double b) { return a + b; }
static inline double dsub(double a, double b) { return a - b; }
static inline double dmul(double a, double b) { return a * b; }
static inline double ddiv(double a, double b) { return a / b; }
template <typename T> static inline void st_stream(T *p, T v) { *p = v; }
}
template <typename T> static inline T __ldg(const T *p) { return *p; }
template <typename T> static inline T __ldcs(const T *p) { return *p; }
static inline int __double2int_rd(double d) { return static_cast<int>(std::floor(d)); }
static inline int __double2int_ru(double d) { return static_cast<int>(std::ceil(d)); }
static inline int __double2int_rn(double d) { return static_cast<int>(std::nearbyint(d)); }
static inline float __fsub_rn(float a, float b) { return a - b; }
// lanes of the warp that have not left the kernel: every lane is either here or gone (see xrsh_lane_state)
static int xrsh_lane_state[XRSH_MAX_WARPS][32];  // 0 running, 1 returned, 2 at __activemask
static inline unsigned __activemask() {
    const int w = static_cast<int>(threadIdx.x >> 5), l = xrsh_l();
    __atomic_store_n(&xrsh_lane_state[w][l], 2, __ATOMIC_RELEASE);
    unsigned m = 0;
    for (int k = 0; k < 32; ++k) {
        int s;
        while ((s = __atomic_load_n(&xrsh_lane_state[w][k], __ATOMIC_ACQUIRE)) == 0) sched_yield();
        if (s == 2) m |= 1u << k;
    }
    return m;
}
static int xrsh_and_acc[2] = {1, 1};
static thread_local unsigned xrsh_and_n = 0;
static inline int __syncthreads_and(int p) {
    const unsigned k = xrsh_and_n++ & 1u;
    if (!p) __atomic_store_n(&xrsh_and_acc[k], 0, __ATOMIC_RELEASE);
    __syncthreads();
    const int r = __atomic_load_n(&xrsh_and_acc[k], __ATOMIC_ACQUIRE);
    __syncthreads();
    if (threadIdx.x == 0) __atomic_store_n(&xrsh_and_acc[k], 1, __ATOMIC_RELEASE);
    return r;
}
"""

K3K_EXPORT = r"""
namespace {
struct XrshK3Launch { unsigned gx, gy; const std::function<void()> *body; };
struct XrshK3Thread { unsigned tid; const XrshK3Launch *l; };
void *xrsh_k3_thread(void *p) {
    const XrshK3Thread *a = static_cast<const XrshK3Thread *>(p);
    const XrshK3Launch &l = *a->l;
    threadIdx.x = a->tid; blockDim.x = xrs::K3T_THREADS; gridDim.x = l.gx; gridDim.y = l.gy;
    const int w = static_cast<int>(a->tid >> 5), lane = static_cast<int>(a->tid & 31);
    for (unsigned by = 0; by < l.gy; ++by)
        for (unsigned bx = 0; bx < l.gx; ++bx) {
            blockIdx.x = bx; blockIdx.y = by;
            __atomic_store_n(&xrsh_lane_state[w][lane], 0, __ATOMIC_RELEASE);
            __atomic_store_n(&xrsh_warps[w].gen[lane], 0u, __ATOMIC_RELEASE);
            xrsh_gen = 0;
            __syncthreads();   // every lane is "running" and at generation 0 before any collective of this CTA
            (*l.body)();
            __atomic_store_n(&xrsh_lane_state[w][lane], 1, __ATOMIC_RELEASE);
            __syncthreads();   // the next CTA reuses the shared arrays
        }
    return nullptr;
}
void xrsh_k3_launch(unsigned gx, unsigned gy, const std::function<void()> &body) {
    XrshK3Launch l{gx, gy, &body};
    const int threads = xrs::K3T_THREADS;
    pthread_barrier_init(&xrsh_block_bar, nullptr, threads);
    for (int k = 0; k < threads / 32; ++k) pthread_barrier_init(&xrsh_warps[k].bar, nullptr, 32);
    std::vector<pthread_t> th(threads);
    std::vector<XrshK3Thread> args(threads);
    for (int t = 0; t < threads; ++t) {
        args[t] = XrshK3Thread{static_cast<unsigned>(t), &l};
        pthread_create(&th[t], nullptr, xrsh_k3_thread, &args[t]);
    }
    for (int t = 0; t < threads; ++t) pthread_join(th[t], nullptr);
    pthread_barrier_destroy(&xrsh_block_bar);
    for (int k = 0; k < threads / 32; ++k) pthread_barrier_destroy(&xrsh_warps[k].bar);
}

// launch_reproject of reproject.cu: plan, lattice pre-kernel, band chunks, separable or general kernel
template <typename T, typename OUT, int METHOD>
int xrsh_launch_reproject(const xrs::K3Geom &g_in, const T *src, int64_t band_stride, OUT *dst, int n_bands, double fill,
                          int exact_only, int use_nodes, long *stats) {
    using namespace xrs;
    K3Geom g = g_in;
    g.lat_nodes = nullptr;
    const int64_t rows = g.row_end - g.row_begin;
    const unsigned gx = static_cast<unsigned>(ceil_div(g.dst_w, K3T_COLS)), gy = static_cast<unsigned>(ceil_div(g.row_end - g.row_tile0, K3T_ROWS));
    const T fill_t = cast_fill<T>(fill);
    const int plan = choose_plan(g.from, g.to) | (exact_only ? K3_PLAN_EXACT_ONLY : 0);
    const bool axis_only = (g.from.kind == XRS_PROJ_GEOGRAPHIC || g.from.kind == XRS_PROJ_WEBMERC) &&
                           (g.to.kind == XRS_PROJ_GEOGRAPHIC || g.to.kind == XRS_PROJ_WEBMERC);
    std::vector<double> nodes;
    if (use_nodes && XRS_K3_LATTICE && !axis_only && !(plan & K3_PLAN_EXACT_ONLY) && g.dst_w > 1 && g.dst_h > 1) {
        const int n_tiles = static_cast<int>(gx * gy);
        nodes.assign(static_cast<size_t>(n_tiles) * 34, 0.0);
        blockDim.x = 256; gridDim.x = static_cast<unsigned>(ceil_div(static_cast<int64_t>(n_tiles) * 32, 256));
        for (unsigned b = 0; b < gridDim.x; ++b)
            for (unsigned t = 0; t < 256; ++t) { blockIdx.x = b; threadIdx.x = t; k3_lattice_nodes(g, nodes.data(), static_cast<int>(gx), n_tiles); }
        g.lat_nodes = nodes.data();
    }
    stats[0] = plan; stats[1] = axis_only; stats[2] = g.lat_nodes != nullptr;
    for (int b0 = 0; b0 < n_bands; b0 += K3_MAX_BANDS) {
        const int nb = std::min(K3_MAX_BANDS, n_bands - b0);
        K3Planes<T, OUT> planes = {};
        for (int b = 0; b < nb; ++b) {
            planes.src[b] = src + (b0 + b) * band_stride;
            planes.dst[b] = dst + (b0 + b) * rows * g.dst_w;
        }
        if (axis_only) xrsh_k3_launch(gx, gy, [&] { k3_reproject<T, OUT, METHOD, true>(g, planes, nb, fill_t, plan); });
        else xrsh_k3_launch(gx, gy, [&] { k3_reproject<T, OUT, METHOD, false>(g, planes, nb, fill_t, plan); });
    }
    return 0;
}
}

template <typename T>
int xrsh_reproject_t(const xrs::K3Geom &g, const void *src_v, long band_stride, int n_bands, int out_f64, int method,
                     double fill, int exact_only, int use_nodes, void *dst, long *stats) {
    const T *src = static_cast<const T *>(src_v);
    switch (method) {
    case XRS_NEAREST:
        return xrsh_launch_reproject<T, T, XRS_NEAREST>(g, src, band_stride, static_cast<T *>(dst), n_bands, fill, exact_only, use_nodes, stats);
    case XRS_TRIANGULAR:
        return xrsh_launch_reproject<T, T, XRS_TRIANGULAR>(g, src, band_stride, static_cast<T *>(dst), n_bands, fill, exact_only, use_nodes, stats);
    case XRS_BILINEAR:
        if (out_f64) return xrsh_launch_reproject<T, double, XRS_BILINEAR>(g, src, band_stride, static_cast<double *>(dst), n_bands, fill, exact_only, use_nodes, stats);
        return xrsh_launch_reproject<T, T, XRS_BILINEAR>(g, src, band_stride, static_cast<T *>(dst), n_bands, fill, exact_only, use_nodes, stats);
    }
    return 2;
}

// xrs_reproject: out_f64 = 1 writes float64 (bilinear as the reference returns it), otherwise the source dtype.  src
// points at the resident window's origin (win_i0, win_j0).
extern "C" int xrsh_reproject(const void *src, int dtype, long band_stride, int n_bands, int out_f64, long src_h, long src_w, long src_pitch,
                              long win_i0, long win_j0, long win_w, long win_h, const xrs_proj *src_crs, const xrs_proj *dst_crs,
                              const double *dst_x, const double *dst_y, long dst_h, long dst_w, int tile_h, int tile_w,
                              const double *tile_x0, const double *tile_y0, const int32_t *tile_i0, const int32_t *tile_j0,
                              int tile_win_w, int tile_win_h, double src_x_res, double src_y_res, int method, double fill,
                              long row_begin, long row_end, int exact_only, int use_nodes, void *dst, long *stats) {
    using namespace xrs;
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
    int rc = 3;
    XRSH_DISPATCH_DTYPE(dtype, T, rc = xrsh_reproject_t<T>(g, src, band_stride, n_bands, out_f64, method, fill, exact_only, use_nodes, dst, stats));
    return rc;
}
"""


def build_k3(out_dir: str) -> str:
    """Host build of proj.cuh + reproject.cu up to (and including) choose_plan."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    proj = open(os.path.join(CSRC, "proj.cuh")).read()
    proj, n = re.subn(r'#include "common.cuh"\n', "", proj)
    assert n == 1, "proj.cuh no longer includes common.cuh exactly once"
    proj = proj.replace("#pragma once\n", "")
    text = open(os.path.join(CSRC, "reproject.cu")).read()
    for inc in ('"proj.cuh"', '"tma.cuh"'):
        text, n = re.subn(r"#include " + re.escape(inc) + r"\n", "", text)
        assert n == 1, f"reproject.cu no longer includes {inc} exactly once"
    text, n = re.subn(r'asm volatile\("prefetch\.global\.L2 \[%0\];" ::"l"\(planes\.src\[b\] \+ off\)\);',
                      "(void)(planes.src[b] + off);", text)
    assert n == 1, "the L2 prefetch instruction of k3_prefetch_box moved"
    cut = text.find("// The scratch of k3_lattice_nodes comes from")
    assert cut > 0 and "<<<" not in text[:cut] and "static int choose_plan" in text[:cut], "layout of reproject.cu changed"
    src = os.path.join(out_dir, "k3_host.cpp")
    with open(src, "w") as fh:
        fh.write(K3K_SHIM + "#include <functional>\n" + proj + text[:cut] + "\n}  // namespace xrs\n" + K3K_EXPORT)
    so = os.path.join(out_dir, "libxrs_k3host.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of reproject.cu failed:\n" + res.stderr[-6000:])
    return so


def k3_reproject(so_path: str, src, src_gm, tgt_gm, windows, method: str, fill, out_f64=None, rows=None, window=None,
                 exact_only: bool = False, use_nodes: bool = True):
    """``xrs_reproject`` through the host build: ``(out, (plan, separable kernel, lattice nodes))``; the output has the
    source's dtype, or float64 with ``out_f64`` (default: bilinear, as the reference returns it).
    ``src_gm`` / ``tgt_gm``: the product's GridMappings; ``windows``: ``reproject.SourceWindows``; ``window`` =
    (i0, j0, i1, j1) resident part of the source; arguments are prepared as ``ReprojectPlan`` does."""
    from xcube_resampling_b200._lib import XrsProj

    lib = ctypes.CDLL(so_path)
    dt, me = _k2_codes()
    src = np.ascontiguousarray(src)
    nb, h, w = src.shape
    if out_f64 is None:
        out_f64 = method == "bilinear"
    r0, r1 = rows if rows is not None else (0, tgt_gm.height)
    out = np.empty((nb, r1 - r0, tgt_gm.width), dtype=np.float64 if out_f64 else src.dtype)
    base, bstride, pitch, i0, j0, ww, wh = _k2_window(src, window)
    sp, dp = XrsProj.from_crs(src_gm.crs), XrsProj.from_crs(tgt_gm.crs)
    dst_x = np.ascontiguousarray(tgt_gm.x_values, dtype=np.float64)
    dst_y = np.ascontiguousarray(tgt_gm.y_values, dtype=np.float64)
    x0 = np.ascontiguousarray(windows.x0.astype(np.float64).ravel())
    y0 = np.ascontiguousarray(windows.y0.astype(np.float64).ravel())
    ti0 = np.ascontiguousarray(windows.i0.astype(np.int32).ravel())
    tj0 = np.ascontiguousarray(windows.j0.astype(np.int32).ravel())
    stats = np.zeros(3, dtype=np.int64)
    c_d, c_l, c_i, c_p = ctypes.c_double, ctypes.c_long, ctypes.c_int, ctypes.c_void_p
    lib.xrsh_reproject.restype = c_i
    lib.xrsh_reproject.argtypes = [c_p, c_i, c_l, c_i, c_i, c_l, c_l, c_l, c_l, c_l, c_l, c_l, c_p, c_p, c_p, c_p, c_l, c_l, c_i, c_i,
                                   c_p, c_p, c_p, c_p, c_i, c_i, c_d, c_d, c_i, c_d, c_l, c_l, c_i, c_i, c_p, c_p]
    rc = lib.xrsh_reproject(base, dt[src.dtype], bstride, nb, int(out_f64), src_gm.height, src_gm.width, pitch, i0, j0, ww, wh,
                            ctypes.addressof(sp), ctypes.addressof(dp), dst_x.ctypes.data, dst_y.ctypes.data, tgt_gm.height,
                            tgt_gm.width, tgt_gm.tile_height, tgt_gm.tile_width, x0.ctypes.data, y0.ctypes.data,
                            ti0.ctypes.data, tj0.ctypes.data, int(windows.win_w), int(windows.win_h), float(src_gm.x_res),
                            float(src_gm.y_res), me[method], float(fill), r0, r1, int(exact_only), int(use_nodes),
                            out.ctypes.data, stats.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"xrsh_reproject failed ({rc})")
    return out, (int(stats[0]), bool(stats[1]), bool(stats[2]))


# ---------------------------------------------------------------------------
# K4 / K5 as kernels (csrc/resample.cu + csrc/resample_fast.cu, launch code and C ABI included)
# ---------------------------------------------------------------------------
# Both files are compiled unchanged apart from one rewrite: every `NAME<<<grid, block, shm, st>>>(args)` becomes
# `xrsh_launch(grid, block, shm, st, &NAME, args)`.  The launcher runs the grid on 32 host threads, one per lane:
# each walks every (block, warp) in the same order, with threadIdx / blockIdx thread-local, so the lanes of a warp
# meet __any_sync together (exchanged through a shared array between two barrier waits).  These kernels have no
# shared memory and no block barriers.  The rest of the shim:
#   * XRS_TIMED records the kernel name (the list `xrsh_take_log` returns), so tests see which kernel ran;
#   * __ldcs / __ldg count every load whose address is not aligned to the loaded type (uint4: 16, uint2: 8, else
#     its size) -- x86 forgives what faults on the GPU, so this count is how the dispatch rules are checked;
#   * the SIMD-in-a-word intrinsics are written per lane from the CUDA Math API definitions (xrsh_simd exports
#     them for their own test).
RSK_SHIM = r"""
#define _GNU_SOURCE 1
#include <pthread.h>
#include <algorithm>
#include <cassert>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <math.h>
#include <string>
#include <thread>
#include <tuple>
#include <type_traits>
#include <vector>
#include "xrs.h"
#define __device__
#define __host__
#define __global__
#define __forceinline__ inline
#define __launch_bounds__(...)
typedef void *cudaStream_t;
using std::isfinite; using std::floor; using std::fabs; using std::sqrt; using std::rint; using std::fmin; using std::fmax;
struct dim3 {
    unsigned x, y, z;
    dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
static thread_local dim3 threadIdx, blockIdx, blockDim, gridDim;
struct uint4 { unsigned x, y, z, w; };
struct uint2 { unsigned x, y; };
template <typename T> struct xrsh_align { static constexpr uintptr_t value = sizeof(T); };
template <> struct xrsh_align<uint4> { static constexpr uintptr_t value = 16; };
template <> struct xrsh_align<uint2> { static constexpr uintptr_t value = 8; };
static long xrsh_misaligned = 0;
static std::vector<std::string> xrsh_log;
static std::string xrsh_error;
template <typename T> static inline T xrsh_load(const T *p) {
    if (reinterpret_cast<uintptr_t>(p) % xrsh_align<T>::value) __atomic_fetch_add(&xrsh_misaligned, 1, __ATOMIC_RELAXED);
    T v;
    std::memcpy(&v, p, sizeof(T));
    return v;
}
template <typename T> static inline T __ldg(const T *p) { return xrsh_load(p); }
template <typename T> static inline T __ldcs(const T *p) { return xrsh_load(p); }
static inline int atomicOr(int *p, int v) { return __atomic_fetch_or(p, v, __ATOMIC_RELAXED); }
static inline int cudaMemsetAsync(void *p, int v, size_t n, cudaStream_t) { std::memset(p, v, n); return 0; }
// one warp = 32 host threads in lock step at its collectives
static pthread_barrier_t xrsh_warp_bar;
static int xrsh_warp_vote[32];
static thread_local int xrsh_lane = 0;
static inline bool __any_sync(unsigned, bool p) {
    xrsh_warp_vote[xrsh_lane] = p ? 1 : 0;
    pthread_barrier_wait(&xrsh_warp_bar);
    bool any = false;
    for (int k = 0; k < 32; ++k) any = any || xrsh_warp_vote[k] != 0;
    pthread_barrier_wait(&xrsh_warp_bar);
    return any;
}
// SIMD-in-a-word intrinsics (CUDA Math API, integer intrinsics / SIMD intrinsics), lane by lane
static inline uint32_t xrsh_lane_of(uint32_t v, int bits, int k) { return (v >> (bits * k)) & ((1u << bits) - 1u); }
template <typename Op> static inline uint32_t xrsh_per_lane(uint32_t a, uint32_t b, int bits, Op op) {
    uint32_t r = 0;
    for (int k = 0; k < 32 / bits; ++k)
        r |= (op(xrsh_lane_of(a, bits, k), xrsh_lane_of(b, bits, k)) & ((1u << bits) - 1u)) << (bits * k);
    return r;
}
static inline uint32_t __byte_perm(uint32_t x, uint32_t y, uint32_t s) {
    const uint64_t v = (static_cast<uint64_t>(y) << 32) | x;
    uint32_t r = 0;
    for (int k = 0; k < 4; ++k) {
        const uint32_t sel = (s >> (4 * k)) & 0xfu;
        assert((sel & 8u) == 0 && "__byte_perm: only the default mode is emulated");
        r |= static_cast<uint32_t>((v >> (8 * sel)) & 0xffu) << (8 * k);
    }
    return r;
}
static inline uint32_t __vminu4(uint32_t a, uint32_t b) { return xrsh_per_lane(a, b, 8, [](uint32_t x, uint32_t y) { return x < y ? x : y; }); }
static inline uint32_t __vmaxu4(uint32_t a, uint32_t b) { return xrsh_per_lane(a, b, 8, [](uint32_t x, uint32_t y) { return x > y ? x : y; }); }
static inline uint32_t __vminu2(uint32_t a, uint32_t b) { return xrsh_per_lane(a, b, 16, [](uint32_t x, uint32_t y) { return x < y ? x : y; }); }
static inline uint32_t __vmaxu2(uint32_t a, uint32_t b) { return xrsh_per_lane(a, b, 16, [](uint32_t x, uint32_t y) { return x > y ? x : y; }); }
static inline uint32_t __vhaddu4(uint32_t a, uint32_t b) { return xrsh_per_lane(a, b, 8, [](uint32_t x, uint32_t y) { return (x + y) >> 1; }); }
static inline uint32_t __vadd4(uint32_t a, uint32_t b) { return xrsh_per_lane(a, b, 8, [](uint32_t x, uint32_t y) { return x + y; }); }
static inline uint32_t __vcmpeq4(uint32_t a, uint32_t b) { return xrsh_per_lane(a, b, 8, [](uint32_t x, uint32_t y) { return x == y ? 0xffu : 0u; }); }
static inline uint32_t __vcmpne4(uint32_t a, uint32_t b) { return xrsh_per_lane(a, b, 8, [](uint32_t x, uint32_t y) { return x != y ? 0xffu : 0u; }); }
static inline uint32_t __vcmpgtu4(uint32_t a, uint32_t b) { return xrsh_per_lane(a, b, 8, [](uint32_t x, uint32_t y) { return x > y ? 0xffu : 0u; }); }
static inline uint32_t __dp4a(uint32_t a, uint32_t b, uint32_t c) {
    for (int k = 0; k < 4; ++k) c += xrsh_lane_of(a, 8, k) * xrsh_lane_of(b, 8, k);
    return c;
}
namespace xrs {
static inline int fail(const std::string &msg) { xrsh_error = msg; return 1; }
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline double dadd(double a, double b) { return a + b; }
static inline double dsub(double a, double b) { return a - b; }
static inline double dmul(double a, double b) { return a * b; }
static inline double ddiv(double a, double b) { return a / b; }
}
#define XRS_CUDA(expr) do { int _rc = (expr); if (_rc) return _rc; } while (0)
#define XRS_LAUNCH_CHECK(name) do { } while (0)
#define XRS_TIMED(name, st, ...) do { xrsh_log.push_back(name); __VA_ARGS__; } while (0)
template <typename... P, typename... A>
static void xrsh_launch(dim3 grid, dim3 block, size_t, cudaStream_t, void (*kernel)(P...), A... args) {
    const std::tuple<P...> params(args...);
    const unsigned threads = block.x * block.y * block.z;
    assert(threads % 32 == 0);
    pthread_barrier_init(&xrsh_warp_bar, nullptr, 32);
    std::vector<std::thread> lanes;
    for (int lane = 0; lane < 32; ++lane)
        lanes.emplace_back([&, lane] {
            xrsh_lane = lane;
            gridDim = grid;
            blockDim = block;
            for (unsigned bz = 0; bz < grid.z; ++bz)
                for (unsigned by = 0; by < grid.y; ++by)
                    for (unsigned bx = 0; bx < grid.x; ++bx)
                        for (unsigned t = static_cast<unsigned>(lane); t < threads; t += 32) {
                            blockIdx = dim3(bx, by, bz);
                            threadIdx = dim3(t % block.x, (t / block.x) % block.y, t / (block.x * block.y));
                            std::apply(kernel, params);
                        }
        });
    for (auto &l : lanes) l.join();
    pthread_barrier_destroy(&xrsh_warp_bar);
}
"""

RSK_EXPORT = r"""
// k5_u8x4_reduce launched directly, as launch_affine_fast would for F = 2 / 4 / 8: its median / mode branches are
// kept for layouts k5_u8x2_sort declines, which the present dispatch never produces
extern "C" int xrsh_u8x4(const uint8_t *src, void *dst, int f, long n, long h, long w, long pitch, long sstride, int agg) {
    xrs::FastGeom g = {};
    g.n_slices = n; g.src_h = h; g.src_w = w; g.src_pitch = pitch; g.src_slice_stride = sstride;
    g.dst_h = h / f; g.dst_w = w / f; g.agg = agg; g.vec = 1;
    switch (f) {
    case 2: return xrs::launch_u8x4<2>(src, dst, g, nullptr);
    case 4: return xrs::launch_u8x4<4>(src, dst, g, nullptr);
    case 8: return xrs::launch_u8x4<8>(src, dst, g, nullptr);
    }
    return 1;
}
// kernel names launched since the last call (';'-separated), misaligned loads, last error message; resets all three
extern "C" long xrsh_take_log(char *names, long cap, char *err, long err_cap) {
    std::string s;
    for (const auto &n : xrsh_log) s += (s.empty() ? "" : ";") + n;
    std::snprintf(names, static_cast<size_t>(cap), "%s", s.c_str());
    std::snprintf(err, static_cast<size_t>(err_cap), "%s", xrsh_error.c_str());
    const long m = xrsh_misaligned;
    xrsh_log.clear(); xrsh_error.clear(); xrsh_misaligned = 0;
    return m;
}
// the SIMD intrinsics on word arrays: op 0 byte_perm(a, b, c), 1 vminu4, 2 vmaxu4, 3 vminu2, 4 vmaxu2, 5 vhaddu4,
// 6 vadd4, 7 vcmpeq4, 8 vcmpne4, 9 vcmpgtu4, 10 dp4a(a, b, c)
extern "C" int xrsh_simd(int op, const uint32_t *a, const uint32_t *b, const uint32_t *c, uint32_t *out, long n) {
    for (long k = 0; k < n; ++k) {
        switch (op) {
        case 0: out[k] = __byte_perm(a[k], b[k], c[k]); break;
        case 1: out[k] = __vminu4(a[k], b[k]); break;
        case 2: out[k] = __vmaxu4(a[k], b[k]); break;
        case 3: out[k] = __vminu2(a[k], b[k]); break;
        case 4: out[k] = __vmaxu2(a[k], b[k]); break;
        case 5: out[k] = __vhaddu4(a[k], b[k]); break;
        case 6: out[k] = __vadd4(a[k], b[k]); break;
        case 7: out[k] = __vcmpeq4(a[k], b[k]); break;
        case 8: out[k] = __vcmpne4(a[k], b[k]); break;
        case 9: out[k] = __vcmpgtu4(a[k], b[k]); break;
        case 10: out[k] = __dp4a(a[k], b[k], c[k]); break;
        default: return 1;
        }
    }
    return 0;
}
"""

SIMD_OPS = ("byte_perm", "vminu4", "vmaxu4", "vminu2", "vmaxu2", "vhaddu4", "vadd4", "vcmpeq4", "vcmpne4", "vcmpgtu4",
            "dp4a")


def _without_include(text: str, inc: str, what: str) -> str:
    text, n = re.subn(r"#include " + re.escape(inc) + r"\n", "", text)
    assert n == 1, f"{what} no longer includes {inc} exactly once"
    return text


def build_resample_kernels(out_dir: str) -> str:
    """Host build of resample_common.cuh + resample_fast.cu + resample.cu, kernels, launch code and the C ABI
    functions xrs_affine / xrs_coarsen / xrs_affine_recover / xrs_has_nan."""
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    common = _without_include(open(os.path.join(CSRC, "common.cuh")).read(), '"xrs.h"', "common.cuh")
    m = re.search(r"#define XRS_DISPATCH_DTYPE\(.*?\n    }\n", common, re.S)
    assert m, "XRS_DISPATCH_DTYPE moved"
    dispatch = m.group(0)
    rc = _without_include(open(os.path.join(CSRC, "resample_common.cuh")).read(), '"common.cuh"', "resample_common.cuh")
    rc = rc.replace("#pragma once\n", "")
    units = []
    for name in ("resample_fast.cu", "resample.cu"):
        text = _without_include(open(os.path.join(CSRC, name)).read(), '"resample_common.cuh"', name)
        text, n = re.subn(r"([A-Za-z_]\w*(?:<[^<>;()]*>)?)<<<([^<>;]*?)>>>\(\s*", r"xrsh_launch(\2, &\1, ", text)
        assert n > 0 and "<<<" not in text, f"launch syntax of {name} changed"
        units.append(text)
    src = os.path.join(out_dir, "resample_kernels_host.cpp")
    with open(src, "w") as fh:
        fh.write(RSK_SHIM + dispatch + "\n" + rc + "".join(units) + RSK_EXPORT)
    so = os.path.join(out_dir, "libxrs_rskhost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off", "-Wl,-Bsymbolic",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of resample.cu / resample_fast.cu failed:\n" + res.stderr[-6000:])
    return so


def aligned_view(a, pitch: int, slice_stride: int, elem_off: int, base_align: int = 256):
    """(n, h, w) copy of ``a`` in a fresh buffer whose first element sits ``elem_off`` elements past a
    ``base_align``-byte boundary, rows ``pitch`` and slices ``slice_stride`` elements apart."""
    a = np.asarray(a)
    n, h, w = a.shape
    es = a.dtype.itemsize
    nbytes = (elem_off + (n - 1) * slice_stride + (h - 1) * pitch + w) * es
    raw = np.zeros(nbytes + base_align, dtype=np.uint8)
    start = (-raw.ctypes.data) % base_align
    flat = raw[start:start + nbytes].view(a.dtype)
    view = np.lib.stride_tricks.as_strided(flat[elem_off:], (n, h, w), (slice_stride * es, pitch * es, es))
    view[...] = a
    return view


class ResampleKernels:
    """The C ABI of the affine / coarsen family on host buffers through :func:`build_resample_kernels`.  Every call
    returns ``(out, kernels, misaligned)``: the kernel names launched and the number of misaligned loads."""

    def __init__(self, so_path: str):
        self.lib = ctypes.CDLL(so_path)
        c_d, c_i, c_l, c_p, c_64 = ctypes.c_double, ctypes.c_int32, ctypes.c_long, ctypes.c_void_p, ctypes.c_int64
        self.lib.xrs_affine.restype = ctypes.c_int
        self.lib.xrs_affine.argtypes = [c_p, c_p, c_i] + [c_64] * 7 + [c_d] * 4 + [c_i, c_d, c_i, c_i, c_i, c_i, c_p]
        self.lib.xrs_affine_recover.restype = ctypes.c_int
        self.lib.xrs_affine_recover.argtypes = [c_p, c_p, c_i] + [c_64] * 7 + [c_d] * 5 + [c_i, c_i, c_i, c_i, c_p]
        self.lib.xrs_coarsen.restype = ctypes.c_int
        self.lib.xrs_coarsen.argtypes = [c_p, c_p, c_i] + [c_64] * 5 + [c_i, c_i, c_i, c_p]
        self.lib.xrs_has_nan.restype = ctypes.c_int
        self.lib.xrs_has_nan.argtypes = [c_p, c_i] + [c_64] * 5 + [c_p, c_p]
        self.lib.xrsh_take_log.restype = c_l
        self.lib.xrsh_take_log.argtypes = [c_p, c_l, c_p, c_l]
        self.lib.xrsh_u8x4.restype = ctypes.c_int
        self.lib.xrsh_u8x4.argtypes = [c_p, c_p, c_i] + [c_l] * 5 + [c_i]
        self.lib.xrsh_simd.restype = ctypes.c_int
        self.lib.xrsh_simd.argtypes = [ctypes.c_int, c_p, c_p, c_p, c_p, c_l]
        self.take()

    def take(self):
        names, err = ctypes.create_string_buffer(1 << 16), ctypes.create_string_buffer(1024)
        mis = self.lib.xrsh_take_log(names, 1 << 16, err, 1024)
        kernels = [k for k in names.value.decode().split(";") if k]
        return kernels, int(mis), err.value.decode()

    def _finish(self, rc, out, what):
        kernels, mis, err = self.take()
        if rc:
            raise RuntimeError(f"{what} failed: {err}")
        return out, kernels, mis

    @staticmethod
    def _geom(view):
        """What the Python layer passes (affine.py): row pitch, and the slice stride (h * pitch for one slice)."""
        n, h, w = view.shape
        es = view.dtype.itemsize
        pitch = view.strides[1] // es
        return n, h, w, pitch, (view.strides[0] // es if n > 1 else h * pitch)

    def affine(self, view, scale_ji, offset_ji, out_hw, order, cval, agg="mean", factors=(1, 1), slice_blend=False):
        from xcube_resampling_b200.constants import AGG_CODES, DTYPE_CODES

        n, h, w, pitch, sstride = self._geom(view)
        f_j, f_i = int(factors[0]), int(factors[1])
        is_float = view.dtype.kind == "f"
        i64 = f_j * f_i > 1 and (agg in ("mode", "count") or (not is_float and agg in ("sum", "prod")))
        out = aligned_view(np.zeros((n, int(out_hw[0]), int(out_hw[1])), np.int64 if i64 else view.dtype),
                           int(out_hw[1]), int(out_hw[0]) * int(out_hw[1]), 0)
        rc = self.lib.xrs_affine(view.ctypes.data, out.ctypes.data, DTYPE_CODES[view.dtype], n, h, w, pitch, sstride,
                                 int(out_hw[0]), int(out_hw[1]), float(scale_ji[0]), float(offset_ji[0]),
                                 float(scale_ji[1]), float(offset_ji[1]), int(order), float(cval), AGG_CODES[agg], f_j, f_i,
                                 int(bool(slice_blend)), None)
        return self._finish(rc, out, "xrs_affine")

    def affine_recover(self, view, scale_ji, offset_ji, out_hw, cval, agg="mean", factors=(1, 1), slice_blend=False):
        from xcube_resampling_b200.constants import AGG_CODES, DTYPE_CODES

        n, h, w, pitch, sstride = self._geom(view)
        out = aligned_view(np.zeros((n, int(out_hw[0]), int(out_hw[1]))), int(out_hw[1]), int(out_hw[0]) * int(out_hw[1]), 0)
        rc = self.lib.xrs_affine_recover(view.ctypes.data, out.ctypes.data, DTYPE_CODES[view.dtype], n, h, w, pitch,
                                         sstride, int(out_hw[0]), int(out_hw[1]), float(scale_ji[0]), float(offset_ji[0]),
                                         float(scale_ji[1]), float(offset_ji[1]), float(cval), AGG_CODES[agg],
                                         int(factors[0]), int(factors[1]), int(bool(slice_blend)), None)
        return self._finish(rc, out, "xrs_affine_recover")

    def coarsen(self, view, factors, agg):
        from xcube_resampling_b200.constants import AGG_CODES, DTYPE_CODES

        n, h, w, pitch, sstride = self._geom(view)
        f_j, f_i = int(factors[0]), int(factors[1])
        i64 = agg in ("mode", "count") or (view.dtype.kind != "f" and agg in ("sum", "prod"))
        oh, ow = h // f_j, w // f_i
        out = aligned_view(np.zeros((n, oh, ow), np.int64 if i64 else view.dtype), ow, oh * ow, 0)
        rc = self.lib.xrs_coarsen(view.ctypes.data, out.ctypes.data, DTYPE_CODES[view.dtype], n, h, w, pitch, sstride,
                                  AGG_CODES[agg], f_j, f_i, None)
        return self._finish(rc, out, "xrs_coarsen")

    def u8x4(self, view, f, agg):
        """k5_u8x4_reduce on its own (every aggregation it implements, median and mode included)."""
        from xcube_resampling_b200.constants import AGG_CODES

        n, h, w, pitch, sstride = self._geom(view)
        i64 = agg in ("mode", "count", "sum")
        out = aligned_view(np.zeros((n, h // f, w // f), np.int64 if i64 else np.uint8), w // f, (h // f) * (w // f), 0)
        rc = self.lib.xrsh_u8x4(view.ctypes.data, out.ctypes.data, int(f), n, h, w, pitch, sstride, AGG_CODES[agg])
        return self._finish(rc, out, "k5_u8x4_reduce")

    def has_nan(self, view):
        from xcube_resampling_b200.constants import DTYPE_CODES

        n, h, w, pitch, sstride = self._geom(view)
        flag = np.full(1, 7, dtype=np.int32)
        rc = self.lib.xrs_has_nan(view.ctypes.data, DTYPE_CODES[view.dtype], n, h, w, pitch, sstride, flag.ctypes.data, None)
        return self._finish(rc, bool(flag[0]), "xrs_has_nan")

    def simd(self, op: str, a, b, c=None) -> np.ndarray:
        a = np.ascontiguousarray(a, dtype=np.uint32)
        b = np.ascontiguousarray(b, dtype=np.uint32)
        c = np.ascontiguousarray(np.zeros_like(a) if c is None else c, dtype=np.uint32)
        out = np.empty_like(a)
        rc = self.lib.xrsh_simd(SIMD_OPS.index(op), a.ctypes.data, b.ctypes.data, c.ctypes.data, out.ctypes.data, a.size)
        assert rc == 0
        return out
