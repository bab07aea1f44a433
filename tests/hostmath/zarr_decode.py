"""Host build of csrc/decode.cu: the kernels, their launch code and the C ABI functions xrs_zarr_decode /
xrs_zarr_decode_workspace_bytes compiled unchanged for the CPU, on the shim of
:func:`tests.hostmath.build_resample_kernels`.  Each launch runs as 32 host threads, one per lane, so the lanes of a
warp run concurrently and meet at every ``__syncwarp`` (a barrier of the 32 threads); device buffers are host
buffers and the table copy is a memcpy."""

from __future__ import annotations

import os
import re
import shutil
import subprocess

from . import CSRC, ROOT, RSK_SHIM, _without_include

DECODE_SHIM = r"""
static inline void __syncwarp(unsigned = 0xffffffffu) { pthread_barrier_wait(&xrsh_warp_bar); }
static inline uint32_t atomicCAS(uint32_t *p, uint32_t cmp, uint32_t v) {
    __atomic_compare_exchange_n(p, &cmp, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED);
    return cmp;
}
static inline float __fmul_rn(float a, float b) { return a * b; }
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline int __float_as_int(float v) { int i; std::memcpy(&i, &v, 4); return i; }
static inline float __int_as_float(int i) { float v; std::memcpy(&v, &i, 4); return v; }
static inline long long __double_as_longlong(double v) { long long i; std::memcpy(&i, &v, 8); return i; }
static inline double __longlong_as_double(long long i) { double v; std::memcpy(&v, &i, 8); return v; }
enum { cudaMemcpyHostToDevice = 1 };
// CUDA's launch limits (grid.x < 2^31, grid.y / grid.z <= 65535, <= 1024 threads a block): a launch beyond them fails
// on the device with "invalid configuration argument"; here it is counted and skipped (xrsh_bad_launches)
static long xrsh_bad = 0;
template <typename... P, typename... A>
static void xrshd_launch(dim3 grid, dim3 block, size_t smem, cudaStream_t st, void (*kernel)(P...), A... args) {
    if (grid.x == 0 || grid.y == 0 || grid.z == 0 || grid.x > 2147483647u || grid.y > 65535u || grid.z > 65535u ||
        block.x * block.y * block.z > 1024u) {
        ++xrsh_bad;
        return;
    }
    xrsh_launch(grid, block, smem, st, kernel, args...);
}

static inline int cudaMemcpyAsync(void *d, const void *s, size_t n, int, cudaStream_t) { std::memcpy(d, s, n); return 0; }
"""

DECODE_EXPORT = r"""
// kernel names launched since the last call (';'-separated) and the last error message; resets both
extern "C" long xrsh_take_log(char *names, long cap, char *err, long err_cap) {
    std::string s;
    for (const auto &n : xrsh_log) s += (s.empty() ? "" : ";") + n;
    std::snprintf(names, static_cast<size_t>(cap), "%s", s.c_str());
    std::snprintf(err, static_cast<size_t>(err_cap), "%s", xrsh_error.c_str());
    xrsh_log.clear(); xrsh_error.clear();
    return 0;
}
extern "C" const char *xrs_last_error(void) { return xrsh_error.c_str(); }
// launches refused by CUDA's limits since the last call; resets the count
extern "C" long xrsh_bad_launches(void) { const long n = xrsh_bad; xrsh_bad = 0; return n; }
"""


def build_decode(out_dir: str) -> str:
    gxx = shutil.which("g++")
    if gxx is None:
        raise RuntimeError("g++ not available")
    common = _without_include(open(os.path.join(CSRC, "common.cuh")).read(), '"xrs.h"', "common.cuh")
    m = re.search(r"#define XRS_DISPATCH_DTYPE\(.*?\n    }\n", common, re.S)
    assert m, "XRS_DISPATCH_DTYPE moved"
    text = _without_include(open(os.path.join(CSRC, "decode.cu")).read(), '"common.cuh"', "decode.cu")
    text, n = re.subn(r"([A-Za-z_]\w*(?:<[^<>;()]*>)?)<<<([^<>;]*?)>>>\(\s*", r"xrshd_launch(\2, &\1, ", text)
    assert n == 3 and "<<<" not in text, "launch syntax of decode.cu changed"
    src = os.path.join(out_dir, "decode_host.cpp")
    with open(src, "w") as fh:
        fh.write(RSK_SHIM + DECODE_SHIM + m.group(0) + "\n" + text + DECODE_EXPORT)
    so = os.path.join(out_dir, "libxrs_decodehost.so")
    cmd = [gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-ffp-contract=off", "-Wl,-Bsymbolic",
           f"-I{os.path.join(ROOT, 'include')}", src, "-o", so]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("host build of decode.cu failed:\n" + res.stderr[-6000:])
    return so
