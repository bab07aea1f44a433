// common.cuh -- shared helpers of libxrs.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <cstdio>
#include <limits>
#include <string>
#include <type_traits>

#include "xrs.h"

namespace xrs {

void set_error(const std::string &msg);
int fail(const std::string &msg);
int check_cuda(cudaError_t e, const char *what);

#define XRS_CUDA(expr)                                   \
    do {                                                 \
        int _rc = ::xrs::check_cuda((expr), #expr);      \
        if (_rc) return _rc;                             \
    } while (0)

void count_launch();

#define XRS_LAUNCH_CHECK(name)            \
    do {                                  \
        ::xrs::count_launch();            \
        XRS_CUDA((cudaGetLastError()));   \
    } while (0)

// Optional per-kernel timing (xrs_profile_enable): brackets one launch with CUDA events on its stream.
void profile_begin(const char *name, cudaStream_t st);
void profile_end(cudaStream_t st);
struct ProfileScope {
    cudaStream_t st;
    ProfileScope(const char *name, cudaStream_t s) : st(s) { profile_begin(name, s); }
    ~ProfileScope() { profile_end(st); }
};
#define XRS_TIMED(name, st, ...)                  \
    do {                                          \
        ::xrs::ProfileScope _xrs_ps((name), (st)); \
        __VA_ARGS__;                              \
    } while (0)

__host__ __device__ static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------
// fp64 arithmetic that must round exactly like the reference's numba / numpy
// code (no FMA contraction, SURVEY.md 7.3-3): explicit _rn intrinsics are never
// fused by nvcc regardless of -fmad.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double ddiv(double a, double b) { return __ddiv_rn(a, b); }

// ---------------------------------------------------------------------------
// mbarrier + bulk async copy (TMA engine, SASS UBLKCP) wrappers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
// Make freshly initialised mbarriers visible to other threads AND to the async proxy (the TMA
// engine completes transactions on them; without the proxy fence it faults on sm_100).
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a byte-count bug must trap, not hang the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 26)) {
            printf("xrs: mbarrier wait timed out (block %d,%d thread %d)\n", blockIdx.x, blockIdx.y, threadIdx.x);
            __trap();
        }
    }
}
// global -> shared bulk copy; dst, src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// streaming (read-once / write-once) accesses
template <typename T>
__device__ __forceinline__ T ld_stream(const T *p) {
    return __ldcs(p);
}
template <typename T>
__device__ __forceinline__ void st_stream(T *p, T v) {
    __stcs(p, v);
}

template <typename T>
struct DTypeOf;
template <> struct DTypeOf<float> { static constexpr int code = XRS_F32; };
template <> struct DTypeOf<double> { static constexpr int code = XRS_F64; };
template <> struct DTypeOf<uint8_t> { static constexpr int code = XRS_U8; };
template <> struct DTypeOf<int8_t> { static constexpr int code = XRS_I8; };
template <> struct DTypeOf<uint16_t> { static constexpr int code = XRS_U16; };
template <> struct DTypeOf<int16_t> { static constexpr int code = XRS_I16; };
template <> struct DTypeOf<int32_t> { static constexpr int code = XRS_I32; };
template <> struct DTypeOf<uint32_t> { static constexpr int code = XRS_U32; };
template <> struct DTypeOf<int64_t> { static constexpr int code = XRS_I64; };

static inline int dtype_size(int dtype) {
    switch (dtype) {
    case XRS_F64: case XRS_I64: return 8;
    case XRS_F32: case XRS_I32: case XRS_U32: return 4;
    case XRS_U16: case XRS_I16: return 2;
    case XRS_U8: case XRS_I8: return 1;
    default: return 0;
    }
}

#define XRS_DISPATCH_DTYPE(dtype, T, ...)                                   \
    switch (dtype) {                                                        \
    case XRS_F32: { using T = float; __VA_ARGS__; break; }                  \
    case XRS_F64: { using T = double; __VA_ARGS__; break; }                 \
    case XRS_U8: { using T = uint8_t; __VA_ARGS__; break; }                 \
    case XRS_I8: { using T = int8_t; __VA_ARGS__; break; }                  \
    case XRS_U16: { using T = uint16_t; __VA_ARGS__; break; }               \
    case XRS_I16: { using T = int16_t; __VA_ARGS__; break; }                \
    case XRS_I32: { using T = int32_t; __VA_ARGS__; break; }                \
    case XRS_U32: { using T = uint32_t; __VA_ARGS__; break; }               \
    case XRS_I64: { using T = int64_t; __VA_ARGS__; break; }                \
    default: return ::xrs::fail("unsupported dtype code " + std::to_string(dtype)); \
    }

}  // namespace xrs
