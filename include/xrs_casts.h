/*
 * xrs_casts.h -- the float64 -> dtype conversions of libxrs.so, for C++ (xrs.h includes this file when compiled as
 * C++).  They are what the ABI promises for `fill` arguments and for every float64 result a kernel stores into an
 * integer variable: the results the reference gets on x86-64.  The same text compiles for the device (nvcc) and
 * for the host, so host builds of the kernels convert exactly as the GPU does.
 */
#ifndef XRS_CASTS_H_
#define XRS_CASTS_H_

#include <stdint.h>

#include <type_traits>

#if defined(__CUDACC__)
#define XRS_CAST_FN __host__ __device__ __forceinline__
#else
#define XRS_CAST_FN inline
#endif

namespace xrs {

// float64 -> T the way numpy's astype and numba's stores do it on x86-64 (the reference assigns float64 results
// into arrays of the source dtype: rectify.py:734, reproject.py:299-300): types up to 32 bits go through a
// 32-bit cvttsd2si (uint32 through the 64-bit one), whose out-of-range / NaN result is the "integer indefinite"
// value 0x80000000 (0x8000000000000000), and are then truncated to the destination width.  So NaN gives
// INT32_MIN / INT64_MIN for int32 / int64 and 0 for the other integer types, and 2^63 gives INT64_MIN.  A plain
// C cast is undefined there, and the device's cvt.rzi saturates instead (2^63 -> INT64_MAX, NaN -> 0).
template <typename OUT>
XRS_CAST_FN OUT cast_like_numpy(double v) {
    if constexpr (std::is_floating_point<OUT>::value) {
        return static_cast<OUT>(v);
    } else if constexpr (sizeof(OUT) == 8 || std::is_same<OUT, uint32_t>::value) {
        const bool ok = v > -9223372036854775809.0 && v < 9223372036854775808.0;
        const long long w = ok ? static_cast<long long>(v) : static_cast<long long>(0x8000000000000000ull);
        return static_cast<OUT>(w);
    } else {
        const bool ok = v > -2147483649.0 && v < 2147483648.0;
        const int w = ok ? static_cast<int>(v) : static_cast<int>(0x80000000u);
        return static_cast<OUT>(w);
    }
}

// A fill value reaches the C ABI as a double (the Python layer passes float(fill_value)) and is converted like
// numpy's np.full(shape, float_value, dtype): NaN into an integer variable is cast_like_numpy's x86 result, -1.0
// into uint32 is 0xFFFFFFFF, and int64 fills beyond 2^53 arrive already rounded to the nearest double.
template <typename T>
XRS_CAST_FN T cast_fill(double fill) {
    return cast_like_numpy<T>(fill);
}

}  // namespace xrs

#undef XRS_CAST_FN
#endif /* XRS_CASTS_H_ */
