// Whole-array reductions of doubles for the build kernels: warp shuffles, then one atomic per warp into global memory.
// Minimum and maximum are exact in any order; a sum is not (its callers say why that is acceptable).
#pragma once
#include <cuda_runtime.h>

namespace rrt {

__device__ __forceinline__ double warp_min_f64(double v) {
    for (int off = 16; off > 0; off >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}
__device__ __forceinline__ double warp_max_f64(double v) {
    for (int off = 16; off > 0; off >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}
__device__ __forceinline__ double warp_sum_f64(double v) {
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// *a = min(*a, v) / max(*a, v): a compare-and-swap only while v still improves on what is stored
__device__ __forceinline__ void atomic_min_f64(double* a, double v) {
    unsigned long long* p = reinterpret_cast<unsigned long long*>(a);
    unsigned long long old = *reinterpret_cast<volatile unsigned long long*>(p);
    while (v < __longlong_as_double((long long)old)) {
        const unsigned long long seen = atomicCAS(p, old, (unsigned long long)__double_as_longlong(v));
        if (seen == old) break;
        old = seen;
    }
}
__device__ __forceinline__ void atomic_max_f64(double* a, double v) {
    unsigned long long* p = reinterpret_cast<unsigned long long*>(a);
    unsigned long long old = *reinterpret_cast<volatile unsigned long long*>(p);
    while (v > __longlong_as_double((long long)old)) {
        const unsigned long long seen = atomicCAS(p, old, (unsigned long long)__double_as_longlong(v));
        if (seen == old) break;
        old = seen;
    }
}

}  // namespace rrt
