// The two streaming passes around the f64 walk for fp32 callers (include/rrt.h, rrt_intersect_f32 and relatives).
// One thread per record, 16-byte vector loads and stores; the conversions themselves are rays_f32.cuh's.  Kept apart
// from trace_kernel on purpose: 32 + 64 + 32 + 16 extra bytes of HBM traffic per ray against a walk that moves
// kilobytes, and no new variants of the hottest kernel.
#include <cuda_runtime.h>

#include "rays_f32.cuh"
#include "rays_f32.hpp"

namespace rrt {
namespace {

constexpr unsigned kThreads = 256;

__global__ void __launch_bounds__(kThreads) promote_rays_kernel(uint64_t n, const float4* __restrict__ in,
                                                                double2* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    union {
        float4 v[2];
        rrt_ray_f32 r;
    } a;
    a.v[0] = in[2 * i];
    a.v[1] = in[2 * i + 1];
    union {
        rrt_ray r;
        double2 v[4];
    } b;
    b.r = promote_ray(a.r);
#pragma unroll
    for (int k = 0; k < 4; ++k) out[4 * i + k] = b.v[k];
}

__global__ void __launch_bounds__(kThreads) compact_hits_kernel(uint64_t n, const double2* __restrict__ in,
                                                                uint4* __restrict__ out) {
    const uint64_t i = (uint64_t)blockIdx.x * kThreads + threadIdx.x;
    if (i >= n) return;
    union {
        double2 v[2];
        rrt_hit h;
    } a;
    a.v[0] = in[2 * i];
    a.v[1] = in[2 * i + 1];
    union {
        rrt_hit_f32 h;
        uint4 v;
    } b;
    b.h = compact_hit(a.h);
    out[i] = b.v;
}

unsigned blocks_for(uint64_t n) { return (unsigned)((n + kThreads - 1) / kThreads); }

}  // namespace

int launch_promote_rays(uint64_t n, const rrt_ray_f32* in, rrt_ray* out, void* stream) {
    if (n == 0) return cudaSuccess;
    promote_rays_kernel<<<blocks_for(n), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        n, reinterpret_cast<const float4*>(in), reinterpret_cast<double2*>(out));
    return cudaGetLastError();
}

int launch_compact_hits(uint64_t n, const rrt_hit* in, rrt_hit_f32* out, void* stream) {
    if (n == 0) return cudaSuccess;
    compact_hits_kernel<<<blocks_for(n), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        n, reinterpret_cast<const double2*>(in), reinterpret_cast<uint4*>(out));
    return cudaGetLastError();
}

}  // namespace rrt
