// The surface pass of the intersect API (include/rrt.h, rrt_intersect_surface and rrt_intersect_surface_device): what
// BVHAccel::intersect leaves in `si` for the winning primitive (primitives.rs:56-57, interaction.rs:85-113), rebuilt
// from the f64 hit by the renderer's own make_surface_body in its FULL form, so there is one statement of the triangle,
// sphere and instance code (triangle.rs, sphere.rs:127-255, transform.rs:604-656) on the device.
//
// One thread per ray.  A record is 336 bytes, 42 doubles: a thread fills its record in shared memory (stride 43 doubles,
// odd, so that the 8-byte stores of a warp do not collide on banks), then the block writes its records out as one
// contiguous run, consecutive lanes on consecutive doubles: every store instruction of a warp covers 256 contiguous bytes.
#include <cuda_runtime.h>

#include <new>

#include "scene_tables.cuh"
#include "surface.hpp"

namespace rrt {

struct SurfaceTables {
    ShadeScene sc{};
    std::vector<void*> allocations;
};

namespace {

constexpr unsigned kThreads = 128;
constexpr unsigned kWords = sizeof(rrt_surface) / sizeof(double);  // 42
constexpr unsigned kStride = kWords + 1;
static_assert(sizeof(rrt_surface) == 336 && kWords * sizeof(double) == sizeof(rrt_surface), "rrt_surface layout");

__device__ __forceinline__ void put3(double* w, V3 v) {
    w[0] = v.x;
    w[1] = v.y;
    w[2] = v.z;
}

__global__ void __launch_bounds__(kThreads) surface_kernel(ShadeScene sc, uint64_t n, const double* __restrict__ rays,
                                                           const double* __restrict__ hits, double* __restrict__ out) {
    __shared__ double stage[kThreads * kStride];
    const uint64_t base = (uint64_t)blockIdx.x * kThreads;
    const uint64_t i = base + threadIdx.x;
    if (i < n) {
        double* w = stage + threadIdx.x * kStride;
        // the hit, word for word (prim_id and reserved share the first word)
        const double h0 = hits[4 * i], t = hits[4 * i + 1], bu = hits[4 * i + 2], bv = hits[4 * i + 3];
        w[0] = h0;
        w[1] = t;
        w[2] = bu;
        w[3] = bv;
        const uint32_t prim_id = (uint32_t)(unsigned long long)__double_as_longlong(h0);
        if (prim_id != RRT_NO_HIT) {
            const double* r = rays + 8 * i;
            Surface s;
            BumpPartials bp;
            GeomNormalPartials gp;
            make_surface_body<true>(sc, prim_id, t, bu, bv, v3(r[0], r[1], r[2]), v3(r[3], r[4], r[5]), &s, &bp, &gp);
            put3(w + 4, s.p);
            put3(w + 7, s.wo);
            put3(w + 10, s.n);
            w[13] = s.uv.x;
            w[14] = s.uv.y;
            put3(w + 15, s.dpdu);
            put3(w + 18, s.dpdv);
            put3(w + 21, gp.dndu);
            put3(w + 24, gp.dndv);
            put3(w + 27, s.shn);
            put3(w + 30, s.shdpdu);
            put3(w + 33, bp.shdpdv);
            put3(w + 36, bp.shdndu);
            put3(w + 39, bp.shdndv);
        } else {
#pragma unroll
            for (unsigned k = 4; k < kWords; ++k) w[k] = 0.0;
        }
    }
    __syncthreads();
    const uint64_t left = n - base;
    const unsigned words = (unsigned)(left < kThreads ? left : kThreads) * kWords;
    double* dst = out + base * kWords;
    for (unsigned j = threadIdx.x; j < words; j += kThreads) dst[j] = stage[(j / kWords) * kStride + j % kWords];
}

}  // namespace

int surface_tables_create(const HostScene& scene, SurfaceTables** out, std::string* err) {
    *out = nullptr;
    SurfaceTables* t = new (std::nothrow) SurfaceTables();
    if (!t) {
        if (err) *err = "out of host memory";
        return RRT_ERR_INVALID;
    }
    const int rc = upload_geometry_tables(scene, &t->sc, &t->allocations, err);
    if (rc != RRT_OK) {
        surface_tables_destroy(t);
        return rc;
    }
    *out = t;
    return RRT_OK;
}

void surface_tables_destroy(SurfaceTables* t) {
    if (!t) return;
    for (void* p : t->allocations) cudaFree(p);
    delete t;
}

const ShadeScene* surface_tables_view(const SurfaceTables* t) { return &t->sc; }

int launch_surfaces(const ShadeScene& tables, bool literal, uint64_t n, const rrt_ray* rays, const rrt_hit* hits,
                    rrt_surface* out, void* stream) {
    if (n == 0) return cudaSuccess;
    ShadeScene sc = tables;
    sc.literal = literal ? 1u : 0u;
    surface_kernel<<<(unsigned)((n + kThreads - 1) / kThreads), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        sc, n, reinterpret_cast<const double*>(rays), reinterpret_cast<const double*>(hits), reinterpret_cast<double*>(out));
    return cudaGetLastError();
}

}  // namespace rrt
