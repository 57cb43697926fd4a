// The device image of rrt_scene_update_mesh (mesh_update.hpp): upload, the re-bake of one mesh's primitives, the
// reductions that fix the node frame and format, and the gather of the primitive records in tree order.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>

#include "bake_core.h"
#include "device_layout.h"
#include "mesh_update.hpp"
#include "reduce.cuh"

namespace rrt {

namespace {

#define MU_CUDA(call)                                                           \
    do {                                                                        \
        cudaError_t e_ = (call);                                                \
        if (e_ != cudaSuccess) {                                                \
            if (err) *err = std::string(#call) + ": " + cudaGetErrorString(e_); \
            return RRT_ERR_CUDA;                                                \
        }                                                                       \
    } while (0)

struct FrameSums {
    double lo[3], hi[3];
    double growth;
    uint32_t inexact, pad;
};

// grid-stride kernels over the primitives: every warp of the grid reaches the shuffles of the reductions
unsigned reduce_blocks(size_t n) { return (unsigned)std::min<size_t>((n + 255) / 256, 1024); }

// One thread per triangle of the mesh's runs (binary search for the run): the host bake's arithmetic (bake_core.h).
__global__ void __launch_bounds__(256) rebake_kernel(const MeshImage::Run* __restrict__ runs, uint32_t n_runs, uint32_t total,
                                                      const double* __restrict__ p, const uint32_t* __restrict__ vi,
                                                      BakedPrim* __restrict__ world, Aabb* __restrict__ box,
                                                      uint8_t* __restrict__ exact) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total) return;
    uint32_t lo = 0, hi = n_runs - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) / 2;
        if (runs[mid].offset <= g) lo = mid;
        else hi = mid - 1;
    }
    const MeshImage::Run& r = runs[lo];
    const uint32_t k = g - r.offset, prim = r.first_prim + k;
    double v[9];
    bake::world_triangle(p, vi, r.first_tri + k, r.has_m ? r.m : nullptr, v);
    for (int j = 0; j < 9; ++j) world[prim].v[j] = v[j];
    bake::triangle_box(v, box[prim].lo, box[prim].hi);
    exact[prim] = bake::fp32_exact(v, 9) ? 1 : 0;
}

__global__ void __launch_bounds__(256) frame_kernel(uint64_t n, const Aabb* __restrict__ box, const uint8_t* __restrict__ exact,
                                                     FrameSums* __restrict__ out) {
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    bool inexact = false;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        for (int k = 0; k < 3; ++k) {
            lo[k] = fmin(lo[k], box[i].lo[k]);
            hi[k] = fmax(hi[k], box[i].hi[k]);
        }
        inexact |= exact[i] == 0;
    }
    for (int k = 0; k < 3; ++k) {
        lo[k] = warp_min_f64(lo[k]);
        hi[k] = warp_max_f64(hi[k]);
    }
    inexact = __any_sync(0xffffffffu, inexact);
    if ((threadIdx.x & 31u) == 0) {
        for (int k = 0; k < 3; ++k) {
            atomic_min_f64(&out->lo[k], lo[k]);
            atomic_max_f64(&out->hi[k], hi[k]);
        }
        if (inexact) atomicOr(&out->inexact, 1u);
    }
}

__global__ void __launch_bounds__(256) growth_kernel(uint64_t n, const Aabb* __restrict__ box, double cells, FrameSums* __restrict__ out) {
    double part = 0.0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const Aabb& b = box[i];
        const double hp = (b.hi[0] - b.lo[0]) + (b.hi[1] - b.lo[1]) + (b.hi[2] - b.lo[2]);
        part += fmin(1.0, cells / fmax(hp, 1e-300));
    }
    part = warp_sum_f64(part);
    if ((threadIdx.x & 31u) == 0) atomicAdd(&out->growth, part);
}

// DeviceAggregate::build's make_record, one slot per thread
template <bool WIDE>
__global__ void __launch_bounds__(256) gather_kernel(uint32_t n, const uint32_t* __restrict__ order, const BakedPrim* __restrict__ world,
                                                      const uint8_t* __restrict__ kind, const uint32_t* __restrict__ inst,
                                                      void* __restrict__ out) {
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n) return;
    const uint32_t pi = order[slot];
    const BakedPrim& w = world[pi];
    if (WIDE) {
        PrimRec96 r;
        for (int j = 0; j < 9; ++j) r.v[j] = w.v[j];
        r.prim_id = pi;
        r.kind = kind[pi];
        r.pad[0] = inst[pi];
        r.pad[1] = r.pad[2] = r.pad[3] = 0;
        static_cast<PrimRec96*>(out)[slot] = r;
    } else {
        PrimRec48 r;
        for (int j = 0; j < 12; ++j) r.words[j] = 0;
        if (kind[pi] == PRIM_TRIANGLE) {
            for (int j = 0; j < 3; ++j) {
                r.tri.v0[j] = (float)w.v[j];
                r.tri.v1[j] = (float)w.v[3 + j];
                r.tri.v2[j] = (float)w.v[6 + j];
            }
            r.tri.prim_id = pi;
            r.tri.kind = PRIM_TRIANGLE;
        } else {
            for (int j = 0; j < 3; ++j) r.sph.c[j] = w.v[j];
            r.sph.radius = w.v[3];
            r.sph.prim_id = pi;
            r.sph.kind = kind[pi];
            r.sph.instance = inst[pi];
        }
        static_cast<PrimRec48*>(out)[slot] = r;
    }
}

}  // namespace

MeshImage::~MeshImage() {
    cudaFree(d_world_);
    cudaFree(d_box_);
    cudaFree(d_kind_);
    cudaFree(d_exact_);
    cudaFree(d_inst_);
    cudaFree(d_red_);
    for (Mesh& m : meshes_) {
        cudaFree(m.d_p);
        cudaFree(m.d_vi);
        cudaFree(m.d_runs);
    }
}

int MeshImage::create(int device, const HostScene& scene, std::string* err) {
    device_ = device;
    n_ = scene.prims.size();
    WorldBake bake(n_);
    if (int rc = bake_world(scene, &bake, err)) return rc;
    std::vector<uint32_t> inst(n_);
    // the runs: consecutive triangles of one mesh under one instance (each rrt_scene_add_triangles call makes one per
    // instance, or one for the bare mesh)
    std::vector<std::vector<Run>> runs(scene.meshes.size());
    for (size_t i = 0; i < n_; ++i) {
        const Primitive& pr = scene.prims[i];
        inst[i] = pr.instance >= 0 ? (uint32_t)pr.instance : 0xFFFFFFFFu;
        if (pr.kind != SHAPE_TRIANGLE) continue;
        std::vector<Run>& rs = runs[pr.shape];
        if (!rs.empty()) {
            Run& last = rs.back();
            const Primitive& prev = scene.prims[i - 1];
            if (last.first_prim + last.count == i && prev.kind == SHAPE_TRIANGLE && prev.shape == pr.shape &&
                prev.instance == pr.instance && prev.tri + 1 == pr.tri) {
                last.count += 1;
                continue;
            }
        }
        Run r{};
        r.first_prim = (uint32_t)i;
        r.first_tri = pr.tri;
        r.count = 1;
        r.has_m = pr.instance >= 0 ? 1 : 0;
        if (pr.instance >= 0) std::memcpy(r.m, &scene.instances[pr.instance].m.m[0][0], sizeof(r.m));
        rs.push_back(r);
    }
    MU_CUDA(cudaSetDevice(device));
    MU_CUDA(cudaMalloc(&d_world_, n_ * sizeof(BakedPrim)));
    MU_CUDA(cudaMalloc(&d_box_, n_ * sizeof(Aabb)));
    MU_CUDA(cudaMalloc(&d_kind_, n_));
    MU_CUDA(cudaMalloc(&d_exact_, n_));
    MU_CUDA(cudaMalloc(&d_inst_, n_ * sizeof(uint32_t)));
    MU_CUDA(cudaMalloc(&d_red_, sizeof(FrameSums)));
    MU_CUDA(cudaMemcpy(d_world_, bake.world.get(), n_ * sizeof(BakedPrim), cudaMemcpyHostToDevice));
    MU_CUDA(cudaMemcpy(d_box_, bake.boxes.get(), n_ * sizeof(Aabb), cudaMemcpyHostToDevice));
    MU_CUDA(cudaMemcpy(d_kind_, bake.kind.get(), n_, cudaMemcpyHostToDevice));
    MU_CUDA(cudaMemcpy(d_exact_, bake.exact.get(), n_, cudaMemcpyHostToDevice));
    MU_CUDA(cudaMemcpy(d_inst_, inst.data(), n_ * sizeof(uint32_t), cudaMemcpyHostToDevice));
    meshes_.resize(scene.meshes.size());
    for (size_t m = 0; m < scene.meshes.size(); ++m) {
        const TriangleMesh& tm = scene.meshes[m];
        Mesh& dm = meshes_[m];
        MU_CUDA(cudaMalloc(&dm.d_p, tm.p.size() * sizeof(double)));
        MU_CUDA(cudaMemcpy(dm.d_p, tm.p.data(), tm.p.size() * sizeof(double), cudaMemcpyHostToDevice));
        MU_CUDA(cudaMalloc(&dm.d_vi, tm.vi.size() * sizeof(uint32_t)));
        MU_CUDA(cudaMemcpy(dm.d_vi, tm.vi.data(), tm.vi.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
        uint32_t offset = 0;
        for (Run& r : runs[m]) {
            r.offset = offset;
            offset += r.count;
        }
        dm.n_runs = (uint32_t)runs[m].size();
        dm.n_prims = offset;
        if (dm.n_runs) {
            MU_CUDA(cudaMalloc(&dm.d_runs, runs[m].size() * sizeof(Run)));
            MU_CUDA(cudaMemcpy(dm.d_runs, runs[m].data(), runs[m].size() * sizeof(Run), cudaMemcpyHostToDevice));
        }
    }
    has_spheres = bake.has_spheres;
    inst_w2p = std::move(bake.inst_w2p);
    gspheres = std::move(bake.gspheres);
    return RRT_OK;
}

int MeshImage::rebake(uint32_t mesh, std::string* err) {
    const Mesh& m = meshes_[mesh];
    if (m.n_prims == 0) return RRT_OK;
    MU_CUDA(cudaSetDevice(device_));
    rebake_kernel<<<(m.n_prims + 255) / 256, 256>>>(m.d_runs, m.n_runs, m.n_prims, m.d_p, m.d_vi, d_world_, d_box_, d_exact_);
    MU_CUDA(cudaGetLastError());
    return RRT_OK;
}

int MeshImage::frame(Aabb* world_box, bool* all_fp32, std::string* err) {
    FrameSums s = {{INFINITY, INFINITY, INFINITY}, {-INFINITY, -INFINITY, -INFINITY}, 0.0, 0u, 0u};
    FrameSums* d = static_cast<FrameSums*>(d_red_);
    MU_CUDA(cudaMemcpy(d, &s, sizeof(s), cudaMemcpyHostToDevice));
    frame_kernel<<<reduce_blocks(n_), 256>>>(n_, d_box_, d_exact_, d);
    MU_CUDA(cudaGetLastError());
    MU_CUDA(cudaMemcpy(&s, d, sizeof(s), cudaMemcpyDeviceToHost));
    for (int k = 0; k < 3; ++k) {
        world_box->lo[k] = s.lo[k];
        world_box->hi[k] = s.hi[k];
    }
    *all_fp32 = s.inexact == 0;
    return RRT_OK;
}

int MeshImage::growth(double cells, double* sum, std::string* err) {
    FrameSums* d = static_cast<FrameSums*>(d_red_);
    MU_CUDA(cudaMemset(&d->growth, 0, sizeof(double)));
    growth_kernel<<<reduce_blocks(n_), 256>>>(n_, d_box_, cells, d);
    MU_CUDA(cudaGetLastError());
    MU_CUDA(cudaMemcpy(sum, &d->growth, sizeof(double), cudaMemcpyDeviceToHost));
    return RRT_OK;
}

int MeshImage::gather(const uint32_t* d_order, bool wide, void* d_records, std::string* err) {
    const unsigned blocks = (unsigned)((n_ + 255) / 256);
    if (wide) gather_kernel<true><<<blocks, 256>>>((uint32_t)n_, d_order, d_world_, d_kind_, d_inst_, d_records);
    else gather_kernel<false><<<blocks, 256>>>((uint32_t)n_, d_order, d_world_, d_kind_, d_inst_, d_records);
    MU_CUDA(cudaGetLastError());
    return RRT_OK;
}

}  // namespace rrt
