// Host BVH construction for the Tier-F ("fast") aggregate: a binned surface-area-heuristic
// binary tree over world-space primitive boxes, built top-down with the upper levels fanned
// out over host threads.  It replaces BVHAccel::hlbvh_build (src/bvh.rs:365-514) for the GPU
// path — Tier-F results are independent of tree topology (DESIGN.md §2), so the tree is chosen
// for traversal cost, not for likeness to the reference's Morton treelets.
#pragma once
#include <cstdint>
#include <memory>
#include <utility>
#include <vector>

#include "host_scene.hpp"

namespace rrt {

struct Bvh2Node {
    Aabb box;
    int32_t left = -1, right = -1;  // interior: child node indices
    uint32_t first = 0, count = 0;  // leaf: range in Bvh2::order
    // subtree totals (a leaf: n_interior = 0, n_prims = count): what lets the packer lay a subtree out without walking
    // the ones before it (bvh_pack_plan.hpp)
    uint32_t n_interior = 0, n_prims = 0;
};

// Allocator whose value-less construct() does nothing: resize() then leaves the elements uninitialised.  The builder
// writes every field of every node it hands out, on the thread that builds that node — a value-initialising resize of
// 8.4 M nodes was 0.3 s of one thread zero-filling (and page-faulting) half a gigabyte before the build could start.
template <class T>
struct NoInitAlloc : std::allocator<T> {
    template <class U>
    struct rebind {
        using other = NoInitAlloc<U>;
    };
    NoInitAlloc() = default;
    template <class U>
    NoInitAlloc(const NoInitAlloc<U>&) {}
    template <class U>
    void construct(U*) noexcept {}
    template <class U, class A0, class... Args>
    void construct(U* p, A0&& a0, Args&&... args) {
        ::new ((void*)p) U(std::forward<A0>(a0), std::forward<Args>(args)...);
    }
};

struct Bvh2 {
    std::vector<Bvh2Node, NoInitAlloc<Bvh2Node>> nodes;
    // primitive indices, leaf ranges are contiguous; with spatial splits a primitive may appear in several leaves, so this
    // holds the references (as many as nodes[root].n_prims), not one entry per primitive
    std::vector<uint32_t> order;
    uint32_t root = 0;
    uint32_t max_depth = 0;
    uint32_t n_leaves = 0;
};

struct SahParams {
    uint32_t max_leaf = 4;      // BVHAccel's max_prims_in_node (capped at 8 by the leaf encoding)
    double cost_traverse = 1.0;
    double cost_intersect = 2.0;
    int n_threads = 0;          // 0 = hardware_concurrency
    // Spatial splits (SBVH, Stich et al. 2009), used only when the builder is given triangle vertices: a node tries one
    // when its best object split's children overlap by more than split_alpha x the root's surface area, and the tree
    // holds at most split_cap x n references.  (DESIGN.md §3: measured on configs 3 and 5.)
    double split_alpha = 1e-5;
    double split_cap = 1.3;
};

// World-space triangle vertices for spatial splits: primitive i's are verts[9 i .. 9 i + 8] (v0, v1, v2) when
// is_tri is null or is_tri[i] != 0.  Other primitives (spheres) stay whole references.
struct SplitTriangles {
    const double* verts = nullptr;
    const uint8_t* is_tri = nullptr;
};

// object splits only: one reference per primitive
void build_sah(AabbSpan boxes, const SahParams& params, Bvh2* out);
// object and spatial splits: triangles may be referenced from several leaves, each time with the box of the part of
// the triangle inside that leaf
void build_sah(AabbSpan boxes, const SplitTriangles& tris, const SahParams& params, Bvh2* out);

}  // namespace rrt
