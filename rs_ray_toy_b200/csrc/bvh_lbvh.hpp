// Device LBVH builder (RRT_BUILD_DEVICE_LBVH) — see bvh_lbvh.cu / lbvh_core.h.
#pragma once
#include <cmath>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/rrt.h"
#include "host_scene.hpp"

namespace rrt {

// The numeric frame both builders pack nodes in (DESIGN.md §3): the fp32-rounding margin `delta` of Node64
// boxes and the 15-bit grid of Node32.
struct NodeFrame {
    double scale, delta;
    double grid_lo[3], grid_c[3];
    float grid_ext[3];
};
inline NodeFrame make_node_frame(const Aabb& world_box) {
    NodeFrame f;
    f.scale = 0.0;
    for (int k = 0; k < 3; ++k) f.scale = std::fmax(f.scale, std::fmax(std::fabs(world_box.lo[k]), std::fabs(world_box.hi[k])));
    if (!(f.scale > 0.0)) f.scale = 1.0;
    // Widening that absorbs every fp32 rounding of the slab test: the fp32 copy of the origin
    // (<= scale * 2^-24 after prepare_ray), of 1/d and of the products.
    f.delta = f.scale * std::ldexp(1.0, -19);
    for (int k = 0; k < 3; ++k) {
        // fp32-rounding margins around the root's (already widened) children, and an extent that is an fp32 value
        f.grid_lo[k] = world_box.lo[k] - 4.0 * f.delta;
        double ext = (world_box.hi[k] + 4.0 * f.delta) - f.grid_lo[k];
        ext = std::fmax(ext, f.scale * std::ldexp(1.0, -10));
        float e = (float)(ext * (1.0 + std::ldexp(1.0, -20)));
        if ((double)e < ext) e = std::nextafterf(e, INFINITY);
        f.grid_ext[k] = e;
        f.grid_c[k] = f.grid_lo[k] - (double)f.grid_ext[k];
    }
    return f;
}

struct LbvhResult {
    void* d_nodes = nullptr;  // Node32[] or Node64[] in device memory (caller owns)
    size_t node_bytes = 0;
    uint32_t n_nodes = 0, n_leaves = 0, max_depth = 0;
    std::vector<uint32_t> order;  // primitive index at every sorted position (= record order)
    const uint32_t* d_order = nullptr;  // build_lbvh_device_boxes: the same order in device memory, in the arena
    double root_lo[3], root_hi[3];
    float device_ms = 0.0f;       // keys -> emitted nodes, CUDA events
    uint64_t total_usec = 0;      // including allocations and transfers
};

// Device memory the builds over device boxes reuse: the scratch arrays, grown to the largest build, freed with it.
struct LbvhArena {
    void* d = nullptr;
    size_t bytes = 0;
    LbvhArena() = default;
    LbvhArena(const LbvhArena&) = delete;
    LbvhArena& operator=(const LbvhArena&) = delete;
    ~LbvhArena();
};

int build_lbvh_device(int device, AabbSpan boxes, uint32_t max_leaf, double delta, bool quantise,
                      const double grid_lo[3], const float grid_ext[3], LbvhResult* out, std::string* err);

// The same build from f64 boxes already in device memory (d_boxes[n]): the fp32 conversion and the centroid frame are
// made on the device, the scratch lives in *arena, and the order stays there (out->d_order, valid until the arena's
// next build; out->order is left empty).
int build_lbvh_device_boxes(int device, const Aabb* d_boxes, uint32_t n, uint32_t max_leaf, double delta, bool quantise,
                            const double grid_lo[3], const float grid_ext[3], LbvhArena* arena, LbvhResult* out,
                            std::string* err);

int lbvh_host_probe(const std::vector<Aabb>& boxes, uint32_t max_leaf, double delta, bool quantise, const double grid_lo[3],
                    const float grid_ext[3], std::vector<uint8_t>* nodes_out, std::vector<uint32_t>* order_out, uint32_t* depth_out,
                    uint32_t* leaves_out);

}  // namespace rrt
