// The GPU aggregate: device-resident tree + primitive records and the launchers of the
// closest-hit / any-hit kernels.  Host-visible part (no CUDA types in the interface besides
// the opaque stream pointer) so capi.cpp can be compiled by the plain host compiler.
#pragma once
#include <chrono>
#include <cstdint>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/rrt.h"
#include "bvh_lbvh.hpp"
#include "bvh_sah.hpp"
#include "host_scene.hpp"

namespace rrt {

struct GenSphere;
class MeshImage;

struct AggregateStats {
    uint64_t n_nodes = 0, n_leaves = 0, max_depth = 0, device_bytes = 0, build_usec = 0, n_records = 0,
             wide_records = 0, n_prims = 0;
    uint64_t tree_device_usec = 0;  // RRT_BUILD_DEVICE_LBVH: keys -> emitted nodes on the GPU (CUDA events)
};

// Kernel-side view, passed by value to every launch.
struct AggView {
    const void* nodes;   // Node64[]
    const void* prims;   // PrimRec48[] or PrimRec96[]
    const double* inst_w2p;  // world->primitive 3x4 (row-major f64) per instance; sphere (u,v) only
    const void* gspheres;    // GenSphere[] (sphere_core.cuh): partial spheres and spheres under non-rigid transforms
    double world_lo[3];  // tight world box of the tree, used to pull far-away origins close
    double world_hi[3];
    double scene_scale;  // max |coordinate| of the world box
    double grid_c[3];    // Node32: quantisation grid, lo - extent per axis (plane = grid_c + f * grid_ext)
    float grid_ext[3];   //             extent per axis (an fp32 value)
    int32_t quantised;   // 1 => nodes is Node32[] (15-bit planes on the grid), 0 => Node64[]
    int32_t root;        // interior node index of the root (always 0)
    int32_t wide;        // 1 => PrimRec96
    int32_t has_spheres;
    int32_t sort_mode;   // ray-queue key: 0 cell, 1 cell|octant, 2 octant|cell
    int32_t reserved;    // always 0
};
// a kernel parameter, and copied whole into the header of an exported tree: its layout is part of the blob format
static_assert(sizeof(AggView) == 152, "AggView layout changed: exported trees would no longer import");

// What the C ABI and the renderer need from an aggregate: batches of closest-hit / any-hit
// queries, with the batch size on the host or in device memory.
class RayTracer {
  public:
    virtual ~RayTracer() = default;
    virtual int closest_hit(uint64_t n, const rrt_ray* d_rays, rrt_hit* d_hits, void* stream, std::string* err,
                            int* launches = nullptr) const = 0;
    virtual int any_hit(uint64_t n, const rrt_ray* d_rays, uint8_t* d_occluded, void* stream, std::string* err,
                        int* launches = nullptr) const = 0;
    virtual int closest_hit_indirect(uint64_t capacity, const uint32_t* d_count, const rrt_ray* d_rays, rrt_hit* d_hits,
                                     void* stream, std::string* err, int* launches = nullptr) const = 0;
    virtual int any_hit_indirect(uint64_t capacity, const uint32_t* d_count, const rrt_ray* d_rays, uint8_t* d_occluded,
                                 void* stream, std::string* err, int* launches = nullptr) const = 0;
    virtual const AggregateStats& stats() const = 0;
    virtual bool literal() const { return false; }
};

class DeviceAggregate : public RayTracer {
  public:
    DeviceAggregate() = default;
    ~DeviceAggregate();
    DeviceAggregate(const DeviceAggregate&) = delete;
    DeviceAggregate& operator=(const DeviceAggregate&) = delete;

    // Bake primitives to world space, build the SAH tree, pack Node64 / PrimRec and upload.
    // Returns an rrt_status; on failure *err holds the reason.
    // `device_lbvh`: build the tree on the GPU (bvh_lbvh.cu) instead of the host SAH builder.
    int build(int device, const HostScene& scene, uint32_t max_prims_in_node, std::string* err, bool device_lbvh = false);
    // Whether build(device_lbvh = true) makes the tree on the device for n primitives: more than 16, and more than one
    // leaf holds.  Otherwise it builds the host SAH tree.
    static bool device_tree_fits(size_t n, uint32_t max_prims_in_node);
    // The aggregate build(device_lbvh = true) makes, from a scene baked on the device (rrt_scene_update_mesh): world box,
    // node format, device LBVH and records, without the primitives going through the host.  For n that
    // device_tree_fits.  *too_deep: the radix tree is deeper than the traversal stack; nothing was built, and build()
    // (which falls back to the SAH tree) is the caller's answer.
    int build_from_image(int device, MeshImage& image, uint32_t max_prims_in_node, bool* too_deep, std::string* err);

    // Asynchronous on `stream`; *launches (optional) receives the number of kernels launched.
    int closest_hit(uint64_t n, const rrt_ray* d_rays, rrt_hit* d_hits, void* stream, std::string* err,
                    int* launches = nullptr) const override;
    int any_hit(uint64_t n, const rrt_ray* d_rays, uint8_t* d_occluded, void* stream, std::string* err,
                int* launches = nullptr) const override;

    // Wavefront queues: the number of rays is read from device memory (*d_count <= capacity), so a
    // whole bounce loop can be enqueued without a host round trip.
    int closest_hit_indirect(uint64_t capacity, const uint32_t* d_count, const rrt_ray* d_rays, rrt_hit* d_hits,
                             void* stream, std::string* err, int* launches = nullptr) const override;
    int any_hit_indirect(uint64_t capacity, const uint32_t* d_count, const rrt_ray* d_rays, uint8_t* d_occluded,
                         void* stream, std::string* err, int* launches = nullptr) const override;

    // The committed aggregate as a relocatable blob (header + node / record / instance / sphere tables) and back: one rank
    // builds, the others upload.  `buffer` = nullptr: only *bytes is set.
    int export_blob(void* buffer, uint64_t capacity, uint64_t* bytes, std::string* err) const;
    int import_blob(int device, const void* blob, uint64_t bytes, uint64_t n_prims_expected, std::string* err);

    const AggView& view() const { return view_; }
    const AggregateStats& stats() const override { return stats_; }

  private:
    // Scratch for the ray sort + the persistent kernel's cursor: one per stream that calls in (the host-buffer pipeline
    // of capi.cpp runs three), so that a chunk's sort does not wait for the previous chunk's walk; past kMaxWorkspaces
    // streams the first one is shared, ordered by an event.
    static constexpr size_t kMaxWorkspaces = 8;
    struct Workspace {
        uint32_t *d_bins = nullptr, *d_block_sums = nullptr, *d_key = nullptr, *d_rank = nullptr, *d_perm = nullptr;
        void* d_small = nullptr;
        uint64_t capacity = 0;
        struct CUevent_st* last_use = nullptr;
        bool used = false;
        void* last_stream = nullptr;
        int n_sms = 0;
    };
    int ensure_workspace(Workspace& w, uint64_t n, std::string* err) const;
    template <bool ANY>
    int trace(uint64_t n, const rrt_ray* d_rays, rrt_hit* d_hits, uint8_t* d_occ, void* stream, std::string* err,
              int* launches, const uint32_t* n_dev) const;
    mutable std::map<void*, Workspace> ws_;
    mutable std::mutex ws_mutex_;
    bool sort_rays_ = true;
    int stack_levels_ = 2;
    AggView view_{};
    AggregateStats stats_{};
    void* d_nodes_ = nullptr;
    void* d_prims_ = nullptr;
    void* d_inst_ = nullptr;
    void* d_gspheres_ = nullptr;
    uint64_t node_bytes_ = 0, prim_bytes_ = 0, inst_bytes_ = 0, gsphere_bytes_ = 0;
    int device_ = 0;
    void configure_kernels(bool quantised);
    int upload_tables(const std::vector<double>& inst_w2p, const std::vector<GenSphere>& gspheres, std::string* err);
    struct Built {
        Aabb world_box;
        NodeFrame frame;
        bool quantise, wide, has_spheres;
        uint64_t n_nodes, n_leaves, max_depth, tree_device_usec, node_bytes, prim_bytes, n_records, n_prims;
    };
    void install(const Built& b, std::chrono::steady_clock::time_point t_start);
};

}  // namespace rrt
