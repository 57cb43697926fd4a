// Every primitive of a scene baked to world space: what DeviceAggregate::build packs into records and what the
// device image of rrt_scene_update_mesh (mesh_update.hpp) starts from.  Shared by aggregate.cu and mesh_update.cu.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "host_scene.hpp"
#include "sphere_core.cuh"

namespace rrt {

// A triangle's three world vertices; a full sphere's world centre and radius in v[0..3]; a sphere that needs the
// object-space test: the index of its GenSphere entry in v[0] and its radius in v[3].  Unused entries are 0.
struct BakedPrim {
    double v[9];
};

struct WorldBake {
    explicit WorldBake(size_t n) : world(n), boxes(n), kind(n), exact(n) {}
    RawBuf<BakedPrim> world;
    RawBuf<Aabb> boxes;
    RawBuf<uint8_t> kind;   // PRIM_TRIANGLE, PRIM_SPHERE or PRIM_SPHERE_GENERAL (device_layout.h)
    RawBuf<uint8_t> exact;  // 1: every vertex coordinate is an fp32 value (spheres: always 1)
    bool all_fp32 = true;
    bool has_spheres = false;
    std::vector<GenSphere> gspheres;
    std::vector<double> inst_w2p;  // world -> primitive 3x4 per instance, when the scene has spheres (their (u, v))
};

// Bakes scene.prims in parallel over the host threads.  RRT_ERR_UNSUPPORTED for a clipped sphere with a transform of
// its own (see the function).
int bake_world(const HostScene& scene, WorldBake* out, std::string* err);

}  // namespace rrt
