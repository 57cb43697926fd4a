// The surface pass of rrt_intersect_surface / rrt_intersect_surface_device (surface.cu): after the walk, one thread per
// ray rebuilds the winner's SurfaceInteraction with the renderer's make_surface_body and writes a 336-byte rrt_surface.
// Host-visible, no CUDA types: the launcher returns a cudaError_t value (0 = success) and is asynchronous on `stream`.
#pragma once
#include <cstdint>
#include <string>

#include "../../include/rrt.h"

namespace rrt {

struct HostScene;
struct ShadeScene;   // shading.cuh: the device geometry tables the pass reads
struct SurfaceTables;  // a scene's own copy of those tables (Tier F)

// upload_geometry_tables over `scene` (one synchronous upload); freed by surface_tables_destroy
int surface_tables_create(const HostScene& scene, SurfaceTables** out, std::string* err);
void surface_tables_destroy(SurfaceTables* t);
const ShadeScene* surface_tables_view(const SurfaceTables* t);

// n < 2^32 rays and their f64 hits -> n records.  `literal`: the Tier-L instance / sphere ray rule (Q6) is applied.
int launch_surfaces(const ShadeScene& tables, bool literal, uint64_t n, const rrt_ray* rays, const rrt_hit* hits,
                    rrt_surface* out, void* stream);

}  // namespace rrt
