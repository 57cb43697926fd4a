// Launchers of the fp32 format's streaming passes (rays_f32.cu): rrt_ray_f32 -> rrt_ray before the walk, rrt_hit ->
// rrt_hit_f32 after it.  Host-visible, no CUDA types: both return a cudaError_t value (0 = success) and are
// asynchronous on `stream`.  n < 2^32; every pointer 16-byte aligned.
#pragma once
#include <cstdint>

#include "../../include/rrt.h"

namespace rrt {

int launch_promote_rays(uint64_t n, const rrt_ray_f32* in, rrt_ray* out, void* stream);
int launch_compact_hits(uint64_t n, const rrt_hit* in, rrt_hit_f32* out, void* stream);

}  // namespace rrt
