// The fp32 ray / hit format of rrt_intersect_f32 and relatives (include/rrt.h): what a 32-byte rrt_ray_f32 means as
// an rrt_ray, and how an rrt_hit becomes a 16-byte rrt_hit_f32.  Host + device, so that the CPU tests run the same
// conversions the streaming kernels of rays_f32.cu run (rrt_rays_f32_host_probe).
//
// Exactness: every float is a double (24-bit significand, exponent range inside double's, subnormals included), so
// the promotion loses nothing and the f64 walk sees exactly the rays the caller meant.  The way back rounds each field
// once, to nearest even: the same float as numpy's astype(np.float32) of the f64 result.
#pragma once
#include "../../include/rrt.h"
#include "rmath.cuh"

namespace rrt {

#if defined(__CUDA_ARCH__)
RRT_HD float round_to_f32(double x) { return __double2float_rn(x); }
#else
RRT_HD float round_to_f32(double x) { return static_cast<float>(x); }  // the host's default rounding: to nearest even
#endif

RRT_HD rrt_ray promote_ray(const rrt_ray_f32& r) {
    rrt_ray o;
    for (int k = 0; k < 3; ++k) {
        o.o[k] = static_cast<double>(r.o[k]);
        o.d[k] = static_cast<double>(r.d[k]);
    }
    o.t_max = static_cast<double>(r.t_max);
    o.time = 0.0;
    return o;
}

RRT_HD rrt_hit_f32 compact_hit(const rrt_hit& h) {
    rrt_hit_f32 o;
    o.prim_id = h.prim_id;
    o.t = round_to_f32(h.t);
    o.u = round_to_f32(h.u);
    o.v = round_to_f32(h.v);
    return o;
}

}  // namespace rrt
