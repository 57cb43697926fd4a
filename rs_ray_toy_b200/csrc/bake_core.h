// Baking a triangle to world space: Transform::point (src/transform.rs:451-488) and the per-vertex loop of
// HostScene::world_triangle, written once as __host__ __device__ functions so that the commit's host bake and the
// device re-bake of rrt_scene_update_mesh (mesh_update.cu) produce the same bits.  Both sides are compiled without
// FMA contraction (--fmad=false, -ffp-contract=off): each product and sum below is rounded on its own, in this order.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define BAKE_HD __host__ __device__ __forceinline__
#else
#define BAKE_HD inline
#endif

namespace rrt {
namespace bake {

// Transform::point with the row-major 4x4 matrix m (transform.rs:451-488)
BAKE_HD void xf_point(const double* m, double x, double y, double z, double out[3]) {
    const double xp = m[0] * x + m[1] * y + m[2] * z + m[3];
    const double yp = m[4] * x + m[5] * y + m[6] * z + m[7];
    const double zp = m[8] * x + m[9] * y + m[10] * z + m[11];
    const double wp = m[12] * x + m[13] * y + m[14] * z + m[15];
    if (wp == 1.0) {
        out[0] = xp;
        out[1] = yp;
        out[2] = zp;
        return;
    }
    const double inv_w = 1.0 / wp;
    out[0] = inv_w * xp;
    out[1] = inv_w * yp;
    out[2] = inv_w * zp;
}

// World-space vertices of triangle `tri` of the mesh (p: 3 doubles per vertex, vi: 3 indices per triangle), through
// the instance matrix m (row-major 4x4) or none (m = nullptr: a bare triangle).
BAKE_HD void world_triangle(const double* p, const uint32_t* vi, uint32_t tri, const double* m, double v[9]) {
    for (int k = 0; k < 3; ++k) {
        const uint32_t x = vi[3 * (size_t)tri + k];
        const double* q = p + 3 * (size_t)x;
        if (m) {
            xf_point(m, q[0], q[1], q[2], v + 3 * k);
        } else {
            v[3 * k] = q[0];
            v[3 * k + 1] = q[1];
            v[3 * k + 2] = q[2];
        }
    }
}

// Every value is an fp32 value: the triangle's record may be a PrimRec48 (device_layout.h)
BAKE_HD bool fp32_exact(const double* v, int n) {
    for (int i = 0; i < n; ++i)
        if ((double)(float)v[i] != v[i]) return false;
    return true;
}

// The f64 box of a baked triangle, grown vertex by vertex like Aabb::grow
BAKE_HD void triangle_box(const double v[9], double lo[3], double hi[3]) {
    for (int k = 0; k < 3; ++k) {
        lo[k] = __builtin_huge_val();
        hi[k] = -__builtin_huge_val();
    }
    for (int j = 0; j < 3; ++j)
        for (int k = 0; k < 3; ++k) {
            if (v[3 * j + k] < lo[k]) lo[k] = v[3 * j + k];
            if (v[3 * j + k] > hi[k]) hi[k] = v[3 * j + k];
        }
}

}  // namespace bake
}  // namespace rrt
