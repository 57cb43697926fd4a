#include "host_scene.hpp"

#include "bake_core.h"

namespace rrt {

Transform Transform::identity() {
    Transform t;
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) t.m.m[i][j] = t.inv.m[i][j] = (i == j) ? 1.0 : 0.0;
    return t;
}

bool Transform::is_identity() const {
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j)
            if (m.m[i][j] != ((i == j) ? 1.0 : 0.0)) return false;
    return true;
}

Vec3d Transform::point(Vec3d p) const {
    double q[3];
    bake::xf_point(&m.m[0][0], p.x, p.y, p.z, q);
    return {q[0], q[1], q[2]};
}

Vec3d Transform::vector(Vec3d v) const {
    const auto& a = m.m;
    return {a[0][0] * v.x + a[0][1] * v.y + a[0][2] * v.z, a[1][0] * v.x + a[1][1] * v.y + a[1][2] * v.z,
            a[2][0] * v.x + a[2][1] * v.y + a[2][2] * v.z};
}

Vec3d Transform::normal(Vec3d n) const {
    const auto& a = inv.m;
    return {a[0][0] * n.x + a[1][0] * n.y + a[2][0] * n.z, a[0][1] * n.x + a[1][1] * n.y + a[2][1] * n.z,
            a[0][2] * n.x + a[1][2] * n.y + a[2][2] * n.z};
}

void HostScene::world_triangle(size_t i, double v[9]) const {
    const Primitive& pr = prims[i];
    const TriangleMesh& m = meshes[pr.shape];
    bake::world_triangle(m.p.data(), m.vi.data(), pr.tri, pr.instance >= 0 ? &instances[pr.instance].m.m[0][0] : nullptr, v);
}

namespace {
// The reference's Bounds3f::t_by walks the corners in this exact order (transform.rs:539-616)
// and Bounds3::union uses `<` / `>` selects, so a plain min/max reproduces it bit for bit.
Aabb transform_bounds(const Transform& t, const Aabb& b) {
    const int order[8][3] = {{0, 0, 0}, {1, 0, 0}, {0, 1, 0}, {0, 0, 1}, {0, 1, 1}, {1, 1, 0}, {1, 0, 1}, {1, 1, 1}};
    Aabb r;
    for (int c = 0; c < 8; ++c) {
        Vec3d p{order[c][0] ? b.hi[0] : b.lo[0], order[c][1] ? b.hi[1] : b.lo[1], order[c][2] ? b.hi[2] : b.lo[2]};
        Vec3d q = t.point(p);
        double a[3] = {q.x, q.y, q.z};
        r.grow(a);
    }
    return r;
}
}  // namespace

Aabb HostScene::reference_world_bound(size_t i) const {
    const Primitive& pr = prims[i];
    Aabb b;
    if (pr.kind == SHAPE_TRIANGLE) {
        const TriangleMesh& m = meshes[pr.shape];
        for (int k = 0; k < 3; ++k) {
            uint32_t vi = m.vi[3 * (size_t)pr.tri + k];
            b.grow(&m.p[3 * (size_t)vi]);
        }
    } else {
        const Sphere& s = spheres[pr.shape];
        Aabb ob;
        double lo[3] = {-s.radius, -s.radius, s.z_min}, hi[3] = {s.radius, s.radius, s.z_max};
        // Bounds3::new orders the corners componentwise (geometry.rs:1570-1585)
        for (int k = 0; k < 3; ++k) {
            ob.lo[k] = lo[k] > hi[k] ? hi[k] : lo[k];
            ob.hi[k] = lo[k] > hi[k] ? lo[k] : hi[k];
        }
        b = transform_bounds(s.obj_to_world, ob);
    }
    if (pr.instance >= 0) b = transform_bounds(instances[pr.instance], b);
    return b;
}

}  // namespace rrt
