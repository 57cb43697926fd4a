#include "literal.hpp"

#include <cuda_runtime.h>

#include <chrono>

#include "bvh_hlbvh.hpp"
#include "scene_tables.cuh"

namespace rrt {
namespace {

constexpr double kMaxDist = 1999999999.0;  // main.rs:51
constexpr int kLitStack = 64;             // bvh.rs:133,193

struct LitView {
    const LinearNode* nodes;
    const uint32_t* ordered;
    ShadeScene sc;  // geometry tables only
};

#define LIT_CUDA(call)                                                          \
    do {                                                                        \
        cudaError_t e_ = (call);                                                \
        if (e_ != cudaSuccess) {                                                \
            if (err) *err = std::string(#call) + ": " + cudaGetErrorString(e_); \
            return RRT_ERR_CUDA;                                                \
        }                                                                       \
    } while (0)

// Bounds3f::intersect_p (geometry.rs:1767-1800): corner select by dir_is_neg, far planes padded by
// 1 + 2 * gamma(3), accept iff t_min < ray.t_max && t_max > 0
__device__ __forceinline__ bool slab_literal(const LinearNode& b, V3 o, double ray_tmax, V3 inv, const int neg[3]) {
    const double gamma3 = (3.0 * kMachineEps) / (1.0 - 3.0 * kMachineEps);  // misc.rs:40-42
    const double pad = 1.0 + 2.0 * gamma3;
    double t_min = ((neg[0] ? b.hi[0] : b.lo[0]) - o.x) * inv.x;
    double t_max = ((neg[0] ? b.lo[0] : b.hi[0]) - o.x) * inv.x;
    const double ty_min = ((neg[1] ? b.hi[1] : b.lo[1]) - o.y) * inv.y;
    double ty_max = ((neg[1] ? b.lo[1] : b.hi[1]) - o.y) * inv.y;
    t_max *= pad;
    ty_max *= pad;
    if (t_min > ty_max || ty_min > t_max) return false;
    if (ty_min > t_min) t_min = ty_min;
    if (ty_max < t_max) t_max = ty_max;
    const double tz_min = ((neg[2] ? b.hi[2] : b.lo[2]) - o.z) * inv.z;
    double tz_max = ((neg[2] ? b.lo[2] : b.hi[2]) - o.z) * inv.z;
    tz_max *= pad;
    if (t_min > tz_max || tz_min > t_max) return false;
    if (tz_min > t_min) t_min = tz_min;
    if (tz_max < t_max) t_max = tz_max;
    return (t_min < ray_tmax) && (t_max > 0.0);
}

// The ray a shape receives from a TransformedPrimitive / a Sphere's world_to_object: Transformable
// for Ray normalises d, Ray::new normalises it again (transform.rs:525-537, geometry.rs:1841-1848; Q6)
__device__ __forceinline__ void xf_ray_literal(const M34& inv, V3* o, V3* d) {
    *o = xf_point(inv, *o);
    *d = normalize(normalize(xf_vector(inv, *d)));
}

// Shape::intersect of primitive `prim` on world ray (o, d): returns the accepted t (local units,
// copied to the world ray unscaled: primitives.rs:132) — the shapes never look at ray.t_max (Q3)
__device__ bool prim_intersect_literal(const ShadeScene& sc, uint32_t prim, V3 o, V3 d, double* t, double* u, double* v) {
    const PrimInfo pi = sc.prims[prim];
    if (pi.instance >= 0) xf_ray_literal(sc.instances[pi.instance].inv, &o, &d);
    if ((pi.kind & kPrimKindMask) == 0) {  // Triangle::intersect (triangle.rs:226-265)
        const MeshInfo mi = sc.meshes[pi.shape];
        const uint32_t* vi = sc.mesh_vi + mi.vi_off + 3ull * pi.tri;
        const double* pb = sc.mesh_p + 3 * mi.p_off;
        const V3 p0 = ld3(pb, vi[0]), p1 = ld3(pb, vi[1]), p2 = ld3(pb, vi[2]);
        const V3 E1 = p1 - p0, E2 = p2 - p0;
        const V3 P = cross(d, E2);
        const double a = dot(E1, P);
        if (a > -0.0000001 && a < 0.0000001) return false;
        const double f = 1.0 / a;
        const V3 T = o - p0;
        const double uu = f * dot(T, P);
        if (uu < 0.0 || uu > 1.0) return false;
        const V3 Q = cross(T, E1);
        const double vv = f * dot(d, Q);
        if (vv < 0.0 || (uu + vv) > 1.0) return false;
        const double tt = f * dot(E2, Q);
        if (tt < 0.0000001) return false;
        // triangle.rs:283-291: a degenerate geometric normal rejects the hit after the fact
        if (length_sq(cross(p2 - p0, p1 - p0)) == 0.0) {
            // only reached through the degenerate-uv fallback; with the default uvs the determinant is 1
        }
        *t = tt;
        *u = uu;
        *v = vv;
        return true;
    }
    // Sphere::intersect (sphere.rs:124-198), full spheres
    const SphereInfo& sp = sc.spheres[pi.shape];
    V3 so = o, sd = d;
    xf_ray_literal(sp.w2o, &so, &sd);
    const double a = sd.x * sd.x + sd.y * sd.y + sd.z * sd.z;
    const double b = 2.0 * (sd.x * so.x + sd.y * so.y + sd.z * so.z);
    const double c = so.x * so.x + so.y * so.y + so.z * so.z - sp.radius * sp.radius;
    double t0, t1;
    if (!quadratic(a, b, c, &t0, &t1)) return false;
    if (t0 > kMaxDist || t1 <= 0.0) return false;  // Q5b: MAX_DIST, not ray.t_max
    double ts = t0;
    if (t0 <= 0.0) {
        ts = t1;
        if (ts > kMaxDist) return false;
    }
    *t = ts;
    *u = 0.0;
    *v = 0.0;
    return true;
}

// Shape::intersect_p: Triangle uses E2 = p2 - p1 (Q4, triangle.rs:175) and ignores t_max
__device__ bool prim_intersect_p_literal(const ShadeScene& sc, uint32_t prim, V3 o, V3 d) {
    const PrimInfo pi = sc.prims[prim];
    if ((pi.kind & kPrimKindMask) != 0) {
        // sphere.rs:50-109: for a full sphere the any-hit accept rule is the closest-hit one (the clip
        // test runs on an uninitialised p_hit = 0, phi = 0 and never fires, Q5c)
        double t, u, v;
        return prim_intersect_literal(sc, prim, o, d, &t, &u, &v);
    }
    if (pi.instance >= 0) xf_ray_literal(sc.instances[pi.instance].inv, &o, &d);
    {
        const MeshInfo mi = sc.meshes[pi.shape];
        const uint32_t* vi = sc.mesh_vi + mi.vi_off + 3ull * pi.tri;
        const double* pb = sc.mesh_p + 3 * mi.p_off;
        const V3 p0 = ld3(pb, vi[0]), p1 = ld3(pb, vi[1]), p2 = ld3(pb, vi[2]);
        const V3 E1 = p1 - p0, E2 = p2 - p1;
        const V3 P = cross(d, E2);
        const double a = dot(E1, P);
        if (a > -0.0000001 && a < 0.0000001) return false;
        const double f = 1.0 / a;
        const V3 T = o - p0;
        const double uu = f * dot(T, P);
        if (uu < 0.0 || uu > 1.0) return false;
        const V3 Q = cross(T, E1);
        const double vv = f * dot(d, Q);
        if (vv < 0.0 || (uu + vv) > 1.0) return false;
        const double tt = f * dot(E2, Q);
        return !(tt < 0.0000001);
    }
}

template <bool ANY>
__global__ void __launch_bounds__(128) literal_kernel(LitView V, uint64_t n, const rrt_ray* __restrict__ rays,
                                                       rrt_hit* __restrict__ hits, uint8_t* __restrict__ occluded,
                                                       const uint32_t* __restrict__ n_dev) {
    if (n_dev) n = *n_dev;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double2* rp = reinterpret_cast<const double2*>(rays + i);
    const double2 q0 = rp[0], q1 = rp[1], q2 = rp[2], q3 = rp[3];
    const V3 o = v3(q0.x, q0.y, q1.x), d = v3(q1.y, q2.x, q2.y);
    double t_max = q3.x;
    const V3 inv = v3(1.0 / d.x, 1.0 / d.y, 1.0 / d.z);
    const int neg[3] = {inv.x < 0.0 ? 1 : 0, inv.y < 0.0 ? 1 : 0, inv.z < 0.0 ? 1 : 0};
    uint32_t stack[kLitStack];
    int to_visit = 0;
    uint32_t cur = 0;
    bool hit = false;
    uint32_t best = RRT_NO_HIT;
    double bu = 0.0, bv = 0.0;
    for (;;) {
        const LinearNode node = V.nodes[cur];
        if (slab_literal(node, o, t_max, inv, neg)) {
            if (node.n_primitives > 0) {
                for (uint32_t k = 0; k < node.n_primitives; ++k) {
                    const uint32_t prim = V.ordered[node.offset + k];
                    if (ANY) {
                        if (prim_intersect_p_literal(V.sc, prim, o, d)) {
                            occluded[i] = 1;
                            return;
                        }
                    } else {
                        double t, u, v;
                        if (prim_intersect_literal(V.sc, prim, o, d, &t, &u, &v)) {
                            hit = true;  // every accepted candidate overwrites si and r.t_max (Q3)
                            best = prim;
                            t_max = t;
                            bu = u;
                            bv = v;
                        }
                    }
                }
                if (to_visit == 0) break;
                cur = stack[--to_visit];
            } else if (neg[node.axis]) {
                stack[to_visit++] = cur + 1;
                cur = node.offset;
            } else {
                stack[to_visit++] = node.offset;
                cur = cur + 1;
            }
        } else {
            if (to_visit == 0) break;
            cur = stack[--to_visit];
        }
    }
    if (ANY) {
        occluded[i] = 0;
    } else {
        rrt_hit h;
        h.prim_id = hit ? best : RRT_NO_HIT;
        h.reserved = 0;
        h.t = hit ? t_max : 0.0;
        h.u = hit ? bu : 0.0;
        h.v = hit ? bv : 0.0;
        hits[i] = h;
    }
}

}  // namespace

struct LiteralAggregate::Impl {
    LitView view{};
    std::vector<void*> allocations;
};

LiteralAggregate::~LiteralAggregate() {
    if (!impl_) return;
    cudaSetDevice(device_);
    for (void* p : impl_->allocations) cudaFree(p);
    delete impl_;
}

int LiteralAggregate::build(int device, const HostScene& scene, uint32_t max_prims_in_node, std::string* err) {
    auto t0 = std::chrono::steady_clock::now();
    device_ = device;
    if (scene.prims.empty()) {
        if (err) *err = "BVHAccel::new needs at least one primitive (bvh.rs:319)";
        return RRT_ERR_EMPTY;
    }
    for (const Primitive& p : scene.prims)
        if (p.kind == SHAPE_SPHERE && !scene.spheres[p.shape].is_full()) {
            if (err) *err = "partial spheres (z_min / z_max / phi_max) are outside the device scope";
            return RRT_ERR_UNSUPPORTED;
        }
    std::vector<Aabb> bounds(scene.prims.size());
    for (size_t i = 0; i < scene.prims.size(); ++i) bounds[i] = scene.reference_world_bound(i);
    LiteralBvh tree;
    try {
        build_hlbvh_literal(bounds, max_prims_in_node == 0 ? 4 : max_prims_in_node, &tree);
    } catch (const std::exception& e) {
        if (err) *err = std::string("HLBVH build: ") + e.what();
        return RRT_ERR_INVALID;
    }
    if (tree.max_depth + 1 > (uint32_t)kLitStack) {
        // Q27: the reference indexes a [usize; 64] stack with bounds checks and would panic
        if (err) *err = "literal tree deeper than the reference's 64-entry traversal stack (bvh.rs:133)";
        return RRT_ERR_UNSUPPORTED;
    }
    LIT_CUDA(cudaSetDevice(device));
    impl_ = new Impl();
    void* d = nullptr;
    int rc = upload_vector(tree.nodes, &d, err);
    if (rc != RRT_OK) return rc;
    impl_->allocations.push_back(d);
    impl_->view.nodes = static_cast<const LinearNode*>(d);
    rc = upload_vector(tree.ordered, &d, err);
    if (rc != RRT_OK) return rc;
    impl_->allocations.push_back(d);
    impl_->view.ordered = static_cast<const uint32_t*>(d);
    rc = upload_geometry_tables(scene, &impl_->view.sc, &impl_->allocations, err);
    if (rc != RRT_OK) return rc;
    for (int k = 0; k < 3; ++k) {
        root_bounds_[k] = tree.nodes[0].lo[k];
        root_bounds_[3 + k] = tree.nodes[0].hi[k];
    }
    stats_.n_nodes = tree.nodes.size();
    stats_.max_depth = tree.max_depth;
    stats_.n_prims = scene.prims.size();
    stats_.n_records = tree.ordered.size();
    stats_.device_bytes = tree.nodes.size() * sizeof(LinearNode) + tree.ordered.size() * 4;
    for (const LinearNode& nd : tree.nodes) stats_.n_leaves += nd.n_primitives > 0 ? 1 : 0;
    stats_.build_usec = (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    return RRT_OK;
}

namespace {
template <bool ANY>
int launch_literal(const LitView& v, uint64_t n, const rrt_ray* rays, rrt_hit* hits, uint8_t* occ, void* stream,
                   const uint32_t* n_dev, std::string* err, int* launches) {
    if (n == 0) return RRT_OK;
    const uint64_t blocks = (n + 127) / 128;
    if (blocks > 0x7fffffffull) {
        if (err) *err = "batch too large for one launch";
        return RRT_ERR_INVALID;
    }
    literal_kernel<ANY><<<(unsigned)blocks, 128, 0, static_cast<cudaStream_t>(stream)>>>(v, n, rays, hits, occ, n_dev);
    LIT_CUDA(cudaGetLastError());
    if (launches) *launches = 1;
    return RRT_OK;
}
}  // namespace

const ShadeScene& LiteralAggregate::geometry_tables() const { return impl_->view.sc; }

int LiteralAggregate::closest_hit(uint64_t n, const rrt_ray* r, rrt_hit* h, void* s, std::string* err, int* l) const {
    return launch_literal<false>(impl_->view, n, r, h, nullptr, s, nullptr, err, l);
}
int LiteralAggregate::any_hit(uint64_t n, const rrt_ray* r, uint8_t* o, void* s, std::string* err, int* l) const {
    return launch_literal<true>(impl_->view, n, r, nullptr, o, s, nullptr, err, l);
}
int LiteralAggregate::closest_hit_indirect(uint64_t cap, const uint32_t* c, const rrt_ray* r, rrt_hit* h, void* s,
                                           std::string* err, int* l) const {
    return launch_literal<false>(impl_->view, cap, r, h, nullptr, s, c, err, l);
}
int LiteralAggregate::any_hit_indirect(uint64_t cap, const uint32_t* c, const rrt_ray* r, uint8_t* o, void* s,
                                       std::string* err, int* l) const {
    return launch_literal<true>(impl_->view, cap, r, nullptr, o, s, c, err, l);
}

}  // namespace rrt
