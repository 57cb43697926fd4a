// sm_100a closest-hit / any-hit traversal of the GPU aggregate.
//
// Replaces BVHAccel::intersect / intersect_p (src/bvh.rs:183-236, :123-174) together with
// the per-candidate Triangle / Sphere tests (src/shape/triangle.rs:226-265, :167-205,
// src/shape/sphere.rs:124-155, :50-86) for a whole batch of rays.
//
// Precision split (DESIGN.md §3): the *culling* (box slabs) runs in fp32 on boxes that were
// widened on the host so that no fp32 rounding can drop a true candidate; the *deciding*
// arithmetic (Möller–Trumbore, sphere quadratic) runs in f64 with the reference's operation
// order and with FMA contraction disabled (__dmul_rn / __dadd_rn), so t, u, v are the same
// bits the reference's f64 code produces.  B200's FP64 pipe is half-rate FP32, which makes
// this affordable; the box tests dominate the instruction count.
#include <cuda_runtime.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <atomic>
#include <cstring>
#include <thread>
#include <utility>
#include <vector>

#include "aggregate.hpp"
#include "bvh_lbvh.hpp"
#include "bvh_pack_plan.hpp"
#include "device_layout.h"
#include "bake_core.h"
#include "mesh_update.hpp"
#include "sphere_core.cuh"
#include "world_bake.hpp"

namespace rrt {

namespace {

constexpr int kStack = 64;
#ifndef RRT_BLOCK
#define RRT_BLOCK 128
#endif
#ifndef RRT_UNROLL
#define RRT_UNROLL 2
#endif
constexpr int kBlock = RRT_BLOCK;

struct D3 {
    double x, y, z;
};
// f64 helpers that can never be contracted into FMAs: bit-compatible with the reference's
// plain Rust arithmetic (geometry.rs:110-117 dot3, :1099-1107 cross).
__device__ __forceinline__ D3 sub3(D3 a, D3 b) { return {__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y), __dsub_rn(a.z, b.z)}; }
__device__ __forceinline__ double dot3(D3 a, D3 b) {
    return __dadd_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), __dmul_rn(a.z, b.z));
}
__device__ __forceinline__ D3 cross3(D3 a, D3 b) {
    return {__dsub_rn(__dmul_rn(a.y, b.z), __dmul_rn(a.z, b.y)), __dsub_rn(__dmul_rn(a.z, b.x), __dmul_rn(a.x, b.z)),
            __dsub_rn(__dmul_rn(a.x, b.y), __dmul_rn(a.y, b.x))};
}

// Möller–Trumbore exactly as triangle.rs:233-265 (closest) — with Q4 fixed it is also the
// any-hit test.  Returns true and t,u,v when the candidate is accepted (t_max not applied here).
__device__ __forceinline__ bool tri_test(D3 o, D3 d, D3 p0, D3 p1, D3 p2, double* t, double* u, double* v) {
    D3 E1 = sub3(p1, p0);
    D3 E2 = sub3(p2, p0);
    D3 P = cross3(d, E2);
    double a = dot3(E1, P);
    if (a > -0.0000001 && a < 0.0000001) return false;
    double f = __ddiv_rn(1.0, a);
    D3 T = sub3(o, p0);
    double uu = __dmul_rn(f, dot3(T, P));
    if (uu < 0.0 || uu > 1.0) return false;
    D3 Q = cross3(T, E1);
    double vv = __dmul_rn(f, dot3(d, Q));
    if (vv < 0.0 || __dadd_rn(uu, vv) > 1.0) return false;
    double tt = __dmul_rn(f, dot3(E2, Q));
    if (tt < 0.0000001) return false;
    *t = tt;
    *u = uu;
    *v = vv;
    return true;
}

// Full sphere in world space: sphere.rs:127-155 with MAX_DIST -> t_max (Q5b) and the Tier-F
// self-hit floor (Q8).  misc.rs:231-251 quadratic.
__device__ __forceinline__ bool sphere_test(D3 o, D3 d, D3 c, double radius, double t_far, double* t) {
    D3 oc = sub3(o, c);
    double a = dot3(d, d);
    double b = __dmul_rn(2.0, dot3(d, oc));
    double cc = __dsub_rn(dot3(oc, oc), __dmul_rn(radius, radius));
    double discrim = __dsub_rn(__dmul_rn(b, b), __dmul_rn(__dmul_rn(4.0, a), cc));
    if (discrim < 0.0) return false;
    double root = __dsqrt_rn(discrim);
    double q = (b < 0.0) ? __dmul_rn(-0.5, __dsub_rn(b, root)) : __dmul_rn(-0.5, __dadd_rn(b, root));
    double t0 = __ddiv_rn(q, a);
    double t1 = __ddiv_rn(cc, q);
    if (t0 > t1) {
        double s = t0;
        t0 = t1;
        t1 = s;
    }
    const double t_near = 1e-7 * fmax(1.0, radius);
    if (t0 > t_far || t1 <= t_near) return false;
    double ts = t0;
    if (t0 <= t_near) {
        ts = t1;
        if (ts > t_far) return false;
    }
    *t = ts;
    return true;
}

// One 256-bit load (LDG.E.256 on sm_100a): half a Node64 per request instead of a quarter.
struct F8 {
    float a, b, c, d, e, f, g, h;
};
__device__ __forceinline__ F8 ldg256(const void* p) {
    F8 r;
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(r.a), "=f"(r.b), "=f"(r.c), "=f"(r.d), "=f"(r.e), "=f"(r.f), "=f"(r.g), "=f"(r.h)
                 : "l"(p));
    return r;
}

struct RayF {
    float idx, idy, idz;     // 1/d (fp32)
    float oidx, oidy, oidz;  // o * (1/d)
};

__device__ __forceinline__ float safe_inv(double d) {
    float f = (float)d;
    if (fabsf(f) < 1e-30f) f = copysignf(1e-30f, f == 0.0f ? (signbit(d) ? -1.0f : 1.0f) : f);
    return 1.0f / f;
}

// Slab test of one child box; `tcull` is the current closest t (rounded up).  Returns entry t.
__device__ __forceinline__ bool slab(const RayF& r, float lox, float hix, float loy, float hiy, float loz, float hiz,
                                     float tcull, float* tnear) {
    float tx0 = fmaf(lox, r.idx, -r.oidx), tx1 = fmaf(hix, r.idx, -r.oidx);
    float ty0 = fmaf(loy, r.idy, -r.oidy), ty1 = fmaf(hiy, r.idy, -r.oidy);
    float tz0 = fmaf(loz, r.idz, -r.oidz), tz1 = fmaf(hiz, r.idz, -r.oidz);
    float tmin = fmaxf(fmaxf(fminf(tx0, tx1), fminf(ty0, ty1)), fmaxf(fminf(tz0, tz1), 0.0f));
    float tmax = fminf(fminf(fmaxf(tx0, tx1), fmaxf(ty0, ty1)), fminf(fmaxf(tz0, tz1), tcull));
    *tnear = tmin;
    return tmin <= tmax;
}

// Node32 planes: a word holds lo | hi << 16 (device_layout.h); these decode the lo / hi plane
__device__ __forceinline__ float qlo(uint32_t w) { return __uint_as_float(__byte_perm(w, 0x3Fu, 0x4105)); }
__device__ __forceinline__ float qhi(uint32_t w) { return __uint_as_float(__byte_perm(w, 0x3Fu, 0x4325)); }

template <bool WIDE>
__device__ __forceinline__ void load_prim(const void* prims, uint32_t idx, D3* a, D3* b, D3* c, uint32_t* prim_id,
                                          uint32_t* kind) {
    if (!WIDE) {
        const float4* p = reinterpret_cast<const float4*>(static_cast<const PrimRec48*>(prims) + idx);
        float4 r0 = __ldg(p), r1 = __ldg(p + 1), r2 = __ldg(p + 2);
        *prim_id = __float_as_uint(r2.y);
        *kind = __float_as_uint(r2.z);
        if (*kind == PRIM_TRIANGLE) {
            *a = {(double)r0.x, (double)r0.y, (double)r0.z};
            *b = {(double)r0.w, (double)r1.x, (double)r1.y};
            *c = {(double)r1.z, (double)r1.w, (double)r2.x};
        } else {
            // sphere: centre + radius as four f64 in the first 32 bytes
            double cx = __hiloint2double(__float_as_int(r0.y), __float_as_int(r0.x));
            double cy = __hiloint2double(__float_as_int(r0.w), __float_as_int(r0.z));
            double cz = __hiloint2double(__float_as_int(r1.y), __float_as_int(r1.x));
            double rr = __hiloint2double(__float_as_int(r1.w), __float_as_int(r1.z));
            *a = {cx, cy, cz};
            *b = {rr, 0.0, 0.0};
        }
    } else {
        const double2* p = reinterpret_cast<const double2*>(static_cast<const PrimRec96*>(prims) + idx);
        double2 r0 = __ldg(p), r1 = __ldg(p + 1), r2 = __ldg(p + 2), r3 = __ldg(p + 3), r4 = __ldg(p + 4);
        *prim_id = (uint32_t)__double2loint(r4.y);
        *kind = (uint32_t)__double2hiint(r4.y);
        *a = {r0.x, r0.y, r1.x};
        *b = {r1.y, r2.x, r2.y};
        *c = {r3.x, r3.y, r4.x};
    }
}

// Brings a ray whose origin lies far outside the world box close to it (in f64), so that the
// fp32 traversal copy keeps |o| comparable to the scene and the host-side box widening holds.
__device__ __noinline__ bool prepare_ray(const AggView& A, D3 o, D3 d, double t_max, float* t_shift, RayF* rf) {
    // Scene::intersect asserts d != 0 (scene.rs:70); here a ray without a direction, or with a
    // non-finite component, simply hits nothing
    const double len2 = d.x * d.x + d.y * d.y + d.z * d.z;
    if (!(len2 > 0.0) || !(len2 < 1e300) || !(o.x == o.x) || !(o.y == o.y) || !(o.z == o.z) ||
        fabs(o.x) > 1e300 || fabs(o.y) > 1e300 || fabs(o.z) > 1e300)
        return false;
    double ts = 0.0;
    bool outside = o.x < A.world_lo[0] || o.x > A.world_hi[0] || o.y < A.world_lo[1] || o.y > A.world_hi[1] ||
                   o.z < A.world_lo[2] || o.z > A.world_hi[2];
    if (outside) {
        double t0 = 0.0, t1 = t_max;
        const double oo[3] = {o.x, o.y, o.z}, dd[3] = {d.x, d.y, d.z};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            if (dd[k] == 0.0) {
                if (oo[k] < A.world_lo[k] || oo[k] > A.world_hi[k]) return false;
                continue;
            }
            double inv = 1.0 / dd[k];
            double ta = (A.world_lo[k] - oo[k]) * inv, tb = (A.world_hi[k] - oo[k]) * inv;
            double tn = fmin(ta, tb), tf = fmax(ta, tb);
            tf *= 1.0 + 1e-12;
            t0 = fmax(t0, tn);
            t1 = fmin(t1, tf);
        }
        if (t0 > t1 * (1.0 + 1e-12) + 1e-300) return false;
        double len = sqrt(d.x * d.x + d.y * d.y + d.z * d.z);
        ts = fmax(0.0, t0 - A.scene_scale / len);
    }
    // the shift is kept as an fp32 value (rounded toward the origin) so the walk can carry it in one register
    const float tsf = __double2float_rd(ts);
    ts = (double)tsf;
    *t_shift = tsf;
    double sx = o.x + d.x * ts, sy = o.y + d.y * ts, sz = o.z + d.z * ts;
    const float ix = safe_inv(d.x), iy = safe_inv(d.y), iz = safe_inv(d.z);
    if (A.quantised) {
        // Node32 planes: distance = f * (extent / d) - (o - (lo - extent)) / d, f in [1, 2) straight from the node
        rf->idx = A.grid_ext[0] * ix;
        rf->idy = A.grid_ext[1] * iy;
        rf->idz = A.grid_ext[2] * iz;
        rf->oidx = (float)(sx - A.grid_c[0]) * ix;
        rf->oidy = (float)(sy - A.grid_c[1]) * iy;
        rf->oidz = (float)(sz - A.grid_c[2]) * iz;
    } else {
        rf->idx = ix;
        rf->idy = iy;
        rf->idz = iz;
        rf->oidx = (float)sx * ix;
        rf->oidy = (float)sy * iy;
        rf->oidz = (float)sz * iz;
    }
    return true;
}

// Partial spheres and spheres under non-rigid transforms: the whole of Sphere::intersect in object space
// (sphere_core.cuh).  Out of line: scenes without such spheres never pay for it.
__device__ __noinline__ bool general_sphere_test(const AggView& A, double index, D3 o, D3 d, double t_far, double* t) {
    const GenSphere& g = static_cast<const GenSphere*>(A.gspheres)[(uint32_t)index];
    V3 p;
    double phi;
    return gen_sphere_hit(g, v3(o.x, o.y, o.z), v3(d.x, d.y, d.z), t_far, t, &p, &phi);
}

// Surface parameters of the winning record.  Sphere hit, sphere.rs:157-198 for a full sphere: the hit point is taken
// on the ray the shape was handed (the instance-space ray, Q5a), phi = atan2(y, x) wrapped to
// [0, 2pi), u = phi / phi_max, v = (theta - theta_min) / (theta_max - theta_min) with
// theta_min = acos(-1), theta_max = acos(1).  Only the winning record pays for this.
template <bool WIDE>
__device__ __noinline__ void hit_params(const AggView& A, uint32_t rec, D3 o, D3 d, double t, double* u, double* v) {
    D3 a, b, c;
    uint32_t pid, kind, inst = 0xFFFFFFFFu;
    load_prim<WIDE>(A.prims, rec, &a, &b, &c, &pid, &kind);
    if (kind == PRIM_TRIANGLE) {
        // the walk keeps only (t, record); the barycentrics of the winner are recomputed here with
        // the same operations, hence the same bits (triangle.rs:245-256)
        double tt;
        tri_test(o, d, a, b, c, &tt, u, v);
        return;
    }
    if (kind == PRIM_SPHERE_GENERAL) {
        // replay the accepted hit (t_far = t reproduces the walk's root and clipping decisions) for its point
        const GenSphere& g = static_cast<const GenSphere*>(A.gspheres)[(uint32_t)a.x];
        V3 p;
        double phi, tt;
        *u = *v = 0.0;
        if (gen_sphere_hit(g, v3(o.x, o.y, o.z), v3(d.x, d.y, d.z), t, &tt, &p, &phi)) gen_sphere_uv(g, p, phi, u, v);
        return;
    }
    if (!WIDE) inst = static_cast<const PrimRec48*>(A.prims)[rec].words[8];
    else inst = static_cast<const PrimRec96*>(A.prims)[rec].pad[0];
    D3 lo = o, ld = d;
    if (inst != 0xFFFFFFFFu) {
        // Transform::t(ray) with world_to_primitive (transform.rs:451-502), row by row
        const double* m = A.inst_w2p + 12 * (size_t)inst;
        lo = {__dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(m[0], o.x), __dmul_rn(m[1], o.y)), __dmul_rn(m[2], o.z)), m[3]),
              __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(m[4], o.x), __dmul_rn(m[5], o.y)), __dmul_rn(m[6], o.z)), m[7]),
              __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(m[8], o.x), __dmul_rn(m[9], o.y)), __dmul_rn(m[10], o.z)), m[11])};
        ld = {__dadd_rn(__dadd_rn(__dmul_rn(m[0], d.x), __dmul_rn(m[1], d.y)), __dmul_rn(m[2], d.z)),
              __dadd_rn(__dadd_rn(__dmul_rn(m[4], d.x), __dmul_rn(m[5], d.y)), __dmul_rn(m[6], d.z)),
              __dadd_rn(__dadd_rn(__dmul_rn(m[8], d.x), __dmul_rn(m[9], d.y)), __dmul_rn(m[10], d.z))};
    }
    const double radius = b.x;
    double px = __dadd_rn(lo.x, __dmul_rn(ld.x, t)), py = __dadd_rn(lo.y, __dmul_rn(ld.y, t)),
           pz = __dadd_rn(lo.z, __dmul_rn(ld.z, t));
    if (px == 0.0 && py == 0.0) px = __dmul_rn(1e-5, radius);
    double phi = atan2(py, px);
    const double kPi = 3.14159265358979323846;
    if (phi < 0.0) phi = __dadd_rn(phi, __dmul_rn(2.0, kPi));
    const double phi_max = __dmul_rn(360.0, kPi / 180.0);
    *u = __ddiv_rn(phi, phi_max);
    double cz = __ddiv_rn(pz, radius);
    cz = cz < -1.0 ? -1.0 : (cz > 1.0 ? 1.0 : cz);
    double theta = acos(cz);
    const double theta_min = kPi, theta_max = 0.0;  // acos(-1), acos(1)
    *v = __ddiv_rn(__dsub_rn(theta, theta_min), __dsub_rn(theta_max, theta_min));
}

// ---------------------------------------------------------------------------------------------
// The traversal kernel.  Persistent warps pull rays from a global cursor; every lane owns one ray
// at a time.  Control flow is kept warp-uniform (all 32 lanes vote on every loop exit):
//   * interior phase: lanes walk Node64 records; a lane that reaches a leaf parks it ("postponed
//     leaf") and keeps walking speculatively until every lane that has work holds a leaf
//     (Aila & Laine's speculative while-while) — box tests done while waiting are never wasted
//     on correctness: they can only visit subtrees a later, closer hit would have culled;
//   * leaf phase: every parked leaf is tested in f64;
//   * refill: when at least kRefill lanes have finished their ray the warp takes that many new
//     rays with one atomicAdd (rays are Morton-sorted by sort_rays, so neighbours in the queue
//     are neighbours in space and the refilled lanes re-join warm cache lines).
// ---------------------------------------------------------------------------------------------
constexpr int32_t kDone = 0x7fffffff;  // "stack empty": a positive value no node index reaches
constexpr int32_t kNoLeaf = 0;         // leaf references are negative, so 0 means "none parked"
#ifndef RRT_REFILL
#define RRT_REFILL 8
#endif
#ifndef RRT_NODE32
#define RRT_NODE32 1  // 0: never quantise, 1: per scene (quantise when the grid is fine enough), 2: always
#endif
#ifndef RRT_STATS
#define RRT_STATS 0
#endif
#ifndef RRT_WALK_MIN
#define RRT_WALK_MIN 12
#endif
#ifndef RRT_LEAF_MIN
#define RRT_LEAF_MIN 8
#endif
#ifndef RRT_LEAFQ
#define RRT_LEAFQ 3  // postponed leaves per lane (measured: with one, 10 of 32 lanes stand at their second leaf)
#endif
static_assert(RRT_LEAFQ >= 2, "the leaf queue holds the head leaf and at least one more");
#ifndef RRT_MINBLOCKS
#define RRT_MINBLOCKS 7  // Node64 kernels: 72 registers
#endif
#ifndef RRT_MINBLOCKS_Q
#define RRT_MINBLOCKS_Q 8  // Node32 kernels: 64 registers (measured best, profiles/r1_sweep8.txt)
#endif
constexpr int kRefill = RRT_REFILL;


// GEN: the scene holds spheres that need the object-space test (PRIM_SPHERE_GENERAL); every other scene runs the
// instantiation without that branch, whose register allocation is the measured one.
template <bool ANY, bool WIDE, bool QUANT, bool GEN>
__global__ void __launch_bounds__(kBlock, QUANT ? RRT_MINBLOCKS_Q : RRT_MINBLOCKS) trace_kernel(AggView A, uint64_t n, const rrt_ray* __restrict__ rays,
                                                        rrt_hit* __restrict__ hits, uint8_t* __restrict__ occluded,
                                                        const uint32_t* __restrict__ perm,
                                                        const uint32_t* __restrict__ use_perm,
                                                        unsigned long long* __restrict__ cursor,
                                                        const uint32_t* __restrict__ n_dev, int /*stack_levels*/) {
    const unsigned FULL = 0xffffffffu;
    if (n_dev) n = *n_dev;  // wavefront queues: the batch size lives on the device
    const unsigned lane = threadIdx.x & 31u;
    const Node64* __restrict__ nodes = static_cast<const Node64*>(A.nodes);
    const bool permuted = perm != nullptr && (use_perm == nullptr || *use_perm != 0u);

    // Traversal stack: entirely in shared memory, laid out [level][thread] so that 32 lanes at 32
    // different depths still hit 32 different banks (one wavefront per push / pop).  Level 0 holds
    // the "stack empty" marker, so a pop never needs an underflow test.  The launch sizes it from
    // the tree depth (trace_smem_bytes).
    extern __shared__ int32_t sstack[];
    int32_t* const my_stack = sstack + threadIdx.x;
#define RRT_POP()                     \
    do {                              \
        --sp;                         \
        node = my_stack[sp * kBlock]; \
    } while (0)
    int sp = 1;
    int32_t node = kDone;     // >= 0 interior index, < 0 leaf reference, kDone = nothing left
    int32_t leaf = kNoLeaf;   // parked leaf reference (head of the queue)
    int32_t lq[RRT_LEAFQ - 1];  // further parked leaves: the walk goes on past RRT_LEAFQ untested leaves
#pragma unroll
    for (int k = 0; k < RRT_LEAFQ - 1; ++k) lq[k] = kNoLeaf;
    // filled front to back, so the queue is full exactly when its last slot is taken
#define RRT_PARK()                                         \
    do {                                                   \
        bool placed_ = false;                              \
        if (leaf == kNoLeaf) {                             \
            leaf = node;                                   \
            placed_ = true;                                \
        }                                                  \
        _Pragma("unroll") for (int k_ = 0; k_ < RRT_LEAFQ - 1; ++k_) { \
            if (!placed_ && lq[k_] == kNoLeaf) {           \
                lq[k_] = node;                             \
                placed_ = true;                            \
            }                                              \
        }                                                  \
    } while (0)
    bool have_ray = false;
    bool exhausted = false;   // the global queue is empty (warp-uniform)
    uint64_t ray_index = 0;
    D3 o = {0, 0, 0}, d = {0, 0, 0};
    RayF rf = {0, 0, 0, 0, 0, 0};
    double best_t = 0.0;
    float t_shift = 0.0f, tcull = 0.0f;
    uint32_t best_id = RRT_NO_HIT, best_rec = 0;
    bool found = false;
#if RRT_STATS  // diagnostic build: where do the lanes of an interior / leaf trip stand? (tools/sweep.py "STATS=1")
    unsigned long long st_trips = 0, st_walk = 0, st_noray = 0, st_drained = 0, st_second = 0, st_ltrips = 0, st_lact = 0;
#endif

    for (;;) {
        // ---- retire finished rays, refill idle lanes ----
        const bool finished = have_ray && node == kDone && leaf == kNoLeaf;
        if (finished) {
            if (ANY) {
                occluded[ray_index] = found ? 1 : 0;
            } else {
                double bu = 0.0, bv = 0.0;
                const bool got = best_id != RRT_NO_HIT;
                if (got) hit_params<WIDE>(A, best_rec, o, d, best_t, &bu, &bv);
                double2* hp = reinterpret_cast<double2*>(hits + ray_index);
                double2 w0, w1;
                w0.x = __hiloint2double(0, (int)best_id);
                w0.y = got ? best_t : 0.0;
                w1.x = bu;
                w1.y = bv;
                __stcs(hp, w0);
                __stcs(hp + 1, w1);
            }
            have_ray = false;
        }
        const unsigned idle = __ballot_sync(FULL, !have_ray);
        if (idle != 0u && !exhausted && (__popc(idle) >= kRefill)) {
            const int want = __popc(idle);
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(cursor, (unsigned long long)want);
            base = __shfl_sync(FULL, base, 0);
            if (base + (unsigned long long)want >= n) exhausted = true;
            if (!have_ray) {
                const unsigned long long q = base + (unsigned long long)__popc(idle & ((1u << lane) - 1u));
                if (q < n) {
                    ray_index = permuted ? (uint64_t)__ldcs(perm + q) : (uint64_t)q;  // read once: streaming
                    const double2* rp = reinterpret_cast<const double2*>(rays + ray_index);
                    const double2 q0 = __ldcs(rp), q1 = __ldcs(rp + 1), q2 = __ldcs(rp + 2), q3 = __ldcs(rp + 3);
                    o = {q0.x, q0.y, q1.x};
                    d = {q1.y, q2.x, q2.y};
                    best_t = q3.x;
                    best_id = RRT_NO_HIT;
                    found = false;
                    have_ray = true;
                    sp = 1;
                    my_stack[0] = kDone;
                    leaf = kNoLeaf;
#pragma unroll
                    for (int k = 0; k < RRT_LEAFQ - 1; ++k) lq[k] = kNoLeaf;
                    const bool live = prepare_ray(A, o, d, best_t, &t_shift, &rf) && !(best_t < 0.0);
                    node = live ? A.root : kDone;
                    tcull = __double2float_ru(best_t - (double)t_shift);
                }
            }
        }
        if (__ballot_sync(FULL, have_ray) == 0u) {
            if (exhausted) break;
            continue;  // fewer than kRefill idle lanes cannot happen here (all 32 are idle)
        }

        // ---- interior phase ----
        for (;;) {
#pragma unroll
          for (int step = 0; step < RRT_UNROLL; ++step) {
            const bool walking = node >= 0 && node != kDone;
#if RRT_STATS
            st_trips += 1;
            st_walk += __popc(__ballot_sync(FULL, walking));
            st_noray += __popc(__ballot_sync(FULL, !have_ray));
            st_drained += __popc(__ballot_sync(FULL, have_ray && node == kDone));
            st_second += __popc(__ballot_sync(FULL, have_ray && node < 0));
#endif
            if (walking) {
                int32_t ch_x, ch_y;
                float tn0, tn1;
                bool h0, h1;
                if (QUANT) {
                    // one 256-bit load: 12 quantised planes + two child references; a plane becomes the float
                    // 1 + q / 32768 with one byte permute (device_layout.h)
                    const F8 v = ldg256(reinterpret_cast<const char*>(A.nodes) + (size_t)node * sizeof(Node32));
                    const uint32_t w0 = __float_as_uint(v.a), w1 = __float_as_uint(v.b), w2 = __float_as_uint(v.c);
                    const uint32_t w3 = __float_as_uint(v.d), w4 = __float_as_uint(v.e), w5 = __float_as_uint(v.f);
                    ch_x = __float_as_int(v.g);
                    ch_y = __float_as_int(v.h);
                    h0 = slab(rf, qlo(w0), qhi(w0), qlo(w1), qhi(w1), qlo(w2), qhi(w2), tcull, &tn0);
                    h1 = slab(rf, qlo(w3), qhi(w3), qlo(w4), qhi(w4), qlo(w5), qhi(w5), tcull, &tn1);
                } else {
                    const char* np = reinterpret_cast<const char*>(nodes + node);
                    const F8 lo = ldg256(np);        // c0 x/y slabs, c1 x/y slabs
                    const F8 hi = ldg256(np + 32);   // z slabs of both, child references
                    ch_x = __float_as_int(hi.e);
                    ch_y = __float_as_int(hi.f);
                    h0 = slab(rf, lo.a, lo.b, lo.c, lo.d, hi.a, hi.b, tcull, &tn0);
                    h1 = slab(rf, lo.e, lo.f, lo.g, lo.h, hi.c, hi.d, tcull, &tn1);
                }
                // branch-free step: both hit -> push the far child, go near; one hit -> go there;
                // none -> pop
                const bool both = h0 && h1;
                const bool swap = !ANY && (tn1 < tn0);
                const int32_t near_c = swap ? ch_y : ch_x, far_c = swap ? ch_x : ch_y;
                if (both) my_stack[sp * kBlock] = far_c;
                sp += both ? 1 : 0;
                node = both ? near_c : (h0 ? ch_x : ch_y);
                if (!(h0 || h1)) RRT_POP();
            }
            if (node < 0 && lq[RRT_LEAFQ - 2] == kNoLeaf) {  // park the leaf, keep walking
                RRT_PARK();
                RRT_POP();
            }
          }
            // leave when no lane is still looking for its first leaf
            if (!__any_sync(FULL, leaf == kNoLeaf && node != kDone)) break;
#if RRT_WALK_MIN > 0
            // ... or when too few lanes are left walking to fill the warp (the rest stand at a full leaf queue or
            // have emptied their stack): the searching lanes resume after the leaf phase
            if (__popc(__ballot_sync(FULL, node >= 0 && node != kDone)) < RRT_WALK_MIN) break;
#endif
        }

        // ---- leaf phase ----
#if RRT_LEAF_MIN > 0
        // a leaf trip is worth its ~150 f64 instructions only with enough lanes in it: below RRT_LEAF_MIN the
        // remaining leaves stay queued while the others walk on — unless nobody is left to walk
        for (;;) {
            const unsigned with_leaf = __ballot_sync(FULL, leaf != kNoLeaf);
            if (with_leaf == 0u) break;
            if (__popc(with_leaf) < RRT_LEAF_MIN && __any_sync(FULL, node >= 0 && node != kDone)) break;
#else
        while (__any_sync(FULL, leaf != kNoLeaf)) {
#endif
#if RRT_STATS
            st_ltrips += 1;
            st_lact += __popc(__ballot_sync(FULL, leaf != kNoLeaf));
#endif
            if (leaf != kNoLeaf) {
                const uint32_t ref = ~(uint32_t)leaf;
                const uint32_t first = ref >> 3, cnt = (ref & 7u) + 1u;
                // every record of the leaf through the deciding arithmetic: f64, reference operation order
                uint32_t cand = (1u << cnt) - 1u;
                while (cand != 0u) {
                    const uint32_t k = (uint32_t)__ffs((int)cand) - 1u;
                    cand &= cand - 1u;
                    D3 a, b, c;
                    uint32_t pid, kind;
                    load_prim<WIDE>(A.prims, first + k, &a, &b, &c, &pid, &kind);
                    double t, u, v;
                    bool hit;
                    if (kind == PRIM_TRIANGLE) {
                        hit = tri_test(o, d, a, b, c, &t, &u, &v) && !(t > best_t);
                    } else if (!GEN || kind == PRIM_SPHERE) {
                        hit = sphere_test(o, d, a, b.x, best_t, &t);
                    } else {
                        hit = general_sphere_test(A, a.x, o, d, best_t, &t);
                    }
                    if (hit) {
                        if (ANY) {
                            found = true;
                            break;
                        }
                        // Tier F accept rule: closest t, exact ties go to the lowest prim id
                        if (t < best_t || best_id == RRT_NO_HIT || pid < best_id) {
                            best_t = t;
                            best_id = pid;
                            best_rec = first + k;
                            tcull = __double2float_ru(best_t - (double)t_shift);
                        }
                    }
                }
                leaf = lq[0];
#pragma unroll
                for (int k = 0; k < RRT_LEAFQ - 2; ++k) lq[k] = lq[k + 1];
                lq[RRT_LEAFQ - 2] = kNoLeaf;
                if (ANY && found) {
                    node = kDone;
                    leaf = kNoLeaf;
#pragma unroll
                    for (int k = 0; k < RRT_LEAFQ - 1; ++k) lq[k] = kNoLeaf;
                } else if (node < 0) {  // the walk stands at one more leaf: it takes the slot that came free
                    RRT_PARK();
                    RRT_POP();
                }
            }
        }
    }
#if RRT_STATS
    if (lane == 0) {
        atomicAdd(cursor + 2, st_trips);
        atomicAdd(cursor + 3, st_walk);
        atomicAdd(cursor + 4, st_noray);
        atomicAdd(cursor + 5, st_drained);
        atomicAdd(cursor + 6, st_second);
        atomicAdd(cursor + 7, st_ltrips);
        atomicAdd(cursor + 8, st_lact);
    }
#endif
#undef RRT_POP
#undef RRT_PARK
}

// ---------------------------------------------------------------------------------------------
// Ray sorting: a counting sort of ray indices by the Morton code of the ray origin (7 bits per
// axis inside the world box, + the direction octant).  Incoherent batches become queues whose
// neighbours start in the same ~1/128 cell, which is what keeps a warp's 32 walks on the same
// cache lines.  Batches that are already coherent (camera rays: one origin -> one huge bin)
// are detected by the largest bin and left in input order (use_perm = 0).
// ---------------------------------------------------------------------------------------------
#ifndef RRT_SORTBITS
#define RRT_SORTBITS 7
#endif
constexpr int kSortBits = RRT_SORTBITS;
constexpr uint32_t kSortBins = (1u << (3 * kSortBits)) * 8u;

__device__ __forceinline__ uint32_t spread3(uint32_t x) {  // 10 bits -> every third bit
    x = (x | (x << 16)) & 0x030000FFu;
    x = (x | (x << 8)) & 0x0300F00Fu;
    x = (x | (x << 4)) & 0x030C30C3u;
    x = (x | (x << 2)) & 0x09249249u;
    return x;
}

__device__ __forceinline__ uint32_t ray_key(const AggView& A, const rrt_ray* r, int bits) {
    const double2* rp = reinterpret_cast<const double2*>(r);
    const double2 q0 = __ldg(rp), q1 = __ldg(rp + 1), q2 = __ldg(rp + 2);
    const double o[3] = {q0.x, q0.y, q1.x};
    const double dd[3] = {q1.y, q2.x, q2.y};
    uint32_t c[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        double ext = A.world_hi[k] - A.world_lo[k];
        double f = ext > 0.0 ? (o[k] - A.world_lo[k]) / ext : 0.0;
        f = f < 0.0 ? 0.0 : (f > 1.0 ? 1.0 : f);
        if (!(f == f)) f = 0.0;
        uint32_t q = (uint32_t)(f * (double)(1u << bits));
        c[k] = q >= (1u << bits) ? (1u << bits) - 1u : q;
    }
    const uint32_t cell = spread3(c[0]) | (spread3(c[1]) << 1) | (spread3(c[2]) << 2);
    const uint32_t oct = (dd[0] < 0.0 ? 1u : 0u) | (dd[1] < 0.0 ? 2u : 0u) | (dd[2] < 0.0 ? 4u : 0u);
    if (A.sort_mode == 0) return cell;
    if (A.sort_mode == 2) return (oct << (3 * bits)) | cell;
    return (cell << 3) | oct;
}

// (grid-stride: the wavefront renderer launches these for a queue's CAPACITY while the live count sits on the device;
// a grid of a few CTAs per SM walks whatever is there instead of tens of thousands of CTAs that find nothing)
__global__ void __launch_bounds__(256) sort_count_kernel(AggView A, uint64_t n, const rrt_ray* __restrict__ rays,
                                                          uint32_t* __restrict__ bins, uint32_t* __restrict__ key_out,
                                                          uint32_t* __restrict__ rank_out,
                                                          const uint32_t* __restrict__ n_dev, int bits) {
    if (n_dev) n = *n_dev;
    const unsigned lane = threadIdx.x & 31u;
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < n; base += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t i = base + threadIdx.x;
        const bool valid = i < n;
        const uint32_t key = valid ? ray_key(A, rays + i, bits) : 0xFFFFFFFFu;
        // one atomic per distinct key per warp
        const unsigned peers = __match_any_sync(0xffffffffu, key);
        const int leader = __ffs(peers) - 1;
        uint32_t first = 0;
        if (valid && (int)lane == leader) first = atomicAdd(bins + key, (uint32_t)__popc(peers));
        first = __shfl_sync(0xffffffffu, first, leader);
        if (valid) {
            key_out[i] = key;
            rank_out[i] = first + (uint32_t)__popc(peers & ((1u << lane) - 1u));
        }
    }
}

// Exclusive scan of the bins in three small launches (per-block sums, scan of the sums, apply).
constexpr int kScanBlock = 1024;
__global__ void __launch_bounds__(kScanBlock) scan_block_kernel(uint32_t* __restrict__ bins, uint32_t nbins,
                                                                 uint32_t* __restrict__ block_sums,
                                                                 uint32_t* __restrict__ max_bin) {
    __shared__ uint32_t warp_sums[32];
    const uint32_t i = blockIdx.x * kScanBlock + threadIdx.x;
    const uint32_t v = i < nbins ? bins[i] : 0u;
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, x, off);
        if ((int)lane >= off) x += y;
    }
    uint32_t m = v;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, off));
    if (lane == 31) warp_sums[warp] = x;
    if (lane == 0 && m > 0) atomicMax(max_bin, m);
    __syncthreads();
    if (warp == 0) {
        uint32_t w = warp_sums[lane];
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, w, off);
            if ((int)lane >= off) w += y;
        }
        warp_sums[lane] = w;
    }
    __syncthreads();
    const uint32_t incl = x + (warp > 0 ? warp_sums[warp - 1] : 0u);
    if (i < nbins) bins[i] = incl - v;  // exclusive within the block
    if (threadIdx.x == kScanBlock - 1) block_sums[blockIdx.x] = incl;
}
__global__ void __launch_bounds__(kScanBlock) scan_sums_kernel(uint32_t* __restrict__ block_sums, uint32_t nblocks,
                                                                const uint32_t* __restrict__ max_bin, uint64_t n,
                                                                uint32_t* __restrict__ use_perm,
                                                                const uint32_t* __restrict__ n_dev) {
    if (n_dev) n = *n_dev;
    // nblocks <= kScanBlock * 16: a serial carry over chunks of kScanBlock
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) {
        carry = 0;
        // coherent batches (one bin holding > 1/64 of the rays, and at least 4096) keep input order
        const uint32_t mb = *max_bin;
        *use_perm = (((uint64_t)mb * 64u > n && mb >= 4096u) || n < 4096u) ? 0u : 1u;
    }
    __syncthreads();
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    for (uint32_t base = 0; base < nblocks; base += kScanBlock) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < nblocks ? block_sums[i] : 0u;
        uint32_t x = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, x, off);
            if ((int)lane >= off) x += y;
        }
        if (lane == 31) warp_sums[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = warp_sums[lane];
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                uint32_t y = __shfl_up_sync(0xffffffffu, w, off);
                if ((int)lane >= off) w += y;
            }
            warp_sums[lane] = w;
        }
        __syncthreads();
        const uint32_t incl = x + (warp > 0 ? warp_sums[warp - 1] : 0u) + carry;
        if (i < nblocks) block_sums[i] = incl - v;
        __syncthreads();
        if (threadIdx.x == kScanBlock - 1) carry = incl;
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256) sort_scatter_kernel(uint64_t n, const uint32_t* __restrict__ bins,
                                                            const uint32_t* __restrict__ block_sums,
                                                            const uint32_t* __restrict__ key,
                                                            const uint32_t* __restrict__ rank,
                                                            const uint32_t* __restrict__ use_perm,
                                                            uint32_t* __restrict__ perm,
                                                            const uint32_t* __restrict__ n_dev) {
    if (n_dev) n = *n_dev;
    if (*use_perm == 0u) return;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t k = key[i];
        perm[bins[k] + block_sums[k / kScanBlock] + rank[i]] = (uint32_t)i;
    }
}

// ---- trace_kernel launch facts: which instantiation, how much dynamic shared memory ----
using TraceKernel = decltype(&trace_kernel<false, false, false, false>);

// table[wide | any << 1 | quant << 2 | gen << 3]
template <int... V>
TraceKernel trace_kernel_table(int v, std::integer_sequence<int, V...>) {
    static const TraceKernel table[] = {trace_kernel<(V & 2) != 0, (V & 1) != 0, (V & 4) != 0, (V & 8) != 0>...};
    return table[v];
}
// The instantiation that serves one launch: any hit or closest hit, PrimRec96 records, Node32 nodes, general spheres.
TraceKernel trace_kernel_for(bool any, bool wide, bool quant, bool gen) {
    return trace_kernel_table((wide ? 1 : 0) | (any ? 2 : 0) | (quant ? 4 : 0) | (gen ? 8 : 0),
                              std::make_integer_sequence<int, 16>{});
}

// The traversal stack, stack_levels entries per thread, is all of trace_kernel's dynamic shared memory.
size_t trace_smem_bytes(int stack_levels) { return (size_t)stack_levels * kBlock * sizeof(int32_t); }

inline float round_down(double v) {
    float f = (float)v;
    if ((double)f > v) f = std::nextafterf(f, -INFINITY);
    return f;
}
inline float round_up(double v) {
    float f = (float)v;
    if ((double)f < v) f = std::nextafterf(f, INFINITY);
    return f;
}

// Splits [0, n) over the host threads (per-primitive loops of the commit: baking, record packing).
template <class F>
void parallel_ranges(size_t n, F f) {
    unsigned t = std::thread::hardware_concurrency();
    if (t == 0) t = 1;
    if (t > 32) t = 32;
    if (n < 65536 || t == 1) {
        f((size_t)0, n);
        return;
    }
    std::vector<std::thread> pool;
    const size_t step = (n + t - 1) / t;
    for (unsigned k = 0; k < t; ++k) {
        const size_t a = (size_t)k * step, b = std::min(n, a + step);
        if (a >= b) break;
        pool.emplace_back([=]() { f(a, b); });
    }
    for (auto& th : pool) th.join();
}

// Node32 when the grid costs the primitive boxes little (see DeviceAggregate::build): `growth` is the sum over the
// primitive boxes of min(1, grid_cells / half-perimeter).  RRT_QUANTISE overrides.
bool quantise_for(double growth, size_t n) {
    bool quantise = RRT_NODE32 == 2;
    if (RRT_NODE32 == 1) quantise = growth / (double)n < 0.05;
    if (const char* e = std::getenv("RRT_QUANTISE")) quantise = atoi(e) != 0;
    return quantise;
}
double grid_cells(const float grid_ext[3]) {
    return 2.0 * ((double)grid_ext[0] + (double)grid_ext[1] + (double)grid_ext[2]) / 32768.0;
}

// The device builder makes ONE-primitive leaves whatever max_prims_in_node says (Tier-F answers do not depend on
// it): without SAH the collapsed 2-4 primitive leaves cost more f64 tests than they save nodes — measured 1364
// (1) / 1261 (2) / 1076 (4) Mrays/s on config 3 (profiles/r1_bench_build_lbvh.txt).  RRT_LBVH_LEAF overrides.
uint32_t lbvh_leaf_for(uint32_t max_prims_in_node) {
    const uint32_t max_leaf = max_prims_in_node == 0 ? 4 : (max_prims_in_node > 8 ? 8 : max_prims_in_node);
    uint32_t lbvh_leaf = 1;
    if (const char* e = std::getenv("RRT_LBVH_LEAF")) lbvh_leaf = (uint32_t)std::max(1, std::min(8, atoi(e)));
    return std::min(max_leaf, lbvh_leaf);
}

#define RRT_CUDA(call)                                                                  \
    do {                                                                                \
        cudaError_t e_ = (call);                                                        \
        if (e_ != cudaSuccess) {                                                        \
            if (err) *err = std::string(#call) + ": " + cudaGetErrorString(e_);         \
            return RRT_ERR_CUDA;                                                        \
        }                                                                               \
    } while (0)

}  // namespace

int bake_world(const HostScene& scene, WorldBake* out, std::string* err) {
    const size_t n = scene.prims.size();
    BakedPrim* const world = out->world.get();
    Aabb* const boxes = out->boxes.get();
    uint8_t* const kind = out->kind.get();
    uint8_t* const exact = out->exact.get();
    // (default-initialised buffers: the worker threads below touch — and so place — their own pages; a value-initialised
    // std::vector would zero half a gigabyte on one thread first: measured 170 -> see profiles/r2_build_timing.txt)
    std::atomic<int> not_fp32{0}, clipped_with_own_transform{0};
    parallel_ranges(n, [&](size_t i0, size_t i1) {
    bool all_fp32 = true;
    for (size_t i = i0; i < i1; ++i) {
        const Primitive& pr = scene.prims[i];
        new (&boxes[i]) Aabb();
        exact[i] = 1;
        if (pr.kind == SHAPE_TRIANGLE) {
            kind[i] = PRIM_TRIANGLE;
            scene.world_triangle(i, world[i].v);
            bake::triangle_box(world[i].v, boxes[i].lo, boxes[i].hi);
            exact[i] = bake::fp32_exact(world[i].v, 9) ? 1 : 0;
            if (!exact[i]) all_fp32 = false;
        } else {
            for (int k = 0; k < 9; ++k) world[i].v[k] = 0.0;  // a PrimRec96 copies all nine
            kind[i] = PRIM_SPHERE;
            const Sphere& s = scene.spheres[pr.shape];
            auto general_sphere = [&]() {
                // box of the object-space extent [-r, r]^2 x [z_min, z_max] (Sphere::object_bound, sphere.rs:262-268)
                // carried to world space corner by corner; the GenSphere entry itself is made after this loop
                kind[i] = PRIM_SPHERE_GENERAL;
                const double zl = std::fmax(std::fmin(s.z_min, s.z_max), -s.radius), zh = std::fmin(std::fmax(s.z_min, s.z_max), s.radius);
                for (int k = 0; k < 8; ++k) {
                    Vec3d q = s.obj_to_world.point(Vec3d{(k & 1) ? s.radius : -s.radius, (k & 2) ? s.radius : -s.radius, (k & 4) ? zh : zl});
                    if (pr.instance >= 0) q = scene.instances[pr.instance].point(q);
                    const double pad = 1e-12 * (std::fabs(q.x) + std::fabs(q.y) + std::fabs(q.z) + s.radius);
                    const double lo[3] = {q.x - pad, q.y - pad, q.z - pad}, hi[3] = {q.x + pad, q.y + pad, q.z + pad};
                    boxes[i].grow(lo);
                    boxes[i].grow(hi);
                }
            };
            if (!s.is_full()) {
                // Q5a (sphere.rs:157): the first root is clipped by the z / phi of the INSTANCE-space point.  With a
                // transform of the sphere's own that accepts points outside the shape's bound, which the reference
                // finds only when the ray happens to cross the leaf's box: the answer depends on the tree.  A clipped
                // sphere is therefore placed through instances[] (as config 4 places its spheres), where both spaces
                // are one and the same.
                if (!s.obj_to_world.is_identity()) {
                    clipped_with_own_transform = 1;
                    continue;
                }
                general_sphere();
                continue;
            }
            // world centre; the instance / object transforms must be rigid (unit scale)
            Vec3d c = s.obj_to_world.point(Vec3d{0, 0, 0});
            Vec3d ex = s.obj_to_world.vector(Vec3d{1, 0, 0}), ey = s.obj_to_world.vector(Vec3d{0, 1, 0}),
                  ez = s.obj_to_world.vector(Vec3d{0, 0, 1});
            if (pr.instance >= 0) {
                const Transform& t = scene.instances[pr.instance];
                c = t.point(c);
                ex = t.vector(ex);
                ey = t.vector(ey);
                ez = t.vector(ez);
            }
            auto len = [](Vec3d a) { return std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); };
            auto dt = [](Vec3d a, Vec3d b) { return a.x * b.x + a.y * b.y + a.z * b.z; };
            double tol = 1e-9;
            if (std::fabs(len(ex) - 1) > tol || std::fabs(len(ey) - 1) > tol || std::fabs(len(ez) - 1) > tol ||
                std::fabs(dt(ex, ey)) > tol || std::fabs(dt(ex, ez)) > tol || std::fabs(dt(ey, ez)) > tol) {
                general_sphere();
                continue;
            }
            world[i].v[0] = c.x;
            world[i].v[1] = c.y;
            world[i].v[2] = c.z;
            world[i].v[3] = s.radius;
            double lo[3] = {c.x - s.radius, c.y - s.radius, c.z - s.radius};
            double hi[3] = {c.x + s.radius, c.y + s.radius, c.z + s.radius};
            // one ulp of slack: centre +- r is rounded
            for (int k = 0; k < 3; ++k) {
                lo[k] = std::nextafter(lo[k], -INFINITY);
                hi[k] = std::nextafter(hi[k], INFINITY);
            }
            boxes[i].grow(lo);
            boxes[i].grow(hi);
        }
    }
    if (!all_fp32) not_fp32 = 1;
    });
    if (clipped_with_own_transform) {
        if (err)
            *err = "a sphere clipped by z_min / z_max / phi_max must get its placement from instances[], not from a transform of "
                   "its own: the reference clips the first root in instance space (Q5a) and its answer then depends on the tree";
        return RRT_ERR_UNSUPPORTED;
    }
    out->gspheres.clear();
    for (size_t i = 0; i < n; ++i) {
        if (kind[i] != PRIM_SPHERE_GENERAL) continue;
        const Primitive& pr = scene.prims[i];
        const Sphere& s = scene.spheres[pr.shape];
        GenSphere g{};
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 4; ++c) {
                g.inst_inv.m[4 * r + c] = pr.instance >= 0 ? scene.instances[pr.instance].inv.m[r][c] : (r == c ? 1.0 : 0.0);
                g.w2o.m[4 * r + c] = s.obj_to_world.inv.m[r][c];
            }
        // Sphere::new (sphere.rs:28-47)
        const double kPiD = 3.14159265358979323846264338327950288;
        g.clip.radius = s.radius;
        g.clip.z_min = s.z_min;
        g.clip.z_max = s.z_max;
        g.theta_min = std::acos(std::fmin(std::fmax(std::fmin(s.z_min, s.z_max) / s.radius, -1.0), 1.0));
        g.theta_max = std::acos(std::fmin(std::fmax(std::fmax(s.z_min, s.z_max) / s.radius, -1.0), 1.0));
        g.clip.phi_max = std::fmin(std::fmax(s.phi_max_deg, 0.0), 360.0) * (kPiD / 180.0);
        world[i].v[0] = (double)out->gspheres.size();
        world[i].v[3] = s.radius;
        out->gspheres.push_back(g);
    }
    out->all_fp32 = not_fp32 == 0;
    out->has_spheres = false;
    for (const Primitive& pr : scene.prims) out->has_spheres |= pr.kind == SHAPE_SPHERE;
    out->inst_w2p.clear();
    if (out->has_spheres && !scene.instances.empty()) {
        out->inst_w2p.resize(12 * scene.instances.size());
        for (size_t i = 0; i < scene.instances.size(); ++i)
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 4; ++c) out->inst_w2p[12 * i + 4 * r + c] = scene.instances[i].inv.m[r][c];
    }
    return RRT_OK;
}

bool DeviceAggregate::device_tree_fits(size_t n, uint32_t max_prims_in_node) {
    const uint32_t max_leaf = max_prims_in_node == 0 ? 4 : (max_prims_in_node > 8 ? 8 : max_prims_in_node);
    return n > 16 && n > max_leaf;
}

DeviceAggregate::~DeviceAggregate() {
    if (d_nodes_) cudaFree(d_nodes_);
    if (d_prims_) cudaFree(d_prims_);
    if (d_inst_) cudaFree(d_inst_);
    if (d_gspheres_) cudaFree(d_gspheres_);
    for (auto& kv : ws_) {
        Workspace& w = kv.second;
        if (w.d_bins) cudaFree(w.d_bins);
        if (w.d_block_sums) cudaFree(w.d_block_sums);
        if (w.d_small) cudaFree(w.d_small);
        if (w.d_key) cudaFree(w.d_key);
        if (w.d_rank) cudaFree(w.d_rank);
        if (w.d_perm) cudaFree(w.d_perm);
        if (w.last_use) cudaEventDestroy(w.last_use);
    }
}

int DeviceAggregate::build(int device, const HostScene& scene, uint32_t max_prims_in_node, std::string* err, bool device_lbvh) {
    auto t_start = std::chrono::steady_clock::now();
    const bool timing = std::getenv("RRT_BUILD_TIMING") != nullptr;
    auto lap = [&, t_last = t_start](const char* what) mutable {
        if (!timing) return;
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "RRT_BUILD_TIMING %-22s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
        t_last = now;
    };
    device_ = device;
    const size_t n = scene.prims.size();
    if (n == 0) {
        if (err) *err = "BVHAccel::new needs at least one primitive (bvh.rs:319)";
        return RRT_ERR_EMPTY;
    }
    if (n >= (1u << 28)) {
        if (err) *err = "too many primitives for the 28-bit leaf reference";
        return RRT_ERR_UNSUPPORTED;
    }
    // ---- bake to world space ----
    WorldBake bake(n);
    if (int rc = bake_world(scene, &bake, err)) return rc;
    const BakedPrim* const world = bake.world.get();
    Aabb* const boxes = bake.boxes.get();
    const bool all_fp32 = bake.all_fp32;
    lap("bake to world space");
    // ---- frame: world box, fp32 margin, Node32 grid, node format ----
    Aabb world_box;
    {
        std::mutex m;
        parallel_ranges(n, [&](size_t i0, size_t i1) {
            Aabb part;
            for (size_t i = i0; i < i1; ++i) part.grow(boxes[i]);
            std::lock_guard<std::mutex> lock(m);
            world_box.grow(part);
        });
    }
    const NodeFrame frame = make_node_frame(world_box);
    const double delta = frame.delta;
    const double* grid_lo = frame.grid_lo;
    const float* grid_ext = frame.grid_ext;
    // The grid costs every box up to one cell per side.  That is nothing for a scene whose primitives are much
    // larger than extent / 32768 (configs 1-5: under 1% of a primitive box's half-perimeter), and it would ruin
    // the culling of a scene with small details in a huge box; such scenes keep the fp32 node.
    double growth = 0.0;
    if (RRT_NODE32 == 1) {
        const double cells = grid_cells(grid_ext);
        // (summed per contiguous range, then over the ranges in order: the same total whatever the thread count is not
        // guaranteed to the last bit, and does not need to be — it is compared with 5 %)
        std::mutex m;
        parallel_ranges(n, [&](size_t i0, size_t i1) {
            double part = 0.0;
            for (size_t i = i0; i < i1; ++i) {
                const double hp = (boxes[i].hi[0] - boxes[i].lo[0]) + (boxes[i].hi[1] - boxes[i].lo[1]) + (boxes[i].hi[2] - boxes[i].lo[2]);
                part += std::fmin(1.0, cells / std::fmax(hp, 1e-300));
            }
            std::lock_guard<std::mutex> lock(m);
            growth += part;
        });
    }
    const bool quantise = quantise_for(growth, n);
    const bool on_device = device_lbvh && device_tree_fits(n, max_prims_in_node);

    lap("frame + node format");
    // ---- tree ----
    Bvh2 tree;
    LbvhResult lb;
    bool on_device_ok = on_device;
    if (on_device) {
        int rc = build_lbvh_device(device, AabbSpan(boxes, n), lbvh_leaf_for(max_prims_in_node), delta, quantise, grid_lo, grid_ext, &lb, err);
        if (rc != RRT_OK) return rc;
        tree.max_depth = lb.max_depth + 1;
        tree.n_leaves = lb.n_leaves;
        if (tree.max_depth + 2 > (uint32_t)kStack) {
            // thousands of primitives with one centroid make a radix tree deeper than the traversal stack:
            // such scenes get the SAH tree (which splits equal centroids by count)
            cudaFree(lb.d_nodes);
            lb = LbvhResult();
            on_device_ok = false;
        }
    }
    if (!on_device_ok) {
        SahParams sp;
        sp.max_leaf = max_prims_in_node == 0 ? 4 : max_prims_in_node;
        if (const char* e = std::getenv("RRT_SAH_CI")) sp.cost_intersect = atof(e);
        // spatial splits (DESIGN.md §3); RRT_SBVH_CAP=1 builds the object-split tree, one reference per primitive
        if (const char* e = std::getenv("RRT_SBVH_ALPHA")) sp.split_alpha = atof(e);
        if (const char* e = std::getenv("RRT_SBVH_CAP")) sp.split_cap = atof(e);
        // spatial splits clip the triangles' world-space vertices; spheres stay whole references
        RawBuf<uint8_t> is_tri(n);
        bool all_tri = true;
        for (size_t i = 0; i < n; ++i) {
            is_tri[i] = scene.prims[i].kind == SHAPE_TRIANGLE ? 1 : 0;
            all_tri = all_tri && is_tri[i];
        }
        SplitTriangles tris;
        tris.verts = world->v;  // (BakedPrim is nine doubles: primitive i's vertices start at 9 i)
        tris.is_tri = all_tri ? nullptr : is_tri.get();
        build_sah(AabbSpan(boxes, n), tris, sp, &tree);
        if (tree.max_depth + 2 > (uint32_t)kStack) {
            // duplicated references can deepen a tree past the traversal stack; the object-split tree splits every
            // node by count at worst, and is the one such a scene gets
            tree = Bvh2();
            build_sah(AabbSpan(boxes, n), sp, &tree);
        }
    }
    if (tree.max_depth + 2 > (uint32_t)kStack) {
        if (on_device_ok) cudaFree(lb.d_nodes);
        if (err) *err = "tree deeper than the traversal stack (" + std::to_string(tree.max_depth) + " levels)";
        return RRT_ERR_UNSUPPORTED;
    }

    lap(on_device_ok ? "device LBVH (total)" : "host SAH tree");
    // ---- pack: interior nodes in DFS order, leaves become references ----
    std::vector<Node64> nodes;
    nodes.reserve(tree.nodes.size() / 2 + 2);
    const bool wide = !all_fp32;
    // one record per leaf reference (the device tree and the object-split host tree: one per primitive; spatial splits
    // reference a triangle from every leaf that holds a part of it) — every slot is written below
    const size_t n_refs = on_device_ok ? n : tree.order.size();
    RawBuf<PrimRec48> rec48(wide ? 0 : n_refs);
    RawBuf<PrimRec96> rec96(wide ? n_refs : 0);
    size_t n_rec = 0;  // host tree: records are appended leaf by leaf
    auto make_record = [&](uint32_t pi, size_t slot) {
        {
            const Primitive& pr = scene.prims[pi];
            if (wide) {
                PrimRec96 r;
                std::memset(&r, 0, sizeof(r));
                std::memcpy(r.v, world[pi].v, sizeof(double) * 9);
                r.prim_id = pi;
                r.kind = bake.kind[pi];
                r.pad[0] = pr.instance >= 0 ? (uint32_t)pr.instance : 0xFFFFFFFFu;
                rec96[slot] = r;
            } else {
                PrimRec48 r;
                std::memset(&r, 0, sizeof(r));
                if (pr.kind == SHAPE_TRIANGLE) {
                    for (int j = 0; j < 3; ++j) {
                        r.tri.v0[j] = (float)world[pi].v[j];
                        r.tri.v1[j] = (float)world[pi].v[3 + j];
                        r.tri.v2[j] = (float)world[pi].v[6 + j];
                    }
                    r.tri.prim_id = pi;
                    r.tri.kind = PRIM_TRIANGLE;
                } else {
                    for (int j = 0; j < 3; ++j) r.sph.c[j] = world[pi].v[j];
                    r.sph.radius = world[pi].v[3];
                    r.sph.prim_id = pi;
                    r.sph.kind = bake.kind[pi];
                    r.sph.instance = pr.instance >= 0 ? (uint32_t)pr.instance : 0xFFFFFFFFu;
                }
                rec48[slot] = r;
            }
        }
    };
    auto emit_leaf = [&](const Bvh2Node& nd) -> int32_t {
        uint32_t first = (uint32_t)n_rec;
        for (uint32_t k = 0; k < nd.count; ++k) make_record(tree.order[nd.first + k], n_rec++);
        return make_leaf_ref(first, nd.count);
    };
    auto set_child = [&](Node64& out, int which, const Aabb& b) {
        float lo[3], hi[3];
        for (int k = 0; k < 3; ++k) {
            lo[k] = round_down(b.lo[k] - delta);
            hi[k] = round_up(b.hi[k] + delta);
        }
        if (which == 0) {
            out.c0_lox = lo[0]; out.c0_hix = hi[0]; out.c0_loy = lo[1]; out.c0_hiy = hi[1];
            out.c0_loz = lo[2]; out.c0_hiz = hi[2];
        } else {
            out.c1_lox = lo[0]; out.c1_hix = hi[0]; out.c1_loy = lo[1]; out.c1_hiy = hi[1];
            out.c1_loz = lo[2]; out.c1_hiz = hi[2];
        }
    };
    if (on_device_ok) {
        // the device tree's leaves are runs of the sorted order: records simply follow it
        parallel_ranges(n, [&](size_t r0, size_t r1) {
            for (size_t r = r0; r < r1; ++r) make_record(lb.order[r], r);
        });
    } else {
        const Bvh2Node& root = tree.nodes[tree.root];
        if (root.count > 0) {
            // the whole scene fits one leaf: the root's two children both reference that leaf
            // (a candidate tested twice cannot change a closest or an any hit)
            Node64 r;
            std::memset(&r, 0, sizeof(r));
            set_child(r, 0, root.box);
            set_child(r, 1, root.box);
            r.child0 = emit_leaf(root);
            r.child1 = r.child0;
            nodes.push_back(r);
        } else {
            // Two passes.  (1) DECIDE: the slot of every interior node (sibling interiors get adjacent slots — one 128-byte
            // line —, the left subtree's descendants follow, then the right subtree's) and the first record of every leaf,
            // in the order a depth-first walk meets them — bvh_pack_plan.hpp: subtrees are planned side by side from the
            // builder's subtree totals, with the plan one thread's walk would make.  (2) All threads fill the slots and the
            // records.  (Filling inside the walk cost 1.3 s for 4 Mi triangles, the one-thread walk alone 0.25 s.)
            PackPlan pack;
            plan_parallel(tree, &pack, (int)std::max(1u, std::thread::hardware_concurrency()));
            const auto& plan = pack.slots;
            const auto& leaves = pack.leaves;
            n_rec = pack.n_records;
            nodes.resize(plan.size());
            parallel_ranges(plan.size(), [&](size_t i0, size_t i1) {
                for (size_t i = i0; i < i1; ++i) {
                    const Bvh2Node& nd = tree.nodes[plan[i].tn];
                    Node64 o;
                    std::memset(&o, 0, sizeof(o));
                    set_child(o, 0, tree.nodes[nd.left].box);
                    set_child(o, 1, tree.nodes[nd.right].box);
                    o.child0 = plan[i].child0;
                    o.child1 = plan[i].child1;
                    nodes[i] = o;
                }
            });
            parallel_ranges(leaves.size(), [&](size_t i0, size_t i1) {
                for (size_t i = i0; i < i1; ++i) {
                    const Bvh2Node& nd = tree.nodes[leaves[i].tn];
                    for (uint32_t k = 0; k < nd.count; ++k) make_record(tree.order[nd.first + k], (size_t)leaves[i].first + k);
                }
            });
        }
    }

    // ---- quantise the host tree: Node64 (fp32 planes) -> Node32 (15-bit planes on the grid) ----
    std::vector<Node32> nodes32;
    if (quantise && !on_device_ok) {
        nodes32.resize(nodes.size());
        // the device evaluates fmaf(f, ext / d, -(o - c) / d) in fp32: 11 roundings of magnitude <= 2 ext / |d|
        // (DESIGN.md §3), i.e. less than ext * 2^-20 in position; the planes move outward by twice that
        auto quant = [&](double plane, int k, bool upper) -> uint32_t {
            const double cell = (double)grid_ext[k] / 32768.0;
            const double margin = (double)grid_ext[k] * std::ldexp(1.0, -19);
            double q = upper ? std::ceil((plane + margin - grid_lo[k]) / cell) : std::floor((plane - margin - grid_lo[k]) / cell);
            if (q < 0.0) q = 0.0;
            if (q > 32767.0) q = 32767.0;
            return 0x8000u | (uint32_t)q;
        };
        parallel_ranges(nodes.size(), [&](size_t i0, size_t i1) {
        for (size_t i = i0; i < i1; ++i) {
            const Node64& s = nodes[i];
            Node32 o;
            o.p[0] = quant(s.c0_lox, 0, false) | (quant(s.c0_hix, 0, true) << 16);
            o.p[1] = quant(s.c0_loy, 1, false) | (quant(s.c0_hiy, 1, true) << 16);
            o.p[2] = quant(s.c0_loz, 2, false) | (quant(s.c0_hiz, 2, true) << 16);
            o.p[3] = quant(s.c1_lox, 0, false) | (quant(s.c1_hix, 0, true) << 16);
            o.p[4] = quant(s.c1_loy, 1, false) | (quant(s.c1_hiy, 1, true) << 16);
            o.p[5] = quant(s.c1_loz, 2, false) | (quant(s.c1_hiz, 2, true) << 16);
            o.child0 = s.child0;
            o.child1 = s.child1;
            nodes32[i] = o;
        }
        });
    }
    lap("pack nodes + records");
    // ---- upload ----
    RRT_CUDA(cudaSetDevice(device));
    const size_t node_bytes = on_device_ok ? lb.node_bytes : (quantise ? nodes32.size() * sizeof(Node32) : nodes.size() * sizeof(Node64));
    const void* node_src = quantise ? (const void*)nodes32.data() : (const void*)nodes.data();
    size_t prim_bytes = wide ? n_refs * sizeof(PrimRec96) : n_refs * sizeof(PrimRec48);
    if (on_device_ok) {
        d_nodes_ = lb.d_nodes;
    } else {
        RRT_CUDA(cudaMalloc(&d_nodes_, node_bytes));
        RRT_CUDA(cudaMemcpy(d_nodes_, node_src, node_bytes, cudaMemcpyHostToDevice));
    }
    RRT_CUDA(cudaMalloc(&d_prims_, prim_bytes));
    RRT_CUDA(cudaMemcpy(d_prims_, wide ? (const void*)rec96.get() : (const void*)rec48.get(), prim_bytes,
                        cudaMemcpyHostToDevice));
    if (int rc = upload_tables(bake.inst_w2p, bake.gspheres, err)) return rc;
    lap("upload");
    Built b;
    b.world_box = world_box;
    b.frame = frame;
    b.quantise = quantise;
    b.wide = wide;
    b.has_spheres = bake.has_spheres;
    b.n_nodes = on_device_ok ? lb.n_nodes : nodes.size();
    b.tree_device_usec = on_device_ok ? (uint64_t)(lb.device_ms * 1000.0f) : 0;
    b.n_leaves = tree.n_leaves;
    b.max_depth = tree.max_depth;
    b.node_bytes = node_bytes;
    b.prim_bytes = prim_bytes;
    b.n_records = n_refs;
    b.n_prims = n;
    install(b, t_start);
    return RRT_OK;
}

int DeviceAggregate::build_from_image(int device, MeshImage& image, uint32_t max_prims_in_node, bool* too_deep,
                                      std::string* err) {
    const auto t_start = std::chrono::steady_clock::now();
    const bool timing = std::getenv("RRT_BUILD_TIMING") != nullptr;
    auto lap = [&, t_last = t_start](const char* what) mutable {
        if (!timing) return;
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "RRT_BUILD_TIMING %-22s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
        t_last = now;
    };
    *too_deep = false;
    device_ = device;
    RRT_CUDA(cudaSetDevice(device));
    const size_t n = image.n_prims();
    // ---- frame: world box (device min / max, then make_node_frame on its 48 bytes), node format ----
    Aabb world_box;
    bool all_fp32 = true;
    if (int rc = image.frame(&world_box, &all_fp32, err)) return rc;
    const NodeFrame frame = make_node_frame(world_box);
    // The growth sum is a parallel sum on the device, rounded differently from the host's: only a scene within rounding
    // of the 5 % threshold can get the other node format than a fresh commit.
    double growth = 0.0;
    if (RRT_NODE32 == 1)
        if (int rc = image.growth(grid_cells(frame.grid_ext), &growth, err)) return rc;
    const bool quantise = quantise_for(growth, n);
    lap("frame + node format");
    // ---- tree ----
    LbvhResult lb;
    if (int rc = build_lbvh_device_boxes(device, image.boxes(), (uint32_t)n, lbvh_leaf_for(max_prims_in_node), frame.delta,
                                         quantise, frame.grid_lo, frame.grid_ext, &image.arena(), &lb, err))
        return rc;
    if (lb.max_depth + 1 + 2 > (uint32_t)kStack) {
        cudaFree(lb.d_nodes);
        *too_deep = true;
        return RRT_OK;
    }
    d_nodes_ = lb.d_nodes;
    lap("device LBVH (total)");
    // ---- records in tree order, tables ----
    const bool wide = !all_fp32;
    const size_t prim_bytes = n * (wide ? sizeof(PrimRec96) : sizeof(PrimRec48));
    RRT_CUDA(cudaMalloc(&d_prims_, prim_bytes));
    if (int rc = image.gather(lb.d_order, wide, d_prims_, err)) return rc;
    if (int rc = upload_tables(image.inst_w2p, image.gspheres, err)) return rc;
    RRT_CUDA(cudaStreamSynchronize(0));
    lap("records + tables");
    Built b;
    b.world_box = world_box;
    b.frame = frame;
    b.quantise = quantise;
    b.wide = wide;
    b.has_spheres = image.has_spheres;
    b.n_nodes = lb.n_nodes;
    b.tree_device_usec = (uint64_t)(lb.device_ms * 1000.0f);
    b.n_leaves = lb.n_leaves;
    b.max_depth = lb.max_depth + 1;
    b.node_bytes = lb.node_bytes;
    b.prim_bytes = prim_bytes;
    b.n_records = n;
    b.n_prims = n;
    install(b, t_start);
    return RRT_OK;
}

int DeviceAggregate::upload_tables(const std::vector<double>& inst_w2p, const std::vector<GenSphere>& gspheres, std::string* err) {
    if (!inst_w2p.empty()) {
        RRT_CUDA(cudaMalloc(&d_inst_, inst_w2p.size() * sizeof(double)));
        RRT_CUDA(cudaMemcpy(d_inst_, inst_w2p.data(), inst_w2p.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    if (!gspheres.empty()) {
        RRT_CUDA(cudaMalloc(&d_gspheres_, gspheres.size() * sizeof(GenSphere)));
        RRT_CUDA(cudaMemcpy(d_gspheres_, gspheres.data(), gspheres.size() * sizeof(GenSphere), cudaMemcpyHostToDevice));
    }
    inst_bytes_ = inst_w2p.size() * sizeof(double);
    gsphere_bytes_ = gspheres.size() * sizeof(GenSphere);
    return RRT_OK;
}

// The view, statistics and launch set-up of a built aggregate whose nodes, records and tables are on the device.
void DeviceAggregate::install(const Built& b, std::chrono::steady_clock::time_point t_start) {
    view_.gspheres = d_gspheres_;
    view_.inst_w2p = static_cast<const double*>(d_inst_);
    view_.has_spheres = b.has_spheres ? 1 : 0;
    view_.nodes = d_nodes_;
    view_.prims = d_prims_;
    for (int k = 0; k < 3; ++k) {
        view_.world_lo[k] = b.world_box.lo[k] - b.frame.delta;
        view_.world_hi[k] = b.world_box.hi[k] + b.frame.delta;
    }
    view_.scene_scale = b.frame.scale;
    for (int k = 0; k < 3; ++k) {
        view_.grid_c[k] = b.frame.grid_c[k];
        view_.grid_ext[k] = b.frame.grid_ext[k];
    }
    view_.quantised = b.quantise ? 1 : 0;
    view_.root = 0;
    view_.wide = b.wide ? 1 : 0;
    view_.sort_mode = 0;
    if (const char* e = std::getenv("RRT_SORT_MODE")) view_.sort_mode = atoi(e);
    if (const char* e = std::getenv("RRT_SORT")) sort_rays_ = atoi(e) != 0;
    stats_.n_nodes = b.n_nodes;
    stats_.tree_device_usec = b.tree_device_usec;
    stats_.n_leaves = b.n_leaves;
    stats_.max_depth = b.max_depth;
    stats_.device_bytes = b.node_bytes + b.prim_bytes;
    stats_.n_records = b.n_records;
    stats_.wide_records = b.wide;
    stats_.n_prims = b.n_prims;
    stats_.build_usec =
        (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t_start).count();
    stack_levels_ = (int)b.max_depth + 2;
    node_bytes_ = b.node_bytes;
    prim_bytes_ = b.prim_bytes;
    configure_kernels(b.quantise);
}

// the only shared memory is the traversal stack (one entry per tree level + the marker, trace_smem_bytes);
// everything else of the 256 KB stays L1
void DeviceAggregate::configure_kernels(bool quantise) {
    const size_t smem = trace_smem_bytes(stack_levels_);
    int carve = (int)(((quantise ? RRT_MINBLOCKS_Q : RRT_MINBLOCKS) * smem * 100 + 227 * 1024 - 1) / (227 * 1024)) + 2;
    if (carve > 100) carve = 100;
    for (int v = 0; v < 16; ++v) {
        const void* fn = (const void*)trace_kernel_for(v & 1, v & 2, v & 4, v & 8);
        // (the attribute belongs to the kernel, shared by every aggregate in the process: it is set to what the deepest
        // tree needs, so that configuring a shallower aggregate never refuses a deeper one's launch)
        cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)trace_smem_bytes(kStack));
        cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
    }
}

namespace {
struct BlobHeader {
    uint64_t magic, version;
    AggView view;          // device pointers are meaningless in the blob
    AggregateStats stats;
    int32_t stack_levels, sort_rays;
    uint64_t node_bytes, prim_bytes, inst_bytes, gsphere_bytes;
};
static_assert(sizeof(BlobHeader) == 280, "BlobHeader layout changed: bump the blob version");
constexpr uint64_t kBlobMagic = 0x3130454552545252ull;  // "RRTREE01"
}  // namespace

int DeviceAggregate::export_blob(void* buffer, uint64_t capacity, uint64_t* bytes, std::string* err) const {
    const uint64_t total = sizeof(BlobHeader) + node_bytes_ + prim_bytes_ + inst_bytes_ + gsphere_bytes_;
    *bytes = total;
    if (!buffer) return RRT_OK;
    if (capacity < total) {
        if (err) *err = "export_blob: buffer too small";
        return RRT_ERR_INVALID;
    }
    BlobHeader h{};
    h.magic = kBlobMagic;
    h.version = 1;
    h.view = view_;
    h.view.nodes = h.view.prims = h.view.gspheres = nullptr;
    h.view.inst_w2p = nullptr;
    h.stats = stats_;
    h.stack_levels = stack_levels_;
    h.sort_rays = sort_rays_ ? 1 : 0;
    h.node_bytes = node_bytes_;
    h.prim_bytes = prim_bytes_;
    h.inst_bytes = inst_bytes_;
    h.gsphere_bytes = gsphere_bytes_;
    char* out = static_cast<char*>(buffer);
    std::memcpy(out, &h, sizeof(h));
    out += sizeof(h);
    RRT_CUDA(cudaSetDevice(device_));
    RRT_CUDA(cudaMemcpy(out, d_nodes_, node_bytes_, cudaMemcpyDeviceToHost));
    out += node_bytes_;
    RRT_CUDA(cudaMemcpy(out, d_prims_, prim_bytes_, cudaMemcpyDeviceToHost));
    out += prim_bytes_;
    if (inst_bytes_) RRT_CUDA(cudaMemcpy(out, d_inst_, inst_bytes_, cudaMemcpyDeviceToHost));
    out += inst_bytes_;
    if (gsphere_bytes_) RRT_CUDA(cudaMemcpy(out, d_gspheres_, gsphere_bytes_, cudaMemcpyDeviceToHost));
    return RRT_OK;
}

int DeviceAggregate::import_blob(int device, const void* blob, uint64_t bytes, uint64_t n_prims_expected, std::string* err) {
    auto t_start = std::chrono::steady_clock::now();
    BlobHeader h;
    if (bytes < sizeof(h)) {
        if (err) *err = "import_blob: truncated";
        return RRT_ERR_INVALID;
    }
    std::memcpy(&h, blob, sizeof(h));
    if (h.magic != kBlobMagic || h.version != 1 ||
        bytes != sizeof(h) + h.node_bytes + h.prim_bytes + h.inst_bytes + h.gsphere_bytes) {
        if (err) *err = "import_blob: not a tree exported by this library version";
        return RRT_ERR_INVALID;
    }
    if (h.stats.n_prims != n_prims_expected) {
        if (err) *err = "import_blob: the tree was built over " + std::to_string(h.stats.n_prims) + " primitives, the scene holds " + std::to_string(n_prims_expected);
        return RRT_ERR_INVALID;
    }
    if (h.stack_levels < 2 || h.stack_levels > kStack) {
        if (err) *err = "import_blob: bad stack depth";
        return RRT_ERR_INVALID;
    }
    device_ = device;
    RRT_CUDA(cudaSetDevice(device));
    const char* in = static_cast<const char*>(blob) + sizeof(h);
    RRT_CUDA(cudaMalloc(&d_nodes_, h.node_bytes));
    RRT_CUDA(cudaMemcpy(d_nodes_, in, h.node_bytes, cudaMemcpyHostToDevice));
    in += h.node_bytes;
    RRT_CUDA(cudaMalloc(&d_prims_, h.prim_bytes));
    RRT_CUDA(cudaMemcpy(d_prims_, in, h.prim_bytes, cudaMemcpyHostToDevice));
    in += h.prim_bytes;
    if (h.inst_bytes) {
        RRT_CUDA(cudaMalloc(&d_inst_, h.inst_bytes));
        RRT_CUDA(cudaMemcpy(d_inst_, in, h.inst_bytes, cudaMemcpyHostToDevice));
    }
    in += h.inst_bytes;
    if (h.gsphere_bytes) {
        RRT_CUDA(cudaMalloc(&d_gspheres_, h.gsphere_bytes));
        RRT_CUDA(cudaMemcpy(d_gspheres_, in, h.gsphere_bytes, cudaMemcpyHostToDevice));
    }
    view_ = h.view;
    view_.nodes = d_nodes_;
    view_.prims = d_prims_;
    view_.inst_w2p = static_cast<const double*>(d_inst_);
    view_.gspheres = d_gspheres_;
    stats_ = h.stats;
    stack_levels_ = h.stack_levels;
    sort_rays_ = h.sort_rays != 0;
    node_bytes_ = h.node_bytes;
    prim_bytes_ = h.prim_bytes;
    inst_bytes_ = h.inst_bytes;
    gsphere_bytes_ = h.gsphere_bytes;
    stats_.build_usec =
        (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t_start).count();
    configure_kernels(view_.quantised != 0);
    return RRT_OK;
}

int DeviceAggregate::ensure_workspace(Workspace& w, uint64_t n, std::string* err) const {
    if (!w.d_small) {
        RRT_CUDA(cudaMalloc(&w.d_bins, (size_t)kSortBins * sizeof(uint32_t)));
        RRT_CUDA(cudaMalloc(&w.d_block_sums, (size_t)(kSortBins / kScanBlock) * sizeof(uint32_t)));
        RRT_CUDA(cudaMalloc(&w.d_small, 128));
        RRT_CUDA(cudaEventCreateWithFlags(&w.last_use, cudaEventDisableTiming));
        int dev = 0, sms = 0;
        RRT_CUDA(cudaGetDevice(&dev));
        RRT_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        w.n_sms = sms;
    }
    if (n > w.capacity) {
        if (w.d_key) cudaFree(w.d_key);
        if (w.d_rank) cudaFree(w.d_rank);
        if (w.d_perm) cudaFree(w.d_perm);
        w.d_key = w.d_rank = w.d_perm = nullptr;
        w.capacity = 0;
        RRT_CUDA(cudaMalloc(&w.d_key, n * sizeof(uint32_t)));
        RRT_CUDA(cudaMalloc(&w.d_rank, n * sizeof(uint32_t)));
        RRT_CUDA(cudaMalloc(&w.d_perm, n * sizeof(uint32_t)));
        w.capacity = n;
    }
    return RRT_OK;
}

template <bool ANY>
int DeviceAggregate::trace(uint64_t n, const rrt_ray* d_rays, rrt_hit* d_hits, uint8_t* d_occ, void* stream,
                           std::string* err, int* launches, const uint32_t* n_dev) const {
    if (n == 0) return RRT_OK;
    if (n >= (1ull << 32)) {
        if (err) *err = "batch too large for one call (2^32 rays)";
        return RRT_ERR_INVALID;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    std::lock_guard<std::mutex> lock(ws_mutex_);
    Workspace& w = (ws_.count(stream) || ws_.size() < kMaxWorkspaces) ? ws_[stream] : ws_.begin()->second;
    int rc = ensure_workspace(w, n, err);
    if (rc != RRT_OK) return rc;
    // a workspace that another stream used last (only past kMaxWorkspaces streams): order this call after that one
    if (w.used && w.last_stream != stream) RRT_CUDA(cudaStreamWaitEvent(s, w.last_use, 0));
    uint32_t* small = static_cast<uint32_t*>(w.d_small);  // [0..1] cursor, [2] max_bin, [3] use_perm
    RRT_CUDA(cudaMemsetAsync(small, 0, 128, s));
    const bool sorting = sort_rays_ && n >= 4096;
    int count = 0;
    if (sorting) {
        // about one ray per cell: 7 bits per axis for >= 1 Mi rays, fewer for short queues
        int bits = kSortBits;
        while (bits > 4 && (1ull << (3 * bits)) > 2 * n) --bits;
        const uint32_t nbins = (1u << (3 * bits)) * (view_.sort_mode == 0 ? 1u : 8u);
        RRT_CUDA(cudaMemsetAsync(w.d_bins, 0, (size_t)nbins * sizeof(uint32_t), s));
        const unsigned sb = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)w.n_sms * 16u);
        sort_count_kernel<<<sb, 256, 0, s>>>(view_, n, d_rays, w.d_bins, w.d_key, w.d_rank, n_dev, bits);
        scan_block_kernel<<<nbins / kScanBlock, kScanBlock, 0, s>>>(w.d_bins, nbins, w.d_block_sums, small + 2);
        scan_sums_kernel<<<1, kScanBlock, 0, s>>>(w.d_block_sums, nbins / kScanBlock, small + 2, n, small + 3, n_dev);
        sort_scatter_kernel<<<sb, 256, 0, s>>>(n, w.d_bins, w.d_block_sums, w.d_key, w.d_rank, small + 3, w.d_perm,
                                               n_dev);
        count += 4;
    }
    const TraceKernel kernel = trace_kernel_for(ANY, view_.wide != 0, view_.quantised != 0, view_.gspheres != nullptr);
    const size_t smem = trace_smem_bytes(stack_levels_);
    int per_sm = 0;
    RRT_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kBlock, smem));
    if (per_sm < 1) per_sm = 1;
    uint64_t blocks = (uint64_t)w.n_sms * (uint64_t)per_sm;
    const uint64_t needed = (n + kBlock - 1) / kBlock;
    if (blocks > needed) blocks = needed;
    kernel<<<(unsigned)blocks, kBlock, smem, s>>>(view_, n, d_rays, d_hits, d_occ, sorting ? w.d_perm : nullptr,
                                               sorting ? small + 3 : nullptr,
                                               reinterpret_cast<unsigned long long*>(small), n_dev, stack_levels_);
    count += 1;
    RRT_CUDA(cudaGetLastError());
#if RRT_STATS
    {
        unsigned long long h[16];
        RRT_CUDA(cudaStreamSynchronize(s));
        RRT_CUDA(cudaMemcpy(h, small, 128, cudaMemcpyDeviceToHost));
        if (n >= (1u << 20))
            fprintf(stderr, "RRT_STATS any=%d n=%llu interior trips %llu: walking %.2f no-ray %.2f drained %.2f at-2nd-leaf %.2f | leaf trips %llu: active %.2f\n",
                    (int)ANY, (unsigned long long)n, h[2], (double)h[3] / h[2], (double)h[4] / h[2], (double)h[5] / h[2],
                    (double)h[6] / h[2], h[7], (double)h[8] / (h[7] ? h[7] : 1));
    }
#endif
    RRT_CUDA(cudaEventRecord(w.last_use, s));
    w.used = true;
    w.last_stream = stream;
    if (launches) *launches = count;
    return RRT_OK;
}

int DeviceAggregate::closest_hit(uint64_t n, const rrt_ray* d_rays, rrt_hit* d_hits, void* stream, std::string* err,
                                 int* launches) const {
    return trace<false>(n, d_rays, d_hits, nullptr, stream, err, launches, nullptr);
}
int DeviceAggregate::closest_hit_indirect(uint64_t capacity, const uint32_t* d_count, const rrt_ray* d_rays,
                                          rrt_hit* d_hits, void* stream, std::string* err, int* launches) const {
    return trace<false>(capacity, d_rays, d_hits, nullptr, stream, err, launches, d_count);
}
int DeviceAggregate::any_hit_indirect(uint64_t capacity, const uint32_t* d_count, const rrt_ray* d_rays,
                                      uint8_t* d_occluded, void* stream, std::string* err, int* launches) const {
    return trace<true>(capacity, d_rays, nullptr, d_occluded, stream, err, launches, d_count);
}

int DeviceAggregate::any_hit(uint64_t n, const rrt_ray* d_rays, uint8_t* d_occluded, void* stream, std::string* err,
                             int* launches) const {
    return trace<true>(n, d_rays, nullptr, d_occluded, stream, err, launches, nullptr);
}

}  // namespace rrt
