// The CPU oracle's SurfaceInteraction for rrt_intersect_surface (tests/surface_oracle.py, tests/test_gpu_surface.py).
//
// Built into its own shared library with the oracle's shape and BVH sources (oracle/rt_geom.cpp, rt_shapes.cpp,
// rt_bvh.cpp) and the oracle's compiler flags.  Scenes are assembled exactly as oracle/oracle_capi.cpp assembles them;
// sor_intersect_si runs BVH::intersect with a SurfaceInteraction to fill and returns every field of it: the statement
// each rrt_surface record is checked against.
#include <algorithm>
#include <atomic>
#include <cstring>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "rt_bvh.hpp"

using namespace orc;

namespace {
thread_local std::string g_err;
Xform xf_from(const double* m16, const double* inv16) {
    Xform t;
    std::memcpy(t.m.m, m16, 16 * sizeof(double));
    std::memcpy(t.inv.m, inv16, 16 * sizeof(double));
    return t;
}
struct Scene {
    Geometry geom;
    BVH bvh;
    bool built = false;
};
template <class F>
void parallel_for(uint64_t n, int nthreads, F f) {
    if (nthreads <= 1 || n < 1024) {
        f(0, n);
        return;
    }
    std::vector<std::thread> th;
    const uint64_t per = (n + nthreads - 1) / nthreads;
    for (int i = 0; i < nthreads; ++i) {
        const uint64_t b = per * i, e = std::min(n, b + per);
        if (b >= e) break;
        th.emplace_back([=] { f(b, e); });
    }
    for (auto& t : th) t.join();
}
}  // namespace

extern "C" {

const char* sor_last_error() { return g_err.c_str(); }

// quirk_mask as orc_scene_new: bit i set = fix Q(1,2,3,4,5b,6,8,9,5c)[i]; 0 = literal reference, 0x1FF = Tier F.
void* sor_scene_new(uint32_t mask) {
    Scene* s = new Scene();
    Quirks& q = s->geom.q;
    q.fix_q1 = mask & 1u;
    q.fix_q2 = mask & 2u;
    q.fix_q3 = mask & 4u;
    q.fix_q4 = mask & 8u;
    q.fix_q5b = mask & 16u;
    q.fix_q6 = mask & 32u;
    q.fix_q8 = mask & 64u;
    q.fix_q9 = mask & 128u;
    q.fix_q5c = mask & 256u;
    return s;
}
void sor_scene_free(void* sp) { delete (Scene*)sp; }

// create_triangle_mesh (triangle.rs:131-165), as orc_add_mesh: 0-based indices, n = 0 / null for absent attributes.
int32_t sor_add_mesh(void* sp, uint32_t nv, const double* p, uint32_t ntri, const uint32_t* vi, uint32_t nn, const double* n,
                     const uint32_t* ni, uint32_t nuv, const double* uv, const uint32_t* uvi) {
    Scene* s = (Scene*)sp;
    TriMesh m;
    m.p.resize(nv);
    for (uint32_t i = 0; i < nv; ++i) m.p[i] = V3(p[3 * i], p[3 * i + 1], p[3 * i + 2]);
    m.vi.assign(vi, vi + 3 * (size_t)ntri);
    if (nn && n) {
        m.n.resize(nn);
        for (uint32_t i = 0; i < nn; ++i) m.n[i] = V3(n[3 * i], n[3 * i + 1], n[3 * i + 2]);
        if (ni) m.ni.assign(ni, ni + 3 * (size_t)ntri);
    }
    if (nuv && uv) {
        m.uv.resize(nuv);
        for (uint32_t i = 0; i < nuv; ++i) m.uv[i] = P2(uv[2 * i], uv[2 * i + 1]);
        if (uvi) m.uvi.assign(uvi, uvi + 3 * (size_t)ntri);
    }
    s->geom.meshes.push_back(std::move(m));
    return (int32_t)s->geom.meshes.size() - 1;
}
// Sphere::new (sphere.rs:28-47)
int32_t sor_add_sphere(void* sp, const double* m16, const double* inv16, double radius, double z_min, double z_max,
                       double phi_max_deg) {
    Scene* s = (Scene*)sp;
    const Xform o2w = xf_from(m16, inv16);
    s->geom.spheres.push_back(sphere_new(o2w, xf_inverse(o2w), radius, z_min, z_max, phi_max_deg));
    return (int32_t)s->geom.spheres.size() - 1;
}
int32_t sor_add_geo_triangles(void* sp, int32_t mesh) {
    Scene* s = (Scene*)sp;
    const int32_t first = (int32_t)s->geom.geos.size();
    const size_t nt = s->geom.meshes[mesh].n_triangles();
    for (size_t i = 0; i < nt; ++i) s->geom.geos.push_back(GeoPrim{SHAPE_TRIANGLE, mesh, (int32_t)i, 0});
    return first;
}
int32_t sor_add_geo_sphere(void* sp, int32_t sphere) {
    Scene* s = (Scene*)sp;
    s->geom.geos.push_back(GeoPrim{SHAPE_SPHERE, sphere, 0, 0});
    return (int32_t)s->geom.geos.size() - 1;
}
int32_t sor_add_xform(void* sp, const double* m16, const double* inv16) {
    Scene* s = (Scene*)sp;
    s->geom.xforms.push_back(xf_from(m16, inv16));
    return (int32_t)s->geom.xforms.size() - 1;
}
// `count` top-level primitives geo = first_geo.., wrapped in a TransformedPrimitive when xf >= 0
void sor_add_prims(void* sp, int32_t first_geo, int32_t count, int32_t xf) {
    Scene* s = (Scene*)sp;
    for (int32_t i = 0; i < count; ++i) s->geom.prims.push_back(Prim{first_geo + i, xf});
}
int32_t sor_build(void* sp, uint32_t max_prims_in_node) {
    Scene* s = (Scene*)sp;
    try {
        s->bvh.build(&s->geom, max_prims_in_node);
        s->built = true;
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}

// Scene::intersect over a batch with the SurfaceInteraction it leaves (interaction.rs:85-113).  rays: n x 7 doubles
// (o, d, t_max).  prim[n] (-1 miss), t[n], uv[2n] (the hit's u, v); si[38n] in rrt_surface's order after its hit: p, wo, n,
// uv, dpdu, dpdv, dndu, dndv, shading n, dpdu, dpdv, dndu, dndv; +0.0 throughout for a miss.
int32_t sor_intersect_si(void* sp, uint64_t n, const double* rays, int32_t* prim, double* t, double* uv, double* si_out,
                         int32_t nthreads) {
    Scene* s = (Scene*)sp;
    if (!s->built) {
        g_err = "sor_intersect_si: scene not built";
        return -1;
    }
    std::atomic<int> failed{0};
    std::string err;
    parallel_for(n, nthreads, [&](uint64_t b, uint64_t e) {
        try {
            for (uint64_t i = b; i < e; ++i) {
                const double* rr = rays + 7 * i;
                Ray r;
                r.o = V3(rr[0], rr[1], rr[2]);
                r.d = V3(rr[3], rr[4], rr[5]);
                r.t_max = rr[6];
                HitRecord h;
                SI si;
                const bool hit = s->bvh.intersect(r, &h, &si, nullptr);
                prim[i] = hit ? h.prim : -1;
                t[i] = hit ? h.t : 0.0;
                uv[2 * i] = hit ? h.u : 0.0;
                uv[2 * i + 1] = hit ? h.v : 0.0;
                double* g = si_out + 38 * i;
                if (!hit) {
                    for (int k = 0; k < 38; ++k) g[k] = 0.0;
                    continue;
                }
                const V3 vecs[12] = {si.p, si.wo, si.n, si.dpdu, si.dpdv, si.dndu, si.dndv,
                                     si.sh.n, si.sh.dpdu, si.sh.dpdv, si.sh.dndu, si.sh.dndv};
                int k = 0;
                for (int j = 0; j < 12; ++j) {
                    g[k++] = vecs[j].x;
                    g[k++] = vecs[j].y;
                    g[k++] = vecs[j].z;
                    if (j == 2) {  // uv follows n
                        g[k++] = si.uv[0];
                        g[k++] = si.uv[1];
                    }
                }
            }
        } catch (const std::exception& ex) {
            if (!failed.exchange(1)) err = ex.what();
        }
    });
    if (failed) {
        g_err = err;
        return -1;
    }
    return 0;
}

}  // extern "C"
