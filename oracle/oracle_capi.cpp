// ORACLE — TEST INFRASTRUCTURE ONLY (see rt_geom.hpp).
//
// C entry points so that tests/ (ctypes) and bench.py's cpu_baseline leg can drive the
// CPU restatement.  Nothing in the product links or loads this file.
#include <algorithm>
#include <atomic>
#include <memory>
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "rt_bvh.hpp"
#include "rt_sampling.hpp"

using namespace orc;

namespace {
thread_local std::string g_err;
Xform xf_from(const double* m16, const double* inv16) {
    Xform t;
    std::memcpy(t.m.m, m16, 16 * sizeof(double));
    std::memcpy(t.inv.m, inv16, 16 * sizeof(double));
    return t;
}
Quirks quirks_from_mask(uint32_t mask) {
    Quirks q;
    q.fix_q1 = mask & 1u;
    q.fix_q2 = mask & 2u;
    q.fix_q3 = mask & 4u;
    q.fix_q4 = mask & 8u;
    q.fix_q5b = mask & 16u;
    q.fix_q6 = mask & 32u;
    q.fix_q8 = mask & 64u;
    q.fix_q9 = mask & 128u;
    q.fix_q5c = mask & 256u;
    return q;
}
struct Scene {
    Geometry geom;
    BVH bvh;
    bool built = false;
};
template <class F>
void parallel_for(uint64_t n, int nthreads, F f) {
    if (nthreads <= 1 || n < 1024) {
        f(0, n, 0);
        return;
    }
    std::vector<std::thread> th;
    uint64_t per = (n + nthreads - 1) / nthreads;
    for (int i = 0; i < nthreads; ++i) {
        uint64_t b = per * i, e = std::min(n, b + per);
        if (b >= e) break;
        th.emplace_back([=] { f(b, e, i); });
    }
    for (auto& t : th) t.join();
}
}  // namespace

extern "C" {

const char* orc_last_error() { return g_err.c_str(); }

// quirk_mask: bit i set = fix Q(1,2,3,4,5b,6,8,9,5c)[i]; 0 = literal reference, 0x1FF = Tier F.
void* orc_scene_new(uint32_t quirk_mask) {
    Scene* s = new Scene();
    s->geom.q = quirks_from_mask(quirk_mask);
    return s;
}

// create_triangle_mesh (triangle.rs:131-165).  Index arrays are 0-based; pass n=0 / null
// for absent normals / uvs.  Returns the mesh index.
int32_t orc_add_mesh(void* sp, uint32_t nv, const double* p, uint32_t ntri, const uint32_t* vi, uint32_t nn,
                     const double* n, const uint32_t* ni, uint32_t nuv, const double* uv, const uint32_t* uvi) {
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

// Sphere::new (sphere.rs:28-47); o2w given as matrix + inverse (Transform carries both).
int32_t orc_add_sphere(void* sp, const double* m16, const double* inv16, double radius, double z_min, double z_max,
                       double phi_max_deg) {
    Scene* s = (Scene*)sp;
    Xform o2w = xf_from(m16, inv16);
    s->geom.spheres.push_back(sphere_new(o2w, xf_inverse(o2w), radius, z_min, z_max, phi_max_deg));
    return (int32_t)s->geom.spheres.size() - 1;
}

// One GeometricPrimitive per mesh triangle (renderprocess.rs:1255-1263). Returns first geo index.
int32_t orc_add_geo_triangles(void* sp, int32_t mesh, int32_t material) {
    Scene* s = (Scene*)sp;
    int32_t first = (int32_t)s->geom.geos.size();
    size_t nt = s->geom.meshes[mesh].n_triangles();
    for (size_t i = 0; i < nt; ++i) s->geom.geos.push_back(GeoPrim{SHAPE_TRIANGLE, mesh, (int32_t)i, material});
    return first;
}
int32_t orc_add_geo_sphere(void* sp, int32_t sphere, int32_t material) {
    Scene* s = (Scene*)sp;
    s->geom.geos.push_back(GeoPrim{SHAPE_SPHERE, sphere, 0, material});
    return (int32_t)s->geom.geos.size() - 1;
}
int32_t orc_add_xform(void* sp, const double* m16, const double* inv16) {
    Scene* s = (Scene*)sp;
    s->geom.xforms.push_back(xf_from(m16, inv16));
    return (int32_t)s->geom.xforms.size() - 1;
}
// Append `count` top-level primitives geo = first_geo..first_geo+count, wrapped in a
// TransformedPrimitive when xf >= 0 (renderprocess.rs:1265-1281).
void orc_add_prims(void* sp, int32_t first_geo, int32_t count, int32_t xf) {
    Scene* s = (Scene*)sp;
    for (int32_t i = 0; i < count; ++i) s->geom.prims.push_back(Prim{first_geo + i, xf});
}
uint32_t orc_num_prims(void* sp) { return (uint32_t)((Scene*)sp)->geom.prims.size(); }

// BVHAccel::new(prims, max_prims_in_node, HLBVH).  0 = ok.
int32_t orc_build(void* sp, uint32_t max_prims_in_node) {
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
uint32_t orc_num_nodes(void* sp) { return (uint32_t)((Scene*)sp)->bvh.nodes.size(); }
uint32_t orc_num_ordered(void* sp) { return (uint32_t)((Scene*)sp)->bvh.ordered.size(); }
// bounds6[n*6] (lo,hi), meta[n*3] (offset, n_primitives, axis), ordered[num_ordered]
void orc_get_nodes(void* sp, double* bounds6, uint32_t* meta3, uint32_t* ordered) {
    Scene* s = (Scene*)sp;
    for (size_t i = 0; i < s->bvh.nodes.size(); ++i) {
        const LinearNode& n = s->bvh.nodes[i];
        if (bounds6) {
            double* b = bounds6 + 6 * i;
            b[0] = n.bounds.lo.x; b[1] = n.bounds.lo.y; b[2] = n.bounds.lo.z;
            b[3] = n.bounds.hi.x; b[4] = n.bounds.hi.y; b[5] = n.bounds.hi.z;
        }
        if (meta3) {
            meta3[3 * i] = n.offset;
            meta3[3 * i + 1] = n.n_primitives;
            meta3[3 * i + 2] = n.axis;
        }
    }
    if (ordered) std::memcpy(ordered, s->bvh.ordered.data(), s->bvh.ordered.size() * sizeof(uint32_t));
}
void orc_world_bound(void* sp, double* out6) {
    B3 b = ((Scene*)sp)->bvh.world_bound();
    out6[0] = b.lo.x; out6[1] = b.lo.y; out6[2] = b.lo.z;
    out6[3] = b.hi.x; out6[4] = b.hi.y; out6[5] = b.hi.z;
}

// Scene::intersect over a batch (scene.rs:69-72 -> bvh.rs:183-236).
// rays: n x 7 doubles (o, d, t_max) — d is used as given, like the reference's aggregate.
// Outputs (any may be null): prim[n] (orig prim id, -1 miss), t[n], uv[n*2],
// geom_out[n*9] = hit point p, geometric normal n, shading normal ns (world space).
// stats5: rays, nodes_visited, prims_tested, max_stack, stack_overflow.
int32_t orc_intersect(void* sp, uint64_t n, const double* rays, int32_t* prim, double* t, double* uv,
                      double* geom_out, uint64_t* stats5, int32_t nthreads) {
    Scene* s = (Scene*)sp;
    if (!s->built) {
        g_err = "orc_intersect: scene not built";
        return -1;
    }
    std::vector<TraversalStats> st(std::max(1, nthreads));
    std::atomic<int> failed{0};
    std::string err;
    parallel_for(n, nthreads, [&](uint64_t b, uint64_t e, int tid) {
        try {
            for (uint64_t i = b; i < e; ++i) {
                const double* rr = rays + 7 * i;
                Ray r;
                r.o = V3(rr[0], rr[1], rr[2]);
                r.d = V3(rr[3], rr[4], rr[5]);
                r.t_max = rr[6];
                HitRecord h;
                SI si;
                bool hit = s->bvh.intersect(r, &h, geom_out ? &si : nullptr, &st[tid]);
                if (prim) prim[i] = hit ? h.prim : -1;
                if (t) t[i] = hit ? h.t : 0.0;
                if (uv) {
                    uv[2 * i] = hit ? h.u : 0.0;
                    uv[2 * i + 1] = hit ? h.v : 0.0;
                }
                if (geom_out) {
                    double* g = geom_out + 9 * i;
                    if (hit) {
                        g[0] = si.p.x; g[1] = si.p.y; g[2] = si.p.z;
                        g[3] = si.n.x; g[4] = si.n.y; g[5] = si.n.z;
                        g[6] = si.sh.n.x; g[7] = si.sh.n.y; g[8] = si.sh.n.z;
                    } else {
                        for (int k = 0; k < 9; ++k) g[k] = 0.0;
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
    if (stats5) {
        TraversalStats tot;
        for (auto& x : st) {
            tot.rays += x.rays;
            tot.nodes_visited += x.nodes_visited;
            tot.prims_tested += x.prims_tested;
            tot.max_stack = std::max(tot.max_stack, x.max_stack);
            tot.stack_overflow += x.stack_overflow;
        }
        stats5[0] = tot.rays; stats5[1] = tot.nodes_visited; stats5[2] = tot.prims_tested;
        stats5[3] = tot.max_stack; stats5[4] = tot.stack_overflow;
    }
    return 0;
}

// Scene::intersect_p over a batch (scene.rs:75-80 -> bvh.rs:123-174).
int32_t orc_intersect_p(void* sp, uint64_t n, const double* rays, uint8_t* occluded, uint64_t* stats5,
                        int32_t nthreads) {
    Scene* s = (Scene*)sp;
    if (!s->built) {
        g_err = "orc_intersect_p: scene not built";
        return -1;
    }
    std::vector<TraversalStats> st(std::max(1, nthreads));
    std::atomic<int> failed{0};
    std::string err;
    parallel_for(n, nthreads, [&](uint64_t b, uint64_t e, int tid) {
        try {
            for (uint64_t i = b; i < e; ++i) {
                const double* rr = rays + 7 * i;
                Ray r;
                r.o = V3(rr[0], rr[1], rr[2]);
                r.d = V3(rr[3], rr[4], rr[5]);
                r.t_max = rr[6];
                occluded[i] = s->bvh.intersect_p(r, &st[tid]) ? 1 : 0;
            }
        } catch (const std::exception& ex) {
            if (!failed.exchange(1)) err = ex.what();
        }
    });
    if (failed) {
        g_err = err;
        return -1;
    }
    if (stats5) {
        TraversalStats tot;
        for (auto& x : st) {
            tot.rays += x.rays;
            tot.nodes_visited += x.nodes_visited;
            tot.prims_tested += x.prims_tested;
            tot.max_stack = std::max(tot.max_stack, x.max_stack);
            tot.stack_overflow += x.stack_overflow;
        }
        stats5[0] = tot.rays; stats5[1] = tot.nodes_visited; stats5[2] = tot.prims_tested;
        stats5[3] = tot.max_stack; stats5[4] = tot.stack_overflow;
    }
    return 0;
}

// Brute force over every top-level primitive (no BVH): the topology-independent checker.
// Same accept rules as the Tier-F traversal (closest t, ties -> lowest prim id).
int32_t orc_brute_force(void* sp, uint64_t n, const double* rays, int32_t* prim, double* t, int32_t nthreads) {
    Scene* s = (Scene*)sp;
    const Geometry& g = s->geom;
    parallel_for(n, nthreads, [&](uint64_t b, uint64_t e, int) {
        for (uint64_t i = b; i < e; ++i) {
            const double* rr = rays + 7 * i;
            Ray r;
            r.o = V3(rr[0], rr[1], rr[2]);
            r.d = V3(rr[3], rr[4], rr[5]);
            r.t_max = rr[6];
            int32_t best = -1;
            for (size_t pi = 0; pi < g.prims.size(); ++pi) {
                Ray q = r;
                double u, v;
                if (g.prim_intersect(g.prims[pi], q, &u, &v, nullptr, false)) {
                    if (best < 0 || q.t_max < r.t_max) {
                        best = (int32_t)pi;
                        r.t_max = q.t_max;
                    }
                }
            }
            prim[i] = best;
            t[i] = best >= 0 ? r.t_max : 0.0;
        }
    });
    return 0;
}

// ---- known-answer-test hooks (geometry.rs tests, bvh.rs helpers) -------------------------
void orc_kat_vec3(const double* a3, const double* b3, double s, double* out) {
    V3 a(a3[0], a3[1], a3[2]), b(b3[0], b3[1], b3[2]);
    out[0] = length_sq(a);
    V3 m = a * s;
    out[1] = m.x; out[2] = m.y; out[3] = m.z;
    out[4] = dot(a, b);
    V3 c = cross(a, b);
    out[5] = c.x; out[6] = c.y; out[7] = c.z;
}
void orc_kat_bounds(const double* p1, const double* p2, const double* p3, double* out10) {
    B3 b = b3_new(V3(p1[0], p1[1], p1[2]), V3(p2[0], p2[1], p2[2]));
    b = b3_union(b, V3(p3[0], p3[1], p3[2]));
    out10[0] = b.lo.x; out10[1] = b.lo.y; out10[2] = b.lo.z;
    out10[3] = b.hi.x; out10[4] = b.hi.y; out10[5] = b.hi.z;
    V3 c;
    double r;
    b3_bounding_sphere(b, &c, &r);
    out10[6] = c.x; out10[7] = c.y; out10[8] = c.z; out10[9] = r;
}
// test_bnd2 (geometry.rs:1974-1980): the points of `for p in b.into_iter()`, and Bounds2i::inside of each
uint64_t orc_kat_bounds2i_iter(int64_t x0, int64_t y0, int64_t x1, int64_t y1, int64_t* out_xy_inside, uint64_t cap) {
    Bounds2iIter it(x0, y0, x1, y1);
    uint64_t n = 0;
    int64_t px, py;
    while (it.next(&px, &py)) {
        if (n < cap) {
            out_xy_inside[3 * n] = px;
            out_xy_inside[3 * n + 1] = py;
            out_xy_inside[3 * n + 2] = bounds2i_inside(px, py, x0, y0, x1, y1) ? 1 : 0;
        }
        ++n;
    }
    return n;
}
// PixelSampler<Stratified> for one pixel: the 1D tables [ndims][n], the 2D tables [ndims][n][2] as start_pixel leaves
// them, and for every sample the first four overflow draws (a get_1d past the tables).
void orc_kat_stratified(uint64_t seed, int64_t xres, int64_t px, int64_t py, uint32_t xs, uint32_t ys, uint32_t ndims,
                        int32_t jitter, double* out1d, double* out2d, double* overflow4) {
    StratifiedParams sp;
    sp.xs = xs; sp.ys = ys; sp.ndims = ndims; sp.jitter = jitter != 0; sp.seed = seed; sp.xres = xres;
    StratifiedSampler sm;
    sm.sp = &sp;
    sm.samples_per_pixel = (uint64_t)xs * ys;
    sm.start_pixel(px, py);
    const uint32_t n = xs * ys;
    for (uint32_t d = 0; d < ndims; ++d)
        for (uint32_t i = 0; i < n; ++i) {
            out1d[d * n + i] = sm.s1[d][i];
            out2d[2 * (d * n + i)] = sm.s2[d][i].x;
            out2d[2 * (d * n + i) + 1] = sm.s2[d][i].y;
        }
    uint32_t k = 1;
    while (sm.start_next_sample()) {
        for (uint32_t d = 0; d < ndims; ++d) sm.get_1d();
        for (int j = 0; j < 4; ++j) overflow4[4 * k + j] = sm.get_1d();
        ++k;
    }
}
uint32_t orc_kat_left_shift3(uint32_t x) { return left_shift3(x); }
uint32_t orc_kat_morton(double x, double y, double z) { return encode_morton3(V3(x, y, z)); }
void orc_kat_radix_sort(uint32_t n, uint32_t* idx, uint32_t* codes) {
    std::vector<MortonPrim> v(n);
    for (uint32_t i = 0; i < n; ++i) v[i] = MortonPrim{idx[i], codes[i]};
    radix_sort(v);
    for (uint32_t i = 0; i < n; ++i) {
        idx[i] = v[i].primitive_index;
        codes[i] = v[i].morton_code;
    }
}
// make_to_world (renderprocess.rs:242-252): translate * rotate(angle, normalize(axis)) * scale
void orc_make_to_world(const double* pos3, const double* axis3, double angle_deg, const double* scale3, double* m16,
                       double* inv16) {
    V3 axis = normalize_vec(V3(axis3[0], axis3[1], axis3[2]));
    Xform t = xf_mul(xf_mul(xf_translate(V3(pos3[0], pos3[1], pos3[2])), xf_rotate(angle_deg, axis)),
                     xf_scale(scale3[0], scale3[1], scale3[2]));
    std::memcpy(m16, t.m.m, sizeof(t.m.m));
    std::memcpy(inv16, t.inv.m, sizeof(t.inv.m));
}
void orc_m44_inverse(const double* m16, double* out16) {
    M44 m;
    std::memcpy(m.m, m16, sizeof(m.m));
    M44 r = m44_inverse(m);
    std::memcpy(out16, r.m, sizeof(r.m));
}
// Ray::new_od helper: returns the normalised direction exactly as the reference would.
void orc_normalize(const double* v3, double* out3) {
    V3 n = normalize_vec(V3(v3[0], v3[1], v3[2]));
    out3[0] = n.x; out3[1] = n.y; out3[2] = n.z;
}
// Single-primitive tests (primitives.rs test_primitive / sphere.rs test_sphere).
int32_t orc_prim_intersect_p(void* sp, uint32_t prim, const double* ray7) {
    Scene* s = (Scene*)sp;
    Ray r;
    r.o = V3(ray7[0], ray7[1], ray7[2]);
    r.d = V3(ray7[3], ray7[4], ray7[5]);
    r.t_max = ray7[6];
    return s->geom.prim_intersect_p(s->geom.prims[prim], r) ? 1 : 0;
}
int32_t orc_hardware_threads() { return (int32_t)std::thread::hardware_concurrency(); }

}  // extern "C"

// ================================ rendering ==================================================
#include "rt_render.hpp"

namespace {
struct EnvImage {
    uint64_t w = 0, h = 0;
    std::vector<uint8_t> rgb8;
};
struct RenderSetup {
    std::vector<std::unique_ptr<MipMap>> images;  // ImageTexture mip maps (stable addresses)
    std::vector<EnvImage> env_images;             // InfiniteAreaLight maps, kept raw until the world bound is known
    std::vector<Light> inf_specs;                 // the scene file's `infinite_lights` list
    std::vector<Xform> inf_xf;
    std::vector<Texture> textures;
    std::vector<Material> materials;
    std::vector<Light> light_specs;  // distant: w_light holds the raw (from - to) until render time
    std::vector<Xform> light_xf;
};
std::vector<std::pair<void*, RenderSetup>> g_setups;
RenderSetup& setup_of(void* s) {
    for (auto& p : g_setups)
        if (p.first == s) return p.second;
    g_setups.emplace_back(s, RenderSetup());
    return g_setups.back().second;
}
}  // namespace

extern "C" {

// Drops the scene's render setup too: a later scene may be allocated at the same address.
void orc_scene_free(void* s) {
    for (size_t i = 0; i < g_setups.size(); ++i)
        if (g_setups[i].first == s) {
            g_setups.erase(g_setups.begin() + i);
            break;
        }
    delete (Scene*)s;
}

// Debug ray log (rt_render.hpp raylog()): begin, render single-threaded, then take the records.
void orc_raylog_begin() {
    static std::vector<double> store;
    store.clear();
    raylog() = &store;
}
uint64_t orc_raylog_take(double* out, uint64_t cap_records) {
    std::vector<double>* v = raylog();
    raylog() = nullptr;
    if (!v) return 0;
    uint64_t n = v->size() / 10;
    if (out) std::memcpy(out, v->data(), sizeof(double) * 10 * std::min(n, cap_records));
    return n;
}

// Material table.  72 doubles per material (tests/oracle_scene.py material_row):
//  0 kind (MaterialKind) | 1-3 kd | 4-6 ks | 7-9 kr | 10-12 kt | 13-15 metal eta | 16-18 metal k |
//  19 sigma | 20 roughness | 21 u_roughness (<0 = None) | 22 v_roughness | 23 glass eta | 24 remap | 25 pad |
//  26-36 texture ids of those parameters | 37 bump map | 40-49 Disney metallic specular_tint anisotropic sheen sheen_tint
//  clearcoat clearcoat_gloss spec_trans flatness diff_trans | 50-52 scatter_distance | 53 thin | 54-64 their texture ids
void orc_set_materials(void* sp, uint32_t n, const double* m) {
    RenderSetup& rs = setup_of(sp);
    rs.materials.clear();
    for (uint32_t i = 0; i < n; ++i) {
        const double* a = m + 72 * (size_t)i;
        Material mat;
        mat.kind = (uint32_t)a[0];
        mat.kd = Rgb(a[1], a[2], a[3]);
        mat.ks = Rgb(a[4], a[5], a[6]);
        mat.kr = Rgb(a[7], a[8], a[9]);
        mat.kt = Rgb(a[10], a[11], a[12]);
        mat.eta_rgb = Rgb(a[13], a[14], a[15]);
        mat.k_rgb = Rgb(a[16], a[17], a[18]);
        mat.sigma = a[19];
        mat.roughness = a[20];
        mat.u_roughness = a[21];
        mat.v_roughness = a[22];
        mat.eta = a[23];
        mat.remap_roughness = a[24] != 0.0;
        for (int k = 0; k < 11; ++k) mat.tex[k] = (int32_t)a[26 + k];
        mat.bump_tex = (int32_t)a[37];
        double* ds[10] = {&mat.metallic, &mat.specular_tint, &mat.anisotropic, &mat.sheen, &mat.sheen_tint, &mat.clearcoat,
                          &mat.clearcoat_gloss, &mat.spec_trans, &mat.flatness, &mat.diff_trans};
        for (int k = 0; k < 10; ++k) *ds[k] = a[40 + k];
        mat.scatter_distance = Rgb(a[50], a[51], a[52]);
        mat.thin = a[53] != 0.0;
        for (int k = 0; k < 11; ++k) mat.dtex[k] = (int32_t)a[54 + k];
        rs.materials.push_back(mat);
    }
}
// Lights.  24 doubles per light: 0 kind | 1-3 I or L | 4-6 point: p_light, distant: from - to |
// 7-22 light_to_world m (row-major) | 23 pad.  (The inverse is not needed: vectors use m.)
// Texture table, 48 doubles per texture (tests/oracle_scene.py texture_rows): 0 kind | 1 is_rgb | 2 mapping | 3 aa |
// 4 t1 | 5 t2 | 6 amount | 8-19 v[4][3] | 20-27 map[8] | 28-43 IdentityMapping3D matrix (row-major).
// load_image (renderprocess.rs:535-566): 8-bit RGB rows as decoded (top row first); returns the image's index.
int32_t orc_add_image(void* sp, uint64_t w, uint64_t h, const uint8_t* rgb8, int32_t trilinear, double max_aniso, uint32_t wrap) {
    try {
        RenderSetup& rs = setup_of(sp);
        auto m = std::make_unique<MipMap>();
        m->create(w, h, texels_from_rgb8(rgb8, w, h), trilinear != 0, max_aniso, wrap);
        rs.images.push_back(std::move(m));
        return (int32_t)rs.images.size() - 1;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}
int32_t orc_add_env_image(void* sp, uint64_t w, uint64_t h, const uint8_t* rgb8) {
    RenderSetup& rs = setup_of(sp);
    EnvImage e;
    e.w = w;
    e.h = h;
    e.rgb8.assign(rgb8, rgb8 + 3 * w * h);
    rs.env_images.push_back(std::move(e));
    return (int32_t)rs.env_images.size() - 1;
}
// MIPMap probe: out = levels, then per level u_res, v_res; lookups: for each of n points (st, dstdx, dstdy: 6 doubles)
// lookup_d -> rgb and lookup_w(st, width = dstdx.x) -> rgb (6 doubles per point)
int32_t orc_mipmap_probe(void* sp, int32_t image, uint64_t n, const double* q6, double* out6, uint64_t* info) {
    try {
        RenderSetup& rs = setup_of(sp);
        const MipMap& m = *rs.images.at((size_t)image);
        info[0] = m.levels();
        for (uint64_t l = 0; l < m.levels() && l < 15; ++l) {
            info[1 + 2 * l] = m.pyramid[l].u_res;
            info[2 + 2 * l] = m.pyramid[l].v_res;
        }
        for (uint64_t i = 0; i < n; ++i) {
            const double* a = q6 + 6 * i;
            Rgb d = m.lookup_d(P2(a[0], a[1]), P2(a[2], a[3]), P2(a[4], a[5]));
            Rgb w = m.lookup_w(P2(a[0], a[1]), a[2]);
            for (int k = 0; k < 3; ++k) {
                out6[6 * i + k] = d.c[k];
                out6[6 * i + 3 + k] = w.c[k];
            }
        }
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}
// InfiniteAreaLight probe: per query (ref point[3], u[2], w[3]) -> sample_li: Li[3], wi[3], pdf; pdf_li(w); le(w)[3]; p1.x
int32_t orc_envlight_probe(uint64_t w, uint64_t h, const uint8_t* rgb8, const double* to_world16, const double* to_local16,
                           const double* wb6, uint64_t n, const double* in8, double* out12) {
    try {
        InfiniteLight il;
        Xform l2w, w2l;
        std::memcpy(l2w.m.m, to_world16, 16 * sizeof(double));
        std::memcpy(l2w.inv.m, to_local16, 16 * sizeof(double));
        w2l = xf_inverse(l2w);
        B3 wb;
        wb.lo = V3(wb6[0], wb6[1], wb6[2]);
        wb.hi = V3(wb6[3], wb6[4], wb6[5]);
        il.init(rgb8, w, h, l2w, w2l, wb);
        for (uint64_t i = 0; i < n; ++i) {
            const double* a = in8 + 8 * i;
            double* o = out12 + 12 * i;
            V3 wi, p1;
            double pdf = 0.0;
            Rgb li = il.sample_li(V3(a[0], a[1], a[2]), P2(a[3], a[4]), &wi, &pdf, &p1);
            V3 dir(a[5], a[6], a[7]);
            Rgb le = il.le(dir);
            o[0] = li.c[0]; o[1] = li.c[1]; o[2] = li.c[2]; o[3] = wi.x; o[4] = wi.y; o[5] = wi.z; o[6] = pdf;
            o[7] = il.pdf_li(dir); o[8] = le.c[0]; o[9] = le.c[1]; o[10] = le.c[2]; o[11] = p1.x;
        }
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}
void orc_set_textures(void* sp, uint32_t n, const double* t) {
    RenderSetup& rs = setup_of(sp);
    rs.textures.clear();
    if (n > (uint32_t)kMaxTextures) {
        g_err = "more textures than the restated evaluator holds";
        return;
    }
    for (uint32_t i = 0; i < n; ++i) {
        const double* a = t + 48 * (size_t)i;
        Texture x;
        x.kind = (uint32_t)a[0];
        x.mapping = (uint32_t)a[2];
        x.aa = (uint32_t)a[3];
        x.t1 = (int32_t)a[4];
        x.t2 = (int32_t)a[5];
        x.amount = (int32_t)a[6];
        for (int k = 0; k < 4; ++k) x.v[k] = Rgb(a[8 + 3 * k], a[9 + 3 * k], a[10 + 3 * k]);
        for (int k = 0; k < 8; ++k) x.map[k] = a[20 + k];
        std::memcpy(x.w2t.m.m, a + 28, 16 * sizeof(double));
        x.w2t.inv = x.w2t.m;  // unused
        if (x.kind == TEX_IMAGE) {
            if (x.t1 < 0 || (size_t)x.t1 >= rs.images.size()) {
                g_err = "image texture names an image that was not added";
                return;
            }
            x.image = rs.images[(size_t)x.t1].get();
        }
        rs.textures.push_back(x);
    }
}
// Texture probe: evaluates the table at (uv, p) and returns every texture's value (3 doubles each).  `diff` (may be
// null) = dpdx[3] dpdy[3] dudx dvdx dudy dvdy as compute_differentials would leave them.
void orc_texture_probe(uint32_t n, const double* table, const double* uv2, const double* p3, const double* diff, double* out) {
    void* tmp = orc_scene_new(0);
    orc_set_textures(tmp, n, table);
    RenderSetup& rs = setup_of(tmp);
    Rgb vals[kMaxTextures];
    TexPoint q;
    q.uv = P2(uv2[0], uv2[1]);
    q.p = V3(p3[0], p3[1], p3[2]);
    if (diff) {
        q.dpdx = V3(diff[0], diff[1], diff[2]);
        q.dpdy = V3(diff[3], diff[4], diff[5]);
        q.dudx = diff[6];
        q.dvdx = diff[7];
        q.dudy = diff[8];
        q.dvdy = diff[9];
    }
    tex_eval_all(rs.textures, q, vals);
    for (uint32_t i = 0; i < n && i < (uint32_t)kMaxTextures; ++i)
        for (int c = 0; c < 3; ++c) out[3 * i + c] = vals[i].c[c];
    orc_scene_free(tmp);
}
// compute_differentials probe: in = p n dpdu dpdv rx_o rx_d ry_o ry_d (3 doubles each); out = dpdx dpdy dudx dvdx dudy dvdy
void orc_differentials_probe(const double* in24, double* out10) {
    auto v = [&](int k) { return V3(in24[3 * k], in24[3 * k + 1], in24[3 * k + 2]); };
    SI si;
    si.p = v(0);
    si.n = v(1);
    si.dpdu = v(2);
    si.dpdv = v(3);
    RayDiff rd;
    rd.has_differentials = true;
    rd.rx_o = v(4);
    rd.rx_d = v(5);
    rd.ry_o = v(6);
    rd.ry_d = v(7);
    TexPoint q = compute_differentials(si, &rd);
    const double o[10] = {q.dpdx.x, q.dpdx.y, q.dpdx.z, q.dpdy.x, q.dpdy.y, q.dpdy.z, q.dudx, q.dvdx, q.dudy, q.dvdy};
    for (int k = 0; k < 10; ++k) out10[k] = o[k];
}
// Light table, 80 doubles per light (tests/oracle_scene.py light_row).
void orc_set_lights(void* sp, uint32_t n, const double* l) {
    RenderSetup& rs = setup_of(sp);
    rs.light_specs.clear();
    rs.light_xf.clear();
    for (uint32_t i = 0; i < n; ++i) {
        const double* a = l + 80 * (size_t)i;
        Light lt;
        lt.kind = (uint32_t)a[0];
        lt.intensity = Rgb(a[1], a[2], a[3]);
        lt.p_light = V3(a[4], a[5], a[6]);
        lt.w_light = V3(a[4], a[5], a[6]);
        Xform x;
        std::memcpy(x.m.m, a + 7, 16 * sizeof(double));
        x.inv = x.m;  // unused
        if (lt.kind == LIGHT_DIFFUSE_AREA) {
            lt.shape_kind = (uint32_t)a[23];
            Xform o2w, w2o;
            std::memcpy(o2w.m.m, a + 24, 16 * sizeof(double));
            std::memcpy(o2w.inv.m, a + 40, 16 * sizeof(double));
            w2o = xf_inverse(o2w);
            lt.sphere = sphere_new(o2w, w2o, a[56], a[57], a[58], a[59]);
            for (int k = 0; k < 3; ++k) {
                lt.tp[k] = V3(a[60 + 3 * k], a[61 + 3 * k], a[62 + 3 * k]);
                lt.tn[k] = V3(a[69 + 3 * k], a[70 + 3 * k], a[71 + 3 * k]);
            }
            lt.tri_has_n = a[78] != 0.0;
        }
        if (lt.kind == LIGHT_INFINITE) {
            lt.env_image = (int)a[23];
            std::memcpy(x.inv.m, a + 40, 16 * sizeof(double));  // world_to_light as make_to_world composed it
        }
        rs.light_specs.push_back(lt);
        rs.light_xf.push_back(x);
    }
}
// the scene file's `infinite_lights` list (same rows): PathIntegrator reads it for escaped rays (path.rs:84)
void orc_set_infinite_lights(void* sp, uint32_t n, const double* l) {
    RenderSetup& rs = setup_of(sp);
    std::vector<Light> keep = rs.light_specs;
    std::vector<Xform> keep_xf = rs.light_xf;
    orc_set_lights(sp, n, l);
    rs.inf_specs = rs.light_specs;
    rs.inf_xf = rs.light_xf;
    rs.light_specs = keep;
    rs.light_xf = keep_xf;
}

// DiffuseAreaLight::sample_li probe for one light row (80 doubles): out10 = wi[3], pdf, p_shape[3], L[3].
void orc_area_light_probe(const double* row80, const double* ref_p3, const double* u2, double* out10) {
    void* tmp = orc_scene_new(0);
    orc_set_lights(tmp, 1, row80);
    RenderSetup& rs = setup_of(tmp);
    RenderScene sc;
    V3 wi, p1;
    double pdf = 0.0;
    Rgb L = sc.area_sample_li(rs.light_specs[0], V3(ref_p3[0], ref_p3[1], ref_p3[2]), P2(u2[0], u2[1]), &wi, &pdf, &p1);
    const double o[10] = {wi.x, wi.y, wi.z, pdf, p1.x, p1.y, p1.z, L.c[0], L.c[1], L.c[2]};
    std::memcpy(out10, o, sizeof(o));
    orc_scene_free(tmp);
}

// params (doubles):
//  0 xres 1 yres 2 diagonal_mm 3 filter kind 4 rx 5 ry 6 alpha 7 scale 8 max_sample_luminance
//  9-11 camera world_pos 12-14 look 15-17 up 18 shutter_open 19 shutter_close 20 aperture_diameter
//  21 focus_distance 22 simple_weighting 23 nsamp 24 sample_at_center 25 seed 26 integrator kind
//  27 max_depth 28 rr_threshold 29 tile_mod 30 tile_rank 31 crop flag 32-35 crop x0 y0 x1 y1 36 want_dump
//  37 light strategy (DirectLighting: 0 one, 1 all)
// outputs: rgb[3*npix] (Film::write_image values before the PNG quantisation), raw[4*npix]
// (xyz + filter_weight_sum), stats[16], dump (6 doubles per camera sample, capacity dump_cap).
int32_t orc_render(void* sp, const double* prm, const double* lens_data, uint32_t n_lens_values, double* rgb,
                   double* raw, uint64_t* stats16, double* dump, uint64_t dump_cap, uint64_t* dump_count,
                   int32_t nthreads) {
    Scene* s = (Scene*)sp;
    if (!s->built) {
        g_err = "orc_render: scene not built";
        return -1;
    }
    try {
        RenderSetup& rs = setup_of(sp);
        RenderJob job;
        job.scene.geom = &s->geom;
        job.scene.bvh = &s->bvh;
        job.scene.materials = rs.materials;
        job.scene.textures = rs.textures;
        job.scene.fix_q9 = s->geom.q.fix_q9;
        for (const GeoPrim& g : s->geom.geos)
            if (g.material < 0 || (size_t)g.material >= rs.materials.size()) throw std::runtime_error("material index out of range");
        B3 wb = s->bvh.world_bound();
        std::vector<std::unique_ptr<InfiniteLight>> env_lights;
        auto make_infinite = [&](const Light& lt, const Xform& to_world) -> const InfiniteLight* {
            if (lt.env_image < 0 || (size_t)lt.env_image >= rs.env_images.size()) throw std::runtime_error("infinite light names no map");
            const EnvImage& e = rs.env_images[(size_t)lt.env_image];
            auto il = std::make_unique<InfiniteLight>();
            il->init(e.rgb8.data(), e.w, e.h, to_world, xf_inverse(to_world), wb);
            env_lights.push_back(std::move(il));
            return env_lights.back().get();
        };
        for (size_t i = 0; i < rs.light_specs.size(); ++i) {
            Light lt = rs.light_specs[i];
            if (lt.kind == LIGHT_POINT) {
                lt.p_light = V3(0.0, 0.0, 0.0);  // Q17: PointLight::new(.., Point3f::default(), ..), light_to_world unused
            } else if (lt.kind == LIGHT_DIFFUSE_AREA) {
                // the light's own shape, kept apart from the aggregate (Shape::pdf_ref intersects it)
                Geometry& lg = job.scene.light_shapes;
                lg.q = s->geom.q;
                GeoPrim g;
                g.material = -1;
                if (lt.shape_kind == 0) {
                    lg.spheres.push_back(lt.sphere);
                    g.kind = SHAPE_SPHERE;
                    g.a = (int32_t)lg.spheres.size() - 1;
                    g.b = 0;
                } else {
                    TriMesh m;
                    m.p = {lt.tp[0], lt.tp[1], lt.tp[2]};
                    m.vi = {0, 1, 2};
                    if (lt.tri_has_n) {
                        m.n = {lt.tn[0], lt.tn[1], lt.tn[2]};
                        m.ni = {0, 1, 2};
                    }
                    lg.meshes.push_back(m);
                    g.kind = SHAPE_TRIANGLE;
                    g.a = (int32_t)lg.meshes.size() - 1;
                    g.b = 0;
                }
                lg.geos.push_back(g);
                lt.probe_geo = (int)lg.geos.size() - 1;
            } else if (lt.kind == LIGHT_INFINITE) {
                lt.inf = make_infinite(lt, rs.light_xf[i]);
            } else {
                lt.w_light = normalize_vec(xf_vector(rs.light_xf[i], lt.w_light));  // distant.rs:30
                b3_bounding_sphere(wb, &lt.world_center, &lt.world_radius);
            }
            job.scene.lights.push_back(lt);
        }
        for (const Material& m : rs.materials)  // checked here: the worker threads have nobody to catch for them
            if (m.kind == MAT_DISNEY && !m.thin && (m.dtex[10] >= 0 || !m.scatter_distance.is_black()))
                throw std::runtime_error("oracle: DisneyMaterial with scatter_distance builds a BSSRDF (outside the restated path)");
        for (size_t i = 0; i < rs.inf_specs.size(); ++i) {  // Scene::infinite_lights: only Light::le is ever asked of them
            Light lt = rs.inf_specs[i];
            if (lt.kind == LIGHT_INFINITE) lt.inf = make_infinite(lt, rs.inf_xf[i]);
            job.scene.infinite_lights.push_back(lt);
        }
        Filter f;
        f.kind = (uint32_t)prm[3];
        f.rx = prm[4];
        f.ry = prm[5];
        f.alpha = prm[6];
        job.film.init((int64_t)prm[0], (int64_t)prm[1], prm[2], f, prm[7], prm[8]);
        Xform to_camera = xf_look_at(V3(prm[9], prm[10], prm[11]), V3(prm[12], prm[13], prm[14]), V3(prm[15], prm[16], prm[17]));
        std::vector<double> lens(lens_data, lens_data + n_lens_values);
        job.camera.init(xf_inverse(to_camera), prm[18], prm[19], prm[20], prm[21], &job.film, lens, prm[22] != 0.0,
                        std::max(1, nthreads));
        job.samples_per_pixel = (uint64_t)prm[23];
        job.halton.init(job.film.crop[2] - job.film.crop[0], job.film.crop[3] - job.film.crop[1], prm[24] != 0.0);
        job.perms = compute_radical_inverse_permutations((uint64_t)prm[25]);
        // prm[38] sampler kind (0 Halton, 1 Stratified: make_sampler, renderprocess.rs:1306-1325), 39 jitter,
        // 40 xsamp, 41 ysamp, 42 dimension
        job.sampler_kind = (int)prm[38];
        if (job.sampler_kind == 1) {
            job.stratified.xs = (uint32_t)prm[40];
            job.stratified.ys = (uint32_t)prm[41];
            job.stratified.ndims = (uint32_t)prm[42];
            job.stratified.jitter = prm[39] != 0.0;
            job.stratified.seed = (uint64_t)prm[25];
            job.stratified.xres = job.film.xres;
            job.samples_per_pixel = (uint64_t)job.stratified.xs * job.stratified.ys;
        }
        job.integrator.kind = (uint32_t)prm[26];
        job.integrator.max_depth = (uint32_t)prm[27];
        job.integrator.rr_threshold = prm[28];
        job.integrator.sample_all_lights = prm[37] != 0.0;
        job.want_dump = prm[36] != 0.0 && dump != nullptr;
        int64_t crop[4] = {(int64_t)prm[32], (int64_t)prm[33], (int64_t)prm[34], (int64_t)prm[35]};
        mip_panics().store(0);  // lookups made outside a render (the MIPMap probes of tests/test_images.py) are not this frame's
        job.render(std::max(1, nthreads), std::max<uint32_t>(1, (uint32_t)prm[29]), (uint32_t)prm[30],
                   prm[31] != 0.0 ? crop : nullptr);
        size_t npix = job.film.pixels.size();
        if (rgb) film_to_rgb(job.film, rgb);
        if (raw)
            for (size_t i = 0; i < npix; ++i) {
                raw[4 * i] = job.film.pixels[i].xyz[0];
                raw[4 * i + 1] = job.film.pixels[i].xyz[1];
                raw[4 * i + 2] = job.film.pixels[i].xyz[2];
                raw[4 * i + 3] = job.film.pixels[i].filter_weight_sum;
            }
        job.stats.asserts += mip_panics().exchange(0);
        if (stats16) {
            const RenderStats& st = job.stats;
            uint64_t v[16] = {st.camera_rays, st.extension_rays, st.shadow_rays, st.bounces, st.zero_weight, st.asserts,
                              st.closest.rays, st.closest.nodes_visited, st.closest.prims_tested, st.closest.max_stack,
                              st.any.rays, st.any.nodes_visited, st.any.prims_tested, st.any.max_stack,
                              st.closest.stack_overflow + st.any.stack_overflow, st.mis_probe_rays};
            std::memcpy(stats16, v, sizeof(v));
        }
        if (dump_count) *dump_count = job.dump.size();
        if (job.want_dump) {
            std::sort(job.dump.begin(), job.dump.end(), [](const HitDump& a, const HitDump& b) {
                if (a.py != b.py) return a.py < b.py;
                if (a.px != b.px) return a.px < b.px;
                return a.sample < b.sample;
            });
            uint64_t n = std::min<uint64_t>(dump_cap, job.dump.size());
            for (uint64_t i = 0; i < n; ++i) {
                const HitDump& d = job.dump[i];
                double* o = dump + 6 * i;
                o[0] = d.px; o[1] = d.py; o[2] = d.sample; o[3] = d.prim; o[4] = d.t; o[5] = d.weight;
            }
        }
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}

// Camera-only probe: the CameraSample, world ray and weight of every sample of one pixel
// (13 doubles per sample: p_film 2, p_lens 2, time, o 3, d 3, weight, halton index as double).
int32_t orc_camera_samples(const double* prm, const double* lens_data, uint32_t n_lens_values, int64_t px, int64_t py,
                           double* out, uint32_t max_samples, int32_t nthreads) {
    try {
        Film film;
        Filter f;
        f.kind = (uint32_t)prm[3];
        f.rx = prm[4];
        f.ry = prm[5];
        f.alpha = prm[6];
        film.init((int64_t)prm[0], (int64_t)prm[1], prm[2], f, prm[7], prm[8]);
        RealisticCamera cam;
        Xform to_camera = xf_look_at(V3(prm[9], prm[10], prm[11]), V3(prm[12], prm[13], prm[14]), V3(prm[15], prm[16], prm[17]));
        std::vector<double> lens(lens_data, lens_data + n_lens_values);
        cam.init(xf_inverse(to_camera), prm[18], prm[19], prm[20], prm[21], &film, lens, prm[22] != 0.0, std::max(1, nthreads));
        HaltonParams hp;
        hp.init(film.crop[2] - film.crop[0], film.crop[3] - film.crop[1], prm[24] != 0.0);
        std::vector<uint16_t> perms = compute_radical_inverse_permutations((uint64_t)prm[25]);
        HaltonSampler sm;
        sm.hp = &hp;
        sm.perms = perms.data();
        sm.samples_per_pixel = (uint64_t)prm[23];
        sm.start_pixel(px, py);
        uint32_t k = 0;
        while (sm.start_next_sample() && k < max_samples) {
            CameraSample cs;
            P2 a = sm.get_2d();
            cs.p_film = P2((double)px + a.x, (double)py + a.y);
            P2 b = sm.get_2d();
            cs.p_lens = P2(b.x + 0.5, b.y + 0.5);
            cs.time = sm.get_1d() + 0.5;
            RayDiff rd;
            double w = cam.generate_ray_differential(cs, &rd);
            double* o = out + 13 * (size_t)k;
            o[0] = cs.p_film.x; o[1] = cs.p_film.y; o[2] = cs.p_lens.x; o[3] = cs.p_lens.y; o[4] = cs.time;
            o[5] = rd.ray.o.x; o[6] = rd.ray.o.y; o[7] = rd.ray.o.z; o[8] = rd.ray.d.x; o[9] = rd.ray.d.y; o[10] = rd.ray.d.z;
            o[11] = w; o[12] = (double)sm.interval_sample_index;
            ++k;
        }
        return (int32_t)k;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}

// Halton KAT hooks (lowdiscrepancy.rs / halton.rs)
double orc_radical_inverse(int32_t base_index, uint64_t a) { return radical_inverse(base_index, a); }
double orc_scrambled_radical_inverse(int32_t base_index, uint64_t a, uint64_t seed) {
    std::vector<uint16_t> perms = compute_radical_inverse_permutations(seed);
    return scrambled_radical_inverse(base_index, a, perms.data() + prime_table().sums[base_index]);
}
uint64_t orc_halton_index(int64_t xres, int64_t yres, int64_t px, int64_t py, uint64_t sample_num, uint64_t* stride) {
    HaltonParams hp;
    hp.init(xres, yres, false);
    if (stride) *stride = hp.sample_stride;
    return hp.offset_for_pixel(px, py) + sample_num * hp.sample_stride;
}
void orc_halton_perms(uint64_t seed, uint16_t* out, uint32_t n) {
    std::vector<uint16_t> perms = compute_radical_inverse_permutations(seed);
    std::memcpy(out, perms.data(), std::min<size_t>(n, perms.size()) * sizeof(uint16_t));
}
// BSDF probe for unit tests: evaluates f, pdf and one sample of a material's Bsdf in a frame with
// shading normal +z, dpdu +x.  `m72`: one orc_set_materials row.  out: f(3), pdf, sample f(3), wi(3), pdf, sampled_type
void orc_bsdf_probe(const double* m72, const double* wo3, const double* wi3, const double* u2, int32_t allow_multiple,
                    double* out12) {
    Material mat;
    const double* a = m72;
    {
        double* ds[10] = {&mat.metallic, &mat.specular_tint, &mat.anisotropic, &mat.sheen, &mat.sheen_tint, &mat.clearcoat,
                          &mat.clearcoat_gloss, &mat.spec_trans, &mat.flatness, &mat.diff_trans};
        for (int k = 0; k < 10; ++k) *ds[k] = a[40 + k];
        mat.scatter_distance = Rgb(a[50], a[51], a[52]);
        mat.thin = a[53] != 0.0;
    }
    mat.kind = (uint32_t)a[0];
    mat.kd = Rgb(a[1], a[2], a[3]); mat.ks = Rgb(a[4], a[5], a[6]); mat.kr = Rgb(a[7], a[8], a[9]);
    mat.kt = Rgb(a[10], a[11], a[12]); mat.eta_rgb = Rgb(a[13], a[14], a[15]); mat.k_rgb = Rgb(a[16], a[17], a[18]);
    mat.sigma = a[19]; mat.roughness = a[20]; mat.u_roughness = a[21]; mat.v_roughness = a[22]; mat.eta = a[23];
    mat.remap_roughness = a[24] != 0.0;
    SI si = si_new(V3(0, 0, 0), P2(0, 0), V3(wo3[0], wo3[1], wo3[2]), V3(1, 0, 0), V3(0, 1, 0), V3(), V3(), 0.0);
    Bsdf b;
    material_bsdf(mat, si, allow_multiple != 0, &b);
    V3 wo(wo3[0], wo3[1], wo3[2]), wi(wi3[0], wi3[1], wi3[2]);
    Rgb f = b.f(wo, wi, BXDF_ALL);
    out12[0] = f.c[0]; out12[1] = f.c[1]; out12[2] = f.c[2];
    out12[3] = b.pdf(wo, wi, BXDF_ALL);
    V3 swi;
    double pdf = 0.0;
    uint8_t ty = 0;
    Rgb sf = b.sample_f(wo, &swi, P2(u2[0], u2[1]), &pdf, BXDF_ALL, &ty);
    out12[4] = sf.c[0]; out12[5] = sf.c[1]; out12[6] = sf.c[2];
    out12[7] = swi.x; out12[8] = swi.y; out12[9] = swi.z;
    out12[10] = pdf; out12[11] = (double)ty;
}

}  // extern "C"
