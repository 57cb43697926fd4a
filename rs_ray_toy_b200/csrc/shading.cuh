// Device-side shading for the wavefront path tracer: hit record -> surface frame
// (src/shape/triangle.rs:266-388, src/shape/sphere.rs:157-258, src/transform.rs:618-656),
// material -> lobes (src/material/{matte,plastic,metal,mirror,glass}.rs), and the Bsdf
// f / pdf / sample_f logic over those lobes (src/reflection.rs:216-404 with the BxDFs at
// :622-1026 and the Trowbridge–Reitz distribution of src/microfacet.rs:253-425).
//
// A material kind fixes its lobe list, so there is no per-hit allocation (the reference builds a
// Vec<Arc<dyn BxDF>> per hit): at most two lobes live in registers.  Scenes with a Translucent, Disney or Debug
// material (translucent.rs, disney.rs, debug_material.rs: up to eight lobes, Bsdf::MAX_BxDFS) run the NL = 8
// instantiation of everything below; every other scene runs NL = 2, whose code is what it was before those existed.  Quirks kept (Appendix A):
// Q15 (Bsdf::sample_f: other lobes' pdfs added only when the chosen lobe is not reflective, the
// recomputed multi-lobe f discarded), Q16 (Plastic's specular lobe gated on kd), Q5a (sphere hit
// point taken on the instance-space ray), FresnelSpecular's type = SPECULAR | ALL.
#pragma once
#ifndef RRT_SHADE_NOINLINE
#define RRT_SHADE_NOINLINE 1  // measured: 160 registers without spills, +3% (profiles/r1_sweep_shade_noinline.txt)
#endif
#if RRT_SHADE_NOINLINE
#define RRT_SHADE_FN static __device__ __noinline__
#else
#define RRT_SHADE_FN static __device__
#endif
#include "rmath.cuh"
#include "sphere_core.cuh"
#include "texture_core.h"

namespace rrt {

// ---- scene tables in HBM ---------------------------------------------------------------------------
struct PrimInfo {       // one per entry of the primitive list (prim_id order)
    uint32_t kind;      // low byte: 0 triangle, 1 sphere; kPrimHasUv / kPrimHasNormals: the mesh has uv / vertex normals
    uint32_t material;
    int32_t instance;   // -1 = bare GeometricPrimitive
    uint32_t shape;     // triangle: mesh id; sphere: sphere id
    uint32_t tri;       // triangle number inside the mesh
    // triangle: its three vertices as indices into the pooled mesh_p — the hit's vertex loads then depend on this record
    // alone instead of on the chain prims -> meshes -> mesh_vi -> mesh_p (two dependent gathers fewer per hit)
    uint32_t gv[3];
};
constexpr uint32_t kPrimKindMask = 0xffu, kPrimHasUv = 0x100u, kPrimHasNormals = 0x200u;
struct MeshInfo {
    uint64_t p_off, vi_off, n_off, ni_off, uv_off, uvi_off;  // element offsets into the pooled arrays
    uint32_t has_n, has_ni, has_uv, has_uvi;
};
struct SphereInfo {
    M34 o2w, w2o;
    double radius, theta_min, theta_max, phi_max;
    double z_min, z_max;
    uint32_t partial, pad;  // z_min / z_max / phi_max clip the sphere: the hit point depends on which root was taken
};
struct InstanceXf {
    M34 m, inv;
    uint32_t is_identity, pad;
};
struct MaterialRec {  // rrt_material, flattened
    uint32_t kind, remap_roughness;
    Rgb kd, ks, kr, kt, metal_eta, metal_k;
    double sigma, roughness, u_roughness, v_roughness, eta;
    // texture index per parameter (rrt_material_slot order; -1 = the constant above) and the bits of every
    // texture those reach; 0 = a constant-valued material, which is never copied
    int32_t tex[12];   // [11] = bump_map
    uint32_t needed;   // closure of the parameter textures (the bump map's own closure: bump_needed)
    uint32_t bump_needed, pad;
};
// DisneyMaterial's own parameters (disney.rs:464-483), a table beside `materials` that only the NL = 8 kernels read
struct DisneyRec {
    double v[10];      // metallic specular_tint anisotropic sheen sheen_tint clearcoat clearcoat_gloss spec_trans flatness diff_trans
    int32_t tex[10];   // texture index per parameter, -1 = the constant
    uint32_t thin, pad;
};
enum { DZ_METALLIC = 0, DZ_SPECULAR_TINT, DZ_ANISOTROPIC, DZ_SHEEN, DZ_SHEEN_TINT, DZ_CLEARCOAT, DZ_CLEARCOAT_GLOSS, DZ_SPEC_TRANS,
       DZ_FLATNESS, DZ_DIFF_TRANS };
struct LightRec {
    uint32_t kind, shape_kind;
    Rgb intensity;    // point: I; distant: L; diffuse area: lemit
    V3 p_light;       // point
    V3 w_light;       // distant (normalised, world space)
    double world_radius;
    // DiffuseAreaLight's shape (lights/diffuse.rs; renderprocess.rs:1078-1106)
    M34 o2w, w2o;     // sphere
    double radius;
    V3 tp[3], tn[3];  // triangle vertices and vertex normals
    uint32_t tri_has_n;
    int32_t env;      // InfiniteAreaLight: index into ShadeScene::envs
};
struct ShadeScene {
    const PrimInfo* prims;
    const MeshInfo* meshes;
    const double* mesh_p;     // xyz per vertex (object space; the obj transform is never applied, Q7)
    const uint32_t* mesh_vi;
    const double* mesh_n;
    const uint32_t* mesh_ni;
    const double* mesh_uv;
    const uint32_t* mesh_uvi;
    const SphereInfo* spheres;
    const InstanceXf* instances;
    const MaterialRec* materials;
    const TextureRec* textures;
    uint32_t n_textures;
    uint32_t bump;  // some material has a bump map: the textured shade kernel asks make_surface for the partials it reads
    // camera-ray differentials per path slot (null unless a texture filters with them: a closed-form checkerboard)
    const RayDiffRec* ray_diffs;
    const LightRec* lights;
    uint32_t n_lights;
    uint32_t literal;  // Tier L: instance / sphere rays are renormalised like the reference (Q6)
    const MipView* mips;        // one per ImageTexture (TextureRec::t1)
    const EnvLightView* envs;   // the InfiniteAreaLights of `lights` and of `infinite_lights`
    const int32_t* escape_envs; // Scene::infinite_lights: indices into envs (PathIntegrator, path.rs:84)
    uint32_t n_escape_envs, pad_sc;
    const DisneyRec* disney;    // one per material when some material is Translucent / Disney / Debug, else null
};

// What the integrator reads of a SurfaceInteraction (interaction.rs:95-113)
struct Surface {
    V3 p, n, wo;       // BaseInteraction: point, geometric normal, outgoing direction
    V3 shn, shdpdu;    // shading.n, shading.dpdu
    // what textures read (filled only for scenes that have textures): SurfaceInteraction::uv, dpdu, dpdv
    P2 uv;
    V3 dpdu, dpdv;
    uint32_t material;
};
// What Material::bump reads on top of that: shading.dpdv, shading.dndu, shading.dndv.  Kept out of Surface so that
// kernels for scenes without bump maps carry none of it (measured: 2-3 % of the frame when it sat in Surface).
struct BumpPartials {
    V3 shdpdv, shdndu, shdndv;
};

__device__ __forceinline__ V3 ld3(const double* a, uint64_t i) { return v3(a[3 * i], a[3 * i + 1], a[3 * i + 2]); }

// transform.rs:618-656
__device__ __forceinline__ void xf_surface(const M34& m, const M34& inv, Surface* s) {
    s->p = xf_point(m, s->p);
    s->wo = xf_vector(m, s->wo);
    s->n = xf_normal_inv(inv, s->n);
    s->shn = normalize_n(xf_normal_inv(inv, s->shn));
    s->shdpdu = xf_vector(m, s->shdpdu);
    s->shn = faceforward(s->shn, s->n);
}
__device__ __forceinline__ void xf_surface_partials(const M34& m, Surface* s) {
    s->dpdu = xf_vector(m, s->dpdu);
    s->dpdv = xf_vector(m, s->dpdv);
}
__device__ __forceinline__ void xf_surface_bump_partials(const M34& m, const M34& inv, BumpPartials* s) {
    s->shdpdv = xf_vector(m, s->shdpdv);
    s->shdndu = xf_normal_inv(inv, s->shdndu);
    s->shdndv = xf_normal_inv(inv, s->shdndv);
}

// sphere.rs:205-232: shading.dpdv and dndu / dndv from the second derivatives (Weingarten equations), carried to the
// sphere's world space like the rest of the SurfaceInteraction (sphere.rs:245-255)
static __device__ __noinline__ void sphere_bump_partials(const SphereInfo& sp, V3 p, V3 dpdu, V3 dpdv, double cos_phi, double sin_phi,
                                                         BumpPartials* bp) {
    const double dtheta = sp.theta_max - sp.theta_min;
    const V3 d2pduu = v3(p.x, p.y, 0.0) * -sp.phi_max * sp.phi_max;
    const V3 d2pduv = v3(-sin_phi, cos_phi, 0.0) * dtheta * p.z * sp.phi_max;
    const V3 d2pdvv = p * -dtheta * dtheta;
    const double E = dot(dpdu, dpdu), F = dot(dpdu, dpdv), G = dot(dpdv, dpdv);
    const V3 N = normalize(cross(dpdu, dpdv));
    const double e = dot(N, d2pduu), ff = dot(N, d2pduv), gg = dot(N, d2pdvv);
    const double inv_EGF2 = 1.0 / (E * G - F * F);
    bp->shdpdv = dpdv;
    bp->shdndu = dpdu * ((ff * F - e * G) * inv_EGF2) + dpdv * ((e * F - ff * E) * inv_EGF2);
    bp->shdndv = dpdu * ((gg * F - ff * G) * inv_EGF2) + dpdv * ((ff * F - gg * E) * inv_EGF2);
    xf_surface_bump_partials(sp.o2w, sp.w2o, bp);
}

// The geometric dndu / dndv of a SurfaceInteraction (interaction.rs:85-113): only the intersect API's surface records carry
// them.  Zero for triangles (Triangle::intersect hands SurfaceInteraction::new zero vectors); a sphere's are the Weingarten
// values that sphere_bump_partials computes for its shading frame (SurfaceInteraction::new copies them into `shading`).
struct GeomNormalPartials {
    V3 dndu, dndv;
};

// Rebuilds the surface frame of hit (prim_id, t, u, v) for the world ray (o, d).
// FULL = false (the renderer): uv / dpdu / dpdv only for scenes with textures, the shading partials only when `bp` is given.
// FULL = true (rrt_intersect_surface): every field of the SurfaceInteraction; `bp` and `gp` must be given.
template <bool FULL = false>
__device__ __forceinline__ void make_surface_body(const ShadeScene& sc, uint32_t prim_id, double t, double bu, double bv, V3 o, V3 d,
                                                  Surface* out, BumpPartials* bp, GeomNormalPartials* gp = nullptr) {
    const PrimInfo pi = sc.prims[prim_id];
    V3 lo = o, ld = d;
    if (pi.instance >= 0) {  // TransformedPrimitive::intersect (primitives.rs:126-139), Q6 fixed: d keeps its length
        const InstanceXf& x = sc.instances[pi.instance];
        lo = xf_point(x.inv, o);
        ld = xf_vector(x.inv, d);
        if (sc.literal) ld = normalize(normalize(ld));  // transform.rs:525-537 + Ray::new
    }
    Surface s;
    s.material = pi.material;
    const bool textured = FULL || sc.n_textures != 0;
    if ((pi.kind & kPrimKindMask) == 0) {
        const V3 p0 = ld3(sc.mesh_p, pi.gv[0]), p1 = ld3(sc.mesh_p, pi.gv[1]), p2 = ld3(sc.mesh_p, pi.gv[2]);
        MeshInfo mi = {};  // read only for meshes that carry uv or normals
        if (pi.kind & (kPrimHasUv | kPrimHasNormals)) mi = sc.meshes[pi.shape];
        // triangle.rs:113-129 get_uvs
        P2 uv0 = {0.0, 0.0}, uv1 = {1.0, 0.0}, uv2 = {1.0, 1.0};
        if (mi.has_uv) {
            const double* uvb = sc.mesh_uv + 2 * mi.uv_off;
            uint32_t i0 = 0, i1 = 0, i2 = 0;
            if (mi.has_uvi) {
                const uint32_t* ui = sc.mesh_uvi + mi.uvi_off + 3ull * pi.tri;
                i0 = ui[0]; i1 = ui[1]; i2 = ui[2];
            }
            uv0 = P2{uvb[2 * i0], uvb[2 * i0 + 1]};
            uv1 = P2{uvb[2 * i1], uvb[2 * i1 + 1]};
            uv2 = P2{uvb[2 * i2], uvb[2 * i2 + 1]};
        }
        const double du02 = uv0.x - uv2.x, dv02 = uv0.y - uv2.y, du12 = uv1.x - uv2.x, dv12 = uv1.y - uv2.y;
        const V3 dp02 = p0 - p2, dp12 = p1 - p2;
        const double determinant = du02 * dv12 - dv02 * du12;
        const bool degenerate_uv = fabs(determinant) < 1e-8;
        V3 dpdu = v3(0, 0, 0), dpdv = v3(0, 0, 0);
        if (!degenerate_uv) {
            const double i_det = 1.0 / determinant;
            dpdu = (dp02 * dv12 - dp12 * dv02) * i_det;
            dpdv = (dp02 * -du12 + dp12 * du02) * i_det;
        }
        if (degenerate_uv || length_sq(cross(dpdu, dpdv)) == 0.0) {
            V3 ng = cross(p2 - p0, p1 - p0);
            coordinate_system(normalize(ng), &dpdu, &dpdv);
        }
        s.p = lo + ld * t;
        s.wo = -ld;
        if (textured) {  // triangle.rs:289: uv[0] * (1 - u - v) + uv[1] * u + uv[2] * v
            const double b0 = sub(sub(1.0, bu), bv);
            s.uv = P2{add(add(mul(uv0.x, b0), mul(uv1.x, bu)), mul(uv2.x, bv)), add(add(mul(uv0.y, b0), mul(uv1.y, bu)), mul(uv2.y, bv))};
            s.dpdu = dpdu;
            s.dpdv = dpdv;
        }
        const V3 ist_n = normalize(cross(dp02, dp12));
        s.n = ist_n;
        s.shn = ist_n;
        s.shdpdu = dpdu;
        if (bp) {
            bp->shdpdv = dpdv;
            bp->shdndu = bp->shdndv = v3(0, 0, 0);
        }
        if constexpr (FULL) gp->dndu = gp->dndv = v3(0, 0, 0);
        if (mi.has_n && mi.has_ni) {
            const uint32_t* ni = sc.mesh_ni + mi.ni_off + 3ull * pi.tri;
            const double* nb = sc.mesh_n + 3 * mi.n_off;
            const V3 n0 = ld3(nb, ni[0]), n1 = ld3(nb, ni[1]), n2 = ld3(nb, ni[2]);
            V3 ns = n0 * (1.0 - bu - bv) + n1 * bu + n2 * bv;
            ns = length_sq(ns) > 0.0 ? normalize_n(ns) : ist_n;
            V3 ss = normalize(dpdu);
            V3 ts = cross(ss, ns);
            if (length_sq(ts) > 0.0) {
                ts = normalize(ts);
                ss = cross(ts, ns);
            } else {
                coordinate_system(ns, &ss, &ts);
            }
            // set_shading_geometry(ss, ts, .., orientation_is_authoritative = true): the shading
            // normal is the GEOMETRIC normal flipped towards ss x ts (interaction.rs:186-202)
            V3 nn = normalize(cross(ss, ts));
            s.shn = faceforward(s.n, nn);
            s.shdpdu = ss;
            if (bp) {  // triangle.rs:331-366: dndu / dndv from the vertex normals, shading.dpdv = ts
                bp->shdpdv = ts;
                const V3 dn1 = n0 - n2, dn2 = n1 - n2;
                if (degenerate_uv) {
                    const V3 dn = cross(n2 - n0, n1 - n0);
                    if (length_sq(dn) != 0.0) coordinate_system(dn, &bp->shdndu, &bp->shdndv);
                } else {
                    const double i_det = 1.0 / determinant;
                    bp->shdndu = (dn1 * dv12 - dn2 * dv02) * i_det;
                    bp->shdndv = (dn1 * -du12 + dn2 * du02) * i_det;
                }
            }
        }
    } else {
        const SphereInfo& sp = sc.spheres[pi.shape];
        // sphere.rs:127-128: the shape works on the object-space ray, but the first hit point is
        // taken on the ray it was handed (Q5a)
        V3 od = xf_vector(sp.w2o, ld);
        if (sc.literal) od = normalize(normalize(od));
        V3 p = lo + ld * t;
        if (p.x == 0.0 && p.y == 0.0) p.x = 1e-5 * sp.radius;
        double phi = atan2(p.y, p.x);
        if (phi < 0.0) phi += 2.0 * kPi;
        if (sp.partial && !sc.literal) {
            // a clipped sphere may have been hit at its far root, whose point is taken on the object-space ray and
            // re-projected (sphere.rs:171-186): replay the accepted hit (t_far = t reproduces the decisions)
            const SphereClip clip = {sp.radius, sp.z_min, sp.z_max, sp.phi_max};
            V3 q;
            double tt, f;
            if (sphere_hit_local(sp.w2o, clip, lo, ld, t, &tt, &q, &f)) {
                p = q;
                phi = f;
            }
        }
        const double theta = acos(clampd(p.z / sp.radius, -1.0, 1.0));
        const double z_radius = sqrt(p.x * p.x + p.y * p.y);
        const double inv_z_radius = 1.0 / z_radius;
        const double cos_phi = p.x * inv_z_radius, sin_phi = p.y * inv_z_radius;
        const V3 dpdu = v3(-sp.phi_max * p.y, sp.phi_max * p.x, 0.0);
        const V3 dpdv = v3(p.z * cos_phi, p.z * sin_phi, -sp.radius * sin(theta)) * (sp.theta_max - sp.theta_min);
        if (bp) sphere_bump_partials(sp, p, dpdu, dpdv, cos_phi, sin_phi, bp);  // out of line: bump-mapped scenes only
        if constexpr (FULL) {
            gp->dndu = bp->shdndu;
            gp->dndv = bp->shdndv;
        }
        s.p = p;
        s.wo = -od;
        s.n = normalize(cross(dpdu, dpdv));
        s.shn = s.n;
        s.shdpdu = dpdu;
        xf_surface(sp.o2w, sp.w2o, &s);  // sphere.rs:245-255: always applied
        if (textured) {
            s.uv = P2{phi / sp.phi_max, sub(theta, sp.theta_min) / sub(sp.theta_max, sp.theta_min)};  // sphere.rs:157-160
            s.dpdu = dpdu;
            s.dpdv = dpdv;
            xf_surface_partials(sp.o2w, &s);
        }
    }
    if (pi.instance >= 0) {
        const InstanceXf& x = sc.instances[pi.instance];
        if (!x.is_identity) {
            xf_surface(x.m, x.inv, &s);  // primitives.rs:135-137
            if (textured) xf_surface_partials(x.m, &s);
            if (bp) xf_surface_bump_partials(x.m, x.inv, bp);
            if constexpr (FULL) {
                gp->dndu = xf_normal_inv(x.inv, gp->dndu);
                gp->dndv = xf_normal_inv(x.inv, gp->dndv);
            }
        }
    }
    *out = s;
}
// Out of line for the general kernels (measured: 160 registers without spills, +3 %); the kernels specialised by material
// kind inline the body.
static __device__ __noinline__ void make_surface(const ShadeScene& sc, uint32_t prim_id, double t, double bu, double bv, V3 o, V3 d,
                                                 Surface* out, BumpPartials* bp = nullptr) {
    make_surface_body(sc, prim_id, t, bu, bv, o, d, out, bp);
}

// ---- reflection.rs helpers ---------------------------------------------------------------------------
__device__ __forceinline__ double cos2_theta(V3 w) { return w.z * w.z; }
__device__ __forceinline__ double abs_cos_theta(V3 w) { return fabs(w.z); }
__device__ __forceinline__ double sin2_theta(V3 w) { return rmax(0.0, 1.0 - cos2_theta(w)); }
__device__ __forceinline__ double sin_theta(V3 w) { return sqrt(sin2_theta(w)); }
__device__ __forceinline__ double tan_theta(V3 w) { return sin_theta(w) / w.z; }
__device__ __forceinline__ double tan2_theta(V3 w) { return sin2_theta(w) / cos2_theta(w); }
__device__ __forceinline__ double cos_phi(V3 w) {
    double s = sin_theta(w);
    return s == 0.0 ? 1.0 : clampd(w.x / s, -1.0, 1.0);
}
__device__ __forceinline__ double sin_phi(V3 w) {
    double s = sin_theta(w);
    return s == 0.0 ? 0.0 : clampd(w.y / s, -1.0, 1.0);
}
__device__ __forceinline__ bool same_hemisphere(V3 a, V3 b) { return a.z * b.z > 0.0; }
__device__ __forceinline__ V3 reflect_about(V3 wo, V3 n) { return -wo + n * 2.0 * dot(wo, n); }
__device__ __forceinline__ bool refract_dir(V3 wi, V3 n, double eta, V3* wt) {
    double cos_i = dot(n, wi);
    double sin2_i = rmax(0.0, 1.0 - cos_i * cos_i);
    double sin2_t = eta * eta * sin2_i;
    if (sin2_t >= 1.0) return false;
    double cos_t = sqrt(1.0 - sin2_t);
    *wt = -wi * eta + n * (eta * cos_i - cos_t);
    return true;
}
// reflection.rs:145-168
static __device__ double fr_dielectric(double cos_i, double eta_i, double eta_t) {
    cos_i = clampd(cos_i, -1.0, 1.0);
    if (!(cos_i > 0.0)) {
        double s = eta_i;
        eta_i = eta_t;
        eta_t = s;
        cos_i = fabs(cos_i);
    }
    double sin_i = sqrt(rmax(0.0, 1.0 - cos_i * cos_i));
    double sin_t = eta_i / eta_t * sin_i;
    if (sin_t >= 1.0) return 1.0;
    double cos_t = sqrt(rmax(0.0, 1.0 - sin_t * sin_t));
    double r_parl = ((eta_t * cos_i) - (eta_i * cos_t)) / ((eta_t * cos_i) + (eta_i * cos_t));
    double r_perp = ((eta_i * cos_i) - (eta_t * cos_t)) / ((eta_i * cos_i) + (eta_t * cos_t));
    return (r_parl * r_parl + r_perp * r_perp) / 2.0;
}
// reflection.rs:170-195
static __device__ Rgb fr_conductor(double cos_i, Rgb eta_i, Rgb eta_t, Rgb k) {
    cos_i = clampd(cos_i, -1.0, 1.0);
    Rgb eta = eta_t / eta_i, eta_k = k / eta_i;
    double cos2 = cos_i * cos_i, sin2 = 1.0 - cos2;
    Rgb eta_2 = eta * eta, eta_k2 = eta_k * eta_k;
    Rgb t0 = eta_2 - eta_k2 - rgb(sin2);
    Rgb a2_plus_b2 = sqrt_rgb(t0 * t0 + eta_2 * eta_k2 * rgb(4.0));
    Rgb t1 = a2_plus_b2 + rgb(cos2);
    Rgb a = sqrt_rgb((a2_plus_b2 + t0) * 0.5);
    Rgb t2 = a * 2.0 * cos_i;
    Rgb rs = (t1 - t2) / (t1 + t2);
    Rgb t3 = a2_plus_b2 * cos2 + rgb(sin2 * sin2);
    Rgb t4 = t2 * sin2;
    Rgb rp = rs * (t3 - t4) / (t3 + t4);
    return (rp + rs) * rgb(0.5);
}
// microfacet.rs:12-20
static __device__ double roughness_to_alpha(double roughness) {
    roughness = rmax(roughness, 1e-3);
    double x = log(roughness);
    return 1.62142 + 0.819955 * x + 0.1734 * x * x + 0.0171201 * x * x * x + 0.000640711 * x * x * x * x;
}

// ---- lobes -----------------------------------------------------------------------------------------------
enum : uint32_t { BXDF_REFLECTION = 1, BXDF_TRANSMISSION = 2, BXDF_DIFFUSE = 4, BXDF_GLOSSY = 8, BXDF_SPECULAR = 16, BXDF_ALL = 31 };
enum : uint32_t { LOBE_LAMBERT = 0, LOBE_OREN_NAYAR, LOBE_MICROFACET, LOBE_SPEC_REFL, LOBE_SPEC_TRANS, LOBE_FRESNEL_SPEC,
                  LOBE_MICROFACET_TRANS,
                  // NL = 8 only
                  LOBE_LAMBERT_TRANS,     // reflection.rs:843-898
                  LOBE_DISNEY_DIFFUSE,    // disney.rs:33-75
                  LOBE_DISNEY_FAKESS,     // disney.rs:77-131   (eta_a = roughness)
                  LOBE_DISNEY_RETRO,      // disney.rs:133-180  (eta_a = roughness)
                  LOBE_DISNEY_SHEEN,      // disney.rs:182-224
                  LOBE_DISNEY_CLEARCOAT,  // disney.rs:226-303  (eta_a = weight, eta_b = gloss)
                  LOBE_DEBUG_DIFFUSE,     // debug_material.rs:10-20
                  LOBE_DEBUG_SPECULAR };  // debug_material.rs:22-32: typed specular, cosine-sampled
// FRESNEL_DISNEY (disney.rs:305-326): cond_eta = r0, a = metallic, b = eta.  NL = 8 lobes may also carry
// FRESNEL_SEPARABLE_G: DisneyMicrofacetDistribution's g = g1(wo) * g1(wi) (disney.rs:329-360).
enum : uint32_t { FRESNEL_NOOP = 0, FRESNEL_DIELECTRIC = 1, FRESNEL_CONDUCTOR = 2, FRESNEL_DISNEY = 3, FRESNEL_SEPARABLE_G = 256 };

// ---- lobe sets ---------------------------------------------------------------------------------------------------
// A material kind fixes which lobe kinds (bits 0..15) and Fresnel terms (bits 16..) its Bsdf can hold.  Every function
// below takes that set as a template parameter: kLobesAll is the general code (out of line, the Bsdf in local memory — what
// the textured / eight-lobe / environment kernels and the "any kind" shade kernel run); a narrower set prunes the other
// lobes' code at compile time, is inlined into its caller and indexes the lobes statically, so that the Bsdf of a Matte,
// Plastic or Metal hit lives in registers (shade_range_kernel<KIND>, render_kernels.cuh).  Same functions, same operation
// order: a specialised kernel's results are bit-identical to the general one's.
constexpr uint32_t kLobesAll = 0xffffffffu;
__host__ __device__ constexpr uint32_t lobe_bit(uint32_t k) { return 1u << k; }
__host__ __device__ constexpr uint32_t fresnel_bit(uint32_t f) { return 1u << (16u + f); }
constexpr uint32_t kLobesMatte = lobe_bit(LOBE_LAMBERT) | lobe_bit(LOBE_OREN_NAYAR) | fresnel_bit(FRESNEL_NOOP);
constexpr uint32_t kLobesPlastic = lobe_bit(LOBE_LAMBERT) | lobe_bit(LOBE_MICROFACET) | fresnel_bit(FRESNEL_NOOP) | fresnel_bit(FRESNEL_DIELECTRIC);
constexpr uint32_t kLobesMetal = lobe_bit(LOBE_MICROFACET) | fresnel_bit(FRESNEL_CONDUCTOR);
#define RRT_LOBE_IN(MASK, K) ((((MASK) >> (K)) & 1u) != 0u)
#define RRT_FRESNEL_IN(MASK, F) ((((MASK) >> (16u + (F))) & 1u) != 0u)
__host__ __device__ constexpr bool lobe_set_is_single(uint32_t mask) { return (mask & 0xffffu) != 0u && ((mask & 0xffffu) & ((mask & 0xffffu) - 1u)) == 0u; }
__host__ __device__ constexpr uint32_t lobe_set_first(uint32_t mask) {
    uint32_t k = 0;
    while (k < 16u && !((mask >> k) & 1u)) ++k;
    return k;
}

struct Lobe {
    uint32_t kind, fresnel;
    Rgb r, t;           // reflectance / transmittance
    Rgb cond_eta, cond_k;  // FresnelConductor eta_t, k (eta_i = 1)
    double a, b;        // FresnelDielectric eta_i, eta_t of the lobe's Fresnel term
    double eta_a, eta_b;   // specular transmission / FresnelSpecular indices; Oren–Nayar A, B
    double alpha_x, alpha_y;
};
template <uint32_t MASK>
__device__ __forceinline__ uint32_t lobe_kind(const Lobe& l) {  // a one-lobe set knows its kind at compile time
    if (MASK != kLobesAll && lobe_set_is_single(MASK)) return lobe_set_first(MASK);
    return l.kind;
}
template <bool BIG = false, uint32_t MASK = kLobesAll>
__device__ __forceinline__ uint32_t lobe_type(const Lobe& l) {
    switch (lobe_kind<MASK>(l)) {
        case LOBE_LAMBERT:
        case LOBE_OREN_NAYAR: return BXDF_DIFFUSE | BXDF_REFLECTION;
        case LOBE_MICROFACET: return BXDF_GLOSSY | BXDF_REFLECTION;
        case LOBE_SPEC_REFL: return BXDF_REFLECTION | BXDF_SPECULAR;
        case LOBE_SPEC_TRANS: return BXDF_SPECULAR | BXDF_TRANSMISSION;
        case LOBE_MICROFACET_TRANS: return BXDF_GLOSSY | BXDF_TRANSMISSION;  // reflection.rs:1143-1145
        default: break;
    }
    if (BIG) {
        switch (lobe_kind<MASK>(l)) {
            case LOBE_LAMBERT_TRANS: return BXDF_DIFFUSE | BXDF_TRANSMISSION;
            case LOBE_DISNEY_DIFFUSE:
            case LOBE_DISNEY_FAKESS:
            case LOBE_DISNEY_RETRO:
            case LOBE_DISNEY_SHEEN:
            case LOBE_DEBUG_DIFFUSE: return BXDF_DIFFUSE | BXDF_REFLECTION;
            // disney.rs:300-302: neither REFLECTION nor TRANSMISSION — Bsdf::f never adds the clearcoat lobe, it is
            // only seen through sample_f and pdf (Q37)
            case LOBE_DISNEY_CLEARCOAT: return BXDF_DIFFUSE | BXDF_GLOSSY;
            case LOBE_DEBUG_SPECULAR: return BXDF_SPECULAR | BXDF_REFLECTION;
            default: break;
        }
    }
    return BXDF_SPECULAR | BXDF_ALL;  // FresnelSpecular, reflection.rs:801-803
}
template <bool BIG = false, uint32_t MASK = kLobesAll>
__device__ __forceinline__ bool lobe_matches(const Lobe& l, uint32_t flags) { return (lobe_type<BIG, MASK>(l) & flags) == lobe_type<BIG, MASK>(l); }
// reflection.rs:13-24, misc.rs:223-228 (lerp(t, a, b) = a * (1 - t) + b * t)
__device__ __forceinline__ double schlick_weight(double c) {
    const double m = clampd(1.0 - c, 0.0, 1.0);
    return (m * m) * (m * m) * m;
}
__device__ __forceinline__ double lerp_f(double t, double a, double b) { return a * (1.0 - t) + b * t; }
__device__ __forceinline__ Rgb lerp_rgb(double t, Rgb a, Rgb b) { return a * (1.0 - t) + b * t; }
template <bool BIG = false, uint32_t MASK = kLobesAll>
static __device__ Rgb lobe_fresnel(const Lobe& l, double cos_i) {  // reflection.rs:603-619
    const uint32_t fk = BIG ? (l.fresnel & 255u) : l.fresnel;
    if (BIG && fk == FRESNEL_DISNEY)
        return lerp_rgb(l.a, rgb(fr_dielectric(cos_i, 1.0, l.b)), lerp_rgb(schlick_weight(cos_i), l.cond_eta, rgb(1.0)));
    if (RRT_FRESNEL_IN(MASK, FRESNEL_DIELECTRIC) && fk == FRESNEL_DIELECTRIC) return rgb(fr_dielectric(cos_i, l.a, l.b));
    if (RRT_FRESNEL_IN(MASK, FRESNEL_CONDUCTOR) && fk == FRESNEL_CONDUCTOR) return fr_conductor(fabs(cos_i), rgb(1.0), l.cond_eta, l.cond_k);
    return rgb(1.0);
}
// TrowbridgeReitzDistribution (microfacet.rs:364-390)
static __device__ double tr_d(const Lobe& l, V3 wh) {
    double tan2 = tan2_theta(wh);
    if (isinf(tan2)) return 0.0;
    double cos4 = cos2_theta(wh) * cos2_theta(wh);
    double cp = cos_phi(wh), spv = sin_phi(wh);
    double e = ((cp * cp) / (l.alpha_x * l.alpha_x) + (spv * spv) / (l.alpha_y * l.alpha_y)) * tan2;
    return 1.0 / (kPi * l.alpha_x * l.alpha_y * cos4 * (1.0 + e) * (1.0 + e));
}
static __device__ double tr_lambda(const Lobe& l, V3 w) {
    double abs_tan = fabs(tan_theta(w));
    if (isinf(abs_tan)) return 0.0;
    double cp = cos_phi(w), spv = sin_phi(w);
    double alpha = sqrt((cp * cp) * (l.alpha_x * l.alpha_x) + (spv * spv) * (l.alpha_y * l.alpha_y));
    double a2t2 = (alpha * abs_tan) * (alpha * abs_tan);
    return (-1.0 + sqrt(1.0 + a2t2)) / 2.0;
}
static __device__ double tr_pdf(const Lobe& l, V3 wo, V3 wh) {  // microfacet.rs:30-36, sample_visible_area
    return tr_d(l, wh) * (1.0 / (1.0 + tr_lambda(l, wo))) * absdot(wo, wh) / abs_cos_theta(wo);
}
template <bool BIG = false>
__device__ __forceinline__ double tr_g(const Lobe& l, V3 wo, V3 wi) {  // (a narrowed lobe set is never BIG)
    if (BIG && (l.fresnel & FRESNEL_SEPARABLE_G)) return (1.0 / (1.0 + tr_lambda(l, wo))) * (1.0 / (1.0 + tr_lambda(l, wi)));
    return 1.0 / (1.0 + tr_lambda(l, wo) + tr_lambda(l, wi));
}
// disney.rs:20-31; gtr1 divides by log10(alpha^2) where pbrt has the natural logarithm: kept (Q36)
static __device__ double gtr1(double cos_t, double alpha) {
    const double alpha2 = alpha * alpha;
    return (alpha2 - 1.0) / (kPi * log10(alpha2) * (1.0 + (alpha2 - 1.0) * cos_t * cos_t));
}
static __device__ double smith_g_ggx(double cos_t, double alpha) {
    const double alpha2 = alpha * alpha, cos2 = cos_t * cos_t;
    return 1.0 / (cos_t + sqrt(alpha2 + cos2 - alpha2 * cos2));
}
// microfacet.rs:270-362
static __device__ V3 tr_sample_visible(V3 wi, double ax, double ay, double u1, double u2) {
    V3 ws = normalize(v3(ax * wi.x, ay * wi.y, wi.z));
    double slope_x, slope_y;
    const double cos_t = ws.z;
    if (cos_t > 0.9999) {
        double r = sqrt(u1 / (1.0 - u1));
        double phi = 6.28318530718 * u2;
        slope_x = r * cos(phi);
        slope_y = r * sin(phi);
    } else {
        double sin_t = sqrt(rmax(0.0, 1.0 - cos_t * cos_t));
        double tan_t = sin_t / cos_t;
        double a = 1.0 / tan_t;
        double g1 = 2.0 / (1.0 + sqrt(1.0 + 1.0 / (a * a)));
        a = 2.0 * u1 / g1 - 1.0;
        double tmp = 1.0 / (a * a - 1.0);
        if (tmp > 1e10) tmp = 1e10;
        double b = tan_t;
        double dd = sqrt(rmax(b * b * tmp * tmp - (a * a - b * b) * tmp, 0.0));
        double sx1 = b * tmp - dd, sx2 = b * tmp + dd;
        slope_x = (a < 0.0 || sx2 > 1.0 / tan_t) ? sx1 : sx2;
        double s, nu2;
        if (u2 > 0.5) {
            s = 1.0;
            nu2 = 2.0 * (u2 - 0.5);
        } else {
            s = -1.0;
            nu2 = 2.0 * (0.5 - u2);
        }
        double z = (nu2 * (nu2 * (nu2 * 0.27385 - 0.73369) + 0.46341)) /
                   (nu2 * (nu2 * (nu2 * 0.093073 + 0.309420) - 1.0) + 0.597999);
        slope_y = s * z * sqrt(1.0 + slope_x * slope_x);
    }
    double tmp = cos_phi(ws) * slope_x - sin_phi(ws) * slope_y;
    slope_y = sin_phi(ws) * slope_x + cos_phi(ws) * slope_y;
    slope_x = tmp;
    slope_x *= ax;
    slope_y *= ay;
    return normalize(v3(-slope_x, -slope_y, 1.0));
}

template <bool BIG, uint32_t MASK>
__device__ __forceinline__ Rgb lobe_f_body(const Lobe& l, V3 wo, V3 wi) {
    if (BIG) {
        switch (l.kind) {
            case LOBE_LAMBERT_TRANS: return l.t / kPi;
            case LOBE_DEBUG_DIFFUSE: return Rgb{0.0, 1.0, 0.0};
            case LOBE_DEBUG_SPECULAR: return Rgb{0.0, 0.0, 1.0};
            case LOBE_DISNEY_DIFFUSE: {
                const double fo = schlick_weight(abs_cos_theta(wo)), fi = schlick_weight(abs_cos_theta(wi));
                return l.r / kPi * (1.0 - fo / 2.0) * (1.0 - fi / 2.0);
            }
            case LOBE_DISNEY_FAKESS:
            case LOBE_DISNEY_RETRO:
            case LOBE_DISNEY_SHEEN:
            case LOBE_DISNEY_CLEARCOAT: {
                V3 wh = wi + wo;
                if (wh.x == 0.0 && wh.y == 0.0 && wh.z == 0.0) return rgb(0.0);
                wh = normalize(wh);
                if (l.kind == LOBE_DISNEY_CLEARCOAT) {
                    const double dr = gtr1(abs_cos_theta(wh), l.eta_b);
                    const double fr = lerp_f(schlick_weight(dot(wo, wh)), 0.04, 1.0);
                    const double gr = smith_g_ggx(abs_cos_theta(wo), 0.25) * smith_g_ggx(abs_cos_theta(wi), 0.25);
                    return rgb(l.eta_a * gr * fr * dr / 4.0);
                }
                const double cos_theta_d = dot(wi, wh);
                if (l.kind == LOBE_DISNEY_SHEEN) return l.r * schlick_weight(cos_theta_d);
                const double fo = schlick_weight(abs_cos_theta(wo)), fi = schlick_weight(abs_cos_theta(wi));
                if (l.kind == LOBE_DISNEY_RETRO) {
                    const double r_r = 2.0 * l.eta_a * cos_theta_d * cos_theta_d;
                    return l.r / kPi * r_r * (fo + fi + fo * fi * (r_r - 1.0));
                }
                const double fss_90 = cos_theta_d * cos_theta_d * l.eta_a;
                const double fss = lerp_f(fo, 1.0, fss_90) * lerp_f(fi, 1.0, fss_90);
                const double ss = 1.25 * (fss * (1.0 / (abs_cos_theta(wo) + abs_cos_theta(wi)) - 0.5) + 0.5);
                return l.r / kPi * ss;
            }
            default: break;
        }
    }
    switch (lobe_kind<MASK>(l)) {
        case LOBE_LAMBERT:
            if (!RRT_LOBE_IN(MASK, LOBE_LAMBERT)) break;
            return l.r / kPi;
        case LOBE_OREN_NAYAR: {  // reflection.rs:916-941
            if (!RRT_LOBE_IN(MASK, LOBE_OREN_NAYAR)) break;
            double sin_i = sin_theta(wi), sin_o = sin_theta(wo), max_cos = 0.0;
            if (sin_i > 1e-4 && sin_o > 1e-4) {
                double d_cos = cos_phi(wi) * cos_phi(wo) + sin_phi(wi) * sin_phi(wo);
                max_cos = rmax(d_cos, 0.0);
            }
            double sin_alpha, tan_beta;
            if (abs_cos_theta(wi) > abs_cos_theta(wo)) {
                sin_alpha = sin_o;
                tan_beta = sin_i / abs_cos_theta(wi);
            } else {
                sin_alpha = sin_i;
                tan_beta = sin_o / abs_cos_theta(wo);
            }
            return l.r / kPi * (l.eta_a + l.eta_b * max_cos * sin_alpha * tan_beta);
        }
        case LOBE_MICROFACET: {  // reflection.rs:970-990
            if (!RRT_LOBE_IN(MASK, LOBE_MICROFACET)) break;
            double cos_o = abs_cos_theta(wo), cos_i = abs_cos_theta(wi);
            V3 wh = wi + wo;
            if (cos_i == 0.0 || cos_o == 0.0) return rgb(0.0);
            if (wh.x == 0.0 && wh.y == 0.0 && wh.z == 0.0) return rgb(0.0);
            wh = normalize(wh);
            Rgb fr = lobe_fresnel<BIG, MASK>(l, dot(wi, faceforward(wh, v3(0.0, 0.0, 1.0))));
            double g = tr_g<BIG>(l, wo, wi);
            return l.r * tr_d(l, wh) * g * fr / (4.0 * cos_i * cos_o);
        }
        case LOBE_MICROFACET_TRANS: {  // MicrofacetTransmission::f (reflection.rs:1058-1099), TransportMode::Radiance
            if (!RRT_LOBE_IN(MASK, LOBE_MICROFACET_TRANS)) break;
            if (same_hemisphere(wo, wi)) return rgb(0.0);
            const double cos_o = wo.z, cos_i = wi.z;
            if (cos_i == 0.0 || cos_o == 0.0) return rgb(0.0);
            const double eta = wo.z > 0.0 ? l.eta_b / l.eta_a : l.eta_a / l.eta_b;
            V3 wh = normalize(wo + wi * eta);
            if (wh.z < 0.0) wh = -wh;
            const Rgb fr = rgb(fr_dielectric(dot(wo, wh), l.eta_a, l.eta_b));
            const double sqrt_denom = dot(wo, wh) + eta * dot(wi, wh);
            const double factor = 1.0 / eta;
            const double g = tr_g<BIG>(l, wo, wi);
            return (rgb(1.0) - fr) * l.t *
                   fabs(tr_d(l, wh) * g * eta * eta * absdot(wi, wh) * absdot(wo, wh) * factor * factor /
                        (cos_i * cos_o * sqrt_denom * sqrt_denom));
        }
        default: break;
    }
    return rgb(0.0);
}
template <bool BIG>
RRT_SHADE_FN Rgb lobe_f_out(const Lobe& l, V3 wo, V3 wi) { return lobe_f_body<BIG, kLobesAll>(l, wo, wi); }
template <bool BIG = false, uint32_t MASK = kLobesAll>
__device__ __forceinline__ Rgb lobe_f(const Lobe& l, V3 wo, V3 wi) {
    if constexpr (MASK == kLobesAll) return lobe_f_out<BIG>(l, wo, wi);
    else return lobe_f_body<BIG, MASK>(l, wo, wi);
}
template <bool BIG, uint32_t MASK>
__device__ __forceinline__ double lobe_pdf_body(const Lobe& l, V3 wo, V3 wi) {
    if (BIG) {
        switch (l.kind) {
            case LOBE_DISNEY_DIFFUSE:
            case LOBE_DISNEY_FAKESS:
            case LOBE_DISNEY_RETRO:
            case LOBE_DISNEY_SHEEN:
            case LOBE_DEBUG_DIFFUSE:
            case LOBE_DEBUG_SPECULAR: return same_hemisphere(wo, wi) ? abs_cos_theta(wi) / kPi : 0.0;  // reflection.rs:480-486
            case LOBE_LAMBERT_TRANS: return !same_hemisphere(wo, wi) ? abs_cos_theta(wi) / kPi : 0.0;
            case LOBE_DISNEY_CLEARCOAT: {  // disney.rs:283-299
                if (!same_hemisphere(wo, wi)) return 0.0;
                V3 wh = wi + wo;
                if (wh.x == 0.0 && wh.y == 0.0 && wh.z == 0.0) return 0.0;
                wh = normalize(wh);
                const double dr = gtr1(abs_cos_theta(wh), l.eta_b);
                return dr * abs_cos_theta(wh) / (4.0 * dot(wo, wh));
            }
            default: break;
        }
    }
    switch (lobe_kind<MASK>(l)) {
        case LOBE_LAMBERT:
        case LOBE_OREN_NAYAR: return same_hemisphere(wo, wi) ? abs_cos_theta(wi) / kPi : 0.0;
        case LOBE_MICROFACET: {
            if (!RRT_LOBE_IN(MASK, LOBE_MICROFACET)) break;
            if (!same_hemisphere(wo, wi)) return 0.0;
            V3 wh = normalize(wo + wi);
            return tr_pdf(l, wo, wh) / (4.0 * dot(wo, wh));
        }
        case LOBE_MICROFACET_TRANS: {  // reflection.rs:1127-1142
            if (!RRT_LOBE_IN(MASK, LOBE_MICROFACET_TRANS)) break;
            if (same_hemisphere(wo, wi)) return 0.0;
            const double eta = wo.z > 0.0 ? l.eta_b / l.eta_a : l.eta_a / l.eta_b;
            const V3 wh = normalize(wo + wi * eta);
            const double sqrt_denom = dot(wo, wh) + dot(wi, wh) * eta;
            const double dwh_dwi = fabs((eta * eta * dot(wi, wh)) / (sqrt_denom * sqrt_denom));
            return tr_pdf(l, wo, wh) * dwh_dwi;
        }
        default: break;
    }
    return 0.0;
}
template <bool BIG>
RRT_SHADE_FN double lobe_pdf_out(const Lobe& l, V3 wo, V3 wi) { return lobe_pdf_body<BIG, kLobesAll>(l, wo, wi); }
template <bool BIG = false, uint32_t MASK = kLobesAll>
__device__ __forceinline__ double lobe_pdf(const Lobe& l, V3 wo, V3 wi) {
    if constexpr (MASK == kLobesAll) return lobe_pdf_out<BIG>(l, wo, wi);
    else return lobe_pdf_body<BIG, MASK>(l, wo, wi);
}
// BxDF::sample_f of each lobe; *pdf is left untouched on the early-outs (the caller zeroed it)
template <bool BIG, uint32_t MASK>
__device__ __forceinline__ Rgb lobe_sample_f_body(const Lobe& l, V3 wo, V3* wi, P2 u, double* pdf, uint32_t* sampled_type) {
    if (BIG) {
        switch (l.kind) {
            case LOBE_DISNEY_DIFFUSE:
            case LOBE_DISNEY_FAKESS:
            case LOBE_DISNEY_RETRO:
            case LOBE_DISNEY_SHEEN:
            case LOBE_DEBUG_DIFFUSE:
            case LOBE_DEBUG_SPECULAR: {  // BxDF's default sample_f, reflection.rs:428-443
                *wi = cosine_sample_hemisphere(u);
                if (wo.z < 0.0) wi->z *= -1.0;
                *pdf = lobe_pdf<BIG>(l, wo, *wi);
                return lobe_f<BIG>(l, wo, *wi);
            }
            case LOBE_LAMBERT_TRANS: {  // reflection.rs:857-871
                *wi = cosine_sample_hemisphere(u);
                if (wo.z > 0.0) wi->z *= -1.0;
                *pdf = lobe_pdf<BIG>(l, wo, *wi);
                return lobe_f<BIG>(l, wo, *wi);
            }
            case LOBE_DISNEY_CLEARCOAT: {  // disney.rs:254-282; the square root covers the denominator only (Q36)
                if (wo.z == 0.0) return rgb(0.0);
                const double alpha2 = l.eta_b * l.eta_b;
                const double cos_t = (1.0 - pow(alpha2, 1.0 - u.x)) / sqrt(rmax(1.0 - alpha2, 0.0));
                const double sin_t = sqrt(rmax(1.0 - cos_t * cos_t, 0.0));
                const double phi = 2.0 * kPi * u.y;
                V3 wh = v3(sin_t * cos(phi), sin_t * sin(phi), cos_t);
                if (!same_hemisphere(wo, wh)) wh = -wh;
                *wi = reflect_about(wo, wh);
                if (!same_hemisphere(wo, *wi)) return rgb(0.0);
                *pdf = lobe_pdf<BIG>(l, wo, *wi);
                return lobe_f<BIG>(l, wo, *wi);
            }
            default: break;
        }
    }
    switch (lobe_kind<MASK>(l)) {
        case LOBE_LAMBERT:
        case LOBE_OREN_NAYAR: {  // reflection.rs:428-443
            if (!RRT_LOBE_IN(MASK, LOBE_LAMBERT) && !RRT_LOBE_IN(MASK, LOBE_OREN_NAYAR)) break;
            *wi = cosine_sample_hemisphere(u);
            if (wo.z < 0.0) wi->z *= -1.0;
            *pdf = lobe_pdf<BIG, MASK>(l, wo, *wi);
            return lobe_f<BIG, MASK>(l, wo, *wi);
        }
        case LOBE_MICROFACET: {  // reflection.rs:991-1015
            if (!RRT_LOBE_IN(MASK, LOBE_MICROFACET)) break;
            if (wo.z == 0.0) return rgb(0.0);
            V3 wh = wo.z < 0.0 ? -tr_sample_visible(-wo, l.alpha_x, l.alpha_y, u.x, u.y)
                               : tr_sample_visible(wo, l.alpha_x, l.alpha_y, u.x, u.y);
            if (dot(wo, wh) < 0.0) return rgb(0.0);
            *wi = reflect_about(wo, wh);
            if (!same_hemisphere(wo, *wi)) return rgb(0.0);
            *pdf = tr_pdf(l, wo, wh) / (4.0 * dot(wo, wh));
            return lobe_f<BIG, MASK>(l, wo, *wi);
        }
        case LOBE_SPEC_REFL: {  // reflection.rs:638-649
            if (!RRT_LOBE_IN(MASK, LOBE_SPEC_REFL)) break;
            *wi = v3(-wo.x, -wo.y, wo.z);
            *pdf = 1.0;
            return lobe_fresnel<BIG, MASK>(l, wi->z) * l.r / abs_cos_theta(*wi);
        }
        case LOBE_SPEC_TRANS: {  // reflection.rs:686-714, TransportMode::Radiance
            if (!RRT_LOBE_IN(MASK, LOBE_SPEC_TRANS)) break;
            bool entering = wo.z > 0.0;
            double ei = entering ? l.eta_a : l.eta_b, et = entering ? l.eta_b : l.eta_a;
            if (!refract_dir(wo, faceforward(v3(0.0, 0.0, 1.0), wo), ei / et, wi)) return rgb(0.0);
            *pdf = 1.0;
            Rgb ft = l.t * (rgb(1.0) - rgb(fr_dielectric(wi->z, l.eta_a, l.eta_b)));
            ft = ft * ((ei * ei) / (et * et));
            return ft / abs_cos_theta(*wi);
        }
        case LOBE_MICROFACET_TRANS: {  // reflection.rs:1100-1126
            if (!RRT_LOBE_IN(MASK, LOBE_MICROFACET_TRANS)) break;
            if (wo.z == 0.0) return rgb(0.0);
            const V3 wh = wo.z < 0.0 ? -tr_sample_visible(-wo, l.alpha_x, l.alpha_y, u.x, u.y)
                                     : tr_sample_visible(wo, l.alpha_x, l.alpha_y, u.x, u.y);
            if (dot(wo, wh) < 0.0) return rgb(0.0);
            const double eta = wo.z > 0.0 ? l.eta_a / l.eta_b : l.eta_b / l.eta_a;
            if (!refract_dir(wo, wh, eta, wi)) return rgb(0.0);
            *pdf = lobe_pdf<BIG, MASK>(l, wo, *wi);
            return lobe_f<BIG, MASK>(l, wo, *wi);
        }
        default: {  // FresnelSpecular, reflection.rs:751-797
            if (!RRT_LOBE_IN(MASK, LOBE_FRESNEL_SPEC)) break;
            double fr = fr_dielectric(wo.z, l.eta_a, l.eta_b);
            if (u.x < fr) {
                *wi = v3(-wo.x, -wo.y, wo.z);
                *sampled_type = BXDF_SPECULAR | BXDF_REFLECTION;
                *pdf = fr;
                return l.r * fr / abs_cos_theta(*wi);
            }
            bool entering = wo.z > 0.0;
            double ei = entering ? l.eta_a : l.eta_b, et = entering ? l.eta_b : l.eta_a;
            if (!refract_dir(wo, faceforward(v3(0.0, 0.0, 1.0), wo), ei / et, wi)) return rgb(0.0);
            Rgb ft = l.t * (1.0 - fr);
            ft = ft * ((ei * ei) / (et * et));
            *sampled_type = BXDF_SPECULAR | BXDF_TRANSMISSION;
            *pdf = 1.0 - fr;
            return ft / abs_cos_theta(*wi);
        }
    }
    return rgb(0.0);  // (a lobe kind outside MASK: unreachable)
}
template <bool BIG>
RRT_SHADE_FN Rgb lobe_sample_f_out(const Lobe& l, V3 wo, V3* wi, P2 u, double* pdf, uint32_t* sampled_type) {
    return lobe_sample_f_body<BIG, kLobesAll>(l, wo, wi, u, pdf, sampled_type);
}
template <bool BIG = false, uint32_t MASK = kLobesAll>
__device__ __forceinline__ Rgb lobe_sample_f(const Lobe& l, V3 wo, V3* wi, P2 u, double* pdf, uint32_t* sampled_type) {
    if constexpr (MASK == kLobesAll) return lobe_sample_f_out<BIG>(l, wo, wi, u, pdf, sampled_type);
    else return lobe_sample_f_body<BIG, MASK>(l, wo, wi, u, pdf, sampled_type);
}

// ---- Bsdf over at most NL lobes (reflection.rs:205-404) ---------------------------------------------------
// MASK = the lobe set (above).  A narrowed set walks its lobes with a compile-time bound and static indices (RRT_FOR_LOBES:
// the loop over NL <= 2 slots unrolls), the general one with the run-time count as it always did.
template <int NL, uint32_t MASK = kLobesAll>
struct BsdfT {
    V3 ns, ng, ss, ts;
    double eta;
    int n_lobes;
    bool present;
    Lobe lobes[NL];
};
using Bsdf = BsdfT<2>;
using BsdfBig = BsdfT<8>;  // Bsdf::MAX_BxDFS (reflection.rs:207)
#define RRT_FOR_LOBES(i, b)                                     \
    _Pragma("unroll (MASK != kLobesAll ? NL : 1)")              \
    for (int i = 0; i < (MASK != kLobesAll ? NL : (b).n_lobes); ++i) \
        if (MASK == kLobesAll || i < (b).n_lobes)
template <int NL, uint32_t MASK>
__device__ __forceinline__ V3 to_local(const BsdfT<NL, MASK>& b, V3 v) { return v3(dot(v, b.ss), dot(v, b.ts), dot(v, b.ns)); }
template <int NL, uint32_t MASK>
__device__ __forceinline__ V3 to_world(const BsdfT<NL, MASK>& b, V3 v) {
    return v3(b.ss.x * v.x + b.ts.x * v.y + b.ns.x * v.z, b.ss.y * v.x + b.ts.y * v.y + b.ns.y * v.z,
              b.ss.z * v.x + b.ts.z * v.y + b.ns.z * v.z);
}
template <int NL, uint32_t MASK>
static __device__ int bsdf_num_components(const BsdfT<NL, MASK>& b, uint32_t flags) {
    int n = 0;
    RRT_FOR_LOBES(i, b) n += lobe_matches<(NL > 2), MASK>(b.lobes[i], flags) ? 1 : 0;
    return n;
}
template <int NL, uint32_t MASK>
__device__ __forceinline__ Rgb bsdf_f_body(const BsdfT<NL, MASK>& b, V3 wo_w, V3 wi_w, uint32_t flags) {
    constexpr bool BIG = NL > 2;
    V3 wi = to_local(b, wi_w), wo = to_local(b, wo_w);
    if (wo.z == 0.0) return rgb(0.0);
    bool reflect = dot(wi_w, b.ng) * dot(wo_w, b.ng) > 0.0;
    Rgb f = rgb(0.0);
    RRT_FOR_LOBES(i, b) {
        const Lobe& l = b.lobes[i];
        const uint32_t ty = lobe_type<BIG, MASK>(l);
        if (lobe_matches<BIG, MASK>(l, flags) && ((reflect && (ty & BXDF_REFLECTION)) || (!reflect && (ty & BXDF_TRANSMISSION))))
            f = f + lobe_f<BIG, MASK>(l, wo, wi);
    }
    return f;
}
template <int NL>
RRT_SHADE_FN Rgb bsdf_f_out(const BsdfT<NL, kLobesAll>& b, V3 wo_w, V3 wi_w, uint32_t flags) { return bsdf_f_body(b, wo_w, wi_w, flags); }
template <int NL, uint32_t MASK>
__device__ __forceinline__ Rgb bsdf_f(const BsdfT<NL, MASK>& b, V3 wo_w, V3 wi_w, uint32_t flags) {
    if constexpr (MASK == kLobesAll) return bsdf_f_out(b, wo_w, wi_w, flags);
    else return bsdf_f_body(b, wo_w, wi_w, flags);
}
// Bsdf::pdf (reflection.rs:382-404)
template <int NL, uint32_t MASK>
__device__ __forceinline__ double bsdf_pdf_body(const BsdfT<NL, MASK>& b, V3 wo_w, V3 wi_w, uint32_t flags) {
    constexpr bool BIG = NL > 2;
    if (b.n_lobes == 0) return 0.0;
    V3 wo = to_local(b, wo_w), wi = to_local(b, wi_w);
    if (wo.z == 0.0) return 0.0;
    double pdf = 0.0;
    int matching = 0;
    RRT_FOR_LOBES(i, b)
        if (lobe_matches<BIG, MASK>(b.lobes[i], flags)) {
            matching += 1;
            pdf += lobe_pdf<BIG, MASK>(b.lobes[i], wo, wi);
        }
    return matching > 0 ? pdf / (double)matching : 0.0;
}
template <int NL>
RRT_SHADE_FN double bsdf_pdf_out(const BsdfT<NL, kLobesAll>& b, V3 wo_w, V3 wi_w, uint32_t flags) { return bsdf_pdf_body(b, wo_w, wi_w, flags); }
template <int NL, uint32_t MASK>
__device__ __forceinline__ double bsdf_pdf(const BsdfT<NL, MASK>& b, V3 wo_w, V3 wi_w, uint32_t flags) {
    if constexpr (MASK == kLobesAll) return bsdf_pdf_out(b, wo_w, wi_w, flags);
    else return bsdf_pdf_body(b, wo_w, wi_w, flags);
}
// sampling.rs:233-242
__device__ __forceinline__ V3 uniform_sample_sphere(P2 u) {
    double z = 1.0 - 2.0 * u.x;
    double r = sqrt(rmax(0.0, 1.0 - z * z));
    double phi = 2.0 * kPi * u.y;
    return v3(r * cos(phi), r * sin(phi), z);
}
// sampling.rs:324-328
__device__ __forceinline__ double power_heuristic(int nf, double f_pdf, int ng, double g_pdf) {
    double f = (double)nf * f_pdf, g = (double)ng * g_pdf;
    return (f * f) / (f * f + g * g);
}
// DiffuseAreaLight::sample_li (diffuse.rs:62-79) over Shape::sample_ref (shape/mod.rs:33-48) over Shape::sample
// (sphere.rs:265-284: uniform over the whole sphere; triangle.rs:393-417: "barycentrics" from uniform_sample_sphere,
// Q20).  sample_ref ASSIGNS distance^2 / |cos| to the pdf, dropping Shape::sample's 1 / area (Q28).
RRT_SHADE_FN Rgb area_sample_li(const LightRec& l, V3 ref_p, P2 u, V3* wi, double* pdf, V3* p1) {
    V3 ps, ns;
    if (l.shape_kind == 0) {
        V3 p_obj = v3(0.0, 0.0, 0.0) + uniform_sample_sphere(u) * l.radius;
        ns = normalize_n(xf_normal_inv(l.w2o, p_obj));
        p_obj = p_obj * (l.radius / length(p_obj - v3(0.0, 0.0, 0.0)));
        ps = xf_point(l.o2w, p_obj);
    } else {
        V3 b = uniform_sample_sphere(u);
        ps = l.tp[0] * b.x + l.tp[1] * b.y + l.tp[2] * b.z;
        ns = normalize(cross(l.tp[1] - l.tp[0], l.tp[2] - l.tp[0]));
        if (l.tri_has_n) ns = faceforward(ns, l.tn[0] * b.x + l.tn[1] * b.y + l.tn[2] * b.z);
    }
    V3 w = ps - ref_p;
    const double len_sq = length_sq(w);
    if (len_sq == 0.0) {
        *pdf = 0.0;
    } else {
        w = normalize(w);
        *pdf = len_sq / absdot(-w, ns);
        if (isinf(*pdf)) *pdf = 0.0;
    }
    if (*pdf == 0.0 || length_sq(ps - ref_p) == 0.0) {
        *pdf = 0.0;
        return rgb(0.0);
    }
    *wi = normalize(ps - ref_p);
    *p1 = ps;
    return dot(ns, -*wi) > 0.0 ? l.intensity : rgb(0.0);  // AreaLight::l (diffuse.rs:134-140)
}

template <int NL, uint32_t MASK>
__device__ __forceinline__ Rgb bsdf_sample_f_body(const BsdfT<NL, MASK>& b, V3 wo_w, V3* wi_w, P2 u, double* pdf, uint32_t flags,
                                                  uint32_t* sampled_type) {
    constexpr bool BIG = NL > 2;
    const int matching = bsdf_num_components(b, flags);
    if (matching == 0) {
        *pdf = 0.0;
        *sampled_type = 0;
        return rgb(0.0);
    }
    uint64_t c64 = as_u64(floor(u.x * (double)matching));
    int comp = c64 > (uint64_t)matching ? matching : (int)c64;
    int count = comp, chosen = 0;
    bool searching = true;
    RRT_FOR_LOBES(i, b)
        if (searching && lobe_matches<BIG, MASK>(b.lobes[i], flags)) {
            if (count == 0) {
                chosen = i;
                searching = false;
                if (MASK == kLobesAll) break;
            }
            count -= 1;
        }
    P2 ur = {rmin(u.x * (double)matching - (double)comp, kOneMinusEps), u.y};
    V3 wi = v3(0, 0, 0), wo = to_local(b, wo_w);
    if (wo.z == 0.0) return rgb(0.0);  // NB: *pdf is not touched here either (reflection.rs:343-345)
    *pdf = 0.0;
    Rgb f = rgb(0.0);
    uint32_t chosen_type = 0;
    if constexpr (MASK == kLobesAll) {
        const Lobe& l = b.lobes[chosen];
        chosen_type = lobe_type<BIG, MASK>(l);
        *sampled_type = chosen_type;
        f = lobe_sample_f<BIG, MASK>(l, wo, &wi, ur, pdf, sampled_type);
    } else {  // static lobe indices: each slot's code is the one lobe kind that slot can hold
#pragma unroll
        for (int i = 0; i < NL; ++i)
            if (i == chosen) {
                chosen_type = lobe_type<BIG, MASK>(b.lobes[i]);
                *sampled_type = chosen_type;
                f = lobe_sample_f<BIG, MASK>(b.lobes[i], wo, &wi, ur, pdf, sampled_type);
            }
    }
    if (*pdf == 0.0) {
        *sampled_type = 0;
        return rgb(0.0);
    }
    *wi_w = to_world(b, wi);
    if (!(chosen_type & BXDF_REFLECTION) && matching > 1) {
        RRT_FOR_LOBES(i, b)
            if (i != chosen && lobe_matches<BIG, MASK>(b.lobes[i], flags)) *pdf += lobe_pdf<BIG, MASK>(b.lobes[i], wo, wi);
    }
    if (matching > 1) *pdf /= (double)matching;
    return f;  // Q15: the multi-lobe re-evaluation is computed into a shadowed variable and dropped
}
template <int NL>
RRT_SHADE_FN Rgb bsdf_sample_f_out(const BsdfT<NL, kLobesAll>& b, V3 wo_w, V3* wi_w, P2 u, double* pdf, uint32_t flags, uint32_t* sampled_type) {
    return bsdf_sample_f_body(b, wo_w, wi_w, u, pdf, flags, sampled_type);
}
template <int NL, uint32_t MASK>
__device__ __forceinline__ Rgb bsdf_sample_f(const BsdfT<NL, MASK>& b, V3 wo_w, V3* wi_w, P2 u, double* pdf, uint32_t flags, uint32_t* sampled_type) {
    if constexpr (MASK == kLobesAll) return bsdf_sample_f_out(b, wo_w, wi_w, u, pdf, flags, sampled_type);
    else return bsdf_sample_f_body(b, wo_w, wi_w, u, pdf, flags, sampled_type);
}

// Material::bump (material/mod.rs:22-65): the shading frame after displacement by the material's bump map.  Literal:
// du = |dudx| * 0.5 + |dudy| (the 0.5 binds to the first term only), dv = (|dvdx| + |dvdy|) * 0.5; 0.0005 without
// differentials.  The shifted evaluations move p along shading.dpdu / dpdv and uv by (du, 0) / (0, dv).
static __device__ __noinline__ void material_bump(const ShadeScene& sc, const MaterialRec& m, const RayDiffRec* diff, Surface* s,
                                                  const BumpPartials& bp) {
    Rgb vals[kMaxTextures];
    TexPoint q = tex_point(s->uv, s->p);
    if (diff) compute_differentials(s->n, s->dpdu, s->dpdv, *diff, &q);
    const int32_t b = m.tex[11];
    double du = add(mul(fabs(q.dudx), 0.5), fabs(q.dudy));
    if (du == 0.0) du = 0.0005;
    TexPoint e = q;
    e.p = s->p + s->shdpdu * du;
    e.uv = P2{add(s->uv.x, du), add(s->uv.y, 0.0)};
    texture_eval_table(sc.textures, sc.n_textures, m.bump_needed, e, vals, sc.mips);
    const double u_displace = vals[b].r;
    double dv = mul(add(fabs(q.dvdx), fabs(q.dvdy)), 0.5);
    if (dv == 0.0) dv = 0.0005;
    e.p = s->p + bp.shdpdv * dv;
    e.uv = P2{add(s->uv.x, 0.0), add(s->uv.y, dv)};
    texture_eval_table(sc.textures, sc.n_textures, m.bump_needed, e, vals, sc.mips);
    const double v_displace = vals[b].r;
    texture_eval_table(sc.textures, sc.n_textures, m.bump_needed, q, vals, sc.mips);
    const double displace = vals[b].r;
    const V3 dpdu = s->shdpdu + (s->shn * sub(u_displace, displace)) / du + bp.shdndu * displace;
    const V3 dpdv = bp.shdpdv + (s->shn * sub(v_displace, displace)) / dv + bp.shdndv * displace;
    // set_shading_geometry(dpdu, dpdv, .., orientation_is_authoritative = false) (interaction.rs:186-202)
    s->shn = faceforward(normalize(cross(dpdu, dpdv)), s->n);
    s->shdpdu = dpdu;
}

// The material with every textured parameter evaluated at the hit (each compute_scattering_functions starts with
// Texture::evaluate(si), material/*.rs; si.compute_differentials ran just before, interaction.rs:203-214).  Only
// called for materials with `needed != 0`.  `diff` = the camera ray's differentials at a path's first hit, or null.
static __device__ __noinline__ void material_at(const ShadeScene& sc, const MaterialRec& m, const Surface& s, const RayDiffRec* diff,
                                                MaterialRec* out) {
    Rgb vals[kMaxTextures];
    TexPoint q = tex_point(s.uv, s.p);
    if (diff) compute_differentials(s.n, s.dpdu, s.dpdv, *diff, &q);
    texture_eval_table(sc.textures, sc.n_textures, m.needed, q, vals, sc.mips);
    MaterialRec r = m;
    Rgb* const colours[6] = {&r.kd, &r.ks, &r.kr, &r.kt, &r.metal_eta, &r.metal_k};
#pragma unroll
    for (int k = 0; k < 6; ++k)
        if (m.tex[k] >= 0) *colours[k] = vals[m.tex[k]];
    double* const scalars[5] = {&r.sigma, &r.roughness, &r.u_roughness, &r.v_roughness, &r.eta};
#pragma unroll
    for (int k = 0; k < 5; ++k)
        if (m.tex[6 + k] >= 0) *scalars[k] = vals[m.tex[6 + k]].r;
    *out = r;
}

// material_at for the NL = 8 kernels: DisneyMaterial's own parameters too (disney.rs:538-551 evaluates every texture)
static __device__ __noinline__ void material_at_big(const ShadeScene& sc, const MaterialRec& m, const Surface& s, const RayDiffRec* diff,
                                                    MaterialRec* out, DisneyRec* dz) {
    Rgb vals[kMaxTextures];
    TexPoint q = tex_point(s.uv, s.p);
    if (diff) compute_differentials(s.n, s.dpdu, s.dpdv, *diff, &q);
    texture_eval_table(sc.textures, sc.n_textures, m.needed, q, vals, sc.mips);
    MaterialRec r = m;
    Rgb* const colours[6] = {&r.kd, &r.ks, &r.kr, &r.kt, &r.metal_eta, &r.metal_k};
    for (int k = 0; k < 6; ++k)
        if (m.tex[k] >= 0) *colours[k] = vals[m.tex[k]];
    double* const scalars[5] = {&r.sigma, &r.roughness, &r.u_roughness, &r.v_roughness, &r.eta};
    for (int k = 0; k < 5; ++k)
        if (m.tex[6 + k] >= 0) *scalars[k] = vals[m.tex[6 + k]].r;
    *out = r;
    for (int k = 0; k < 10; ++k)
        if (dz->tex[k] >= 0) dz->v[k] = vals[dz->tex[k]].r;
}

// Material::compute_scattering_functions once the parameters are values.  `dz`: the material's DisneyRec (NL = 8 only).
// KIND >= 0: the caller knows every hit it shades carries a material of that kind (0 Matte, 1 Plastic, 2 Metal).
template <int KIND, int NL, uint32_t MASK>
__device__ __forceinline__ void make_bsdf_body(const MaterialRec& m, const Surface& s, bool allow_multiple_lobes, BsdfT<NL, MASK>* b,
                                               const DisneyRec* dz) {
    b->ns = s.shn;
    b->ss = normalize(s.shdpdu);
    b->ng = s.n;
    b->ts = cross(b->ns, b->ss);
    b->eta = 1.0;
    b->n_lobes = 0;
    b->present = true;
    Lobe l;
    l.fresnel = FRESNEL_NOOP;
    l.r = rgb(0.0);
    l.t = rgb(0.0);
    l.cond_eta = rgb(0.0);
    l.cond_k = rgb(0.0);
    l.a = l.b = 1.0;
    l.eta_a = l.eta_b = 1.0;
    l.alpha_x = l.alpha_y = 0.0;
    if (NL > 2 && m.kind >= 5) {
        if (m.kind == 5) {  // TranslucentMaterial (translucent.rs:51-107): reflect = kr, transmit = kt
            const double eta = 1.5;
            b->eta = eta;
            const Rgb r = clamp_rgb(m.kr, 0.0, kInfD), t = clamp_rgb(m.kt, 0.0, kInfD);
            if (is_black(r) && is_black(t)) {
                b->present = false;
                return;
            }
            const Rgb kd = clamp_rgb(m.kd, 0.0, kInfD);
            if (!is_black(kd)) {
                if (!is_black(r)) {
                    l.kind = LOBE_LAMBERT;
                    l.r = r * kd;
                    b->lobes[b->n_lobes++] = l;
                }
                if (!is_black(t)) {
                    l.kind = LOBE_LAMBERT_TRANS;
                    l.r = rgb(0.0);
                    l.t = t * kd;
                    b->lobes[b->n_lobes++] = l;
                }
            }
            const Rgb ks = clamp_rgb(m.ks, 0.0, kInfD);
            if (!is_black(ks) && (!is_black(r) || !is_black(t))) {
                double rough = m.roughness;
                if (m.remap_roughness) rough = roughness_to_alpha(rough);
                l.alpha_x = l.alpha_y = rough;
                if (!is_black(r)) {
                    l.kind = LOBE_MICROFACET;
                    l.r = r * ks;
                    l.t = rgb(0.0);
                    l.fresnel = FRESNEL_DIELECTRIC;
                    l.a = 1.0;
                    l.b = eta;
                    b->lobes[b->n_lobes++] = l;
                }
                if (!is_black(t)) {
                    l.kind = LOBE_MICROFACET_TRANS;
                    l.fresnel = FRESNEL_NOOP;
                    l.r = rgb(0.0);
                    l.t = t * ks;
                    l.eta_a = 1.0;
                    l.eta_b = eta;
                    b->lobes[b->n_lobes++] = l;
                }
            }
            return;
        }
        if (m.kind == 7) {  // DebugMaterial (debug_material.rs:37-50)
            l.kind = LOBE_DEBUG_DIFFUSE;
            b->lobes[b->n_lobes++] = l;
            l.kind = LOBE_DEBUG_SPECULAR;
            b->lobes[b->n_lobes++] = l;
            return;
        }
        // DisneyMaterial (disney.rs:524-680); a BSSRDF-producing record was refused when the scene was set up
        const Rgb c = clamp_rgb(m.kd, 0.0, kInfD);
        const double metallic_weight = dz->v[DZ_METALLIC], e = m.eta, strans = dz->v[DZ_SPEC_TRANS];
        const double diffuse_weight = (1.0 - metallic_weight) * (1.0 - strans);
        const double dt = dz->v[DZ_DIFF_TRANS], rough = m.roughness;
        const double luminance = lum(c);
        const Rgb c_tint = luminance > 0.0 ? c / luminance : rgb(1.0);
        const double sheen_weight = dz->v[DZ_SHEEN];
        Rgb c_sheen = rgb(0.0);
        if (sheen_weight > 0.0) c_sheen = lerp_rgb(dz->v[DZ_SHEEN_TINT], rgb(1.0), c_tint);
        if (diffuse_weight > 0.0) {
            if (dz->thin) {
                const double flat = dz->v[DZ_FLATNESS];
                l.kind = LOBE_DISNEY_DIFFUSE;
                l.r = c * diffuse_weight * (1.0 - flat) * (1.0 - dt);
                b->lobes[b->n_lobes++] = l;
                l.kind = LOBE_DISNEY_FAKESS;
                l.r = c * diffuse_weight * flat * (1.0 - dt);
                l.eta_a = rough;
                b->lobes[b->n_lobes++] = l;
            } else {
                l.kind = LOBE_DISNEY_DIFFUSE;
                l.r = c * diffuse_weight;
                b->lobes[b->n_lobes++] = l;
            }
            l.kind = LOBE_DISNEY_RETRO;
            l.r = c * diffuse_weight;
            l.eta_a = rough;
            b->lobes[b->n_lobes++] = l;
            if (sheen_weight > 0.0) {
                l.kind = LOBE_DISNEY_SHEEN;
                l.r = c_sheen * sheen_weight * diffuse_weight;
                b->lobes[b->n_lobes++] = l;
            }
        }
        const double aspect = sqrt(1.0 - dz->v[DZ_ANISOTROPIC] * 0.9);
        const double ax = rmax((rough * rough) / aspect, 0.001), ay = rmax((rough * rough) * aspect, 0.001);
        const double q0 = (e - 1.0) / (e + 1.0);  // schlick_r0_from_eta (reflection.rs:28-30)
        const Rgb c_spec_0 = lerp_rgb(metallic_weight, lerp_rgb(dz->v[DZ_SPECULAR_TINT], rgb(1.0), c_tint) * (q0 * q0), c);
        l.kind = LOBE_MICROFACET;
        l.r = rgb(1.0);
        l.alpha_x = ax;
        l.alpha_y = ay;
        l.fresnel = FRESNEL_DISNEY | FRESNEL_SEPARABLE_G;
        l.cond_eta = c_spec_0;
        l.a = metallic_weight;
        l.b = e;
        l.eta_a = l.eta_b = 1.0;
        b->lobes[b->n_lobes++] = l;
        l.fresnel = FRESNEL_NOOP;
        l.cond_eta = rgb(0.0);
        l.a = l.b = 1.0;
        const double cc = dz->v[DZ_CLEARCOAT];
        if (cc > 0.0) {
            l.kind = LOBE_DISNEY_CLEARCOAT;
            l.r = rgb(0.0);
            l.eta_a = cc;
            l.eta_b = lerp_f(dz->v[DZ_CLEARCOAT_GLOSS], 0.1, 0.001);
            b->lobes[b->n_lobes++] = l;
        }
        if (strans > 0.0) {
            l.kind = LOBE_MICROFACET_TRANS;
            l.r = rgb(0.0);
            l.t = sqrt_rgb(c) * strans;
            l.eta_a = 1.0;
            l.eta_b = e;
            if (dz->thin) {  // a plain TrowbridgeReitzDistribution over the IOR-scaled roughness (Burley 2015, figure 15)
                const double r_scaled = (0.65 * e - 0.35) * rough;
                l.alpha_x = rmax((r_scaled * r_scaled) / aspect, 0.001);
                l.alpha_y = rmax((r_scaled * r_scaled) * aspect, 0.001);
            } else {
                l.fresnel = FRESNEL_SEPARABLE_G;
            }
            b->lobes[b->n_lobes++] = l;
            l.fresnel = FRESNEL_NOOP;
        }
        if (dz->thin) {
            l.kind = LOBE_LAMBERT_TRANS;
            l.r = rgb(0.0);
            l.t = c * dt;
            b->lobes[b->n_lobes++] = l;
        }
        return;
    }
    switch (KIND >= 0 ? (uint32_t)KIND : m.kind) {
        case 0: {  // MatteMaterial (matte.rs:36-61)
            Rgb r = clamp_rgb(m.kd, 0.0, kInfD);
            double sig = clampd(m.sigma, 0.0, 90.0);
            if (!is_black(r)) {
                l.r = r;
                if (sig == 0.0) {
                    l.kind = LOBE_LAMBERT;
                } else {
                    l.kind = LOBE_OREN_NAYAR;  // reflection.rs:906-912: A, B kept in eta_a / eta_b
                    double sr = (kPi / 180.0) * sig;
                    double sigma2 = sr * sr;
                    l.eta_a = 1.0 - (sigma2 / (2.0 * (sigma2 + 0.33)));
                    l.eta_b = 0.45 * sigma2 / (sigma2 + 0.09);
                }
                b->lobes[b->n_lobes++] = l;
            }
            return;
        }
        case 1: {  // PlasticMaterial (plastic.rs:42-73), Q16
            Rgb kd = clamp_rgb(m.kd, 0.0, kInfD), ks = clamp_rgb(m.ks, 0.0, kInfD);
            if (!is_black(kd)) {
                l.kind = LOBE_LAMBERT;
                l.r = kd;
                b->lobes[b->n_lobes++] = l;
                double rough = m.roughness;
                if (m.remap_roughness) rough = roughness_to_alpha(rough);
                l.kind = LOBE_MICROFACET;
                l.r = ks;
                l.alpha_x = l.alpha_y = rough;
                l.fresnel = FRESNEL_DIELECTRIC;
                l.a = 1.5;
                l.b = 1.0;
                b->lobes[b->n_lobes++] = l;
            }
            return;
        }
        case 2: {  // MetalMaterial (metal.rs:48-90)
            double ur = m.u_roughness >= 0.0 ? m.u_roughness : m.roughness;
            double vr = m.v_roughness >= 0.0 ? m.v_roughness : m.roughness;
            if (m.remap_roughness) {
                ur = roughness_to_alpha(ur);
                vr = roughness_to_alpha(vr);
            }
            l.kind = LOBE_MICROFACET;
            l.r = rgb(1.0);
            l.alpha_x = ur;
            l.alpha_y = vr;
            l.fresnel = FRESNEL_CONDUCTOR;
            l.cond_eta = m.metal_eta;
            l.cond_k = m.metal_k;
            b->lobes[b->n_lobes++] = l;
            return;
        }
        case 3: {  // MirrorMaterial (mirror.rs:28-48)
            Rgb r = clamp_rgb(m.kr, 0.0, kInfD);
            if (!is_black(r)) {
                l.kind = LOBE_SPEC_REFL;
                l.r = r;
                b->lobes[b->n_lobes++] = l;
            }
            return;
        }
        default: {  // GlassMaterial (glass.rs:52-113)
            Rgb r = clamp_rgb(m.kr, 0.0, kInfD), t = clamp_rgb(m.kt, 0.0, kInfD);
            double ur = rmax(m.u_roughness, 0.0), vr = rmax(m.v_roughness, 0.0);
            b->eta = m.eta;
            if (is_black(r) && is_black(t)) {
                b->present = false;
                return;
            }
            const bool is_specular = ur == 0.0 && vr == 0.0;
            if (is_specular && allow_multiple_lobes) {
                l.kind = LOBE_FRESNEL_SPEC;
                l.r = r;
                l.t = t;
                l.eta_a = 1.0;
                l.eta_b = m.eta;
                b->lobes[b->n_lobes++] = l;
                return;
            }
            if (m.remap_roughness) {
                ur = roughness_to_alpha(ur);
                vr = roughness_to_alpha(vr);
            }
            l.alpha_x = ur;  // TrowbridgeReitzDistribution::new(u_rough, v_rough, true) for both rough lobes
            l.alpha_y = vr;
            if (!is_black(r)) {
                l.kind = is_specular ? LOBE_SPEC_REFL : LOBE_MICROFACET;
                l.r = r;
                l.fresnel = FRESNEL_DIELECTRIC;
                l.a = 1.0;
                l.b = m.eta;
                b->lobes[b->n_lobes++] = l;
            }
            if (!is_black(t)) {
                l.kind = is_specular ? LOBE_SPEC_TRANS : LOBE_MICROFACET_TRANS;
                l.fresnel = FRESNEL_NOOP;
                l.r = rgb(0.0);
                l.t = t;
                l.eta_a = 1.0;
                l.eta_b = m.eta;
                b->lobes[b->n_lobes++] = l;
            }
            return;
        }
    }
}
template <int NL>
RRT_SHADE_FN void make_bsdf_out(const MaterialRec& m, const Surface& s, bool allow_multiple_lobes, BsdfT<NL, kLobesAll>* b, const DisneyRec* dz) {
    make_bsdf_body<-1>(m, s, allow_multiple_lobes, b, dz);
}
template <int KIND = -1, int NL, uint32_t MASK>
__device__ __forceinline__ void make_bsdf(const MaterialRec& m, const Surface& s, bool allow_multiple_lobes, BsdfT<NL, MASK>* b,
                                          const DisneyRec* dz = nullptr) {
    if constexpr (MASK == kLobesAll) make_bsdf_out(m, s, allow_multiple_lobes, b, dz);
    else make_bsdf_body<KIND>(m, s, allow_multiple_lobes, b, dz);
}

}  // namespace rrt
