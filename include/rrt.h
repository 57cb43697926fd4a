/* rrt.h — C ABI of librrt_sm100.so, the B200 (sm_100a) ray-intersection and path-tracing core
 * that stands behind rs_ray_toy's aggregate seam.
 *
 * Every entry point names the reference interface it replaces (file:line under
 * pppKin/rs_ray_toy `src/`).  Plain pointers and sizes only; no C++ / torch / Rust types.
 * All functions return RRT_OK (0) or a negative rrt_status; rrt_last_error() gives the text of
 * the last failure on the calling thread.  No exception or panic crosses this boundary
 * (the reference reports the same conditions with assert!/panic!, e.g. bvh.rs:319, scene.rs:70).
 *
 * Threading: an rrt_scene is immutable after rrt_scene_commit(); intersect / render calls on it
 * are stream-ordered and may be issued from several host threads (the reference's
 * `Primitive: Send + Sync`, primitives.rs:14).
 */
#ifndef RRT_H_
#define RRT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum rrt_status {
    RRT_OK = 0,
    RRT_ERR_INVALID = -1,     /* bad argument / call order                                      */
    RRT_ERR_CUDA = -2,        /* CUDA runtime failure (text in rrt_last_error)                  */
    RRT_ERR_UNSUPPORTED = -3, /* reference feature outside the hot-path scope (DESIGN.md)       */
    RRT_ERR_EMPTY = -4,       /* BVHAccel::new on zero primitives (bvh.rs:319 asserts)          */
    RRT_ERR_IO = -5           /* scene.json / .obj could not be read or parsed                  */
} rrt_status;

typedef struct rrt_ctx rrt_ctx;     /* one per CUDA device                                       */
typedef struct rrt_scene rrt_scene; /* the GPU aggregate: replaces BVHAccel behind Arc<dyn Primitive> */

/* geometry.rs:73-79 `Ray{o,d,t_max,time,medium}` — f64 like the reference; `medium` is out of
 * scope.  d is used as given (the aggregate never renormalises it, bvh.rs:186).  64 bytes.      */
typedef struct rrt_ray {
    double o[3];
    double d[3];
    double t_max;
    double time;
} rrt_ray;

/* What BVHAccel::intersect hands back through `r.t_max` and `si` (bvh.rs:183-236,
 * primitives.rs:56-57): the primitive that won, its hit distance and surface parameters.
 * prim_id indexes the primitive list in the order it was added (= the Vec passed to
 * BVHAccel::new, renderprocess.rs:1299); RRT_NO_HIT when the ray escaped.
 * (u,v): triangle barycentrics of triangle.rs:245-256, or the sphere's (phi/phi_max, theta
 * fraction) of sphere.rs:195-198.  32 bytes.                                                    */
#define RRT_NO_HIT 0xFFFFFFFFu
typedef struct rrt_hit {
    uint32_t prim_id;
    uint32_t reserved;
    double t;
    double u;
    double v;
} rrt_hit;

/* Compact records for callers that hold their rays in fp32 (rrt_intersect_f32 and relatives below).  The aggregate
 * still decides in f64: every float is promoted exactly to double on the device (`time` = 0, which the aggregate never
 * reads: its transforms are static), the f64 walk runs unchanged, and each f64 result field is rounded to nearest
 * (__double2float_rn) on the way out.  So a call on rrt_ray_f32 records returns bit for bit the rrt_intersect answer
 * on the promoted rays, rounded.  t_max may be +inf.  32 bytes: two 16-byte loads per ray.                         */
typedef struct rrt_ray_f32 {
    float o[3];
    float t_max;
    float d[3];
    uint32_t reserved; /* ignored */
} rrt_ray_f32;
/* rrt_hit with t, u, v rounded to nearest fp32; prim_id copied unchanged (RRT_NO_HIT on a miss, when t, u, v are the
 * rounded values the f64 record carries).  16 bytes.                                                            */
typedef struct rrt_hit_f32 {
    uint32_t prim_id;
    float t;
    float u;
    float v;
} rrt_hit_f32;

/* BVHSplitMethod (bvh.rs:111-114) plus the parity tier (SURVEY.md §8c).                         */
typedef enum rrt_build_flags {
    RRT_BUILD_FAST = 0,    /* Tier F: own SAH tree, true closest hit, ties -> lowest prim id     */
    RRT_BUILD_LITERAL = 1, /* Tier L: the reference's HLBVH topology, visiting order and accept rules
                              with every quirk kept (last accepted hit wins, ...): bit-for-bit what
                              BVHAccel returns; one thread per ray, meant for parity not throughput */
    RRT_BUILD_DEVICE_LBVH = 2 /* Tier F with the tree built ON the GPU: Morton keys, radix sort, binary radix
                              tree, bottom-up boxes (the device counterpart of hlbvh_build's Morton half,
                              bvh.rs:365-612).  Milliseconds instead of a host SAH build; same answers (Tier-F
                              results do not depend on topology), a tree 2-5% slower to walk              */
} rrt_build_flags;

/* ---- context ----------------------------------------------------------------------------- */
int rrt_create(int device_ordinal, rrt_ctx** out);
void rrt_destroy(rrt_ctx* ctx);
const char* rrt_last_error(void);
/* Number of kernels launched by this library on `ctx` since creation (bench.py's gpu_launches). */
uint64_t rrt_launch_count(const rrt_ctx* ctx);
/* Pinned host memory for ray / hit batches (cudaHostAlloc); plain malloc'd buffers also work.   */
int rrt_host_alloc(rrt_ctx* ctx, size_t bytes, void** out);
int rrt_host_free(rrt_ctx* ctx, void* p);

/* ---- scene assembly: what make_aggregate builds (renderprocess.rs:1178-1304) --------------- */
int rrt_scene_begin(rrt_ctx* ctx, rrt_scene** out);
void rrt_scene_destroy(rrt_scene* scene);

/* create_triangle_mesh (shape/triangle.rs:131-165): vertex positions p[3*nv] (f64), 0-based
 * vertex indices vi[3*ntri]; optional normals n[3*nn] with ni[3*ntri], optional uv[2*nuv] with
 * uvi[3*ntri] (null when absent).  The obj-level transform is NOT applied to vertices, exactly
 * like the reference (Q7, renderprocess.rs:884-903).  Returns the mesh handle in *mesh_id.     */
int rrt_scene_add_mesh(rrt_scene* scene, uint32_t nv, const double* p, uint32_t ntri, const uint32_t* vi,
                       uint32_t nn, const double* n, const uint32_t* ni, uint32_t nuv, const double* uv,
                       const uint32_t* uvi, uint32_t* mesh_id);

/* One GeometricPrimitive per mesh triangle (renderprocess.rs:1255-1263), appended to the
 * primitive list once per instance transform (TransformedPrimitive, primitives.rs:27-30) or
 * once bare when n_instances == 0.  instance_m / instance_minv: n_instances 4x4 row-major
 * matrices and their inverses (Transform carries both, transform.rs:177-180).                  */
int rrt_scene_add_triangles(rrt_scene* scene, uint32_t mesh_id, uint32_t material_id, uint32_t n_instances,
                            const double* instance_m, const double* instance_minv);

/* Sphere::new (shape/sphere.rs:28-47) wrapped in a GeometricPrimitive, appended bare or once per
 * instance like the triangles above (renderprocess.rs:1187-1227).                              */
int rrt_scene_add_sphere(rrt_scene* scene, const double* obj_to_world_m, const double* obj_to_world_minv,
                         double radius, double z_min, double z_max, double phi_max_deg, uint32_t material_id,
                         uint32_t n_instances, const double* instance_m, const double* instance_minv);

/* BVHAccel::new(prims, max_prims_in_node, split_method) (bvh.rs:307-363): host build, flatten to
 * the linear SoA layout, upload to HBM.                                                         */
int rrt_scene_commit(rrt_scene* scene, uint32_t max_prims_in_node, uint32_t build_flags);
/* Dynamic scenes (SURVEY §8f row 1, "refit for instance updates"): replaces the transforms of instances
 * [first_instance, first_instance + n) — numbered in the order the rrt_scene_add_* calls appended them — and brings the
 * aggregate up to date: the moved primitives are re-baked to world space and the tree is made anew ON the device
 * (Morton keys, radix sort, radix tree, bottom-up boxes: milliseconds).  Fast tier; integrators made over the scene
 * must be destroyed first, since they hold its tables.                                                              */
int rrt_scene_update_instances(rrt_scene* scene, uint32_t first_instance, uint32_t n, const double* instance_m,
                               const double* instance_minv);
int rrt_scene_num_prims(const rrt_scene* scene, uint32_t* out);
/* Primitive::world_bound (bvh.rs:177-182): out6 = p_min, p_max.                                 */
int rrt_world_bound(const rrt_scene* scene, double out6[6]);
/* The committed aggregate — tree, primitive records, instance tables — as one relocatable blob, so that ONE rank builds
 * and the others replicate (SURVEY §5: "scene replicated per GPU"): rrt_scene_export_tree with buffer = NULL returns the
 * size; rrt_scene_commit_from_tree commits a scene that received the SAME rrt_scene_add_* calls without building a tree
 * of its own (the blob's primitive count is checked).  Fast tier only.                                             */
int rrt_scene_export_tree(const rrt_scene* scene, void* buffer, uint64_t capacity, uint64_t* bytes);
int rrt_scene_commit_from_tree(rrt_scene* scene, const void* blob, uint64_t bytes);
/* Build statistics: nodes, leaves, max depth, bytes uploaded, host build seconds (x1e6).        */
int rrt_scene_stats(const rrt_scene* scene, uint64_t out8[8]);

/* How the tree was built: out4 = { microseconds the GPU spent building it (0 for a host build), bytes per
 * interior node (32 or 64), 1 if built on the device, reserved }.                                            */
int rrt_scene_build_info(const rrt_scene* scene, uint64_t out4[4]);

/* ---- the hot path ------------------------------------------------------------------------- */
/* Scene::intersect -> BVHAccel::intersect (scene.rs:69-72, bvh.rs:183-236) over a batch.
 * rays / hits are DEVICE pointers; the call is asynchronous on `cuda_stream` (a cudaStream_t,
 * 0 = default stream).                                                                          */
int rrt_intersect_device(const rrt_scene* scene, uint64_t n, const rrt_ray* d_rays, rrt_hit* d_hits,
                         void* cuda_stream);
/* Scene::intersect_p -> BVHAccel::intersect_p (scene.rs:75-80, bvh.rs:123-174): occluded[i] = 1
 * when any primitive is hit within (0, t_max].                                                  */
int rrt_intersect_p_device(const rrt_scene* scene, uint64_t n, const rrt_ray* d_rays, uint8_t* d_occluded,
                           void* cuda_stream);
/* Same two calls with HOST buffers: chunked, double-buffered H2D -> kernel -> D2H; returns when
 * `hits` / `occluded` are complete.  This is the call a Rust `impl Primitive for GpuAggregate`
 * binds (INTEGRATION.md).                                                                       */
int rrt_intersect(const rrt_scene* scene, uint64_t n, const rrt_ray* rays, rrt_hit* hits);
int rrt_intersect_p(const rrt_scene* scene, uint64_t n, const rrt_ray* rays, uint8_t* occluded);

/* The same four calls on fp32 rays (rrt_ray_f32, 32 B) and compact hits (rrt_hit_f32, 16 B): Scene::intersect /
 * intersect_p (scene.rs:69-80, bvh.rs:123-236) for callers whose rays are fp32 already, at half the link bytes per
 * ray up and down.  Errors, limits and threading are those of the f64 call each one mirrors.
 * Host buffers: the same chunked pipeline as rrt_intersect; the first fp32 call on a context adds one staging buffer
 * of 32 MiB to each of its four pipeline slots (128 MiB of device memory, kept until rrt_destroy).                   */
int rrt_intersect_f32(const rrt_scene* scene, uint64_t n, const rrt_ray_f32* rays, rrt_hit_f32* hits);
int rrt_intersect_p_f32(const rrt_scene* scene, uint64_t n, const rrt_ray_f32* rays, uint8_t* occluded);
/* Device buffers, asynchronous on `cuda_stream`.  The promoted f64 rays and the f64 hits live in scratch memory the
 * scene keeps per calling stream: 96 bytes per ray for rrt_intersect_f32_device, 64 for rrt_intersect_p_f32_device,
 * grown to the largest batch seen on that stream and freed by rrt_scene_destroy.  Past eight streams the scratch of
 * the first one is shared, each call ordered after the last one that used it (as the tree walk's own workspaces).  */
int rrt_intersect_f32_device(const rrt_scene* scene, uint64_t n, const rrt_ray_f32* d_rays, rrt_hit_f32* d_hits,
                             void* cuda_stream);
int rrt_intersect_p_f32_device(const rrt_scene* scene, uint64_t n, const rrt_ray_f32* d_rays, uint8_t* d_occluded,
                               void* cuda_stream);

/* ---- the render loop ------------------------------------------------------------------------
 * What deploy_render builds and runs (renderprocess.rs:92-105): make_scene + make_integrator,
 * then Integrator::render -> SamplerIntegrator::si_render (integrator/mod.rs:48-139), executed
 * as a wavefront of generate / extend / shade / shadow / accumulate kernels.                    */

/* Material::compute_scattering_functions inputs with constant-valued textures
 * (material/{matte,plastic,metal,mirror,glass,translucent,disney,debug_material}.rs; make_materials,
 * renderprocess.rs:664-871).  MixMaterial has no record: the reference panics while loading one (Q25).            */
typedef enum rrt_material_kind {
    RRT_MAT_MATTE = 0, RRT_MAT_PLASTIC = 1, RRT_MAT_METAL = 2, RRT_MAT_MIRROR = 3, RRT_MAT_GLASS = 4,
    RRT_MAT_TRANSLUCENT = 5, /* translucent.rs: kd, ks, roughness; reflect = kr, transmit = kt; up to four lobes     */
    RRT_MAT_DISNEY = 6,      /* disney.rs: color = kd, roughness, eta and the Disney block below; up to eight lobes.
                              * thin = 0 with a non-black scatter_distance asks for the BSSRDF: refused             */
    RRT_MAT_DEBUG = 7        /* debug_material.rs: no parameters                                                    */
} rrt_material_kind;
typedef struct rrt_material {
    uint32_t kind;
    uint32_t remap_roughness;
    double kd[3], ks[3], kr[3], kt[3];
    double metal_eta[3], metal_k[3];  /* FresnelConductor eta / k (default: copper)             */
    double sigma;                     /* Matte: Oren-Nayar sigma in degrees                     */
    double roughness;                 /* Plastic / Metal                                        */
    double u_roughness, v_roughness;  /* Metal: < 0 = None (use roughness); Glass: values; non-zero = rough
                                       * glass, MicrofacetReflection + MicrofacetTransmission (glass.rs:77-108) */
    double eta;                       /* Glass / Disney index                                   */
    /* DisneyMaterial (disney.rs:464-483; the loader's defaults, renderprocess.rs:810-836, are 0 but for
     * sheen_tint 0.5, clearcoat_gloss 1, diff_trans 1, roughness 0.5, eta 1.5, color 0.5)                          */
    double metallic, specular_tint, anisotropic, sheen, sheen_tint, clearcoat, clearcoat_gloss, spec_trans,
           flatness, diff_trans;
    double scatter_distance[3];
    uint32_t thin, pad;
} rrt_material;

/* Textures a material parameter can name (make_textures, renderprocess.rs:298-515): the scene's float and rgb
 * textures flattened into ONE table in definition order (float textures first).  A texture can only name textures
 * defined before it (the loader looks names up in the maps it is filling; an unknown name becomes a constant,
 * get_text_fallback :282-296), so children always have smaller indices.  Float textures use v[.][0].
 * texture/{bilerp,mix,scale,checkerboard,uv,windy,wrinkled}.rs; mappings texture/mod.rs:206-347 with their screen-space
 * differentials: the renderer carries the camera ray's differentials (RealisticCamera::generate_ray_differential,
 * camera.rs:582-628, scaled by 1/sqrt(spp), integrator/mod.rs:92-94) to the first hit and runs
 * SurfaceInteraction::compute_differentials (interaction.rs:223-284) there when a texture asks for them (a
 * closed-form checkerboard, a noise texture); every later hit has none, like the reference's spawned rays.               */
typedef enum rrt_texture_kind {
    RRT_TEX_CONSTANT = 0, RRT_TEX_BILERP = 1, RRT_TEX_SCALE = 2, RRT_TEX_MIX = 3, RRT_TEX_CHECKER2D = 4,
    RRT_TEX_CHECKER3D = 5, RRT_TEX_UV = 6,
    RRT_TEX_WINDY = 7,    /* windy.rs: |fbm(0.1 p, 3 octaves)| * fbm(p, 6 octaves) over Perlin noise (texture/mod.rs:75-155) */
    RRT_TEX_WRINKLED = 8, /* wrinkled.rs: turbulence(p, omega = map[1], octaves = map[0]) (texture/mod.rs:157-188)     */
    RRT_TEX_IMAGE = 9     /* imagemap.rs + mipmap.rs: an rgb texture over an image added with rrt_scene_add_image*: t1 = the
                           * image's index, aa = do_trilinear, v[0][0] = max_aniso (default 8), v[0][1] = wrap (rrt_image_wrap);
                           * EWA or trilinear MIPMap lookups exactly as the reference runs them (csrc/mipmap_core.h: Q31, Q32) */
} rrt_texture_kind;
typedef enum rrt_image_wrap { RRT_WRAP_REPEAT = 0, RRT_WRAP_BLACK = 1, RRT_WRAP_CLAMP = 2 } rrt_image_wrap;
typedef enum rrt_texture_mapping {
    RRT_TEXMAP_UV = 0, RRT_TEXMAP_PLANAR = 1, RRT_TEXMAP_SPHERICAL = 2, RRT_TEXMAP_CYLINDRICAL = 3
} rrt_texture_mapping;
#define RRT_MAX_TEXTURES 32
typedef struct rrt_texture {
    uint32_t kind, mapping;
    int32_t t1, t2, amount;       /* child texture indices (< own index); amount: a float texture (Mix)        */
    uint32_t aa;                  /* Checkerboard 2D: 0 = AAMethod::AANone, 1 = ClosedForm (the loader's default) */
    double v[4][3];               /* Constant: v[0]; Bilerp: v00 v01 v10 v11                                   */
    double map[8];                /* uv: su sv du dv; planar: vs[3] vt[3] ds dt                                */
    double world_to_texture[16];  /* Checkerboard 3D / Windy / Wrinkled (IdentityMapping3D), spherical /
                                   * cylindrical: row-major                                                   */
} rrt_texture;
/* Which texture drives each parameter of a material; -1 = the constant held in rrt_material.               */
typedef enum rrt_material_slot {
    RRT_SLOT_KD = 0, RRT_SLOT_KS, RRT_SLOT_KR, RRT_SLOT_KT, RRT_SLOT_METAL_ETA, RRT_SLOT_METAL_K, RRT_SLOT_SIGMA,
    RRT_SLOT_ROUGHNESS, RRT_SLOT_U_ROUGHNESS, RRT_SLOT_V_ROUGHNESS, RRT_SLOT_ETA,
    RRT_SLOT_BUMP_MAP, /* Material::bump (material/mod.rs:22-65): a float texture displaces the shading frame         */
    /* DisneyMaterial's scalars in rrt_material order, then scatter_distance (color = KD, roughness, eta as above)   */
    RRT_SLOT_METALLIC, RRT_SLOT_SPECULAR_TINT, RRT_SLOT_ANISOTROPIC, RRT_SLOT_SHEEN, RRT_SLOT_SHEEN_TINT,
    RRT_SLOT_CLEARCOAT, RRT_SLOT_CLEARCOAT_GLOSS, RRT_SLOT_SPEC_TRANS, RRT_SLOT_FLATNESS, RRT_SLOT_DIFF_TRANS,
    RRT_SLOT_SCATTER_DISTANCE,
    RRT_MATERIAL_SLOTS
} rrt_material_slot;

/* lights/point.rs, lights/distant.rs, lights/diffuse.rs (make_light, renderprocess.rs:967-1053).
 * A DiffuseAreaLight samples a shape of its own — make_light_shape (renderprocess.rs:1078-1095): a Sphere with its
 * own transform, or one triangle of a loaded mesh (untransformed vertices, Q7).  That shape is not in the aggregate
 * and the loader attaches no area light to any primitive (Q22): the emitter is sampled by next-event estimation only. */
/* RRT_LIGHT_INFINITE: lights/infinite.rs — an environment map sampled through its luminance distribution, with the
 * BSDF-sampling half of estimate_direct live (integrator/mod.rs:484-556): `env_image` = index of an image added with
 * rrt_scene_add_image*, `to_world` = light_to_world, `shape_to_world_inv` = world_to_light (make_to_world's own inverse).
 * `intensity` is carried but, like the reference (Q34), never multiplied in.                                         */
typedef enum rrt_light_kind { RRT_LIGHT_POINT = 0, RRT_LIGHT_DISTANT = 1, RRT_LIGHT_DIFFUSE_AREA = 2, RRT_LIGHT_INFINITE = 3 } rrt_light_kind;
typedef enum rrt_light_shape_kind { RRT_LIGHT_SHAPE_SPHERE = 0, RRT_LIGHT_SHAPE_TRIANGLE = 1 } rrt_light_shape_kind;
typedef struct rrt_light {
    uint32_t kind;
    uint32_t shape_kind;  /* area: rrt_light_shape_kind                                          */
    double intensity[3];  /* point: I ("spectrum"); distant: l * scale; area: lemit ("spectrum") */
    double dir[3];        /* distant: from - to                                                 */
    double to_world[16];  /* light_to_world matrix, row-major (unused by point lights: Q17)     */
    /* area light shape */
    double shape_to_world[16], shape_to_world_inv[16]; /* sphere: make_sphere's transform and inverse */
    double radius, z_min, z_max, phi_max_deg;          /* sphere (sampling ignores the clipping; area() does not) */
    double tri_p[9];      /* triangle: p0 p1 p2                                                 */
    double tri_n[9];      /* triangle: vertex normals (when tri_has_n)                          */
    uint32_t tri_has_n;
    uint32_t env_image;   /* infinite: image index                                              */
} rrt_light;

typedef enum rrt_filter_kind { RRT_FILTER_BOX = 0, RRT_FILTER_GAUSSIAN = 1, RRT_FILTER_TRIANGLE = 2 } rrt_filter_kind;
/* PathIntegrator (integrator/path.rs), DirectLightingIntegrator (integrator/directlighting.rs, with its specular
 * recursion, integrator/mod.rs:150-301), IntersectDebugIntegrator (integrator/intersect_debug.rs:56-89: a constant 0.1 per
 * hit + uniform_sample_all_lights + the same recursion — what samples/scene.json asks for).                          */
typedef enum rrt_integrator_kind { RRT_INTEGRATOR_PATH = 0, RRT_INTEGRATOR_DIRECT = 1, RRT_INTEGRATOR_DEBUG = 2 } rrt_integrator_kind;
/* make_sampler (renderprocess.rs:1306-1325) */
typedef enum rrt_sampler_kind { RRT_SAMPLER_HALTON = 0, RRT_SAMPLER_STRATIFIED = 1 } rrt_sampler_kind;

/* make_film / make_camera / make_sampler / make_integrator arguments (renderprocess.rs:1306-1499). */
typedef struct rrt_render_desc {
    /* Film */
    int64_t xres, yres;
    double diagonal_mm, scale, max_sample_luminance;
    uint32_t filter_kind, pad0;
    double filter_radius[2], filter_alpha;
    /* Camera (RealisticCamera) */
    double cam_pos[3], cam_look[3], cam_up[3];
    double shutter_open, shutter_close, aperture_diameter, focus_distance;
    uint32_t simple_weighting, n_lens_values;
    const double* lens_data;          /* 4 values per element interface, millimetres            */
    /* Sampler (HaltonSampler) */
    uint64_t nsamp;                   /* the reference renders nsamp - 1 samples per pixel (Q10) */
    uint32_t sample_at_center;
    uint32_t light_strategy;          /* DirectLighting: 0 = UniformSampleOne, 1 = UniformSampleAll (one sample per
                                       * light: the reference's sample arrays never reach its tile samplers, Q30) */
    uint64_t seed;                    /* digit-permutation seed (0 = identity); DESIGN.md §6    */
    /* Integrator */
    uint32_t integrator_kind, max_depth;
    double rr_threshold;
    /* Sampler, continued (fields added after round 1 sit at the end: older callers' zeroes mean HaltonSampler) */
    uint32_t sampler_kind;            /* rrt_sampler_kind                                        */
    uint32_t strat_xsamp, strat_ysamp;/* StratifiedSampler: xsamp * ysamp samples per pixel, of which the first is
                                       * never rendered (Q10); `nsamp` is ignored                 */
    uint32_t strat_dimension;         /* sampled dimensions; a draw past them is U[-1, 1) (Q12)  */
    uint32_t strat_jitter, pad1;      /* `seed` also seeds the jitter / shuffle streams (csrc/stratified.cuh) */
} rrt_render_desc;

typedef struct rrt_render rrt_render; /* Box<dyn Integrator> + its film, camera and sampler      */

int rrt_scene_set_materials(rrt_scene* scene, uint32_t n, const rrt_material* materials);
int rrt_scene_set_lights(rrt_scene* scene, uint32_t n, const rrt_light* lights);
/* Scene::infinite_lights (scene.rs:17-30, make_all_lights renderprocess.rs:945-960): the second light list, which only
 * PathIntegrator reads — an escaped camera ray or specular bounce adds every entry's Light::le (path.rs:79-88).       */
int rrt_scene_set_infinite_lights(rrt_scene* scene, uint32_t n, const rrt_light* lights);
/* Images for RRT_TEX_IMAGE textures and RRT_LIGHT_INFINITE lights: 8-bit RGB, rows top first (what
 * `image::io::Reader::open(..).decode().into_rgb8()` hands load_image, renderprocess.rs:535-566), or a PNG file read by the
 * library (non-interlaced, 8 bits per channel or palette).  *index receives the image's number.                      */
int rrt_scene_add_image(rrt_scene* scene, uint32_t width, uint32_t height, const uint8_t* rgb8, uint32_t* index);
int rrt_scene_add_image_png(rrt_scene* scene, const char* path, uint32_t* index);
/* The texture table (n <= RRT_MAX_TEXTURES) and, per material set with rrt_scene_set_materials, the
 * RRT_MATERIAL_SLOTS texture indices of its parameters (slots[material * RRT_MATERIAL_SLOTS + slot], -1 = constant).
 * Optional: a scene without these calls has constant-valued materials.                                        */
int rrt_scene_set_textures(rrt_scene* scene, uint32_t n, const rrt_texture* textures);
int rrt_scene_set_material_textures(rrt_scene* scene, uint32_t n_materials, const int32_t* slots);
/* deploy_render's loader: parses scene.json (+ the .obj files it names, relative to it) into a
 * committed scene and the integrator that renders it.  `overrides_json` (may be NULL) replaces
 * top-level keys (e.g. {"Integrator": {...}, "Sampler": {...}}) before the factories run.       */
int rrt_scene_load_json(rrt_ctx* ctx, const char* path, const char* overrides_json, uint64_t seed, rrt_scene** scene,
                        rrt_render** render);
/* The same with the parity tier chosen (RRT_BUILD_FAST / RRT_BUILD_LITERAL): in the literal tier the
 * integrator also keeps the reference's shadow-ray construction (Q9) and instance-ray rule (Q6). */
int rrt_scene_load_json_tier(rrt_ctx* ctx, const char* path, const char* overrides_json, uint64_t seed,
                             uint32_t build_flags, rrt_scene** scene, rrt_render** render);
/* make_integrator for an assembled scene.                                                       */
int rrt_render_create(rrt_scene* scene, const rrt_render_desc* desc, rrt_render** out);
void rrt_render_destroy(rrt_render* render);
/* Integrator::render for the 16x16 sample tiles t with t % tile_mod == tile_rank
 * (integrator/mod.rs:55-71; tile index = tile_y * n_tiles_x + tile_x).  (1, 0) renders the frame.
 * `crop` (may be NULL) = pixel rectangle x0,y0,x1,y1 to sample.  Accumulates into the film;
 * returns after the device finished.                                                            */
int rrt_render_run(rrt_render* render, uint32_t tile_mod, uint32_t tile_rank, const int64_t* crop);
int rrt_render_clear(rrt_render* render);
/* Film::write_image up to the float image (film.rs:323-366): rgb[yres*xres*3]; raw (may be NULL)
 * [yres*xres*4] = pixel xyz + filter_weight_sum as the reference's Film would hold them.        */
int rrt_render_read_film(rrt_render* render, double* rgb, double* raw);
/* write_image (renderprocess.rs:1501-1530): sRGB gamma + `clamp(255 g + 0.5) as u8`, alpha 255.
 * rgba8[yres*xres*4]; rrt_render_write_png also writes the file (`save_to` of deploy_render).   */
int rrt_render_read_rgba8(rrt_render* render, uint8_t* rgba8);
int rrt_render_write_png(rrt_render* render, const char* path);
/* The same quantisation for a caller-held float image (host only; no device is touched).        */
int rrt_rgb_to_png(const double* rgb, uint32_t xres, uint32_t yres, const char* path, uint8_t* rgba8_or_null);
/* Device pointer to the accumulation film (4 f64 per pixel: RGB contribution sum, filter weight sum)
 * for a multi-GPU gather/reduce; *n_doubles = 4 * xres * yres.                                   */
int rrt_render_film_device(rrt_render* render, void** d_film, uint64_t* n_doubles);
/* Copies the accumulation film to (to_render = 0) or from (to_render = 1) a caller-owned DEVICE
 * buffer of n_doubles f64 on `cuda_stream` — the hand-off to a collective that sums ranks' films
 * (merge_film_tile across ranks, film.rs:248-263).                                              */
int rrt_render_film_copy(rrt_render* render, void* d_buffer, int to_render, void* cuda_stream);
/* The film GATHER of a multi-GPU frame (renderprocess.rs tiling dealt to ranks; merge_film_tile, film.rs:248-263).  With a
 * filter radius <= 0.5 the tiles t % tile_mod == tile_rank own their pixels, so a rank ships only those: 1 / G of the film.
 *   rrt_render_owned_doubles : size of that rank's packed tiles (1024 doubles per 16 x 16 tile);
 *   rrt_render_pack_owned    : film -> caller-owned DEVICE buffer, on `cuda_stream` (ordered after the render);
 *   rrt_render_unpack_owned  : DEVICE buffer -> film (the root calls it once per sender, with the sender's rank);
 *   rrt_film_gather          : ONE process driving n renderers on n devices, renders[r] having run (n, r): packs every
 *                              rank's tiles, copies them to renders[root]'s device (peer copy over NVLink) and unpacks.
 * Processes-per-GPU callers move the packed buffers with their own collective (NCCL gather; rs_ray_toy_b200/parallel.py).
 * Wider filters splat across tile borders: RRT_ERR_UNSUPPORTED here, use rrt_render_film_copy + a sum.               */
int rrt_render_owned_doubles(const rrt_render* render, uint32_t tile_mod, uint32_t tile_rank, uint64_t* n_doubles);
int rrt_render_pack_owned(rrt_render* render, uint32_t tile_mod, uint32_t tile_rank, void* d_buffer, uint64_t capacity_doubles,
                          void* cuda_stream);
int rrt_render_unpack_owned(rrt_render* render, uint32_t tile_mod, uint32_t tile_rank, const void* d_buffer,
                            uint64_t capacity_doubles, void* cuda_stream);
int rrt_film_gather(rrt_render* const* renders, uint32_t n, uint32_t root);
/* out16: camera rays, extension rays, shadow rays, bounces, zero-weight samples, samples, kernels
 * launched, render microseconds, set-up microseconds, chunks, neighbour lens rays decided by the fp32
 * walk, neighbour lens rays it handed to the f64 walk, ...                                       */
int rrt_render_stats(const rrt_render* render, uint64_t out16[16]);
/* First-hit record of every camera sample of the last run, in launch order: 6 doubles per sample
 * (pixel x, pixel y, sample number, prim id or -1 miss / -2 zero weight, t, ray weight).         */
int rrt_render_hit_dump(rrt_render* render, int enable, double* out, uint64_t capacity, uint64_t* count);

#ifdef __cplusplus
}
#endif
#endif /* RRT_H_ */
