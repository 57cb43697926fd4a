/* rrt_test.h — TEST-ONLY entry points of librrt_sm100.so.
 *
 * These run pieces of the PRODUCT's own code on the host so that the CPU test-suite (`pytest -m "not gpu"`) can
 * check them without a device: the device LBVH builder's per-element code, the literal tier's HLBVH, the texture
 * evaluator, the Halton tables, compute_differentials, the scene.json loader.  They are
 * checkers, not a CPU path: none of them traces a ray or renders a sample.  A Rust `rrt-sys` crate binds
 * include/rrt.h only; nothing here belongs in it.                                                                  */
#ifndef RRT_TEST_H
#define RRT_TEST_H
#include "rrt.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Host-only probe of the device LBVH builder's per-element code (lbvh_core.h runs unchanged on the host; this
 * is a checker for the CPU tests, not a product path): world bounds in (6 doubles each), out: the emitted
 * Node64 array (16 x 4-byte words per node: 12 fp32 planes as laid out in device_layout.h, child0, child1, pad),
 * the primitive order, and info3 = { nodes, max depth, leaves }.  *n_nodes is set also when capacity is short. */
int rrt_lbvh_host_probe(uint32_t n, const double* bounds6, uint32_t max_prims_in_node, uint32_t capacity_nodes,
                        uint32_t* n_nodes, uint32_t* node_words16, uint32_t* order, uint32_t info3[3]);

/* Host-only probe of the literal tier's tree builder (BVHAccel::new with HLBVH, bvh.rs:307-751) on a
 * list of primitive world bounds (6 doubles each: p_min, p_max).  Returns the flattened
 * LinearBVHNode array: node_bounds6[6 * i], node_meta3[3 * i] = (offset, n_primitives, axis), and the
 * reordered primitive list.  *n_nodes receives the node count (also when capacity is too small).   */
int rrt_hlbvh_literal_probe(uint32_t n, const double* bounds6, uint32_t max_prims_in_node, uint32_t capacity_nodes,
                            uint32_t* n_nodes, double* node_bounds6, uint32_t* node_meta3, uint32_t* ordered);

/* Host-only evaluation of a texture table at (uv, p) with the product's own evaluator (csrc/texture_core.h, the
 * code the shade kernel runs): out[3 * i + c] for every texture i.  `diff` (may be NULL = none) holds the
 * screen-space differentials dpdx[3] dpdy[3] dudx dvdx dudy dvdy.  For the CPU test-suite.                    */
int rrt_texture_host_probe(uint32_t n, const rrt_texture* textures, const double uv[2], const double p[3],
                           const double* diff, double* out);

/* Host-only HaltonSampler probe (csrc/halton.cuh, the code the kernels run): for each i the sample index of
 * (px, py, sample) (Halton::get_index_for_sample, halton.rs:75-105) and its value in dimension dim
 * (sample_dimension, :107-128) for a film of xres x yres and the given permutation seed.  use_tables = 1 takes the
 * table-driven paths the device takes (per-dimension constants, exact multiply-shift division, per-pixel index
 * terms), 0 the generic digit loops: both must give the same bits.                                            */
int rrt_halton_host_probe(int64_t xres, int64_t yres, uint64_t seed, int use_tables, uint64_t n, const int64_t* px,
                          const int64_t* py, const uint64_t* sample, const uint32_t* dim, uint64_t* index_out, double* value_out);

/* Host-only SurfaceInteraction::compute_differentials with the product's code (csrc/texture_core.h): in = p[3] n[3]
 * dpdu[3] dpdv[3] rx_origin[3] rx_direction[3] ry_origin[3] ry_direction[3]; out = dpdx[3] dpdy[3] dudx dvdx dudy dvdy. */
int rrt_differentials_host_probe(const double in24[24], double out10[10]);

/* Host-only view of what the loader reads (no device is touched): out8 = primitives, meshes,
 * spheres, instances, materials, lights, max_prims_in_node, lens values; desc = the render
 * description (lens_data pointer left NULL).  Used by the CPU test-suite and by tooling.          */
int rrt_scene_json_probe(const char* path, const char* overrides_json, uint64_t out8[8], rrt_render_desc* desc);

/* Host-only view of the loader's texture table and materials: textures (room for RRT_MAX_TEXTURES, may be NULL),
 * the first max_materials materials and their RRT_MATERIAL_SLOTS texture indices each (may be NULL).          */
int rrt_scene_json_texture_probe(const char* path, const char* overrides_json, uint32_t* n_textures, rrt_texture* textures,
                                 uint32_t max_materials, uint32_t* n_materials, rrt_material* materials, int32_t* slots);

/* Host-only probe of the device StratifiedSampler (csrc/stratified.cuh, the code the kernels run): for one pixel the
 * 1D tables out1d[ndims][xs * ys], the 2D tables out2d[ndims][xs * ys][2] as PixelSampler::start_pixel leaves them, and
 * for every sample k >= 1 the first four draws past the sampled dimensions overflow4[k][4].                           */
int rrt_stratified_host_probe(uint64_t seed, int64_t xres, int64_t px, int64_t py, uint32_t xs, uint32_t ys, uint32_t ndims,
                              int jitter, double* out1d, double* out2d, double* overflow4);

/* Host-only probes of the image path.  rrt_png_host_probe: the library's PNG reader (csrc/image_host.cpp) -> 8-bit RGB.
 * rrt_mipmap_host_probe: MIPMap::create on the host, then for each of n queries (st[2], dstdx[2], dstdy[2]) the device
 * lookups of csrc/mipmap_core.h run on the host: lookup_d -> out6[0..2], lookup_w(st, width = dstdx[0]) -> out6[3..5];
 * info = levels, then (u_res, v_res) per level.  rrt_envlight_host_probe: InfiniteAreaLight::new's distribution, then per
 * query (ref point[3], u[2], w[3]): sample_li -> Li[3], wi[3], pdf; pdf_li(w); le(w)[3]; p1.x.                        */
/* Host-only probe of the fp32 record format (csrc/rays_f32.cuh, the conversions the streaming kernels around the walk
 * run): promoted[i] = rays[i] as the rrt_ray the walk sees, compact[i] = hits[i] as the rrt_hit_f32 the caller gets. */
int rrt_rays_f32_host_probe(uint64_t n_rays, const rrt_ray_f32* rays, rrt_ray* promoted, uint64_t n_hits, const rrt_hit* hits,
                            rrt_hit_f32* compact);

int rrt_png_host_probe(const char* path, uint32_t* width, uint32_t* height, uint8_t* rgb8, uint64_t capacity);
int rrt_mipmap_host_probe(uint32_t width, uint32_t height, const uint8_t* rgb8, int trilinear, double max_aniso, uint32_t wrap,
                          uint64_t n, const double* q6, double* out6, uint64_t info[32]);
int rrt_envlight_host_probe(uint32_t width, uint32_t height, const uint8_t* rgb8, const double to_world16[16],
                            const double to_local16[16], double world_radius, uint64_t n, const double* in8, double* out12);

#ifdef __cplusplus
}
#endif
#endif /* RRT_TEST_H */
