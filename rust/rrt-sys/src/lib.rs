//! Raw FFI over `include/rrt.h` (librrt_sm100.so).  Every function returns `RRT_OK` (0) or a negative `rrt_status`;
//! `rrt_last_error()` gives the text of the calling thread's last failure.  No panic or exception crosses the ABI.
#![allow(non_camel_case_types)]
use std::mem::size_of;
use std::os::raw::{c_char, c_int, c_void};

pub const RRT_OK: c_int = 0;
pub const RRT_ERR_INVALID: c_int = -1;
pub const RRT_ERR_CUDA: c_int = -2;
pub const RRT_ERR_UNSUPPORTED: c_int = -3;
pub const RRT_ERR_EMPTY: c_int = -4;
pub const RRT_ERR_IO: c_int = -5;
pub const RRT_NO_HIT: u32 = 0xFFFF_FFFF;
pub const RRT_BUILD_FAST: u32 = 0;
pub const RRT_BUILD_LITERAL: u32 = 1;
pub const RRT_BUILD_DEVICE_LBVH: u32 = 2;
pub const RRT_MAX_TEXTURES: usize = 32;
pub const RRT_MATERIAL_SLOTS: usize = 23;

#[repr(C)] pub struct rrt_ctx { _p: [u8; 0] }
#[repr(C)] pub struct rrt_scene { _p: [u8; 0] }
#[repr(C)] pub struct rrt_render { _p: [u8; 0] }

/// geometry.rs:73-79 `Ray` (f64; `medium` out of scope)
#[repr(C)] #[derive(Copy, Clone, Debug, Default)]
pub struct rrt_ray { pub o: [f64; 3], pub d: [f64; 3], pub t_max: f64, pub time: f64 }
/// what BVHAccel::intersect hands back through `r.t_max` and `si`
#[repr(C)] #[derive(Copy, Clone, Debug, Default)]
pub struct rrt_hit { pub prim_id: u32, pub reserved: u32, pub t: f64, pub u: f64, pub v: f64 }
/// fp32 ray for rrt_intersect_f32 and relatives: promoted exactly to `rrt_ray` (time 0) on the device
#[repr(C)] #[derive(Copy, Clone, Debug, Default)]
pub struct rrt_ray_f32 { pub o: [f32; 3], pub t_max: f32, pub d: [f32; 3], pub reserved: u32 }
/// `rrt_hit` with t, u, v rounded to nearest fp32
#[repr(C)] #[derive(Copy, Clone, Debug, Default)]
pub struct rrt_hit_f32 { pub prim_id: u32, pub t: f32, pub u: f32, pub v: f32 }

/// material/{matte,plastic,metal,mirror,glass,translucent,disney,debug_material}.rs with constant parameters
/// (kind: 0 Matte .. 4 Glass, 5 Translucent, 6 Disney, 7 Debug)
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct rrt_material {
    pub kind: u32, pub remap_roughness: u32,
    pub kd: [f64; 3], pub ks: [f64; 3], pub kr: [f64; 3], pub kt: [f64; 3],
    pub metal_eta: [f64; 3], pub metal_k: [f64; 3],
    pub sigma: f64, pub roughness: f64, pub u_roughness: f64, pub v_roughness: f64, pub eta: f64,
    pub metallic: f64, pub specular_tint: f64, pub anisotropic: f64, pub sheen: f64, pub sheen_tint: f64,
    pub clearcoat: f64, pub clearcoat_gloss: f64, pub spec_trans: f64, pub flatness: f64, pub diff_trans: f64,
    pub scatter_distance: [f64; 3],
    pub thin: u32, pub pad: u32,
}
/// one row of the flattened texture table (kind: 0 Constant .. 8 Wrinkled, 9 Image)
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct rrt_texture {
    pub kind: u32, pub mapping: u32,
    pub t1: i32, pub t2: i32, pub amount: i32,
    pub aa: u32,
    pub v: [[f64; 3]; 4],
    pub map: [f64; 8],
    pub world_to_texture: [f64; 16],
}
/// lights/{point,distant,diffuse,infinite}.rs (kind: 0 point, 1 distant, 2 diffuse area, 3 infinite)
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct rrt_light {
    pub kind: u32, pub shape_kind: u32,
    pub intensity: [f64; 3], pub dir: [f64; 3],
    pub to_world: [f64; 16], pub shape_to_world: [f64; 16], pub shape_to_world_inv: [f64; 16],
    pub radius: f64, pub z_min: f64, pub z_max: f64, pub phi_max_deg: f64,
    pub tri_p: [f64; 9], pub tri_n: [f64; 9],
    pub tri_has_n: u32, pub env_image: u32,
}
/// make_film / make_camera / make_sampler / make_integrator arguments (renderprocess.rs:1306-1499)
#[repr(C)] #[derive(Copy, Clone, Debug)]
pub struct rrt_render_desc {
    pub xres: i64, pub yres: i64,
    pub diagonal_mm: f64, pub scale: f64, pub max_sample_luminance: f64,
    pub filter_kind: u32, pub pad0: u32,
    pub filter_radius: [f64; 2], pub filter_alpha: f64,
    pub cam_pos: [f64; 3], pub cam_look: [f64; 3], pub cam_up: [f64; 3],
    pub shutter_open: f64, pub shutter_close: f64, pub aperture_diameter: f64, pub focus_distance: f64,
    pub simple_weighting: u32, pub n_lens_values: u32,
    pub lens_data: *const f64,
    pub nsamp: u64,
    pub sample_at_center: u32, pub light_strategy: u32,
    pub seed: u64,
    pub integrator_kind: u32, pub max_depth: u32,
    pub rr_threshold: f64,
    pub sampler_kind: u32, pub strat_xsamp: u32, pub strat_ysamp: u32, pub strat_dimension: u32,
    pub strat_jitter: u32, pub pad1: u32,
}

// the C sizes (tests/test_capi_exports.py compares them with sizeof on the C side)
const _: () = assert!(size_of::<rrt_ray>() == 64);
const _: () = assert!(size_of::<rrt_hit>() == 32);
const _: () = assert!(size_of::<rrt_material>() == 304);
const _: () = assert!(size_of::<rrt_texture>() == 312);
const _: () = assert!(size_of::<rrt_light>() == 624);
const _: () = assert!(size_of::<rrt_render_desc>() == 256);
// the fp32 records (tests/test_rays_f32.py checks these sizes against the C side)
const _: () = assert!(size_of::<rrt_ray_f32>() == 32);
const _: () = assert!(size_of::<rrt_hit_f32>() == 16);

extern "C" {
    // ---- context ----
    pub fn rrt_create(device_ordinal: c_int, out: *mut *mut rrt_ctx) -> c_int;
    pub fn rrt_destroy(ctx: *mut rrt_ctx);
    pub fn rrt_last_error() -> *const c_char;
    pub fn rrt_launch_count(ctx: *const rrt_ctx) -> u64;
    pub fn rrt_host_alloc(ctx: *mut rrt_ctx, bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn rrt_host_free(ctx: *mut rrt_ctx, p: *mut c_void) -> c_int;
    // ---- scene assembly (make_aggregate, renderprocess.rs:1178-1304) ----
    pub fn rrt_scene_begin(ctx: *mut rrt_ctx, out: *mut *mut rrt_scene) -> c_int;
    pub fn rrt_scene_destroy(scene: *mut rrt_scene);
    pub fn rrt_scene_add_mesh(scene: *mut rrt_scene, nv: u32, p: *const f64, ntri: u32, vi: *const u32, nn: u32, n: *const f64,
                              ni: *const u32, nuv: u32, uv: *const f64, uvi: *const u32, mesh_id: *mut u32) -> c_int;
    pub fn rrt_scene_add_triangles(scene: *mut rrt_scene, mesh_id: u32, material_id: u32, n_instances: u32,
                                   instance_m: *const f64, instance_minv: *const f64) -> c_int;
    pub fn rrt_scene_add_sphere(scene: *mut rrt_scene, obj_to_world_m: *const f64, obj_to_world_minv: *const f64, radius: f64,
                                z_min: f64, z_max: f64, phi_max_deg: f64, material_id: u32, n_instances: u32,
                                instance_m: *const f64, instance_minv: *const f64) -> c_int;
    pub fn rrt_scene_commit(scene: *mut rrt_scene, max_prims_in_node: u32, build_flags: u32) -> c_int;
    pub fn rrt_scene_update_instances(scene: *mut rrt_scene, first_instance: u32, n: u32, instance_m: *const f64, instance_minv: *const f64) -> c_int;
    pub fn rrt_scene_num_prims(scene: *const rrt_scene, out: *mut u32) -> c_int;
    pub fn rrt_world_bound(scene: *const rrt_scene, out6: *mut f64) -> c_int;
    pub fn rrt_scene_export_tree(scene: *const rrt_scene, buffer: *mut c_void, capacity: u64, bytes: *mut u64) -> c_int;
    pub fn rrt_scene_commit_from_tree(scene: *mut rrt_scene, blob: *const c_void, bytes: u64) -> c_int;
    pub fn rrt_scene_stats(scene: *const rrt_scene, out8: *mut u64) -> c_int;
    pub fn rrt_scene_build_info(scene: *const rrt_scene, out4: *mut u64) -> c_int;
    // ---- the hot path (Scene::intersect / intersect_p, scene.rs:69-80) ----
    pub fn rrt_intersect_device(scene: *const rrt_scene, n: u64, d_rays: *const rrt_ray, d_hits: *mut rrt_hit, cuda_stream: *mut c_void) -> c_int;
    pub fn rrt_intersect_p_device(scene: *const rrt_scene, n: u64, d_rays: *const rrt_ray, d_occluded: *mut u8, cuda_stream: *mut c_void) -> c_int;
    pub fn rrt_intersect(scene: *const rrt_scene, n: u64, rays: *const rrt_ray, hits: *mut rrt_hit) -> c_int;
    pub fn rrt_intersect_p(scene: *const rrt_scene, n: u64, rays: *const rrt_ray, occluded: *mut u8) -> c_int;
    // ---- the same over fp32 rays and compact hits ----
    pub fn rrt_intersect_f32(scene: *const rrt_scene, n: u64, rays: *const rrt_ray_f32, hits: *mut rrt_hit_f32) -> c_int;
    pub fn rrt_intersect_p_f32(scene: *const rrt_scene, n: u64, rays: *const rrt_ray_f32, occluded: *mut u8) -> c_int;
    pub fn rrt_intersect_f32_device(scene: *const rrt_scene, n: u64, d_rays: *const rrt_ray_f32, d_hits: *mut rrt_hit_f32, cuda_stream: *mut c_void) -> c_int;
    pub fn rrt_intersect_p_f32_device(scene: *const rrt_scene, n: u64, d_rays: *const rrt_ray_f32, d_occluded: *mut u8, cuda_stream: *mut c_void) -> c_int;
    // ---- shading tables ----
    pub fn rrt_scene_set_materials(scene: *mut rrt_scene, n: u32, materials: *const rrt_material) -> c_int;
    pub fn rrt_scene_set_lights(scene: *mut rrt_scene, n: u32, lights: *const rrt_light) -> c_int;
    pub fn rrt_scene_set_infinite_lights(scene: *mut rrt_scene, n: u32, lights: *const rrt_light) -> c_int;
    pub fn rrt_scene_add_image(scene: *mut rrt_scene, width: u32, height: u32, rgb8: *const u8, index: *mut u32) -> c_int;
    pub fn rrt_scene_add_image_png(scene: *mut rrt_scene, path: *const c_char, index: *mut u32) -> c_int;
    pub fn rrt_scene_set_textures(scene: *mut rrt_scene, n: u32, textures: *const rrt_texture) -> c_int;
    pub fn rrt_scene_set_material_textures(scene: *mut rrt_scene, n_materials: u32, slots: *const i32) -> c_int;
    // ---- the render loop (deploy_render, renderprocess.rs:92-105) ----
    pub fn rrt_scene_load_json(ctx: *mut rrt_ctx, path: *const c_char, overrides_json: *const c_char, seed: u64,
                               scene: *mut *mut rrt_scene, render: *mut *mut rrt_render) -> c_int;
    pub fn rrt_scene_load_json_tier(ctx: *mut rrt_ctx, path: *const c_char, overrides_json: *const c_char, seed: u64, build_flags: u32,
                                    scene: *mut *mut rrt_scene, render: *mut *mut rrt_render) -> c_int;
    pub fn rrt_render_create(scene: *mut rrt_scene, desc: *const rrt_render_desc, out: *mut *mut rrt_render) -> c_int;
    pub fn rrt_render_destroy(render: *mut rrt_render);
    pub fn rrt_render_run(render: *mut rrt_render, tile_mod: u32, tile_rank: u32, crop: *const i64) -> c_int;
    pub fn rrt_render_clear(render: *mut rrt_render) -> c_int;
    pub fn rrt_render_read_film(render: *mut rrt_render, rgb: *mut f64, raw: *mut f64) -> c_int;
    pub fn rrt_render_read_rgba8(render: *mut rrt_render, rgba8: *mut u8) -> c_int;
    pub fn rrt_render_write_png(render: *mut rrt_render, path: *const c_char) -> c_int;
    pub fn rrt_rgb_to_png(rgb: *const f64, xres: u32, yres: u32, path: *const c_char, rgba8_or_null: *mut u8) -> c_int;
    pub fn rrt_render_film_device(render: *mut rrt_render, d_film: *mut *mut c_void, n_doubles: *mut u64) -> c_int;
    pub fn rrt_render_film_copy(render: *mut rrt_render, d_buffer: *mut c_void, to_render: c_int, cuda_stream: *mut c_void) -> c_int;
    // ---- multi-GPU: the film gather of a frame whose tiles were dealt to ranks ----
    pub fn rrt_render_owned_doubles(render: *const rrt_render, tile_mod: u32, tile_rank: u32, n_doubles: *mut u64) -> c_int;
    pub fn rrt_render_pack_owned(render: *mut rrt_render, tile_mod: u32, tile_rank: u32, d_buffer: *mut c_void, capacity_doubles: u64,
                                 cuda_stream: *mut c_void) -> c_int;
    pub fn rrt_render_unpack_owned(render: *mut rrt_render, tile_mod: u32, tile_rank: u32, d_buffer: *const c_void, capacity_doubles: u64,
                                   cuda_stream: *mut c_void) -> c_int;
    pub fn rrt_film_gather(renders: *const *mut rrt_render, n: u32, root: u32) -> c_int;
    pub fn rrt_render_stats(render: *const rrt_render, out16: *mut u64) -> c_int;
    pub fn rrt_render_hit_dump(render: *mut rrt_render, enable: c_int, out: *mut f64, capacity: u64, count: *mut u64) -> c_int;
}

/// `rrt_last_error()` as a Rust string
pub fn last_error() -> String {
    unsafe {
        let p = rrt_last_error();
        if p.is_null() { String::new() } else { std::ffi::CStr::from_ptr(p).to_string_lossy().into_owned() }
    }
}
/// Turns a status into a `Result`; the reference reports the same conditions with `assert!` / `panic!`
pub fn check(status: c_int) -> Result<(), String> {
    if status == RRT_OK { Ok(()) } else { Err(format!("rrt status {}: {}", status, last_error())) }
}
