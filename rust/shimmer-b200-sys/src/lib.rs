//! Raw declarations of `include/shimmer_b200.h` (one per exported symbol, same order as the header).
//! Hand-written so that the crate builds without libclang; `--features bindgen` regenerates them into
//! `OUT_DIR/bindings.rs` for comparison.  `tests/test_rust_binding.py` checks names and arities against the header.
#![allow(non_camel_case_types)]

use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct shim_scene {
    _private: [u8; 0],
}

pub const SHIM_OK: c_int = 0;
pub const SHIM_ERR_INVALID: c_int = -1;
pub const SHIM_ERR_UNSUPPORTED: c_int = -2;
pub const SHIM_ERR_CUDA: c_int = -3;
pub const SHIM_ERR_STATE: c_int = -4;

pub const SHIM_OPT_DEVICE_BVH: c_int = 1;
pub const SHIM_DEVICE_BVH_SAH: c_int = 0;
pub const SHIM_DEVICE_BVH_REFERENCE: c_int = 1;

pub const SHIM_RENDER_RAW_SUM: i32 = 1;
pub const SHIM_RENDER_PREDICTORS: i32 = 2;
pub const SHIM_RENDER_COUNT_NODES: i32 = 4;
pub const SHIM_RENDER_PROFILE: i32 = 8;
pub const SHIM_RENDER_KEEP_PREDICTORS: i32 = 16;

pub const SHIM_SHARD_SAMPLES: c_int = 0;
pub const SHIM_SHARD_TILES: c_int = 1;

/// The nine `Camera::new` arguments (camera.rs:44-54).
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct shim_camera {
    pub look_from: [f32; 3],
    pub look_at: [f32; 3],
    pub view_up: [f32; 3],
    pub vertical_fov: f32,
    pub aspect_ratio: f32,
    pub aperture: f32,
    pub focus_dist: f32,
    pub time_start: f32,
    pub time_end: f32,
}

/// Arguments of `Renderer::render` (renderer.rs:42-52) plus sharding and the Philox key.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct shim_render_params {
    pub width: i32,
    pub height: i32,
    pub samples_per_pixel: i32,
    pub max_depth: i32,
    pub tile_width: i32,
    pub tile_height: i32,
    pub background: [f32; 3],
    pub seed: u64,
    pub sample_begin: i32,
    pub sample_count: i32,
    pub tile_rank: i32,
    pub tile_world: i32,
    pub flags: i32,
    pub pool_paths: i32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct shim_stats {
    pub rays: u64,
    pub samples: u64,
    pub node_visits: u64,
    pub prim_tests: u64,
    pub hrpp_true_positive: u64,
    pub hrpp_false_positive: u64,
    pub hrpp_no_prediction: u64,
    pub kernel_launches: u64,
    pub iterations: u64,
    pub device_ms: f64,
    pub extend_ms: f64,
    pub shade_ms: f64,
    pub generate_ms: f64,
    pub extend_launches: u64,
    pub extend_variant: u64,
    pub pool_paths: u64,
    pub pool_bytes: u64,
    pub devices: u64,
    pub wall_ms: f64,
}

/// `Hittable::hit`'s `HitRecord` (hittable.rs:15-52) plus the id of what was hit; 48 bytes (`shim_trace_hit`).
/// `hittable == -1`: a miss (`material == -1`, `t == +inf`, everything else 0).
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct shim_hit_record {
    pub point: [f32; 3],
    pub normal: [f32; 3],
    pub t: f32,
    pub u: f32,
    pub v: f32,
    pub front_face: i32,
    pub material: i32,
    pub hittable: i32,
}

extern "C" {
    pub fn shim_last_error() -> *const c_char;
    pub fn shim_version() -> c_int;

    pub fn shim_scene_create() -> *mut shim_scene;
    pub fn shim_scene_destroy(s: *mut shim_scene);

    pub fn shim_texture_solid(s: *mut shim_scene, r: f32, g: f32, b: f32) -> c_int;
    pub fn shim_texture_checker(s: *mut shim_scene, scale: f32, even_tex: c_int, odd_tex: c_int) -> c_int;
    pub fn shim_texture_marble(s: *mut shim_scene, scale: f32, perlin_seed: u32) -> c_int;
    pub fn shim_texture_image(s: *mut shim_scene, rgb8: *const u8, width: c_int, height: c_int) -> c_int;

    pub fn shim_material_lambertian(s: *mut shim_scene, albedo_tex: c_int) -> c_int;
    pub fn shim_material_metal(s: *mut shim_scene, r: f32, g: f32, b: f32, fuzz: f32) -> c_int;
    pub fn shim_material_dielectric(s: *mut shim_scene, index_of_refraction: f32) -> c_int;
    pub fn shim_material_diffuse_light(s: *mut shim_scene, emission_tex: c_int) -> c_int;
    pub fn shim_material_isotropic(s: *mut shim_scene, albedo_tex: c_int) -> c_int;

    pub fn shim_sphere(s: *mut shim_scene, cx: f32, cy: f32, cz: f32, radius: f32, material: c_int) -> c_int;
    pub fn shim_moving_sphere(
        s: *mut shim_scene, c0x: f32, c0y: f32, c0z: f32, c1x: f32, c1y: f32, c1z: f32,
        time_start: f32, time_end: f32, radius: f32, material: c_int,
    ) -> c_int;
    pub fn shim_xy_rect(s: *mut shim_scene, x0: f32, x1: f32, y0: f32, y1: f32, z: f32, material: c_int) -> c_int;
    pub fn shim_xz_rect(s: *mut shim_scene, x0: f32, x1: f32, z0: f32, z1: f32, y: f32, material: c_int) -> c_int;
    pub fn shim_yz_rect(s: *mut shim_scene, y0: f32, y1: f32, z0: f32, z1: f32, x: f32, material: c_int) -> c_int;
    pub fn shim_tri(s: *mut shim_scene, p0p1p2: *const f32, material: c_int) -> c_int;
    pub fn shim_cube(s: *mut shim_scene, minx: f32, miny: f32, minz: f32, maxx: f32, maxy: f32, maxz: f32, material: c_int) -> c_int;
    pub fn shim_list_create(s: *mut shim_scene) -> c_int;
    pub fn shim_list_add(s: *mut shim_scene, list: c_int, hittable: c_int) -> c_int;
    pub fn shim_tris_bulk(s: *mut shim_scene, xyz: *const f32, n_tris: c_int, material: c_int, list: c_int) -> c_int;
    pub fn shim_bvh(s: *mut shim_scene, list: c_int, time0: f32, time1: f32, axis_seed: u64, with_predictor: c_int) -> c_int;
    pub fn shim_bvh_from_nodes(
        s: *mut shim_scene, n_nodes: c_int, left: *const i32, right: *const i32, root: c_int,
        time0: f32, time1: f32, with_predictor: c_int,
    ) -> c_int;
    pub fn shim_translate(s: *mut shim_scene, hittable: c_int, dx: f32, dy: f32, dz: f32) -> c_int;
    pub fn shim_rotate_y(s: *mut shim_scene, hittable: c_int, degrees: f32) -> c_int;
    pub fn shim_constant_medium(s: *mut shim_scene, boundary: c_int, density: f32, albedo_tex: c_int) -> c_int;
    pub fn shim_world_add(s: *mut shim_scene, hittable: c_int) -> c_int;
    pub fn shim_scene_set_option(s: *mut shim_scene, option: c_int, value: c_int) -> c_int;
    pub fn shim_commit(s: *mut shim_scene) -> c_int;

    pub fn shim_bvh_info(s: *mut shim_scene, bvh: c_int, n_nodes: *mut c_int, root: *mut c_int, height: *mut c_int) -> c_int;
    pub fn shim_bvh_nodes(s: *mut shim_scene, bvh: c_int, left: *mut i32, right: *mut i32, parent: *mut i32, boxes6: *mut f32) -> c_int;
    pub fn shim_scene_device_bytes(s: *mut shim_scene) -> u64;

    pub fn shim_render(
        s: *mut shim_scene, cam: *const shim_camera, p: *const shim_render_params, out_rgb: *mut f32, stats: *mut shim_stats,
    ) -> c_int;
    pub fn shim_host_alloc(floats: usize) -> *mut f32;
    pub fn shim_host_free(p: *mut f32);
    pub fn shim_render_device(
        s: *mut shim_scene, cam: *const shim_camera, p: *const shim_render_params, d_out_rgb: *mut f32,
        stats: *mut shim_stats, cuda_stream: *mut c_void,
    ) -> c_int;

    pub fn shim_render_multi(
        s: *mut shim_scene, cam: *const shim_camera, p: *const shim_render_params, n_devices: c_int, devices: *const c_int,
        mode: c_int, out_rgb: *mut f32, stats: *mut shim_stats,
    ) -> c_int;
    pub fn shim_shutdown() -> c_int;
    pub fn shim_pool_bytes(device: c_int) -> u64;

    pub fn shim_trace_closest(
        s: *mut shim_scene, rays: *const f32, n: i64, t_min: f32, t_max: f32, seed: u64,
        prim_id: *mut i32, t: *mut f32, counters3: *mut u64,
    ) -> c_int;
    pub fn shim_trace_closest_device(
        s: *mut shim_scene, d_rays: *const f32, n: i64, t_min: f32, t_max: f32, seed: u64,
        d_prim_id: *mut i32, d_t: *mut f32, cuda_stream: *mut c_void,
    ) -> c_int;
    pub fn shim_trace_hit(
        s: *mut shim_scene, rays: *const f32, n: i64, t_min: f32, t_max: f32, seed: u64,
        out: *mut shim_hit_record, counters3: *mut u64,
    ) -> c_int;
    pub fn shim_trace_hit_device(
        s: *mut shim_scene, d_rays: *const f32, n: i64, t_min: f32, t_max: f32, seed: u64,
        d_out: *mut shim_hit_record, cuda_stream: *mut c_void,
    ) -> c_int;
    pub fn shim_trace_occluded(
        s: *mut shim_scene, rays: *const f32, n: i64, t_min: f32, t_max: f32, seed: u64,
        occluded: *mut u8, counters3: *mut u64,
    ) -> c_int;
    pub fn shim_trace_occluded_device(
        s: *mut shim_scene, d_rays: *const f32, n: i64, t_min: f32, t_max: f32, seed: u64,
        d_occluded: *mut u8, cuda_stream: *mut c_void,
    ) -> c_int;

    pub fn shim_tile_layout(image_width: c_int, image_height: c_int, tile_width: c_int, tile_height: c_int, out4: *mut i32, cap: c_int) -> c_int;
    pub fn shim_camera_fields(cam: *const shim_camera, out21: *mut f32) -> c_int;
    pub fn shim_aabb_hit(
        min3: *const f32, max3: *const f32, origin3: *const f32, direction3: *const f32, t_min: f32, t_max: f32, layout: c_int,
    ) -> c_int;
    pub fn shim_hrpp_hash(origin3: *const f32, direction3: *const f32) -> u64;
    pub fn shim_write_ppm(rgb: *const f32, width: c_int, height: c_int, path: *const c_char) -> i64;
}
