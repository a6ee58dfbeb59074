//! Raw bindings: one item per declaration of include/rttnw_b200.h (ABI version 1; tests/test_host_cpu.py keeps the
//! function names in step with the header).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const RTX_OK: c_int = 0;
pub const RTX_ERR_INVALID: c_int = -1;
pub const RTX_MISS: i32 = -1;

// rtx_node_kind
pub const RTX_NODE_SPHERE: i32 = 1;
pub const RTX_NODE_MOVING_SPHERE: i32 = 2;
pub const RTX_NODE_RECT_XY: i32 = 3;
pub const RTX_NODE_RECT_XZ: i32 = 4;
pub const RTX_NODE_RECT_YZ: i32 = 5;
pub const RTX_NODE_CUBE: i32 = 6;
pub const RTX_NODE_LIST: i32 = 7;
pub const RTX_NODE_BVH: i32 = 8;
pub const RTX_NODE_TRANSLATE: i32 = 9;
pub const RTX_NODE_ROTATE_Y: i32 = 10;
pub const RTX_NODE_MEDIUM: i32 = 11;
// rtx_material_kind
pub const RTX_MAT_LAMBERTIAN: i32 = 1;
pub const RTX_MAT_METAL: i32 = 2;
pub const RTX_MAT_DIELECTRIC: i32 = 3;
pub const RTX_MAT_DIFFUSE_LIGHT: i32 = 4;
pub const RTX_MAT_ISOTROPIC: i32 = 5;
// rtx_texture_kind
pub const RTX_TEX_SOLID: i32 = 1;
pub const RTX_TEX_CHECKER: i32 = 2;
pub const RTX_TEX_NOISE: i32 = 3;
pub const RTX_TEX_IMAGE: i32 = 4;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_node {
    pub kind: i32,
    pub material: i32,
    pub child: i32,
    pub n_children: i32,
    pub f: [f64; 10],
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_material {
    pub kind: i32,
    pub texture: i32,
    pub albedo: [f64; 3],
    pub param: f64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_texture {
    pub kind: i32,
    pub a: i32,
    pub b: i32,
    pub _pad: i32,
    pub f: [f64; 4],
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_perlin {
    pub ranvec: [[f64; 3]; 256],
    pub perm_x: [i32; 256],
    pub perm_y: [i32; 256],
    pub perm_z: [i32; 256],
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_image {
    pub width: i32,
    pub height: i32,
    pub rgba: *const u8,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_camera {
    pub lookfrom: [f64; 3],
    pub lookat: [f64; 3],
    pub view_up: [f64; 3],
    pub vertical_fov: f64,
    pub aspect_ratio: f64,
    pub aperture: f64,
    pub focus_distance: f64,
    pub open_time: f64,
    pub close_time: f64,
}
#[repr(C)]
pub struct rtx_scene_desc {
    pub nodes: *const rtx_node,
    pub n_nodes: i32,
    pub root: i32,
    pub children: *const i32,
    pub n_children: i32,
    pub n_materials: i32,
    pub materials: *const rtx_material,
    pub textures: *const rtx_texture,
    pub n_textures: i32,
    pub n_perlins: i32,
    pub perlins: *const rtx_perlin,
    pub images: *const rtx_image,
    pub n_images: i32,
    pub _pad: i32,
    pub background: [f64; 3],
    pub camera: rtx_camera,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_ray {
    pub origin: [f64; 3],
    pub direction: [f64; 3],
    pub time: f64,
    pub t_min: f64,
    pub t_max: f64,
    pub xi: f64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_hit {
    pub prim_id: i32,
    pub material: i32,
    pub front_face: i32,
    pub _pad: i32,
    pub t: f64,
    pub p: [f64; 3],
    pub normal: [f64; 3],
    pub u: f64,
    pub v: f64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_render_params {
    pub width: i32,
    pub height: i32,
    pub spp_begin: i32,
    pub spp_count: i32,
    pub max_depth: i32,
    pub _pad: i32,
    pub seed: u64,
}

/// Mean per-ray work counters of the traversal (`rtx_trace_rays_stats`, `rtx_render_counted`).
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct rtx_trace_stats {
    pub rays: f64,
    pub box_tests: f64,
    pub node_visits: f64,
    pub sphere_tests: f64,
    pub rect_tests: f64,
    pub instance_enters: f64,
    pub medium_tests: f64,
}
/// Adaptive sampling settings (`rtx_render_adaptive`); `rtx_render_params.spp_count` is the largest spp.
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct rtx_adaptive_params {
    pub threshold: f64,
    pub min_spp: i32,
    pub step_spp: i32,
}
/// What an adaptive render spent (`rtx_render_adaptive`).
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct rtx_adaptive_stats {
    pub path_samples: i64,
    pub rounds: i32,
    pub tiles: i32,
    pub tiles_converged: i32,
    pub tiles_at_max: i32,
}
/// Settings of the denoiser (`rtx_denoise`; the exact filter is written out in rttnw_b200.h).
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_denoise_params {
    pub iterations: i32,
    pub sigma_normal: f32,
    pub sigma_albedo: f32,
    pub sigma_luminance: f32,
}
impl Default for rtx_denoise_params {
    fn default() -> Self {
        rtx_denoise_params { iterations: 5, sigma_normal: 0.25, sigma_albedo: 0.1, sigma_luminance: 8.0 }
    }
}
/// The scene table of src/main.rs:66-183 and the defaults of :255.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtx_scene_defaults {
    pub width: i32,
    pub height: i32,
    pub samples: i32,
    pub max_depth: i32,
    pub name: *const c_char,
}

pub enum rtx_ctx {}
pub enum rtx_scene {}
pub enum rtx_comm {}

extern "C" {
    pub fn rtx_abi_version() -> c_int;
    pub fn rtx_last_error() -> *const c_char;
    pub fn rtx_device_count(count: *mut c_int) -> c_int;
    pub fn rtx_ctx_create(device: c_int, stream: *mut c_void, out: *mut *mut rtx_ctx) -> c_int;
    pub fn rtx_ctx_destroy(ctx: *mut rtx_ctx) -> c_int;
    pub fn rtx_ctx_sync(ctx: *mut rtx_ctx) -> c_int;
    pub fn rtx_ctx_set_async(ctx: *mut rtx_ctx, on: c_int) -> c_int;
    pub fn rtx_ctx_stream(ctx: *mut rtx_ctx) -> *mut c_void;
    pub fn rtx_ctx_set_bvh_builder(ctx: *mut rtx_ctx, kind: c_int) -> c_int;
    pub fn rtx_ctx_kernel_launches(ctx: *mut rtx_ctx, out: *mut u64) -> c_int;
    pub fn rtx_ctx_set_profiling(ctx: *mut rtx_ctx, on: c_int) -> c_int;
    pub fn rtx_ctx_profile_read(ctx: *mut rtx_ctx, shade_ms: *mut f64, trace_ms: *mut f64, iterations: *mut u64, reset: c_int) -> c_int;
    pub fn rtx_ctx_measure_l2_read(ctx: *mut rtx_ctx, bytes: u64, repeats: c_int, gbytes_per_s: *mut f64) -> c_int;
    pub fn rtx_scene_create(ctx: *mut rtx_ctx, desc: *const rtx_scene_desc, out: *mut *mut rtx_scene) -> c_int;
    pub fn rtx_scene_destroy(scene: *mut rtx_scene) -> c_int;
    pub fn rtx_cache_trim(device: c_int) -> c_int;
    pub fn rtx_scene_info(scene: *const rtx_scene, n_bvh_nodes: *mut i32, n_records: *mut i32, n_xform_ops: *mut i32, device_bytes: *mut i64) -> c_int;
    pub fn rtx_trace_rays(ctx: *mut rtx_ctx, scene: *const rtx_scene, n: i64, rays: *const rtx_ray, hits: *mut rtx_hit) -> c_int;
    pub fn rtx_trace_rays_device(ctx: *mut rtx_ctx, scene: *const rtx_scene, n: i64, d_rays: *const rtx_ray, d_hits: *mut rtx_hit) -> c_int;
    pub fn rtx_trace_rays_stats(ctx: *mut rtx_ctx, scene: *const rtx_scene, n: i64, d_rays: *const rtx_ray, out: *mut rtx_trace_stats) -> c_int;
    pub fn rtx_render(ctx: *mut rtx_ctx, scene: *const rtx_scene, params: *const rtx_render_params, d_accum: *mut f32, d_ray_count: *mut u64) -> c_int;
    pub fn rtx_render_counted(ctx: *mut rtx_ctx, scene: *const rtx_scene, params: *const rtx_render_params, d_accum: *mut f32, out: *mut rtx_trace_stats) -> c_int;
    pub fn rtx_render_adaptive(ctx: *mut rtx_ctx, scene: *const rtx_scene, params: *const rtx_render_params, adaptive: *const rtx_adaptive_params, d_accum: *mut f32, d_aux: *mut f32, stats: *mut rtx_adaptive_stats) -> c_int;
    pub fn rtx_adaptive_error(ctx: *mut rtx_ctx, d_accum: *const f32, d_aux: *const f32, width: i32, height: i32, d_tile_error: *mut f32) -> c_int;
    pub fn rtx_render_aov(ctx: *mut rtx_ctx, scene: *const rtx_scene, params: *const rtx_render_params, d_albedo: *mut f32, d_normal: *mut f32, d_depth: *mut f32) -> c_int;
    pub fn rtx_denoise(ctx: *mut rtx_ctx, d_accum: *const f32, d_half: *const f32, d_albedo: *const f32, d_normal: *const f32, width: i32, height: i32, params: *const rtx_denoise_params, d_out: *mut f32) -> c_int;
    pub fn rtx_tonemap_rgba8(ctx: *mut rtx_ctx, d_accum: *const f32, width: i32, height: i32, out: *mut u8, out_on_device: c_int) -> c_int;
    pub fn rtx_reduce_tonemap_peers(ctx: *mut rtx_ctx, d_accum: *mut f32, d_peer_accums: *const *const f32, n_peers: i32, width: i32, height: i32, d_rgba8: *mut u8) -> c_int;
    pub fn rtx_reduce_tonemap_slice(ctx: *mut rtx_ctx, d_accums: *const *const f32, n_ranks: i32, rank: i32, width: i32, height: i32, d_rgba8_root: *mut u8) -> c_int;
    pub fn rtx_comm_unique_id(id_out: *mut u8) -> c_int;
    pub fn rtx_comm_create(ctx: *mut rtx_ctx, n_ranks: i32, rank: i32, id: *const u8, out: *mut *mut rtx_comm) -> c_int;
    pub fn rtx_comm_wrap(nccl_comm: *mut c_void, out: *mut *mut rtx_comm) -> c_int;
    pub fn rtx_comm_destroy(comm: *mut rtx_comm) -> c_int;
    pub fn rtx_accum_reduce(ctx: *mut rtx_ctx, comm: *mut rtx_comm, d_accum: *mut f32, width: i32, height: i32, root: i32) -> c_int;
    pub fn rtx_malloc(ctx: *mut rtx_ctx, bytes: usize, out: *mut *mut c_void) -> c_int;
    pub fn rtx_free(ctx: *mut rtx_ctx, ptr: *mut c_void) -> c_int;
    pub fn rtx_memset_zero(ctx: *mut rtx_ctx, ptr: *mut c_void, bytes: usize) -> c_int;
    pub fn rtx_memcpy_h2d(ctx: *mut rtx_ctx, dst: *mut c_void, src: *const c_void, bytes: usize) -> c_int;
    pub fn rtx_memcpy_d2h(ctx: *mut rtx_ctx, dst: *mut c_void, src: *const c_void, bytes: usize) -> c_int;
    pub fn rtx_memcpy_d2d(ctx: *mut rtx_ctx, dst: *mut c_void, src: *const c_void, bytes: usize) -> c_int;
    pub fn rtx_ipc_export(ctx: *mut rtx_ctx, d_ptr: *mut c_void, handle_out: *mut u8) -> c_int;
    pub fn rtx_ipc_open(ctx: *mut rtx_ctx, handle: *const u8, d_ptr_out: *mut *mut c_void) -> c_int;
    pub fn rtx_ipc_close(ctx: *mut rtx_ctx, d_ptr: *mut c_void) -> c_int;
    pub fn rtx_builtin_scene_defaults(scene_number: c_int, out: *mut rtx_scene_defaults) -> c_int;
    pub fn rtx_builtin_scene(scene_number: c_int, seed: u64, earth_png_path: *const c_char, out: *mut *mut rtx_scene_desc) -> c_int;
    pub fn rtx_scene_desc_free(desc: *mut rtx_scene_desc) -> c_int;
    pub fn rtx_flatten_check(desc: *const rtx_scene_desc, n_bvh_nodes: *mut i32, n_records: *mut i32, n_prim_ids: *mut i32) -> c_int;
    pub fn rtx_png_read_rgba8(path: *const c_char, width: *mut i32, height: *mut i32, rgba_out: *mut *mut u8) -> c_int;
    pub fn rtx_png_write_rgba8(path: *const c_char, width: i32, height: i32, rgba: *const u8) -> c_int;
    pub fn rtx_pfm_write(path: *const c_char, width: i32, height: i32, channels: i32, data: *const f32) -> c_int;
    pub fn rtx_buffer_free(p: *mut c_void) -> c_int;
}
