//! Raw bindings to `include/rtiow_cuda.h` (ABI version 4).  One `extern "C"` item per exported symbol, one
//! `#[repr(C)]` struct per C struct; layouts are asserted in `tests/test_host_cabi.py::test_struct_layouts_match_header`
//! (Camera 176 B, Params 48 B, Stats 72 B, Spheres/Materials 48 B).
//!
//! NOT compiled in this repository's build container (no rustc).  `tests/test_rust_header_lock.py` parses this file and the
//! header and fails when symbol names, argument counts, struct field order or the constants drift apart.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const RTIOW_ABI_VERSION: c_int = 4;

pub const RTIOW_OK: c_int = 0;
pub const RTIOW_ERR_INVALID_ARG: c_int = -1;
pub const RTIOW_ERR_UNSUPPORTED: c_int = -2;
pub const RTIOW_ERR_CUDA: c_int = -3;
pub const RTIOW_ERR_NCCL: c_int = -4;
pub const RTIOW_ERR_NO_DEVICE: c_int = -5;
pub const RTIOW_ERR_NOMEM: c_int = -6;
pub const RTIOW_ERR_CANCELLED: c_int = -7;

pub const RTIOW_MAT_LAMBERTIAN: u32 = 0;
pub const RTIOW_MAT_METAL: u32 = 1;
pub const RTIOW_MAT_DIELECTRIC: u32 = 2;

pub const RTIOW_PRECISION_F32: u8 = 0;
pub const RTIOW_PRECISION_F64: u8 = 1;

pub const RTIOW_SCAN_AUTO: c_int = 0;
pub const RTIOW_SCAN_FP32: c_int = 1;
pub const RTIOW_SCAN_TENSOR: c_int = 2;

pub const RTIOW_GATHER_AUTO: c_int = 0;
pub const RTIOW_GATHER_NCCL: c_int = 1;
pub const RTIOW_GATHER_FUSED: c_int = 2;
pub const RTIOW_NCCL_UNIQUE_ID_BYTES: usize = 128;

#[repr(C)]
pub struct rtiow_ctx { _private: [u8; 0] }

#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtiow_spheres {
    pub cx: *const f64, pub cy: *const f64, pub cz: *const f64,
    pub radius: *const f64,
    pub mat_index: *const u32,
    pub n: u32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtiow_materials {
    pub kind: *const u32,
    pub albedo_r: *const f64, pub albedo_g: *const f64, pub albedo_b: *const f64,
    pub param: *const f64,
    pub n: u32,
}

/// The 8 private fields of `Camera` (camera.rs:4-13).
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct rtiow_camera {
    pub origin: [f64; 3], pub lower_left_corner: [f64; 3], pub horizontal: [f64; 3], pub vertical: [f64; 3],
    pub u: [f64; 3], pub v: [f64; 3], pub w: [f64; 3],
    pub lens_radius: f64,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct rtiow_params {
    pub width: u32, pub height: u32, pub spp: u32,
    pub max_depth: i32,
    pub t_min: f64,
    pub seed: u64,
    pub alpha: u8, pub precision: u8, pub reserved: [u8; 6],
    pub tile_rows: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct rtiow_stats {
    pub kernel_ms: f64, pub total_ms: f64,
    pub paths: u64, pub rays_traced: u64, pub sphere_tests: u64, pub h2d_bytes: u64, pub d2h_bytes: u64,
    pub kernel_launches: u32, pub n_gpus: u32, pub scan_backend: u32, pub reserved: u32,
}

/// int (*)(void* user, uint32_t pass, uint32_t n_passes, uint32_t spp_done, const uint8_t* rgba); non-zero return cancels
pub type rtiow_progress_fn = unsafe extern "C" fn(user: *mut c_void, pass: u32, n_passes: u32, spp_done: u32, rgba: *const u8) -> c_int;

extern "C" {
    pub fn rtiow_abi_version() -> c_int;
    pub fn rtiow_last_error() -> *const c_char;
    pub fn rtiow_device_count(out_count: *mut c_int) -> c_int;
    pub fn rtiow_ctx_create(n_gpus: c_int, out: *mut *mut rtiow_ctx) -> c_int;
    pub fn rtiow_ctx_create_on_device(device: c_int, out: *mut *mut rtiow_ctx) -> c_int;
    pub fn rtiow_ctx_destroy(ctx: *mut rtiow_ctx);
    pub fn rtiow_ctx_set_scan_backend(ctx: *mut rtiow_ctx, backend: c_int) -> c_int;
    pub fn rtiow_ctx_set_filter_bypass(ctx: *mut rtiow_ctx, on: c_int) -> c_int;
    pub fn rtiow_nccl_unique_id(out_id: *mut c_void) -> c_int;
    pub fn rtiow_ctx_create_rank(device: c_int, rank: c_int, world: c_int, nccl_unique_id: *const c_void, out: *mut *mut rtiow_ctx) -> c_int;
    pub fn rtiow_ctx_set_stream(ctx: *mut rtiow_ctx, stream: *mut c_void) -> c_int;
    pub fn rtiow_ctx_set_gather(ctx: *mut rtiow_ctx, mode: c_int) -> c_int;
    pub fn rtiow_ctx_gather_info(ctx: *mut rtiow_ctx, buf: *mut c_char, n: usize) -> c_int;
    pub fn rtiow_scene_upload(ctx: *mut rtiow_ctx, spheres: *const rtiow_spheres, materials: *const rtiow_materials) -> c_int;
    pub fn rtiow_camera_new(look_from: *const f64, look_at: *const f64, v_up: *const f64, v_fov_deg: f64, aspect_ratio: f64,
                            aperture: f64, focus_dist: f64, out: *mut rtiow_camera) -> c_int;
    pub fn rtiow_params_default(p: *mut rtiow_params);
    pub fn rtiow_render(ctx: *mut rtiow_ctx, cam: *const rtiow_camera, p: *const rtiow_params, out_rgba: *mut u8,
                        stats: *mut rtiow_stats) -> c_int;
    pub fn rtiow_render_aov(ctx: *mut rtiow_ctx, cam: *const rtiow_camera, p: *const rtiow_params, out_rgba: *mut u8, out_color: *mut f32,
                            out_albedo: *mut f32, out_normal: *mut f32, out_depth: *mut f32, stats: *mut rtiow_stats) -> c_int;
    pub fn rtiow_render_adaptive(ctx: *mut rtiow_ctx, cam: *const rtiow_camera, p: *const rtiow_params, min_spp: u32, tolerance: f64,
                                 out_rgba: *mut u8, out_spp: *mut u32, out_error: *mut f32, stats: *mut rtiow_stats) -> c_int;
    pub fn rtiow_render_views(ctx: *mut rtiow_ctx, cams: *const rtiow_camera, n_views: u32, p: *const rtiow_params, out_rgba: *mut u8,
                              stats: *mut rtiow_stats) -> c_int;
    pub fn rtiow_render_progressive(ctx: *mut rtiow_ctx, cam: *const rtiow_camera, p: *const rtiow_params, n_passes: u32,
                                    on_pass: Option<rtiow_progress_fn>, user: *mut c_void, out_rgba: *mut u8, stats: *mut rtiow_stats) -> c_int;
    pub fn rtiow_render_rank(ctx: *mut rtiow_ctx, cam: *const rtiow_camera, p: *const rtiow_params, out_rgba: *mut u8, stats: *mut rtiow_stats) -> c_int;
    pub fn rtiow_render_rank_device(ctx: *mut rtiow_ctx, cam: *const rtiow_camera, p: *const rtiow_params, d_frame: *mut *const c_void,
                                    stats: *mut rtiow_stats) -> c_int;
    pub fn rtiow_render_rank_enqueue(ctx: *mut rtiow_ctx, cam: *const rtiow_camera, p: *const rtiow_params, d_frame: *mut *const c_void) -> c_int;
    pub fn rtiow_ctx_synchronize(ctx: *mut rtiow_ctx, stats: *mut rtiow_stats) -> c_int;
    pub fn rtiow_tile_buffer_bytes(p: *const rtiow_params, world: c_int, out_bytes: *mut usize) -> c_int;
    pub fn rtiow_render_tiles_device(ctx: *mut rtiow_ctx, cam: *const rtiow_camera, p: *const rtiow_params, rank: c_int, world: c_int,
                                     d_tiles: *mut c_void, stream: *mut c_void, stats: *mut rtiow_stats) -> c_int;
    pub fn rtiow_render_to_frame_device(ctx: *mut rtiow_ctx, cam: *const rtiow_camera, p: *const rtiow_params, rank: c_int, world: c_int,
                                        d_frame: *mut c_void, stream: *mut c_void, stats: *mut rtiow_stats) -> c_int;
    pub fn rtiow_deinterleave_device(ctx: *mut rtiow_ctx, d_gathered: *const c_void, p: *const rtiow_params, world: c_int,
                                     d_frame: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn rtiow_sphere_hit_batch(ctx: *mut rtiow_ctx, precision: c_int, n: i64, center: *const f64, radius: *const f64, orig: *const f64,
                                  dir: *const f64, t_min: *const f64, t_max: *const f64, hit: *mut i32, t: *mut f64, p: *mut f64,
                                  normal: *mut f64, front_face: *mut i32) -> c_int;
    pub fn rtiow_hitlist_batch(ctx: *mut rtiow_ctx, precision: c_int, n: i64, orig: *const f64, dir: *const f64, t_min: f64, hit: *mut i32,
                               index: *mut i32, t: *mut f64, p: *mut f64, normal: *mut f64, front_face: *mut i32) -> c_int;
    pub fn rtiow_scatter_batch(ctx: *mut rtiow_ctx, precision: c_int, n: i64, kind: *const i32, albedo: *const f64, param: *const f64,
                               r_orig: *const f64, r_dir: *const f64, p: *const f64, normal: *const f64, front_face: *const i32,
                               sample: *const f64, some: *mut i32, attenuation: *mut f64, s_orig: *mut f64, s_dir: *mut f64) -> c_int;
    pub fn rtiow_get_ray_batch(ctx: *mut rtiow_ctx, precision: c_int, cam: *const rtiow_camera, n: i64, s: *const f64, t: *const f64,
                               disk_xy: *const f64, orig: *mut f64, dir: *mut f64) -> c_int;
    pub fn rtiow_to_rgba_batch(ctx: *mut rtiow_ctx, precision: c_int, n: i64, color: *const f64, alpha: u8, spp: u64, out_rgba: *mut u8) -> c_int;
    pub fn rtiow_reflect_batch(ctx: *mut rtiow_ctx, precision: c_int, n: i64, v: *const f64, nrm: *const f64, out: *mut f64) -> c_int;
    pub fn rtiow_refract_batch(ctx: *mut rtiow_ctx, precision: c_int, n: i64, uv: *const f64, nrm: *const f64, eta: *const f64, out: *mut f64) -> c_int;
    pub fn rtiow_ray_color_batch(ctx: *mut rtiow_ctx, precision: c_int, n: i64, orig: *const f64, dir: *const f64, pixel: *const u32,
                                 sample: *const u32, seed: u64, max_depth: i32, t_min: f64, color: *mut f64, rays: *mut u64) -> c_int;
    pub fn rtiow_ray_color_trace_batch(ctx: *mut rtiow_ctx, precision: c_int, n: i64, orig: *const f64, dir: *const f64, pixel: *const u32,
                                       sample: *const u32, seed: u64, max_depth: i32, t_min: f64, color: *mut f64, rays: *mut u64,
                                       trace_index: *mut i32, trace_ray: *mut f64) -> c_int;
    pub fn rtiow_sampler_batch(ctx: *mut rtiow_ctx, precision: c_int, n: i64, pixel: *const u32, sample: *const u32, bounce: *const u32,
                               seed: u64, out: *mut f64) -> c_int;
    pub fn rtiow_fp32_peak_probe(ctx: *mut rtiow_ctx, packed: c_int, target_ms: f64, out_tflops: *mut f64, out_ms: *mut f64) -> c_int;
    pub fn rtiow_flush_l2(ctx: *mut rtiow_ctx) -> c_int;
    pub fn rtiow_random_scene(seed: u64, half_extent: i32, material_mode: i32, cap: u32, cx: *mut f64, cy: *mut f64, cz: *mut f64,
                              radius: *mut f64, mat_kind: *mut u32, albedo_rgb: *mut f64, mat_param: *mut f64, out_n: *mut u32) -> c_int;
    pub fn rtiow_scene_save(path: *const c_char, n: u32, cx: *const f64, cy: *const f64, cz: *const f64, radius: *const f64,
                            mat_kind: *const u32, albedo_rgb: *const f64, mat_param: *const f64) -> c_int;
    pub fn rtiow_scene_load(path: *const c_char, cap: u32, cx: *mut f64, cy: *mut f64, cz: *mut f64, radius: *mut f64, mat_kind: *mut u32,
                            albedo_rgb: *mut f64, mat_param: *mut f64, out_n: *mut u32) -> c_int;
}
