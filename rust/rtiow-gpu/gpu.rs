//! gpu.rs — drop this file into the reference crate as `src/gpu.rs` (`pub mod gpu;` in main.rs) together with the
//! four small additions listed in INTEGRATION.md.  It adds ONE call, `gpu::render`, that replaces the rayon pixel loop,
//! the collect and the row flip of main.rs:122-145 with the B200 backend.  Everything else in the crate is unchanged:
//! `Hit::hit`, `Scatter::scatter` and `Camera::get_ray` keep working on the CPU for callers that use them directly,
//! but `render` never falls back to them.
//!
//! NOT compiled in this repository's build container (no rustc/cargo there).
use std::ffi::CStr;
use std::ptr;

use rtiow_cuda_sys as sys;

use crate::camera::Camera;
use crate::shapes::HittableList;

/// What `Hit::describe` returns for a shape the GPU knows (only spheres exist in the reference, shapes/sphere.rs:9-13).
pub struct SphereDesc { pub center: [f64; 3], pub radius: f64, pub mat: std::sync::Arc<dyn crate::materials::Scatter> }

/// What `Scatter::describe` returns (materials.rs:9-11,34-37,64-66).  `param` = fuzz (Metal) or ir (Dialectric).
#[derive(Clone, Copy)]
pub struct MaterialDesc { pub kind: u32, pub albedo: [f64; 3], pub param: f64 }

/// Runtime form of the compile-time constants main.rs:24-28,44,137.
#[derive(Clone, Debug)]
pub struct RenderParams {
    pub width: u32, pub height: u32, pub spp: u32, pub max_depth: i32, pub t_min: f64,
    pub seed: u64, pub n_gpus: i32, pub alpha: u8,
}

impl Default for RenderParams {
    fn default() -> Self {       // IMAGE_WIDTH 200, 3:2 -> 133 rows, 100 spp, depth 50, t_min 0.0001, alpha 255
        RenderParams { width: 200, height: 133, spp: 100, max_depth: 50, t_min: 0.0001, seed: 1, n_gpus: 1, alpha: 255 }
    }
}

#[derive(Debug)]
pub enum RenderError { InvalidArg(String), Unsupported(String), Cuda(String), Nccl(String), NoDevice(String), NoMem(String), Cancelled(String) }

fn err(code: i32) -> RenderError {
    let msg = unsafe { CStr::from_ptr(sys::rtiow_last_error()) }.to_string_lossy().into_owned();
    match code {
        sys::RTIOW_ERR_UNSUPPORTED => RenderError::Unsupported(msg),
        sys::RTIOW_ERR_CUDA => RenderError::Cuda(msg),
        sys::RTIOW_ERR_NCCL => RenderError::Nccl(msg),
        sys::RTIOW_ERR_NO_DEVICE => RenderError::NoDevice(msg),
        sys::RTIOW_ERR_NOMEM => RenderError::NoMem(msg),
        sys::RTIOW_ERR_CANCELLED => RenderError::Cancelled(msg),
        _ => RenderError::InvalidArg(msg),
    }
}

struct Ctx(*mut sys::rtiow_ctx);
impl Drop for Ctx { fn drop(&mut self) { unsafe { sys::rtiow_ctx_destroy(self.0) } } }   // Send, !Sync: one caller per ctx

/// Replaces main.rs:122-145.  Returns top-down RGBA8, `4*width*height` bytes: exactly the `Vec<u8>` handed to
/// `ImageBuffer::from_vec(IMAGE_WIDTH, IMAGE_HEIGHT, pixels)` at main.rs:147.
pub fn render(cam: &Camera, world: &HittableList, p: &RenderParams) -> Result<Vec<u8>, RenderError> {
    render_impl(cam, world, p, 0, None)
}

/// Many cameras of one world in one call (a turntable, a stereo pair, a camera sweep): the views' top-down RGBA8 frames one
/// after the other, `4*width*height` bytes each.  Frame `v` is byte-identical to `render(&cams[v], world, p)`.
pub fn render_views(cams: &[Camera], world: &HittableList, p: &RenderParams) -> Result<Vec<u8>, RenderError> {
    unsafe {
        let mut raw: *mut sys::rtiow_ctx = ptr::null_mut();
        let rc = sys::rtiow_ctx_create(p.n_gpus, &mut raw);
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        let ctx = Ctx(raw);
        upload(&ctx, world)?;
        let prm = raw_params(p);
        let raw_cams: Vec<sys::rtiow_camera> = cams.iter().map(|c| c.raw()).collect();
        let mut pixels = vec![0u8; 4 * p.width as usize * p.height as usize * cams.len()];
        let rc = sys::rtiow_render_views(ctx.0, raw_cams.as_ptr(), cams.len() as u32, &prm, pixels.as_mut_ptr(), ptr::null_mut());
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        Ok(pixels)
    }
}

/// The float buffers of `render_aov`, top-down: `color`, `albedo` and `normal` hold 3 floats per pixel, `depth` one.
pub struct Aovs { pub color: Vec<f32>, pub albedo: Vec<f32>, pub normal: Vec<f32>, pub depth: Vec<f32> }

/// `render`'s frame, byte for byte, plus the float buffers a denoiser takes: linear colour, and the albedo, normal and distance of
/// each camera ray's first hit, averaged over the samples (include/rtiow_cuda.h, rtiow_render_aov).
pub fn render_aov(cam: &Camera, world: &HittableList, p: &RenderParams) -> Result<(Vec<u8>, Aovs), RenderError> {
    unsafe {
        let mut raw: *mut sys::rtiow_ctx = ptr::null_mut();
        let rc = sys::rtiow_ctx_create(p.n_gpus, &mut raw);
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        let ctx = Ctx(raw);
        upload(&ctx, world)?;
        let prm = raw_params(p);
        let n = p.width as usize * p.height as usize;
        let mut pixels = vec![0u8; 4 * n];
        let mut a = Aovs { color: vec![0.0; 3 * n], albedo: vec![0.0; 3 * n], normal: vec![0.0; 3 * n], depth: vec![0.0; n] };
        let rc = sys::rtiow_render_aov(ctx.0, &cam.raw(), &prm, pixels.as_mut_ptr(), a.color.as_mut_ptr(), a.albedo.as_mut_ptr(),
                                       a.normal.as_mut_ptr(), a.depth.as_mut_ptr(), ptr::null_mut());
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        Ok((pixels, a))
    }
}

/// Adaptive sampling: each pixel gets between `min_spp` and `p.spp` samples, as many as its own noise asks for, and is
/// byte-identical to `render` at its own count.  Returns the frame, each pixel's count and its error at the last boundary it
/// reached (one standard error of the displayed value in 8-bit levels; include/rtiow_cuda.h, rtiow_render_adaptive).
pub fn render_adaptive(cam: &Camera, world: &HittableList, p: &RenderParams, min_spp: u32, tolerance: f64)
                       -> Result<(Vec<u8>, Vec<u32>, Vec<f32>), RenderError> {
    unsafe {
        let mut raw: *mut sys::rtiow_ctx = ptr::null_mut();
        let rc = sys::rtiow_ctx_create(p.n_gpus, &mut raw);
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        let ctx = Ctx(raw);
        upload(&ctx, world)?;
        let prm = raw_params(p);
        let n = p.width as usize * p.height as usize;
        let mut pixels = vec![0u8; 4 * n];
        let mut spp = vec![0u32; n];
        let mut error = vec![0.0f32; n];
        let rc = sys::rtiow_render_adaptive(ctx.0, &cam.raw(), &prm, min_spp, tolerance, pixels.as_mut_ptr(), spp.as_mut_ptr(),
                                            error.as_mut_ptr(), ptr::null_mut());
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        Ok((pixels, spp, error))
    }
}

/// The parameters of `denoise`: the defaults the library chose on the final scene (`rtiow_denoise_params_default`).
pub fn default_denoise_params() -> sys::rtiow_denoise_params {
    let mut dp = sys::rtiow_denoise_params::default();
    unsafe { sys::rtiow_denoise_params_default(&mut dp) };
    dp
}

/// An edge-avoiding a-trous denoiser over `render_aov`'s buffers (include/rtiow_cuda.h, rtiow_denoise): returns the denoised
/// linear colour (3 floats per pixel) and its top-down RGBA8 frame.  Runs on GPU 0 and needs no scene.
pub fn denoise(width: u32, height: u32, aovs: &Aovs, dp: &sys::rtiow_denoise_params) -> Result<(Vec<f32>, Vec<u8>), RenderError> {
    let n = width as usize * height as usize;
    if aovs.color.len() != 3 * n || aovs.albedo.len() != 3 * n || aovs.normal.len() != 3 * n || aovs.depth.len() != n {
        return Err(RenderError::InvalidArg("denoise: AOV buffers do not match width x height".into()));
    }
    unsafe {
        let mut raw: *mut sys::rtiow_ctx = ptr::null_mut();
        let rc = sys::rtiow_ctx_create(1, &mut raw);
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        let ctx = Ctx(raw);
        let mut color = vec![0.0f32; 3 * n];
        let mut pixels = vec![0u8; 4 * n];
        let rc = sys::rtiow_denoise(ctx.0, width, height, aovs.color.as_ptr(), aovs.albedo.as_ptr(), aovs.normal.as_ptr(), aovs.depth.as_ptr(),
                                    dp, color.as_mut_ptr(), pixels.as_mut_ptr(), ptr::null_mut());
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        Ok((color, pixels))
    }
}

/// `render_aov` and `denoise` in one call, the AOVs kept on the GPU (include/rtiow_cuda.h, rtiow_render_denoised): returns the
/// denoised linear colour (3 floats per pixel) and its top-down RGBA8 frame, both bit-identical to `denoise` over `render_aov`'s
/// buffers.
pub fn render_denoised(cam: &Camera, world: &HittableList, p: &RenderParams, dp: &sys::rtiow_denoise_params)
                       -> Result<(Vec<f32>, Vec<u8>), RenderError> {
    unsafe {
        let mut raw: *mut sys::rtiow_ctx = ptr::null_mut();
        let rc = sys::rtiow_ctx_create(p.n_gpus, &mut raw);
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        let ctx = Ctx(raw);
        upload(&ctx, world)?;
        let prm = raw_params(p);
        let n = p.width as usize * p.height as usize;
        let mut color = vec![0.0f32; 3 * n];
        let mut pixels = vec![0u8; 4 * n];
        let rc = sys::rtiow_render_denoised(ctx.0, &cam.raw(), &prm, dp, color.as_mut_ptr(), pixels.as_mut_ptr(), ptr::null_mut());
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        Ok((color, pixels))
    }
}

/// The same frame in `n_passes` slices of the samples, with the frame so far handed to `on_pass(pass, n_passes, spp_done, rgba)`
/// after each — the role of the indicatif bar (main.rs:120,124) and the piston preview window (main.rs:151-171).  The returned
/// frame is bit-identical to `render`'s.  `on_pass` returning `true` stops the render: `Err(RenderError::Cancelled)`.
pub fn render_progressive(cam: &Camera, world: &HittableList, p: &RenderParams, n_passes: u32,
                          on_pass: &mut dyn FnMut(u32, u32, u32, &[u8]) -> bool) -> Result<Vec<u8>, RenderError> {
    render_impl(cam, world, p, n_passes.max(1), Some(on_pass))
}

struct Progress<'a> { f: &'a mut dyn FnMut(u32, u32, u32, &[u8]) -> bool, len: usize }
unsafe extern "C" fn progress_trampoline(user: *mut std::os::raw::c_void, pass: u32, n_passes: u32, spp_done: u32, rgba: *const u8) -> std::os::raw::c_int {
    let p = &mut *(user as *mut Progress);
    (p.f)(pass, n_passes, spp_done, std::slice::from_raw_parts(rgba, p.len)) as std::os::raw::c_int
}

/// One process per GPU (MPI ranks, one Rust process per device): rank 0 makes the id, hands its 128 bytes to the other ranks by
/// any means, and every rank calls `render_rank` with the same camera, world and params.  The gather happens inside
/// librtiow_cuda.so (one ncclAllGather per frame, or epilogue stores into rank 0's frame over NVLink): rank 0 gets
/// `Some(pixels)`, the others `None`.  The frame is byte-identical to `render`'s on one GPU.
pub fn nccl_unique_id() -> Result<[u8; 128], RenderError> {
    let mut id = [0u8; 128];
    let rc = unsafe { sys::rtiow_nccl_unique_id(id.as_mut_ptr() as *mut std::os::raw::c_void) };
    if rc != sys::RTIOW_OK { return Err(err(rc)); }
    Ok(id)
}

pub fn render_rank(cam: &Camera, world: &HittableList, p: &RenderParams, device: i32, rank: i32, ranks: i32,
                   nccl_id: &[u8; 128]) -> Result<Option<Vec<u8>>, RenderError> {
    unsafe {
        let mut raw: *mut sys::rtiow_ctx = ptr::null_mut();
        let rc = sys::rtiow_ctx_create_rank(device, rank, ranks, nccl_id.as_ptr() as *const std::os::raw::c_void, &mut raw);
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        let ctx = Ctx(raw);
        upload(&ctx, world)?;
        let prm = raw_params(p);
        let mut pixels = if rank == 0 { vec![0u8; 4 * p.width as usize * p.height as usize] } else { vec![] };
        let out = if rank == 0 { pixels.as_mut_ptr() } else { ptr::null_mut() };
        let rc = sys::rtiow_render_rank(ctx.0, &cam.raw(), &prm, out, ptr::null_mut());
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        Ok(if rank == 0 { Some(pixels) } else { None })
    }
}

unsafe fn raw_params(p: &RenderParams) -> sys::rtiow_params {
    let mut prm: sys::rtiow_params = std::mem::zeroed();
    sys::rtiow_params_default(&mut prm);
    prm.width = p.width; prm.height = p.height; prm.spp = p.spp; prm.max_depth = p.max_depth; prm.t_min = p.t_min;
    prm.seed = p.seed; prm.alpha = p.alpha;
    prm
}

/// `&world` (main.rs:62-99) -> SoA arrays -> rtiow_scene_upload
unsafe fn upload(ctx: &Ctx, world: &HittableList) -> Result<(), RenderError> {
    // flatten the trait objects through the provided describe() methods; unknown ones are an error, not a CPU fallback
    let (mut cx, mut cy, mut cz, mut radius, mut mat_index) = (vec![], vec![], vec![], vec![], vec![]);
    let (mut kind, mut ar, mut ag, mut ab, mut param) = (vec![], vec![], vec![], vec![], vec![]);
    let mut seen: Vec<*const ()> = vec![];
    for shape in world.iter() {
        let s = shape.describe().ok_or_else(|| RenderError::Unsupported("shape without a GPU description".into()))?;
        let m = s.mat.describe().ok_or_else(|| RenderError::Unsupported("material without a GPU description".into()))?;
        let key = std::sync::Arc::as_ptr(&s.mat) as *const ();
        let id = match seen.iter().position(|k| *k == key) {
            Some(i) => i,
            None => { seen.push(key); kind.push(m.kind); ar.push(m.albedo[0]); ag.push(m.albedo[1]); ab.push(m.albedo[2]); param.push(m.param); seen.len() - 1 }
        };
        cx.push(s.center[0]); cy.push(s.center[1]); cz.push(s.center[2]); radius.push(s.radius); mat_index.push(id as u32);
    }
    {
        let spheres = sys::rtiow_spheres { cx: cx.as_ptr(), cy: cy.as_ptr(), cz: cz.as_ptr(), radius: radius.as_ptr(), mat_index: mat_index.as_ptr(), n: radius.len() as u32 };
        let mats = sys::rtiow_materials { kind: kind.as_ptr(), albedo_r: ar.as_ptr(), albedo_g: ag.as_ptr(), albedo_b: ab.as_ptr(), param: param.as_ptr(), n: kind.len() as u32 };
        let rc = sys::rtiow_scene_upload(ctx.0, &spheres, &mats);
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        Ok(())
    }
}

fn render_impl(cam: &Camera, world: &HittableList, p: &RenderParams, n_passes: u32,
               on_pass: Option<&mut dyn FnMut(u32, u32, u32, &[u8]) -> bool>) -> Result<Vec<u8>, RenderError> {
    unsafe {
        let mut raw: *mut sys::rtiow_ctx = ptr::null_mut();
        let rc = sys::rtiow_ctx_create(p.n_gpus, &mut raw);
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        let ctx = Ctx(raw);
        upload(&ctx, world)?;
        let prm = raw_params(p);
        let mut pixels = vec![0u8; 4 * p.width as usize * p.height as usize];
        let rc = match on_pass {
            None if n_passes == 0 => sys::rtiow_render(ctx.0, &cam.raw(), &prm, pixels.as_mut_ptr(), ptr::null_mut()),
            None => sys::rtiow_render_progressive(ctx.0, &cam.raw(), &prm, n_passes, None, ptr::null_mut(), pixels.as_mut_ptr(), ptr::null_mut()),
            Some(f) => {
                let mut pr = Progress { f, len: pixels.len() };
                sys::rtiow_render_progressive(ctx.0, &cam.raw(), &prm, n_passes, Some(progress_trampoline),
                                              &mut pr as *mut Progress as *mut std::os::raw::c_void, pixels.as_mut_ptr(), ptr::null_mut())
            }
        };
        if rc != sys::RTIOW_OK { return Err(err(rc)); }
        Ok(pixels)
    }
}
