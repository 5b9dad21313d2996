/*
 * rtiow_cuda.h — C ABI of librtiow_cuda.so: the B200 (sm_100a) render backend for Druthyn/rtiow.
 *
 * The reference has no FFI/plugin interface: it is one Rust binary whose render loop
 * (/root/reference/src/main.rs:122-145) calls private functions.  This header IS the drop-in
 * boundary: one call, rtiow_render(), replaces main.rs:122-145, and the scene/camera structs
 * below carry exactly the private fields of the reference's types.  A Rust `-sys` crate binds these
 * symbols 1:1 (INTEGRATION.md); the C++ host mirror (rtiow_b200/host/rtiow.hpp) and the ctypes
 * binding (rtiow_b200/capi.py) are the callers exercised here, because this image has no rustc.
 *
 * Conventions: plain pointers and sizes only; host-facing scalars are double (the Rust side is
 * f64) and are narrowed inside the library; every function returns RTIOW_OK (0) or a negative
 * rtiow_status and never aborts or throws (contrast main.rs:147,156,177 unwrap/panic);
 * rtiow_last_error() returns a thread-local message.  The caller owns every host buffer; the
 * library owns the ctx.  A ctx is single-caller (Send, !Sync).  There is NO CPU fallback: with no
 * CUDA device every compute entry point returns RTIOW_ERR_NO_DEVICE.
 */
#ifndef RTIOW_CUDA_H
#define RTIOW_CUDA_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTIOW_ABI_VERSION 4

typedef enum {
    RTIOW_OK = 0,
    RTIOW_ERR_INVALID_ARG = -1,
    RTIOW_ERR_UNSUPPORTED = -2,   /* shape/material the GPU path does not know: no CPU fallback */
    RTIOW_ERR_CUDA = -3,
    RTIOW_ERR_NCCL = -4,
    RTIOW_ERR_NO_DEVICE = -5,
    RTIOW_ERR_NOMEM = -6,
    RTIOW_ERR_CANCELLED = -7      /* rtiow_render_progressive: the callback asked to stop; out_rgba holds the frame so far */
} rtiow_status;

/* materials.rs:9-11 (Lambertian), 34-37 (Metal), 64-66 (Dialectric) */
typedef enum { RTIOW_MAT_LAMBERTIAN = 0, RTIOW_MAT_METAL = 1, RTIOW_MAT_DIELECTRIC = 2 } rtiow_material_kind;

/* arithmetic the render runs in.  F32 is the product path; F64 restates the reference's f64
 * arithmetic on the GPU for parity triage (same kernels, real_t = double). */
typedef enum { RTIOW_PRECISION_F32 = 0, RTIOW_PRECISION_F64 = 1 } rtiow_precision;

/* Where the sphere FILTER of the F32 scan runs (HittableList::hit, shapes/mod.rs:56-69: every ray against every sphere).
 * FP32: 7 packed FFMA2 per sphere pair on the CUDA cores.  TENSOR: the discriminant as a [rays x 11] x [11 x spheres]
 * contraction on the tcgen05 tensor cores (fp16 hi/lo split, fp32 accumulate in TMEM).  Both are conservative filters in
 * front of the SAME precise test, so hits, images and ray counts are identical bit for bit.  AUTO = TENSOR when the scene
 * qualifies (its small spheres fit one CTA's shared memory), else FP32. */
typedef enum { RTIOW_SCAN_AUTO = 0, RTIOW_SCAN_FP32 = 1, RTIOW_SCAN_TENSOR = 2 } rtiow_scan_backend;

/* HittableList of Sphere (shapes/mod.rs:52, shapes/sphere.rs:9-13) as a structure of arrays,
 * in LIST ORDER (order decides exact-tie hits: later index wins, sphere.rs:29,31 + mod.rs:61-66).
 * radius may be negative (sphere.rs:45-51 does not validate; flips the outward normal). */
typedef struct {
    const double* cx; const double* cy; const double* cz;   /* Sphere.center */
    const double* radius;                                   /* Sphere.radius */
    const uint32_t* mat_index;                              /* Sphere.mat -> index into rtiow_materials */
    uint32_t n;
} rtiow_spheres;

/* Arc<dyn Scatter> records (materials.rs).  param = fuzz (Metal, NOT clamped, materials.rs:40-45)
 * or ir (Dialectric); ignored for Lambertian.  albedo ignored for Dialectric.
 * The albedo of a Lambertian or Metal material and the param of a Metal or Dialectric one must be finite when a sphere
 * uses the material (RTIOW_ERR_INVALID_ARG otherwise), as the sphere centres and radii must; ignored fields may be anything. */
typedef struct {
    const uint32_t* kind;                                   /* rtiow_material_kind */
    const double* albedo_r; const double* albedo_g; const double* albedo_b;
    const double* param;
    uint32_t n;
} rtiow_materials;

/* The 8 private fields of Camera (camera.rs:4-13), as Camera::new leaves them. */
typedef struct {
    double origin[3], lower_left_corner[3], horizontal[3], vertical[3], u[3], v[3], w[3];
    double lens_radius;
} rtiow_camera;

/* Runtime replacement of the compile-time constants main.rs:24-28,44,137. */
typedef struct {
    uint32_t width, height;       /* IMAGE_WIDTH / IMAGE_HEIGHT (main.rs:25-26); both >= 2 */
    uint32_t spp;                 /* SAMPLES_PER_PIXEL (main.rs:27) */
    int32_t  max_depth;           /* MAX_DEPTH (main.rs:28): at most max_depth rays per path */
    double   t_min;               /* 0.0001 at main.rs:44; >= 0.  Below ~1e-12 (0 included) the reference's own
                                     self-intersections depend on the last bit of its f64 rounding, and no f32 render
                                     can be compared with it there */
    uint64_t seed;                /* Philox key; the reference's thread_rng is unseedable */
    uint8_t  alpha;               /* 255 at main.rs:137 */
    uint8_t  precision;           /* rtiow_precision */
    uint8_t  reserved[6];
    uint32_t tile_rows;           /* rows per interleaved tile when the frame is split across GPUs (>=1) */
} rtiow_params;

/* How the row tiles of a multi-GPU frame reach rank 0 (the reference's collect(), main.rs:139).
 * NCCL : equal-size (padded) tile buffers + ONE ncclAllGather per frame + a de-interleave kernel (SURVEY §8e).
 * FUSED: every rank's epilogue stores its pixels straight into their top-down place in rank 0's frame through NVLink peer
 *        memory (cudaDeviceEnablePeerAccess inside one process, a CUDA IPC mapping across processes); across processes a
 *        1-int ncclAllReduce is the frame-complete barrier.  No tile buffer, no de-interleave pass.
 * AUTO : FUSED when the mapping is possible, else NCCL.  All three give the same bytes. */
typedef enum { RTIOW_GATHER_AUTO = 0, RTIOW_GATHER_NCCL = 1, RTIOW_GATHER_FUSED = 2 } rtiow_gather_mode;
#define RTIOW_NCCL_UNIQUE_ID_BYTES 128

typedef struct {
    double   kernel_ms;           /* CUDA-event time of the render kernels: this rank, or the slowest device of an n-GPU ctx */
    double   total_ms;            /* host wall time of the call */
    uint64_t paths;               /* width*height*spp handled by this call */
    uint64_t rays_traced;         /* exact count of world.hit calls (main.rs:44) */
    uint64_t sphere_tests;        /* rays_traced * n_spheres: the linear scan of shapes/mod.rs:61-66 */
    uint64_t h2d_bytes, d2h_bytes;
    uint32_t kernel_launches;
    uint32_t n_gpus;
    uint32_t scan_backend;        /* rtiow_scan_backend the render launch used: RTIOW_SCAN_FP32 or RTIOW_SCAN_TENSOR */
    uint32_t reserved;
} rtiow_stats;

typedef struct rtiow_ctx rtiow_ctx;

int         rtiow_abi_version(void);
const char* rtiow_last_error(void);
int         rtiow_device_count(int* out_count);

/* One process driving n_gpus devices (0..n_gpus-1); the frame is split into interleaved row tiles
 * and gathered on device 0.  n_gpus = 1 is the single-GPU path. */
int  rtiow_ctx_create(int n_gpus, rtiow_ctx** out);
/* One process per GPU (torchrun / MPI style): this ctx drives `device` only. */
int  rtiow_ctx_create_on_device(int device, rtiow_ctx** out);
void rtiow_ctx_destroy(rtiow_ctx* ctx);
/* Select the filter backend of every later F32 call on this ctx (render and unit-level batches).  RTIOW_SCAN_TENSOR on a
 * scene that does not qualify makes those calls return RTIOW_ERR_UNSUPPORTED (never a silent fallback). */
int  rtiow_ctx_set_scan_backend(rtiow_ctx* ctx, int backend);

/* One process per GPU (MPI / torchrun style) with the gather INSIDE the library.  Rank 0 calls rtiow_nccl_unique_id and hands
 * the RTIOW_NCCL_UNIQUE_ID_BYTES bytes to every rank by any means (MPI_Bcast, a file, torch.distributed); every rank then
 * calls rtiow_ctx_create_rank (collective: ncclCommInitRank).  world = 1 needs no id and no NCCL.  NCCL is loaded at run time
 * (libnccl.so.2); if it is missing these return RTIOW_ERR_NCCL. */
int  rtiow_nccl_unique_id(void* out_id);
int  rtiow_ctx_create_rank(int device, int rank, int world, const void* nccl_unique_id, rtiow_ctx** out);
/* a one-device ctx works on the caller's cudaStream_t from now on (NULL: back to its own stream), so the caller's events and
 * copies on that stream are ordered with the library's kernels and collectives */
int  rtiow_ctx_set_stream(rtiow_ctx* ctx, void* stream);
/* rtiow_gather_mode of every later multi-GPU render on this ctx (an n-GPU ctx or a rank ctx) */
int  rtiow_ctx_set_gather(rtiow_ctx* ctx, int mode);
/* one line describing the gather the last render used (for logs and bench lines) */
int  rtiow_ctx_gather_info(rtiow_ctx* ctx, char* buf, size_t n);

/* Replaces building `world` for the GPU (main.rs:62-99 push calls): validates, converts to the
 * device SoA and uploads to every device of the ctx.  May be called again to replace the scene. */
int rtiow_scene_upload(rtiow_ctx* ctx, const rtiow_spheres* spheres, const rtiow_materials* materials);

/* Camera::new, camera.rs:17-45 (host, f64). */
int rtiow_camera_new(const double look_from[3], const double look_at[3], const double v_up[3], double v_fov_deg,
                     double aspect_ratio, double aperture, double focus_dist, rtiow_camera* out);

/* Defaults mirroring main.rs:24-28,44,137: 200x133, 100 spp, depth 50, t_min 1e-4, alpha 255. */
void rtiow_params_default(rtiow_params* p);

/* THE drop-in call: replaces main.rs:122-145.  Writes 4*width*height bytes, top-down RGBA8 — the
 * buffer handed to ImageBuffer::from_vec at main.rs:147 — into caller-owned HOST memory. */
int rtiow_render(rtiow_ctx* ctx, const rtiow_camera* cam, const rtiow_params* p, uint8_t* out_rgba, rtiow_stats* stats);

/* Many views of one scene (turntables, animations, stereo pairs, camera sweeps) in one call: out_rgba receives n_views top-down
 * RGBA8 frames of 4*width*height bytes each, in view order, in caller-owned HOST memory.  Frame v equals
 * rtiow_render(ctx, &cams[v], p, ...) byte for byte, so the views share their sample streams (same seed, same pixel keys);
 * decorrelated views are separate calls with other seeds.  One render launch per device pays the fixed per-launch cost once
 * per batch.  An n-GPU ctx renders a contiguous block of whole views on each device.  n_views * width * height must be
 * <= 0xfffffff0.  A rank ctx with world > 1 returns RTIOW_ERR_UNSUPPORTED.  Stats cover the whole batch (kernel_ms: the
 * slowest device's). */
int rtiow_render_views(rtiow_ctx* ctx, const rtiow_camera* cams, uint32_t n_views, const rtiow_params* p, uint8_t* out_rgba,
                       rtiow_stats* stats);

/* The reference shows progress per row (indicatif bar, main.rs:120,124) and the finished frame in a piston window
 * (main.rs:151-171).  The GPU equivalent: the spp samples are rendered in n_passes slices (clamped to spp); after each slice
 * on_pass(user, pass [1-based], n_passes, spp_done, rgba) receives the frame so far — out_rgba, top-down RGBA8, quantised
 * with the samples done so far (vec3.rs:404-420).  A non-zero return stops the render (RTIOW_ERR_CANCELLED; out_rgba keeps
 * the last frame).  on_pass may be NULL.  The final frame is bit-identical to rtiow_render's; stats are summed over passes. */
typedef int (*rtiow_progress_fn)(void* user, uint32_t pass, uint32_t n_passes, uint32_t spp_done, const uint8_t* rgba);
int rtiow_render_progressive(rtiow_ctx* ctx, const rtiow_camera* cam, const rtiow_params* p, uint32_t n_passes,
                             rtiow_progress_fn on_pass, void* user, uint8_t* out_rgba, rtiow_stats* stats);

/* The drop-in call of a rank ctx (collective: every rank calls it with the same camera and params).  Renders this rank's rows
 * {y : (y / tile_rows) % world == rank}, gathers inside the library, and writes the whole top-down RGBA8 frame into out_rgba
 * (HOST memory) on rank 0 — and on every rank that passes a buffer when the gather is NCCL.  out_rgba may be NULL on ranks > 0.
 * stats describe this rank (paths, rays, kernel_ms of its own rows). */
int rtiow_render_rank(rtiow_ctx* ctx, const rtiow_camera* cam, const rtiow_params* p, uint8_t* out_rgba, rtiow_stats* stats);
/* the same, leaving the frame in DEVICE memory: *d_frame = the whole frame on rank 0 (NCCL gather: on every rank; FUSED: NULL
 * on ranks > 0), owned by the ctx and valid until its next render. */
int rtiow_render_rank_device(rtiow_ctx* ctx, const rtiow_camera* cam, const rtiow_params* p, const void** d_frame, rtiow_stats* stats);
/* Frames back to back (an animation loop; the reference renders one frame per process, main.rs:104-149, so this replaces nothing
 * there): rtiow_render_rank_device WITHOUT the host synchronisation — kernel, epilogue / gather and the frame-complete barrier are
 * enqueued on the ctx's stream and the call returns.  *d_frame as above; with the FUSED gather two frame buffers alternate, so a
 * frame stays valid until the second-next enqueue.  rtiow_ctx_synchronize waits for everything enqueued; its stats (may be NULL)
 * carry the MEAN kernel_ms of the frames enqueued since the last synchronize and the paths / rays of the last one.  At most 1024
 * frames may be enqueued between two synchronizes (one event pair each). */
int rtiow_render_rank_enqueue(rtiow_ctx* ctx, const rtiow_camera* cam, const rtiow_params* p, const void** d_frame);
int rtiow_ctx_synchronize(rtiow_ctx* ctx, rtiow_stats* stats);

/* --- lower-level one-process-per-GPU pieces for callers that own the gather (rank r of world G renders rows {y : (y / tile_rows) % G == r}) ---- */
/* bytes of one rank's tile buffer (equal on every rank; padded when the tile count does not divide) */
int rtiow_tile_buffer_bytes(const rtiow_params* p, int world, size_t* out_bytes);
/* render this rank's tiles into DEVICE memory d_tiles (>= rtiow_tile_buffer_bytes), rank-local
 * top-down order, on `stream` (a cudaStream_t, may be NULL).  Asynchronous unless stats != NULL. */
int rtiow_render_tiles_device(rtiow_ctx* ctx, const rtiow_camera* cam, const rtiow_params* p, int rank, int world,
                              void* d_tiles, void* stream, rtiow_stats* stats);
/* the same render with the gather FUSED into the epilogue: d_frame is the whole top-down frame (4*width*height bytes) in DEVICE
 * memory — usually rank 0's buffer mapped into this process (CUDA IPC, torch symmetric memory) — and this rank's pixels are
 * stored straight into their rows of it, over NVLink when it is remote.  Replaces tiles + all-gather + rtiow_deinterleave_device;
 * the caller synchronises the ranks before rank 0 reads the frame. */
int rtiow_render_to_frame_device(rtiow_ctx* ctx, const rtiow_camera* cam, const rtiow_params* p, int rank, int world,
                                 void* d_frame, void* stream, rtiow_stats* stats);
/* d_gathered = the G tile buffers concatenated in rank order (what an allgather leaves);
 * writes the top-down frame (4*width*height bytes) to DEVICE memory d_frame. */
int rtiow_deinterleave_device(rtiow_ctx* ctx, const void* d_gathered, const rtiow_params* p, int world, void* d_frame,
                              void* stream);

/* --- unit-level entry points: the SAME __device__ functions the renderer uses, on explicit inputs
 *     with injected random numbers (SURVEY Appendix B).  All arrays are HOST memory, row-major
 *     [n][3] for vectors.  precision selects the float or double instantiation. ---------------------- */
/* Sphere::hit, sphere.rs:16-41 + HitRecord::new, mod.rs:20-30 — one (sphere, ray) pair per item */
int rtiow_sphere_hit_batch(rtiow_ctx* ctx, int precision, int64_t n, const double* center, const double* radius,
                           const double* orig, const double* dir, const double* t_min, const double* t_max,
                           int32_t* hit, double* t, double* p, double* normal, int32_t* front_face);
/* HittableList::hit, mod.rs:56-69, against the uploaded scene — the renderer's scan */
int rtiow_hitlist_batch(rtiow_ctx* ctx, int precision, int64_t n, const double* orig, const double* dir, double t_min,
                        int32_t* hit, int32_t* index, double* t, double* p, double* normal, int32_t* front_face);
/* Scatter::scatter x3, materials.rs:22-30,50-61,77-104; sample = injected random (see oracle header) */
int rtiow_scatter_batch(rtiow_ctx* ctx, int precision, int64_t n, const int32_t* kind, const double* albedo,
                        const double* param, const double* r_orig, const double* r_dir, const double* p,
                        const double* normal, const int32_t* front_face, const double* sample, int32_t* some,
                        double* attenuation, double* s_orig, double* s_dir);
/* Camera::get_ray, camera.rs:47-54; disk_xy = accepted random_in_unit_disk sample */
int rtiow_get_ray_batch(rtiow_ctx* ctx, int precision, const rtiow_camera* cam, int64_t n, const double* s,
                        const double* t, const double* disk_xy, double* orig, double* dir);
/* Color::to_rgba, vec3.rs:404-420 */
int rtiow_to_rgba_batch(rtiow_ctx* ctx, int precision, int64_t n, const double* color, uint8_t alpha, uint64_t spp,
                        uint8_t* out_rgba);
/* Vec3::reflect / Vec3::refract, vec3.rs:116-125 */
int rtiow_reflect_batch(rtiow_ctx* ctx, int precision, int64_t n, const double* v, const double* nrm, double* out);
int rtiow_refract_batch(rtiow_ctx* ctx, int precision, int64_t n, const double* uv, const double* nrm,
                        const double* eta, double* out);
/* ray_color, main.rs:38-57, as the renderer's iterative bounce loop, on explicit rays against the
 * uploaded scene; randoms are Philox blocks keyed (seed; pixel[i], sample[i], bounce). */
int rtiow_ray_color_batch(rtiow_ctx* ctx, int precision, int64_t n, const double* orig, const double* dir,
                          const uint32_t* pixel, const uint32_t* sample, uint64_t seed, int32_t max_depth, double t_min,
                          double* color, uint64_t* rays);
/* the same, also recording every ray of every path: trace_index[i][k] = list index hit by the k-th ray of path i (-1: miss
 * or no such ray), trace_ray[i][k] = (origin, unit direction) of that ray; both [n][max_depth], either may be NULL.  The
 * parity tests use it to compare GPU and oracle paths ray by ray. */
int rtiow_ray_color_trace_batch(rtiow_ctx* ctx, int precision, int64_t n, const double* orig, const double* dir,
                                const uint32_t* pixel, const uint32_t* sample, uint64_t seed, int32_t max_depth, double t_min,
                                double* color, uint64_t* rays, int32_t* trace_index, double* trace_ray);
/* the sampler mapping itself: Philox4x32-10 block (seed; pixel, sample, bounce) -> 4 uniforms, the
 * lens-disk sample, the unit vector and the in-unit-sphere vector derived from them.  out: [n][12] */
int rtiow_sampler_batch(rtiow_ctx* ctx, int precision, int64_t n, const uint32_t* pixel, const uint32_t* sample,
                        const uint32_t* bounce, uint64_t seed, double* out);

/* --- measurement ------------------------------------------------------------------------------- */
/* FP32-pipe calibration for the roofline (MEASURED_PEAKS.json has no FP32 entry): runs an
 * FFMA-saturating kernel for about `target_ms` and reports achieved TFLOP/s.  packed=1 uses the
 * f32x2 form the scan uses. */
int rtiow_fp32_peak_probe(rtiow_ctx* ctx, int packed, double target_ms, double* out_tflops, double* out_ms);
/* writes `bytes` of device memory (> L2) to evict the L2 between timed iterations */
int rtiow_flush_l2(rtiow_ctx* ctx);

/* --- seeded scene builder (SURVEY §8f #1): random_scene, main.rs:59-102, with an explicit seed.
 *     material_mode: 0 = reference mix, 1 = all Lambertian, 2 = all Metal, 3 = all Dialectric
 *     (+ one hollow shell r=-0.9 inside the big glass sphere).  half_extent 11 = the reference grid.
 *     Arrays are caller-allocated with capacity `cap` spheres (one material per sphere);
 *     *out_n receives the count.  Host-only: works without a GPU. */
int rtiow_random_scene(uint64_t seed, int32_t half_extent, int32_t material_mode, uint32_t cap, double* cx, double* cy,
                       double* cz, double* radius, uint32_t* mat_kind, double* albedo_rgb, double* mat_param,
                       uint32_t* out_n);

/* --- scene dump / load (SURVEY §8f #1): the same world for this library, the oracle and a cargo build of the reference.
 *     Text: "rtiow-scene 1", "n <count>", then one line per sphere in list order:
 *     cx cy cz radius kind albedo_r albedo_g albedo_b param   (17 significant digits: f64 round-trips bit for bit).
 *     rtiow_scene_load with cap = 0 only returns the count; a file larger than cap gives RTIOW_ERR_NOMEM with *out_n = the count.
 *     Host-only. */
int rtiow_scene_save(const char* path, uint32_t n, const double* cx, const double* cy, const double* cz, const double* radius,
                     const uint32_t* mat_kind, const double* albedo_rgb, const double* mat_param);
int rtiow_scene_load(const char* path, uint32_t cap, double* cx, double* cy, double* cz, double* radius, uint32_t* mat_kind,
                     double* albedo_rgb, double* mat_param, uint32_t* out_n);

#ifdef __cplusplus
}
#endif
#endif /* RTIOW_CUDA_H */
