// rt_render.cuh — the render megakernel: the pixel/sample loop (main.rs:122-139), ray_color
// (main.rs:38-57) as an iterative bounce loop, and the quantise + row flip (main.rs:137,141-145).
//
// Execution model (B200, 148 SMs): a persistent grid of kCtasPerSm x SM-count CTAs.  Every lane owns
// one PATH at a time; when its path ends (miss -> sky, absorbed, depth exhausted) the lane pulls the
// next (pixel, sample) from its warp's chunk, so the sphere scan — >95 % of the work — always runs
// with 32 live lanes regardless of the heavy-tailed path length (1..max_depth rays).
// Sample radiance is accumulated in 32.32 fixed point with RED.ADD.U64 (integer adds are associative),
// so the image is bit-identical for any chunk size, grid size or GPU count.
#pragma once
#include "rt_scene.cuh"
#include "rt_umma_scan.cuh"

namespace rt {

template <typename T> struct RenderArgs {
    SceneDev scene;
    CameraT<T> cam;
    uint32_t width, height, spp;   // spp: samples per pixel rendered by THIS launch (a progressive pass renders a slice)
    uint32_t smp_begin;            // index of the launch's first sample: the Philox key uses smp_begin + local index
    int32_t max_depth;
    T t_min;
    T inv_wm1, inv_hm1;            // 1/(width-1), 1/(height-1): the jitter denominators of main.rs:131-132
    PhiloxKey key;                 // Philox4x32-10 round keys of the sample seed
    // frame partition: this launch renders rows {y : (y / tile_rows) % world == rank}
    uint32_t rank, world, tile_rows, local_rows;
    uint32_t chunk_samples;        // samples per chunk (<= spp); chunks never straddle pixels
    uint32_t chunks_per_pixel;
    uint32_t chunks_per_fetch;     // chunks per fetch from the work counter while plenty are left ...
    uint32_t guided_div;           // ... and (chunks left) / guided_div towards the end (guided_div = 2 x warps of the grid)
    uint64_t n_chunks;
    T sample_cap;                  // min(1e9, the frame's total spp): the largest value a sample adds (to_fix)
    uint32_t saturate;             // total spp > 65535: sums could pass 2^32, accumulate with add_saturating
    unsigned long long* accum;     // [3][local_rows*width] 32.32 fixed-point radiance sums
    unsigned long long* work_counter;
    unsigned long long* ray_counter;
};

#define RT_FIX_SCALE 4294967296.0f   // 2^32

// What a render launch produces; every kind runs the same loop (render_kernel, render_kernel_umma):
//   Frame     a frame, or a rank's rows of one;
//   Views     a batch of views on one device, one camera per view in `cams` (rtiow_render_views);
//   Aov       a frame, and every camera ray's first hit in `aov` (AovArgs, rtiow_render_aov);
//   Adaptive  one round of rtiow_render_adaptive: the pixels of `ad.list` only, with their noise sums (AdaptArgs).
enum class Loop { Frame, Views, Aov, Adaptive };

// The first-hit accumulators of rtiow_render_aov (Loop::Aov), beside RenderArgs::accum and over the same local pixels.
// Every camera ray adds one fixed-point sample per channel with an integer RED.ADD, so the AOVs are bit-identical for any grid,
// chunking or GPU count.  Each per-sample value is clamped to a range whose sum over 2^32 - 1 samples stays below 2^64, so no
// sum can wrap at any spp and none needs add_saturating:
//   albedo  [3][n_lp]  per sample in [0, 1] (the range a denoiser's albedo guide takes), scale 2^32;
//   normal  [3][n_lp]  per sample n + 1 in [0, 2] (a unit normal, offset so that a sample is never negative), scale 2^31;
//   depth   [n_lp]     per sample in [0, 65536] scene units, scale 2^16 (resolution 1.5e-5);
//   hits    [n_lp]     camera rays that hit a sphere (32-bit: at most spp of them).
// A miss adds its sky value to the albedo and nothing else, so finalize_aov_kernel removes the offset of the hits alone.
// 16-byte aligned: as a kernel parameter after the 8-byte `cams` it still starts on a 16-byte boundary, so the render loop
// loads both pointers with one 128-bit constant load.
struct __align__(16) AovArgs {
    unsigned long long* sum;       // [7][n_lp]: albedo r, g, b, normal x, y, z, depth
    unsigned int* hits;            // [n_lp]
};
#define RT_AOV_NORMAL_SCALE 2147483648.0   // 2^31
#define RT_AOV_DEPTH_SCALE 65536.0         // 2^16
#define RT_AOV_DEPTH_MAX 65536.0           // a farther hit is recorded at this distance

// One round of rtiow_render_adaptive (Loop::Adaptive): the launch renders its sample range of the pixels in `list`
// only (local pixel indices, n_chunks / chunks_per_pixel of them), and every finished non-black path also adds its noise value
// y = clamp((r + g + b) / 3, 0, 1) to two per-pixel fixed-point sums, S1 += round(y 2^32) and S2 += round(y^2 2^32).  Each
// value is at most 2^32, so neither sum can wrap at any u32 spp.  The pixels' own radiance sums stay RenderArgs::accum.
struct AdaptArgs {
    const uint32_t* list;          // the round's active local pixels, in the frame's bottom-up drawing order
    unsigned long long* lum_sum;   // [2][n_lp]: S1, S2
};

// A sample's 32.32 value, clamped to [0, cap].  NaN/negative -> 0: a poisoned sample contributes nothing (the reference would
// turn the whole pixel black through NaN -> `as u8` = 0, vec3.rs:415-417; the upload rejects non-finite materials, so only
// an overflow to inf x 0 can make one).  cap = min(1e9, total spp) changes no byte: a sample of >= spp alone brings the
// pixel's mean to >= 1, which quantises to 255 with or without the clamp (vec3.rs:404-420).
__device__ __forceinline__ unsigned long long to_fix(float c, float cap)
{
    return __float2ull_rn(fminf(fmaxf(c, 0.0f), cap) * RT_FIX_SCALE);
}
__device__ __forceinline__ unsigned long long to_fix(double c, double cap)
{
    return __double2ull_rn(fmin(fmax(c, 0.0), cap) * 4294967296.0);
}

// local row -> global top-down row under the interleaved-tile partition
__device__ __forceinline__ uint32_t local_to_global_row(uint32_t lr, uint32_t tile_rows, uint32_t world, uint32_t rank)
{
    const uint32_t tl = lr / tile_rows, within = lr - tl * tile_rows;
    return (tl * world + rank) * tile_rows + within;
}

// One path in flight (one lane).  The ray is (o, dhat) with |dir| folded into tmin_n; self_* name the
// sphere the ray starts on (rt_scene.cuh, candidate_self).  The Philox event number of the path's next scatter is
// max_depth - depth + 1 (event 0 is the camera ray), so no separate bounce counter is carried.
template <typename T> struct PathState {
    V3<T> o, dhat, thr, self_n;
    T tmin_n;
    int self_code;
    uint32_t pix_key, smp;
    int depth;
};

// float: one MUFU.RSQ gives 1/|dir| (2 ulp); dhat is then unit to ~2e-7, which the precise test absorbs through inv_a
__device__ __forceinline__ void inv_and_len(float l2, float* inv, float* len) { *inv = rsqrtf(l2); *len = l2 * *inv; }
__device__ __forceinline__ void inv_and_len(double l2, double* inv, double* len) { *len = sqrt(l2); *inv = 1.0 / *len; }

template <typename T> __device__ __forceinline__ void start_ray(PathState<T>& ps, V3<T> orig, V3<T> dir, T t_min)
{
    T inv, len; inv_and_len(length_squared(dir), &inv, &len);
    ps.o = orig; ps.dhat = dir * inv;
    ps.tmin_n = t_min * len;                        // t is measured in |dir| units (Appendix C.3)
}

template <typename T> __device__ __forceinline__ void init_path(PathState<T>& ps)
{
    ps.o = mk<T>(0, 0, 0); ps.dhat = mk<T>(0, 1, 0); ps.thr = mk<T>(0, 0, 0); ps.self_n = mk<T>(0, 1, 0);
    ps.tmin_n = T(0); ps.self_code = RT_SELF_NONE; ps.pix_key = 0; ps.smp = 0; ps.depth = 0;
}

// world.hit(r, t_min, INFINITY) (main.rs:44) for every lane of the warp (all 32 must call: the scan's warp-level
// operations need them); lanes without a ray get a result they ignore.
template <typename T, bool kSmem>
__device__ __forceinline__ void world_hit(const SceneDev& sc, const float* table, uint16_t* cand, int cand_stride, const PathState<T>& ps,
                                          T* t_hit, int* idx, int* code)
{
    if (sizeof(T) == 4) {
        const HitF h = closest_hit<kSmem>(sc, table, mk<float>((float)ps.o.x, (float)ps.o.y, (float)ps.o.z),
                                          mk<float>((float)ps.dhat.x, (float)ps.dhat.y, (float)ps.dhat.z), (float)ps.tmin_n, ps.self_code,
                                          mk<float>((float)ps.self_n.x, (float)ps.self_n.y, (float)ps.self_n.z), cand, cand_stride);
        *t_hit = (T)h.t; *idx = h.idx; *code = h.code;
    } else {
        double td;
        closest_hit_f64(sc, mk<double>(ps.o.x, ps.o.y, ps.o.z), mk<double>(ps.dhat.x, ps.dhat.y, ps.dhat.z), (double)ps.tmin_n, ps.self_code,
                        mk<double>(ps.self_n.x, ps.self_n.y, ps.self_n.z), &td, idx);
        *t_hit = (T)td; *code = *idx;
    }
}

// The hit branch of ray_color (main.rs:46-52) for one lane: HitRecord::new at p (sphere.rs:36-39), Scatter::scatter
// (main.rs:47) with the event's random numbers, then the scattered ray.  (sa, sb, z) is the event's uniform unit vector
// (materials.rs:23 adds it to the normal; materials.rs:53 scales it into the ball by cbrt(u2)); u0 is xi for glass
// (materials.rs:96).  Returns false when the path ends here in black (absorbed: main.rs:51, or depth exhausted: main.rs:40-42).
template <typename T>
__device__ __forceinline__ bool scatter_at_hit(const SceneDev& sc, T t_min, PathState<T>& ps, V3<T> p, int idx, int code, T sa, T sb, T z, T u0, T u2)
{
    V3<T> cen; T rad; V3<T> albedo; T param;
    if (sizeof(T) == 4) {
        const float4 s = sc.sph[idx], m = sc.mat[idx];
        cen = mk<T>(s.x, s.y, s.z); rad = s.w; albedo = mk<T>(m.x, m.y, m.z); param = m.w;
    } else {
        const double4 s = sc.sphd[idx], m = sc.matd[idx];
        cen = mk<T>(s.x, s.y, s.z); rad = s.w; albedo = mk<T>(m.x, m.y, m.z); param = m.w;
    }
    const int kind = sc.kind[idx];
    V3<T> n; bool ff; hit_record(p, cen, rad, ps.dhat, &n, &ff);             // sphere.rs:36-39
    V3<T> sample = mk<T>(u0, 0, 0);
    if (kind != MAT_DIELECTRIC) {
        sample = mk<T>(sa, sb, z);
        if (kind == MAT_METAL) sample = sample * cbrt_t(u2);
    }
    V3<T> att, nd;
    const bool some = scatter<T, sizeof(T) == 4>(kind, albedo, param, ps.dhat, n, ff, sample, &att, &nd);   // main.rs:47
    --ps.depth;
    if (!some || ps.depth <= 0) return false;
    ps.thr = ps.thr * att;                                                    // main.rs:49 as a running product
    start_ray(ps, p, nd, t_min);
    ps.self_code = code;
    const V3<T> pc = p - cen;
    T inv, len; inv_and_len(length_squared(pc), &inv, &len);
    ps.self_n = pc * inv;
    return true;
}

// The event's shared sampler: one sincospi and one sqrt serve the lens disk of a camera ray (camera.rs:48: radius
// sqrt(u2), angle 2 pi u3 — direct_disk) and the unit vector of a scatter (z = 1 - 2 u0, angle 2 pi u1 — direct_unit_vector).
template <typename T>
__device__ __forceinline__ void event_sample(bool camera, const Uniform4<T>& u, T* sa, T* sb, T* z)
{
    *z = T(1) - T(2) * u.u0;
    T sn, cs; sincospi_t(T(2) * (camera ? u.u3 : u.u1), &sn, &cs);
    const T rr = sqrt_t(camera ? u.u2 : max_t(T(0), T(1) - *z * *z));
    *sa = rr * cs; *sb = rr * sn;
}

// One iteration of ray_color (main.rs:38-57) for a lane on an explicit ray (rtiow_ray_color_batch), after the scan found
// (t_hit, idx, code): miss -> sky / hit -> scatter.  Returns the lane's new `active`; when the path ends, *radiance receives
// its value (throughput x sky, or black).  The render kernel below runs the same pieces in a different order (scatter of
// the previous hit and camera rays share one Philox block + sampler per iteration).
template <typename T>
__device__ __forceinline__ bool bounce_step(const SceneDev& sc, const PhiloxKey& key, int max_depth, T t_min, PathState<T>& ps, T t_hit, int idx, int code,
                                            V3<T>* radiance)
{
    if (idx < 0) {                                                            // miss: sky (main.rs:54-56)
        *radiance = ps.thr * sky<T, sizeof(T) == 4>(ps.dhat);
        return false;
    }
    const V3<T> p = ps.o + ps.dhat * t_hit;                                   // ray.rs:15-17
    const Uniform4<T> u = event_uniforms<T>(key, ps.pix_key, ps.smp, (uint32_t)(max_depth - ps.depth) + 1u);
    T sa, sb, z; event_sample(false, u, &sa, &sb, &z);
    if (!scatter_at_hit(sc, t_min, ps, p, idx, code, sa, sb, z, u.u0, u.u2)) { *radiance = mk<T>(0, 0, 0); return false; }
    return true;
}

// ---- the pixel/sample loop's bookkeeping (main.rs:122-135) ---------------------------------------------------------
// warp-uniform cursor over the work: chunks (<= 256 samples of ONE pixel) fetched from a global atomic counter
struct WorkCursor {
    uint32_t cs = 0, ce = 0, c_lp = 0, c_x = 0, c_y = 0, c_v = 0;
    unsigned long long cc = 0, cce = 0;
    bool exhausted = false;
};

// Every lane whose slot is free (`busy` false) takes the next (pixel, sample) of the warp's chunk (main.rs:130).  Returns
// true for the lanes that received one; their pixel column / bottom-up row come back in *px, *pj.
// Loop::Views: the launch renders a batch of views on one device as ONE frame n_views * height rows tall, so local row lr is
// row lr % height of view lr / height.  *pv receives the view; pj and the Philox pixel key are those of the row within the
// view, exactly as the view's own frame computes them, which makes every view byte-identical to it.
// Loop::Adaptive: chunk c belongs to pixel ad.list[c / chunks_per_pixel] (AdaptArgs), a round's subset of the pixels in the same order.
template <Loop L, typename T>
__device__ __forceinline__ bool assign_work(const RenderArgs<T>& a, const AdaptArgs& ad, WorkCursor& wc, unsigned lt_mask, bool busy, PathState<T>& ps,
                                            uint32_t& acc_lp, uint32_t* px, uint32_t* pj, uint32_t* pv)
{
    bool fresh = false;
    unsigned need = __ballot_sync(RT_FULL, !busy);
    while (need && !wc.exhausted) {
        if (wc.cs == wc.ce) {
            if (wc.cc == wc.cce) {
                // guided self-scheduling: a fetch takes chunks_per_fetch chunks while plenty are left and 1/guided_div of the
                // rest towards the end of the frame, so that the warps of the persistent grid run dry together
                unsigned long long base = 0, take = a.chunks_per_fetch;
                if (lt_mask == 0u) {                                                                             // lane 0
                    const unsigned long long seen = *(volatile unsigned long long*)a.work_counter;
                    const unsigned long long left = a.n_chunks > seen ? a.n_chunks - seen : 0ull;
                    take = min(take, max(1ull, left / a.guided_div));
                    base = atomicAdd(a.work_counter, take);
                }
                wc.cc = __shfl_sync(RT_FULL, base, 0);
                wc.cce = wc.cc + __shfl_sync(RT_FULL, take, 0); if (wc.cce > a.n_chunks) wc.cce = a.n_chunks;
                if (wc.cc >= a.n_chunks) { wc.exhausted = true; break; }
            }
            // chunks walk the frame BOTTOM-UP, like the reference's row index j (main.rs:122,132): the top rows come last, and
            // in these scenes they are sky — one-ray paths — so the frame does not end on freshly started 50-bounce paths
            const unsigned long long c = wc.cc++;
            const uint32_t pix = (uint32_t)(c / a.chunks_per_pixel);
            const uint32_t part = (uint32_t)(c - (unsigned long long)pix * a.chunks_per_pixel);
            wc.c_lp = L == Loop::Adaptive ? ad.list[pix] : a.local_rows * a.width - 1u - pix;
            wc.cs = part * a.chunk_samples; wc.ce = min(wc.cs + a.chunk_samples, a.spp);
            const uint32_t lr = wc.c_lp / a.width;
            wc.c_x = wc.c_lp - lr * a.width;
            wc.c_y = local_to_global_row(lr, a.tile_rows, a.world, a.rank);
            if constexpr (L == Loop::Views) { wc.c_v = lr / a.height; wc.c_y = lr - wc.c_v * a.height; }
        }
        const uint32_t avail = wc.ce - wc.cs;
        const uint32_t r = __popc(need & lt_mask);
        if (!busy && !fresh && r < avail) {
            fresh = true;
            acc_lp = wc.c_lp;
            ps.smp = a.smp_begin + wc.cs + r;
            *px = wc.c_x;
            *pv = wc.c_v;
            *pj = a.height - 1u - wc.c_y;                            // j = 0 is the bottom row (main.rs:132,141-145)
            ps.pix_key = *pj * a.width + wc.c_x;
        }
        wc.cs += min((uint32_t)__popc(need), avail);
        need = __ballot_sync(RT_FULL, !busy && !fresh);
    }
    return fresh;
}

// One channel's add, saturating at 2^64 - 1 (a sum of 2^32: any spp below 2^32 quantises it to 255, as the reference's
// unbounded f64 sum would be).  An add that wraps sees old + v < old and raises the sum to the maximum; any later add wraps
// again and does the same, so whatever the order of the adds, a channel that passed 2^32 ends at 2^64 - 1 and every other
// one holds its exact sum.  It waits for the old value, so it is only used where a sum can pass 2^32 (RenderArgs::saturate).
__device__ __forceinline__ void add_saturating(unsigned long long* sum, unsigned long long v)
{
    const unsigned long long old = atomicAdd(sum, v);
    if (old + v < old) atomicMax(sum, ~0ull);
}

// pixel_color += ray_color (main.rs:135): 32.32 fixed-point RED.ADD.U64 straight into the frame's accumulators
// (integer adds commute: any order, any GPU count, same bits); black paths add nothing.  With every sample clamped to
// sample_cap <= spp, a channel's sum stays below spp^2 <= 65535^2 < 2^32 and cannot wrap; larger spp saturate instead.
template <typename T>
__device__ __forceinline__ void accumulate(const RenderArgs<T>& a, uint32_t acc_lp, V3<T> rad)
{
    if (rad.x != T(0) || rad.y != T(0) || rad.z != T(0)) {
        const size_t n_lp = (size_t)a.local_rows * a.width;
        unsigned long long* const sum = a.accum + acc_lp;
        const unsigned long long vx = to_fix(rad.x, a.sample_cap), vy = to_fix(rad.y, a.sample_cap), vz = to_fix(rad.z, a.sample_cap);
        if (a.saturate) {
            add_saturating(sum, vx); add_saturating(sum + n_lp, vy); add_saturating(sum + 2 * n_lp, vz);
        } else {
            atomicAdd(sum, vx); atomicAdd(sum + n_lp, vy); atomicAdd(sum + 2 * n_lp, vz);
        }
    }
}

// Step 2 of the render iteration (below) for one lane: the camera ray of a fresh sample, or the scatter at the pending hit
// on sphere hit_idx at ps.o.  Returns whether the lane has a ray for this iteration's scan.  The camera is a.cam, or with
// Loop::Views the camera of the sample's view pv.
template <Loop L, typename T>
__device__ __forceinline__ bool next_ray(const RenderArgs<T>& a, const CameraT<T>* cams, PathState<T>& ps, bool fresh, bool pending, int hit_idx, int hit_code,
                                         uint32_t px, uint32_t pj, uint32_t pv)
{
    const Uniform4<T> u = event_uniforms<T>(a.key, ps.pix_key, ps.smp, fresh ? 0u : (uint32_t)(a.max_depth - ps.depth) + 1u);
    T sa, sb, z; event_sample(fresh, u, &sa, &sb, &z);
    bool active = false;
    if (fresh) {
        const T su = (T(px) + u.u0) * a.inv_wm1;                 // main.rs:131
        const T sv = (T(pj) + u.u1) * a.inv_hm1;                 // main.rs:132
        const CameraT<T>& cam = L == Loop::Views ? cams[pv] : a.cam;
        V3<T> ro, rd; get_ray(cam, su, sv, sa, sb, &ro, &rd);    // main.rs:134
        start_ray(ps, ro, rd, a.t_min);
        ps.thr = mk<T>(1, 1, 1); ps.self_code = RT_SELF_NONE;
        ps.depth = a.max_depth;
        active = ps.depth > 0;                                   // main.rs:40-42
    } else if (pending) {
        active = scatter_at_hit(a.scene, a.t_min, ps, ps.o, hit_idx, hit_code, sa, sb, z, u.u0, u.u2);
    }
    return active;
}

// a per-sample AOV value clamped to [0, hi] in fixed point (AovArgs); NaN -> 0
__device__ __forceinline__ unsigned long long aov_fix(float v, float hi, float scale) { return __float2ull_rn(fminf(fmaxf(v, 0.0f), hi) * scale); }
__device__ __forceinline__ unsigned long long aov_fix(double v, double hi, double scale) { return __double2ull_rn(fmin(fmax(v, 0.0), hi) * scale); }

// The first hit of a camera ray into the AOV accumulators (AovArgs): the albedo of the material hit (Lambertian / Metal: its
// albedo, Dielectric: 1) or the sky value on a miss (main.rs:54-56), and on a hit HitRecord::new's normal (hit_record) and
// the distance t_hit (the ray's direction is unit: rt_render.cuh, start_ray).
template <typename T>
__device__ __forceinline__ void record_first_hit(const RenderArgs<T>& a, const AovArgs& aov, const PathState<T>& ps, uint32_t acc_lp, T t_hit, int idx)
{
    const size_t n_lp = (size_t)a.local_rows * a.width;
    unsigned long long* const sum = aov.sum + acc_lp;
    V3<T> alb;
    if (idx < 0) {
        alb = sky<T, sizeof(T) == 4>(ps.dhat);
    } else {
        V3<T> cen; T rad;
        if (sizeof(T) == 4) {
            const float4 s = a.scene.sph[idx], m = a.scene.mat[idx];
            cen = mk<T>(s.x, s.y, s.z); rad = s.w; alb = mk<T>(m.x, m.y, m.z);
        } else {
            const double4 s = a.scene.sphd[idx], m = a.scene.matd[idx];
            cen = mk<T>(s.x, s.y, s.z); rad = s.w; alb = mk<T>(m.x, m.y, m.z);
        }
        if (a.scene.kind[idx] == MAT_DIELECTRIC) alb = mk<T>(1, 1, 1);
        V3<T> n; bool ff; hit_record(ps.o + ps.dhat * t_hit, cen, rad, ps.dhat, &n, &ff);          // sphere.rs:36-39
        atomicAdd(sum + 3 * n_lp, aov_fix(n.x + T(1), T(2), T(RT_AOV_NORMAL_SCALE)));
        atomicAdd(sum + 4 * n_lp, aov_fix(n.y + T(1), T(2), T(RT_AOV_NORMAL_SCALE)));
        atomicAdd(sum + 5 * n_lp, aov_fix(n.z + T(1), T(2), T(RT_AOV_NORMAL_SCALE)));
        atomicAdd(sum + 6 * n_lp, aov_fix(t_hit, T(RT_AOV_DEPTH_MAX), T(RT_AOV_DEPTH_SCALE)));
        atomicAdd(aov.hits + acc_lp, 1u);
    }
    atomicAdd(sum, aov_fix(alb.x, T(1), T(RT_FIX_SCALE)));
    atomicAdd(sum + n_lp, aov_fix(alb.y, T(1), T(RT_FIX_SCALE)));
    atomicAdd(sum + 2 * n_lp, aov_fix(alb.z, T(1), T(RT_FIX_SCALE)));
}

// A finished path's noise value into the sums of rtiow_render_adaptive (AdaptArgs): y = clamp((r + g + b) / 3, 0, 1) of its
// radiance in the render's precision, S1 += round(y 2^32), S2 += round(y^2 2^32).  A black path adds nothing, as in accumulate.
template <typename T>
__device__ __forceinline__ void accumulate_noise(const RenderArgs<T>& a, const AdaptArgs& ad, uint32_t acc_lp, V3<T> rad)
{
    if (rad.x != T(0) || rad.y != T(0) || rad.z != T(0)) {
        const size_t n_lp = (size_t)a.local_rows * a.width;
        const T y = (rad.x + rad.y + rad.z) / T(3);
        const T yc = y > T(0) ? (y < T(1) ? y : T(1)) : T(0);                  // NaN -> 0, as to_fix does
        atomicAdd(ad.lum_sum + acc_lp, aov_fix(yc, T(1), T(RT_FIX_SCALE)));
        atomicAdd(ad.lum_sum + n_lp + acc_lp, aov_fix(yc * yc, T(1), T(RT_FIX_SCALE)));
    }
}

// Step 4 for one lane after the scan found (t_hit, idx, code); on a hit the lane moves to the hit point and keeps the
// sphere in *hit_idx, *hit_code.  Returns whether a scatter is now pending.  Loop::Aov: a camera ray (depth still max_depth)
// also records its first hit (record_first_hit).  Loop::Adaptive: a path that ends on the sky also adds its noise value
// (accumulate_noise); paths that end black add nothing anywhere.
template <Loop L, typename T>
__device__ __forceinline__ bool take_hit(const RenderArgs<T>& a, const AovArgs& aov, const AdaptArgs& ad, PathState<T>& ps, bool active, uint32_t acc_lp,
                                         T t_hit, int idx, int code, int* hit_idx, int* hit_code)
{
    if (!active) return false;
    if (L == Loop::Aov && ps.depth == a.max_depth) record_first_hit(a, aov, ps, acc_lp, t_hit, idx);
    if (idx < 0) {                                                                                        // miss: sky (main.rs:54-56)
        const V3<T> rad = ps.thr * sky<T, sizeof(T) == 4>(ps.dhat);
        accumulate(a, acc_lp, rad);
        if constexpr (L == Loop::Adaptive) accumulate_noise(a, ad, acc_lp, rad);
        return false;
    }
    ps.o = ps.o + ps.dhat * t_hit; *hit_idx = idx; *hit_code = code;                                    // ray.rs:15-17
    return true;
}

// The render kernel.  Per iteration of a warp:
//   1. lanes without a path take the next (pixel, sample);
//   2. ONE Philox block + ONE sincospi/sqrt per lane serve whatever event the lane is at — the camera ray of a fresh
//      sample (main.rs:131-134) or the scatter at the hit found by the previous iteration (main.rs:47) — so the expensive
//      common part runs once, converged, instead of once per divergent branch;
//   3. the scan (world.hit) for all 32 lanes;
//   4. miss -> throughput x sky is added to the pixel and the lane is free again; hit -> the lane keeps the hit for step 2.
// Steps 2 and 4 are next_ray and take_hit, which the tensor-core kernel below calls too.  L is what the launch produces (Loop).
template <typename T, bool kSmem, int kThreads, Loop L>
__device__ __forceinline__ void render_loop(const RenderArgs<T>& a, const CameraT<T>* cams, const AovArgs& aov, const AdaptArgs& ad)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint16_t* cand;
    const float* table = setup_scan_smem<kSmem>(smem_raw, a.scene, kThreads, &cand);
    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;

    PathState<T> ps; init_path(ps);
    uint32_t acc_lp = 0;                                // local pixel of the path in flight
    bool pending = false;                               // the lane's ray hit sphere hit_idx at ps.o: scatter to be evaluated
    int hit_idx = -1, hit_code = RT_SELF_NONE;
    uint32_t n_rays_w = 0;                              // warp-uniform: rays traced by this warp
    WorkCursor wc;

    for (;;) {
        uint32_t px = 0, pj = 0, pv = 0;
        const bool fresh = assign_work<L>(a, ad, wc, lt_mask, pending, ps, acc_lp, &px, &pj, &pv);
        if (!__any_sync(RT_FULL, fresh || pending)) break;

        const bool active = next_ray<L>(a, cams, ps, fresh, pending, hit_idx, hit_code, px, pj, pv);
        n_rays_w += __popc(__ballot_sync(RT_FULL, active));          // world.hit call count (main.rs:44)
        T t_hit; int idx, code;
        world_hit<T, kSmem>(a.scene, table, cand, kThreads, ps, &t_hit, &idx, &code);
        pending = take_hit<L>(a, aov, ad, ps, active, acc_lp, t_hit, idx, code, &hit_idx, &hit_code);
    }
    if (lane == 0) atomicAdd(a.ray_counter, (unsigned long long)n_rays_w);
}

template <typename T, bool kSmem, int kThreads, int kMinCtas, Loop L>
__global__ void __launch_bounds__(kThreads, kMinCtas)
render_kernel(const RenderArgs<T> a, const CameraT<T>* __restrict__ cams, const AovArgs aov, const AdaptArgs ad)
{
    render_loop<T, kSmem, kThreads, L>(a, cams, aov, ad);
}

// The same render loop with the sphere filter on the tensor cores (rt_umma_scan.cuh): G groups of 128 ray threads + G
// MMA-issuer warps per CTA, one CTA per SM.  Everything per ray is the code above — work distribution (assign_work), the
// Philox event and camera / scatter (next_ray), sky and accumulation (take_hit), and in the scan the precise test of the
// filter's survivors and the f64 large-sphere test; only the filter moves from 7 FFMA2 per sphere pair to three
// tcgen05.mma per 128 rays x NC spheres, and the warp-level "any lane alive" vote becomes a 128-thread one, because a
// group's 128 rays form one MMA.
template <int G, int NC, Loop L>
__device__ __forceinline__ void render_loop_umma(const RenderArgs<float>& a, const CameraT<float>* cams, const AovArgs& aov, const AdaptArgs& ad)
{
    extern __shared__ __align__(1024) unsigned char smem_umma[];
    uint32_t tmem_base;
    UmmaCtx ux = umma_setup<G, NC>(smem_umma, a.scene, &tmem_base);
    const unsigned lane = threadIdx.x & 31u;
    if (ux.issuer_warp) {
        // the issuer warps (and the warps that pad them to whole warpgroups) give registers back, the ray warps take them:
        // 1024 threads x 64 registers is the whole file; 8 warps down to 32 frees 8 K, 24 ray warps up to 72 take 6 K
        umma::setmaxnreg_dec<RT_UMMA_ISSUER_REGS>();
        if ((threadIdx.x >> 5) < 5 * G) umma_issuer<G, NC>(ux);
    } else {
        umma::setmaxnreg_inc<RT_UMMA_RAY_REGS>();
        const unsigned lt_mask = (1u << lane) - 1u;
        PathState<float> ps; init_path(ps);
        uint32_t acc_lp = 0;
        bool pending = false;
        int hit_idx = -1, hit_code = RT_SELF_NONE;
        uint32_t n_rays_w = 0;
        WorkCursor wc;
        for (;;) {
            uint32_t px = 0, pj = 0, pv = 0;
            RT_STAMP(1);
            const bool fresh = assign_work<L>(a, ad, wc, lt_mask, pending, ps, acc_lp, &px, &pj, &pv);
            RT_STAMP(2);
            if (!umma_group_any(ux, fresh || pending)) { umma_group_quit(ux); break; }
            RT_STAMP(3);

            const bool active = next_ray<L>(a, cams, ps, fresh, pending, hit_idx, hit_code, px, pj, pv);
            n_rays_w += __popc(__ballot_sync(RT_FULL, active));              // world.hit call count (main.rs:44)
            RT_STAMP(4);
            const HitF h = closest_hit_umma<G, NC>(ux, a.scene, ps.o, ps.dhat, ps.tmin_n, ps.self_code, ps.self_n, active);
            RT_STAMP(9);
            pending = take_hit<L>(a, aov, ad, ps, active, acc_lp, h.t, h.idx, h.code, &hit_idx, &hit_code);
        }
        if (lane == 0) atomicAdd(a.ray_counter, (unsigned long long)n_rays_w);
    }
    umma_teardown(tmem_base);
}

template <int G, int NC, Loop L>
__global__ void __launch_bounds__(UmmaShape<G, NC>::kRenderThreads, 1)
render_kernel_umma(const RenderArgs<float> a, const CameraT<float>* __restrict__ cams, const AovArgs aov, const AdaptArgs ad)
{
    render_loop_umma<G, NC, L>(a, cams, aov, ad);
}

// Color::to_rgba (vec3.rs:404-420) + the row flip (main.rs:141-145): fixed-point sums -> RGBA8, each pixel quantised at spp, or
// at its own sample count spp_px[i] when spp_px is given (rtiow_render_adaptive).  Local pixel i is stored at its top-down place
// in `out` under the partition (world, rank).  A tile buffer in rank-local row order is the partition (1, 0).  A whole frame
// fuses the gather into the epilogue (single-process multi-GPU): `out` is then rank 0's frame, a peer pointer
// (cudaDeviceEnablePeerAccess), so for ranks > 0 these are st.global over NVLink — no tile buffer, no copy, no de-interleave
// pass.  Rows are written as whole 4-byte-per-pixel runs, i.e. coalesced 128-byte stores.
__global__ void finalize_kernel(const unsigned long long* __restrict__ accum, uint32_t n_lp, uint32_t spp, const uint32_t* __restrict__ spp_px,
                                uint32_t alpha, uint32_t width, uint32_t tile_rows, uint32_t world, uint32_t rank, uint32_t* __restrict__ out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_lp) return;
    const double k = 1.0 / 4294967296.0;
    const V3<double> sum = mk<double>((double)accum[i] * k, (double)accum[n_lp + i] * k, (double)accum[2 * (size_t)n_lp + i] * k);
    const uint32_t lr = i / width, x = i - lr * width;
    const uint32_t y = local_to_global_row(lr, tile_rows, world, rank);
    out[(size_t)y * width + x] = to_rgba<double>(sum, alpha, (uint64_t)(spp_px ? spp_px[i] : spp));
}

// The float epilogue of rtiow_render_aov: the frame's sums and the AOV accumulators (AovArgs) -> per-pixel means in this
// rank's local row order, each buffer [n_lp][3] (depth [n_lp]) one after the other in `out`: colour = sum / spp, albedo =
// sum / spp, normal = (sum - hits x 2^31) / 2^31 / spp (exact in 64-bit integers: the hits' offsets come off before any
// rounding, misses add 0), depth = sum / 2^16 / hits, or +inf when no camera ray of the pixel hit anything.
__global__ void finalize_aov_kernel(const unsigned long long* __restrict__ accum, const unsigned long long* __restrict__ aov_sum,
                                    const unsigned int* __restrict__ hits, uint32_t n_lp, uint32_t spp, float* __restrict__ out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_lp) return;
    const double inv_spp = 1.0 / (double)spp;
    const uint32_t h = hits[i];
    for (int c = 0; c < 3; ++c) {
        out[3 * (size_t)i + c] = (float)((double)accum[c * (size_t)n_lp + i] * (inv_spp / 4294967296.0));
        out[3 * ((size_t)n_lp + i) + c] = (float)((double)aov_sum[c * (size_t)n_lp + i] * (inv_spp / 4294967296.0));
        const long long nrm = (long long)(aov_sum[(3 + c) * (size_t)n_lp + i] - ((unsigned long long)h << 31));
        out[3 * (2 * (size_t)n_lp + i) + c] = (float)((double)nrm * (inv_spp / RT_AOV_NORMAL_SCALE));
    }
    out[9 * (size_t)n_lp + i] = h ? (float)((double)aov_sum[6 * (size_t)n_lp + i] / (RT_AOV_DEPTH_SCALE * h)) : __int_as_float(0x7f800000);
}

// ---- rtiow_render_adaptive: the rounds' bookkeeping (the epilogue is finalize_kernel at per-pixel counts) ---------------
// The error of a pixel at a boundary of n samples (include/rtiow_cuda.h): with m = S1 2^-32 / n and q = S2 2^-32 / n,
// err = 128 sqrt(max(0, q - m^2) / ((n - 1) max(m, 2^-16))), one standard error of the displayed value 256 sqrt(m) in 8-bit
// levels; +inf for n = 1.  Every operation is rounded on its own (no contraction), so a restatement in IEEE double from the
// same sums gives the same bits.
__device__ __forceinline__ double adapt_error(unsigned long long s1, unsigned long long s2, uint32_t n)
{
    if (n <= 1) return __longlong_as_double(0x7ff0000000000000ll);
    const double k = 1.0 / 4294967296.0, nd = (double)n;
    const double m = __ddiv_rn(__dmul_rn(__ull2double_rn(s1), k), nd);
    const double q = __ddiv_rn(__dmul_rn(__ull2double_rn(s2), k), nd);
    const double var = fmax(0.0, __dadd_rn(q, -__dmul_rn(m, m)));
    const double den = __dmul_rn((double)(n - 1), fmax(m, 1.0 / 65536.0));
    return __dmul_rn(128.0, __dsqrt_rn(__ddiv_rn(var, den)));
}

// the rule: a pixel at boundary n stays active iff its error, as out_error reports it (float), exceeds the tolerance and n is
// not the maximum
__device__ __forceinline__ bool adapt_keep(float err, double tol, uint32_t n, uint32_t n_max) { return n < n_max && (double)err > tol; }

#define RT_ADAPT_BLOCK 1024   // the select and compact kernels share their blocks: one list entry per thread, 32 warps

// the first round's list: every local pixel, bottom-up like the frame's chunks (assign_work)
__global__ void adapt_first_list_kernel(uint32_t n_lp, uint32_t* __restrict__ list)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_lp) list[i] = n_lp - 1u - i;
}

// After a round that brought every pixel of `list` to n samples: each gets its count and error, and each block counts the
// pixels that stay active (adapt_keep) into block_keep[block].
__global__ void __launch_bounds__(RT_ADAPT_BLOCK) adapt_select_kernel(const uint32_t* __restrict__ list, uint32_t n_act,
                                                                      const unsigned long long* __restrict__ lum_sum, uint32_t n_lp, uint32_t n,
                                                                      uint32_t n_max, double tol, uint32_t* __restrict__ spp_out,
                                                                      float* __restrict__ err_out, uint32_t* __restrict__ block_keep)
{
    const uint32_t i = blockIdx.x * RT_ADAPT_BLOCK + threadIdx.x;
    bool keep = false;
    if (i < n_act) {
        const uint32_t lp = list[i];
        const float err = (float)adapt_error(lum_sum[lp], lum_sum[n_lp + lp], n);
        spp_out[lp] = n; err_out[lp] = err;
        keep = adapt_keep(err, tol, n, n_max);
    }
    const int kept = __syncthreads_count(keep);
    if (threadIdx.x == 0) block_keep[blockIdx.x] = (uint32_t)kept;
}

// The next round's list: the active pixels of `list` in their order (a stable compaction, so every round still walks the frame
// bottom-up and ends on the sky rows).  A block's offset is the sum of the counts of the blocks before it; the last block also
// writes the length of the new list to *n_next.
__global__ void __launch_bounds__(RT_ADAPT_BLOCK) adapt_compact_kernel(const uint32_t* __restrict__ list, uint32_t n_act,
                                                                       const float* __restrict__ err_out, uint32_t n, uint32_t n_max, double tol,
                                                                       const uint32_t* __restrict__ block_keep, uint32_t* __restrict__ next,
                                                                       uint32_t* __restrict__ n_next)
{
    __shared__ uint32_t warp_n[32];
    __shared__ uint32_t base;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t before = 0;
    for (uint32_t b = threadIdx.x; b < blockIdx.x; b += RT_ADAPT_BLOCK) before += block_keep[b];
    before = __reduce_add_sync(RT_FULL, before);
    if (lane == 0) warp_n[warp] = before;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t s = 0; for (int w = 0; w < 32; ++w) s += warp_n[w]; base = s; }
    __syncthreads();
    const uint32_t i = blockIdx.x * RT_ADAPT_BLOCK + threadIdx.x;
    const bool keep = i < n_act && adapt_keep(err_out[list[i]], tol, n, n_max);
    const unsigned kept = __ballot_sync(RT_FULL, keep);
    if (lane == 0) warp_n[warp] = __popc(kept);
    __syncthreads();
    if (warp == 0) {                                          // exclusive scan of the 32 warps' counts
        const uint32_t v = warp_n[lane];
        uint32_t incl = v;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t u = __shfl_up_sync(RT_FULL, incl, o); if (lane >= (unsigned)o) incl += u; }
        warp_n[lane] = incl - v;
    }
    __syncthreads();
    if (keep) next[base + warp_n[warp] + __popc(kept & ((1u << lane) - 1u))] = list[i];
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) *n_next = base + block_keep[blockIdx.x];
}

// gathered tile buffers (rank-major, rank-local rows) -> top-down frame
__global__ void deinterleave_kernel(const uint32_t* __restrict__ gathered, uint32_t width, uint32_t height, uint32_t tile_rows,
                                    uint32_t world, size_t tile_buf_pixels, uint32_t* __restrict__ frame)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)width * height) return;
    const uint32_t y = (uint32_t)(i / width), x = (uint32_t)(i - (size_t)y * width);
    const uint32_t tg = y / tile_rows, within = y - tg * tile_rows;
    const uint32_t rank = tg % world, lr = (tg / world) * tile_rows + within;
    frame[i] = gathered[rank * tile_buf_pixels + (size_t)lr * width + x];
}

}  // namespace rt
