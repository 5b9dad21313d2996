// rt_unit.cuh — unit-level kernels behind the rtiow_*_batch entry points: thin wrappers that run
// the renderer's own __device__ functions on explicit inputs with injected random numbers
// (SURVEY Appendix B), so that parity is checked on the code that renders.
// I/O is double on both sides; the arithmetic in between is real_t = T.
#pragma once
#include "rt_render.cuh"

namespace rt {

template <typename T> __device__ __forceinline__ V3<T> ld3(const double* a, int64_t i) { return mk<T>((T)a[3 * i], (T)a[3 * i + 1], (T)a[3 * i + 2]); }
template <typename T> __device__ __forceinline__ void st3(double* a, int64_t i, V3<T> v) { a[3 * i] = (double)v.x; a[3 * i + 1] = (double)v.y; a[3 * i + 2] = (double)v.z; }

// Sphere::hit (sphere.rs:16-41) + HitRecord::new (mod.rs:20-30), one (sphere, ray) pair per thread
template <typename T>
__global__ void sphere_hit_kernel(int64_t n, const double* center, const double* radius, const double* orig, const double* dir,
                                  const double* t_min, const double* t_max, int32_t* hit, double* t, double* p, double* normal,
                                  int32_t* front_face)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const V3<T> c = ld3<T>(center, i), o = ld3<T>(orig, i), d = ld3<T>(dir, i);
    const T r = (T)radius[i];
    const T len = length(d), inv_len = T(1) / len;
    const V3<T> dhat = d * inv_len;
    const T tmin_n = (T)t_min[i] * len, tmax_n = (T)t_max[i] * len;
    T root = T(0);
    bool h = sphere_roots(c - o, dhat, T(1) / length_squared(dhat), r * r, tmin_n, tmax_n, &root);
    V3<T> pp = mk<T>(0, 0, 0), nn = mk<T>(0, 0, 0); bool ff = false;
    if (h) { pp = o + dhat * root; hit_record(pp, c, r, dhat, &nn, &ff); }
    hit[i] = h ? 1 : 0; t[i] = h ? (double)(root * inv_len) : 0.0;
    st3(p, i, pp); st3(normal, i, nn); front_face[i] = ff ? 1 : 0;
}

// Ray i of a hitlist batch as the scan takes it (a lane past n gets a dummy ray): ps.o, ps.dhat, ps.tmin_n, no self sphere.
// Returns 1/|dir|, which takes t back to |dir| units; it is a division, not start_ray's rsqrtf.
template <typename T>
__device__ __forceinline__ T hitlist_ray(PathState<T>& ps, int64_t i, int64_t n, const double* orig, const double* dir, double t_min)
{
    V3<T> o = mk<T>(0, 0, 0), d = mk<T>(0, 1, 0);
    if (i < n) { o = ld3<T>(orig, i); d = ld3<T>(dir, i); }
    const T len = length(d), inv_len = T(1) / len;
    ps.o = o; ps.dhat = d * inv_len; ps.tmin_n = (T)t_min * len;
    ps.self_code = RT_SELF_NONE; ps.self_n = mk<T>(0, 1, 0);
    return inv_len;
}

// HittableList::hit's result for ray i: the closest hit (t_hit, idx) found by the scan, with its HitRecord (mod.rs:20-30).
// ps is taken by value: by reference, nvcc contracts hitlist_ray's |dir|^2 in another order, which moves the last bits of t.
template <typename T>
__device__ __forceinline__ void store_hit(const SceneDev& sc, int64_t i, const PathState<T> ps, T inv_len, T t_hit, int idx,
                                          int32_t* hit, int32_t* index, double* t, double* p, double* normal, int32_t* front_face)
{
    V3<T> pp = mk<T>(0, 0, 0), nn = mk<T>(0, 0, 0); bool ff = false;
    if (idx >= 0) {
        V3<T> cen; T rad;
        if (sizeof(T) == 4) { const float4 s = sc.sph[idx]; cen = mk<T>(s.x, s.y, s.z); rad = s.w; }
        else { const double4 s = sc.sphd[idx]; cen = mk<T>(s.x, s.y, s.z); rad = s.w; }
        pp = ps.o + ps.dhat * t_hit; hit_record(pp, cen, rad, ps.dhat, &nn, &ff);
    }
    hit[i] = idx >= 0; index[i] = idx; t[i] = idx >= 0 ? (double)(t_hit * inv_len) : 0.0;
    st3(p, i, pp); st3(normal, i, nn); front_face[i] = ff ? 1 : 0;
}

// HittableList::hit (mod.rs:56-69) through the renderer's scan
template <typename T, bool kSmem, int kThreads>
__global__ void __launch_bounds__(kThreads) hitlist_kernel(SceneDev sc, int64_t n, const double* orig, const double* dir, double t_min,
                                                           int32_t* hit, int32_t* index, double* t, double* p, double* normal, int32_t* front_face)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint16_t* cand;
    const float* table = setup_scan_smem<kSmem>(smem_raw, sc, kThreads, &cand);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    PathState<T> ps;
    const T inv_len = hitlist_ray(ps, i, n, orig, dir, t_min);
    T th; int idx, code;
    world_hit<T, kSmem>(sc, table, cand, kThreads, ps, &th, &idx, &code);
    if (i < n) store_hit(sc, i, ps, inv_len, th, idx, hit, index, t, p, normal, front_face);
}

// the same through the tensor-core scan (rt_umma_scan.cuh): 128 rays per group, G groups + G issuer warps per CTA
template <int G, int NC>
__global__ void __launch_bounds__(G * 160, 1) hitlist_kernel_umma(SceneDev sc, int64_t n, const double* orig, const double* dir, double t_min,
                                                                  int32_t* hit, int32_t* index, double* t, double* p, double* normal, int32_t* front_face)
{
    extern __shared__ __align__(1024) unsigned char smem_umma[];
    uint32_t tmem_base;
    UmmaCtx ux = umma_setup<G, NC>(smem_umma, sc, &tmem_base);
    if (ux.issuer_warp) {
        umma_issuer<G, NC>(ux);
    } else {
        const int64_t i = (int64_t)blockIdx.x * (G * 128) + threadIdx.x;
        PathState<float> ps;
        const float inv_len = hitlist_ray(ps, i, n, orig, dir, t_min);
        const HitF h = closest_hit_umma<G, NC>(ux, sc, ps.o, ps.dhat, ps.tmin_n, ps.self_code, ps.self_n);
        umma_group_quit(ux);
        if (i < n) store_hit(sc, i, ps, inv_len, h.t, h.idx, hit, index, t, p, normal, front_face);
    }
    umma_teardown(tmem_base);
}

// Scatter::scatter (materials.rs:22-30,50-61,77-104)
template <typename T>
__global__ void scatter_kernel(int64_t n, const int32_t* kind, const double* albedo, const double* param, const double* r_orig,
                               const double* r_dir, const double* p, const double* normal, const int32_t* front_face,
                               const double* sample, int32_t* some, double* attenuation, double* s_orig, double* s_dir)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    (void)r_orig;
    V3<T> att = mk<T>(0, 0, 0), nd = mk<T>(0, 0, 0);
    const bool s = scatter<T>(kind[i], ld3<T>(albedo, i), (T)param[i], ld3<T>(r_dir, i), ld3<T>(normal, i), front_face[i] != 0,
                              ld3<T>(sample, i), &att, &nd);
    some[i] = s ? 1 : 0;
    if (!s) { att = mk<T>(0, 0, 0); }
    st3(attenuation, i, att); st3(s_orig, i, ld3<T>(p, i)); st3(s_dir, i, nd);
}

// Camera::get_ray (camera.rs:47-54)
template <typename T>
__global__ void get_ray_kernel(CameraT<T> cam, int64_t n, const double* s, const double* t, const double* disk_xy, double* orig, double* dir)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    V3<T> o, d; get_ray<T>(cam, (T)s[i], (T)t[i], (T)disk_xy[2 * i], (T)disk_xy[2 * i + 1], &o, &d);
    st3(orig, i, o); st3(dir, i, d);
}

// Color::to_rgba (vec3.rs:404-420)
template <typename T>
__global__ void to_rgba_kernel(int64_t n, const double* color, uint32_t alpha, uint64_t spp, uint32_t* out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = to_rgba<T>(ld3<T>(color, i), alpha, spp);
}

template <typename T> __global__ void reflect_kernel(int64_t n, const double* v, const double* nrm, double* out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    st3(out, i, reflect(ld3<T>(v, i), ld3<T>(nrm, i)));                  // vec3.rs:116-118
}
template <typename T> __global__ void refract_kernel(int64_t n, const double* uv, const double* nrm, const double* eta, double* out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    st3(out, i, refract(ld3<T>(uv, i), ld3<T>(nrm, i), (T)eta[i]));      // vec3.rs:120-125
}

// the sampler mapping: out[i] = {u0,u1,u2,u3, disk.x,disk.y, unit.xyz, ball.xyz}
template <typename T>
__global__ void sampler_kernel(int64_t n, const uint32_t* pixel, const uint32_t* sample, const uint32_t* bounce, uint64_t seed, double* out)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Uniform4<T> u = event_uniforms<T>(seed, pixel[i], sample[i], bounce[i]);
    T dx, dy; direct_disk(u.u2, u.u3, &dx, &dy);
    const V3<T> uv = direct_unit_vector(u.u0, u.u1), bv = direct_in_unit_sphere(u.u0, u.u1, u.u2);
    double* o = out + 12 * i;
    o[0] = u.u0; o[1] = u.u1; o[2] = u.u2; o[3] = u.u3; o[4] = dx; o[5] = dy;
    o[6] = uv.x; o[7] = uv.y; o[8] = uv.z; o[9] = bv.x; o[10] = bv.y; o[11] = bv.z;
}

// The path of ray i of a ray_color batch: throughput 1, depth max_depth, keyed (pixel[i], sample[i]).  Returns whether the
// lane has a ray (a lane past n gets a dummy path).
template <typename T>
__device__ __forceinline__ bool ray_color_start(PathState<T>& ps, int64_t i, int64_t n, const double* orig, const double* dir, const uint32_t* pixel,
                                                const uint32_t* sample, int32_t max_depth, double t_min)
{
    init_path(ps);
    ps.thr = mk<T>(1, 1, 1); ps.depth = max_depth;
    if (i < n) { start_ray(ps, ld3<T>(orig, i), ld3<T>(dir, i), (T)t_min); ps.pix_key = pixel[i]; ps.smp = sample[i]; }
    return i < n && max_depth > 0;
}

// bounce_step for a lane whose scan found (t_hit, idx, code) for its ray nr, which goes to trace_ray / trace_idx when they
// are given.  Returns the lane's new `active`; when the path ends, *result receives its radiance.
template <typename T>
__device__ __forceinline__ bool ray_color_bounce(const SceneDev& sc, const PhiloxKey& key, int32_t max_depth, double t_min, int64_t i, uint32_t& nr,
                                                 int32_t* trace_idx, double* trace_ray, PathState<T>& ps, T t_hit, int idx, int code, V3<T>* result)
{
    const size_t k = (size_t)i * max_depth + nr++;                            // world.hit call count (main.rs:44)
    if (trace_ray) { double* tr = trace_ray + k * 6; tr[0] = ps.o.x; tr[1] = ps.o.y; tr[2] = ps.o.z; tr[3] = ps.dhat.x; tr[4] = ps.dhat.y; tr[5] = ps.dhat.z; }
    if (trace_idx) trace_idx[k] = idx;
    return bounce_step(sc, key, max_depth, (T)t_min, ps, t_hit, idx, code, result);
}

// ray_color (main.rs:38-57): the renderer's bounce loop on explicit rays
template <typename T, bool kSmem, int kThreads>
__global__ void __launch_bounds__(kThreads) ray_color_kernel(SceneDev sc, int64_t n, const double* orig, const double* dir, const uint32_t* pixel,
                                                             const uint32_t* sample, uint64_t seed, int32_t max_depth, double t_min,
                                                             double* color, unsigned long long* rays, int32_t* trace_idx, double* trace_ray)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint16_t* cand;
    const float* table = setup_scan_smem<kSmem>(smem_raw, sc, kThreads, &cand);
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    PathState<T> ps;
    bool active = ray_color_start(ps, i, n, orig, dir, pixel, sample, max_depth, t_min);
    const PhiloxKey key = philox_key(seed);
    V3<T> result = mk<T>(0, 0, 0);
    uint32_t nr = 0;
    while (__any_sync(RT_FULL, active)) {
        T t_hit; int idx, code;
        world_hit<T, kSmem>(sc, table, cand, kThreads, ps, &t_hit, &idx, &code);
        if (active) active = ray_color_bounce(sc, key, max_depth, t_min, i, nr, trace_idx, trace_ray, ps, t_hit, idx, code, &result);
    }
    if (i < n) { st3(color, i, result); if (rays) rays[i] = nr; }
}

// ray_color through the tensor-core scan: the same bounce loop, 128 rays per group in lock step
template <int G, int NC>
__global__ void __launch_bounds__(G * 160, 1) ray_color_kernel_umma(SceneDev sc, int64_t n, const double* orig, const double* dir, const uint32_t* pixel,
                                                                    const uint32_t* sample, uint64_t seed, int32_t max_depth, double t_min,
                                                                    double* color, unsigned long long* rays, int32_t* trace_idx, double* trace_ray)
{
    extern __shared__ __align__(1024) unsigned char smem_umma[];
    uint32_t tmem_base;
    UmmaCtx ux = umma_setup<G, NC>(smem_umma, sc, &tmem_base);
    if (ux.issuer_warp) {
        umma_issuer<G, NC>(ux);
    } else {
        const int64_t i = (int64_t)blockIdx.x * (G * 128) + threadIdx.x;
        PathState<float> ps;
        bool active = ray_color_start(ps, i, n, orig, dir, pixel, sample, max_depth, t_min);
        const PhiloxKey key = philox_key(seed);
        V3<float> result = mk<float>(0, 0, 0);
        uint32_t nr = 0;
        while (umma_group_any(ux, active)) {
            const HitF h = closest_hit_umma<G, NC>(ux, sc, ps.o, ps.dhat, ps.tmin_n, ps.self_code, ps.self_n, active);
            if (active) active = ray_color_bounce(sc, key, max_depth, t_min, i, nr, trace_idx, trace_ray, ps, h.t, h.idx, h.code, &result);
        }
        umma_group_quit(ux);
        if (i < n) { st3(color, i, result); if (rays) rays[i] = nr; }
    }
    umma_teardown(tmem_base);
}

// ---- FP32-pipe calibration kernels (roofline denominator) -----------------------------------------
__global__ void __launch_bounds__(256) probe_ffma_kernel(float* out, int iters, float a, float b)
{
    float x[8];
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = threadIdx.x * 0.001f + i;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
#pragma unroll
            for (int i = 0; i < 8; i++) x[i] = fmaf(x[i], a, b);
        }
    }
    float s = 0;
    for (int i = 0; i < 8; i++) s += x[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void __launch_bounds__(256) probe_ffma2_kernel(float* out, int iters, float a, float b)
{
    float2 x[8];
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = make_float2(threadIdx.x * 0.001f + i, i * 0.5f);
    const float2 A = bc2(a), B = bc2(b);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
#pragma unroll
            for (int i = 0; i < 8; i++) x[i] = ffma2(x[i], A, B);
        }
    }
    float s = 0;
    for (int i = 0; i < 8; i++) s += x[i].x + x[i].y;
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void flush_kernel(uint4* buf, size_t n, uint32_t v)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) buf[i] = make_uint4(v, v, v, v);
}

}  // namespace rt
