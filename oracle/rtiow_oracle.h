/*
 * rtiow_oracle.h — CPU oracle for the rtiow render hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * A plain-C, f64 restatement of the reference's algorithm (Druthyn/rtiow, Rust), function by
 * function, each citing the reference file:line it follows.  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load this library, and only as the
 * checker or as the timed CPU baseline — never on the product path.
 *
 * PARITY PINNING.  The reference ships no tests, golden vectors or seeded RNG path, and its
 * toolchain (rustc/cargo) is absent here, so the reference itself cannot be run.  Its only
 * result-bearing artefact is rtiow_part1_final.png (1200x800), and this oracle is pinned on every part of
 * that render that does not depend on the random small spheres (tests/test_oracle_golden.py):
 *   - the 58 sky-only rows: Camera::new + the miss branch of ray_color + Color::to_rgba + the row flip,
 *     within 1 LSB per pixel, four pixels exactly (tests/golden/png_sky_rows.json);
 *   - the sky-mirroring cap of the fixed Metal sphere (main.rs:98-99): Camera::get_ray, Sphere::hit (point,
 *     normal), Metal::scatter (reflect, albedo), the recursion — 391 9x9-block means within 0.25 LSB
 *     (measured: 0.05);
 *   - the sky seen through the fixed glass sphere (main.rs:93-94): Dialectric::scatter (refract, Schlick) —
 *     49 block means within -1.0 .. +2.5 LSB; and the top of the fixed Lambertian sphere (main.rs:95-96):
 *     Lambertian::scatter — 35 block means within -0.5 .. +4.5 LSB (the reference's random neighbourhood
 *     shades both slightly; tests/golden/png_big_spheres.json, generator committed);
 *   - the defocused horizon band beside the sphere field: the f64 ground sphere at grazing incidence, the thin
 *     lens and the Lambertian ground under open sky — 132 block means within 2.5 LSB, unbiased (|mean| <= 0.4).
 * What stays **parity unpinned** by the reference: Metal fuzz > 0 (the fixed sphere has fuzz 0), total
 * internal reflection and the exact rejection-sampler streams (thread_rng is unseedable), and `t` /
 * front_face as separate outputs; those are checked against analytic known answers and an independently
 * written numpy restatement (tests/np_restatement.py) only.
 *
 * Third-party arithmetic outside /root/reference: rand = "0.8.5" (Cargo.toml:11, Cargo.lock not
 * committed).  thread_rng() is OS-seeded ChaCha12 and cannot be reproduced; only its distributions
 * matter: gen::<f64>() = 53-bit uniform in [0,1); gen_range(a..b)/(a..=b) on f64 = uniform on the
 * range.  The oracle draws those from a counter-based Philox4x32-10 stream instead.
 */
#ifndef RTIOW_ORACLE_H
#define RTIOW_ORACLE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct { double x, y, z; } o_vec3;               /* vec3.rs:4-9 */
typedef struct { o_vec3 orig, dir; } o_ray;              /* ray.rs:5-8 */

typedef struct {                                          /* camera.rs:4-13 */
    o_vec3 origin, lower_left_corner, horizontal, vertical, u, v, w;
    double lens_radius;
} o_camera;

enum { O_MAT_LAMBERTIAN = 0, O_MAT_METAL = 1, O_MAT_DIELECTRIC = 2 };
typedef struct { int32_t kind; o_vec3 albedo; double param; } o_material; /* materials.rs:9-11,34-37,64-66 */

typedef struct { o_vec3 center; double radius; int32_t mat; } o_sphere;    /* sphere.rs:9-13 */

typedef struct {                                          /* shapes/mod.rs:10-16 */
    o_vec3 p, normal; int32_t mat; double t; int32_t front_face;
} o_hit_record;

typedef struct { const o_sphere* spheres; int32_t n_spheres; const o_material* materials; int32_t n_materials; } o_world;

/* ---- vec3.rs ------------------------------------------------------------------------------ */
o_vec3 o_v(double x, double y, double z);
o_vec3 o_add(o_vec3 a, o_vec3 b);          /* vec3.rs:137-147 */
o_vec3 o_sub(o_vec3 a, o_vec3 b);          /* vec3.rs:243-253 */
o_vec3 o_mul_s(o_vec3 a, double s);        /* vec3.rs:330-353 */
o_vec3 o_mul_v(o_vec3 a, o_vec3 b);        /* vec3.rs:355-367 */
o_vec3 o_div_s(o_vec3 a, double s);        /* vec3.rs:371-376: self * (1.0/scalar) */
double o_length_squared(o_vec3 a);         /* vec3.rs:87-89 */
double o_length(o_vec3 a);                 /* vec3.rs:83-85 */
double o_dot(o_vec3 a, o_vec3 b);          /* vec3.rs:95-97 */
o_vec3 o_cross(o_vec3 a, o_vec3 b);        /* vec3.rs:99-105 */
o_vec3 o_unit_vector(o_vec3 a);            /* vec3.rs:107-109 (norm at 91-93 is identical) */
int    o_is_near_zero(o_vec3 a);           /* vec3.rs:111-114 */
o_vec3 o_reflect(o_vec3 v, o_vec3 n);      /* vec3.rs:116-118 */
o_vec3 o_refract(o_vec3 uv, o_vec3 n, double etai_over_etat); /* vec3.rs:120-125 */
void   o_to_rgba(o_vec3 c, uint8_t alpha, uint64_t spp, uint8_t out[4]); /* vec3.rs:404-420 */

/* ---- ray.rs ------------------------------------------------------------------------------- */
o_vec3 o_ray_at(const o_ray* r, double t); /* ray.rs:15-17 */

/* ---- camera.rs ---------------------------------------------------------------------------- */
void  o_camera_new(o_camera* cam, o_vec3 look_from, o_vec3 look_at, o_vec3 v_up, double v_fov,
                   double aspect_ratio, double aperture, double focus_dist);           /* camera.rs:17-45 */
/* disk_x, disk_y: the ACCEPTED sample of Vec3::random_in_unit_disk (injection point, camera.rs:48) */
o_ray o_camera_get_ray(const o_camera* cam, double s, double t, double disk_x, double disk_y); /* camera.rs:47-54 */

/* ---- shapes -------------------------------------------------------------------------------- */
int o_sphere_hit(const o_sphere* s, const o_ray* r, double t_min, double t_max, o_hit_record* rec);  /* sphere.rs:16-41 + mod.rs:20-30 */
int o_world_hit(const o_world* w, const o_ray* r, double t_min, double t_max, o_hit_record* rec, int32_t* index); /* mod.rs:56-69 */

/* ---- materials.rs (random numbers injected) ---------------------------------------------------
 * sample: Lambertian — the accepted in-unit-sphere vector BEFORE normalisation (vec3.rs:47-49);
 *         Metal      — the accepted in-unit-sphere vector (materials.rs:53);
 *         Dialectric — sample.x is the uniform xi of materials.rs:96 (ignored under TIR).
 * returns 1 = Some((attenuation, scattered)), 0 = None. */
int o_scatter(const o_material* m, const o_ray* r_in, const o_hit_record* rec, o_vec3 sample,
              o_vec3* attenuation, o_ray* scattered);                                  /* materials.rs:22-30,50-61,77-104 */
double o_reflectance(double cosine, double ref_idx);                                   /* materials.rs:78-82 */

/* ---- Philox4x32-10 (Salmon et al., SC'11; Random123) --------------------------------------- */
void o_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

/* ---- samplers --------------------------------------------------------------------------------
 * Two ways of turning random bits into the distributions of Appendix B:
 *  O_SAMPLER_REJECTION  reference-faithful rejection loops (vec3.rs:37-49,59-68) and draw order
 *                       (main.rs:131-132, camera.rs:48, materials.rs:23,53,96), fed by a per-path
 *                       counter stream of 53-bit uniforms;
 *  O_SAMPLER_DIRECT     the CUDA path's mapping: ONE Philox block per event keyed
 *                       (seed; pixel, sample, bounce), 24-bit uniforms, inversion sampling of the
 *                       same distributions.  Lets oracle and GPU follow the same paths.          */
enum { O_SAMPLER_REJECTION = 0, O_SAMPLER_DIRECT = 1 };

typedef struct {
    uint32_t key[2];
    uint32_t pixel, sample;
    uint32_t draw;            /* REJECTION: running draw index inside this path */
    int32_t  mode;
} o_rng;

void   o_rng_init(o_rng* g, uint64_t seed, uint32_t pixel, uint32_t sample, int32_t mode);
double o_rng_f64(o_rng* g);                                  /* gen::<f64>() : [0,1), 53 bits */
double o_rng_range(o_rng* g, double lo, double hi);         /* gen_range(lo..hi) / (lo..=hi) */
o_vec3 o_random_in_unit_sphere(o_rng* g);                    /* vec3.rs:37-45 */
o_vec3 o_random_unit_vector(o_rng* g);                       /* vec3.rs:47-49 */
o_vec3 o_random_in_unit_disk(o_rng* g);                      /* vec3.rs:59-68 */
/* DIRECT mapping of one Philox block (4 x 24-bit uniforms u[0..3] in [0,1)) */
void   o_direct_uniforms(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t bounce, double u[4]);
void   o_direct_disk(double u2, double u3, double* x, double* y);
o_vec3 o_direct_unit_vector(double u0, double u1);
o_vec3 o_direct_in_unit_sphere(double u0, double u1, double u2);

/* ---- main.rs integrator -------------------------------------------------------------------- */
typedef struct { uint64_t rays, sphere_tests; } o_counters;
/* ray_color, main.rs:38-57 — recursive exactly as written.  bounce = index of this ray in its path
 * (0 = camera ray); in DIRECT mode the scatter at this ray's hit uses Philox block (bounce+1). */
o_vec3 o_ray_color(const o_ray* r, const o_world* w, int32_t depth, double t_min, o_rng* g,
                   uint32_t bounce, o_counters* cnt);

typedef struct {
    uint32_t width, height, spp;
    int32_t  max_depth;
    double   t_min;
    uint64_t seed;
    uint8_t  alpha;
    int32_t  sampler;          /* O_SAMPLER_* */
    int32_t  n_threads;        /* 0 = all */
    uint32_t row_begin, row_end; /* top-down output rows to render [begin,end); 0,0 = all */
} o_render_params;

/* pixel/sample loop + quantise + row flip, main.rs:122-145.  out_rgba: 4*width*height bytes,
 * top-down.  accum (optional, may be NULL): 3*width*height doubles, per-pixel radiance SUM,
 * top-down, before to_rgba.  Rows are OpenMP schedule(dynamic,1), mirroring rayon-per-row. */
int o_render(const o_world* w, const o_camera* cam, const o_render_params* p, uint8_t* out_rgba,
             double* accum, o_counters* cnt);

/* o_render with the DIRECT sampler (the same bytes, sums and counters), plus margin[H][W] (top-down): how far each pixel is
 * from a decision an f32 render could take the other way.  It is the smallest margin over every ray of the pixel's paths;
 * a ray's margin is the smallest of these normalised distances from a decision boundary, each divided by the ray's error
 * growth (below):
 *   grazing    |r^2 - dist(centre, line)^2| / (|r| L) for every sphere with a root in [t_min, t_winner], or whose line
 *              passes outside it with tca in that range (a near miss in front of the winner);
 *   t_min      |root - t_min| |dir| / L for every root of every sphere (not the near-zero root of the sphere the ray
 *              starts on, which the renderer drops without computing it);
 *   near tie   (t2 - t1) |dir| / L between the two smallest accepted roots (not between coincident spheres, which tie
 *              exactly in f32 too);
 *   dielectric |ratio sin(theta) - 1| and, when it can refract, |reflectance - xi|;
 *   metal      dot(d, n) / |d| (the absorption test);
 *   lambertian |n + unit(sample)| (the near-zero fallback).
 * L = |o| + |o - c| + |r| is the size of the numbers the sphere's roots are computed from: f32 rounding moves a root by
 * about eps32 L.  The growth starts at 1 on the camera ray and is multiplied at every hit by 1 + k L_next / |r| (L_next:
 * the distance from the hit to the point of the next ray being judged; k = O_MARGIN_K_SPECULAR for a mirror or glass
 * bounce, whose direction turns by twice the normal's error, O_MARGIN_K_LAMBERTIAN for a diffuse one, whose direction is
 * offset by the normal's), and by Snell's amplification ratio cos(theta) / cos(theta_out) on a refraction.  Without the
 * growth, long mirror and glass chains look robust where an f32 render leaves them. */
#define O_MARGIN_K_SPECULAR 2.0
#define O_MARGIN_K_LAMBERTIAN 1.0
int o_render_margins(const o_world* w, const o_camera* cam, const o_render_params* p, uint8_t* out_rgba, double* accum,
                     double* margin, o_counters* cnt);

/* one path: pixel (i, j) with j=0 the BOTTOM row (main.rs:131-135), sample index s */
o_vec3 o_path_radiance(const o_world* w, const o_camera* cam, const o_render_params* p,
                       uint32_t i, uint32_t j, uint32_t s, o_counters* cnt);

/* ---- batch helpers (plain loops over the functions above; arrays are row-major [n][3]) ------ */
void o_sphere_hit_batch(int64_t n, const double* center, const double* radius, const double* orig,
                        const double* dir, const double* t_min, const double* t_max,
                        int32_t* hit, double* t, double* p, double* normal, int32_t* front_face);
void o_world_hit_batch(const o_world* w, int64_t n, const double* orig, const double* dir, double t_min,
                       double t_max, int32_t* hit, int32_t* index, double* t, double* p, double* normal,
                       int32_t* front_face);
void o_scatter_batch(int64_t n, const int32_t* kind, const double* albedo, const double* param,
                     const double* r_orig, const double* r_dir, const double* p, const double* normal,
                     const int32_t* front_face, const double* sample, int32_t* some,
                     double* attenuation, double* s_orig, double* s_dir);
void o_get_ray_batch(const o_camera* cam, int64_t n, const double* s, const double* t,
                     const double* disk_xy, double* orig, double* dir);
void o_to_rgba_batch(int64_t n, const double* color, uint8_t alpha, uint64_t spp, uint8_t* out);
void o_reflect_batch(int64_t n, const double* v, const double* nrm, double* out);
void o_refract_batch(int64_t n, const double* uv, const double* nrm, const double* eta, double* out);
/* n draws of a reference rejection sampler (which: 0 = random_in_unit_disk, 1 = random_in_unit_sphere,
 * 2 = random_unit_vector), stream (seed; pixel = i, sample = 0).  out: [n][3] */
void o_rejection_samples(uint64_t seed, int64_t n, int32_t which, double* out);
/* ray_color on explicit rays with the DIRECT sampler keyed (seed; pixel[i], sample[i], bounce) */
void o_ray_color_batch(const o_world* w, int64_t n, const double* orig, const double* dir,
                       const uint32_t* pixel, const uint32_t* sample, uint64_t seed, int32_t max_depth,
                       double t_min, double* color, uint64_t* rays);

#ifdef __cplusplus
}
#endif
#endif
