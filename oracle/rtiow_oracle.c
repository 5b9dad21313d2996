/*
 * rtiow_oracle.c — CPU oracle (f64) for the rtiow render hot path.  TEST INFRASTRUCTURE ONLY.
 * See rtiow_oracle.h for the scope statement and the "parity unpinned" note.
 *
 * Every function restates one reference function; the citation is /root/reference/src/<file>:<lines>.
 * Build with -ffp-contract=off: rustc never fuses a*b+c, so neither may this file.
 */
#include "rtiow_oracle.h"
#include <math.h>
#include <string.h>
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ============================== vec3.rs ================================================== */

o_vec3 o_v(double x, double y, double z) { o_vec3 r = { x, y, z }; return r; }      /* vec3.rs:17-19 */
o_vec3 o_add(o_vec3 a, o_vec3 b) { return o_v(a.x + b.x, a.y + b.y, a.z + b.z); }  /* vec3.rs:137-147 */
o_vec3 o_sub(o_vec3 a, o_vec3 b) { return o_v(a.x - b.x, a.y - b.y, a.z - b.z); }  /* vec3.rs:243-253 */
o_vec3 o_mul_s(o_vec3 a, double s) { return o_v(a.x * s, a.y * s, a.z * s); }      /* vec3.rs:330-353 */
o_vec3 o_mul_v(o_vec3 a, o_vec3 b) { return o_v(a.x * b.x, a.y * b.y, a.z * b.z); }/* vec3.rs:355-367 */

/* vec3.rs:371-376 — Div<f64> is `self * (1.0/scalar)`: one reciprocal, three multiplies. */
o_vec3 o_div_s(o_vec3 a, double s) { return o_mul_s(a, 1.0 / s); }

/* vec3.rs:87-89 — x.powi(2)+y.powi(2)+z.powi(2); powi(2) is x*x, summed left to right. */
double o_length_squared(o_vec3 a) { return a.x * a.x + a.y * a.y + a.z * a.z; }
double o_length(o_vec3 a) { return sqrt(o_length_squared(a)); }                      /* vec3.rs:83-85 */
double o_dot(o_vec3 a, o_vec3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }      /* vec3.rs:95-97 */

o_vec3 o_cross(o_vec3 a, o_vec3 b)                                                   /* vec3.rs:99-105 */
{
    return o_v(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}

o_vec3 o_unit_vector(o_vec3 a) { return o_div_s(a, o_length(a)); }                   /* vec3.rs:107-109 */

int o_is_near_zero(o_vec3 a)                                                         /* vec3.rs:111-114 */
{
    const double s = 1e-8;
    return fabs(a.x) < s && fabs(a.y) < s && fabs(a.z) < s;
}

/* vec3.rs:116-118 — self - 2.0*self.dot(n) * *n : (2*dot) first, then scalar*vector. */
o_vec3 o_reflect(o_vec3 v, o_vec3 n) { return o_sub(v, o_mul_s(n, 2.0 * o_dot(v, n))); }

o_vec3 o_refract(o_vec3 uv, o_vec3 n, double etai_over_etat)                         /* vec3.rs:120-125 */
{
    double cos_theta = fmin(1.0, -o_dot(uv, n));
    o_vec3 r_out_perp = o_mul_s(o_add(uv, o_mul_s(n, cos_theta)), etai_over_etat);
    o_vec3 r_out_parallel = o_mul_s(n, -sqrt(fabs(1.0 - o_length_squared(r_out_perp))));
    return o_add(r_out_perp, r_out_parallel);
}

/* Rust `f64 as u8`: truncate toward zero, saturate to [0,255], NaN -> 0. */
static uint8_t rust_f64_as_u8(double v)
{
    if (isnan(v)) return 0;
    if (v <= 0.0) return 0;
    if (v >= 255.0) return 255;
    return (uint8_t)v;
}

/* Rust f64::clamp(min,max): NaN stays NaN. */
static double rust_clamp(double v, double lo, double hi)
{
    if (v < lo) return lo;
    if (v > hi) return hi;
    return v;
}

void o_to_rgba(o_vec3 c, uint8_t alpha, uint64_t spp, uint8_t out[4])               /* vec3.rs:404-420 */
{
    double scale = 1.0 / (double)spp;
    double r = sqrt(scale * c.x), g = sqrt(scale * c.y), b = sqrt(scale * c.z);
    out[0] = rust_f64_as_u8(256.0 * rust_clamp(r, 0.0, 0.999));
    out[1] = rust_f64_as_u8(256.0 * rust_clamp(g, 0.0, 0.999));
    out[2] = rust_f64_as_u8(256.0 * rust_clamp(b, 0.0, 0.999));
    out[3] = alpha;
}

/* ============================== ray.rs =================================================== */

o_vec3 o_ray_at(const o_ray* r, double t) { return o_add(r->orig, o_mul_s(r->dir, t)); } /* ray.rs:15-17 */

/* ============================== camera.rs ================================================ */

void o_camera_new(o_camera* cam, o_vec3 look_from, o_vec3 look_at, o_vec3 v_up, double v_fov,
                  double aspect_ratio, double aperture, double focus_dist)           /* camera.rs:17-45 */
{
    /* f64::to_radians multiplies by the constant PI/180 (camera.rs:25) */
    double theta = v_fov * (3.14159265358979323846264338327950288 / 180.0);
    double viewport_height = 2.0 * tan(theta / 2.0);
    double viewport_width = aspect_ratio * viewport_height;

    o_vec3 w = o_unit_vector(o_sub(look_from, look_at));
    o_vec3 u = o_unit_vector(o_cross(v_up, w));
    o_vec3 v = o_cross(w, u);

    /* focus_dist * viewport_width * u parses as (focus_dist*viewport_width) * u (camera.rs:33-34) */
    o_vec3 horizontal = o_mul_s(u, focus_dist * viewport_width);
    o_vec3 vertical = o_mul_s(v, focus_dist * viewport_height);
    o_vec3 llc = o_sub(o_sub(o_sub(look_from, o_div_s(horizontal, 2.0)), o_div_s(vertical, 2.0)),
                       o_mul_s(w, focus_dist));                                     /* camera.rs:35 */
    cam->origin = look_from;
    cam->lower_left_corner = llc;
    cam->horizontal = horizontal;
    cam->vertical = vertical;
    cam->u = u; cam->v = v; cam->w = w;
    cam->lens_radius = aperture / 2.0;
}

o_ray o_camera_get_ray(const o_camera* cam, double s, double t, double disk_x, double disk_y) /* camera.rs:47-54 */
{
    o_vec3 rd = o_mul_s(o_v(disk_x, disk_y, 0.0), cam->lens_radius);
    o_vec3 offset = o_add(o_mul_s(cam->u, rd.x), o_mul_s(cam->v, rd.y));
    o_ray r;
    r.orig = o_add(cam->origin, offset);
    r.dir = o_sub(o_sub(o_add(o_add(cam->lower_left_corner, o_mul_s(cam->horizontal, s)),
                              o_mul_s(cam->vertical, t)), cam->origin), offset);
    return r;
}

/* ============================== shapes ==================================================== */

int o_sphere_hit(const o_sphere* s, const o_ray* r, double t_min, double t_max, o_hit_record* rec)
{                                                                                    /* sphere.rs:16-41 */
    o_vec3 oc = o_sub(r->orig, s->center);
    double a = o_length_squared(r->dir);
    double half_b = o_dot(oc, r->dir);
    double c = o_length_squared(oc) - s->radius * s->radius;

    double discriminant = half_b * half_b - a * c;
    if (discriminant < 0.0) return 0;
    double sqrtd = sqrt(discriminant);

    double root = (-half_b - sqrtd) / a;
    if (root < t_min || t_max < root) {
        root = (-half_b + sqrtd) / a;
        if (root < t_min || t_max < root) return 0;
    }
    o_vec3 p = o_ray_at(r, root);
    o_vec3 outward_normal = o_div_s(o_sub(p, s->center), s->radius);
    /* HitRecord::new, shapes/mod.rs:20-30 */
    int front_face = o_dot(r->dir, outward_normal) < 0.0;
    rec->p = p;
    rec->normal = front_face ? outward_normal : o_sub(o_v(0, 0, 0), outward_normal);
    rec->mat = s->mat;
    rec->t = root;
    rec->front_face = front_face;
    return 1;
}

int o_world_hit(const o_world* w, const o_ray* r, double t_min, double t_max, o_hit_record* rec, int32_t* index)
{                                                                                    /* shapes/mod.rs:56-69 */
    int found = 0;
    double closest_so_far = t_max;
    o_hit_record tmp;
    for (int32_t i = 0; i < w->n_spheres; ++i) {
        if (o_sphere_hit(&w->spheres[i], r, t_min, closest_so_far, &tmp)) {
            closest_so_far = tmp.t;
            *rec = tmp;
            if (index) *index = i;
            found = 1;
        }
    }
    return found;
}

/* ============================== materials.rs ============================================== */

double o_reflectance(double cosine, double ref_idx)                                  /* materials.rs:78-82 */
{
    double r0 = (1.0 - ref_idx) / (1.0 + ref_idx);
    r0 = r0 * r0;
    double m = 1.0 - cosine;
    return r0 + (1.0 - r0) * (m * m * m * m * m);
}

int o_scatter(const o_material* m, const o_ray* r_in, const o_hit_record* rec, o_vec3 sample,
              o_vec3* attenuation, o_ray* scattered)
{
    switch (m->kind) {
    case O_MAT_LAMBERTIAN: {                                                         /* materials.rs:22-30 */
        o_vec3 scatter_direction = o_add(rec->normal, o_unit_vector(sample));        /* vec3.rs:47-49 */
        if (o_is_near_zero(scatter_direction)) scatter_direction = rec->normal;
        scattered->orig = rec->p;
        scattered->dir = scatter_direction;
        *attenuation = m->albedo;
        return 1;
    }
    case O_MAT_METAL: {                                                              /* materials.rs:50-61 */
        o_vec3 reflected = o_unit_vector(o_reflect(r_in->dir, rec->normal));
        scattered->orig = rec->p;
        scattered->dir = o_add(reflected, o_mul_s(sample, m->param));
        if (o_dot(scattered->dir, rec->normal) <= 0.0) return 0;
        *attenuation = m->albedo;
        return 1;
    }
    case O_MAT_DIELECTRIC: {                                                         /* materials.rs:77-104 */
        double refraction_ratio = rec->front_face ? 1.0 / m->param : m->param;
        o_vec3 unit_direction = o_unit_vector(r_in->dir);
        double cos_theta = fmin(1.0, -o_dot(unit_direction, rec->normal));
        double sin_theta = sqrt(1.0 - cos_theta * cos_theta);
        int can_refract = refraction_ratio * sin_theta <= 1.0;
        o_vec3 direction;
        /* short-circuit: xi is consumed only when can_refract (materials.rs:96) */
        if (can_refract && o_reflectance(cos_theta, refraction_ratio) <= sample.x)
            direction = o_refract(unit_direction, rec->normal, refraction_ratio);
        else
            direction = o_reflect(unit_direction, rec->normal);
        scattered->orig = rec->p;
        scattered->dir = direction;
        *attenuation = o_v(1, 1, 1);
        return 1;
    }
    default:
        return 0;
    }
}

/* ============================== Philox4x32-10 ============================================ */

void o_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4])
{
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
    uint32_t k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* ============================== samplers ================================================== */

#define O_STREAM_REJECTION 0x52454A43u  /* "REJC": keeps the rejection stream disjoint from DIRECT blocks */

void o_rng_init(o_rng* g, uint64_t seed, uint32_t pixel, uint32_t sample, int32_t mode)
{
    g->key[0] = (uint32_t)seed; g->key[1] = (uint32_t)(seed >> 32);
    g->pixel = pixel; g->sample = sample; g->draw = 0; g->mode = mode;
}

double o_rng_f64(o_rng* g)
{
    uint32_t ctr[4] = { g->pixel, g->sample, g->draw >> 1, O_STREAM_REJECTION }, out[4];
    o_philox4x32_10(ctr, g->key, out);
    uint32_t lo = out[2 * (g->draw & 1u)], hi = out[2 * (g->draw & 1u) + 1];
    g->draw++;
    uint64_t bits = ((uint64_t)hi << 32) | lo;
    return (double)(bits >> 11) * (1.0 / 9007199254740992.0);   /* 2^-53, rand 0.8 Standard for f64 */
}

double o_rng_range(o_rng* g, double lo, double hi) { return lo + (hi - lo) * o_rng_f64(g); }

o_vec3 o_random_in_unit_sphere(o_rng* g)                                             /* vec3.rs:37-45 */
{
    for (;;) {
        /* Vec3::random_in_range(-1,1): x, y, z drawn in that order (vec3.rs:26-35) */
        double x = o_rng_range(g, -1.0, 1.0);
        double y = o_rng_range(g, -1.0, 1.0);
        double z = o_rng_range(g, -1.0, 1.0);
        o_vec3 p = o_v(x, y, z);
        if (o_length_squared(p) < 1.0) return p;
    }
}

o_vec3 o_random_unit_vector(o_rng* g) { return o_unit_vector(o_random_in_unit_sphere(g)); } /* vec3.rs:47-49 */

o_vec3 o_random_in_unit_disk(o_rng* g)                                               /* vec3.rs:59-68 */
{
    for (;;) {
        double x = o_rng_range(g, -1.0, 1.0);
        double y = o_rng_range(g, -1.0, 1.0);
        o_vec3 p = o_v(x, y, 0.0);
        if (o_length_squared(p) < 1.0) return p;
    }
}

void o_direct_uniforms(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t bounce, double u[4])
{
    uint32_t key[2] = { (uint32_t)seed, (uint32_t)(seed >> 32) };
    uint32_t ctr[4] = { pixel, sample, bounce, 0u }, out[4];
    o_philox4x32_10(ctr, key, out);
    for (int i = 0; i < 4; ++i) u[i] = (double)(out[i] >> 8) * (1.0 / 16777216.0);
}

#define O_TWO_PI 6.28318530717958647692528676655900577

void o_direct_disk(double u2, double u3, double* x, double* y)
{
    double r = sqrt(u2), phi = O_TWO_PI * u3;     /* uniform on the unit disk (area measure) */
    *x = r * cos(phi); *y = r * sin(phi);
}

o_vec3 o_direct_unit_vector(double u0, double u1)
{
    double z = 1.0 - 2.0 * u0;                      /* Archimedes: z uniform on [-1,1] */
    double rxy = sqrt(fmax(0.0, 1.0 - z * z)), phi = O_TWO_PI * u1;
    return o_v(rxy * cos(phi), rxy * sin(phi), z);
}

o_vec3 o_direct_in_unit_sphere(double u0, double u1, double u2)
{
    return o_mul_s(o_direct_unit_vector(u0, u1), cbrt(u2));   /* radius cdf r^3 */
}

/* ============================== main.rs: ray_color ========================================= */

o_vec3 o_ray_color(const o_ray* r, const o_world* w, int32_t depth, double t_min, o_rng* g,
                   uint32_t bounce, o_counters* cnt)                                  /* main.rs:38-57 */
{
    if (depth <= 0) return o_v(0, 0, 0);

    o_hit_record rec;
    if (cnt) { cnt->rays++; cnt->sphere_tests += (uint64_t)w->n_spheres; }
    if (o_world_hit(w, r, t_min, INFINITY, &rec, NULL)) {                             /* main.rs:44 */
        const o_material* m = &w->materials[rec.mat];
        o_vec3 sample = o_v(0, 0, 0);
        if (g->mode == O_SAMPLER_DIRECT) {
            double u[4];
            uint64_t seed = ((uint64_t)g->key[1] << 32) | g->key[0];
            o_direct_uniforms(seed, g->pixel, g->sample, bounce + 1u, u);
            if (m->kind == O_MAT_LAMBERTIAN) sample = o_direct_unit_vector(u[0], u[1]);
            else if (m->kind == O_MAT_METAL) sample = o_direct_in_unit_sphere(u[0], u[1], u[2]);
            else sample = o_v(u[0], 0, 0);
        } else {
            if (m->kind == O_MAT_LAMBERTIAN || m->kind == O_MAT_METAL) {
                sample = o_random_in_unit_sphere(g);                                  /* materials.rs:23,53 */
            } else {
                /* draw xi only if can_refract (materials.rs:96); recompute the predicate as scatter does */
                double ratio = rec.front_face ? 1.0 / m->param : m->param;
                o_vec3 ud = o_unit_vector(r->dir);
                double cos_theta = fmin(1.0, -o_dot(ud, rec.normal));
                double sin_theta = sqrt(1.0 - cos_theta * cos_theta);
                if (ratio * sin_theta <= 1.0) sample.x = o_rng_f64(g);
            }
        }
        o_vec3 att; o_ray scat;
        if (o_scatter(m, r, &rec, sample, &att, &scat)) {
            return o_mul_v(att, o_ray_color(&scat, w, depth - 1, t_min, g, bounce + 1u, cnt)); /* main.rs:49 */
        }
        return o_v(0, 0, 0);                                                          /* main.rs:51 */
    }
    o_vec3 unit_direction = o_unit_vector(r->dir);                                    /* main.rs:54-56 */
    double t = 0.5 * (unit_direction.y + 1.0);
    return o_add(o_mul_s(o_v(1, 1, 1), 1.0 - t), o_mul_s(o_v(0.5, 0.7, 1.0), t));
}

o_vec3 o_path_radiance(const o_world* w, const o_camera* cam, const o_render_params* p,
                       uint32_t i, uint32_t j, uint32_t s, o_counters* cnt)            /* main.rs:131-135 */
{
    o_rng g;
    o_rng_init(&g, p->seed, j * p->width + i, s, p->sampler);
    double ju, jv, dx, dy;
    if (p->sampler == O_SAMPLER_DIRECT) {
        double u[4];
        o_direct_uniforms(p->seed, g.pixel, g.sample, 0u, u);
        ju = u[0]; jv = u[1];
        o_direct_disk(u[2], u[3], &dx, &dy);
    } else {
        ju = o_rng_f64(&g);                                                           /* main.rs:131 */
        jv = o_rng_f64(&g);                                                           /* main.rs:132 */
        o_vec3 d = o_random_in_unit_disk(&g);                                         /* camera.rs:48 */
        dx = d.x; dy = d.y;
    }
    double u = ((double)i + ju) / (double)(p->width - 1);
    double v = ((double)j + jv) / (double)(p->height - 1);
    o_ray r = o_camera_get_ray(cam, u, v, dx, dy);                                    /* main.rs:134 */
    return o_ray_color(&r, w, p->max_depth, p->t_min, &g, 0u, cnt);                   /* main.rs:135 */
}

int o_render(const o_world* w, const o_camera* cam, const o_render_params* p, uint8_t* out_rgba,
             double* accum, o_counters* cnt)                                           /* main.rs:122-145 */
{
    if (!w || !cam || !p || !out_rgba || p->width < 2 || p->height < 2 || p->spp == 0) return -1;
    uint32_t rb = p->row_begin, re = p->row_end;
    if (rb == 0 && re == 0) re = p->height;
    if (re > p->height || rb > re) return -1;
    uint64_t rays = 0, tests = 0;
#ifdef _OPENMP
    int nt = p->n_threads > 0 ? p->n_threads : omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 1) num_threads(nt) reduction(+ : rays, tests)
#endif
    for (int64_t y = (int64_t)rb; y < (int64_t)re; ++y) {           /* one task per row (main.rs:122-123) */
        uint32_t j = p->height - 1u - (uint32_t)y;                  /* j=0 is the bottom row; flip = main.rs:141-145 */
        o_counters c = { 0, 0 };
        for (uint32_t i = 0; i < p->width; ++i) {                   /* main.rs:125 */
            o_vec3 pixel_color = o_v(0, 0, 0);                      /* main.rs:127 */
            for (uint32_t s = 0; s < p->spp; ++s)                   /* main.rs:130 */
                pixel_color = o_add(pixel_color, o_path_radiance(w, cam, p, i, j, s, &c));
            size_t px = (size_t)y * p->width + i;
            o_to_rgba(pixel_color, p->alpha, p->spp, out_rgba + 4 * px);              /* main.rs:137 */
            if (accum) { accum[3 * px] = pixel_color.x; accum[3 * px + 1] = pixel_color.y; accum[3 * px + 2] = pixel_color.z; }
        }
        rays += c.rays; tests += c.sphere_tests;
    }
    if (cnt) { cnt->rays = rays; cnt->sphere_tests = tests; }
    return 0;
}

/* ============================== knife-edge margins ========================================= */
/* See rtiow_oracle.h (o_render_margins) for what the margins measure and why.  Nothing below feeds back into the path: the
 * radiance is computed by the same calls, in the same order, as o_ray_color's. */

/* error growth at distance L along a ray whose origin was left by a bounce of kind k (O_MARGIN_K_*) on a sphere of radius r */
static double o_grow(double g, double k_over_r, double L) { return g * (1.0 + k_over_r * fmax(L, 0.0)); }

static int o_same_sphere(const o_sphere* a, const o_sphere* b)
{
    return a->center.x == b->center.x && a->center.y == b->center.y && a->center.z == b->center.z && a->radius == b->radius;
}

/* the hit scan's margin of one ray (o_world_hit with t_win the winner's root, INFINITY on a miss): grazing spheres in
 * [t_min, t_win], roots near t_min and the gap between the two smallest accepted roots, each divided by the growth at the
 * sphere's distance.  `self`: the sphere the ray starts on, whose near-zero root is no decision (and whose far root the
 * renderer computes without a discriminant); a coincident twin of it has the same roots in f64. */
static double o_hit_margin(const o_world* w, const o_ray* r, double t_min, double t_win, int32_t self, double g, double k_over_r)
{
    const double a = o_length_squared(r->dir), dl = sqrt(a), lo = o_length(r->orig);
    double m = INFINITY, t1 = INFINITY, t2 = INFINITY, len1 = 0.0, len2 = 0.0;
    int32_t i1 = -1;
    for (int32_t i = 0; i < w->n_spheres; ++i) {
        const o_sphere* s = &w->spheres[i];
        const int is_self = self >= 0 && o_same_sphere(s, &w->spheres[self]);     /* the sphere, or a coincident twin */
        const o_vec3 oc = o_sub(r->orig, s->center);
        const double hb = o_dot(oc, r->dir), ar = fabs(s->radius);
        const double disc = hb * hb - a * (o_length_squared(oc) - s->radius * s->radius);
        const double len = lo + o_length(oc) + ar;              /* the lengths the sphere's roots are computed from */
        const double tca = -hb / a;
        if (disc < 0.0) {                                        /* a near miss in front of the winner */
            if (!is_self && tca >= t_min && tca <= t_win)
                m = fmin(m, (-disc / a) / (ar * len) / o_grow(g, k_over_r, tca * dl));
            continue;
        }
        const double sq = sqrt(disc), t0 = (-hb - sq) / a, tf = (-hb + sq) / a;
        const double tacc = t0 >= t_min ? t0 : tf >= t_min ? tf : tca;
        const double gi = o_grow(g, k_over_r, tacc * dl);
        if (!is_self && ((t0 >= t_min && t0 <= t_win) || (tf >= t_min && tf <= t_win)))
            m = fmin(m, (disc / a) / (ar * len) / gi);           /* grazing */
        for (int k = 0; k < 2; ++k) {                            /* roots near t_min */
            const double t = k ? tf : t0;
            if (is_self && fabs(t) <= fabs(k ? t0 : tf)) continue;
            m = fmin(m, fabs(t - t_min) * dl / len / gi);
        }
        if (t0 >= t_min || tf >= t_min) {                        /* the two smallest accepted roots; a coincident twin ties exactly */
            if (i1 >= 0 && o_same_sphere(s, &w->spheres[i1])) {
                if (tacc <= t1) { t1 = tacc; i1 = i; }
            } else if (tacc < t1) {
                t2 = t1; len2 = len1; t1 = tacc; len1 = len; i1 = i;
            } else if (tacc < t2) {
                t2 = tacc; len2 = len;
            }
        }
    }
    if (isfinite(t2)) m = fmin(m, (t2 - t1) * dl / fmax(len1, len2) / o_grow(g, k_over_r, t1 * dl));
    return m;
}

/* o_ray_color in DIRECT mode, plus the smallest margin of every ray of the path in *margin.  self: the sphere the ray
 * starts on (-1 for a camera ray); g, k_over_r: the error growth of the ray's origin and of its direction per unit length */
static o_vec3 o_ray_color_m(const o_ray* r, const o_world* w, int32_t depth, double t_min, o_rng* g, uint32_t bounce,
                            o_counters* cnt, int32_t self, double gr, double k_over_r, double* margin)
{
    if (depth <= 0) return o_v(0, 0, 0);

    o_hit_record rec;
    int32_t idx = -1;
    if (cnt) { cnt->rays++; cnt->sphere_tests += (uint64_t)w->n_spheres; }
    if (o_world_hit(w, r, t_min, INFINITY, &rec, &idx)) {
        const o_material* m = &w->materials[rec.mat];
        const double dl = o_length(r->dir);
        *margin = fmin(*margin, o_hit_margin(w, r, t_min, rec.t, self, gr, k_over_r));
        const double gh = o_grow(gr, k_over_r, rec.t * dl);          /* growth at the hit point */
        o_vec3 sample = o_v(0, 0, 0);
        double u[4];
        uint64_t seed = ((uint64_t)g->key[1] << 32) | g->key[0];
        o_direct_uniforms(seed, g->pixel, g->sample, bounce + 1u, u);
        if (m->kind == O_MAT_LAMBERTIAN) sample = o_direct_unit_vector(u[0], u[1]);
        else if (m->kind == O_MAT_METAL) sample = o_direct_in_unit_sphere(u[0], u[1], u[2]);
        else sample = o_v(u[0], 0, 0);
        o_vec3 att; o_ray scat;
        const int some = o_scatter(m, r, &rec, sample, &att, &scat);
        /* the scatter's own decision, and the growth of the direction error it passes on */
        const double ar = fabs(w->spheres[idx].radius);
        double k_next = O_MARGIN_K_SPECULAR, amp = 1.0;
        if (m->kind == O_MAT_LAMBERTIAN) {
            *margin = fmin(*margin, o_length(o_add(rec.normal, o_unit_vector(sample))) / gh);     /* the near-zero fallback */
            k_next = O_MARGIN_K_LAMBERTIAN;
        } else if (m->kind == O_MAT_METAL) {
            const double sl = o_length(scat.dir);
            *margin = fmin(*margin, (sl > 0.0 ? fabs(o_dot(scat.dir, rec.normal)) / sl : 0.0) / gh);   /* absorption */
        } else {
            const double ratio = rec.front_face ? 1.0 / m->param : m->param;
            const o_vec3 ud = o_unit_vector(r->dir);
            const double cos_theta = fmin(1.0, -o_dot(ud, rec.normal));
            const double sin_theta = sqrt(1.0 - cos_theta * cos_theta);
            *margin = fmin(*margin, fabs(ratio * sin_theta - 1.0) / gh);                                    /* TIR */
            if (ratio * sin_theta <= 1.0) {
                *margin = fmin(*margin, fabs(o_reflectance(cos_theta, ratio) - sample.x) / gh);             /* Schlick */
                if (o_reflectance(cos_theta, ratio) <= sample.x) {    /* refracted: Snell's law amplifies the angle's error */
                    const double cos_out = sqrt(fmax(1.0 - ratio * ratio * sin_theta * sin_theta, 1e-300));
                    amp = fmax(1.0, ratio * cos_theta / cos_out);
                }
            }
        }
        if (some) {
            return o_mul_v(att, o_ray_color_m(&scat, w, depth - 1, t_min, g, bounce + 1u, cnt, idx, gh * amp,
                                              k_next / ar, margin));
        }
        return o_v(0, 0, 0);
    }
    *margin = fmin(*margin, o_hit_margin(w, r, t_min, INFINITY, self, gr, k_over_r));
    o_vec3 unit_direction = o_unit_vector(r->dir);
    double t = 0.5 * (unit_direction.y + 1.0);
    return o_add(o_mul_s(o_v(1, 1, 1), 1.0 - t), o_mul_s(o_v(0.5, 0.7, 1.0), t));
}

int o_render_margins(const o_world* w, const o_camera* cam, const o_render_params* p, uint8_t* out_rgba, double* accum,
                     double* margin, o_counters* cnt)
{
    if (!w || !cam || !p || !out_rgba || !margin || p->width < 2 || p->height < 2 || p->spp == 0 || p->sampler != O_SAMPLER_DIRECT)
        return -1;
    uint32_t rb = p->row_begin, re = p->row_end;
    if (rb == 0 && re == 0) re = p->height;
    if (re > p->height || rb > re) return -1;
    uint64_t rays = 0, tests = 0;
#ifdef _OPENMP
    int nt = p->n_threads > 0 ? p->n_threads : omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 1) num_threads(nt) reduction(+ : rays, tests)
#endif
    for (int64_t y = (int64_t)rb; y < (int64_t)re; ++y) {
        uint32_t j = p->height - 1u - (uint32_t)y;
        o_counters c = { 0, 0 };
        for (uint32_t i = 0; i < p->width; ++i) {
            o_vec3 pixel_color = o_v(0, 0, 0);
            double mg = INFINITY;
            for (uint32_t s = 0; s < p->spp; ++s) {
                /* o_path_radiance with the DIRECT sampler */
                o_rng g;
                o_rng_init(&g, p->seed, j * p->width + i, s, p->sampler);
                double u4[4], dx, dy;
                o_direct_uniforms(p->seed, g.pixel, g.sample, 0u, u4);
                o_direct_disk(u4[2], u4[3], &dx, &dy);
                double u = ((double)i + u4[0]) / (double)(p->width - 1);
                double v = ((double)j + u4[1]) / (double)(p->height - 1);
                o_ray r = o_camera_get_ray(cam, u, v, dx, dy);
                pixel_color = o_add(pixel_color, o_ray_color_m(&r, w, p->max_depth, p->t_min, &g, 0u, &c, -1, 1.0, 0.0, &mg));
            }
            size_t px = (size_t)y * p->width + i;
            o_to_rgba(pixel_color, p->alpha, p->spp, out_rgba + 4 * px);
            if (accum) { accum[3 * px] = pixel_color.x; accum[3 * px + 1] = pixel_color.y; accum[3 * px + 2] = pixel_color.z; }
            margin[px] = mg;
        }
        rays += c.rays; tests += c.sphere_tests;
    }
    if (cnt) { cnt->rays = rays; cnt->sphere_tests = tests; }
    return 0;
}

/* ============================== batch helpers ============================================= */

static o_vec3 ld3(const double* a, int64_t i) { return o_v(a[3 * i], a[3 * i + 1], a[3 * i + 2]); }
static void st3(double* a, int64_t i, o_vec3 v) { a[3 * i] = v.x; a[3 * i + 1] = v.y; a[3 * i + 2] = v.z; }

void o_sphere_hit_batch(int64_t n, const double* center, const double* radius, const double* orig,
                        const double* dir, const double* t_min, const double* t_max,
                        int32_t* hit, double* t, double* p, double* normal, int32_t* front_face)
{
    for (int64_t i = 0; i < n; ++i) {
        o_sphere s = { ld3(center, i), radius[i], 0 };
        o_ray r = { ld3(orig, i), ld3(dir, i) };
        o_hit_record rec; memset(&rec, 0, sizeof rec);
        hit[i] = o_sphere_hit(&s, &r, t_min[i], t_max[i], &rec);
        t[i] = rec.t; st3(p, i, rec.p); st3(normal, i, rec.normal); front_face[i] = rec.front_face;
    }
}

void o_world_hit_batch(const o_world* w, int64_t n, const double* orig, const double* dir, double t_min,
                       double t_max, int32_t* hit, int32_t* index, double* t, double* p, double* normal,
                       int32_t* front_face)
{
#ifdef _OPENMP
#pragma omp parallel for schedule(static)
#endif
    for (int64_t i = 0; i < n; ++i) {
        o_ray r = { ld3(orig, i), ld3(dir, i) };
        o_hit_record rec; memset(&rec, 0, sizeof rec);
        int32_t idx = -1;
        hit[i] = o_world_hit(w, &r, t_min, t_max, &rec, &idx);
        index[i] = idx; t[i] = rec.t; st3(p, i, rec.p); st3(normal, i, rec.normal); front_face[i] = rec.front_face;
    }
}

void o_scatter_batch(int64_t n, const int32_t* kind, const double* albedo, const double* param,
                     const double* r_orig, const double* r_dir, const double* p, const double* normal,
                     const int32_t* front_face, const double* sample, int32_t* some,
                     double* attenuation, double* s_orig, double* s_dir)
{
    for (int64_t i = 0; i < n; ++i) {
        o_material m = { kind[i], ld3(albedo, i), param[i] };
        o_ray r = { ld3(r_orig, i), ld3(r_dir, i) };
        o_hit_record rec; memset(&rec, 0, sizeof rec);
        rec.p = ld3(p, i); rec.normal = ld3(normal, i); rec.front_face = front_face[i];
        o_vec3 att = o_v(0, 0, 0); o_ray sc = { o_v(0, 0, 0), o_v(0, 0, 0) };
        some[i] = o_scatter(&m, &r, &rec, ld3(sample, i), &att, &sc);
        st3(attenuation, i, att); st3(s_orig, i, sc.orig); st3(s_dir, i, sc.dir);
    }
}

void o_get_ray_batch(const o_camera* cam, int64_t n, const double* s, const double* t,
                     const double* disk_xy, double* orig, double* dir)
{
    for (int64_t i = 0; i < n; ++i) {
        o_ray r = o_camera_get_ray(cam, s[i], t[i], disk_xy[2 * i], disk_xy[2 * i + 1]);
        st3(orig, i, r.orig); st3(dir, i, r.dir);
    }
}

void o_to_rgba_batch(int64_t n, const double* color, uint8_t alpha, uint64_t spp, uint8_t* out)
{
    for (int64_t i = 0; i < n; ++i) o_to_rgba(ld3(color, i), alpha, spp, out + 4 * i);
}

void o_reflect_batch(int64_t n, const double* v, const double* nrm, double* out)
{
    for (int64_t i = 0; i < n; ++i) st3(out, i, o_reflect(ld3(v, i), ld3(nrm, i)));
}

void o_refract_batch(int64_t n, const double* uv, const double* nrm, const double* eta, double* out)
{
    for (int64_t i = 0; i < n; ++i) st3(out, i, o_refract(ld3(uv, i), ld3(nrm, i), eta[i]));
}

void o_ray_color_batch(const o_world* w, int64_t n, const double* orig, const double* dir,
                       const uint32_t* pixel, const uint32_t* sample, uint64_t seed, int32_t max_depth,
                       double t_min, double* color, uint64_t* rays)
{
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 64)
#endif
    for (int64_t i = 0; i < n; ++i) {
        o_ray r = { ld3(orig, i), ld3(dir, i) };
        o_rng g; o_rng_init(&g, seed, pixel[i], sample[i], O_SAMPLER_DIRECT);
        o_counters c = { 0, 0 };
        st3(color, i, o_ray_color(&r, w, max_depth, t_min, &g, 0u, &c));
        if (rays) rays[i] = c.rays;
    }
}

void o_rejection_samples(uint64_t seed, int64_t n, int32_t which, double* out)
{
    for (int64_t i = 0; i < n; ++i) {
        o_rng g; o_rng_init(&g, seed, (uint32_t)i, 0u, O_SAMPLER_REJECTION);
        o_vec3 v = which == 0 ? o_random_in_unit_disk(&g) : which == 1 ? o_random_in_unit_sphere(&g) : o_random_unit_vector(&g);
        st3(out, i, v);
    }
}
