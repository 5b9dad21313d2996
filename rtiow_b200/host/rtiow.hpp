// rtiow.hpp — C++ host mirror of the reference's caller-facing API (SURVEY Appendix A) over the C ABI.
//
// The reference is a Rust crate and its host code should stay Rust (rust/ in this repo holds that
// crate's sources); this image has no rustc, so the host side that is actually compiled and tested
// here is this header: same module/type/function names, argument meaning and error behaviour as
// /root/reference/src/{vec3,ray,camera,materials,shapes/mod,shapes/sphere}.rs, plus ONE new call,
// rtiow::render(), that replaces main.rs:122-145 with librtiow_cuda.so.
//
// Hit::hit / Scatter::scatter / Camera::get_ray keep working on the host so a caller's own
// ray_color still compiles (Appendix A), but render() never calls them: shapes and materials
// reach the GPU through the defaulted describe() methods, and anything that does not describe
// itself is RenderError::Unsupported — there is no CPU fallback.
#pragma once
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <limits>
#include <functional>
#include <memory>
#include <optional>
#include <ostream>
#include <random>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "rtiow_cuda.h"

namespace rtiow {

// thread_rng stand-in for the host-side samplers (vec3.rs:22,27,61; materials.rs:95): thread-local, OS-seeded
inline std::mt19937_64& thread_rng()
{
    thread_local std::mt19937_64 g{ std::random_device{}() };
    return g;
}
inline double gen_f64() { return std::generate_canonical<double, 53>(thread_rng()); }                 // rng.gen::<f64>()
inline double gen_range(double lo, double hi) { return lo + (hi - lo) * gen_f64(); }                   // gen_range(lo..hi)

// ------------------------------------------------------------------------------------------------ vec3.rs
class Vec3 {                                                                                           // vec3.rs:4-9
    double x_, y_, z_;
public:
    static Vec3 zero() { return Vec3(0.0, 0.0, 0.0); }                                                 // vec3.rs:13
    template <typename T1, typename T2, typename T3> Vec3(T1 x, T2 y, T3 z) : x_(double(x)), y_(double(y)), z_(double(z)) {}   // vec3.rs:17 (Into<f64>)
    Vec3() : x_(0), y_(0), z_(0) {}
    static Vec3 random() { double a = gen_f64(), b = gen_f64(), c = gen_f64(); return Vec3(a, b, c); }  // vec3.rs:21
    template <typename T1, typename T2> static Vec3 random_in_range(T1 mn, T2 mx)                      // vec3.rs:26
    {
        double a = gen_range(double(mn), double(mx)), b = gen_range(double(mn), double(mx)), c = gen_range(double(mn), double(mx));
        return Vec3(a, b, c);
    }
    static Vec3 random_in_unit_sphere() { for (;;) { Vec3 p = random_in_range(-1, 1); if (p.length_squared() < 1.0) return p; } }   // vec3.rs:37
    static Vec3 random_unit_vector() { return random_in_unit_sphere().unit_vector(); }                 // vec3.rs:47
    static Vec3 random_in_hemisphere(const Vec3& normal)                                               // vec3.rs:51
    {
        Vec3 s = random_in_unit_sphere();
        return s.dot(normal) > 0.0 ? s : Vec3::zero() - s;
    }
    static Vec3 random_in_unit_disk() { for (;;) { Vec3 p(gen_range(-1.0, 1.0), gen_range(-1.0, 1.0), 0); if (p.length_squared() < 1.0) return p; } }   // vec3.rs:59
    double x() const { return x_; }
    double y() const { return y_; }
    double z() const { return z_; }
    double length() const { return std::sqrt(length_squared()); }                                      // vec3.rs:83
    double length_squared() const { return x_ * x_ + y_ * y_ + z_ * z_; }                              // vec3.rs:87
    Vec3 norm() const { return *this / length(); }                                                     // vec3.rs:91
    double dot(const Vec3& r) const { return x_ * r.x_ + y_ * r.y_ + z_ * r.z_; }                      // vec3.rs:95
    Vec3 cross(const Vec3& r) const { return Vec3(y_ * r.z_ - z_ * r.y_, z_ * r.x_ - x_ * r.z_, x_ * r.y_ - y_ * r.x_); }   // vec3.rs:99
    Vec3 unit_vector() const { return *this / length(); }                                              // vec3.rs:107
    bool is_near_zero() const { const double s = 1e-8; return std::fabs(x_) < s && std::fabs(y_) < s && std::fabs(z_) < s; }   // vec3.rs:111
    Vec3 reflect(const Vec3& n) const { return *this - (2.0 * dot(n)) * n; }                            // vec3.rs:116
    Vec3 refract(Vec3 n, double etai_over_etat) const                                                  // vec3.rs:120
    {
        double cos_theta = std::fmin(1.0, -dot(n));
        Vec3 perp = etai_over_etat * (*this + n * cos_theta);
        Vec3 par = -std::sqrt(std::fabs(1.0 - perp.length_squared())) * n;
        return perp + par;
    }
    // operators (vec3.rs:137-397); no unary minus, as in the reference
    friend Vec3 operator+(const Vec3& a, const Vec3& b) { return Vec3(a.x_ + b.x_, a.y_ + b.y_, a.z_ + b.z_); }
    friend Vec3 operator+(const Vec3& a, double s) { return Vec3(a.x_ + s, a.y_ + s, a.z_ + s); }
    friend Vec3 operator+(double s, const Vec3& a) { return a + s; }
    friend Vec3 operator-(const Vec3& a, const Vec3& b) { return Vec3(a.x_ - b.x_, a.y_ - b.y_, a.z_ - b.z_); }
    friend Vec3 operator-(const Vec3& a, double s) { return Vec3(a.x_ - s, a.y_ - s, a.z_ - s); }
    friend Vec3 operator-(double s, const Vec3& a) { return Vec3(s - a.x_, s - a.y_, s - a.z_); }
    friend Vec3 operator*(const Vec3& a, double s) { return Vec3(a.x_ * s, a.y_ * s, a.z_ * s); }
    friend Vec3 operator*(double s, const Vec3& a) { return a * s; }
    friend Vec3 operator*(const Vec3& a, const Vec3& b) { return Vec3(a.x_ * b.x_, a.y_ * b.y_, a.z_ * b.z_); }
    friend Vec3 operator/(const Vec3& a, double s) { return a * (1.0 / s); }                            // vec3.rs:371-376
    friend bool operator==(const Vec3& a, const Vec3& b) { return a.x_ == b.x_ && a.y_ == b.y_ && a.z_ == b.z_; }
    friend std::ostream& operator<<(std::ostream& o, const Vec3& v) { return o << "Vec3 (" << v.x_ << ", " << v.y_ << ", " << v.z_ << ")"; }   // vec3.rs:128-132
    // Color::to_rgba (vec3.rs:404-420)
    std::array<uint8_t, 4> to_rgba(uint8_t alpha, uint64_t samples_per_pixel) const
    {
        auto q = [&](double c) -> uint8_t {
            c = std::sqrt((1.0 / double(samples_per_pixel)) * c);
            if (std::isnan(c)) return 0;
            c = c < 0.0 ? 0.0 : (c > 0.999 ? 0.999 : c);
            return uint8_t(256.0 * c);
        };
        return { q(x_), q(y_), q(z_), alpha };
    }
};
using Point3 = Vec3;                                                                                   // vec3.rs:400
using Color = Vec3;                                                                                    // vec3.rs:401

// ------------------------------------------------------------------------------------------------ ray.rs
class Ray {                                                                                            // ray.rs:5-8
    Point3 orig; Vec3 dir;
public:
    Ray(Point3 o, Vec3 d) : orig(o), dir(d) {}
    Point3 at(double t) const { return orig + (t * dir); }                                             // ray.rs:15
    Vec3 direction() const { return dir; }
    Point3 origin() const { return orig; }
    friend std::ostream& operator<<(std::ostream& o, const Ray& r) { return o << "orig: " << r.orig << ", dir: " << r.dir; }   // ray.rs:29-33
};

// ------------------------------------------------------------------------------------------------ materials.rs / shapes
struct MaterialDesc { rtiow_material_kind kind; double albedo[3]; double param; };
struct SphereDesc { double center[3]; double radius; };
class Scatter;

class HitRecord {                                                                                      // shapes/mod.rs:10-16
    Point3 p; Vec3 normal; std::shared_ptr<const Scatter> mat; double t;
    friend class Sphere; friend class HittableList;
    HitRecord(Point3 p_, double t_, const Ray& r, const Vec3& outward, std::shared_ptr<const Scatter> m)   // mod.rs:20-30
        : p(p_), normal(outward), mat(std::move(m)), t(t_), front_face(r.direction().dot(outward) < 0.0)
    {
        if (!front_face) normal = Vec3::zero() - outward;
    }
public:
    bool front_face;
    Vec3 get_normal() const { return normal; }
    Point3 get_p() const { return p; }
    std::shared_ptr<const Scatter> get_mat() const { return mat; }                                     // Arc::clone, mod.rs:40-42
};

class Scatter {                                                                                        // materials.rs:5-7
public:
    virtual ~Scatter() = default;
    virtual std::optional<std::pair<Color, Ray>> scatter(const Ray& r_in, const HitRecord& rec) const = 0;
    // provided method (INTEGRATION.md): how a material reaches the GPU.  nullopt => render() reports Unsupported.
    virtual std::optional<MaterialDesc> describe() const { return std::nullopt; }
};

class Lambertian : public Scatter {                                                                    // materials.rs:9-31
    Color albedo;
public:
    explicit Lambertian(Color a) : albedo(a) {}
    std::optional<std::pair<Color, Ray>> scatter(const Ray&, const HitRecord& rec) const override
    {
        Vec3 d = rec.get_normal() + Vec3::random_unit_vector();
        if (d.is_near_zero()) d = rec.get_normal();
        return std::make_pair(albedo, Ray(rec.get_p(), d));
    }
    std::optional<MaterialDesc> describe() const override { return MaterialDesc{ RTIOW_MAT_LAMBERTIAN, { albedo.x(), albedo.y(), albedo.z() }, 0.0 }; }
};

class Metal : public Scatter {                                                                         // materials.rs:34-62
    Color albedo; double fuzz;
public:
    Metal(Color a, double f) : albedo(a), fuzz(f) {}
    std::optional<std::pair<Color, Ray>> scatter(const Ray& r_in, const HitRecord& rec) const override
    {
        Vec3 reflected = r_in.direction().reflect(rec.get_normal()).unit_vector();
        Ray scattered(rec.get_p(), reflected + fuzz * Vec3::random_in_unit_sphere());
        if (scattered.direction().dot(rec.get_normal()) <= 0.0) return std::nullopt;
        return std::make_pair(albedo, scattered);
    }
    std::optional<MaterialDesc> describe() const override { return MaterialDesc{ RTIOW_MAT_METAL, { albedo.x(), albedo.y(), albedo.z() }, fuzz }; }
};

class Dialectric : public Scatter {                                                                    // materials.rs:64-104 (sic)
    double ir;
    static double reflectence(double cosine, double ref_idx)                                           // materials.rs:78-82 (sic)
    {
        double r0 = (1.0 - ref_idx) / (1.0 + ref_idx); r0 = r0 * r0;
        return r0 + (1.0 - r0) * std::pow(1.0 - cosine, 5);
    }
public:
    explicit Dialectric(double index_of_refraction) : ir(index_of_refraction) {}
    std::optional<std::pair<Color, Ray>> scatter(const Ray& r_in, const HitRecord& rec) const override
    {
        double ratio = rec.front_face ? 1.0 / ir : ir;
        Vec3 ud = r_in.direction().unit_vector();
        double cos_theta = std::fmin(1.0, -ud.dot(rec.get_normal()));
        double sin_theta = std::sqrt(1.0 - cos_theta * cos_theta);
        bool can_refract = ratio * sin_theta <= 1.0;
        Vec3 d = (can_refract && reflectence(cos_theta, ratio) <= gen_f64()) ? ud.refract(rec.get_normal(), ratio) : ud.reflect(rec.get_normal());
        return std::make_pair(Color(1, 1, 1), Ray(rec.get_p(), d));
    }
    std::optional<MaterialDesc> describe() const override { return MaterialDesc{ RTIOW_MAT_DIELECTRIC, { 1, 1, 1 }, ir }; }
};
using Dielectric = Dialectric;     // correctly spelt alias, added — the reference's name stays

class Hit {                                                                                            // shapes/mod.rs:48-50
public:
    virtual ~Hit() = default;
    virtual std::optional<HitRecord> hit(const Ray& r, double t_min, double t_max) const = 0;
    struct Described { SphereDesc sphere; std::shared_ptr<const Scatter> mat; };
    virtual std::optional<Described> describe() const { return std::nullopt; }
};

class Sphere : public Hit {                                                                            // shapes/sphere.rs:9-13
    Point3 center; double radius; std::shared_ptr<const Scatter> mat;
public:
    template <typename T> Sphere(Point3 cen, T r, std::shared_ptr<const Scatter> m) : center(cen), radius(double(r)), mat(std::move(m)) {}   // sphere.rs:45-51
    std::optional<HitRecord> hit(const Ray& r, double t_min, double t_max) const override              // sphere.rs:16-41
    {
        Vec3 oc = r.origin() - center;
        double a = r.direction().length_squared(), half_b = oc.dot(r.direction()), c = oc.length_squared() - radius * radius;
        double disc = half_b * half_b - a * c;
        if (disc < 0.0) return std::nullopt;
        double sqrtd = std::sqrt(disc), root = (-half_b - sqrtd) / a;
        if (root < t_min || t_max < root) {
            root = (-half_b + sqrtd) / a;
            if (root < t_min || t_max < root) return std::nullopt;
        }
        Point3 p = r.at(root);
        return HitRecord(p, root, r, (p - center) / radius, mat);
    }
    std::optional<Described> describe() const override { return Described{ SphereDesc{ { center.x(), center.y(), center.z() }, radius }, mat }; }
};

class HittableList : public Hit {                                                                      // shapes/mod.rs:52: Vec<Box<dyn Hit>>
    std::vector<std::unique_ptr<Hit>> items;
public:
    HittableList() = default;                                                                          // HittableList::new()
    void push(std::unique_ptr<Hit> h) { items.push_back(std::move(h)); }                               // world.push(Box::new(..))
    size_t len() const { return items.size(); }
    const std::vector<std::unique_ptr<Hit>>& iter() const { return items; }
    std::optional<HitRecord> hit(const Ray& r, double t_min, double t_max) const override              // mod.rs:56-69
    {
        std::optional<HitRecord> closest; double closest_so_far = t_max;
        for (const auto& o : items)
            if (auto rec = o->hit(r, t_min, closest_so_far)) { closest_so_far = rec->t; closest = std::move(rec); }
        return closest;
    }
};

// ------------------------------------------------------------------------------------------------ camera.rs
class Camera {                                                                                         // camera.rs:4-13
    rtiow_camera c{};
    static Vec3 v(const double a[3]) { return Vec3(a[0], a[1], a[2]); }
public:
    Camera(Point3 look_from, Point3 look_at, Vec3 v_up, double v_fov, double aspect_ratio, double aperture, double focus_dist)   // camera.rs:17-45
    {
        const double f[3] = { look_from.x(), look_from.y(), look_from.z() }, a[3] = { look_at.x(), look_at.y(), look_at.z() }, u[3] = { v_up.x(), v_up.y(), v_up.z() };
        rtiow_camera_new(f, a, u, v_fov, aspect_ratio, aperture, focus_dist, &c);
    }
    Ray get_ray(double s, double t) const                                                              // camera.rs:47-54
    {
        Vec3 rd = c.lens_radius * Vec3::random_in_unit_disk();
        Vec3 offset = v(c.u) * rd.x() + v(c.v) * rd.y();
        return Ray(v(c.origin) + offset, v(c.lower_left_corner) + s * v(c.horizontal) + t * v(c.vertical) - v(c.origin) - offset);
    }
    const rtiow_camera& raw() const { return c; }
};

// ------------------------------------------------------------------------------------------------ the new call
struct RenderParams {                                     // runtime form of the consts at main.rs:24-28,44,137
    uint32_t width = 200, height = 133; uint32_t spp = 100; int32_t max_depth = 50; double t_min = 0.0001;
    uint64_t seed = 1; int n_gpus = 1; uint8_t alpha = 255; bool f64 = false; uint32_t tile_rows = 1;
    int scan = RTIOW_SCAN_AUTO;                           // where the sphere filter runs: tensor cores when the scene qualifies
    int gather = RTIOW_GATHER_AUTO;                       // n_gpus > 1: how the row tiles reach GPU 0
};

class RenderError : public std::runtime_error {
public:
    enum Kind { InvalidArg = RTIOW_ERR_INVALID_ARG, Unsupported = RTIOW_ERR_UNSUPPORTED, Cuda = RTIOW_ERR_CUDA, Nccl = RTIOW_ERR_NCCL,
                NoDevice = RTIOW_ERR_NO_DEVICE, NoMem = RTIOW_ERR_NOMEM, Cancelled = RTIOW_ERR_CANCELLED };
    Kind kind;
    RenderError(int code, const std::string& msg) : std::runtime_error(msg), kind(Kind(code)) {}
};

// per-pass preview: called with (pass [1-based], n_passes, spp done so far, the frame so far); return true to stop the render
using ProgressFn = std::function<bool(uint32_t, uint32_t, uint32_t, const std::vector<uint8_t>&)>;

namespace detail {
struct ProgressCtx { const ProgressFn* fn; const std::vector<uint8_t>* frame; };
inline int progress_trampoline(void* user, uint32_t pass, uint32_t n_passes, uint32_t spp_done, const uint8_t*)
{
    auto* pc = static_cast<ProgressCtx*>(user);
    return (*pc->fn)(pass, n_passes, spp_done, *pc->frame) ? 1 : 0;
}
}  // namespace detail

// The float buffers of render_aov(), top-down: color, albedo and normal hold 3 floats per pixel, depth one (include/rtiow_cuda.h,
// rtiow_render_aov).
struct Aovs { std::vector<float> color, albedo, normal, depth; };

// The per-pixel results of render_adaptive(), top-down: each pixel's sample count and its error at the last boundary it reached
// (include/rtiow_cuda.h, rtiow_render_adaptive).
struct AdaptiveMaps { std::vector<uint32_t> spp; std::vector<float> error; };
namespace detail { struct Adaptive { uint32_t min_spp; double tolerance; AdaptiveMaps* maps; }; }

// The world as the GPU sees it + one render call; n_passes == 0: rtiow_render, else rtiow_render_progressive; with `views`:
// rtiow_render_views of those cameras (cam is not used); with `aovs`: rtiow_render_aov into them; with `adaptive`:
// rtiow_render_adaptive into its maps.
inline std::vector<uint8_t> render_impl(const Camera& cam, const HittableList& world, const RenderParams& p, rtiow_stats* stats, uint32_t n_passes,
                                        const ProgressFn* on_pass, const std::vector<Camera>* views = nullptr, Aovs* aovs = nullptr,
                                        const detail::Adaptive* adaptive = nullptr)
{
    std::vector<double> cx, cy, cz, rad, ar, ag, ab, prm; std::vector<uint32_t> mi, kind;
    std::vector<const Scatter*> seen;
    for (const auto& h : world.iter()) {
        auto d = h->describe();
        if (!d) throw RenderError(RTIOW_ERR_UNSUPPORTED, "a shape in the HittableList has no GPU description (no CPU fallback)");
        auto m = d->mat ? d->mat->describe() : std::nullopt;
        if (!m) throw RenderError(RTIOW_ERR_UNSUPPORTED, "a material has no GPU description (no CPU fallback)");
        uint32_t id = 0;
        for (; id < seen.size(); ++id) if (seen[id] == d->mat.get()) break;
        if (id == seen.size()) {
            seen.push_back(d->mat.get());
            kind.push_back(m->kind); ar.push_back(m->albedo[0]); ag.push_back(m->albedo[1]); ab.push_back(m->albedo[2]); prm.push_back(m->param);
        }
        cx.push_back(d->sphere.center[0]); cy.push_back(d->sphere.center[1]); cz.push_back(d->sphere.center[2]); rad.push_back(d->sphere.radius); mi.push_back(id);
    }
    rtiow_ctx* ctx = nullptr;
    auto check = [&](int rc) { if (rc != RTIOW_OK) { std::string m = rtiow_last_error(); if (ctx) rtiow_ctx_destroy(ctx); throw RenderError(rc, m); } };
    check(rtiow_ctx_create(p.n_gpus, &ctx));
    check(rtiow_ctx_set_scan_backend(ctx, p.scan));
    check(rtiow_ctx_set_gather(ctx, p.gather));
    rtiow_spheres s{ cx.data(), cy.data(), cz.data(), rad.data(), mi.data(), uint32_t(rad.size()) };
    rtiow_materials m{ kind.data(), ar.data(), ag.data(), ab.data(), prm.data(), uint32_t(kind.size()) };
    check(rtiow_scene_upload(ctx, &s, &m));
    rtiow_params rp; rtiow_params_default(&rp);
    rp.width = p.width; rp.height = p.height; rp.spp = p.spp; rp.max_depth = p.max_depth; rp.t_min = p.t_min; rp.seed = p.seed; rp.alpha = p.alpha;
    rp.precision = p.f64 ? RTIOW_PRECISION_F64 : RTIOW_PRECISION_F32; rp.tile_rows = p.tile_rows;
    std::vector<uint8_t> out(size_t(4) * p.width * p.height * (views ? views->size() : 1));
    if (views) {
        std::vector<rtiow_camera> raw; for (const Camera& v : *views) raw.push_back(v.raw());
        check(rtiow_render_views(ctx, raw.data(), uint32_t(raw.size()), &rp, out.data(), stats));
    } else if (aovs) {
        const size_t n = size_t(p.width) * p.height;
        aovs->color.resize(3 * n); aovs->albedo.resize(3 * n); aovs->normal.resize(3 * n); aovs->depth.resize(n);
        check(rtiow_render_aov(ctx, &cam.raw(), &rp, out.data(), aovs->color.data(), aovs->albedo.data(), aovs->normal.data(), aovs->depth.data(), stats));
    } else if (adaptive) {
        const size_t n = size_t(p.width) * p.height;
        adaptive->maps->spp.resize(n); adaptive->maps->error.resize(n);
        check(rtiow_render_adaptive(ctx, &cam.raw(), &rp, adaptive->min_spp, adaptive->tolerance, out.data(), adaptive->maps->spp.data(),
                                    adaptive->maps->error.data(), stats));
    } else if (n_passes == 0) check(rtiow_render(ctx, &cam.raw(), &rp, out.data(), stats));
    else {
        detail::ProgressCtx pc{ on_pass, &out };
        check(rtiow_render_progressive(ctx, &cam.raw(), &rp, n_passes, on_pass && *on_pass ? detail::progress_trampoline : nullptr, &pc, out.data(), stats));
    }
    rtiow_ctx_destroy(ctx);
    return out;
}

// render(): replaces main.rs:122-145.  Returns top-down RGBA8, 4*W*H bytes — the Vec<u8> handed to
// ImageBuffer::from_vec at main.rs:147.  Throws RenderError (Rust: Err(RenderError)); never aborts.
inline std::vector<uint8_t> render(const Camera& cam, const HittableList& world, const RenderParams& p, rtiow_stats* stats = nullptr)
{
    return render_impl(cam, world, p, stats, 0, nullptr);
}

// render_views(): many cameras of one world in one call (a turntable, a stereo pair, a camera sweep).  Returns the views'
// top-down RGBA8 frames one after the other, 4*W*H bytes each; frame v is byte-identical to render(cams[v], world, p).
inline std::vector<uint8_t> render_views(const std::vector<Camera>& cams, const HittableList& world, const RenderParams& p, rtiow_stats* stats = nullptr)
{
    if (cams.empty()) throw RenderError(RTIOW_ERR_INVALID_ARG, "render_views needs at least one camera");
    return render_impl(cams.front(), world, p, stats, 0, nullptr, &cams);
}

// render_aov(): render()'s frame, byte for byte, plus the float buffers a denoiser takes in *aovs: linear colour, and the
// albedo, normal and distance of each camera ray's first hit, averaged over the samples.
inline std::vector<uint8_t> render_aov(const Camera& cam, const HittableList& world, const RenderParams& p, Aovs* aovs, rtiow_stats* stats = nullptr)
{
    if (!aovs) throw RenderError(RTIOW_ERR_INVALID_ARG, "render_aov needs an Aovs to fill");
    return render_impl(cam, world, p, stats, 0, nullptr, nullptr, aovs);
}

// render_adaptive(): adaptive sampling.  Each pixel gets between min_spp and p.spp samples, as many as its own noise asks for
// (its error, one standard error of the displayed value in 8-bit levels, at most `tolerance`), and is byte-identical to
// render() at its own count; *maps receives every pixel's count and error.
inline std::vector<uint8_t> render_adaptive(const Camera& cam, const HittableList& world, const RenderParams& p, uint32_t min_spp, double tolerance,
                                            AdaptiveMaps* maps, rtiow_stats* stats = nullptr)
{
    if (!maps) throw RenderError(RTIOW_ERR_INVALID_ARG, "render_adaptive needs an AdaptiveMaps to fill");
    const detail::Adaptive a{ min_spp, tolerance, maps };
    return render_impl(cam, world, p, stats, 0, nullptr, nullptr, nullptr, &a);
}

// render_progressive(): the same frame in n_passes slices of the samples, with a preview after each — what the reference's
// progress bar (main.rs:120,124) and preview window (main.rs:151-171) are for.  The returned frame is bit-identical to
// render()'s.  A callback that returns true stops the render: RenderError::Cancelled.
inline std::vector<uint8_t> render_progressive(const Camera& cam, const HittableList& world, const RenderParams& p, uint32_t n_passes,
                                               const ProgressFn& on_pass, rtiow_stats* stats = nullptr)
{
    return render_impl(cam, world, p, stats, n_passes ? n_passes : 1, &on_pass);
}

namespace detail {
inline HittableList world_from_arrays(uint32_t n, const std::vector<double>& cx, const std::vector<double>& cy, const std::vector<double>& cz,
                                      const std::vector<double>& r, const std::vector<uint32_t>& kind, const std::vector<double>& alb, const std::vector<double>& prm)
{
    HittableList world;
    for (uint32_t i = 0; i < n; ++i) {
        std::shared_ptr<const Scatter> m;
        Color a(alb[3 * i], alb[3 * i + 1], alb[3 * i + 2]);
        if (kind[i] == RTIOW_MAT_LAMBERTIAN) m = std::make_shared<Lambertian>(a);
        else if (kind[i] == RTIOW_MAT_METAL) m = std::make_shared<Metal>(a, prm[i]);
        else m = std::make_shared<Dialectric>(prm[i]);
        world.push(std::make_unique<Sphere>(Point3(cx[i], cy[i], cz[i]), r[i], m));
    }
    return world;
}
}  // namespace detail

// random_scene (main.rs:59-102) with an explicit seed
inline HittableList random_scene(uint64_t seed = 1, int half_extent = 11, int material_mode = 0)
{
    const uint32_t cap = uint32_t((2 * half_extent + 1) * (2 * half_extent + 1) + 8);
    std::vector<double> cx(cap), cy(cap), cz(cap), r(cap), alb(3 * size_t(cap)), prm(cap); std::vector<uint32_t> kind(cap); uint32_t n = 0;
    int rc = rtiow_random_scene(seed, half_extent, material_mode, cap, cx.data(), cy.data(), cz.data(), r.data(), kind.data(), alb.data(), prm.data(), &n);
    if (rc != RTIOW_OK) throw RenderError(rc, "rtiow_random_scene failed");
    return detail::world_from_arrays(n, cx, cy, cz, r, kind, alb, prm);
}

// Scene files (rtiow_scene_save / rtiow_scene_load): the same world for this library, the oracle and a cargo build of the
// reference.  save_scene writes one line per sphere of the HittableList; anything that does not describe() itself throws.
inline void save_scene(const HittableList& world, const std::string& path)
{
    std::vector<double> cx, cy, cz, r, alb, prm; std::vector<uint32_t> kind;
    for (const auto& h : world.iter()) {
        auto d = h->describe();
        auto m = d && d->mat ? d->mat->describe() : std::nullopt;
        if (!d || !m) throw RenderError(RTIOW_ERR_UNSUPPORTED, "a shape or material of the HittableList has no description");
        cx.push_back(d->sphere.center[0]); cy.push_back(d->sphere.center[1]); cz.push_back(d->sphere.center[2]); r.push_back(d->sphere.radius);
        kind.push_back(m->kind); alb.insert(alb.end(), m->albedo, m->albedo + 3); prm.push_back(m->param);
    }
    int rc = rtiow_scene_save(path.c_str(), uint32_t(r.size()), cx.data(), cy.data(), cz.data(), r.data(), kind.data(), alb.data(), prm.data());
    if (rc != RTIOW_OK) throw RenderError(rc, "cannot write scene file " + path);
}
inline HittableList load_scene(const std::string& path)
{
    uint32_t n = 0;
    int rc = rtiow_scene_load(path.c_str(), 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, &n);
    if (rc != RTIOW_OK) throw RenderError(rc, "cannot read scene file " + path);
    const uint32_t cap = n ? n : 1;
    std::vector<double> cx(cap), cy(cap), cz(cap), r(cap), alb(3 * size_t(cap)), prm(cap); std::vector<uint32_t> kind(cap);
    rc = rtiow_scene_load(path.c_str(), cap, cx.data(), cy.data(), cz.data(), r.data(), kind.data(), alb.data(), prm.data(), &n);
    if (rc != RTIOW_OK) throw RenderError(rc, "malformed scene file " + path);
    return detail::world_from_arrays(n, cx, cy, cz, r, kind, alb, prm);
}

// ------------------------------------------------------------------------------------------------ output stage (SURVEY §8f #2)
// top-down RGBA8 -> binary PPM (P6, alpha dropped) and PNG (RGBA8, stored deflate blocks: no zlib needed).
inline bool write_ppm(const std::string& path, uint32_t w, uint32_t h, const std::vector<uint8_t>& rgba)
{
    FILE* f = std::fopen(path.c_str(), "wb"); if (!f) return false;
    std::fprintf(f, "P6\n%u %u\n255\n", w, h);
    for (size_t i = 0; i < size_t(w) * h; ++i) std::fwrite(&rgba[4 * i], 1, 3, f);
    return std::fclose(f) == 0;
}
inline bool write_png(const std::string& path, uint32_t w, uint32_t h, const std::vector<uint8_t>& rgba)
{
    auto crc32 = [](const uint8_t* d, size_t n, uint32_t c = 0xffffffffu) { for (size_t i = 0; i < n; ++i) { c ^= d[i]; for (int k = 0; k < 8; ++k) c = (c >> 1) ^ (0xedb88320u & (0u - (c & 1u))); } return c; };
    auto be32 = [](std::vector<uint8_t>& v, uint32_t x) { v.push_back(x >> 24); v.push_back(x >> 16); v.push_back(x >> 8); v.push_back(x); };
    std::vector<uint8_t> raw; raw.reserve((size_t(w) * 4 + 1) * h);
    for (uint32_t y = 0; y < h; ++y) { raw.push_back(0); raw.insert(raw.end(), rgba.begin() + size_t(y) * w * 4, rgba.begin() + size_t(y + 1) * w * 4); }
    std::vector<uint8_t> z = { 0x78, 0x01 };
    uint32_t a = 1, b = 0;
    for (uint8_t c : raw) { a = (a + c) % 65521u; b = (b + a) % 65521u; }
    for (size_t off = 0; off < raw.size();) {
        size_t n = std::min<size_t>(65535, raw.size() - off); bool last = off + n == raw.size();
        z.push_back(last ? 1 : 0); z.push_back(n & 255); z.push_back(n >> 8); z.push_back(~n & 255); z.push_back((~n >> 8) & 255);
        z.insert(z.end(), raw.begin() + off, raw.begin() + off + n); off += n;
    }
    be32(z, (b << 16) | a);
    std::vector<uint8_t> out = { 0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a };
    auto chunk = [&](const char* tag, const std::vector<uint8_t>& d) {
        be32(out, uint32_t(d.size())); std::vector<uint8_t> t(tag, tag + 4); t.insert(t.end(), d.begin(), d.end());
        out.insert(out.end(), t.begin(), t.end()); be32(out, ~crc32(t.data(), t.size()));
    };
    std::vector<uint8_t> ihdr; be32(ihdr, w); be32(ihdr, h); ihdr.insert(ihdr.end(), { 8, 6, 0, 0, 0 });
    chunk("IHDR", ihdr); chunk("IDAT", z); chunk("IEND", {});
    FILE* f = std::fopen(path.c_str(), "wb"); if (!f) return false;
    std::fwrite(out.data(), 1, out.size(), f);
    return std::fclose(f) == 0;
}
// top-down float RGB (render_aov's colour) -> PFM ("PF", scale -1: little-endian floats, rows stored bottom-up)
inline bool write_pfm(const std::string& path, uint32_t w, uint32_t h, const std::vector<float>& rgb)
{
    FILE* f = std::fopen(path.c_str(), "wb"); if (!f) return false;
    std::fprintf(f, "PF\n%u %u\n-1.0\n", w, h);
    for (uint32_t y = h; y-- > 0;) std::fwrite(&rgb[size_t(y) * w * 3], sizeof(float), size_t(w) * 3, f);
    return std::fclose(f) == 0;
}
// per-pixel sample counts (render_adaptive's) -> RGBA8 heat map for write_png: blue at lo samples to red at hi, on a log scale
inline std::vector<uint8_t> spp_heat_map(const std::vector<uint32_t>& spp, uint32_t lo, uint32_t hi)
{
    std::vector<uint8_t> out(spp.size() * 4, 255);
    const double span = hi > lo ? std::log(double(hi) / double(lo)) : 1.0;
    for (size_t i = 0; i < spp.size(); ++i) {
        const double v = std::min(1.0, std::max(0.0, std::log(double(std::max(spp[i], lo)) / double(lo)) / span));
        out[4 * i] = uint8_t(std::lround(255.0 * v)); out[4 * i + 1] = uint8_t(std::lround(255.0 * (1.0 - std::fabs(2.0 * v - 1.0))));
        out[4 * i + 2] = uint8_t(std::lround(255.0 * (1.0 - v)));
    }
    return out;
}
// float RGB in [0, 1] per channel (render_aov's albedo, or 0.5 n + 0.5 of its normal) -> RGBA8 for write_png
inline std::vector<uint8_t> unit_rgb_to_rgba(const std::vector<float>& rgb, float scale = 1.0f, float offset = 0.0f)
{
    std::vector<uint8_t> out(rgb.size() / 3 * 4, 255);
    for (size_t i = 0; i < rgb.size() / 3; ++i)
        for (int c = 0; c < 3; ++c) out[4 * i + c] = uint8_t(std::lround(255.0f * std::min(1.0f, std::max(0.0f, scale * rgb[3 * i + c] + offset))));
    return out;
}

}  // namespace rtiow
