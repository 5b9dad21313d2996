// example_main.cpp — the reference's main() (/root/reference/src/main.rs:104-178) with the render loop
// (main.rs:122-145) replaced by rtiow::render(), and the compile-time constants (main.rs:24-28) turned
// into flags (SURVEY §8f #3).  No preview window (main.rs:151-171 cannot run headless).
//
//   rtiow_host_example [--width W] [--height H] [--spp N] [--depth D] [--seed S] [--scene-seed S] [--gpus G]
//                      [--grid HALF_EXTENT] [--materials 0..3] [--f64] [--passes N] [--views N] [--aov]
//                      [--denoise] [--render-denoised] [--adaptive TOL [--min-spp N]] [--out image.png|image.ppm] [--selftest]
// --views N renders N cameras orbiting the look-at point about the vertical axis in one call and writes out_000.png ...
// (with --out, the frames are named after its stem: --out orbit.ppm writes orbit_000.ppm ...).
// --aov also writes the inputs of a denoiser beside the image: <stem>_color.pfm (linear colour), <stem>_albedo.png and
// <stem>_normal.png (0.5 n + 0.5).  --denoise (implies --aov) also runs the library's a-trous denoiser (default parameters) over
// them and writes <stem>_denoised.png.  --render-denoised writes only <stem>_denoised.png, through one call that keeps the AOVs on
// the GPU (render_denoised; the same bytes as --denoise's).
// --adaptive TOL renders with adaptive sampling (render_adaptive): between --min-spp N (default 16, at most --spp) and --spp
// samples per pixel, until a pixel's error is at most TOL 8-bit levels; it also writes <stem>_spp.png, a heat map of the
// per-pixel counts (blue: min-spp, red: spp, log scale).
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <iostream>

#include "rtiow.hpp"

using namespace rtiow;

// a caller's own ray_color keeps compiling against the mirrored API (main.rs:38-57)
static Color ray_color(const Ray& r, const HittableList& world, int depth)
{
    if (depth <= 0) return Color::zero();
    if (auto shape = world.hit(r, 0.0001, std::numeric_limits<double>::infinity())) {
        if (auto s = shape->get_mat()->scatter(r, *shape)) return s->first * ray_color(s->second, world, depth - 1);
        return Color(0, 0, 0);
    }
    Vec3 ud = r.direction().unit_vector();
    double t = 0.5 * (ud.y() + 1.0);
    return (1.0 - t) * Color(1, 1, 1) + t * Color(0.5, 0.7, 1.0);
}

struct Unknown : Hit {   // a shape the GPU path does not know
    std::optional<HitRecord> hit(const Ray&, double, double) const override { return std::nullopt; }
};

// the reference camera (main.rs:108-118) turned by `angle` radians about the vertical axis through the look-at point
static Camera orbit_camera(double angle, double aspect)
{
    const double c = std::cos(angle), s = std::sin(angle);
    return Camera(Point3(13 * c + 3 * s, 2, 3 * c - 13 * s), Point3(0, 0, 0), Vec3(0, 1, 0), 20.0, aspect, 0.1, 10.0);
}

static int selftest()
{
    int bad = 0;
    auto expect = [&](bool ok, const char* what) { if (!ok) { std::cerr << "FAIL: " << what << "\n"; ++bad; } };
    HittableList world = random_scene(1);
    Camera cam(Point3(13, 2, 3), Point3(0, 0, 0), Vec3(0, 1, 0), 20.0, 16.0 / 9.0, 0.1, 10.0);
    RenderParams p; p.width = 160; p.height = 90; p.spp = 8; p.seed = 1;
    rtiow_stats st{};
    std::vector<uint8_t> a = render(cam, world, p, &st), b = render(cam, world, p);
    expect(a.size() == size_t(4) * 160 * 90 && a == b, "render is deterministic and sized 4*W*H");
    expect(st.paths == 160ull * 90 * 8 && st.rays_traced > st.paths, "stats");
    bool alpha = true; for (size_t i = 3; i < a.size(); i += 4) alpha &= a[i] == 255;
    expect(alpha, "alpha == 255 (main.rs:137)");
    // top rows are sky: B = 255, R in the 150..225 band
    expect(a[2] == 255 && a[0] > 140 && a[0] < 230, "top-left pixel is sky (row 0 is the TOP, main.rs:141-145)");
    // host ray_color on the same world agrees with the image on average over a sky region and a ground region
    double host = 0, gpu = 0; int n = 0;
    for (int y = 70; y < 90; y += 4) for (int x = 0; x < 160; x += 8) {
        Color c = Color::zero();
        for (int s = 0; s < 64; ++s) c = c + ray_color(cam.get_ray((x + gen_f64()) / 159.0, ((89 - y) + gen_f64()) / 89.0), world, 50);
        auto q = c.to_rgba(255, 64);
        host += q[0] + q[1] + q[2]; gpu += a[4 * (y * 160 + x)] + a[4 * (y * 160 + x) + 1] + a[4 * (y * 160 + x) + 2]; ++n;
    }
    expect(std::fabs(host - gpu) / n < 25.0, "host ray_color (mirrored API) and GPU image agree on average");
    try { world.push(std::make_unique<Unknown>()); render(cam, world, p); expect(false, "unknown shape must be Unsupported"); }
    catch (const RenderError& e) { expect(e.kind == RenderError::Unsupported, "unknown shape -> RenderError::Unsupported"); }
    try { RenderParams q = p; q.width = 1; render(cam, random_scene(1), q); expect(false, "width 1 must be InvalidArg"); }
    catch (const RenderError& e) { expect(e.kind == RenderError::InvalidArg, "width 1 -> RenderError::InvalidArg"); }
    // progressive preview: 4 passes of 2 spp; the last frame equals render()'s, the first equals render() at 2 spp
    { std::vector<uint32_t> seen; std::vector<uint8_t> first;
      std::vector<uint8_t> c = render_progressive(cam, random_scene(1), p, 4, [&](uint32_t k, uint32_t n, uint32_t done, const std::vector<uint8_t>& f) {
          seen.push_back(done); if (k == 1) first = f; return n != 4; });
      RenderParams q = p; q.spp = 2;
      expect(c == a && seen == std::vector<uint32_t>({ 2, 4, 6, 8 }) && first == render(cam, random_scene(1), q), "render_progressive: passes, preview and final frame");
      try { render_progressive(cam, random_scene(1), p, 4, [](uint32_t, uint32_t, uint32_t, const std::vector<uint8_t>&) { return true; }); expect(false, "cancel must throw"); }
      catch (const RenderError& e) { expect(e.kind == RenderError::Cancelled, "callback returning true -> RenderError::Cancelled"); } }
    // a batch of views: three orbit cameras in one call, each frame byte-identical to its own render()
    { std::vector<Camera> cams = { orbit_camera(0.0, 16.0 / 9.0), orbit_camera(2.0, 16.0 / 9.0), orbit_camera(4.0, 16.0 / 9.0) };
      rtiow_stats sv{};
      std::vector<uint8_t> v = render_views(cams, random_scene(1), p, &sv);
      const size_t fb = size_t(4) * p.width * p.height;
      bool same = v.size() == 3 * fb;
      uint64_t rays = 0;
      for (size_t k = 0; k < cams.size() && same; ++k) {
          rtiow_stats sk{};
          same = std::equal(v.begin() + k * fb, v.begin() + (k + 1) * fb, render(cams[k], random_scene(1), p, &sk).begin());
          rays += sk.rays_traced;
      }
      expect(same && std::equal(v.begin(), v.begin() + fb, a.begin()), "render_views: every view equals its own render() byte for byte");
      expect(sv.paths == 3ull * p.width * p.height * p.spp && sv.rays_traced == rays, "render_views stats: paths and rays of the batch"); }
    // the frame with AOVs: out_rgba byte-identical to render()'s, the colour its own sums, albedo and normal in range
    { Aovs av; rtiow_stats sa{};
      std::vector<uint8_t> f = render_aov(cam, random_scene(1), p, &av, &sa);
      const size_t n = size_t(p.width) * p.height;
      expect(f == a && sa.rays_traced == st.rays_traced, "render_aov: the frame equals render()'s byte for byte");
      bool sized = av.color.size() == 3 * n && av.albedo.size() == 3 * n && av.normal.size() == 3 * n && av.depth.size() == n, ranged = sized;
      for (size_t i = 0; ranged && i < 3 * n; ++i) ranged = av.color[i] >= 0 && av.albedo[i] >= 0 && av.albedo[i] <= 1 && std::fabs(av.normal[i]) <= 1.0f + 1e-5f;
      expect(ranged && std::isinf(av.depth[0]) && av.depth[n - 1] > 0 && av.depth[n - 1] < 100, "render_aov: buffers sized, in range, sky depth inf, ground depth finite");
      // the denoiser over those buffers: deterministic, sized, and its frame's bytes agree with its own colour's range
      std::vector<float> dc; rtiow_stats sn{};
      const std::vector<uint8_t> d1 = denoise(p.width, p.height, av, default_denoise_params(), &dc, &sn), d2 = denoise(p.width, p.height, av, default_denoise_params());
      expect(d1 == d2 && d1.size() == 4 * n && dc.size() == 3 * n && d1[3] == 255, "denoise: the same bytes on a second call, sized 4*W*H, alpha 255");
      expect(sn.h2d_bytes == 40ull * n && sn.d2h_bytes == 16ull * n && sn.n_gpus == 1 && sn.paths == 0, "denoise stats: 40 B/px up, 16 B/px down");
      // the same render and filter in one call, the AOVs kept on the GPU: the same bytes and colour bits
      std::vector<float> rc; rtiow_stats sr{};
      const std::vector<uint8_t> r1 = render_denoised(cam, random_scene(1), p, default_denoise_params(), &rc, &sr);
      expect(r1 == d1 && rc.size() == dc.size() && std::memcmp(rc.data(), dc.data(), dc.size() * sizeof(float)) == 0,
             "render_denoised equals denoise(render_aov(...)) byte for byte");
      expect(sr.rays_traced == st.rays_traced && sr.d2h_bytes == 16 + 16ull * n, "render_denoised stats: render_aov's rays, 16 B/px + the counters down"); }
    // adaptive sampling with min_spp == spp renders every pixel at spp: render()'s frame, rays and paths
    { AdaptiveMaps am; rtiow_stats sd{};
      std::vector<uint8_t> f = render_adaptive(cam, random_scene(1), p, p.spp, 1.0, &am, &sd);
      bool flat = am.spp.size() == size_t(p.width) * p.height;
      for (size_t i = 0; flat && i < am.spp.size(); ++i) flat = am.spp[i] == p.spp;
      expect(f == a && sd.rays_traced == st.rays_traced && sd.paths == st.paths && flat, "render_adaptive with min_spp == spp equals render() byte for byte"); }
    // the files below go to a private directory: a fixed name in the shared temporary directory may belong to another user
    std::string dir = (std::filesystem::temp_directory_path() / "rtiow_selftest_XXXXXX").string();
    if (!mkdtemp(dir.data())) { std::cerr << "FAIL: cannot create a temporary directory\nselftest FAILED\n"; return 1; }
    // scene files: the world survives a round trip bit for bit, and both filter backends render it
    { save_scene(random_scene(1), dir + "/scene.txt");
      expect(render(cam, load_scene(dir + "/scene.txt"), p) == a, "scene file round trip renders the same frame");
      RenderParams q = p; q.scan = RTIOW_SCAN_FP32; rtiow_stats sq{};
      std::vector<uint8_t> f = render(cam, random_scene(1), q, &sq); size_t diff = 0;
      for (size_t i = 0; i < f.size(); ++i) diff += f[i] != a[i];
      expect(sq.scan_backend == RTIOW_SCAN_FP32 && diff <= f.size() / 1000, "FP32 filter backend renders the same frame (up to last-bit path differences)"); }
    expect(write_png(dir + "/selftest.png", 160, 90, a) && write_ppm(dir + "/selftest.ppm", 160, 90, a), "PNG/PPM written");
    std::error_code ec; std::filesystem::remove_all(dir, ec);
    std::cout << (bad ? "selftest FAILED\n" : "selftest ok\n");
    return bad ? 1 : 0;
}

int main(int argc, char** argv)
{
    RenderParams p; p.width = 200; p.height = 133;                       // main.rs:24-28
    uint64_t scene_seed = 1; int grid = 11, materials = 0; std::string out = "image.png";     // main.rs:177
    bool explicit_h = false, explicit_out = false, aov = false, denoised = false, fused = false; uint32_t passes = 0, views = 0; std::string scene_file, dump_scene;
    double adaptive = -1.0; uint32_t min_spp = 16;
    for (int i = 1; i < argc; ++i) {
        auto next = [&]() -> const char* { if (i + 1 >= argc) { std::cerr << "missing value for " << argv[i] << "\n"; std::exit(2); } return argv[++i]; };
        if (!std::strcmp(argv[i], "--width")) p.width = std::atoi(next());
        else if (!std::strcmp(argv[i], "--height")) { p.height = std::atoi(next()); explicit_h = true; }
        else if (!std::strcmp(argv[i], "--spp")) p.spp = std::atoi(next());
        else if (!std::strcmp(argv[i], "--depth")) p.max_depth = std::atoi(next());
        else if (!std::strcmp(argv[i], "--seed")) p.seed = std::strtoull(next(), nullptr, 10);
        else if (!std::strcmp(argv[i], "--scene-seed")) scene_seed = std::strtoull(next(), nullptr, 10);
        else if (!std::strcmp(argv[i], "--gpus")) p.n_gpus = std::atoi(next());
        else if (!std::strcmp(argv[i], "--grid")) grid = std::atoi(next());
        else if (!std::strcmp(argv[i], "--materials")) materials = std::atoi(next());
        else if (!std::strcmp(argv[i], "--f64")) p.f64 = true;
        else if (!std::strcmp(argv[i], "--passes")) passes = uint32_t(std::atoi(next()));
        else if (!std::strcmp(argv[i], "--views")) views = uint32_t(std::atoi(next()));
        else if (!std::strcmp(argv[i], "--aov")) aov = true;
        else if (!std::strcmp(argv[i], "--denoise")) denoised = aov = true;        // implies --aov
        else if (!std::strcmp(argv[i], "--render-denoised")) fused = true;
        else if (!std::strcmp(argv[i], "--adaptive")) adaptive = std::atof(next());
        else if (!std::strcmp(argv[i], "--min-spp")) min_spp = uint32_t(std::atoi(next()));
        else if (!std::strcmp(argv[i], "--out")) { out = next(); explicit_out = true; }
        else if (!std::strcmp(argv[i], "--scene")) scene_file = next();               // render the world of a scene file instead of random_scene
        else if (!std::strcmp(argv[i], "--dump-scene")) dump_scene = next();          // write the world to a scene file (for the oracle / a cargo build)
        else if (!std::strcmp(argv[i], "--scan")) { const char* v = next(); p.scan = !std::strcmp(v, "fp32") ? RTIOW_SCAN_FP32 : !std::strcmp(v, "tensor") ? RTIOW_SCAN_TENSOR : RTIOW_SCAN_AUTO; }
        else if (!std::strcmp(argv[i], "--gather")) { const char* v = next(); p.gather = !std::strcmp(v, "nccl") ? RTIOW_GATHER_NCCL : !std::strcmp(v, "fused") ? RTIOW_GATHER_FUSED : RTIOW_GATHER_AUTO; }
        else if (!std::strcmp(argv[i], "--selftest")) return selftest();
        else { std::cerr << "unknown flag " << argv[i] << "\n"; return 2; }
    }
    if (!explicit_h) p.height = uint32_t(double(p.width) / (3.0 / 2.0));  // IMAGE_HEIGHT truncates (main.rs:24,26)
    try {
        HittableList world = scene_file.empty() ? random_scene(scene_seed, grid, materials) : load_scene(scene_file);   // main.rs:106
        if (!dump_scene.empty()) { save_scene(world, dump_scene); std::cout << dump_scene << " written (" << world.iter().size() << " spheres)\n"; }
        Camera cam(Point3(13, 2, 3), Point3(0, 0, 0), Vec3(0, 1, 0), 20.0, double(p.width) / double(p.height), 0.1, 10.0);   // main.rs:108-118
        rtiow_stats st{};
        const bool ppm = out.size() > 4 && out.substr(out.size() - 4) == ".ppm";
        if (views > 0) {                                                  // an orbit of `views` cameras in one call
            std::vector<Camera> cams;
            for (uint32_t k = 0; k < views; ++k) cams.push_back(orbit_camera(2.0 * 3.14159265358979323846 * k / views, double(p.width) / double(p.height)));
            std::vector<uint8_t> frames = render_views(cams, world, p, &st);
            std::cout << views << " views of " << p.width << "x" << p.height << " @ " << p.spp << " spp on " << st.n_gpus << " GPU(s): kernel " << st.kernel_ms
                      << " ms, " << double(st.paths) / st.kernel_ms / 1e3 << " Mpaths/s\n";
            const std::string stem = explicit_out ? out.substr(0, out.rfind('.') == std::string::npos ? out.size() : out.rfind('.')) : "out";
            const size_t fb = size_t(4) * p.width * p.height;
            for (uint32_t k = 0; k < views; ++k) {
                char name[32]; std::snprintf(name, sizeof name, "_%03u", k);
                const std::string path = stem + name + (ppm ? ".ppm" : ".png");
                std::vector<uint8_t> f(frames.begin() + k * fb, frames.begin() + (k + 1) * fb);
                if (!(ppm ? write_ppm(path, p.width, p.height, f) : write_png(path, p.width, p.height, f))) { std::cerr << "could not write " << path << "\n"; return 1; }
                std::cout << path << " saved\n";
            }
            return 0;
        }
        if (fused) {                                                      // the denoised frame only, its AOVs kept on the GPU
            const std::vector<uint8_t> dn = render_denoised(cam, world, p, default_denoise_params(), nullptr, &st);
            const std::string stem = out.substr(0, out.rfind('.') == std::string::npos ? out.size() : out.rfind('.'));
            std::cout << p.width << "x" << p.height << " @ " << p.spp << " spp denoised on " << st.n_gpus << " GPU(s): kernel " << st.kernel_ms
                      << " ms, call " << st.total_ms << " ms\n";
            if (!write_png(stem + "_denoised.png", p.width, p.height, dn)) { std::cerr << "could not write " << stem << "_denoised.png\n"; return 1; }
            std::cout << stem << "_denoised.png saved\n";
            return 0;
        }
        if (aov) {                                                        // the frame plus a denoiser's inputs
            Aovs av;
            std::vector<uint8_t> pixels = render_aov(cam, world, p, &av, &st);
            std::cout << p.width << "x" << p.height << " @ " << p.spp << " spp with AOVs on " << st.n_gpus << " GPU(s): kernel " << st.kernel_ms << " ms\n";
            const std::string stem = out.substr(0, out.rfind('.') == std::string::npos ? out.size() : out.rfind('.'));
            const bool ok = (ppm ? write_ppm(out, p.width, p.height, pixels) : write_png(out, p.width, p.height, pixels)) &&
                            write_pfm(stem + "_color.pfm", p.width, p.height, av.color) &&
                            write_png(stem + "_albedo.png", p.width, p.height, unit_rgb_to_rgba(av.albedo)) &&
                            write_png(stem + "_normal.png", p.width, p.height, unit_rgb_to_rgba(av.normal, 0.5f, 0.5f));
            if (!ok) { std::cerr << "could not write " << out << " and its AOV files\n"; return 1; }
            std::cout << out << ", " << stem << "_color.pfm, " << stem << "_albedo.png, " << stem << "_normal.png saved\n";
            if (denoised) {
                rtiow_stats sd{};
                const std::vector<uint8_t> dn = denoise(p.width, p.height, av, default_denoise_params(), nullptr, &sd);
                if (!write_png(stem + "_denoised.png", p.width, p.height, dn)) { std::cerr << "could not write " << stem << "_denoised.png\n"; return 1; }
                std::cout << "denoised: kernel " << sd.kernel_ms << " ms, call " << sd.total_ms << " ms; " << stem << "_denoised.png saved\n";
            }
            return 0;
        }
        if (adaptive >= 0.0) {                                            // per-pixel sample counts + their heat map
            AdaptiveMaps am;
            std::vector<uint8_t> pixels = render_adaptive(cam, world, p, std::min(min_spp, p.spp), adaptive, &am, &st);
            std::cout << p.width << "x" << p.height << " @ " << std::min(min_spp, p.spp) << ".." << p.spp << " spp (tolerance " << adaptive << ") on "
                      << st.n_gpus << " GPU(s): kernel " << st.kernel_ms << " ms, " << double(st.paths) / (double(p.width) * p.height) << " spp on average\n";
            const std::string stem = out.substr(0, out.rfind('.') == std::string::npos ? out.size() : out.rfind('.'));
            const bool ok = (ppm ? write_ppm(out, p.width, p.height, pixels) : write_png(out, p.width, p.height, pixels)) &&
                            write_png(stem + "_spp.png", p.width, p.height, spp_heat_map(am.spp, std::min(min_spp, p.spp), p.spp));
            if (!ok) { std::cerr << "could not write " << out << " and its heat map\n"; return 1; }
            std::cout << out << ", " << stem << "_spp.png saved\n";
            return 0;
        }
        auto t0 = std::chrono::steady_clock::now();
        // main.rs:122-145; with --passes N the progress the reference shows as a bar (main.rs:120,124) is printed per pass
        std::vector<uint8_t> pixels = passes == 0 ? render(cam, world, p, &st)
            : render_progressive(cam, world, p, passes, [](uint32_t k, uint32_t n, uint32_t done, const std::vector<uint8_t>&) {
                  std::cout << "pass " << k << "/" << n << ": " << done << " spp\n"; return false; }, &st);
        double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        std::cout << "\nDone.\n";                                        // main.rs:149
        std::cout << p.width << "x" << p.height << " @ " << p.spp << " spp on " << st.n_gpus << " GPU(s): kernel " << st.kernel_ms << " ms, call " << ms
                  << " ms (incl. ctx + upload), " << double(st.paths) / st.kernel_ms / 1e3 << " Mpaths/s, " << double(st.rays_traced) / double(st.paths) << " rays/path\n";
        bool ok = ppm ? write_ppm(out, p.width, p.height, pixels) : write_png(out, p.width, p.height, pixels);
        if (!ok) { std::cerr << "could not write " << out << "\n"; return 1; }
        std::cout << out << " saved to working directory\n";             // main.rs:196
    } catch (const RenderError& e) {
        std::cerr << "render failed (" << int(e.kind) << "): " << e.what() << "\n";
        return 1;
    }
    return 0;
}
