"""GPU suite, image level: rtiow_render (the drop-in for main.rs:122-145) against the oracle's render of the same
explicit scene.

Three strengths of comparison:
  * SAME PATHS.  The oracle's DIRECT sampler consumes the same Philox blocks as the GPU, so the f64 GPU render must
    reproduce the oracle's image essentially bit for bit, and the f32 render must differ only where f32 rounding
    flipped a knife-edge decision (rare, bounded).
  * STATISTICAL (the bound stated in BASELINE.md): against the oracle's reference-faithful REJECTION sampler,
    RMSE(gpu, oracle) <= 1.25 x RMSE(oracle seed A, oracle seed B) at equal spp, per-channel mean within 0.1/255
    (+ the Monte-Carlo standard error of that mean at test sizes), sky-only pixels within 1 LSB.
  * SIZE-INDEPENDENT PROPERTIES at BASELINE's full frame sizes: determinism, invariance to the row-tile partition
    (any world size / tile height gives the same bytes), ray counts, alpha, empty scenes.
"""
import numpy as np
import pytest

from conftest import final_camera

pytestmark = pytest.mark.gpu


def rmse(a, b):
    return float(np.sqrt(((a[..., :3].astype(float) - b[..., :3].astype(float)) ** 2).mean()))


def render_gpu(ctx, capi, cam, **kw):
    return ctx.render(cam, capi.default_params(**kw))


def test_cfg1_same_paths_f64(ctx_final, capi, oracle, final_scene):
    """BASELINE configs[0]: 400x225, 10 spp, depth 50 — the reference's own CPU-runnable case."""
    _, sc = final_scene
    W, H, spp = 400, 225, 10
    ref, _, cnt = oracle.render(sc, final_camera(oracle, W / H), W, H, spp, seed=1, sampler=oracle.SAMPLER_DIRECT)
    img, st = render_gpu(ctx_final, capi, final_camera(capi, W / H), width=W, height=H, spp=spp, seed=1, precision=capi.F64)
    diff = np.abs(img.astype(int) - ref.astype(int))
    assert (diff > 0).mean() < 2e-4, f"f64 GPU render differs from the oracle on {(diff > 0).sum()} bytes"
    assert diff.max() <= 2 or (diff > 2).sum() <= 6
    assert st["rays_traced"] == cnt["rays"] or abs(st["rays_traced"] - cnt["rays"]) < 1e-5 * cnt["rays"]
    assert st["paths"] == W * H * spp and st["sphere_tests"] == st["rays_traced"] * sc.n


def test_cfg1_same_paths_f32(ctx_final, capi, oracle, final_scene):
    _, sc = final_scene
    W, H, spp = 400, 225, 10
    ref, _, cnt = oracle.render(sc, final_camera(oracle, W / H), W, H, spp, seed=1, sampler=oracle.SAMPLER_DIRECT)
    img, st = render_gpu(ctx_final, capi, final_camera(capi, W / H), width=W, height=H, spp=spp, seed=1)
    diff = np.abs(img[..., :3].astype(int) - ref[..., :3].astype(int)).max(axis=2)
    assert (diff <= 1).mean() > 0.995, f"{(diff > 1).mean():.4%} of pixels differ by more than 1 LSB"
    assert rmse(img, ref) < 1.5                      # two independent seeds at 10 spp differ by RMSE ~ 12.8
    assert abs(st["rays_traced"] / cnt["rays"] - 1) < 2e-3
    assert (img[..., 3] == 255).all()


def test_statistical_parity_vs_reference_sampler(ctx_final, capi, oracle, final_scene):
    """the stated bound, against the reference-faithful rejection sampler with independent streams"""
    _, sc = final_scene
    W, H, spp = 256, 144, 64
    ocam = final_camera(oracle, W / H)
    a, acc_a, _ = oracle.render(sc, ocam, W, H, spp, seed=101, sampler=oracle.SAMPLER_REJECTION, want_accum=True)
    b, acc_b, _ = oracle.render(sc, ocam, W, H, spp, seed=202, sampler=oracle.SAMPLER_REJECTION, want_accum=True)
    img, _ = render_gpu(ctx_final, capi, final_camera(capi, W / H), width=W, height=H, spp=spp, seed=303)
    floor = rmse(a, b)
    assert rmse(img, a) <= 1.25 * floor and rmse(img, b) <= 1.25 * floor, (rmse(img, a), rmse(img, b), floor)
    # bias: per-channel mean of 8-bit values; tolerance 0.1 + 3 standard errors of the mean difference at this size
    se = np.sqrt(2) * floor / np.sqrt(W * H)
    for c in range(3):
        assert abs(img[..., c].astype(float).mean() - a[..., c].astype(float).mean()) <= 0.1 + 3 * se
    # sky-only pixels (top rows of this camera) within 1 LSB
    assert np.abs(img[:8, :, :3].astype(int) - a[:8, :, :3].astype(int)).max() <= 1


def test_statistical_parity_high_spp(ctx_final, capi, oracle, final_scene):
    """north_star's second parity level AT HIGH SPP (VERDICT r1 weak #1d): 400x225 @ 500 spp, where the noise floor is ~1.8 LSB and
    a bias would show.  Stated bound: RMSE(gpu, oracle) <= 1.25 x RMSE(oracle seed A, oracle seed B) and per-channel mean within
    0.1 of an 8-bit unit — no standard-error allowance needed at this size.  Two oracle renders with the reference-faithful
    rejection sampler (~30-45 s each on the host's threads).  The figures go to $RTIOW_REPORT_DIR/parity_image_r2.json when that
    variable is set (committed copy: profiles/parity_image_r2.json)."""
    import json
    import os
    from pathlib import Path
    _, sc = final_scene
    W, H, spp = 400, 225, 500
    ocam = final_camera(oracle, W / H)
    a, _, _ = oracle.render(sc, ocam, W, H, spp, seed=1001, sampler=oracle.SAMPLER_REJECTION)
    b, _, _ = oracle.render(sc, ocam, W, H, spp, seed=2002, sampler=oracle.SAMPLER_REJECTION)
    img, st = render_gpu(ctx_final, capi, final_camera(capi, W / H), width=W, height=H, spp=spp, seed=3003)
    floor, ra, rb = rmse(a, b), rmse(img, a), rmse(img, b)
    means = [float(img[..., c].astype(float).mean() - 0.5 * (a[..., c].astype(float).mean() + b[..., c].astype(float).mean())) for c in range(3)]
    if os.environ.get("RTIOW_REPORT_DIR"):
        out = Path(os.environ["RTIOW_REPORT_DIR"]) / "parity_image_r2.json"
        out.parent.mkdir(parents=True, exist_ok=True)
        out.write_text(json.dumps({"frame": [W, H, spp], "scan_backend": st["scan_backend"], "rmse_oracleA_oracleB": floor, "rmse_gpu_oracleA": ra,
                                   "rmse_gpu_oracleB": rb, "bound": 1.25 * floor, "mean_gpu_minus_oracle_per_channel": means, "mean_bound": 0.1,
                                   "psnr_gpu_oracleA_db": float(20 * np.log10(255.0 / ra))}, indent=1))
    assert 1.2 < floor < 2.6, floor                         # SURVEY §8c measured 1.81 at this size
    assert ra <= 1.25 * floor and rb <= 1.25 * floor, (ra, rb, floor)
    assert max(abs(m) for m in means) <= 0.1, means
    assert np.abs(img[:12, :, :3].astype(int) - a[:12, :, :3].astype(int)).max() <= 1          # sky-only rows


@pytest.mark.parametrize("mode,name", [(1, "all-Lambertian"), (2, "all-Metal"), (3, "all-Dialectric + hollow shell")])
def test_material_isolation_scenes(ctx, capi, oracle, scene_factory, mode, name):
    """BASELINE configs[2] (reduced size): divergence-stress scenes, same-path comparison per material"""
    arrays, sc = scene_factory(seed=2, mode=mode)
    ctx.upload_scene(**arrays)
    W, H, spp = 320, 180, 8
    ref, _, cnt = oracle.render(sc, final_camera(oracle, W / H), W, H, spp, seed=5, sampler=oracle.SAMPLER_DIRECT)
    img, st = render_gpu(ctx, capi, final_camera(capi, W / H), width=W, height=H, spp=spp, seed=5)
    diff = np.abs(img[..., :3].astype(int) - ref[..., :3].astype(int)).max(axis=2)
    assert (diff <= 1).mean() > 0.99, f"{name}: {(diff > 1).mean():.4%} pixels off by > 1 LSB"
    assert abs(st["rays_traced"] / cnt["rays"] - 1) < 5e-3
    img64, _ = render_gpu(ctx, capi, final_camera(capi, W / H), width=W, height=H, spp=spp, seed=5, precision=capi.F64)
    assert (np.abs(img64.astype(int) - ref.astype(int)) > 0).mean() < 5e-4


def test_many_spheres_scene(ctx, capi, oracle, scene_factory):
    """BASELINE configs[3] shape (10k spheres: filter SoA exceeds the small-scene shared-memory layout), tiny frame"""
    arrays, sc = scene_factory(seed=3, half_extent=50)
    assert sc.n > 10_000
    ctx.upload_scene(**arrays)
    W, H, spp = 96, 54, 2
    ref, _, cnt = oracle.render(sc, final_camera(oracle, W / H), W, H, spp, seed=8, sampler=oracle.SAMPLER_DIRECT)
    img, st = render_gpu(ctx, capi, final_camera(capi, W / H), width=W, height=H, spp=spp, seed=8)
    diff = np.abs(img[..., :3].astype(int) - ref[..., :3].astype(int)).max(axis=2)
    assert (diff <= 1).mean() > 0.99
    assert abs(st["rays_traced"] / cnt["rays"] - 1) < 1e-2


def test_determinism_and_seed(ctx_final, capi):
    cam = final_camera(capi, 16 / 9)
    a, sa = render_gpu(ctx_final, capi, cam, width=320, height=180, spp=16, seed=1)
    b, sb = render_gpu(ctx_final, capi, cam, width=320, height=180, spp=16, seed=1)
    c, _ = render_gpu(ctx_final, capi, cam, width=320, height=180, spp=16, seed=2)
    assert np.array_equal(a, b) and sa["rays_traced"] == sb["rays_traced"]       # bit-identical run to run
    assert not np.array_equal(a, c) and rmse(a, c) < 15


@pytest.mark.parametrize("prec", [0, 1])
def test_png_big_spheres_gpu(ctx, capi, prec):
    """the GPU render against the reference's OWN render (rtiow_part1_final.png), on the part of random_scene that is not
    random: metal cap to a quarter of an LSB, refracted sky and diffuse top within the shading of the reference's random
    neighbourhood — same fixture and bounds as the oracle's test (tests/test_oracle_golden.py::test_png_big_spheres)"""
    import json
    from conftest import ROOT
    g = json.load(open(ROOT / "tests" / "golden" / "png_big_spheres.json"))
    s = g["scene"]
    ctx.upload_scene(s["center"], s["radius"], [0, 1, 2, 3], s["mat_kind"], s["mat_albedo"], s["mat_param"])
    cam = capi.camera_new(**{k: v for k, v in g["camera"].items() if k != "cite"})
    img, _ = render_gpu(ctx, capi, cam, width=g["width"], height=g["height"], spp=128, seed=7, precision=prec)
    for name, r in g["regions"].items():
        lo, hi = r["tolerance_lsb_lo_hi"]
        hw, hh = r["half_w"], r["half_h"]
        d = np.array([img[y - hh:y + hh + 1, x - hw:x + hw + 1, :3].reshape(-1, 3).astype(float).mean(0) - np.array(c) for x, y, *c in r["blocks_x_y_r_g_b"]])
        assert lo <= d.min() and d.max() <= hi, f"{name}: block means differ from the reference PNG by {d.min():.2f} .. {d.max():.2f} LSB"
        if "max_abs_mean" in r:
            assert np.abs(d.mean(0)).max() <= r["max_abs_mean"], f"{name}: biased against the reference PNG by {d.mean(0)} LSB"


def test_scene_too_large_for_shared_memory(ctx, capi, oracle, scene_factory):
    """16 k spheres (grid -63..=63): the filter table (257 KB) fits no CTA's shared memory, the scan streams it from global
    memory (L1/L2) — same code, third launch configuration.  Closest hits and a tiny frame against the oracle."""
    arrays, sc = scene_factory(seed=5, half_extent=63)
    assert sc.n > 15_000
    ctx.upload_scene(**arrays)
    rng = np.random.default_rng(2)
    n = 4000
    k = rng.integers(1, sc.n, n)
    u = rng.normal(size=(n, 3)); u[:, 1] = np.abs(u[:, 1]) + 0.05; u /= np.linalg.norm(u, axis=1, keepdims=True)
    o = np.asarray(arrays["center"])[k] + u * rng.uniform(1, 60, (n, 1)); d = -u + rng.normal(size=(n, 3)) * 0.02
    o32, d32 = o.astype(np.float32).astype(np.float64), d.astype(np.float32).astype(np.float64)
    ref = oracle.world_hit_batch(sc, o32, d32)
    got = ctx.hitlist_batch(o32, d32, 1e-4)
    want = np.where(ref["hit"] == 1, ref["index"], -1)
    assert (got["index"] == want).mean() > 0.995 and (want > 0).mean() > 0.25
    W, H, spp = 96, 54, 2
    ref_img, _, cnt = oracle.render(sc, final_camera(oracle, W / H), W, H, spp, seed=8, sampler=oracle.SAMPLER_DIRECT)
    img, st = render_gpu(ctx, capi, final_camera(capi, W / H), width=W, height=H, spp=spp, seed=8)
    diff = np.abs(img[..., :3].astype(int) - ref_img[..., :3].astype(int)).max(axis=2)
    assert (diff <= 1).mean() > 0.99
    assert abs(st["rays_traced"] / cnt["rays"] - 1) < 1e-2


@pytest.mark.parametrize("prec", [0, 1])
def test_progressive_passes_are_prefixes_of_the_frame(ctx_final, capi, prec):
    """rtiow_render_progressive (SURVEY §8f #4: the per-pass preview that stands in for main.rs:120-124,151-171): the
    accumulators are integer sums over (pixel, sample) keys, so the frame after k passes is BIT-IDENTICAL to rtiow_render with
    spp = samples done, the last one to the full render; stats add up; a callback returning true cancels."""
    cam = final_camera(capi, 16 / 9)
    kw = dict(width=320, height=180, seed=3, precision=prec)
    spp, passes = 13, 4                                                   # uneven slices: 3, 3, 3, 4
    full, st_full = ctx_final.render(cam, capi.default_params(spp=spp, **kw))
    seen = []
    def on_pass(k, n, done, frame):
        seen.append((k, n, done, frame.copy()))
        return False
    img, st = ctx_final.render_progressive(cam, capi.default_params(spp=spp, **kw), passes, on_pass)
    assert [(k, n, d) for k, n, d, _ in seen] == [(1, 4, 3), (2, 4, 6), (3, 4, 9), (4, 4, 13)]
    assert np.array_equal(img, full) and np.array_equal(seen[-1][3], full)
    assert st["rays_traced"] == st_full["rays_traced"] and st["paths"] == st_full["paths"] and st["kernel_launches"] == 2 * passes
    for k, n, done, frame in seen[:-1]:
        part, _ = ctx_final.render(cam, capi.default_params(spp=done, **kw))
        assert np.array_equal(frame, part), f"preview after pass {k} differs from a {done}-spp render"
    # more passes than samples: clamped to one sample per pass; no callback at all is allowed
    img2, st2 = ctx_final.render_progressive(cam, capi.default_params(spp=2, **kw), 50)
    assert st2["kernel_launches"] == 4 and np.array_equal(img2, ctx_final.render(cam, capi.default_params(spp=2, **kw))[0])
    # cancel after the second pass: the error is reported, the buffer keeps the frame so far
    out = np.zeros((180, 320, 4), np.uint8)
    with pytest.raises(capi.RtiowError) as e:
        ctx_final.render_progressive(cam, capi.default_params(spp=spp, **kw), passes, lambda k, n, done, frame: k == 2, out=out)
    assert e.value.code == capi.ERR_CANCELLED and np.array_equal(out, seen[1][3])


@pytest.mark.parametrize("W,H,spp", [(1200, 675, 2), (400, 225, 10), (201, 133, 3)])
def test_tile_partition_invariance(ctx_final, capi, W, H, spp):
    """N-GPU image == 1-GPU image, bit for bit: ranks are emulated one after another on this GPU through the
    per-rank entry points the torchrun path uses (rtiow_render_tiles_device + rtiow_deinterleave_device, and
    rtiow_render_to_frame_device, whose epilogue stores into the whole frame)."""
    import torch
    cam = final_camera(capi, W / H)
    base, _ = ctx_final.render(cam, capi.default_params(width=W, height=H, spp=spp, seed=4))
    for world, tile_rows in [(2, 4), (8, 4), (8, 1), (3, 7), (4, 64)]:
        prm = capi.default_params(width=W, height=H, spp=spp, seed=4, tile_rows=tile_rows)
        nbytes = ctx_final.tile_buffer_bytes(prm, world)
        gathered = torch.zeros(world * nbytes, dtype=torch.uint8, device="cuda")
        rays = 0
        for rank in range(world):
            tiles = gathered[rank * nbytes:(rank + 1) * nbytes]
            st = ctx_final.render_tiles_device(cam, prm, rank, world, tiles.data_ptr(), 0, want_stats=True)
            rays += st["rays_traced"]
        frame = torch.empty(H * W * 4, dtype=torch.uint8, device="cuda")
        ctx_final.deinterleave_device(gathered.data_ptr(), prm, world, frame.data_ptr(), 0)
        torch.cuda.synchronize()
        got = frame.cpu().numpy().reshape(H, W, 4)
        assert np.array_equal(got, base), f"world={world} tile_rows={tile_rows}: image differs from the single-GPU image"
        # the gather fused into the epilogue (rtiow_render_to_frame_device): every rank stores straight into the whole frame
        frame2 = torch.zeros(H * W * 4, dtype=torch.uint8, device="cuda")
        rays2 = sum(ctx_final.render_to_frame_device(cam, prm, rank, world, frame2.data_ptr(), 0, want_stats=True)["rays_traced"] for rank in range(world))
        torch.cuda.synchronize()
        assert np.array_equal(frame2.cpu().numpy().reshape(H, W, 4), base) and rays2 == rays, f"world={world} tile_rows={tile_rows}: fused gather differs"


def test_full_size_properties_cfg2(ctx_final, capi, oracle, final_scene):
    """BASELINE configs[1] frame (1200x675) at reduced spp: top-down orientation, alpha, ray statistics, sky rows."""
    _, sc = final_scene
    W, H, spp = 1200, 675, 4
    img, st = render_gpu(ctx_final, capi, final_camera(capi, W / H), width=W, height=H, spp=spp, seed=1)
    assert img.shape == (H, W, 4) and (img[..., 3] == 255).all()
    assert st["paths"] == W * H * spp and 2.4 < st["rays_traced"] / st["paths"] < 2.9          # SURVEY: ~2.66 rays/path
    # top rows are sky: blue-ish, smooth; bottom rows are ground/spheres
    top = img[:20, :, :3].astype(float)
    assert top[..., 2].min() >= 254 and top.std(axis=1).max() < 1.5
    ref, _, _ = oracle.render(sc, final_camera(oracle, W / H), W, H, spp, seed=1, sampler=oracle.SAMPLER_DIRECT, rows=(0, 12))
    assert np.abs(img[:12, :, :3].astype(int) - ref[:12, :, :3].astype(int)).max() <= 1
    # a band through the middle of the frame against the oracle (same paths)
    ref_mid, _, _ = oracle.render(sc, final_camera(oracle, W / H), W, H, spp, seed=1, sampler=oracle.SAMPLER_DIRECT, rows=(400, 408))
    d = np.abs(img[400:408, :, :3].astype(int) - ref_mid[400:408, :, :3].astype(int)).max(axis=2)
    assert (d <= 1).mean() > 0.99


def test_empty_world_and_edge_params(ctx, capi, oracle):
    ctx.upload_scene(np.zeros((0, 3)), np.zeros(0), np.zeros(0, np.uint32), [0], [[1, 1, 1]], [0])
    cam = final_camera(capi, 1.5)
    img, st = render_gpu(ctx, capi, cam, width=64, height=43, spp=3, seed=1, alpha=7)
    assert st["rays_traced"] == 64 * 43 * 3 and (img[..., 3] == 7).all() and img[..., 2].min() == 255
    # max_depth 0: every path is black (main.rs:40-42), no ray is traced
    img0, st0 = render_gpu(ctx, capi, cam, width=64, height=43, spp=3, max_depth=0)
    assert st0["rays_traced"] == 0 and (img0[..., :3] == 0).all()
    # smallest legal frame, spp 1
    img1, _ = render_gpu(ctx, capi, cam, width=2, height=2, spp=1)
    assert img1.shape == (2, 2, 4)
    for bad in (dict(width=1), dict(height=1), dict(spp=0), dict(tile_rows=0), dict(precision=9)):
        with pytest.raises(capi.RtiowError) as e:
            render_gpu(ctx, capi, cam, **{**dict(width=8, height=8, spp=1), **bad})
        assert e.value.code == capi.ERR_INVALID_ARG


def test_unsupported_and_invalid_scene(ctx, capi):
    with pytest.raises(capi.RtiowError) as e:
        ctx.upload_scene([[0, 0, 0]], [1.0], [0], [3], [[1, 1, 1]], [0])          # unknown material kind: no CPU fallback
    assert e.value.code == capi.ERR_UNSUPPORTED
    with pytest.raises(capi.RtiowError) as e:
        ctx.upload_scene([[0, 0, 0]], [1.0], [5], [0], [[1, 1, 1]], [0])          # material index out of range
    assert e.value.code == capi.ERR_INVALID_ARG
    with pytest.raises(capi.RtiowError) as e:
        ctx.upload_scene([[np.nan, 0, 0]], [1.0], [0], [0], [[1, 1, 1]], [0])
    assert e.value.code == capi.ERR_INVALID_ARG
    # a non-finite field a sphere's material reads: the reference's pixel would be black, the render's would not
    for kind, albedo, param in ((1, [[1, np.nan, 1]], [0]), (0, [[1, 1, np.inf]], [0]), (1, [[1, 1, 1]], [np.nan]),
                                (2, [[1, 1, 1]], [-np.inf])):
        with pytest.raises(capi.RtiowError) as e:
            ctx.upload_scene([[0, 0, 0]], [1.0], [0], [kind], albedo, param)
        assert e.value.code == capi.ERR_INVALID_ARG
    # fields the material ignores (a Dielectric's albedo, a Lambertian's param) and materials no sphere uses may be anything
    ctx.upload_scene([[0, 0, 0], [3, 0, 0]], [1.0, 1.0], [0, 1], [2, 0, 1], [[np.nan] * 3, [1, 1, 1], [np.inf] * 3],
                     [1.5, np.nan, np.nan])
