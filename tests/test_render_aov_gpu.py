"""GPU suite: rtiow_render_aov, a frame byte-identical to rtiow_render plus float AOVs for a denoiser.

The render kernel is the frame's loop as Loop::Aov (rt_render.cuh): a camera ray also adds its first hit to integer
accumulators, and finalize_aov_kernel turns them into float buffers.  So:
  * the RGBA8 frame and rays_traced equal rtiow_render's on every scan arm, with the float buffers set and with them NULL;
  * the linear colour quantises to the frame (to_rgba, vec3.rs:404-420) except next to a quantisation step;
  * albedo, normal and depth equal an independent restatement: every camera ray rebuilt from rtiow_sampler_batch (bounce 0)
    and rtiow_get_ray_batch, its first hit from rtiow_hitlist_batch on the same arm, and the fixed-point means in numpy;
  * every buffer is bit-identical across calls, contexts and GPU counts (integer sums).
"""
import numpy as np
import pytest

import edge_scenes as es
import np_restatement as nr
import scan_scenes as ss
from test_render_views_gpu import ARM_CASES, _wide_threads, orbit

pytestmark = pytest.mark.gpu
W, H, SPP = 96, 54, 4
AOVS = ("color", "albedo", "normal", "depth")


@pytest.fixture()
def aov_ctx(ctx, capi):
    yield ctx
    ctx.set_scan_backend(capi.SCAN_AUTO)


def colour_mismatches(img, color, spp):
    """pixels where to_rgba of color * spp differs from the frame, and how many of them are NOT within float rounding of a
    quantisation step (those would be a real disagreement)"""
    c64 = color.astype(np.float64)
    q = nr.to_rgba(c64 * spp, 255, spp)
    off = (q[..., :3] != img[..., :3]).any(-1)
    v = 256.0 * np.sqrt(np.clip(c64, 0.0, 0.999))
    near_step = (np.abs(v - np.round(v)) < 1e-4 * np.maximum(v, 1.0)).any(-1)
    return int(off.sum()), int((off & ~near_step).sum())


def check_frame(ctx, cam, prm):
    """render_aov against render: same bytes, same rays, with every float buffer and with none; returns the AOVs"""
    ref, sr = ctx.render(cam, prm)
    img, bufs, st = ctx.render_aov(cam, prm)
    assert np.array_equal(img, ref), "render_aov's frame differs from rtiow_render's"
    assert st["rays_traced"] == sr["rays_traced"] and st["paths"] == sr["paths"] and st["scan_backend"] == sr["scan_backend"]
    assert st["kernel_launches"] == sr["kernel_launches"] + 1
    n = prm.width * prm.height
    assert st["d2h_bytes"] == sr["d2h_bytes"] + 4 * 10 * n
    img0, none, s0 = ctx.render_aov(cam, prm, color=False, albedo=False, normal=False, depth=False)
    assert none == {} and np.array_equal(img0, ref) and s0["rays_traced"] == sr["rays_traced"]
    assert set(bufs) == set(AOVS)
    assert bufs["color"].shape == bufs["albedo"].shape == bufs["normal"].shape == (prm.height, prm.width, 3)
    assert bufs["depth"].shape == (prm.height, prm.width)
    return img, bufs, st


@pytest.mark.parametrize("name,backend,prec,arm,threads", ARM_CASES, ids=[f"{c[3]}{c[4] or ''}-{c[0]}" for c in ARM_CASES])
def test_frame_unchanged_on_every_arm(aov_ctx, capi, name, backend, prec, arm, threads):
    arrays = ss.build(name, capi)
    b = {"auto": capi.SCAN_AUTO, "fp32": capi.SCAN_FP32}[backend]
    p = {"f32": capi.F32, "f64": capi.F64}[prec]
    assert ss.scan_arm(arrays, b, p)[0] == arm
    if threads:
        assert _wide_threads(arrays) == threads
    aov_ctx.upload_scene(**arrays)
    aov_ctx.set_scan_backend(b)
    if name.startswith("final"):
        cam = orbit(capi, 1)[0]
    else:
        R = ss.scene_info(arrays)["R"]
        cam = orbit(capi, 1, radius=3.0 * R, height=0.5 * R, fov=45.0)[0]
    spp = 2 if prec == "f64" else SPP
    prm = capi.default_params(width=W, height=H, spp=spp, seed=3, precision=p)
    img, bufs, st = check_frame(aov_ctx, cam, prm)
    assert st["scan_backend"] == (capi.SCAN_TENSOR if arm == "Tensor" else capi.SCAN_FP32)
    off, real = colour_mismatches(img, bufs["color"], spp)
    assert real == 0 and off <= max(2, img.shape[0] * img.shape[1] // 500), (off, real)
    hit = np.isfinite(bufs["depth"])
    assert hit.any() and (bufs["depth"][hit] > 0).all()
    assert (bufs["albedo"] >= 0).all() and (bufs["albedo"] <= 1).all()
    assert (np.abs(bufs["normal"]) <= 1 + 1e-5).all() and not bufs["normal"][~hit].any()


# ------------------------------------------------------------------------------------------------ the independent path
def _cam_rays(ctx, capi, cam, prm, prec):
    """every camera ray of the frame as the kernel builds it (rt_render.cuh, next_ray): the bounce-0 sampler event of
    (pixel key, sample), the jittered (s, t) in the render's precision, and Camera::get_ray.  -> (orig, dir) [H, W, spp, 3]"""
    w, h, spp = prm.width, prm.height, prm.spp
    ft = np.float32 if prec == capi.F32 else np.float64
    y, x, s = np.meshgrid(np.arange(h), np.arange(w), np.arange(spp), indexing="ij")
    j = (h - 1 - y).ravel()                                                   # bottom-up row (main.rs:132,141-145)
    key = (j * w + x.ravel()).astype(np.uint32)
    u = ctx.sampler_batch(key, s.ravel().astype(np.uint32), np.zeros(key.size, np.uint32), prm.seed, precision=prec)
    su = ((x.ravel().astype(ft) + u[:, 0].astype(ft)) * ft(1.0 / (w - 1))).astype(np.float64)
    sv = ((j.astype(ft) + u[:, 1].astype(ft)) * ft(1.0 / (h - 1))).astype(np.float64)
    r = ctx.get_ray_batch(cam, su, sv, u[:, 4:6], precision=prec)
    return r["orig"].reshape(h, w, spp, 3), r["dir"].reshape(h, w, spp, 3)


def _restate(ctx, capi, arrays, cam, prm, prec):
    """the AOVs of the rebuilt camera rays through rtiow_hitlist_batch, with the kernel's fixed-point sums (AovArgs) in numpy
    -> (albedo, normal, depth, robust[H, W]: every sample of the pixel is a robust hit with the index the scan found)"""
    o, d = _cam_rays(ctx, capi, cam, prm, prec)
    h, w, spp = prm.height, prm.width, prm.spp
    o2, d2 = o.reshape(-1, 3), d.reshape(-1, 3)
    hl = ctx.hitlist_batch(o2, d2, prm.t_min, precision=prec)
    idx = hl["index"]
    hit = idx >= 0
    ft = np.float32 if prec == capi.F32 else np.float64
    mi = np.asarray(arrays["mat_index"])[np.maximum(idx, 0)]
    alb = np.asarray(arrays["mat_albedo"], float)[mi].astype(ft).astype(np.float64)
    alb[np.asarray(arrays["mat_kind"])[mi] == capi.MAT_DIELECTRIC] = 1.0
    alb = np.where(hit[:, None], alb, nr.sky(d2))
    fix = lambda v, hi, scale: np.rint(np.clip(v, 0.0, hi) * scale).astype(np.uint64)      # noqa: E731
    a_sum = fix(alb, 1.0, 2.0 ** 32).reshape(h, w, spp, 3).sum(2)
    n_fix = np.where(hit[:, None], fix(hl["normal"] + 1.0, 2.0, 2.0 ** 31), 0).reshape(h, w, spp, 3).sum(2)
    dist = hl["t"] * np.linalg.norm(d2, axis=1)
    d_sum = np.where(hit, fix(dist, 65536.0, 2.0 ** 16), 0).reshape(h, w, spp).sum(2)
    hits = hit.reshape(h, w, spp).sum(2)
    inv = (1.0 / spp) / 2.0 ** 32
    albedo = (a_sum.astype(np.float64) * inv).astype(np.float32)
    normal = ((n_fix.astype(np.int64) - (hits.astype(np.int64) << 31)[..., None]).astype(np.float64) * ((1.0 / spp) / 2.0 ** 31)).astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        depth = np.where(hits > 0, d_sum.astype(np.float64) / (65536.0 * hits), np.inf).astype(np.float32)
    rb = ss.robust_closest(arrays, o2, d2, prm.t_min)
    robust = (rb["robust"] & (rb["index"] == idx)).reshape(h, w, spp).all(2)
    return dict(albedo=albedo, normal=normal, depth=depth, robust=robust, all_miss=(hits == 0))


SKY_VIEW = ((13.0, 2.0, 3.0), (13.0, 40.0, 40.0), (0.0, 1.0, 0.0), 20.0, 0.0, 10.0)      # the final scene, looking up: sky only
INDEPENDENT = [("final", "auto", s) for s in (1, 3, 70)] + [("final", "fp32", 3), ("final", "f64", 3),
                                                            ("shells", "auto", 3), ("glass-inside", "auto", 3), ("sky", "auto", 3)]


@pytest.mark.parametrize("scene,arm,spp", INDEPENDENT, ids=[f"{c[0]}-{c[1]}-spp{c[2]}" for c in INDEPENDENT])
def test_aovs_match_an_independent_path(aov_ctx, capi, scene, arm, spp):
    """Albedo equals the restatement exactly on every pixel whose samples are all robust hits.  The rebuilt ray is not bit
    for bit the kernel's (hitlist_batch normalises with a division, the render with rsqrtf; the lens sample comes from the
    sampler's direct_disk), so normal and depth match within 2e-4 and 1e-5 relative + 2^-16 there, and elsewhere on all but
    a few pixels (a sample can change its hit on a knife edge)."""
    w, h = 32, 18
    if scene == "sky":
        arrays = ss.build("final", capi)
        cam = capi.camera_new(*SKY_VIEW[:4], w / h, *SKY_VIEW[4:])
    elif scene == "final":
        arrays = ss.build("final", capi)
        cam = orbit(capi, 1, aspect=w / h)[0]
    else:
        arrays = es.build(scene)
        cam = es.camera(capi, scene, dict(W=w, H=h))
    prec = capi.F64 if arm == "f64" else capi.F32
    aov_ctx.upload_scene(**arrays)
    aov_ctx.set_scan_backend(capi.SCAN_FP32 if arm == "fp32" else capi.SCAN_AUTO)
    prm = capi.default_params(width=w, height=h, spp=spp, seed=5, precision=prec)
    img, got, st = check_frame(aov_ctx, cam, prm)
    ref = _restate(aov_ctx, capi, arrays, cam, prm, prec)
    rob = ref["robust"]
    if scene == "sky":
        assert ref["all_miss"].all() and np.isinf(got["depth"]).all() and not got["normal"].any()
        assert np.abs(got["albedo"] - ref["albedo"]).max() <= 1e-6
        return
    assert rob.mean() > 0.5, f"only {rob.mean():.1%} robust pixels"
    bad = np.argwhere(rob & (got["albedo"] != ref["albedo"]).any(-1))
    assert len(bad) == 0, f"{len(bad)} robust pixels' albedo differ, e.g. {tuple(bad[0])}: {got['albedo'][tuple(bad[0])]} vs {ref['albedo'][tuple(bad[0])]}"
    dn = np.abs(got["normal"] - ref["normal"]).max(-1)
    with np.errstate(invalid="ignore"):
        dd = np.where(np.isinf(ref["depth"]) & np.isinf(got["depth"]), 0.0, np.abs(got["depth"] - ref["depth"]) / np.maximum(ref["depth"], 1e-3))
    assert (np.isinf(got["depth"]) == ref["all_miss"])[rob].all()
    assert dn[rob].max() <= 2e-4 and dd[rob].max() <= 1e-5 + 2.0 ** -16, (dn[rob].max(), dd[rob].max())
    others = (np.abs(got["albedo"] - ref["albedo"]).max(-1) > 1e-5) | (dn > 2e-4) | ~(dd <= 1e-5 + 2.0 ** -16)
    assert others.sum() <= max(2, others.size // 50), f"{others.sum()} of {others.size} pixels differ beyond the tolerances"


# ------------------------------------------------------------------------------------------------ determinism and edges
def test_deterministic_across_calls_and_contexts(aov_ctx, capi, final_scene):
    aov_ctx.upload_scene(**final_scene[0])
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=70, seed=9)            # chunks of 64 + 6 samples
    _, a, _ = aov_ctx.render_aov(cam, prm)
    _, b, _ = aov_ctx.render_aov(cam, prm)
    with capi.Context(device=0) as c:
        c.upload_scene(**final_scene[0])
        _, c_, _ = c.render_aov(cam, prm)
    for k in AOVS:
        assert a[k].tobytes() == b[k].tobytes() == c_[k].tobytes(), k


def test_multi_gpu_matches_one_device(capi, final_scene):
    n = capi.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    cam = orbit(capi, 1)[0]
    with capi.Context(1) as c1:
        c1.upload_scene(**final_scene[0])
        base = {tr: c1.render_aov(cam, capi.default_params(width=W, height=H, spp=SPP, seed=9, tile_rows=tr)) for tr in (1, 5, H)}
    with capi.Context(n) as cn:
        cn.upload_scene(**final_scene[0])
        for tr, (img1, a1, s1) in base.items():
            img, a, st = cn.render_aov(cam, capi.default_params(width=W, height=H, spp=SPP, seed=9, tile_rows=tr))
            assert np.array_equal(img, img1) and st["rays_traced"] == s1["rays_traced"] and st["n_gpus"] == n
            for k in AOVS:
                assert a[k].tobytes() == a1[k].tobytes(), (tr, k)


@pytest.mark.parametrize("missing", AOVS)
def test_each_buffer_may_be_null(aov_ctx, capi, final_scene, missing):
    aov_ctx.upload_scene(**final_scene[0])
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=2)
    ref_img, full, _ = aov_ctx.render_aov(cam, prm)
    img, part, _ = aov_ctx.render_aov(cam, prm, **{missing: False})
    assert np.array_equal(img, ref_img) and set(part) == set(AOVS) - {missing}
    for k in part:
        assert part[k].tobytes() == full[k].tobytes(), k
    only, one, _ = aov_ctx.render_aov(cam, prm, **{k: k == missing for k in AOVS})
    assert np.array_equal(only, ref_img) and one[missing].tobytes() == full[missing].tobytes()


def test_caller_arrays_receive_the_buffers(aov_ctx, capi, final_scene):
    aov_ctx.upload_scene(**final_scene[0])
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=2)
    _, full, _ = aov_ctx.render_aov(cam, prm)
    mine = {k: np.full(H * W * (1 if k == "depth" else 3), np.nan, np.float32) for k in AOVS}
    _, got, _ = aov_ctx.render_aov(cam, prm, **mine)
    for k in AOVS:
        assert np.shares_memory(got[k], mine[k]) and got[k].tobytes() == full[k].tobytes()


EDGES = {"2x2": dict(width=2, height=2), "depth1": dict(max_depth=1), "depth50": dict(max_depth=50),
         "spp70000": dict(width=4, height=3, spp=70000)}


@pytest.mark.parametrize("case", list(EDGES))
def test_edges(aov_ctx, capi, final_scene, case):
    aov_ctx.upload_scene(**final_scene[0])
    e = {**dict(width=W, height=H, spp=SPP, seed=4), **EDGES[case]}
    prm = capi.default_params(**e)
    cam = orbit(capi, 1, aspect=prm.width / prm.height)[0]
    img, bufs, _ = check_frame(aov_ctx, cam, prm)
    off, real = colour_mismatches(img, bufs["color"], prm.spp)
    assert real == 0 and off <= 2
    if case == "depth1":        # one ray per path: a hit ends black, a miss adds its sky value, which is also its albedo
        miss = np.isinf(bufs["depth"])
        assert miss.any() and np.array_equal(bufs["color"][miss], bufs["albedo"][miss])
    if case == "spp70000":      # sums past 2^32 saturate for colour (add_saturating); the AOVs cannot wrap
        assert (bufs["albedo"] <= 1).all() and np.isfinite(bufs["color"]).all()


def test_max_depth_zero_traces_nothing(aov_ctx, capi, final_scene):
    aov_ctx.upload_scene(**final_scene[0])
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=4, max_depth=0)
    img, bufs, st = check_frame(aov_ctx, orbit(capi, 1)[0], prm)
    assert st["rays_traced"] == 0 and not img[..., :3].any()
    assert not bufs["color"].any() and not bufs["albedo"].any() and not bufs["normal"].any() and np.isinf(bufs["depth"]).all()


def test_rank_ctx_of_world_one_renders(capi, final_scene):
    with capi.Context(device=0, rank=0, world=1) as c:
        c.upload_scene(**final_scene[0])
        check_frame(c, orbit(capi, 1)[0], capi.default_params(width=W, height=H, spp=SPP, seed=8))


def test_errors(aov_ctx, capi, final_scene):
    import ctypes as C
    aov_ctx.upload_scene(**final_scene[0])
    prm = capi.default_params(width=W, height=H, spp=1)
    cam = orbit(capi, 1)[0]
    st = capi.Stats()
    assert capi.lib().rtiow_render_aov(aov_ctx._h, C.byref(cam), C.byref(prm), None, None, None, None, None, C.byref(st)) == capi.ERR_INVALID_ARG
    with pytest.raises(capi.RtiowError) as e:
        aov_ctx.render_aov(cam, capi.default_params(width=1, height=H, spp=1))
    assert e.value.code == capi.ERR_INVALID_ARG
    with capi.Context(1) as c:                                             # no scene
        with pytest.raises(capi.RtiowError) as e:
            c.render_aov(cam, prm)
        assert e.value.code == capi.ERR_INVALID_ARG
