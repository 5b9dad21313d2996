"""GPU suite: rtiow_render_adaptive, per-pixel sample counts driven by each pixel's own noise.

The rounds render sample ranges of shrinking pixel lists into the frame's own integer sums, keyed by (seed; pixel, sample,
bounce) like every other call (rt_render.cuh, Loop::Adaptive).  So:
  * every pixel that stopped at n samples equals rtiow_render(spp = n) byte for byte, on every scan arm;
  * min_spp == spp is rtiow_render, and tolerance = +inf is rtiow_render at spp = min_spp (bytes, paths and rays);
  * the call with spp = b_k is the first k + 1 rounds of a call with a larger spp (the rule, exactly);
  * counts, errors and rays equal an independent restatement: each pixel's camera rays rebuilt, their paths traced by
    rtiow_ray_color_batch, and S1, S2, the error and the rule in numpy (include/rtiow_cuda.h);
  * counts grow as the tolerance falls, and every output is identical across calls, contexts and GPU counts.
"""
import ctypes as C

import numpy as np
import pytest

import edge_scenes as es
import scan_scenes as ss
from test_render_aov_gpu import _cam_rays
from test_render_views_gpu import ARM_CASES, _wide_threads, orbit

pytestmark = pytest.mark.gpu
W, H = 48, 27


@pytest.fixture()
def ad_ctx(ctx, capi):
    yield ctx
    ctx.set_scan_backend(capi.SCAN_AUTO)


def boundaries(min_spp, spp):
    b = [min_spp]
    while b[-1] < spp:
        b.append(min(2 * b[-1], spp))
    return b


def check_exact(ctx, cam, prm, min_spp, tol, least_counts=1):
    """the adaptive frame against rtiow_render at every count it used, pixel by pixel; returns (img, maps, stats)"""
    img, maps, st = ctx.render_adaptive(cam, prm, min_spp, tol)
    n = maps["spp"]
    assert set(np.unique(n)) <= set(boundaries(min_spp, prm.spp)), np.unique(n)
    assert st["paths"] == int(n.astype(np.uint64).sum())
    counts = np.unique(n)
    assert len(counts) >= least_counts, f"only the counts {counts}"
    for k in counts:
        ref, _ = ctx.render(cam, capi_params(prm, spp=int(k)))
        mask = n == k
        bad = np.argwhere(mask & (img != ref).any(-1))
        assert len(bad) == 0, f"{len(bad)} pixels at {k} spp differ from rtiow_render(spp={k}), e.g. {tuple(bad[0])}"
    return img, maps, st


def capi_params(prm, **kw):
    from rtiow_b200 import capi
    fields = {k: getattr(prm, k) for k in ("width", "height", "spp", "max_depth", "t_min", "seed", "alpha", "precision", "tile_rows")}
    return capi.default_params(**{**fields, **kw})


def arm_setup(ctx, capi, name, backend, prec, arm, threads):
    arrays = ss.build(name, capi)
    b = {"auto": capi.SCAN_AUTO, "fp32": capi.SCAN_FP32}[backend]
    p = {"f32": capi.F32, "f64": capi.F64}[prec]
    assert ss.scan_arm(arrays, b, p)[0] == arm
    if threads:
        assert _wide_threads(arrays) == threads
    ctx.upload_scene(**arrays)
    ctx.set_scan_backend(b)
    if name.startswith("final"):
        cam = orbit(capi, 1)[0]
    else:
        R = ss.scene_info(arrays)["R"]
        cam = orbit(capi, 1, radius=3.0 * R, height=0.5 * R, fov=45.0)[0]
    return cam, p


@pytest.mark.parametrize("name,backend,prec,arm,threads", ARM_CASES, ids=[f"{c[3]}{c[4] or ''}-{c[0]}" for c in ARM_CASES])
def test_every_pixel_is_render_at_its_count(ad_ctx, capi, name, backend, prec, arm, threads):
    cam, p = arm_setup(ad_ctx, capi, name, backend, prec, arm, threads)
    min_spp, spp = (2, 16) if prec == "f64" else (4, 64)
    prm = capi.default_params(width=W, height=H, spp=spp, seed=3, precision=p)
    for tol in (4.0, 2.0, 1.0, 0.5, 0.25):          # the first tolerance that leaves pixels on three counts or more
        _, maps, _ = ad_ctx.render_adaptive(cam, prm, min_spp, tol)
        if len(np.unique(maps["spp"])) >= 3:
            break
    _, _, st = check_exact(ad_ctx, cam, prm, min_spp, tol, least_counts=3)
    assert st["scan_backend"] == (capi.SCAN_TENSOR if arm == "Tensor" else capi.SCAN_FP32)


def test_degenerate_calls_are_rtiow_render(ad_ctx, capi, final_scene):
    ad_ctx.upload_scene(**final_scene[0])
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=24, seed=6)
    ref, sr = ad_ctx.render(cam, prm)
    img, maps, st = ad_ctx.render_adaptive(cam, prm, 24, 0.0)
    assert np.array_equal(img, ref) and st["paths"] == sr["paths"] and st["rays_traced"] == sr["rays_traced"]
    assert (maps["spp"] == 24).all() and st["kernel_launches"] == 5 and st["kernel_ms"] > 0
    ref, sr = ad_ctx.render(cam, capi_params(prm, spp=5))
    img, maps, st = ad_ctx.render_adaptive(cam, prm, 5, float("inf"))
    assert np.array_equal(img, ref) and st["paths"] == sr["paths"] and st["rays_traced"] == sr["rays_traced"]
    assert (maps["spp"] == 5).all() and np.isfinite(maps["error"]).all()


def test_the_rule_by_truncation(ad_ctx, capi, final_scene):
    """spp = 16 is the first three rounds (4, 8, 16) of spp = 64"""
    ad_ctx.upload_scene(**final_scene[0])
    cam = orbit(capi, 1)[0]
    tol = 2.0
    _, mk, sk = ad_ctx.render_adaptive(cam, capi.default_params(width=W, height=H, spp=16, seed=8), 4, tol)
    _, mm, sm = ad_ctx.render_adaptive(cam, capi.default_params(width=W, height=H, spp=64, seed=8), 4, tol)
    early = mk["spp"] < 16
    assert early.any() and (~early).any()
    assert np.array_equal(mm["spp"][early], mk["spp"][early]) and mm["error"][early].tobytes() == mk["error"][early].tobytes()
    assert np.array_equal(mm["spp"][~early] > 16, mk["error"][~early] > tol)
    for m, top in ((mk, 16), (mm, 64)):
        assert ((m["spp"] >= 4) & (m["spp"] <= top)).all() and set(np.unique(m["spp"])) <= set(boundaries(4, top))
        stopped = m["spp"] < top
        assert (m["error"][stopped] <= tol).all()
    assert sm["rays_traced"] > sk["rays_traced"] and sm["paths"] > sk["paths"]


def _err(s1, s2, n):
    """the error of include/rtiow_cuda.h in IEEE double, each operation rounded on its own, then to float"""
    n = np.asarray(n, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        m = (s1.astype(np.float64) * 2.0 ** -32) / n
        q = (s2.astype(np.float64) * 2.0 ** -32) / n
        var = np.maximum(0.0, q - m * m)
        e = 128.0 * np.sqrt(var / ((n - 1.0) * np.maximum(m, 2.0 ** -16)))
    return np.where(n <= 1, np.inf, e).astype(np.float32)


INDEPENDENT = [("final", "auto", 2.0), ("final", "fp32", 2.0), ("final", "f64", 2.0), ("bright", "auto", 1.0)]


@pytest.mark.parametrize("scene,arm,tol", INDEPENDENT, ids=[f"{c[0]}-{c[1]}" for c in INDEPENDENT])
def test_the_rule_against_an_independent_restatement(ad_ctx, capi, final_scene, scene, arm, tol):
    w, h, min_spp, spp = 24, 14, 2, 32
    if scene == "final":
        arrays = final_scene[0]
        cam = orbit(capi, 1, aspect=w / h)[0]
    else:
        arrays = es.build(scene)
        cam = es.camera(capi, scene, dict(W=w, H=h))
    prec = capi.F64 if arm == "f64" else capi.F32
    ad_ctx.upload_scene(**arrays)
    ad_ctx.set_scan_backend(capi.SCAN_FP32 if arm == "fp32" else capi.SCAN_AUTO)
    prm = capi.default_params(width=w, height=h, spp=spp, seed=5, precision=prec)
    _, got, st = ad_ctx.render_adaptive(cam, prm, min_spp, tol)

    o, d = _cam_rays(ad_ctx, capi, cam, prm, prec)                         # every sample [0, spp) of every pixel
    y_, x_, s_ = np.meshgrid(np.arange(h), np.arange(w), np.arange(spp), indexing="ij")
    key = ((h - 1 - y_) * w + x_).ravel().astype(np.uint32)
    pc = ad_ctx.ray_color_batch(o.reshape(-1, 3), d.reshape(-1, 3), key, s_.ravel().astype(np.uint32), prm.seed, prm.max_depth,
                                prm.t_min, precision=prec)
    ft = np.float32 if prec == capi.F32 else np.float64
    col = pc["color"].astype(ft)
    y = (col[:, 0] + col[:, 1] + col[:, 2]) / ft(3)
    y = np.where(y > 0, np.where(y < 1, y, ft(1)), ft(0)).astype(ft)
    fix = lambda v: np.rint(v.astype(np.float64) * 2.0 ** 32).astype(np.uint64)          # noqa: E731
    s1 = np.cumsum(fix(y).reshape(h, w, spp), axis=2, dtype=np.uint64)
    s2 = np.cumsum(fix((y * y).astype(ft)).reshape(h, w, spp), axis=2, dtype=np.uint64)
    rays = np.cumsum(pc["rays"].astype(np.int64).reshape(h, w, spp), axis=2)

    n = got["spp"].astype(np.int64)
    at = lambda a, k: np.take_along_axis(a, (k - 1)[..., None], 2)[..., 0]             # noqa: E731
    err_n = _err(at(s1, n), at(s2, n), n)
    with np.errstate(invalid="ignore"):
        agree = (err_n == got["error"]) | (np.abs(err_n - got["error"]) <= 1e-4 * np.abs(err_n))
    assert (~agree).sum() <= max(2, agree.size // 100), f"{(~agree).sum()} of {agree.size} pixels' errors differ"
    # the stop decision at every boundary the pixel reached, where the error is clear of the tolerance
    for b in boundaries(min_spp, spp):
        reached = agree & (n >= b)
        e = _err(at(s1, np.full_like(n, b)), at(s2, np.full_like(n, b)), b)
        clear = np.abs(e.astype(np.float64) - tol) > 1e-4 * max(tol, 1.0)
        went_on = n > b
        want = (e.astype(np.float64) > tol) & (b < spp)
        bad = reached & clear & (went_on != want)
        assert not bad.any(), f"{bad.sum()} pixels decided otherwise at {b} spp"
    # the separately compiled kernels agree on all but ~1e-5 of the rays; on a frame this small one path that parts ways moves
    # the count by up to max_depth rays
    want_rays = int(at(rays, n).sum())
    assert abs(st["rays_traced"] - want_rays) <= max(prm.max_depth, 1e-3 * want_rays), (st["rays_traced"], want_rays)


def test_counts_grow_as_the_tolerance_falls(ad_ctx, capi, final_scene):
    ad_ctx.upload_scene(**final_scene[0])
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=64, seed=2)
    prev = None
    for tol in (8.0, 4.0, 2.0, 1.0, 0.5):
        _, m, _ = ad_ctx.render_adaptive(cam, prm, 4, tol)
        if prev is not None:
            assert (m["spp"] >= prev).all()
        prev = m["spp"]


def test_deterministic_across_calls_and_contexts(ad_ctx, capi, final_scene):
    ad_ctx.upload_scene(**final_scene[0])
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=140, seed=9)      # chunks of 64 + a remainder in the last rounds
    a = ad_ctx.render_adaptive(cam, prm, 3, 1.5)
    b = ad_ctx.render_adaptive(cam, prm, 3, 1.5)
    with capi.Context(device=0) as c:
        c.upload_scene(**final_scene[0])
        c_ = c.render_adaptive(cam, prm, 3, 1.5)
    for r in (b, c_):
        assert np.array_equal(r[0], a[0]) and r[2]["rays_traced"] == a[2]["rays_traced"] and r[2]["paths"] == a[2]["paths"]
        for k in ("spp", "error"):
            assert r[1][k].tobytes() == a[1][k].tobytes(), k


def test_multi_gpu_matches_one_device(capi, final_scene):
    n = capi.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    cam = orbit(capi, 1)[0]
    with capi.Context(1) as c1:
        c1.upload_scene(**final_scene[0])
        base = {tr: c1.render_adaptive(cam, capi.default_params(width=W, height=H, spp=64, seed=9, tile_rows=tr), 4, 1.0) for tr in (1, 5, H)}
    with capi.Context(n) as cn:
        cn.upload_scene(**final_scene[0])
        for tr, (img1, m1, s1) in base.items():
            img, m, st = cn.render_adaptive(cam, capi.default_params(width=W, height=H, spp=64, seed=9, tile_rows=tr), 4, 1.0)
            assert np.array_equal(img, img1) and st["rays_traced"] == s1["rays_traced"] and st["paths"] == s1["paths"] and st["n_gpus"] == n
            for k in ("spp", "error"):
                assert m[k].tobytes() == m1[k].tobytes(), (tr, k)


@pytest.mark.parametrize("missing", ["spp_map", "error_map", "both"])
def test_each_map_may_be_null(ad_ctx, capi, final_scene, missing):
    ad_ctx.upload_scene(**final_scene[0])
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=32, seed=2)
    ref_img, full, _ = ad_ctx.render_adaptive(cam, prm, 4, 2.0)
    off = {"spp_map": False, "error_map": False} if missing == "both" else {missing: False}
    img, part, _ = ad_ctx.render_adaptive(cam, prm, 4, 2.0, **off)
    assert np.array_equal(img, ref_img)
    assert set(part) == {"spp", "error"} - {k.split("_")[0] for k in off}
    for k in part:
        assert part[k].tobytes() == full[k].tobytes(), k
    mine = {"spp_map": np.zeros(W * H, np.uint32), "error_map": np.full(W * H, np.nan, np.float32)}
    _, got, _ = ad_ctx.render_adaptive(cam, prm, 4, 2.0, **mine)
    assert np.shares_memory(got["spp"], mine["spp_map"]) and got["spp"].tobytes() == full["spp"].tobytes()
    assert np.shares_memory(got["error"], mine["error_map"]) and got["error"].tobytes() == full["error"].tobytes()


EDGES = {"2x2": dict(width=2, height=2, spp=64), "depth1": dict(max_depth=1), "depth50": dict(max_depth=50),
         "min-spp-1": dict(min_spp=1)}


@pytest.mark.parametrize("case", list(EDGES))
def test_edges(ad_ctx, capi, final_scene, case):
    ad_ctx.upload_scene(**final_scene[0])
    e = {**dict(width=W, height=H, spp=32, seed=4, min_spp=4), **EDGES[case]}
    min_spp = e.pop("min_spp")
    prm = capi.default_params(**e)
    cam = orbit(capi, 1, aspect=prm.width / prm.height)[0]
    _, maps, _ = check_exact(ad_ctx, cam, prm, min_spp, 1.0)
    if case == "min-spp-1":                      # one sample has no error estimate: every pixel goes on to 2
        assert (maps["spp"] >= 2).all()


@pytest.mark.parametrize("scene", ["bright", "shells", "glass-inside"])
def test_edge_scenes(ad_ctx, capi, scene):
    ad_ctx.upload_scene(**es.build(scene))
    cam = es.camera(capi, scene, dict(W=W, H=H))
    prm = capi.default_params(width=W, height=H, spp=64, seed=7)
    check_exact(ad_ctx, cam, prm, 4, 2.0)


def test_max_depth_zero(ad_ctx, capi, final_scene):
    """no ray is traced, so S1 = S2 = 0: every pixel stops at the first boundary of two samples or more, with error 0"""
    ad_ctx.upload_scene(**final_scene[0])
    cam = orbit(capi, 1)[0]
    for min_spp, spp, n_want in ((4, 32, 4), (1, 32, 2), (1, 1, 1), (8, 8, 8)):
        prm = capi.default_params(width=W, height=H, spp=spp, seed=4, max_depth=0)
        img, maps, st = ad_ctx.render_adaptive(cam, prm, min_spp, 0.5)
        assert st["rays_traced"] == 0 and not img[..., :3].any() and (maps["spp"] == n_want).all()
        assert (np.isinf(maps["error"]) if n_want == 1 else (maps["error"] == 0)).all()


@pytest.mark.parametrize("tol", [0.0, 0.05])
def test_saturating_counts(ad_ctx, capi, final_scene, tol):
    """a 2x2 frame up to 70 000 spp (spp > 65535 accumulates with add_saturating): every pixel still equals rtiow_render at its
    count"""
    ad_ctx.upload_scene(**final_scene[0])
    prm = capi.default_params(width=2, height=2, spp=70000, seed=4)
    cam = orbit(capi, 1, aspect=1.0)[0]
    _, maps, _ = check_exact(ad_ctx, cam, prm, 16384, tol)
    if tol == 0.0:
        assert (maps["spp"] == 70000).all()


def test_errors(ad_ctx, capi, final_scene):
    ad_ctx.upload_scene(**final_scene[0])
    prm = capi.default_params(width=W, height=H, spp=8)
    cam = orbit(capi, 1)[0]
    L = capi.lib()
    out = np.zeros((H, W, 4), np.uint8)
    st = capi.Stats()
    call = lambda h, c, m, t, o: L.rtiow_render_adaptive(h, c, C.byref(prm), m, t, o, None, None, C.byref(st))    # noqa: E731
    good = (ad_ctx._h, C.byref(cam), 2, 1.0, out.ctypes.data_as(C.c_void_p))
    assert call(*good) == capi.OK
    for bad in ((None,) + good[1:], (good[0], None) + good[2:], good[:4] + (None,), good[:2] + (0,) + good[3:], good[:2] + (9,) + good[3:],
                good[:3] + (float("nan"),) + good[4:], good[:3] + (-1.0,) + good[4:]):
        assert call(*bad) == capi.ERR_INVALID_ARG
    with pytest.raises(capi.RtiowError) as e:
        ad_ctx.render_adaptive(cam, capi.default_params(width=1, height=H, spp=4), 1, 1.0)
    assert e.value.code == capi.ERR_INVALID_ARG
    with capi.Context(1) as c:                                             # no scene
        with pytest.raises(capi.RtiowError) as e:
            c.render_adaptive(cam, prm, 2, 1.0)
        assert e.value.code == capi.ERR_INVALID_ARG
