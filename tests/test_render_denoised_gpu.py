"""GPU suite for rtiow_render_denoised: rtiow_render_aov's render and rtiow_denoise's filter in one call, the AOVs kept on the device.

The call runs no kernel of its own: the Loop::Aov render and its epilogues, then the three denoise kernels, on the same buffers
in the same order as the two calls.  So out_color must equal ctx.denoise over ctx.render_aov's buffers bit for bit and out_rgba
byte for byte, on every scan arm, at every edge of the render and of the filter, across calls that resize the ctx's buffers,
and on an n-GPU ctx (whose devices copy their rows to device 0 before the filter).
"""
import ctypes as C

import numpy as np
import pytest

import edge_scenes as es
import np_denoise
import scan_scenes as ss
from test_render_views_gpu import ARM_CASES, _wide_threads, orbit

pytestmark = pytest.mark.gpu
W, H, SPP = 96, 54, 4
INF = float("inf")
SKY_VIEW = ((13.0, 2.0, 3.0), (13.0, 40.0, 40.0), (0.0, 1.0, 0.0), 20.0, 0.0, 10.0)      # the final scene, looking up: sky only


@pytest.fixture()
def dn_ctx(ctx, capi):
    yield ctx
    ctx.set_scan_backend(capi.SCAN_AUTO)


def _dp(capi, **kw):
    return capi.default_denoise_params(**kw)


def two_call(ctx, cam, prm, dp):
    """rtiow_render_aov, then rtiow_denoise over its four buffers -> (outputs, AOVs, render_aov's stats)"""
    _, b, sa = ctx.render_aov(cam, prm)
    outs, _ = ctx.denoise(b["color"], b["albedo"], b["normal"], b["depth"], dp)
    return outs, b, sa


def assert_same(got, ref, what=""):
    assert got["color"].view(np.uint32).tobytes() == ref["color"].view(np.uint32).tobytes(), \
        f"{what}: {int((got['color'].view(np.uint32) != ref['color'].view(np.uint32)).sum())} colour values differ"
    assert np.array_equal(got["rgba"], ref["rgba"]), f"{what}: {int((got['rgba'] != ref['rgba']).any(-1).sum())} pixels differ"


def check(ctx, capi, cam, prm, dp=None):
    """render_denoised against the two-call sequence: both outputs, and the render's paths, rays and scan backend"""
    dp = dp if dp is not None else _dp(capi)
    got, st = ctx.render_denoised(cam, prm, dp)
    ref, b, sa = two_call(ctx, cam, prm, dp)
    assert_same(got, ref)
    assert st["rays_traced"] == sa["rays_traced"] and st["paths"] == sa["paths"] and st["scan_backend"] == sa["scan_backend"]
    assert st["sphere_tests"] == sa["sphere_tests"]
    return got, st, b


# ------------------------------------------------------------------------------------------------ exact
@pytest.mark.parametrize("name,backend,prec,arm,threads", ARM_CASES, ids=[f"{c[3]}{c[4] or ''}-{c[0]}" for c in ARM_CASES])
def test_every_arm_matches_the_two_calls(dn_ctx, capi, name, backend, prec, arm, threads):
    arrays = ss.build(name, capi)
    b = {"auto": capi.SCAN_AUTO, "fp32": capi.SCAN_FP32}[backend]
    p = {"f32": capi.F32, "f64": capi.F64}[prec]
    assert ss.scan_arm(arrays, b, p)[0] == arm
    if threads:
        assert _wide_threads(arrays) == threads
    dn_ctx.upload_scene(**arrays)
    dn_ctx.set_scan_backend(b)
    if name.startswith("final"):
        cam = orbit(capi, 1)[0]
    else:
        R = ss.scene_info(arrays)["R"]
        cam = orbit(capi, 1, radius=3.0 * R, height=0.5 * R, fov=45.0)[0]
    prm = capi.default_params(width=W, height=H, spp=2 if prec == "f64" else SPP, seed=3, precision=p)
    _, st, _ = check(dn_ctx, capi, cam, prm)
    assert st["scan_backend"] == (capi.SCAN_TENSOR if arm == "Tensor" else capi.SCAN_FP32)


def test_equals_the_numpy_restatement(ctx_final, capi):
    """independent of rtiow_denoise: np_denoise over render_aov's buffers gives the same bits"""
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=8, seed=2, max_depth=50)
    for dp in (_dp(capi), _dp(capi, levels=3, sigma_color=0.5, sigma_normal=0.3, sigma_depth=0.05)):
        got, _, b = check(ctx_final, capi, cam, prm, dp)
        y, rgba = np_denoise.denoise(b["color"], b["albedo"], b["normal"], b["depth"], dp.levels, dp.sigma_color, dp.sigma_normal,
                                     dp.sigma_depth, dp.alpha)
        assert_same(got, {"color": y, "rgba": rgba}, "numpy")


EDGES = {
    "2x2": (dict(width=2, height=2), {}),
    "97x55": (dict(width=97, height=55), dict(levels=5)),                     # taps at steps up to 16 cross every border
    "levels0": ({}, dict(levels=0)),
    "levels10": ({}, dict(levels=10)),
    "sigmas-inf": ({}, dict(sigma_color=INF, sigma_normal=INF, sigma_depth=INF)),
    "alpha7": ({}, dict(alpha=7)),
    "depth0": (dict(max_depth=0), {}),
    "depth1": (dict(max_depth=1), {}),
    "spp70000-2x2": (dict(width=2, height=2, spp=70000), {}),
}


@pytest.mark.parametrize("case", list(EDGES))
def test_edges(ctx_final, capi, case):
    pk, dk = EDGES[case]
    prm = capi.default_params(**{**dict(width=W, height=H, spp=SPP, seed=4), **pk})
    cam = orbit(capi, 1, aspect=prm.width / prm.height)[0]
    got, st, b = check(ctx_final, capi, cam, prm, _dp(capi, **dk))
    assert got["rgba"].shape == (prm.height, prm.width, 4) and (got["rgba"][..., 3] == dk.get("alpha", 255)).all()
    if case == "depth0":                # no camera ray: colour 0 and depth +inf everywhere, so the denoised frame is black
        assert st["rays_traced"] == 0 and not b["color"].any() and np.isinf(b["depth"]).all()
        assert not got["color"].any() and not got["rgba"][..., :3].any()
    if case == "spp70000-2x2":          # colour sums saturate (2^32 / spp per channel), still inside the filter's ranges
        assert np.isfinite(got["color"]).all()


@pytest.mark.parametrize("scene", ["glass-inside", "sky"])
def test_edge_scenes(dn_ctx, capi, final_scene, scene):
    w, h = 48, 27
    if scene == "sky":
        arrays, cam = final_scene[0], capi.camera_new(*SKY_VIEW[:4], w / h, *SKY_VIEW[4:])
    else:
        arrays, cam = es.build(scene), es.camera(capi, scene, dict(W=w, H=h))
    dn_ctx.upload_scene(**arrays)
    _, _, b = check(dn_ctx, capi, cam, capi.default_params(width=w, height=h, spp=3, seed=3))
    if scene == "sky":
        assert np.isinf(b["depth"]).all()


def test_headline_frame(ctx_final, capi):
    prm = capi.default_params(width=1200, height=675, spp=16, seed=1, max_depth=50)
    check(ctx_final, capi, capi.camera_new((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, 1200 / 675, 0.1, 10.0), prm)


# ------------------------------------------------------------------------------------------------ buffers across calls
def test_buffers_sized_correctly_across_calls(capi, final_scene):
    """96x54, 32x18, 96x54, with render_aov, denoise and render between the fused calls: every result equals the same call in a
    fresh ctx"""
    sizes = [(96, 54), (32, 18), (96, 54)]
    cams = {s: orbit(capi, 1, aspect=s[0] / s[1])[0] for s in set(sizes)}
    prms = {s: capi.default_params(width=s[0], height=s[1], spp=3, seed=6) for s in set(sizes)}
    dp = _dp(capi)
    alone = {}
    for s in set(sizes):
        with capi.Context(1) as c:
            c.upload_scene(**final_scene[0])
            alone[s] = (two_call(c, cams[s], prms[s], dp), c.render(cams[s], prms[s])[0])
    with capi.Context(1) as c:
        c.upload_scene(**final_scene[0])
        for i, s in enumerate(sizes):
            (ref, b, _), frame = alone[s]
            got, _ = c.render_denoised(cams[s], prms[s], dp)
            assert_same(got, ref, f"render_denoised {s}, call {i}")
            img, bb, _ = c.render_aov(cams[s], prms[s])
            assert np.array_equal(img, frame)
            for k in b:
                assert bb[k].tobytes() == b[k].tobytes(), (s, k)
            got, _ = c.render_denoised(cams[s], prms[s], dp, out_color=False)
            assert np.array_equal(got["rgba"], ref["rgba"])
            dn, _ = c.denoise(bb["color"], bb["albedo"], bb["normal"], bb["depth"], dp)
            assert_same(dn, ref, f"denoise {s}, call {i}")
            assert np.array_equal(c.render(cams[s], prms[s])[0], frame)
            got, _ = c.render_denoised(cams[s], prms[s], dp, out_rgba=False)
            assert got["color"].tobytes() == ref["color"].tobytes()


# ------------------------------------------------------------------------------------------------ behaviour
def test_deterministic_across_calls_and_contexts(ctx_final, capi, final_scene):
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=70, seed=9)            # chunks of 64 + 6 samples
    a, _ = ctx_final.render_denoised(cam, prm)
    b, _ = ctx_final.render_denoised(cam, prm)
    with capi.Context(device=0) as c:
        c.upload_scene(**final_scene[0])
        c_, _ = c.render_denoised(cam, prm)
    for k in ("color", "rgba"):
        assert a[k].tobytes() == b[k].tobytes() == c_[k].tobytes(), k


def test_each_output_may_be_null(ctx_final, capi):
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=2)
    both, _ = ctx_final.render_denoised(cam, prm)
    only_c, _ = ctx_final.render_denoised(cam, prm, out_rgba=None)
    only_r, _ = ctx_final.render_denoised(cam, prm, out_color=None)
    assert set(only_c) == {"color"} and set(only_r) == {"rgba"}
    assert only_c["color"].tobytes() == both["color"].tobytes() and np.array_equal(only_r["rgba"], both["rgba"])


def test_pinned_and_pageable_rgba_agree(ctx_final, capi):
    torch = pytest.importorskip("torch")
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=2)
    pageable, _ = ctx_final.render_denoised(cam, prm, out_color=False)
    pinned = torch.zeros((H, W, 4), dtype=torch.uint8, pin_memory=True).numpy()
    got, _ = ctx_final.render_denoised(cam, prm, out_color=False, out_rgba=pinned)
    assert np.shares_memory(got["rgba"], pinned) and np.array_equal(pinned, pageable["rgba"])


@pytest.mark.parametrize("levels", [0, 4, 10])
def test_stats(ctx_final, capi, levels):
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=2)
    dp = _dp(capi, levels=levels)
    n = W * H
    _, sa = ctx_final.render_aov(cam, prm)[1:]
    for oc, orr, d2h in ((True, True, 16 * n), (True, False, 12 * n), (False, True, 4 * n)):
        _, st = ctx_final.render_denoised(cam, prm, dp, out_color=oc, out_rgba=orr)
        assert st["h2d_bytes"] == C.sizeof(capi.Camera) + C.sizeof(capi.Params)
        assert st["d2h_bytes"] == 16 + d2h
        assert st["kernel_launches"] == 3 + levels + 2 and st["n_gpus"] == 1
        assert st["paths"] == sa["paths"] and st["rays_traced"] == sa["rays_traced"] and st["scan_backend"] == sa["scan_backend"]
        assert st["kernel_ms"] > 0 and st["total_ms"] >= st["kernel_ms"]


def test_rank_ctx_of_world_one(capi, final_scene):
    with capi.Context(device=0, rank=0, world=1) as c:
        c.upload_scene(**final_scene[0])
        check(c, capi, orbit(capi, 1)[0], capi.default_params(width=W, height=H, spp=SPP, seed=8))


# ------------------------------------------------------------------------------------------------ errors
def _raw(capi, h, cam, prm, dp, oc, orr):
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)        # noqa: E731
    return capi.lib().rtiow_render_denoised(h, None if cam is None else C.byref(cam), C.byref(prm), None if dp is None else C.byref(dp),
                                            p(oc), p(orr), None)


def test_errors_write_nothing(ctx_final, capi):
    cam = orbit(capi, 1)[0]
    prm = capi.default_params(width=W, height=H, spp=1)
    good = _dp(capi)
    cases = [("null-ctx", None, cam, prm, good), ("null-cam", ctx_final._h, None, prm, good), ("null-dp", ctx_final._h, cam, prm, None),
             ("levels-11", ctx_final._h, cam, prm, _dp(capi, levels=11)),
             ("width-1", ctx_final._h, cam, capi.default_params(width=1, height=H, spp=1), good)]
    for field in ("sigma_color", "sigma_normal", "sigma_depth"):
        for v in (float("nan"), 0.0, 1e-13):
            cases.append((f"{field}={v}", ctx_final._h, cam, prm, _dp(capi, **{field: v})))
    for tag, h, c, pr, dp in cases:
        oc, orr = np.full((H, W, 3), 7, np.float32), np.full((H, W, 4), 7, np.uint8)
        assert _raw(capi, h, c, pr, dp, oc, orr) == capi.ERR_INVALID_ARG, tag
        assert (oc == 7).all() and (orr == 7).all(), tag
    assert _raw(capi, ctx_final._h, cam, prm, good, None, None) == capi.ERR_INVALID_ARG
    with capi.Context(1) as c:                                             # no scene
        oc, orr = np.full((H, W, 3), 7, np.float32), np.full((H, W, 4), 7, np.uint8)
        assert _raw(capi, c._h, cam, prm, good, oc, orr) == capi.ERR_INVALID_ARG
        assert (oc == 7).all() and (orr == 7).all()
        with pytest.raises(capi.RtiowError) as e:
            c.render_denoised(cam, prm)
        assert e.value.code == capi.ERR_INVALID_ARG


# ------------------------------------------------------------------------------------------------ several GPUs
def test_multi_gpu_matches_one_device(capi, final_scene):
    n = capi.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    cam = orbit(capi, 1)[0]
    dp = _dp(capi)
    # tile_rows 1; 4 and 5 end on a short tile; 27 gives two row tiles, fewer than the devices when there are more than two
    trs = [1, 4, 5] + ([27] if n > 2 else [])
    with capi.Context(1) as c1:
        c1.upload_scene(**final_scene[0])
        base = {tr: c1.render_denoised(cam, capi.default_params(width=W, height=H, spp=SPP, seed=9, tile_rows=tr), dp) for tr in trs}
    with capi.Context(n) as cn:
        cn.upload_scene(**final_scene[0])
        for tr, (ref, s1) in base.items():
            got, st = cn.render_denoised(cam, capi.default_params(width=W, height=H, spp=SPP, seed=9, tile_rows=tr), dp)
            assert_same(got, ref, f"tile_rows {tr}")
            rendering = min(n, -(-H // tr))
            assert st["n_gpus"] == n and st["rays_traced"] == s1["rays_traced"] and st["paths"] == s1["paths"]
            assert st["kernel_launches"] == 3 * rendering + dp.levels + 2
