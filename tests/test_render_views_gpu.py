"""rtiow_render_views: many cameras of one scene in one call, each frame byte-identical to its own rtiow_render.

A batch renders on one device as one frame n_views * height rows tall (rt_render.cuh, render_views_kernel): the work split,
the accumulators and the epilogue are the frame's, and only a fresh path's row -> (view, row in the view) split and its camera
differ.  A frame is a pure function of (scene, camera, params) and the accumulation is integer, so every view must equal
rtiow_render of its camera exactly, on every arm plan_scan can choose, and where the work split puts view boundaries inside
one fetch or one warp's assignment.

The CPU tests at the end check the library's kernel inventory and the ctypes binding; everything else needs a GPU.
"""
import ctypes as C
import re
import subprocess

import numpy as np
import pytest

import scan_scenes as ss

W, H, SPP = 96, 54, 4
gpu = pytest.mark.gpu


def orbit(capi, k, radius=13.4, height=2.0, aspect=W / H, fov=20.0, look_at=(0.0, 0.0, 0.0)):
    """k distinct cameras on a circle about the vertical axis through look_at (the first one is the reference camera's
    position when radius and height are the defaults)"""
    cams = []
    for i in range(k):
        a = 0.23 + 2 * np.pi * i / k
        frm = (look_at[0] + radius * np.cos(a), look_at[1] + height, look_at[2] + radius * np.sin(a))
        cams.append(capi.camera_new(frm, look_at, (0, 1, 0), fov, aspect, 0.1, 10.0))
    return cams


def check_views(ctx, capi, cams, prm, distinct=True):
    """the batch against one rtiow_render per camera: bytes, rays, paths, backend, and the copies the call reports"""
    imgs, st = ctx.render_views(cams, prm)
    k = len(cams)
    assert imgs.shape == (k, prm.height, prm.width, 4)
    rays = 0
    for v, cam in enumerate(cams):
        ref, sv = ctx.render(cam, prm)
        assert np.array_equal(imgs[v], ref), f"view {v} of {k} differs from its own rtiow_render"
        rays += sv["rays_traced"]
        assert st["scan_backend"] == sv["scan_backend"]
    if distinct and k > 1:
        assert not np.array_equal(imgs[0], imgs[1]), "the cameras should see different frames"
    assert st["rays_traced"] == rays
    assert st["paths"] == k * prm.width * prm.height * prm.spp
    assert st["h2d_bytes"] == k * C.sizeof(capi.Camera) + C.sizeof(capi.Params)
    return imgs, st


@pytest.fixture()
def views_ctx(ctx, capi):
    """the session's ctx; the scan backend goes back to AUTO afterwards"""
    yield ctx
    ctx.set_scan_backend(capi.SCAN_AUTO)


def _wide_threads(arrays):
    """the CTA width of the Wide arm (launch_render_kernel): 768 threads when their candidate lists fit beside the table"""
    table = (4 * ss.scene_info(arrays)["np"] + 16) * 4
    return 768 if table + 768 * ss.CAND_CAP * 2 <= ss.SMEM_CTA else 512


# (scene, backend, precision, arm, Wide CTA width)
ARM_CASES = [
    ("final", "auto", "f32", "Tensor", None),
    ("final", "fp32", "f32", "Smem", None),
    ("compact-3072", "fp32", "f32", "Wide", 768),
    ("compact-13472", "auto", "f32", "Wide", 512),
    ("final-h63", "auto", "f32", "Global", None),
    ("final", "auto", "f64", "F64", None),
]


@gpu
@pytest.mark.parametrize("name,backend,prec,arm,threads", ARM_CASES, ids=[f"{c[3]}{c[4] or ''}-{c[0]}" for c in ARM_CASES])
def test_every_arm_matches_single_renders(views_ctx, capi, name, backend, prec, arm, threads):
    arrays = ss.build(name, capi)
    b = {"auto": capi.SCAN_AUTO, "fp32": capi.SCAN_FP32}[backend]
    p = {"f32": capi.F32, "f64": capi.F64}[prec]
    assert ss.scan_arm(arrays, b, p)[0] == arm
    if threads:
        assert _wide_threads(arrays) == threads
    views_ctx.upload_scene(**arrays)
    views_ctx.set_scan_backend(b)
    if name.startswith("final"):
        cams = orbit(capi, 3 if prec == "f64" else 5)
    else:
        R = ss.scene_info(arrays)["R"]
        cams = orbit(capi, 4, radius=3.0 * R, height=0.5 * R, fov=45.0)
    prm = capi.default_params(width=W, height=H, spp=2 if prec == "f64" else SPP, seed=3, precision=p)
    _, st = check_views(views_ctx, capi, cams, prm)
    assert st["scan_backend"] == (capi.SCAN_TENSOR if arm == "Tensor" else capi.SCAN_FP32)


# the work split at its edges, on the final scene (AUTO: the tensor arm)
EDGE_CASES = {
    "one-view": dict(k=1, width=W, height=H, spp=SPP),
    "spp70": dict(k=3, width=40, height=24, spp=70),                  # chunks of 64 + 6 samples
    "2x2": dict(k=5, width=2, height=2, spp=SPP),
    "64x16x9": dict(k=64, width=16, height=9, spp=SPP),               # view boundaries inside one fetch and one warp's assignment
    "depth1": dict(k=3, width=W, height=H, spp=SPP, max_depth=1),
    "depth50": dict(k=3, width=W, height=H, spp=SPP, max_depth=50),
}


@gpu
@pytest.mark.parametrize("case", list(EDGE_CASES))
def test_work_split_edges(views_ctx, capi, final_scene, case):
    e = dict(EDGE_CASES[case])
    k = e.pop("k")
    views_ctx.upload_scene(**final_scene[0])
    prm = capi.default_params(seed=11, **e)
    cams = orbit(capi, k, aspect=prm.width / prm.height)
    imgs, st = check_views(views_ctx, capi, cams, prm, distinct=prm.width * prm.height > 4)
    assert st["n_gpus"] == 1 and st["kernel_launches"] == 2
    assert st["d2h_bytes"] == k * prm.width * prm.height * 4 + 16
    if case == "one-view":
        ref, _ = views_ctx.render(cams[0], prm)
        assert np.array_equal(imgs[0], ref)


@gpu
def test_render_after_a_batch_is_unchanged(views_ctx, capi, final_scene):
    """the batch grows the ctx's accumulators and frame buffer; a later plain frame on the same ctx must not notice"""
    views_ctx.upload_scene(**final_scene[0])
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=5)
    cam = orbit(capi, 1)[0]
    before, sb = views_ctx.render(cam, prm)
    views_ctx.render_views(orbit(capi, 8), capi.default_params(width=2 * W, height=2 * H, spp=SPP, seed=6))
    after, sa = views_ctx.render(cam, prm)
    assert np.array_equal(before, after) and sb["rays_traced"] == sa["rays_traced"]


@gpu
def test_pinned_and_pageable_output_agree(views_ctx, capi, final_scene):
    views_ctx.upload_scene(**final_scene[0])
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=7)
    cams = orbit(capi, 3)
    pageable, _ = views_ctx.render_views(cams, prm, out=np.zeros(3 * H * W * 4, np.uint8))
    torch = pytest.importorskip("torch")
    pinned = torch.zeros(3 * H * W * 4, dtype=torch.uint8).pin_memory()
    got, _ = views_ctx.render_views(cams, prm, out=pinned)
    assert np.array_equal(got.numpy(), pageable)


@gpu
@pytest.mark.parametrize("kind", ["on_device", "rank_world1"])
def test_other_one_device_contexts(capi, final_scene, kind):
    """rtiow_ctx_create_on_device and a rank ctx of world 1 render a batch like rtiow_ctx_create(1)"""
    mk = {"on_device": lambda: capi.Context(device=0), "rank_world1": lambda: capi.Context(device=0, rank=0, world=1)}[kind]
    with mk() as c:
        c.upload_scene(**final_scene[0])
        check_views(c, capi, orbit(capi, 3), capi.default_params(width=W, height=H, spp=SPP, seed=8))


def _raw_views(capi, ctx_h, cams, k, prm, out):
    st = capi.Stats()
    return capi.lib().rtiow_render_views(ctx_h, cams, k, C.byref(prm), out, C.byref(st))


@gpu
def test_errors(views_ctx, capi, final_scene):
    views_ctx.upload_scene(**final_scene[0])
    prm = capi.default_params(width=W, height=H, spp=1)
    cams = (capi.Camera * 2)(*orbit(capi, 2))
    out = np.zeros(2 * H * W * 4, np.uint8)
    assert _raw_views(capi, views_ctx._h, cams, 0, prm, out.ctypes.data_as(C.c_void_p)) == capi.ERR_INVALID_ARG
    assert _raw_views(capi, views_ctx._h, None, 2, prm, out.ctypes.data_as(C.c_void_p)) == capi.ERR_INVALID_ARG
    assert _raw_views(capi, views_ctx._h, cams, 2, prm, None) == capi.ERR_INVALID_ARG
    with pytest.raises(capi.RtiowError) as e:
        views_ctx.render_views([], prm)
    assert e.value.code == capi.ERR_INVALID_ARG
    # 256 views of 4096 x 4096 are 2^32 pixels: refused before anything is allocated (the out buffer is never touched)
    big = capi.default_params(width=4096, height=4096, spp=1)
    many = (capi.Camera * 256)(*(orbit(capi, 1) * 256))
    tiny = np.zeros(4, np.uint8)
    assert _raw_views(capi, views_ctx._h, many, 256, big, tiny.ctypes.data_as(C.c_void_p)) == capi.ERR_INVALID_ARG
    assert "batch too large" in capi.lib().rtiow_last_error().decode()
    # TENSOR forced on a scene the tensor filter does not take
    views_ctx.upload_scene(**ss.build("compact-3201", capi))
    views_ctx.set_scan_backend(capi.SCAN_TENSOR)
    with pytest.raises(capi.RtiowError) as e:
        views_ctx.render_views(orbit(capi, 2), prm)
    assert e.value.code == capi.ERR_UNSUPPORTED


@gpu
def test_no_scene(capi):
    with capi.Context(1) as c:
        with pytest.raises(capi.RtiowError) as e:
            c.render_views(orbit(capi, 2), capi.default_params(width=W, height=H, spp=1))
        assert e.value.code == capi.ERR_INVALID_ARG


@gpu
def test_multi_gpu_matches_one_device(capi, final_scene):
    """rtiow_ctx_create(n): each device renders a block of whole views straight into its slice of the output"""
    n = capi.device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=9)
    with capi.Context(1) as c1:
        c1.upload_scene(**final_scene[0])
        base = {k: c1.render_views(orbit(capi, k), prm) for k in (1, n - 1, 2 * n + 1)}
    with capi.Context(n) as cn:
        cn.upload_scene(**final_scene[0])
        for k, (ref, st1) in base.items():
            imgs, st = cn.render_views(orbit(capi, k), prm)
            assert np.array_equal(imgs, ref), f"{k} views on {n} GPUs differ from one GPU"
            assert st["n_gpus"] == n and st["rays_traced"] == st1["rays_traced"] and st["paths"] == st1["paths"]
            assert st["kernel_launches"] == 2 * min(k, n)


# ------------------------------------------------------------------------------------------------ CPU
VIEW_KERNELS = {
    "render_views_kernel<double, false, 256, 2>",     # F64
    "render_views_kernel<float, true, 256, 3>",       # Smem
    "render_views_kernel<float, true, 768, 1>",       # Wide, 768 threads
    "render_views_kernel<float, true, 512, 1>",       # Wide, 512 threads
    "render_views_kernel<float, false, 256, 4>",      # Global
    "render_views_kernel_umma<6, 64>",                # Tensor
}


def test_views_kernels_are_the_plan_arms(capi):
    """one render_views_kernel per arm of the scan plan, the same instantiations as render_kernel's"""
    syms = subprocess.run(["cuobjdump", "-symbols", str(capi.lib_path())], capture_output=True, text=True, check=True).stdout
    names = subprocess.run(["c++filt"], input=syms, capture_output=True, text=True, check=True).stdout
    found = set(re.findall(r"rt::(render_views_kernel(?:_umma)?<[^>]*>)", names))
    assert found == VIEW_KERNELS, f"unexpected: {sorted(found - VIEW_KERNELS)}, missing: {sorted(VIEW_KERNELS - found)}"
    frame = set(re.findall(r"rt::render_kernel((?:_umma)?<[^>]*>)", names))
    assert {n.replace("render_views_kernel", "") for n in VIEW_KERNELS} == frame


@pytest.mark.parametrize("size", [0, 3 * 9 * 16 * 4 - 1, 3 * 9 * 16 * 4 + 4, 2 * 9 * 16 * 4])
def test_binding_rejects_wrongly_sized_output(capi, size):
    """Context.render_views checks `out` before it calls the library (a ctx handle is not even needed)"""
    ctx = object.__new__(capi.Context)
    ctx._h = None
    cams = [capi.Camera() for _ in range(3)]
    with pytest.raises(ValueError):
        ctx.render_views(cams, capi.default_params(width=16, height=9, spp=1), out=np.zeros(size, np.uint8))
    with pytest.raises(ValueError):
        ctx.render_views(cams, capi.default_params(width=16, height=9, spp=1), out=np.zeros(3 * 9 * 16 * 4, np.float32))
