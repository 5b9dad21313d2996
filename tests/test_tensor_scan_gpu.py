"""GPU suite: the two filter backends of the F32 scan (HittableList::hit, shapes/mod.rs:56-69).

RTIOW_SCAN_FP32 (7 FFMA2 per sphere pair on the CUDA cores) and RTIOW_SCAN_TENSOR (the discriminant as a tcgen05.mma
contraction, rt_umma.cuh) are both CONSERVATIVE filters in front of the same precise test: on the same ray they must find
the same sphere, t, p and normal BIT FOR BIT (rtiow_hitlist_batch, millions of rays in tools/diag_tensor.py).  A whole
render goes through two separately compiled kernels, whose scalar code (hit point, scatter) the compiler contracts into
FMAs differently: a last-bit difference in one t is amplified along long specular paths (tools/diag_tensor.py pixel:
40 bounces inside the glass sphere), so images agree on all but ~1 pixel in 10^5 and ray counts to ~1e-5 — the same
kind of difference the f32 render has against the f64 oracle, three orders of magnitude smaller.  The parity tests of the
other files run on whatever RTIOW_SCAN_AUTO selects (the tensor filter for the final scene).
"""
import numpy as np
import pytest

from conftest import final_camera

pytestmark = pytest.mark.gpu


@pytest.fixture()
def restore_backend(ctx, capi):
    yield
    ctx.set_scan_backend(capi.SCAN_AUTO)


def _render(ctx, capi, backend, **kw):
    ctx.set_scan_backend(backend)
    W, H = kw["width"], kw["height"]
    return ctx.render(final_camera(capi, W / H), capi.default_params(**kw))


@pytest.mark.parametrize("W,H,spp", [(400, 225, 10), (333, 187, 3), (64, 36, 33)])
def test_backends_render_identical_images(ctx_final, capi, restore_backend, W, H, spp):
    a, sa = _render(ctx_final, capi, capi.SCAN_FP32, width=W, height=H, spp=spp, seed=7)
    b, sb = _render(ctx_final, capi, capi.SCAN_TENSOR, width=W, height=H, spp=spp, seed=7)
    assert sa["scan_backend"] == capi.SCAN_FP32 and sb["scan_backend"] == capi.SCAN_TENSOR
    assert abs(sa["rays_traced"] - sb["rays_traced"]) <= 1e-4 * sa["rays_traced"]
    differ = (a != b).any(axis=2)
    assert differ.mean() <= 1e-4, f"{differ.sum()} pixels differ between the FP32 and the tensor filter"
    assert np.abs(a.astype(int) - b.astype(int)).max() <= 48          # one sample of spp took another path
    c, sc = _render(ctx_final, capi, capi.SCAN_AUTO, width=W, height=H, spp=spp, seed=7)
    assert sc["scan_backend"] == capi.SCAN_TENSOR and np.array_equal(b, c)          # the final scene qualifies


@pytest.mark.parametrize("mode", [1, 2, 3])
def test_backends_agree_on_material_scenes(ctx, capi, scene_factory, restore_backend, mode):
    """BASELINE configs[2] scenes (all-Lambertian / all-Metal / all-Dialectric + hollow shell with a negative radius)"""
    arrays, _ = scene_factory(1, 11, mode)
    ctx.upload_scene(**arrays)
    a, sa = _render(ctx, capi, capi.SCAN_FP32, width=200, height=112, spp=8, seed=3)
    b, sb = _render(ctx, capi, capi.SCAN_TENSOR, width=200, height=112, spp=8, seed=3)
    assert abs(sa["rays_traced"] - sb["rays_traced"]) <= 2e-4 * sa["rays_traced"] and (a != b).any(axis=2).mean() <= 2e-4


def test_backends_agree_on_hitlist(ctx_final, capi, restore_backend):
    """the unit-level scan: camera rays, rays leaving the ground and the spheres, far origins, rays that miss everything"""
    rng = np.random.default_rng(5)
    n = 40_000
    o = np.empty((n, 3)); d = np.empty((n, 3))
    o[: n // 4] = (13, 2, 3) + 0.05 * rng.standard_normal((n // 4, 3))
    d[: n // 4] = np.stack([rng.uniform(-11, 11, n // 4), rng.uniform(-0.5, 2.5, n // 4), rng.uniform(-11, 11, n // 4)], 1) - o[: n // 4]
    o[n // 4 :] = np.stack([rng.uniform(-12, 12, n - n // 4), rng.uniform(0, 0.4, n - n // 4), rng.uniform(-12, 12, n - n // 4)], 1)
    d[n // 4 :] = rng.standard_normal((n - n // 4, 3))
    o[-2000:] *= 150.0                                  # far origins: the per-ray slack of the foot point
    d[-4000:-2000] *= 1e-3                              # short directions: t scales, the hit does not
    o, d = o.astype(np.float32).astype(float), d.astype(np.float32).astype(float)
    ctx_final.set_scan_backend(capi.SCAN_FP32); a = ctx_final.hitlist_batch(o, d)
    ctx_final.set_scan_backend(capi.SCAN_TENSOR); b = ctx_final.hitlist_batch(o, d)
    assert 0.2 < a["hit"].mean() < 0.999
    for k in ("hit", "index", "front_face"):
        assert np.array_equal(a[k], b[k]), k
    # the same precise test on the same sphere, compiled into two kernels (different FMA contraction): agreement to a few
    # roundings of the lengths involved (|o|, the scene's extent, the distance travelled)
    dl = np.linalg.norm(d, axis=1)
    length = np.abs(a["t"]) * dl + np.linalg.norm(o, axis=1) + 20.0
    assert (np.abs(a["t"] - b["t"]) * dl <= 1e-6 * length).all()
    assert (np.abs(a["p"] - b["p"]).max(axis=1) <= 1e-6 * length).all()
    assert (np.abs(a["normal"] - b["normal"]).max(axis=1) <= 1e-6 * length / 0.2).all()      # (p - c) / r with r >= 0.2


def test_backends_agree_on_ray_color(ctx_final, capi, restore_backend):
    rng = np.random.default_rng(9)
    n = 5000
    o = np.tile([13.0, 2.0, 3.0], (n, 1))
    d = np.stack([rng.uniform(-11, 11, n), rng.uniform(0, 1.5, n), rng.uniform(-11, 11, n)], 1) - o
    d = d.astype(np.float32).astype(float)
    px = rng.integers(0, 1 << 20, n).astype(np.uint32); sm = rng.integers(0, 500, n).astype(np.uint32)
    ctx_final.set_scan_backend(capi.SCAN_FP32); a = ctx_final.ray_color_batch(o, d, px, sm, seed=11)
    ctx_final.set_scan_backend(capi.SCAN_TENSOR); b = ctx_final.ray_color_batch(o, d, px, sm, seed=11)
    same = (a["rays"] == b["rays"]) & (a["color"] == b["color"]).all(axis=1)
    assert same.mean() > 0.99, f"{(~same).sum()} of {n} paths differ"      # long specular paths amplify a last-bit difference
    assert a["rays"].max() > 5


@pytest.mark.parametrize("backend", ["SCAN_FP32", "SCAN_TENSOR"])
def test_ray_color_trace_records_every_ray(ctx_final, capi, final_scene, restore_backend, backend):
    """rtiow_ray_color_trace_batch follows ray_color_batch's paths and records each ray and the sphere it hit"""
    rng = np.random.default_rng(10)
    n, depth = 3000, 50
    o = np.tile([13.0, 2.0, 3.0], (n, 1))
    d = np.stack([rng.uniform(-11, 11, n), rng.uniform(0, 1.5, n), rng.uniform(-11, 11, n)], 1) - o
    d = d.astype(np.float32).astype(float)
    px = rng.integers(0, 1 << 20, n).astype(np.uint32); sm = rng.integers(0, 500, n).astype(np.uint32)
    ctx_final.set_scan_backend(getattr(capi, backend))
    a = ctx_final.ray_color_batch(o, d, px, sm, seed=11, max_depth=depth)
    tr = ctx_final.ray_color_trace_batch(o, d, px, sm, seed=11, max_depth=depth)
    assert np.array_equal(a["color"], tr["color"]) and np.array_equal(a["rays"], tr["rays"])
    rays = tr["rays"].astype(np.int64)[:, None]
    k = np.arange(depth)[None, :]
    assert rays.max() > 5 and (rays >= 1).all()
    assert (tr["index"][k < rays - 1] >= 0).all()                    # every ray but a path's last one hit a sphere
    assert (tr["index"][k >= rays] == -1).all() and (tr["ray"][k >= rays] == 0).all()
    assert np.abs(tr["ray"][:, 0, :3] - o).max() == 0.0
    assert np.abs(tr["ray"][:, 0, 3:] - d / np.linalg.norm(d, axis=1, keepdims=True)).max() < 1e-6
    # ray k + 1 starts on sphere index[k].  The hit point is o + dhat t in f32: both filters put it within 4e-6 of the sphere
    # (hit points up to 53 from the origin, where an f32 ulp is 4e-6).  The bar of 1e-4 allows 25 times that and is still
    # far below 0.2, the smallest radius, so a ray recorded against the wrong sphere or depth fails it.
    cen, rad = np.asarray(final_scene[0]["center"], float), np.abs(np.asarray(final_scene[0]["radius"], float))
    bounce = k[:, :-1] < rays - 1
    i, j = np.nonzero(bounce)
    s = tr["index"][i, j]
    res = np.abs(np.linalg.norm(tr["ray"][i, j + 1, :3] - cen[s], axis=1) - rad[s])
    assert len(res) > n and res.max() < 1e-4, f"max |dist - r| {res.max():.3g}"


def test_selection_rules(ctx, capi, scene_factory, restore_backend):
    """a scene whose sphere table does not fit one CTA's shared memory stays on the FP32 filter; forcing TENSOR is an error, not a fallback"""
    arrays, _ = scene_factory(1, 50, 0)                 # ~10.2 k spheres (BASELINE configs[3])
    ctx.upload_scene(**arrays)
    img, st = _render(ctx, capi, capi.SCAN_AUTO, width=64, height=36, spp=1, seed=1)
    assert st["scan_backend"] == capi.SCAN_FP32
    ctx.set_scan_backend(capi.SCAN_TENSOR)
    with pytest.raises(capi.RtiowError) as e:
        ctx.render(final_camera(capi, 64 / 36), capi.default_params(width=64, height=36, spp=1))
    assert e.value.code == capi.ERR_UNSUPPORTED
    with pytest.raises(capi.RtiowError):
        ctx.set_scan_backend(7)
    # a tiny scene: 3 spheres + ground
    ctx.upload_scene(center=[[0, -1000, 0], [0, 1, 0], [-4, 1, 0], [4, 1, 0]], radius=[1000, 1, 1, 1], mat_index=[0, 1, 2, 3],
                     mat_kind=[0, 2, 0, 1], mat_albedo=[[.5, .5, .5], [1, 1, 1], [.4, .2, .1], [.7, .6, .5]], mat_param=[0, 1.5, 0, 0])
    a, sa = _render(ctx, capi, capi.SCAN_FP32, width=160, height=90, spp=4, seed=2)
    b, sb = _render(ctx, capi, capi.SCAN_TENSOR, width=160, height=90, spp=4, seed=2)
    assert sb["scan_backend"] == capi.SCAN_TENSOR and abs(sa["rays_traced"] - sb["rays_traced"]) <= 2 and (a != b).any(axis=2).mean() <= 2e-4
