"""GPU suite: every arm of the F32 hit scan against the f64 oracle, on scenes at the sizes where plan_scan changes its choice.

plan_scan (rtiow_b200/csrc/capi.cu) runs a scan on the tensor filter (Tensor), on the FP32 filter with its table in shared
memory (Smem), in one wide CTA (Wide) or in global memory (Global), or in f64.  tests/scan_scenes.py builds scenes on both sides
of each rule and mirrors the rules in numpy; here each scene runs on every arm that applies to it (SCAN_TENSOR and SCAN_FP32
forced, F64 on a few), and:
  * the arm the library reports (rtiow_stats.scan_backend) is the mirror's, and forcing TENSOR fails exactly where it should;
  * rtiow_hitlist_batch returns the oracle's sphere on EVERY robust ray (scan_scenes.robust_closest: not grazing, no other
    root within 1e-5 of the scene's size, not at t_min), and every small sphere is the robust winner of some ray — two rays
    per sphere see to that — so a filter that loses one sphere column, one record of a partial word or one candidate fails;
  * t, p and normal stay within the bars of tests/test_parity_unit_gpu.py;
  * rays whose lines meet more spheres than the candidate lists hold (RT_CAND_CAP) find the oracle's hits and paths;
  * the large spheres take the f64 routine in every lane (not representable in f32) or in some lanes of a warp only;
  * one small render per arm follows the oracle's paths (the bars of test_material_isolation_scenes).
"""
from functools import lru_cache

import numpy as np
import pytest

import scan_scenes as ss
from conftest import final_camera
from test_parity_unit_gpu import f32, not_grazing, t_err, vec_err

pytestmark = pytest.mark.gpu

TENSOR, FP32, AUTO, F64 = "tensor", "fp32", "auto", "f64"
# scenes run here (the rest of scan_scenes.SCENES are random_scene sizes, rendered below or only checked by the mirror)
HITLIST_SCENES = [n for n in ss.SCENES if not n.startswith("final-h")]
F64_SCENES = ["compact-129", "row-r0.4", "ball-R121", "big-not-f32"]
OVERFLOW_SCENES = ["field-row", "overlap-lattice", "row-r0.2", "row-r0.4"]
UNCOVERED = {"overlap-lattice"}          # overlapping spheres: some are nowhere the first surface along a ray


def _backend(capi, name):
    return {TENSOR: capi.SCAN_TENSOR, FP32: capi.SCAN_FP32, AUTO: capi.SCAN_AUTO}[name]


def _cases():
    from rtiow_b200 import capi
    out = []
    for name in HITLIST_SCENES:
        arms = ss.SCENES[name][1]
        out += [(name, b) for b in (TENSOR, FP32) if arms[_backend(capi, b)] is not None]
    return out + [(name, F64) for name in F64_SCENES]


@pytest.fixture()
def scan(ctx, capi):
    """the session's ctx; the scan backend goes back to AUTO afterwards"""
    yield ctx
    ctx.set_scan_backend(capi.SCAN_AUTO)


@lru_cache(maxsize=None)
def _reference(name, capi, oracle, kind="hitlist"):
    arrays = ss.build(name, capi)
    o, d = far_ground_rays(arrays) if kind == "far-ground" else ss.rays(name, arrays)
    ref = oracle.world_hit_batch(oracle.Scene(**arrays), o, d)
    return arrays, o, d, ref, ss.robust_closest(arrays, o, d)


def _check_hitlist(arrays, o, d, ref, rc, got, prec, cover=True):
    want = np.where(ref["hit"] == 1, ref["index"], -1)
    rob = rc["robust"]
    assert rob.mean() > 0.3
    assert np.array_equal(rc["index"][rob], want[rob]), "the numpy reference and the oracle disagree on a robust ray"
    if cover:
        lost = np.setdiff1d(ss.scene_info(arrays)["small"], rc["index"][rob])
        assert len(lost) == 0, f"{len(lost)} small spheres are the robust winner of no ray"
    wrong = np.flatnonzero(rob & (got["index"] != want))
    assert len(wrong) == 0, f"{len(wrong)} robust rays hit another sphere, e.g. ray {wrong[0]}: {got['index'][wrong[0]]} instead of {want[wrong[0]]}"
    agree = got["index"] == want
    assert agree.mean() >= 0.999, f"closest-hit index disagrees on {(~agree).sum()} of {len(o)} rays"
    assert np.array_equal(got["hit"], (got["index"] >= 0).astype(np.int32))
    # values: the bars of test_hitlist_closest_hit
    c, r = arrays["center"], arrays["radius"]
    hi = np.maximum(want, 0)
    m = agree & (want >= 0) & not_grazing(c[hi], r[hi], o, d) & (np.abs(ref["t"] - 1e-4) > 1e-5)
    tol = 1e-5 if prec == 0 else 1e-8
    te = t_err(got["t"][m], ref["t"][m], o[m], d[m], c[hi][m])
    assert te.max() < tol, te.max()
    assert vec_err(got["p"][m], ref["p"][m], np.linalg.norm(o[m], axis=1)).max() < tol
    assert np.array_equal(got["front_face"][m], ref["front_face"][m])
    M = np.maximum(np.maximum(np.linalg.norm(o[m], axis=1), np.linalg.norm(c[hi][m], axis=1)), np.linalg.norm(ref["p"][m], axis=1))
    kappa = np.maximum(1.0, 0.25 * M / np.abs(r[hi][m]))
    assert (np.abs(got["normal"][m] - ref["normal"][m]).max(axis=1) / kappa).max() < (1e-5 if prec == 0 else 2e-11)


@pytest.mark.parametrize("name", HITLIST_SCENES + ["final-h27", "final-h28"])
def test_arm_selection(scan, capi, name):
    """AUTO picks the mirror's filter, and forcing TENSOR is refused exactly on the scenes the mirror says do not qualify"""
    arrays = ss.build(name, capi)
    scan.upload_scene(**arrays)
    arm = ss.scan_arm(arrays, capi.SCAN_AUTO)[0]
    _, st = scan.render(final_camera(capi, 16 / 9), capi.default_params(width=16, height=9, spp=1))
    assert st["scan_backend"] == (capi.SCAN_TENSOR if arm == "Tensor" else capi.SCAN_FP32), arm
    scan.set_scan_backend(capi.SCAN_TENSOR)
    if ss.scan_arm(arrays, capi.SCAN_TENSOR)[0] is None:
        with pytest.raises(capi.RtiowError) as e:
            scan.hitlist_batch([[0.0, 0.0, -50.0]], [[0.0, 0.0, 1.0]])
        assert e.value.code == capi.ERR_UNSUPPORTED
    else:
        scan.hitlist_batch([[0.0, 0.0, -50.0]], [[0.0, 0.0, 1.0]])


@pytest.mark.parametrize("name,backend", _cases())
def test_hitlist_vs_oracle(scan, capi, oracle, name, backend):
    arrays, o, d, ref, rc = _reference(name, capi, oracle)
    if name in OVERFLOW_SCENES:
        # a lower bound on the filter's survivors: these rays overflow the candidate lists on either filter
        assert (ss.line_survivors(arrays, o, d) > ss.CAND_CAP).sum() >= 500
    scan.upload_scene(**arrays)
    prec = capi.F64 if backend == F64 else capi.F32
    if backend != F64:
        scan.set_scan_backend(_backend(capi, backend))
    got = scan.hitlist_batch(o, d, 1e-4, precision=prec)
    _check_hitlist(arrays, o, d, ref, rc, got, prec, cover=name not in UNCOVERED)


@pytest.mark.parametrize("backend", [TENSOR, FP32])
@pytest.mark.parametrize("name", ["field-row", "overlap-lattice"])
def test_ray_color_with_candidate_overflow(scan, capi, oracle, name, backend):
    """whole paths through scenes where rays meet more spheres than the candidate lists hold: bounce rays leave a sphere
    inside the crowd, so the overflow branch must skip the sphere the ray starts on (the bars of
    test_ray_color_iterative_vs_recursive, widened where noted for overlapping surfaces)"""
    arrays, o, d, _, _ = _reference(name, capi, oracle)
    pick = np.random.default_rng(21).choice(len(o), min(len(o), 8000), replace=False)
    o, d = o[pick], d[pick]
    rng = np.random.default_rng(22)
    pix = rng.integers(0, 2 ** 31, len(o)).astype(np.uint32); smp = rng.integers(0, 500, len(o)).astype(np.uint32)
    ref = oracle.ray_color_batch(oracle.Scene(**arrays), o, d, pix, smp, seed=77)
    assert ref["rays"].mean() > 2.5                       # paths bounce inside the crowd
    scan.upload_scene(**arrays)
    scan.set_scan_backend(_backend(capi, backend))
    got = scan.ray_color_batch(o, d, pix, smp, seed=77)
    same = got["rays"] == ref["rays"]
    err = np.abs(got["color"] - ref["color"]).max(axis=1)
    # overlapping surfaces put many bounces within f32 rounding of a second root: on a B200 (1000 W) both filters kept 0.971
    # (overlap-lattice) and 0.992 (field-row) of the paths, the same fraction, and precision=F64 all of them; the 99th
    # percentile of the colour error on kept paths was 1.6e-4 on field-row, again the same on both filters
    assert same.mean() > 0.96, same.mean()
    assert np.median(err[same]) < 1e-6 and np.percentile(err[same], 99) < 3e-4
    assert abs(got["color"].mean() - ref["color"].mean()) < 2e-3
    assert got["rays"].max() <= 50 and abs(got["rays"].mean() - ref["rays"].mean()) < 0.04
    # and the other filter takes the same paths (the overflow code of the two is separate)
    scan.set_scan_backend(_backend(capi, FP32 if backend == TENSOR else TENSOR))
    other = scan.ray_color_batch(o, d, pix, smp, seed=77)
    assert (other["rays"] == got["rays"]).mean() > 0.99


def test_large_spheres_not_f32_representable(capi):
    """big-not-f32 really keeps the f32 records of its large spheres off (every lane takes the f64 routine)"""
    arrays = ss.build("big-not-f32", capi)
    big = np.setdiff1d(np.arange(len(arrays["radius"])), ss.scene_info(arrays)["small"])
    assert len(big) == 2 and (f32(arrays["radius"][big]) != arrays["radius"][big]).all()


def far_ground_rays(arrays, n=8192, seed=0):
    """final scene: warps whose even lanes start near the spheres and whose odd lanes start 1e-3 .. 1e-2 above the ground
    200 .. 600 units from the coordinate origin, where |o|^2 - 2 o.c cancels and big_spheres_f32 hands the lane to f64"""
    rng = np.random.default_rng(10_000 + seed)
    h = n // 2
    k = rng.choice(ss.scene_info(arrays)["small"], n)
    target = arrays["center"][k]
    o_near = np.stack([rng.uniform(-11, 11, h), rng.uniform(1e-3, 0.4, h), rng.uniform(-11, 11, h)], 1)
    rho, th = rng.uniform(200, 600, h), rng.uniform(0, 2 * np.pi, h)
    surf = np.stack([rho * np.cos(th), np.sqrt(1000.0 ** 2 - rho ** 2) - 1000.0, rho * np.sin(th)], 1)
    nrm = (surf - [0.0, -1000.0, 0.0]) / 1000.0
    o_far = surf + nrm * rng.uniform(1e-3, 1e-2, (h, 1))
    o = np.empty((n, 3)); o[0::2], o[1::2] = o_near, o_far
    d = target - o
    rnd = rng.normal(size=(n, 3))
    away = rng.random(n) < 0.5                               # half: random directions (sky, the ground, grazing the ground)
    d[away] = rnd[away] * rng.uniform(0.3, 2.0, (away.sum(), 1))
    return f32(o), f32(d)


@pytest.mark.parametrize("backend", [TENSOR, FP32])
def test_far_ground_lanes_mix_f32_and_f64(scan, capi, oracle, backend):
    arrays, o, d, ref, rc = _reference("final", capi, oracle, kind="far-ground")
    # big_spheres_f32's cancellation test, for the ground (K = |c|^2 - r^2 = 0): about half of each warp goes to f64
    oo = (o * o).sum(1); P = o @ np.array([0.0, -1000.0, 0.0]); C = oo - 2 * P
    need64 = (oo + 2 * np.abs(P)) > 16 * np.abs(C)
    per_warp = need64.reshape(-1, 32).mean(1)
    assert ((per_warp > 0.25) & (per_warp < 0.75)).mean() > 0.9
    scan.upload_scene(**arrays)
    scan.set_scan_backend(_backend(capi, backend))
    got = scan.hitlist_batch(o, d, 1e-4)
    _check_hitlist(arrays, o, d, ref, rc, got, 0, cover=False)
    assert (ref["index"][need64 & (ref["hit"] == 1)] == 0).mean() > 0.2        # lanes of both kinds hit the ground


@pytest.mark.parametrize("name,backend,arm", [("final", FP32, "Smem"), ("final-h27", TENSOR, "Tensor"),
                                              ("ball-R121", TENSOR, "Tensor"), ("final-h28", AUTO, "Wide")])
def test_render_vs_oracle(scan, capi, oracle, name, backend, arm):
    """one small frame per arm, same paths as the oracle's DIRECT sampler"""
    arrays = ss.build(name, capi)
    if name == "ball-R121":
        # Lambertian only: its dense glass and metal spheres send long specular paths whose f32 rounding leaves the oracle's
        # paths on ~4 % of the pixels at 4 spp (on the FP32 and the tensor filter alike; precision=F64 follows them)
        arrays = {**arrays, "mat_kind": np.zeros_like(arrays["mat_kind"])}
    assert ss.scan_arm(arrays, _backend(capi, backend))[0] == arm
    W, H, spp = 160, 90, 8
    view = ((40, 12, 25), (0, 0, 0), (0, 1, 0), 30.0, W / H, 0.1, 45.0) if name == "ball-R121" else None
    cam = (lambda mod: mod.camera_new(*view)) if view else (lambda mod: final_camera(mod, W / H))
    ref, _, cnt = oracle.render(oracle.Scene(**arrays), cam(oracle), W, H, spp, seed=5, sampler=oracle.SAMPLER_DIRECT)
    scan.upload_scene(**arrays)
    scan.set_scan_backend(_backend(capi, backend))
    img, st = scan.render(cam(capi), capi.default_params(width=W, height=H, spp=spp, seed=5))
    assert st["scan_backend"] == (capi.SCAN_TENSOR if arm == "Tensor" else capi.SCAN_FP32)
    diff = np.abs(img[..., :3].astype(int) - ref[..., :3].astype(int)).max(axis=2)
    assert (diff <= 1).mean() > 0.99, f"{(diff > 1).mean():.4%} pixels off by > 1 LSB"
    assert abs(st["rays_traced"] / cnt["rays"] - 1) < 5e-3
