"""CPU suite: the oracle's per-pixel knife-edge margin (o_render_margins), which decides where an f32 render must give the
oracle's exact bytes (tests/test_render_exact_gpu.py).

  * o_render_margins renders exactly as o_render does: same bytes, sums and counters;
  * known answers: a grazing ray, a ray at the total-internal-reflection boundary and a metal ray at the absorption boundary
    get a margin of ~0, a ray through the centre of a sphere one of 1 / 11 (the sphere's radius over the lengths its roots
    are computed from);
  * soundness: on every case of tests/edge_scenes.py, renders of the scene with every small sphere's coordinates and radius
    moved by one f32 ulp (up or down at random; coincident spheres together), and of the camera rounded to f32 as the
    library's to_dev_camera rounds it, keep the bytes of every robust pixel.  (Large spheres, which the renderer tests in
    f64, move by one ulp of the small spheres' bounding radius: an ulp of a 1000-unit coordinate is not an error the
    renderer makes.)  Over every case the largest margin of a pixel that did change was 1.8e-6, 11x below MARGIN_TAU;
  * floors: each case keeps a robust fraction above a recorded floor, so the GPU comparison always has pixels to check.
"""
import numpy as np
import pytest

import edge_scenes as es


def _render(oracle, name, p, scene=None, cam=None):
    arrays = es.build(name)
    return oracle.render_margins(scene or oracle.Scene(**arrays), cam or es.camera(oracle, name, p), p["W"], p["H"], p["spp"],
                                 p["max_depth"], p["t_min"], p["seed"])


@pytest.mark.parametrize("cid", ["final", "glass", "contact", "bright", "final[W=33,H=7,spp=129]", "glass[t_min=0.3]"])
def test_same_render_as_o_render(oracle, cid):
    _, name, p = es.CASE[cid]
    scene, cam = oracle.Scene(**es.build(name)), es.camera(oracle, name, p)
    img, acc, cnt = oracle.render(scene, cam, p["W"], p["H"], p["spp"], p["max_depth"], p["t_min"], p["seed"],
                                  sampler=oracle.SAMPLER_DIRECT, want_accum=True)
    img2, acc2, mg, cnt2 = _render(oracle, name, p, scene, cam)
    assert np.array_equal(img, img2) and np.array_equal(acc, acc2) and cnt == cnt2
    assert (mg >= 0).all() and np.isfinite(mg).any()


def _one_ray_margin(oracle, spheres, orig, direction, max_depth=1, t_min=1e-4):
    """the margin of a 2 x 2 frame whose every camera ray is (orig, direction): a pinhole camera with a zero-sized viewport"""
    arrays = es._scene(spheres)
    cam = oracle.Camera()
    cam.origin = oracle.v3(orig)
    cam.lower_left_corner = oracle.v3(np.add(orig, direction))
    cam.horizontal = cam.vertical = oracle.Vec3(0, 0, 0)
    cam.u, cam.v, cam.w = oracle.Vec3(1, 0, 0), oracle.Vec3(0, 1, 0), oracle.Vec3(0, 0, 1)
    cam.lens_radius = 0.0
    _, _, mg, _ = oracle.render_margins(oracle.Scene(**arrays), cam, 2, 2, 1, max_depth, t_min, 1)
    return float(mg.min())


def test_known_answers(oracle):
    mirror = ((0.0, 0.0, 0.0), 1.0, es.METAL, (1.0, 1.0, 1.0), 0.0)
    # through the centre of a mirror: the line passes r from the surface (|r^2 - 0| / (r (|o| + |oc| + r)) = 1 / 11), the
    # roots 4 and 6 are far from t_min, and the reflection goes straight back (dot(d, n) / |d| = 1)
    m = _one_ray_margin(oracle, [mirror], (0.0, 0.0, 5.0), (0.0, 0.0, -1.0))
    assert m == pytest.approx(1 / 11, rel=1e-9)
    # grazing the sphere, and missing it by the same hair (a near miss in front of nothing)
    for y in (1.0 - 1e-9, 1.0 + 1e-9):
        assert _one_ray_margin(oracle, [mirror], (0.0, y, 5.0), (0.0, 0.0, -1.0)) < 1e-9
    # from inside a glass sphere of ir 1.5, a ray that meets the wall at the critical angle: ratio sin(theta) = 1.  A ray
    # along -z from (0, y0, 0) meets the unit sphere at incidence asin(y0)
    glass = ((0.0, 0.0, 0.0), 1.0, es.GLASS, (1.0, 1.0, 1.0), 1.5)
    assert _one_ray_margin(oracle, [glass], (0.0, 1 / 1.5, 0.0), (0.0, 0.0, -1.0)) < 1e-12
    assert _one_ray_margin(oracle, [glass], (0.0, 0.3, 0.0), (0.0, 0.0, -1.0)) > 1e-2
    # a fuzz-0 mirror at incidence 89.99 degrees: the reflection leaves 1.7e-4 above the tangent plane (the absorption test)
    y0 = np.sin(np.radians(89.99))
    m = _one_ray_margin(oracle, [mirror], (0.0, y0, 5.0), (0.0, 0.0, -1.0))
    assert m < 2e-4


def _perturbed(arrays, rng):
    """every small sphere's coordinates and radius one f32 ulp up or down (coincident spheres together); large spheres
    by one ulp of the small spheres' bounding radius"""
    c = np.asarray(arrays["center"], np.float32); r = np.asarray(arrays["radius"], np.float32)
    _, inv = np.unique(np.concatenate([c, r[:, None]], 1), axis=0, return_inverse=True)
    inv = inv.reshape(-1)
    sc = rng.choice([-1.0, 1.0], (inv.max() + 1, 3))[inv]; sr = rng.choice([-1.0, 1.0], inv.max() + 1)[inv]
    out = dict(arrays)
    out["center"] = np.nextafter(c, (np.inf * sc).astype(np.float32)).astype(float)
    out["radius"] = np.nextafter(r, (np.inf * sr).astype(np.float32)).astype(float)
    big = (np.abs(r) > 8) | (np.linalg.norm(c, axis=1) + np.abs(r) > 4096)
    if big.any() and (~big).any():
        u = float(np.spacing(np.float32(max(1.0, float((np.linalg.norm(c[~big], axis=1) + np.abs(r[~big])).max())))))
        out["center"][big] = c[big] + sc[big] * u
        out["radius"][big] = r[big] + sr[big] * u
    return out


@pytest.mark.parametrize("cid", [c[0] for c in es.CASES])
def test_robust_pixels_survive_f32_perturbations(oracle, cid):
    _, name, p = es.CASE[cid]
    arrays = es.build(name)
    scene, cam = oracle.Scene(**arrays), es.camera(oracle, name, p)
    img, acc, mg, _ = _render(oracle, name, p, scene, cam)
    rob = oracle.robust_pixels(acc, mg, p["spp"])
    variants = [(oracle.Scene(**_perturbed(arrays, np.random.default_rng(k))), cam) for k in range(2)]
    variants.append((scene, es.to_dev_camera_f64(cam)))
    for k, (s2, c2) in enumerate(variants):
        img2 = _render(oracle, name, p, s2, c2)[0]
        moved = (img2[..., :3] != img[..., :3]).any(-1) & rob
        assert not moved.any(), f"variant {k}: {moved.sum()} robust pixels changed, margins {mg[moved]}"


# robust fraction floors (measured: glass 0.863, glass-inside 0.777, shells 0.800, metal 0.918, lambert 0.932, bright 0.981,
# contact 0.863, final 0.548, final-h28 0.770, grid 0.639; the sweeps 0.27 (final, 65 / 129 spp: a pixel takes the smallest
# margin of 8x as many paths) .. 0.935).  mirror-box has none: its camera is shut in a mirror, so every path runs into
# max_depth through ever-growing error, and every pixel is black -- the GPU test compares its whole frame instead.
FLOOR = {"final": 0.45, "final-h28": 0.65, "grid": 0.5, "mirror-box": 0.0}


@pytest.mark.parametrize("cid", [c[0] for c in es.CASES])
def test_robust_fraction_floor(oracle, cid):
    _, name, p = es.CASE[cid]
    _, acc, mg, _ = _render(oracle, name, p)
    frac = oracle.robust_pixels(acc, mg, p["spp"]).mean()
    floor = FLOOR.get(name, 0.65)
    if "spp=" in cid and p["spp"] > 64 or p["W"] * p["H"] <= 4:
        floor = 0.2                                     # many paths per pixel, or a frame of 4 pixels
    assert frac >= floor, frac
