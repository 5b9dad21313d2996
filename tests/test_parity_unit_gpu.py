"""GPU suite, unit level: each C-ABI batch entry point (the renderer's own __device__ functions) against the
f64 oracle on identical inputs with injected random numbers (SURVEY §8c, Appendix B).

Bar (BASELINE.json north_star): t / p / normal / scatter direction / attenuation within 1e-5 relative (absolute floor
1e-6 near zero); booleans and indices exact, on inputs that are f32-representable and away from knife edges
(classified below).  precision=F64 runs the same kernels in double: bar 1e-12.
"""
import numpy as np
import pytest

from conftest import final_camera, rel_err

pytestmark = pytest.mark.gpu

TOL = {0: 1e-5, 1: 1e-12}          # capi.F32 / capi.F64


def f32(a):
    return np.asarray(a, np.float32).astype(np.float64)


def not_grazing(c, r, o, d, thr=2e-3):
    """knife-edge classifier for a (sphere, ray) pair: the reference's discriminant (sphere.rs:24) over a, i.e.
    r^2 - dist(centre, line)^2, must not be within thr * r^2 of zero — there sqrt() amplifies any rounding without bound."""
    c, o, d = np.asarray(c, float), np.asarray(o, float), np.asarray(d, float)
    oc = o - c; a = (d * d).sum(-1); hb = (oc * d).sum(-1); cc = (oc * oc).sum(-1) - r * r
    return np.abs((hb * hb - a * cc) / a) > thr * r * r


def t_err(got_t, ref_t, o, d, c):
    """error of a root t, relative to max(t, 10 % of the lengths it is computed from, in the same units).
    t is the difference of two lengths of size ~|o - c| / |d| (sphere.rs:28), so with f32 inputs its absolute error cannot
    be below ~eps32 * |o - c| / |d|; `1e-5 relative` is therefore meant for hits that are not a hair away from the origin."""
    o, d, c = np.asarray(o, float), np.asarray(d, float), np.asarray(c, float)
    # lengths that enter the subtraction: |o - c|, and the coordinates themselves (one f32 ulp of |o| ~ 10 is 1e-6)
    lengths = np.maximum(np.linalg.norm(o - c, axis=-1), 0.1 * np.linalg.norm(o, axis=-1))
    # 10 %: an origin a hair inside/outside a surface makes t = tca +- sq a cancellation of two numbers ~|o - c|; ten f32
    # roundings of that size (6e-8 each) are the floor of ANY f32 evaluation, i.e. ~1e-6 * |o - c| absolute
    scale = np.maximum(np.abs(ref_t), 0.10 * lengths / np.linalg.norm(d, axis=-1))
    return np.abs(np.asarray(got_t) - np.asarray(ref_t)) / scale


def vec_err(a, b, floor=1e-6):
    """error of a vector relative to its length (floor — scalar or per item — for near-zero vectors; for a POSITION the
    floor is the magnitude of the coordinates it was computed from: f32 cannot place a point finer than eps32 * |coords|)"""
    a, b = np.asarray(a, float), np.asarray(b, float)
    return np.linalg.norm(a - b, axis=-1) / np.maximum(np.linalg.norm(b, axis=-1), floor)


def f32_scene(arrays):
    """the scene with every coordinate, radius and material parameter rounded to f32 — identical inputs for oracle and GPU"""
    return {k: (f32(v) if v.dtype == np.float64 else v) for k, v in arrays.items()}


@pytest.mark.parametrize("prec", [0, 1])
def test_sphere_hit(ctx, oracle, prec):
    rng = np.random.default_rng(10)
    n = 200_000
    c = f32(rng.uniform(-8, 8, (n, 3))); r = f32(rng.uniform(0.1, 2.0, n) * rng.choice([1, 1, 1, -1], n))
    o = f32(rng.uniform(-14, 14, (n, 3)))
    d = f32((c - o) * rng.uniform(0.05, 2.0, (n, 1)) + rng.normal(size=(n, 3)) * np.abs(r)[:, None] * 0.8)
    ref = oracle.sphere_hit_batch(c, r, o, d, 1e-4, np.inf)
    got = ctx.sphere_hit_batch(c, r, o, d, 1e-4, np.inf, precision=prec)
    # knife edges: grazing rays (discriminant ~ 0 relative to its terms) and roots at t_min
    safe = not_grazing(c, r, o, d) & ((ref["hit"] == 0) | (np.abs(ref["t"] - 1e-4) > 1e-5))
    assert safe.mean() > 0.97 and 0.3 < ref["hit"].mean() < 0.9
    assert np.array_equal(got["hit"][safe], ref["hit"][safe])
    m = safe & (ref["hit"] == 1)
    assert np.array_equal(got["front_face"][m], ref["front_face"][m])
    tol = TOL[prec]
    assert t_err(got["t"][m], ref["t"][m], o[m], d[m], c[m]).max() < tol
    assert vec_err(got["p"][m], ref["p"][m], np.maximum(np.linalg.norm(o[m], axis=1), np.linalg.norm(c[m], axis=1))).max() < tol
    # outward_normal = (p - c) / r (sphere.rs:37): the position error over the radius, PER ITEM: 1e-5 * kappa, kappa = max(1, 0.25 M / |r|)
    M = np.maximum(np.linalg.norm(o[m], axis=1), np.linalg.norm(c[m], axis=1))
    kappa = np.maximum(1.0, 0.25 * M / np.abs(r[m]))
    assert (np.abs(got["normal"][m] - ref["normal"][m]).max(axis=1) / kappa).max() < (tol if prec == 0 else 5e-12)    # measured 5.3e-6 / 8.5e-13


@pytest.mark.parametrize("prec", [0, 1])
def test_sphere_hit_edge_cases(ctx, oracle, prec):
    """the reference's own special cases: inside origin, tangent, t_max inclusive, negative radius, far sphere"""
    c = [[0, 0, 0]] * 6 + [[0, -1000, 0]]
    r = [1, 1, 1, 1, -1, 1, 1000]
    o = [[0, 0, -5], [0, 0, 0], [0, 0, -5], [0, 0, -5], [0, 0, -5], [2, 0, -5], [1, 3, 2]]
    d = [[0, 0, 2], [1, 0, 0], [0, 0, 1], [0, 0, 1], [0, 0, 1], [0, 0, 1], [0.25, -1, 0.5]]
    tmax = [np.inf, np.inf, 4.0, 3.5, np.inf, np.inf, np.inf]
    ref = oracle.sphere_hit_batch(c, r, o, d, 1e-4, tmax)
    got = ctx.sphere_hit_batch(c, r, o, d, 1e-4, tmax, precision=prec)
    assert list(ref["hit"]) == [1, 1, 1, 0, 1, 0, 1]
    assert np.array_equal(got["hit"], ref["hit"]) and np.array_equal(got["front_face"], ref["front_face"])
    m = ref["hit"] == 1
    cm, om, dm = np.asarray(c, float)[m], np.asarray(o, float)[m], np.asarray(d, float)[m]
    assert t_err(got["t"][m], ref["t"][m], om, dm, cm).max() < TOL[prec]      # 1e-5 * kappa_t per item (r = 1000: t is a difference of lengths ~1000)
    rm = np.abs(np.asarray(r, float)[m])
    kappa = np.maximum(1.0, 0.25 * np.maximum(np.linalg.norm(om, axis=1), np.linalg.norm(cm, axis=1)) / rm)
    assert (np.abs(got["normal"][m] - ref["normal"][m]).max(axis=1) / kappa).max() < (1e-5 if prec == 0 else 1e-12)


@pytest.mark.parametrize("prec", [0, 1])
def test_hitlist_closest_hit(ctx_final, oracle, final_scene, prec):
    """HittableList::hit through the renderer's scan (packed filter + candidates + f64 ground)."""
    arrays = f32_scene(final_scene[0]); sc = oracle.Scene(**arrays)
    ctx_final.upload_scene(**arrays)
    rng = np.random.default_rng(11)
    cam = final_camera(oracle, 16 / 9)
    n1 = 60_000
    prim = oracle.get_ray_batch(cam, rng.uniform(0, 1, n1), rng.uniform(0, 1, n1), rng.uniform(-0.7, 0.7, (n1, 2)))
    # secondary-like rays: origins on sphere surfaces / the ground, random directions and lengths
    n2 = 60_000
    k = rng.integers(1, sc.n, n2)
    nrm = rng.normal(size=(n2, 3)); nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    so = arrays["center"][k] + nrm * arrays["radius"][k][:, None] * 1.05      # on-surface origins: see the ray_color / image tests
    sd = rng.normal(size=(n2, 3)) * rng.uniform(0.05, 2.0, (n2, 1))
    go = np.stack([rng.uniform(-11, 11, n2 // 2), np.full(n2 // 2, 2e-3), rng.uniform(-11, 11, n2 // 2)], 1)
    gd = rng.normal(size=(n2 // 2, 3)) * [1, 0.3, 1]
    o = f32(np.concatenate([prim["orig"], so, go])); d = f32(np.concatenate([prim["dir"], sd, gd]))
    ref = oracle.world_hit_batch(sc, o, d)
    got = ctx_final.hitlist_batch(o, d, 1e-4, precision=prec)
    agree = got["index"] == np.where(ref["hit"] == 1, ref["index"], -1)
    # disagreements may only be knife edges: silhouettes / t ~ t_min.  Count them, bound them, inspect them.
    assert agree.mean() > (0.9995 if prec == 0 else 0.999999), f"closest-hit index disagrees on {(~agree).sum()} of {len(o)} rays"
    m = agree & (ref["hit"] == 1)
    hi = np.maximum(ref["index"], 0)
    m &= not_grazing(arrays["center"][hi], arrays["radius"][hi], o, d) & (np.abs(ref["t"] - 1e-4) > 1e-5)
    assert 0.5 < m.mean() < 0.99
    tol = TOL[prec] if prec == 0 else 1e-8          # f64: two algebraically equal forms of the discriminant differ by conditioning
    te = t_err(got["t"][m], ref["t"][m], o[m], d[m], arrays["center"][hi][m])
    assert te.max() < tol, te.max()
    assert vec_err(got["p"][m], ref["p"][m], np.linalg.norm(o[m], axis=1)).max() < tol
    assert np.array_equal(got["front_face"][m], ref["front_face"][m])
    # normal = (p - c) / r: 1e-5 * kappa per item, kappa = max(1, 0.25 M / |r|) (measured max 5.6e-6 conditioned, 3.8e-5 raw)
    Cm, Rm = arrays["center"][hi][m], np.abs(arrays["radius"][hi][m])
    kappa = np.maximum(1.0, 0.25 * np.maximum(np.maximum(np.linalg.norm(o[m], axis=1), np.linalg.norm(Cm, axis=1)), np.linalg.norm(ref["p"][m], axis=1)) / Rm)
    assert (np.abs(got["normal"][m] - ref["normal"][m]).max(axis=1) / kappa).max() < (1e-5 if prec == 0 else 2e-11)
    assert np.array_equal(got["hit"], (got["index"] >= 0).astype(np.int32))


def test_hitlist_ties_and_order(ctx, oracle):
    """exact ties -> later list index wins (Appendix C.2), for small (f32) and big (f64) spheres alike"""
    center = [[0, 0, 0], [0, 0, 0], [0, 0, 10], [0, 0, 0], [0, -100, 0], [0, -100, 0]]
    radius = [1, 1, 1, 0.5, 99, 99]
    sc = oracle.Scene(center, radius, [0] * 6, [0], [[1, 1, 1]], [0])
    ctx.upload_scene(center, radius, [0] * 6, [0], [[1, 1, 1]], [0])
    o = [[0, 0, -5], [0, 0, 20], [3, 5, 0.5]]; d = [[0, 0, 1], [0, 0, -1], [0, -1, 0]]
    ref = oracle.world_hit_batch(sc, o, d)
    for prec in (0, 1):
        got = ctx.hitlist_batch(o, d, 1e-4, precision=prec)
        assert list(ref["index"]) == [1, 2, 5] and np.array_equal(got["index"], ref["index"])
        assert rel_err(got["t"], ref["t"]).max() < TOL[prec]


@pytest.mark.parametrize("backend", ["fp32", "tensor"])
@pytest.mark.parametrize("n_spheres", [0, 1, 31, 32, 33, 1024 + 7])
def test_hitlist_ragged_scene_sizes(ctx, capi, oracle, n_spheres, backend):
    """empty world, sizes straddling the 32-sphere word and the 1024-sphere segment, on each filter (SCAN_AUTO would pick the
    tensor filter for all of them)"""
    rng = np.random.default_rng(n_spheres)
    c = f32(rng.uniform(-6, 6, (n_spheres, 3))); r = f32(rng.uniform(0.05, 0.6, n_spheres))
    sc = oracle.Scene(c, r, np.zeros(n_spheres, np.uint32), [0], [[1, 1, 1]], [0])
    ctx.upload_scene(c, r, np.zeros(n_spheres, np.uint32), [0], [[1, 1, 1]], [0])
    o = f32(rng.uniform(-9, 9, (5000, 3))); d = f32(rng.normal(size=(5000, 3)))
    ref = oracle.world_hit_batch(sc, o, d)
    ctx.set_scan_backend(capi.SCAN_TENSOR if backend == "tensor" else capi.SCAN_FP32)
    try:
        if backend == "tensor" and n_spheres == 0:          # an empty world does not qualify for the tensor filter
            with pytest.raises(capi.RtiowError) as e:
                ctx.hitlist_batch(o, d, 1e-4)
            assert e.value.code == capi.ERR_UNSUPPORTED
            return
        got = ctx.hitlist_batch(o, d, 1e-4)
    finally:
        ctx.set_scan_backend(capi.SCAN_AUTO)
    want = np.where(ref["hit"] == 1, ref["index"], -1)
    assert (got["index"] == want).mean() > 0.999
    m = (got["index"] == want) & (want >= 0)
    if m.any():
        hi = np.maximum(want, 0)
        m &= not_grazing(c[hi], r[hi], o, d)
        assert t_err(got["t"][m], ref["t"][m], o[m], d[m], c[hi][m]).max() < 1e-5


def test_hitlist_filter_line_point_far_and_degenerate_origins(ctx_final, oracle, final_scene):
    """The f32 filter replaces the ray origin by the point where the ray's LINE enters the scene's bounding R-sphere
    (rt_scene.cuh, make_filter_ray).  Exercise the geometry of that construction: origins 30 ... 2000 units away (|o| >> R),
    the coordinate origin itself, origins outside the R-sphere looking away, and lines that miss the R-sphere altogether.
    A filter that dropped a true hit would show up as a wrong / missing index on a ROBUST hit (chord well inside the sphere)."""
    arrays = f32_scene(final_scene[0]); sc = oracle.Scene(**arrays)
    ctx_final.upload_scene(**arrays)
    rng = np.random.default_rng(23)
    n = 40_000
    k = rng.integers(1, sc.n, n)                                   # aim at (a point inside) sphere k
    inside = rng.normal(size=(n, 3)); inside *= (rng.uniform(0, 0.6, (n, 1)) / np.linalg.norm(inside, axis=1, keepdims=True))
    target = arrays["center"][k] + inside * np.abs(arrays["radius"][k])[:, None]
    u = rng.normal(size=(n, 3)); u[:, 1] = np.abs(u[:, 1]) * 0.5 + 0.05; u /= np.linalg.norm(u, axis=1, keepdims=True)   # from above the ground
    L = 10 ** rng.uniform(1.5, 3.3, (n, 1))
    far_o = target + u * L; far_d = -u * rng.uniform(0.3, 3.0, (n, 1))
    zero_o = np.zeros((2000, 3)); zero_d = rng.normal(size=(2000, 3))
    away_o = far_o[:2000]; away_d = -far_d[:2000]
    perp = np.cross(u[:2000], rng.normal(size=(2000, 3)))          # lines passing ~L away from the scene
    o = f32(np.concatenate([far_o, zero_o, away_o, far_o[:2000]])); d = f32(np.concatenate([far_d, zero_d, away_d, perp]))
    ref = oracle.world_hit_batch(sc, o, d)
    got = ctx_final.hitlist_batch(o, d, 1e-4)
    want = np.where(ref["hit"] == 1, ref["index"], -1)
    hi = np.maximum(want, 0)
    dist = np.linalg.norm(o - arrays["center"][hi], axis=1)
    # robust: the chord is deep inside the sphere, by far more than f32 can misplace a line through an origin `dist` away
    robust = (want >= 0) & not_grazing(arrays["center"][hi], arrays["radius"][hi], o, d, thr=0.2) & (dist * 1e-6 < 0.02 * np.abs(arrays["radius"][hi]))
    assert robust[:n].mean() > 0.5
    # the only excuse for a different winner is that the GPU's winner is itself a knife edge: a sphere in FRONT whose
    # silhouette the line touches within what f32 can resolve from `dist` away (|disc|/a below ~4 r dist 1e-6)
    gi = np.maximum(got["index"], 0)
    cg, rg = arrays["center"][gi], arrays["radius"][gi]
    oc = o - cg; a = (d * d).sum(1)
    disc_g = ((oc * d).sum(1) ** 2 - a * ((oc * oc).sum(1) - rg * rg)) / a
    knife = (got["index"] >= 0) & (np.abs(disc_g) < np.maximum(2e-3 * rg * rg, 4e-6 * np.abs(rg) * np.linalg.norm(oc, axis=1)))
    lost = robust & (got["index"] != want) & ~knife
    assert not lost.any(), f"{lost.sum()} robust hits lost or misplaced"
    assert (got["index"] == want).mean() > 0.995
    tail_w, tail_g = want[n + 2000:], got["index"][n + 2000:]          # looking away / passing far off: sky or the (f64) ground, never a small sphere
    assert (tail_w <= 0).all() and (tail_w == -1).mean() > 0.4 and np.array_equal(tail_g, tail_w)


def test_hitlist_scene_far_from_coordinate_origin(ctx, oracle):
    """a scene centred 360 units from the coordinate origin: the bounding R-sphere is large, the filter's slack balloons
    (more candidates), but every robust hit must still be found — the filter may only err towards keeping a sphere"""
    rng = np.random.default_rng(5)
    n_s = 300
    off = np.array([300.0, 50.0, -200.0])
    c = f32(off + rng.uniform(-8, 8, (n_s, 3))); r = f32(rng.uniform(0.1, 0.8, n_s))
    sc = oracle.Scene(c, r, np.zeros(n_s, np.uint32), [0], [[1, 1, 1]], [0])
    ctx.upload_scene(c, r, np.zeros(n_s, np.uint32), [0], [[1, 1, 1]], [0])
    n = 20_000
    k = rng.integers(0, n_s, n)
    u = rng.normal(size=(n, 3)); u /= np.linalg.norm(u, axis=1, keepdims=True)
    o = f32(c[k] + u * rng.uniform(2, 40, (n, 1)) + rng.normal(size=(n, 3)) * 0.3 * r[k][:, None]); d = f32(-u * rng.uniform(0.5, 2, (n, 1)))
    ref = oracle.world_hit_batch(sc, o, d)
    got = ctx.hitlist_batch(o, d, 1e-4)
    want = np.where(ref["hit"] == 1, ref["index"], -1)
    hi = np.maximum(want, 0)
    robust = (want >= 0) & not_grazing(c[hi], r[hi], o, d, thr=0.2)            # coordinates ~360: one f32 ulp is 3e-5, r >= 0.1
    assert robust.mean() > 0.4
    assert np.array_equal(got["index"][robust], want[robust])
    assert (got["index"] == want).mean() > 0.99


def test_hitlist_many_candidates_per_ray(ctx, oracle):
    """a ray threading a long row of spheres overflows the per-lane candidate list (RT_CAND_CAP) — still exact"""
    n = 200
    c = np.stack([np.arange(n) * 0.5, np.zeros(n), np.zeros(n)], 1); r = np.full(n, 0.2)
    sc = oracle.Scene(c, r, np.zeros(n, np.uint32), [0], [[1, 1, 1]], [0])
    ctx.upload_scene(c, r, np.zeros(n, np.uint32), [0], [[1, 1, 1]], [0])
    o = [[-3, 0.01, 0.02], [200, 0.0, 0.01], [50.25, 3, 0]]; d = [[1, 0, 0], [-1, 0, 0], [0.3, -1, 0]]
    ref = oracle.world_hit_batch(sc, o, d)
    got = ctx.hitlist_batch(o, d, 1e-4)
    assert np.array_equal(got["index"], ref["index"]) and list(ref["index"][:2]) == [0, n - 1]
    assert rel_err(got["t"], ref["t"]).max() < 1e-5


@pytest.mark.parametrize("prec", [0, 1])
def test_scatter(ctx, oracle, prec):
    rng = np.random.default_rng(12)
    n = 150_000
    nrm = rng.normal(size=(n, 3)); nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    rd = rng.normal(size=(n, 3)) * rng.uniform(0.05, 3, (n, 1))
    rd = np.where(((rd * nrm).sum(1) > 0)[:, None], -rd, rd)
    nrm, rd = f32(nrm), f32(rd)
    smp = rng.normal(size=(n, 3)); smp *= (rng.uniform(0, 1, (n, 1)) ** (1 / 3)) / np.linalg.norm(smp, axis=1, keepdims=True)
    smp = f32(smp)
    kind = rng.integers(0, 3, n)
    smp[kind == 2] = f32(np.stack([rng.uniform(0, 1, (kind == 2).sum())] + [np.zeros((kind == 2).sum())] * 2, 1))
    alb = f32(rng.uniform(0, 1, (n, 3))); p = f32(rng.uniform(-10, 10, (n, 3))); ff = rng.integers(0, 2, n)
    param = f32(np.where(kind == 1, rng.uniform(0, 1.2, n), rng.uniform(1.2, 2.4, n)))
    ref = oracle.scatter_batch(kind, alb, param, p, rd, p, nrm, ff, smp)
    got = ctx.scatter_batch(kind, alb, param, p, rd, p, nrm, ff, smp, precision=prec)
    # knife edges: metal absorption boundary dir.n ~ 0; dielectric TIR boundary and R ~ xi; Lambertian dir ~ 0
    dn = (ref["dir"] * nrm).sum(1)
    ud = rd / np.linalg.norm(rd, axis=1, keepdims=True)
    cos_t = np.minimum(1.0, -(ud * nrm).sum(1)); sin_t = np.sqrt(np.maximum(0, 1 - cos_t ** 2))
    ratio = np.where(ff == 1, 1 / param, param)
    r0 = ((1 - ratio) / (1 + ratio)) ** 2; R = r0 + (1 - r0) * (1 - cos_t) ** 5
    edge = ((kind == 1) & (np.abs(dn) < 1e-3)) | ((kind == 2) & ((np.abs(ratio * sin_t - 1) < 1e-3) | (np.abs(R - smp[:, 0]) < 1e-3))) \
        | ((kind == 0) & (np.linalg.norm(ref["dir"], axis=1) < 1e-2))
    s = ~edge
    assert s.mean() > 0.98
    assert np.array_equal(got["some"][s], ref["some"][s])
    m = s & (ref["some"] == 1)
    tol = TOL[prec]
    assert vec_err(got["dir"][m], ref["dir"][m]).max() < tol, vec_err(got["dir"][m], ref["dir"][m]).max()
    assert rel_err(got["attenuation"][m], ref["attenuation"][m]).max() < tol
    assert np.array_equal(got["orig"], p)


@pytest.mark.parametrize("prec", [0, 1])
def test_get_ray_to_rgba_reflect_refract(ctx, capi, oracle, prec):
    rng = np.random.default_rng(13)
    args = ((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, 16 / 9, 0.1, 10.0)
    ocam, gcam = oracle.camera_new(*args), capi.camera_new(*args)
    n = 100_000
    s, t, disk = f32(rng.uniform(0, 1.001, n)), f32(rng.uniform(0, 1.001, n)), f32(rng.uniform(-0.7, 0.7, (n, 2)))
    ref = oracle.get_ray_batch(ocam, s, t, disk); got = ctx.get_ray_batch(gcam, s, t, disk, precision=prec)
    assert vec_err(got["orig"], ref["orig"]).max() < TOL[prec] and vec_err(got["dir"], ref["dir"]).max() < TOL[prec]
    # to_rgba: exact bytes except where sqrt(c/spp)*256 sits within f32 rounding of an integer
    col = f32(rng.uniform(0, 520, (n, 3))); col[:50] = [[500, 125, 0]] * 50; col[50:60] = np.nan; col[60:70] = -1.0
    refb = oracle.to_rgba_batch(col, 255, 500); gotb = ctx.to_rgba_batch(col, 255, 500, precision=prec)
    v = 256 * np.sqrt(np.clip(col / 500, 0, None)); near = np.abs(v - np.round(v)) < (1e-3 if prec == 0 else 1e-9)
    near = np.concatenate([near, np.zeros((n, 1), bool)], 1)
    assert np.array_equal(gotb[~near], refb[~near]) and np.abs(gotb.astype(int) - refb.astype(int)).max() <= 1
    assert list(gotb[0]) == [255, 128, 0, 255] and list(gotb[55]) == [0, 0, 0, 255] and list(gotb[65]) == [0, 0, 0, 255]
    # reflect / refract
    v3 = f32(rng.normal(size=(n, 3))); nn = rng.normal(size=(n, 3)); nn = f32(nn / np.linalg.norm(nn, axis=1, keepdims=True))
    assert vec_err(ctx.reflect_batch(v3, nn, precision=prec), oracle.reflect_batch(v3, nn)).max() < TOL[prec]
    uv = v3 / np.linalg.norm(v3, axis=1, keepdims=True); uv = f32(np.where(((uv * nn).sum(1) > 0)[:, None], -uv, uv))
    eta = f32(rng.choice([1 / 1.5, 1.5, 1 / 2.4], n))
    ok = eta * np.sqrt(np.maximum(0, 1 - (uv * nn).sum(1) ** 2)) < 0.999        # away from |1-|perp|^2| ~ 0
    # refract's parallel part is -sqrt|1 - |perp|^2| n (vec3.rs:123): kappa = max(1, 0.1 / sqrt|1 - |perp|^2|) per item (measured 9.4e-7)
    q = np.abs(1 - eta * eta * np.maximum(0, 1 - (uv * nn).sum(1) ** 2))[ok]
    kappa = np.maximum(1.0, 0.1 / np.sqrt(q))
    assert (vec_err(ctx.refract_batch(uv, nn, eta, precision=prec)[ok], oracle.refract_batch(uv, nn, eta)[ok]) / kappa).max() < TOL[prec]


def test_sampler_mapping(ctx, oracle):
    """Philox block (seed; pixel, sample, bounce) -> uniforms -> disk / unit vector / ball: GPU == oracle"""
    import ctypes as C
    rng = np.random.default_rng(14)
    n = 4000
    pix, smp, bnc = rng.integers(0, 2 ** 32, n, dtype=np.uint64), rng.integers(0, 2 ** 20, n), rng.integers(0, 51, n)
    seed = 0xDEADBEEF12345678
    L = oracle.lib()
    for prec, tol in ((0, 2e-6), (1, 1e-14)):
        out = ctx.sampler_batch(pix, smp, bnc, seed, precision=prec)
        for i in range(0, n, 13):
            u = oracle.direct_uniforms(seed, int(pix[i]), int(smp[i]), int(bnc[i]))
            assert np.array_equal(out[i, :4], u)                       # 24-bit uniforms are bit-identical
            dx, dy = C.c_double(), C.c_double(); L.o_direct_disk(u[2], u[3], C.byref(dx), C.byref(dy))
            want = np.concatenate([[dx.value, dy.value], L.o_direct_unit_vector(u[0], u[1]).np(), L.o_direct_in_unit_sphere(u[0], u[1], u[2]).np()])
            assert np.abs(out[i, 4:] - want).max() < tol


@pytest.mark.parametrize("prec", [0, 1])
def test_ray_color_iterative_vs_recursive(ctx_final, oracle, final_scene, prec):
    """ray_color (main.rs:38-57): the GPU's iterative bounce loop == the oracle's recursion on the same Philox blocks."""
    arrays = f32_scene(final_scene[0]); sc = oracle.Scene(**arrays)
    ctx_final.upload_scene(**arrays)
    rng = np.random.default_rng(15)
    cam = final_camera(oracle, 16 / 9)
    n = 40_000
    r = oracle.get_ray_batch(cam, rng.uniform(0, 1, n), rng.uniform(0, 1, n), rng.uniform(-0.7, 0.7, (n, 2)))
    o, d = f32(r["orig"]), f32(r["dir"])
    pix = rng.integers(0, 2 ** 31, n).astype(np.uint32); smp = rng.integers(0, 500, n).astype(np.uint32)
    ref = oracle.ray_color_batch(sc, o, d, pix, smp, seed=77)
    got = ctx_final.ray_color_batch(o, d, pix, smp, seed=77, precision=prec)
    same = got["rays"] == ref["rays"]
    err = np.abs(got["color"] - ref["color"]).max(axis=1)
    if prec == 1:
        assert same.mean() > 0.9999 and np.percentile(err, 99.9) < 1e-9
    else:
        # f32 rounding can flip a knife-edge decision and send the path elsewhere: rare, and unbiased
        assert same.mean() > 0.995, same.mean()
        assert np.median(err[same]) < 1e-6 and np.percentile(err[same], 99) < 1e-4
        assert abs(got["color"].mean() - ref["color"].mean()) < 2e-3
    assert int(ref["rays"].max()) <= 50 and got["rays"].max() <= 50
    assert abs(got["rays"].mean() - ref["rays"].mean()) < 0.02
