"""GPU suite: the parity REPORT (VERDICT r1 weak #1).  Every unit-level quantity of north_star's first parity level —
intersection t / p / normal / front_face, closest-hit index, per-material scatter direction / attenuation, get_ray, reflect,
refract — is compared with the f64 oracle on identical f32-representable inputs, and for each the test RECORDS

    max and 99.9th-percentile error, raw and conditioned, in f32 and in f64; the fraction of items excluded as knife edges and why

into $RTIOW_REPORT_DIR/parity_r2.json when that variable is set (committed copy: profiles/parity_r2.json).  Assertions are stated as `1e-5 * kappa_i` with the
conditioning factor kappa_i computed PER ITEM, never as a flat loosened tolerance:

  t       kappa = max(1, 0.1 L / (|t| |d|)),  L = max(|o - c|, 0.1 |o|): t is the difference of two lengths of size ~L
          (sphere.rs:28: (-half_b - sqrtd) / a), so ten f32 roundings of L are the floor of ANY f32 evaluation of a small t
  p       relative to M = max(|o|, |c|): f32 cannot place a point finer than eps32 times its coordinates      (kappa = 1)
  normal  kappa = max(1, 0.25 M / |r|): outward_normal = (p - c) / r (sphere.rs:37) divides the position error by the radius
  scatter direction / attenuation, get_ray, reflect, refract: relative to the vector's length                  (kappa = 1)

and each conditioned bound is min(1e-5, 2 x the maximum this file measured on the B200) — BOUND_F32 below, measured values in
profiles/parity_r2.json.
The same kernels run in f64 to 1e-12 (conditioned), which separates "the algorithm differs" from "f32 rounds".
Also here: the Lambertian near-zero guard (vec3.rs:111-114, materials.rs:24-27) on inputs that hit it on BOTH sides.
"""
import json
import os
from pathlib import Path

import numpy as np
import pytest

from conftest import final_camera

pytestmark = pytest.mark.gpu

REPORT = {}
OUT = Path(os.environ["RTIOW_REPORT_DIR"]) / "parity_r2.json" if os.environ.get("RTIOW_REPORT_DIR") else None

# conditioned bounds asserted for f32 (units of north_star's 1e-5 bar) and what was measured on the B200 (profiles/parity_r2.json)
BAR = 1e-5
F64_BAR = 1e-12
# f32, conditioned: min(BAR, 2 x measured maximum) [measured on B200, round 2: profiles/parity_r2.json]
BOUND_F32 = {
    "sphere_hit.t": 2.1e-6,          # measured 1.04e-6
    "sphere_hit.p": 4.2e-6,          # 2.07e-6
    "sphere_hit.normal": 1.0e-5,     # 5.3e-6
    "hitlist.t": 1.0e-5,             # 6.18e-6
    "hitlist.p": 1.3e-6,             # 6.35e-7
    "hitlist.normal": 1.0e-5,        # 5.6e-6 with kappa 0.1 M/|r|; smaller with 0.25
    "scatter.lambertian.direction": 5.2e-6,   # 2.59e-6
    "scatter.metal.direction": 3.1e-6,        # 1.55e-6
    "scatter.dielectric.direction": 4.0e-6,   # 2.00e-6
    "get_ray.orig": 7.4e-8,          # 3.69e-8
    "get_ray.dir": 3.6e-7,           # 1.77e-7
    "reflect": 5.4e-7,               # 2.65e-7
    "refract": 1.9e-6,               # 9.35e-7
}
F64_BOUND = {"sphere_hit.normal": 5e-12, "hitlist.normal": 2e-11}     # f64 normals: (p - c) / r at |p| ~ 15, r = 0.2 (measured 2.1e-12 / 8e-12)


def f32(a):
    return np.asarray(a, np.float32).astype(np.float64)


def record(name, prec, raw, cond, kappa=None, excluded=0.0, why="", n=None):
    raw, cond = np.asarray(raw, float).ravel(), np.asarray(cond, float).ravel()
    e = {"n": int(n if n is not None else len(raw)), "raw_max": float(raw.max()), "raw_p999": float(np.percentile(raw, 99.9)),
         "conditioned_max": float(cond.max()), "conditioned_p999": float(np.percentile(cond, 99.9)),
         "kappa_max": float(np.max(kappa)) if kappa is not None else 1.0,
         "kappa_gt1_fraction": float(np.mean(np.asarray(kappa) > 1)) if kappa is not None else 0.0,
         "excluded_fraction": float(excluded), "excluded_why": why}
    REPORT.setdefault(name, {})["f64" if prec else "f32"] = e
    if OUT is None:
        return e
    OUT.parent.mkdir(parents=True, exist_ok=True)
    OUT.write_text(json.dumps({"bar": BAR, "what": "unit-level parity of the CUDA path against the f64 oracle; conditioned = error / kappa (see tests/test_parity_report_gpu.py)",
                               "quantities": REPORT}, indent=1, sort_keys=True))
    return e


def grazing(c, r, o, d, thr=2e-3):
    """|discriminant / a| (sphere.rs:24) within thr r^2 of zero: sqrt() there amplifies any rounding without bound"""
    oc = o - c; a = (d * d).sum(-1); hb = (oc * d).sum(-1); cc = (oc * oc).sum(-1) - r * r
    return np.abs((hb * hb - a * cc) / a) <= thr * r * r


def kappa_t(t, o, d, c):
    L = np.maximum(np.linalg.norm(o - c, axis=-1), 0.1 * np.linalg.norm(o, axis=-1))
    return np.maximum(1.0, 0.1 * L / np.maximum(np.abs(t) * np.linalg.norm(d, axis=-1), 1e-300))


def check(e, prec, name):
    lim = F64_BOUND.get(name, F64_BAR) if prec else BOUND_F32[name]
    assert lim <= BAR and e["conditioned_max"] <= lim, (name, e, lim)


@pytest.mark.parametrize("prec", [0, 1])
def test_report_sphere_hit(ctx, oracle, prec):
    """Sphere::hit + HitRecord::new (sphere.rs:16-41, mod.rs:20-30)"""
    rng = np.random.default_rng(10)
    n = 400_000
    c = f32(rng.uniform(-8, 8, (n, 3))); r = f32(rng.uniform(0.1, 2.0, n) * rng.choice([1, 1, 1, -1], n))
    o = f32(rng.uniform(-14, 14, (n, 3)))
    d = f32((c - o) * rng.uniform(0.05, 2.0, (n, 1)) + rng.normal(size=(n, 3)) * np.abs(r)[:, None] * 0.8)
    ref = oracle.sphere_hit_batch(c, r, o, d, 1e-4, np.inf)
    got = ctx.sphere_hit_batch(c, r, o, d, 1e-4, np.inf, precision=prec)
    edge = grazing(c, r, o, d) | ((ref["hit"] == 1) & (np.abs(ref["t"] - 1e-4) <= 1e-5))
    why = "grazing: |disc/a| <= 2e-3 r^2 (sqrt amplifies rounding without bound); root within 1e-5 of t_min"
    assert edge.mean() < 0.01, edge.mean()                    # measured 0.3 %
    s = ~edge
    assert np.array_equal(got["hit"][s], ref["hit"][s])
    m = s & (ref["hit"] == 1)
    assert np.array_equal(got["front_face"][m], ref["front_face"][m])
    kt = kappa_t(ref["t"][m], o[m], d[m], c[m])
    raw_t = np.abs(got["t"][m] - ref["t"][m]) / np.abs(ref["t"][m])
    check(record("sphere_hit.t", prec, raw_t, raw_t / kt, kt, edge.mean(), why), prec, "sphere_hit.t")
    M = np.maximum(np.linalg.norm(o[m], axis=1), np.linalg.norm(c[m], axis=1))
    raw_p = np.linalg.norm(got["p"][m] - ref["p"][m], axis=1) / M
    check(record("sphere_hit.p", prec, raw_p, raw_p, None, edge.mean(), why), prec, "sphere_hit.p")
    kn = np.maximum(1.0, 0.25 * M / np.abs(r[m]))
    raw_n = np.abs(got["normal"][m] - ref["normal"][m]).max(axis=1)
    check(record("sphere_hit.normal", prec, raw_n, raw_n / kn, kn, edge.mean(), why), prec, "sphere_hit.normal")
    record("sphere_hit.hit_and_front_face", prec, np.zeros(1), np.zeros(1), None, edge.mean(), why + "; exact on the rest", n=int(s.sum()))


@pytest.mark.parametrize("prec", [0, 1])
def test_report_hitlist(ctx_final, oracle, final_scene, prec):
    """HittableList::hit (mod.rs:56-69) through the renderer's scan — tensor-core filter + precise test + f64 ground"""
    arrays = {k: (f32(v) if v.dtype == np.float64 else v) for k, v in final_scene[0].items()}
    sc = oracle.Scene(**arrays)
    ctx_final.upload_scene(**arrays)
    rng = np.random.default_rng(11)
    cam = final_camera(oracle, 16 / 9)
    n1 = 150_000
    prim = oracle.get_ray_batch(cam, rng.uniform(0, 1, n1), rng.uniform(0, 1, n1), rng.uniform(-0.7, 0.7, (n1, 2)))
    n2 = 150_000
    k = rng.integers(1, sc.n, n2)
    nrm = rng.normal(size=(n2, 3)); nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    so = arrays["center"][k] + nrm * arrays["radius"][k][:, None] * 1.05
    sd = rng.normal(size=(n2, 3)) * rng.uniform(0.05, 2.0, (n2, 1))
    go = np.stack([rng.uniform(-11, 11, n2 // 2), np.full(n2 // 2, 2e-3), rng.uniform(-11, 11, n2 // 2)], 1)
    gd = rng.normal(size=(n2 // 2, 3)) * [1, 0.3, 1]
    o = f32(np.concatenate([prim["orig"], so, go])); d = f32(np.concatenate([prim["dir"], sd, gd]))
    ref = oracle.world_hit_batch(sc, o, d)
    got = ctx_final.hitlist_batch(o, d, 1e-4, precision=prec)
    want = np.where(ref["hit"] == 1, ref["index"], -1)
    agree = got["index"] == want
    # a different winner is only excusable on a silhouette: the sphere one side found and the other did not is grazed
    other = np.where(agree, 0, np.maximum(np.maximum(got["index"], want), 0))
    excusable = agree | grazing(arrays["center"][other], arrays["radius"][other], o, d, thr=5e-3) | (np.abs(ref["t"] - 1e-4) <= 1e-5)
    assert excusable.all(), f"{(~excusable).sum()} closest-hit indices differ away from any silhouette"
    record("hitlist.index", prec, (~agree).astype(float), np.zeros(1), None, float((~agree).mean()),
           "index differs from the oracle's only where the disputed sphere is grazed (|disc/a| <= 5e-3 r^2): measured fraction", n=len(o))
    assert agree.mean() > (0.9997 if prec == 0 else 0.999999)
    hi = np.maximum(want, 0)
    C_, R_ = arrays["center"][hi], arrays["radius"][hi]
    edge = ~agree | ((want >= 0) & (grazing(C_, R_, o, d) | (np.abs(ref["t"] - 1e-4) <= 1e-5)))
    why = "index disagreement (silhouettes) or grazing |disc/a| <= 2e-3 r^2 or root within 1e-5 of t_min"
    m = ~edge & (want >= 0)
    frac = float(edge[want >= 0].mean())
    kt = kappa_t(ref["t"][m], o[m], d[m], C_[m])
    raw_t = np.abs(got["t"][m] - ref["t"][m]) / np.abs(ref["t"][m])
    check(record("hitlist.t", prec, raw_t, raw_t / kt, kt, frac, why), prec, "hitlist.t")
    M = np.maximum(np.linalg.norm(o[m], axis=1), np.linalg.norm(C_[m], axis=1))
    raw_p = np.linalg.norm(got["p"][m] - ref["p"][m], axis=1) / np.maximum(M, np.linalg.norm(ref["p"][m], axis=1))
    check(record("hitlist.p", prec, raw_p, raw_p, None, frac, why), prec, "hitlist.p")
    kn = np.maximum(1.0, 0.25 * np.maximum(M, np.linalg.norm(ref["p"][m], axis=1)) / np.abs(R_[m]))
    raw_n = np.abs(got["normal"][m] - ref["normal"][m]).max(axis=1)
    check(record("hitlist.normal", prec, raw_n, raw_n / kn, kn, frac, why), prec, "hitlist.normal")
    assert np.array_equal(got["front_face"][m], ref["front_face"][m])


@pytest.mark.parametrize("prec", [0, 1])
def test_report_scatter(ctx, oracle, prec):
    """Scatter::scatter x3 (materials.rs:22-30, 50-61, 77-104) with injected samples, per material"""
    rng = np.random.default_rng(12)
    n = 300_000
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
    dn = (ref["dir"] * nrm).sum(1)
    ud = rd / np.linalg.norm(rd, axis=1, keepdims=True)
    cos_t = np.minimum(1.0, -(ud * nrm).sum(1)); sin_t = np.sqrt(np.maximum(0, 1 - cos_t ** 2))
    ratio = np.where(ff == 1, 1 / param, param)
    r0 = ((1 - ratio) / (1 + ratio)) ** 2; R = r0 + (1 - r0) * (1 - cos_t) ** 5
    edges = {
        "lambertian": ((kind == 0) & (np.linalg.norm(ref["dir"], axis=1) < 1e-2), "|normal + unit(sample)| < 1e-2: the direction is a difference of two unit vectors"),
        "metal": ((kind == 1) & (np.abs(dn) < 1e-3), "|dir . n| < 1e-3: absorbed / scattered boundary (materials.rs:56)"),
        "dielectric": ((kind == 2) & ((np.abs(ratio * sin_t - 1) < 1e-3) | (np.abs(R - smp[:, 0]) < 1e-3)), "within 1e-3 of the TIR boundary or of R == xi (materials.rs:96)"),
    }
    for name, (edge, why) in edges.items():
        sel = kind == {"lambertian": 0, "metal": 1, "dielectric": 2}[name]
        s = sel & ~edge
        frac = float(edge[sel].mean())
        assert frac < 0.02                                     # measured: Lambertian 2e-4 %, Metal 0.13 %, Dialectric 0.33 %
        assert np.array_equal(got["some"][s], ref["some"][s]), name
        m = s & (ref["some"] == 1)
        raw = np.linalg.norm(got["dir"][m] - ref["dir"][m], axis=1) / np.maximum(np.linalg.norm(ref["dir"][m], axis=1), 1e-6)
        check(record(f"scatter.{name}.direction", prec, raw, raw, None, frac, why), prec, f"scatter.{name}.direction")
        ra = (np.abs(got["attenuation"][m] - ref["attenuation"][m]) / np.maximum(np.abs(ref["attenuation"][m]), 1e-6)).max(axis=1)
        record(f"scatter.{name}.attenuation", prec, ra, ra, None, frac, why)
        assert np.array_equal(got["attenuation"][m], ref["attenuation"][m]), name      # the albedo (f32-representable) passes through: exact
    assert np.array_equal(got["orig"], p)


@pytest.mark.parametrize("prec", [0, 1])
def test_lambertian_near_zero_guard(ctx, oracle, prec):
    """V5 is_near_zero (vec3.rs:111-114) inside Lambertian::scatter (materials.rs:24-27): sample = -normal (+ a tiny offset) on
    axis-aligned normals, where unit_vector() is exact on both sides, so the guard fires — or just does not — in f32, f64 and the
    oracle alike.  offset 0, 2^-30, 2^-27 (< 1e-8: guard -> direction = normal); 2^-26, 2^-20 (> 1e-8: the tiny vector is kept)."""
    axes = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], float)
    offs = [0.0, 2.0 ** -30, 2.0 ** -27, 2.0 ** -26, 2.0 ** -20]
    nrm, smp, guard = [], [], []
    for a in axes:
        for off in offs:
            e = np.roll(np.abs(a), 1) * off
            nrm.append(a); smp.append(-a + e); guard.append(off < 1e-8)
    nrm, smp, guard = np.array(nrm), np.array(smp), np.array(guard)
    n = len(nrm)
    assert np.array_equal(f32(smp), smp)                       # the inputs are f32-representable
    kind = np.zeros(n, int); alb = np.full((n, 3), 0.5); prm = np.zeros(n); p = np.zeros((n, 3)); rd = -nrm; ff = np.ones(n, int)
    ref = oracle.scatter_batch(kind, alb, prm, p, rd, p, nrm, ff, smp)
    got = ctx.scatter_batch(kind, alb, prm, p, rd, p, nrm, ff, smp, precision=prec)
    assert (ref["some"] == 1).all() and (got["some"] == 1).all()
    assert np.array_equal(ref["dir"][guard], nrm[guard]), "oracle: the guard must replace a near-zero direction by the normal"
    assert np.array_equal(got["dir"][guard], nrm[guard]), "GPU: the guard must replace a near-zero direction by the normal"
    k = ~guard
    assert (np.linalg.norm(ref["dir"][k], axis=1) < 1e-5).all()            # just above the guard: the tiny vector survives ...
    err = np.linalg.norm(got["dir"][k] - ref["dir"][k], axis=1) / np.linalg.norm(ref["dir"][k], axis=1)
    record("scatter.lambertian.near_zero_guard", prec, err, err, None, 0.0, "30 constructed cases: 18 fire the guard (direction == normal exactly), 12 sit just above it", n=n)
    assert err.max() <= (BAR if prec == 0 else F64_BAR)                    # ... and is the same tiny vector


@pytest.mark.parametrize("prec", [0, 1])
def test_report_get_ray_reflect_refract(ctx, capi, oracle, prec):
    """Camera::get_ray (camera.rs:47-54), Vec3::reflect / refract (vec3.rs:116-125)"""
    rng = np.random.default_rng(13)
    args = ((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, 16 / 9, 0.1, 10.0)
    ocam, gcam = oracle.camera_new(*args), capi.camera_new(*args)
    n = 200_000
    s, t, disk = f32(rng.uniform(0, 1.001, n)), f32(rng.uniform(0, 1.001, n)), f32(rng.uniform(-0.7, 0.7, (n, 2)))
    ref = oracle.get_ray_batch(ocam, s, t, disk); got = ctx.get_ray_batch(gcam, s, t, disk, precision=prec)
    for key in ("orig", "dir"):
        raw = np.linalg.norm(got[key] - ref[key], axis=1) / np.linalg.norm(ref[key], axis=1)
        check(record(f"get_ray.{key}", prec, raw, raw), prec, f"get_ray.{key}")
    v3 = f32(rng.normal(size=(n, 3))); nn = rng.normal(size=(n, 3)); nn = f32(nn / np.linalg.norm(nn, axis=1, keepdims=True))
    a, b = ctx.reflect_batch(v3, nn, precision=prec), oracle.reflect_batch(v3, nn)
    raw = np.linalg.norm(a - b, axis=1) / np.linalg.norm(b, axis=1)
    check(record("reflect", prec, raw, raw), prec, "reflect")
    uv = v3 / np.linalg.norm(v3, axis=1, keepdims=True); uv = f32(np.where(((uv * nn).sum(1) > 0)[:, None], -uv, uv))
    eta = f32(rng.choice([1 / 1.5, 1.5, 1 / 2.4], n))
    # refract's parallel part is -sqrt|1 - |perp|^2| n (vec3.rs:123): kappa = 1 / sqrt|1 - |perp|^2| near the critical angle
    sin2 = np.maximum(0, 1 - (uv * nn).sum(1) ** 2); q = np.abs(1 - eta * eta * sin2)
    edge = q < 1e-3
    kap = np.maximum(1.0, 0.1 / np.sqrt(np.maximum(q, 1e-300)))
    a, b = ctx.refract_batch(uv, nn, eta, precision=prec), oracle.refract_batch(uv, nn, eta)
    raw = (np.linalg.norm(a - b, axis=1) / np.maximum(np.linalg.norm(b, axis=1), 1e-6))[~edge]
    check(record("refract", prec, raw, raw / kap[~edge], kap[~edge], float(edge.mean()), "|1 - |r_out_perp|^2| < 1e-3: the critical angle, sqrt of a cancellation"), prec, "refract")


def test_report_is_complete():
    """runs last in this file: every quantity of north_star's first parity level has an f32 and an f64 entry"""
    need = ["sphere_hit.t", "sphere_hit.p", "sphere_hit.normal", "hitlist.index", "hitlist.t", "hitlist.p", "hitlist.normal",
            "scatter.lambertian.direction", "scatter.metal.direction", "scatter.dielectric.direction", "scatter.lambertian.attenuation",
            "scatter.metal.attenuation", "scatter.dielectric.attenuation", "scatter.lambertian.near_zero_guard", "get_ray.orig", "get_ray.dir", "reflect", "refract"]
    if not REPORT:
        pytest.skip("the report tests did not run in this session")
    for k in need:
        assert set(REPORT[k]) == {"f32", "f64"}, k
        assert REPORT[k]["f32"]["conditioned_max"] <= BAR
