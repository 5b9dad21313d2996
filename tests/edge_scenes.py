"""Scenes and parameters at the edges of the renderer's input space (test infrastructure, not a test file).

Every scene here is explicit and f32-representable, so the oracle and the CUDA library render the same inputs, and each has a
camera that sees its feature.  They cover what the C ABI accepts but random_scene never produces: glass with ir < 1, ir = 1
and ir = 2.4, a camera inside glass, concentric shells, mirrors facing each other, fuzz 1 .. 3, albedo 0 and albedo > 1
(up to a radiance sum past 2^32 per pixel), negative radii on Lambertian and Metal spheres, touching, overlapping and
coincident spheres.  `CASES` pairs scenes with render parameters: the final scene on every scan arm, and sweeps of t_min,
max_depth, spp (chunks that split a pixel), frame size and aperture on the final scene and on the glass scene.
"""
from functools import lru_cache

import numpy as np

from test_parity_unit_gpu import f32

LAMB, METAL, GLASS = 0, 1, 2
F32_TWO_THIRDS = float(np.float32(1 / 1.5))                      # an air bubble in glass of ir 1.5


def _scene(spheres):
    """[(centre, radius, kind, albedo, param)] -> the arrays of the C ABI, one material per sphere, f32-rounded"""
    c = np.array([s[0] for s in spheres], float)
    return dict(center=f32(c), radius=f32([s[1] for s in spheres]), mat_index=np.arange(len(spheres), dtype=np.uint32),
                mat_kind=np.array([s[2] for s in spheres], np.uint32), mat_albedo=f32([s[3] for s in spheres]),
                mat_param=f32([s[4] for s in spheres]))


GROUND = ((0.0, -100.0, 0.0), 100.0, LAMB, (0.5, 0.5, 0.5), 0.0)
GREY, RED, BLUE = (0.7, 0.7, 0.7), (0.8, 0.3, 0.2), (0.2, 0.4, 0.9)


def glass():
    """ir 1.5 with an air bubble (ir 1 / 1.5) inside it, ir 1.0 and ir 2.4, on a ground"""
    return _scene([GROUND,
                   ((0.0, 1.0, 0.0), 1.0, GLASS, GREY, 1.5), ((0.0, 1.0, 0.0), 0.5, GLASS, GREY, F32_TWO_THIRDS),
                   ((-2.25, 0.75, 0.5), 0.75, GLASS, GREY, 1.0), ((2.25, 0.75, 0.5), 0.75, GLASS, GREY, 2.4),
                   ((0.0, 0.5, -3.0), 0.5, LAMB, RED, 0.0)])


def glass_inside():
    """the camera inside a glass sphere of radius 3, looking at a Lambertian and a metal sphere inside it"""
    return _scene([GROUND, ((0.0, 1.0, 0.0), 3.0, GLASS, GREY, 1.5),
                   ((0.0, 0.5, -1.5), 0.5, LAMB, RED, 0.0), ((1.25, 0.75, -1.0), 0.5, METAL, BLUE, 0.25)])


def shells():
    """concentric: glass r, hollow glass -0.9 r and a Lambertian core; beside it the same shell around nothing"""
    return _scene([GROUND,
                   ((0.0, 1.0, 0.0), 1.0, GLASS, GREY, 1.5), ((0.0, 1.0, 0.0), -0.9, GLASS, GREY, 1.5),
                   ((0.0, 1.0, 0.0), 0.5, LAMB, BLUE, 0.0),
                   ((2.25, 1.0, 0.0), 1.0, GLASS, GREY, 1.5), ((2.25, 1.0, 0.0), -0.9, GLASS, GREY, 1.5)])


def metal():
    """two mirrors (fuzz 0) 0.25 apart that send rays back and forth, fuzz 1, 1.5 and 3, an albedo-0 mirror"""
    return _scene([GROUND,
                   ((-1.625, 1.5, 0.0), 1.5, METAL, (0.9, 0.9, 0.9), 0.0), ((1.625, 1.5, 0.0), 1.5, METAL, (0.9, 0.9, 0.9), 0.0),
                   ((-2.25, 0.5, 2.5), 0.5, METAL, GREY, 1.0), ((-0.75, 0.5, 2.5), 0.5, METAL, GREY, 1.5),
                   ((0.75, 0.5, 2.5), 0.5, METAL, GREY, 3.0), ((2.25, 0.5, 2.5), 0.5, METAL, (0.0, 0.0, 0.0), 0.0)])


def mirror_box():
    """the camera inside a fuzz-0 mirror sphere with a glass ball and a mirror ball: no path reaches the sky, every one
    runs to max_depth"""
    return _scene([((0.0, 0.0, 0.0), 4.0, METAL, (0.9, 0.9, 0.9), 0.0),
                   ((0.0, 0.0, -2.0), 1.0, GLASS, GREY, 1.5), ((1.5, -1.0, -1.0), 0.75, METAL, GREY, 0.0)])


def lambert():
    """albedo 0, 1, 1.5 and 2, and negative radii on a Lambertian and a metal sphere"""
    return _scene([GROUND,
                   ((-3.0, 0.5, 0.0), 0.5, LAMB, (0.0, 0.0, 0.0), 0.0), ((-1.75, 0.5, 0.0), 0.5, LAMB, (1.0, 1.0, 1.0), 0.0),
                   ((-0.5, 0.5, 0.0), 0.5, LAMB, (1.5, 1.5, 1.5), 0.0), ((0.75, 0.5, 0.0), 0.5, LAMB, (2.0, 1.0, 2.0), 0.0),
                   ((2.0, 0.5, 0.0), -0.5, LAMB, RED, 0.0), ((3.25, 0.5, 0.0), -0.5, METAL, BLUE, 0.125)])


def bright():
    """two Lambertian spheres of albedo 1000 facing each other: a path that bounces between them a few times before it
    escapes carries 1e9 and more, and a pixel's radiance sum passes 2^32"""
    return _scene([((-1.125, 0.0, 0.0), 1.0, LAMB, (1000.0, 1000.0, 1000.0), 0.0),
                   ((1.125, 0.0, 0.0), 1.0, LAMB, (1000.0, 500.0, 1000.0), 0.0)])


def contact():
    """a chain of touching spheres resting on the ground, a lens of two overlapping glass spheres, and a coincident pair
    (Lambertian first, glass second: the later index wins every tie)"""
    return _scene([GROUND,
                   ((-3.0, 0.5, 0.0), 0.5, LAMB, RED, 0.0), ((-2.0, 0.5, 0.0), 0.5, METAL, GREY, 0.0),
                   ((-1.0, 0.5, 0.0), 0.5, LAMB, BLUE, 0.0),
                   ((0.25, 0.75, 1.0), 0.75, GLASS, GREY, 1.5), ((0.875, 0.75, 1.0), 0.75, GLASS, GREY, 1.5),
                   ((2.5, 0.75, 0.0), 0.75, LAMB, RED, 0.0), ((2.5, 0.75, 0.0), 0.75, GLASS, GREY, 1.5)])


def grid(n=128, spacing=0.75):
    """n x n small spheres (r 0.2 .. 0.3, all materials) on the ground: 16 K+ spheres put the FP32 table in global memory"""
    rng = np.random.default_rng(11)
    g = (np.arange(n) - (n - 1) / 2) * spacing
    x, z = np.meshgrid(g, g, indexing="ij")
    r = rng.uniform(0.2, 0.3, n * n)
    kind = rng.choice([LAMB, METAL, GLASS], n * n, p=[0.6, 0.25, 0.15])
    alb = rng.uniform(0.1, 0.95, (n * n, 3))
    prm = np.where(kind == METAL, rng.uniform(0, 0.5, n * n), 1.5)
    sp = [GROUND] + [((x.flat[i], r[i], z.flat[i]), r[i], kind[i], alb[i], prm[i]) for i in range(n * n)]
    return _scene(sp)


def final(half_extent=11):
    from oracle.oracle import random_scene
    from test_parity_unit_gpu import f32_scene
    return f32_scene(random_scene(1, half_extent))


# name -> (builder(), camera (look_from, look_at, v_up, v_fov, aperture, focus_dist))
FINAL_VIEW = ((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, 0.1, 10.0)
SCENES = {
    "final": (lambda: final(), FINAL_VIEW),
    "final-h28": (lambda: final(28), ((40, 6, 10), (0, 0, 0), (0, 1, 0), 30.0, 0.1, 40.0)),
    "grid": (lambda: grid(), ((0, 6, 30), (0, 0, 0), (0, 1, 0), 45.0, 0.0, 30.0)),
    "glass": (lambda: glass(), ((0, 2, 8), (0, 0.8, 0), (0, 1, 0), 40.0, 0.0, 8.0)),
    "glass-inside": (lambda: glass_inside(), ((0, 1, 1.5), (0, 0.7, -1.5), (0, 1, 0), 70.0, 0.0, 3.0)),
    "shells": (lambda: shells(), ((1, 2, 6), (1, 1, 0), (0, 1, 0), 40.0, 0.0, 6.0)),
    "metal": (lambda: metal(), ((0, 2.5, 9), (0, 1, 0), (0, 1, 0), 40.0, 0.0, 9.0)),
    "mirror-box": (lambda: mirror_box(), ((0, 0.5, 2.5), (0, 0, -2), (0, 1, 0), 70.0, 0.0, 4.0)),
    "lambert": (lambda: lambert(), ((0, 2, 8), (0, 0.5, 0), (0, 1, 0), 45.0, 0.0, 8.0)),
    "bright": (lambda: bright(), ((0, 0.5, 6), (0, 0, 0), (0, 1, 0), 40.0, 0.0, 6.0)),
    "contact": (lambda: contact(), ((0, 2.5, 8), (0, 0.5, 0), (0, 1, 0), 45.0, 0.0, 8.0)),
}
EDGE = ["glass", "glass-inside", "shells", "metal", "mirror-box", "lambert", "bright", "contact"]

BASE = dict(W=48, H=27, spp=8, max_depth=50, t_min=1e-4, seed=3)


def _case(scene, **kw):
    p = {**BASE, **kw}
    tag = ",".join(f"{k}={v}" for k, v in kw.items())
    return (f"{scene}[{tag}]" if tag else scene), scene, p


def _sweeps(scene):
    return [_case(scene, t_min=t) for t in (1e-3, 1e-2, 0.3)] + \
           [_case(scene, max_depth=d) for d in (2, 3, 7, 200)] + \
           [_case(scene, W=8, H=5, spp=65), _case(scene, W=33, H=7, spp=129)] + \
           [_case(scene, W=2, H=2), _case(scene, W=2, H=9), _case(scene, W=37, H=11)] + \
           [_case(scene, aperture=0.0), _case(scene, aperture=2.0)]


# (case id, scene name, params): every case renders once in the oracle and on each of its arms
CASES = ([_case(s) for s in EDGE] + [_case("mirror-box", max_depth=200), _case("bright", spp=64)]
         + [_case("final"), _case("final-h28", W=40, H=24, spp=4), _case("grid", W=32, H=18, spp=4)]
         + _sweeps("final") + _sweeps("glass"))
CASE = {c[0]: c for c in CASES}


@lru_cache(maxsize=None)
def build(name):
    """the scene's arrays (built once per process; callers must not modify them)"""
    return SCENES[name][0]()


def view(name, p):
    look_from, look_at, vup, vfov, aperture, focus = SCENES[name][1]
    if "aperture" in p:
        aperture = p["aperture"]
    return look_from, look_at, vup, vfov, p["W"] / p["H"], aperture, focus


def camera(mod, name, p):
    """the case's camera from `mod` (oracle or capi: both take camera_new's arguments)"""
    return mod.camera_new(*view(name, p))


def to_dev_camera_f64(cam):
    """an oracle camera with the fields rounded as capi.cu's to_dev_camera<float> rounds them: origin, llc - origin,
    horizontal, vertical, u, v and the lens radius to f32 (llc then is the f64 sum of the two f32 parts)"""
    def r(v):
        return np.asarray([v.x, v.y, v.z], np.float32).astype(float)
    out = type(cam)()
    o = r(cam.origin)
    llc = np.array([cam.lower_left_corner.x, cam.lower_left_corner.y, cam.lower_left_corner.z]) - \
        np.array([cam.origin.x, cam.origin.y, cam.origin.z])
    from oracle.oracle import v3
    out.origin = v3(o)
    out.lower_left_corner = v3(o + np.asarray(llc, np.float32).astype(float))
    out.horizontal, out.vertical, out.u, out.v = v3(r(cam.horizontal)), v3(r(cam.vertical)), v3(r(cam.u)), v3(r(cam.v))
    out.w = cam.w
    out.lens_radius = float(np.float32(cam.lens_radius))
    return out
