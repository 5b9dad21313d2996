"""ctypes wrapper of the CPU oracle (oracle/rtiow_oracle.c).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module; the product package (rtiow_b200/) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_SO = _HERE / "build" / "librtiow_oracle.so"

MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC = 0, 1, 2
SAMPLER_REJECTION, SAMPLER_DIRECT = 0, 1


_SCENE_SO = _HERE / "build" / "librtiow_scene.so"


def build(force: bool = False) -> Path:
    """Compile the oracle (and the host-only scene library) with the committed Makefile (gcc, -ffp-contract=off, OpenMP)."""
    srcs = [_HERE / "rtiow_oracle.c", _HERE / "rtiow_oracle.h", _HERE / "Makefile", _HERE.parent / "rtiow_b200" / "csrc" / "scene_gen.cpp",
            _HERE.parent / "include" / "rtiow_cuda.h"]
    stale = force or not _SO.exists() or not _SCENE_SO.exists() or any(s.stat().st_mtime > min(_SO.stat().st_mtime, _SCENE_SO.stat().st_mtime) for s in srcs)
    if stale:
        subprocess.run(["make", "-C", str(_HERE), "-B"], check=True, capture_output=True)
    return _SO


def use_native_build() -> bool:
    """bench.py's timed CPU legs: rebuild the oracle with -march=native ON THE BOX THAT RUNS IT (the committed recipe builds for
    baseline x86-64 because the .so travels) and switch lib() to it.  The build goes to a temporary directory, removed once the
    library is loaded: bench.py writes nothing into the tree.  Returns False (and keeps the baseline build) if gcc fails."""
    global _lib
    with tempfile.TemporaryDirectory(prefix="rtiow_oracle_") as td:
        so = Path(td) / "librtiow_oracle.so"
        try:
            subprocess.run(["make", "-C", str(_HERE), "-B", "MARCH=native", f"BUILD={td}", str(so)], check=True, capture_output=True)
        except (subprocess.CalledProcessError, OSError):
            return False
        _lib = C.CDLL(str(so))
    _declare(_lib)
    return True


class Vec3(C.Structure):
    _fields_ = [("x", C.c_double), ("y", C.c_double), ("z", C.c_double)]

    def np(self):
        return np.array([self.x, self.y, self.z])


def v3(a) -> Vec3:
    return Vec3(float(a[0]), float(a[1]), float(a[2]))


class Ray(C.Structure):
    _fields_ = [("orig", Vec3), ("dir", Vec3)]


class Camera(C.Structure):
    _fields_ = [(n, Vec3) for n in ("origin", "lower_left_corner", "horizontal", "vertical", "u", "v", "w")] + [
        ("lens_radius", C.c_double)
    ]


class Material(C.Structure):
    _fields_ = [("kind", C.c_int32), ("albedo", Vec3), ("param", C.c_double)]


class Sphere(C.Structure):
    _fields_ = [("center", Vec3), ("radius", C.c_double), ("mat", C.c_int32)]


class HitRecord(C.Structure):
    _fields_ = [("p", Vec3), ("normal", Vec3), ("mat", C.c_int32), ("t", C.c_double), ("front_face", C.c_int32)]


class World(C.Structure):
    _fields_ = [("spheres", C.POINTER(Sphere)), ("n_spheres", C.c_int32), ("materials", C.POINTER(Material)),
                ("n_materials", C.c_int32)]


class Counters(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("sphere_tests", C.c_uint64)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("spp", C.c_uint32), ("max_depth", C.c_int32),
                ("t_min", C.c_double), ("seed", C.c_uint64), ("alpha", C.c_uint8), ("sampler", C.c_int32),
                ("n_threads", C.c_int32), ("row_begin", C.c_uint32), ("row_end", C.c_uint32)]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(str(_SO))
        _declare(_lib)
    return _lib


def _declare(L):
    d, i32, u32, u64, i64 = C.c_double, C.c_int32, C.c_uint32, C.c_uint64, C.c_int64
    P = C.c_void_p
    for name, res, args in [
        ("o_add", Vec3, [Vec3, Vec3]), ("o_sub", Vec3, [Vec3, Vec3]), ("o_mul_s", Vec3, [Vec3, d]),
        ("o_mul_v", Vec3, [Vec3, Vec3]), ("o_div_s", Vec3, [Vec3, d]), ("o_length_squared", d, [Vec3]),
        ("o_length", d, [Vec3]), ("o_dot", d, [Vec3, Vec3]), ("o_cross", Vec3, [Vec3, Vec3]),
        ("o_unit_vector", Vec3, [Vec3]), ("o_is_near_zero", C.c_int, [Vec3]), ("o_reflect", Vec3, [Vec3, Vec3]),
        ("o_refract", Vec3, [Vec3, Vec3, d]), ("o_to_rgba", None, [Vec3, C.c_uint8, u64, P]),
        ("o_ray_at", Vec3, [C.POINTER(Ray), d]),
        ("o_camera_new", None, [C.POINTER(Camera), Vec3, Vec3, Vec3, d, d, d, d]),
        ("o_camera_get_ray", Ray, [C.POINTER(Camera), d, d, d, d]),
        ("o_sphere_hit", C.c_int, [C.POINTER(Sphere), C.POINTER(Ray), d, d, C.POINTER(HitRecord)]),
        ("o_world_hit", C.c_int, [C.POINTER(World), C.POINTER(Ray), d, d, C.POINTER(HitRecord), C.POINTER(i32)]),
        ("o_scatter", C.c_int, [C.POINTER(Material), C.POINTER(Ray), C.POINTER(HitRecord), Vec3, C.POINTER(Vec3),
                                C.POINTER(Ray)]),
        ("o_reflectance", d, [d, d]),
        ("o_philox4x32_10", None, [P, P, P]),
        ("o_direct_uniforms", None, [u64, u32, u32, u32, P]),
        ("o_direct_disk", None, [d, d, C.POINTER(d), C.POINTER(d)]),
        ("o_direct_unit_vector", Vec3, [d, d]), ("o_direct_in_unit_sphere", Vec3, [d, d, d]),
        ("o_render", C.c_int, [C.POINTER(World), C.POINTER(Camera), C.POINTER(RenderParams), P, P, C.POINTER(Counters)]),
        ("o_render_margins", C.c_int, [C.POINTER(World), C.POINTER(Camera), C.POINTER(RenderParams), P, P, P,
                                       C.POINTER(Counters)]),
        ("o_path_radiance", Vec3, [C.POINTER(World), C.POINTER(Camera), C.POINTER(RenderParams), u32, u32, u32,
                                   C.POINTER(Counters)]),
        ("o_sphere_hit_batch", None, [i64] + [P] * 11),
        ("o_world_hit_batch", None, [C.POINTER(World), i64, P, P, d, d, P, P, P, P, P, P]),
        ("o_scatter_batch", None, [i64] + [P] * 13),
        ("o_get_ray_batch", None, [C.POINTER(Camera), i64, P, P, P, P, P]),
        ("o_to_rgba_batch", None, [i64, P, C.c_uint8, u64, P]),
        ("o_reflect_batch", None, [i64, P, P, P]), ("o_refract_batch", None, [i64, P, P, P, P]),
        ("o_ray_color_batch", None, [C.POINTER(World), i64, P, P, P, P, u64, i32, d, P, P]),
        ("o_rejection_samples", None, [u64, i64, i32, P]),
    ]:
        if not hasattr(L, name):
            continue
        f = getattr(L, name)
        f.restype = res
        f.argtypes = args


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


# --------------------------------------------------------------------------------------------- scene
class Scene:
    """Explicit scene handed identically to the oracle and to the CUDA library."""

    def __init__(self, center, radius, mat_index, mat_kind, mat_albedo, mat_param):
        self.center = _f64(center, (-1, 3))
        self.radius = _f64(radius, (-1,))
        self.mat_index = np.ascontiguousarray(mat_index, dtype=np.uint32).reshape(-1)
        self.mat_kind = np.ascontiguousarray(mat_kind, dtype=np.uint32).reshape(-1)
        self.mat_albedo = _f64(mat_albedo, (-1, 3))
        self.mat_param = _f64(mat_param, (-1,))
        n, m = len(self.radius), len(self.mat_kind)
        assert self.center.shape == (n, 3) and self.mat_index.shape == (n,)
        assert self.mat_albedo.shape == (m, 3) and self.mat_param.shape == (m,)
        self._spheres = (Sphere * max(n, 1))()
        for i in range(n):
            self._spheres[i] = Sphere(v3(self.center[i]), float(self.radius[i]), int(self.mat_index[i]))
        self._materials = (Material * max(m, 1))()
        for i in range(m):
            self._materials[i] = Material(int(self.mat_kind[i]), v3(self.mat_albedo[i]), float(self.mat_param[i]))
        self.world = World(self._spheres, n, self._materials, m)

    @property
    def n(self):
        return len(self.radius)


def camera_new(look_from, look_at, v_up, v_fov, aspect_ratio, aperture, focus_dist) -> Camera:
    cam = Camera()
    lib().o_camera_new(C.byref(cam), v3(look_from), v3(look_at), v3(v_up), v_fov, aspect_ratio, aperture, focus_dist)
    return cam


# --------------------------------------------------------------------------------------------- batches
def sphere_hit_batch(center, radius, orig, direction, t_min, t_max):
    center, orig, direction = _f64(center, (-1, 3)), _f64(orig, (-1, 3)), _f64(direction, (-1, 3))
    n = len(center)
    radius = _f64(np.broadcast_to(radius, (n,)))
    t_min = _f64(np.broadcast_to(t_min, (n,)))
    t_max = _f64(np.broadcast_to(t_max, (n,)))
    hit = np.zeros(n, np.int32); t = np.zeros(n); p = np.zeros((n, 3)); nrm = np.zeros((n, 3)); ff = np.zeros(n, np.int32)
    lib().o_sphere_hit_batch(n, _p(center), _p(radius), _p(orig), _p(direction), _p(t_min), _p(t_max), _p(hit), _p(t),
                             _p(p), _p(nrm), _p(ff))
    return dict(hit=hit, t=t, p=p, normal=nrm, front_face=ff)


def world_hit_batch(scene: Scene, orig, direction, t_min=1e-4, t_max=float("inf")):
    orig, direction = _f64(orig, (-1, 3)), _f64(direction, (-1, 3))
    n = len(orig)
    hit = np.zeros(n, np.int32); idx = np.zeros(n, np.int32); t = np.zeros(n); p = np.zeros((n, 3))
    nrm = np.zeros((n, 3)); ff = np.zeros(n, np.int32)
    lib().o_world_hit_batch(C.byref(scene.world), n, _p(orig), _p(direction), t_min, t_max, _p(hit), _p(idx), _p(t),
                            _p(p), _p(nrm), _p(ff))
    return dict(hit=hit, index=idx, t=t, p=p, normal=nrm, front_face=ff)


def scatter_batch(kind, albedo, param, r_orig, r_dir, p, normal, front_face, sample):
    kind = np.ascontiguousarray(kind, np.int32)
    n = len(kind)
    albedo, r_orig, r_dir = _f64(albedo, (n, 3)), _f64(r_orig, (n, 3)), _f64(r_dir, (n, 3))
    p, normal, sample = _f64(p, (n, 3)), _f64(normal, (n, 3)), _f64(sample, (n, 3))
    param = _f64(param, (n,)); front_face = np.ascontiguousarray(front_face, np.int32)
    some = np.zeros(n, np.int32); att = np.zeros((n, 3)); so = np.zeros((n, 3)); sd = np.zeros((n, 3))
    lib().o_scatter_batch(n, _p(kind), _p(albedo), _p(param), _p(r_orig), _p(r_dir), _p(p), _p(normal), _p(front_face),
                          _p(sample), _p(some), _p(att), _p(so), _p(sd))
    return dict(some=some, attenuation=att, orig=so, dir=sd)


def get_ray_batch(cam: Camera, s, t, disk_xy):
    s, t, disk_xy = _f64(s, (-1,)), _f64(t, (-1,)), _f64(disk_xy, (-1, 2))
    n = len(s)
    o = np.zeros((n, 3)); d = np.zeros((n, 3))
    lib().o_get_ray_batch(C.byref(cam), n, _p(s), _p(t), _p(disk_xy), _p(o), _p(d))
    return dict(orig=o, dir=d)


def to_rgba_batch(color, alpha, spp):
    color = _f64(color, (-1, 3))
    out = np.zeros((len(color), 4), np.uint8)
    lib().o_to_rgba_batch(len(color), _p(color), alpha, spp, _p(out))
    return out


def reflect_batch(v, n):
    v, n = _f64(v, (-1, 3)), _f64(n, (-1, 3))
    out = np.zeros_like(v)
    lib().o_reflect_batch(len(v), _p(v), _p(n), _p(out))
    return out


def refract_batch(uv, n, eta):
    uv, n = _f64(uv, (-1, 3)), _f64(n, (-1, 3))
    eta = _f64(np.broadcast_to(eta, (len(uv),)))
    out = np.zeros_like(uv)
    lib().o_refract_batch(len(uv), _p(uv), _p(n), _p(eta), _p(out))
    return out


def ray_color_batch(scene: Scene, orig, direction, pixel, sample, seed, max_depth=50, t_min=1e-4):
    orig, direction = _f64(orig, (-1, 3)), _f64(direction, (-1, 3))
    n = len(orig)
    pixel = np.ascontiguousarray(pixel, np.uint32); sample = np.ascontiguousarray(sample, np.uint32)
    col = np.zeros((n, 3)); rays = np.zeros(n, np.uint64)
    lib().o_ray_color_batch(C.byref(scene.world), n, _p(orig), _p(direction), _p(pixel), _p(sample), seed, max_depth,
                            t_min, _p(col), _p(rays))
    return dict(color=col, rays=rays)


def rejection_samples(seed, n, which):
    out = np.zeros((n, 3))
    lib().o_rejection_samples(seed, n, which, _p(out))
    return out


def philox4x32_10(ctr, key):
    ctr = np.ascontiguousarray(ctr, np.uint32); key = np.ascontiguousarray(key, np.uint32)
    out = np.zeros(4, np.uint32)
    lib().o_philox4x32_10(_p(ctr), _p(key), _p(out))
    return out


def direct_uniforms(seed, pixel, sample, bounce):
    u = np.zeros(4)
    lib().o_direct_uniforms(seed, pixel, sample, bounce, _p(u))
    return u


def render(scene: Scene, cam: Camera, width, height, spp, max_depth=50, t_min=1e-4, seed=1, alpha=255,
           sampler=SAMPLER_DIRECT, n_threads=0, rows=None, want_accum=False):
    """main.rs:122-145 on the CPU.  Returns (rgba[H,W,4] top-down, accum[H,W,3] | None, counters dict)."""
    rb, re = (0, 0) if rows is None else rows
    prm = RenderParams(width, height, spp, max_depth, t_min, seed, alpha, sampler, n_threads, rb, re)
    out = np.zeros((height, width, 4), np.uint8)
    acc = np.zeros((height, width, 3)) if want_accum else None
    cnt = Counters()
    rc = lib().o_render(C.byref(scene.world), C.byref(cam), C.byref(prm), _p(out), _p(acc) if want_accum else None,
                        C.byref(cnt))
    if rc != 0:
        raise ValueError("o_render: invalid arguments")
    return out, acc, dict(rays=int(cnt.rays), sphere_tests=int(cnt.sphere_tests))


def render_margins(scene: Scene, cam: Camera, width, height, spp, max_depth=50, t_min=1e-4, seed=1, alpha=255, n_threads=0,
                   rows=None):
    """render(..., sampler=SAMPLER_DIRECT, want_accum=True) and each pixel's knife-edge margin (o_render_margins,
    rtiow_oracle.h).  Returns (rgba[H,W,4], accum[H,W,3], margin[H,W], counters dict)."""
    rb, re = (0, 0) if rows is None else rows
    prm = RenderParams(width, height, spp, max_depth, t_min, seed, alpha, SAMPLER_DIRECT, n_threads, rb, re)
    out = np.zeros((height, width, 4), np.uint8)
    acc = np.zeros((height, width, 3))
    mg = np.full((height, width), np.inf)
    cnt = Counters()
    if lib().o_render_margins(C.byref(scene.world), C.byref(cam), C.byref(prm), _p(out), _p(acc), _p(mg), C.byref(cnt)) != 0:
        raise ValueError("o_render_margins: invalid arguments")
    return out, acc, mg, dict(rays=int(cnt.rays), sphere_tests=int(cnt.sphere_tests))


# A pixel is robust -- an f32 render must give it the oracle's exact bytes -- when no ray of its paths comes within TAU of a
# decision (margin >= TAU, o_render_margins) and its exact value 256 sqrt(clamp(sum / spp, 0, 0.999)) is more than DELTA
# from an integer in every channel (or exactly 0: black paths add nothing on either side).
# TAU: the margins are relative distances, and an f32 evaluation of a root, a dot product or a unit vector errs by a few
# eps32 = 6e-8 relative to its inputs, times the growth the margin is already divided by; TAU = 2e-5 is ~300 eps32.
# DELTA: a pixel's value in f32 carries the relative error of its path colours (~1e-6 on long chains, the sky term of a
# unit vector); at 255 that is ~3e-4, and DELTA = 0.01 leaves a factor 30.
MARGIN_TAU = 2e-5
VALUE_DELTA = 0.01


def robust_pixels(accum, margin, spp, tau=MARGIN_TAU, delta=VALUE_DELTA):
    """bool[H, W]: the pixels whose bytes an f32 render must reproduce exactly (see MARGIN_TAU)"""
    v = 256.0 * np.sqrt(np.clip(np.asarray(accum) / spp, 0.0, 0.999))
    frac = np.abs(v - np.round(v))
    exact = (frac > delta) | (np.asarray(accum) == 0.0)
    return (np.asarray(margin) >= tau) & exact.all(axis=-1)


# ---- worlds: the seeded scene builder and scene files, from the HOST-ONLY build of rtiow_b200/csrc/scene_gen.cpp ----------
_scene_lib = None


def scene_lib() -> C.CDLL:
    global _scene_lib
    if _scene_lib is None:
        build()
        L = C.CDLL(str(_SCENE_SO))
        P, u32 = C.c_void_p, C.c_uint32
        L.rtiow_random_scene.restype, L.rtiow_random_scene.argtypes = C.c_int, [C.c_uint64, C.c_int32, C.c_int32, u32, P, P, P, P, P, P, P, C.POINTER(u32)]
        L.rtiow_scene_save.restype, L.rtiow_scene_save.argtypes = C.c_int, [C.c_char_p, u32, P, P, P, P, P, P, P]
        L.rtiow_scene_load.restype, L.rtiow_scene_load.argtypes = C.c_int, [C.c_char_p, u32, P, P, P, P, P, P, P, C.POINTER(u32)]
        _scene_lib = L
    return _scene_lib


def _scene_dict(k, cx, cy, cz, r, kind, alb, prm):
    return dict(center=np.stack([cx[:k], cy[:k], cz[:k]], 1), radius=r[:k].copy(), mat_index=np.arange(k, dtype=np.uint32),
                mat_kind=kind[:k].copy(), mat_albedo=alb[:k].copy(), mat_param=prm[:k].copy())


def random_scene(seed: int = 1, half_extent: int = 11, material_mode: int = 0):
    """Seeded random_scene (main.rs:59-102) without the CUDA library: the arrays rtiow_b200.capi.random_scene returns."""
    cap = (2 * half_extent + 1) ** 2 + 8
    cx, cy, cz, r = (np.zeros(cap) for _ in range(4))
    kind = np.zeros(cap, np.uint32); alb = np.zeros((cap, 3)); prm = np.zeros(cap)
    n = C.c_uint32(0)
    rc = scene_lib().rtiow_random_scene(seed, half_extent, material_mode, cap, _p(cx), _p(cy), _p(cz), _p(r), _p(kind), _p(alb), _p(prm), C.byref(n))
    if rc != 0:
        raise RuntimeError(f"rtiow_random_scene failed: {rc}")
    return _scene_dict(n.value, cx, cy, cz, r, kind, alb, prm)


def load_scene(path):
    n = C.c_uint32(0)
    if scene_lib().rtiow_scene_load(str(path).encode(), 0, None, None, None, None, None, None, None, C.byref(n)) != 0:
        raise RuntimeError(f"cannot read scene file {path}")
    k = max(n.value, 1)
    cx, cy, cz, r = (np.zeros(k) for _ in range(4))
    kind = np.zeros(k, np.uint32); alb = np.zeros((k, 3)); prm = np.zeros(k)
    if scene_lib().rtiow_scene_load(str(path).encode(), k, _p(cx), _p(cy), _p(cz), _p(r), _p(kind), _p(alb), _p(prm), C.byref(n)) != 0:
        raise RuntimeError(f"malformed scene file {path}")
    return _scene_dict(n.value, cx, cy, cz, r, kind, alb, prm)


def host_threads() -> int:
    return os.cpu_count() or 1
