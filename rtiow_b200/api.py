"""Python mirror of the reference's caller-facing API (SURVEY Appendix A), for tests and bench.

Same names and argument meaning as the Rust modules (`Vec3`-triples are plain sequences here):
`Camera::new` -> Camera(...), `Sphere::new(cen, r, mat)`, `Lambertian::new(albedo)`, `Metal::new(albedo, fuzz)`,
`Dialectric::new(ir)` (the reference's spelling, materials.rs:64), `HittableList` = list of shapes, and one new
call `render(cam, world, params)` that replaces main.rs:122-145.  Everything executes in librtiow_cuda.so;
objects here only describe the scene (the `describe()` of INTEGRATION.md).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from . import capi


@dataclass(frozen=True)
class Lambertian:                      # materials.rs:9-20
    albedo: tuple
    kind: int = field(default=capi.MAT_LAMBERTIAN, init=False)
    param: float = field(default=0.0, init=False)


@dataclass(frozen=True)
class Metal:                           # materials.rs:34-47 (fuzz is NOT clamped)
    albedo: tuple
    fuzz: float
    kind: int = field(default=capi.MAT_METAL, init=False)

    @property
    def param(self):
        return self.fuzz


@dataclass(frozen=True)
class Dialectric:                      # materials.rs:64-74 (sic)
    ir: float
    kind: int = field(default=capi.MAT_DIELECTRIC, init=False)
    albedo: tuple = field(default=(1.0, 1.0, 1.0), init=False)

    @property
    def param(self):
        return self.ir


Dielectric = Dialectric                # correctly spelt alias, added not substituted


@dataclass(frozen=True)
class Sphere:                          # sphere.rs:9-13,45-51 (radius unvalidated: negative allowed)
    center: tuple
    radius: float
    mat: object


class HittableList(list):              # shapes/mod.rs:52: Vec<Box<dyn Hit>>
    def push(self, shape):
        self.append(shape)

    def to_arrays(self):
        """describe(): flatten to the SoA the C ABI takes; unknown shapes/materials -> Unsupported."""
        mats, mat_ids, index = [], {}, []
        for s in self:
            if not isinstance(s, Sphere):
                raise capi.RtiowError(capi.ERR_UNSUPPORTED, f"shape {type(s).__name__} has no GPU implementation")
            if not isinstance(s.mat, (Lambertian, Metal, Dialectric)):
                raise capi.RtiowError(capi.ERR_UNSUPPORTED, f"material {type(s.mat).__name__} has no GPU implementation")
            k = id(s.mat)
            if k not in mat_ids:
                mat_ids[k] = len(mats)
                mats.append(s.mat)
            index.append(mat_ids[k])
        return dict(center=np.array([s.center for s in self], np.float64).reshape(-1, 3),
                    radius=np.array([s.radius for s in self], np.float64),
                    mat_index=np.array(index, np.uint32),
                    mat_kind=np.array([m.kind for m in mats], np.uint32),
                    mat_albedo=np.array([m.albedo for m in mats], np.float64).reshape(-1, 3),
                    mat_param=np.array([m.param for m in mats], np.float64))


def Camera(look_from, look_at, v_up, v_fov, aspect_ratio, aperture, focus_dist) -> capi.Camera:
    """Camera::new (camera.rs:17-23): v_fov in degrees."""
    return capi.camera_new(look_from, look_at, v_up, v_fov, aspect_ratio, aperture, focus_dist)


def RenderParams(**kw) -> capi.Params:
    """Defaults mirror main.rs:24-28,44,137."""
    return capi.default_params(**kw)


def random_scene(seed=1, half_extent=11, material_mode=0) -> HittableList:
    """random_scene (main.rs:59-102) with an explicit seed."""
    a = capi.random_scene(seed, half_extent, material_mode)
    world = HittableList()
    for i in range(len(a["radius"])):
        k, alb, prm = int(a["mat_kind"][i]), tuple(a["mat_albedo"][i]), float(a["mat_param"][i])
        mat = Lambertian(alb) if k == capi.MAT_LAMBERTIAN else Metal(alb, prm) if k == capi.MAT_METAL else Dialectric(prm)
        world.push(Sphere(tuple(a["center"][i]), float(a["radius"][i]), mat))
    return world


def render(cam: capi.Camera, world: HittableList, params: capi.Params, n_gpus: int = 1):
    """The drop-in call: top-down RGBA8 [H,W,4] — the buffer of ImageBuffer::from_vec (main.rs:147)."""
    with capi.Context(n_gpus) as ctx:
        ctx.upload_scene(**world.to_arrays())
        img, _ = ctx.render(cam, params)
    return img


def render_aov(cam: capi.Camera, world: HittableList, params: capi.Params, n_gpus: int = 1):
    """render() plus float AOVs for a denoiser -> (rgba[H,W,4], {"color", "albedo", "normal": [H,W,3], "depth": [H,W]} float32):
    linear colour, and the albedo, normal and distance of each camera ray's first hit (include/rtiow_cuda.h, rtiow_render_aov)."""
    with capi.Context(n_gpus) as ctx:
        ctx.upload_scene(**world.to_arrays())
        img, aovs, _ = ctx.render_aov(cam, params)
    return img, aovs


def render_adaptive(cam: capi.Camera, world: HittableList, params: capi.Params, min_spp: int, tolerance: float, n_gpus: int = 1):
    """Adaptive sampling: each pixel gets between min_spp and params.spp samples, as many as its own noise asks for, and equals
    render() at its own count byte for byte -> (rgba[H,W,4], {"spp": uint32[H,W], "error": float32[H,W]}) (include/rtiow_cuda.h,
    rtiow_render_adaptive: the error is one standard error of the displayed value in 8-bit levels, compared with tolerance)."""
    with capi.Context(n_gpus) as ctx:
        ctx.upload_scene(**world.to_arrays())
        img, maps, _ = ctx.render_adaptive(cam, params, min_spp, tolerance)
    return img, maps


def denoise(color, albedo, normal, depth, params: capi.DenoiseParams | None = None, n_gpus: int = 1):
    """An edge-avoiding a-trous denoiser over render_aov()'s buffers (include/rtiow_cuda.h, rtiow_denoise; default parameters when
    params is None) -> (linear colour float32[H,W,3], rgba uint8[H,W,4]).  Needs no scene: it runs on the first GPU."""
    with capi.Context(n_gpus) as ctx:
        outs, _ = ctx.denoise(color, albedo, normal, depth, params)
    return outs["color"], outs["rgba"]


def render_denoised(cam: capi.Camera, world: HittableList, params: capi.Params, dparams: capi.DenoiseParams | None = None, n_gpus: int = 1):
    """A denoised frame in one call -> (linear colour float32[H,W,3], rgba uint8[H,W,4]), bit-identical to denoise() over
    render_aov()'s buffers, which stay on the GPU (include/rtiow_cuda.h, rtiow_render_denoised; default denoise parameters when
    dparams is None)."""
    with capi.Context(n_gpus) as ctx:
        ctx.upload_scene(**world.to_arrays())
        outs, _ = ctx.render_denoised(cam, params, dparams)
    return outs["color"], outs["rgba"]


def render_views(cams, world: HittableList, params: capi.Params, n_gpus: int = 1):
    """Many cameras of one world in one call: [K,H,W,4] top-down RGBA8, frame v byte-identical to render(cams[v], ...)."""
    with capi.Context(n_gpus) as ctx:
        ctx.upload_scene(**world.to_arrays())
        imgs, _ = ctx.render_views(cams, params)
    return imgs


def render_progressive(cam: capi.Camera, world: HittableList, params: capi.Params, n_passes: int, on_pass=None, n_gpus: int = 1):
    """render() in n_passes slices of the samples; on_pass(pass_1based, n_passes, spp_done, rgba[H,W,4]) after each — the role of
    the reference's progress bar and preview window (main.rs:120-124,151-171).  Final frame bit-identical to render()'s."""
    with capi.Context(n_gpus) as ctx:
        ctx.upload_scene(**world.to_arrays())
        img, _ = ctx.render_progressive(cam, params, n_passes, on_pass)
    return img
