"""ctypes binding of librtiow_cuda.so — the same C ABI (include/rtiow_cuda.h) the Rust `-sys` crate binds.

This module is plumbing: it loads the in-tree .so, declares every exported symbol and converts numpy
arrays to the plain pointers the ABI takes.  There is no CPU fallback: if the library is missing the
import of `lib()` raises, and with no CUDA device every compute call raises RtiowError(NO_DEVICE).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from . import build as _build

OK, ERR_INVALID_ARG, ERR_UNSUPPORTED, ERR_CUDA, ERR_NCCL, ERR_NO_DEVICE, ERR_NOMEM, ERR_CANCELLED = 0, -1, -2, -3, -4, -5, -6, -7
MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC = 0, 1, 2
F32, F64 = 0, 1
ABI_VERSION = 4
SCAN_AUTO, SCAN_FP32, SCAN_TENSOR = 0, 1, 2
GATHER_AUTO, GATHER_NCCL, GATHER_FUSED = 0, 1, 2
NCCL_UNIQUE_ID_BYTES = 128

_STATUS = {OK: "OK", ERR_INVALID_ARG: "INVALID_ARG", ERR_UNSUPPORTED: "UNSUPPORTED", ERR_CUDA: "CUDA", ERR_NCCL: "NCCL",
           ERR_NO_DEVICE: "NO_DEVICE", ERR_NOMEM: "NOMEM", ERR_CANCELLED: "CANCELLED"}
# rtiow_progress_fn: int (*)(void* user, uint32_t pass, uint32_t n_passes, uint32_t spp_done, const uint8_t* rgba)
PROGRESS_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p)

# every symbol include/rtiow_cuda.h declares (tests check the .so exports exactly these)
SYMBOLS = [
    "rtiow_abi_version", "rtiow_last_error", "rtiow_device_count", "rtiow_ctx_create", "rtiow_ctx_create_on_device",
    "rtiow_ctx_destroy", "rtiow_ctx_set_scan_backend", "rtiow_ctx_set_filter_bypass", "rtiow_nccl_unique_id", "rtiow_ctx_create_rank", "rtiow_ctx_set_gather", "rtiow_ctx_set_stream",
    "rtiow_ctx_gather_info", "rtiow_render_rank", "rtiow_render_rank_device", "rtiow_render_rank_enqueue", "rtiow_ctx_synchronize", "rtiow_scene_upload", "rtiow_camera_new", "rtiow_params_default", "rtiow_render", "rtiow_render_aov", "rtiow_render_adaptive", "rtiow_render_views", "rtiow_render_progressive",
    "rtiow_tile_buffer_bytes", "rtiow_render_tiles_device", "rtiow_render_to_frame_device", "rtiow_deinterleave_device", "rtiow_sphere_hit_batch",
    "rtiow_hitlist_batch", "rtiow_scatter_batch", "rtiow_get_ray_batch", "rtiow_to_rgba_batch", "rtiow_reflect_batch",
    "rtiow_refract_batch", "rtiow_ray_color_batch", "rtiow_ray_color_trace_batch", "rtiow_sampler_batch", "rtiow_fp32_peak_probe", "rtiow_flush_l2",
    "rtiow_random_scene", "rtiow_scene_save", "rtiow_scene_load",
]


class RtiowError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"rtiow_cuda: {_STATUS.get(code, code)}: {msg}")
        self.code = code


class Spheres(C.Structure):
    _fields_ = [("cx", C.c_void_p), ("cy", C.c_void_p), ("cz", C.c_void_p), ("radius", C.c_void_p), ("mat_index", C.c_void_p),
                ("n", C.c_uint32)]


class Materials(C.Structure):
    _fields_ = [("kind", C.c_void_p), ("albedo_r", C.c_void_p), ("albedo_g", C.c_void_p), ("albedo_b", C.c_void_p),
                ("param", C.c_void_p), ("n", C.c_uint32)]


class Camera(C.Structure):
    _fields_ = [(k, C.c_double * 3) for k in ("origin", "lower_left_corner", "horizontal", "vertical", "u", "v", "w")] + [
        ("lens_radius", C.c_double)]


class Params(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("spp", C.c_uint32), ("max_depth", C.c_int32),
                ("t_min", C.c_double), ("seed", C.c_uint64), ("alpha", C.c_uint8), ("precision", C.c_uint8),
                ("reserved", C.c_uint8 * 6), ("tile_rows", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("kernel_ms", C.c_double), ("total_ms", C.c_double), ("paths", C.c_uint64), ("rays_traced", C.c_uint64),
                ("sphere_tests", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("kernel_launches", C.c_uint32), ("n_gpus", C.c_uint32), ("scan_backend", C.c_uint32), ("reserved", C.c_uint32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib = None


def lib_path() -> Path:
    return _build.LIB


def lib(build_if_missing: bool = True) -> C.CDLL:
    """Load librtiow_cuda.so (building it in-tree with nvcc if it is missing).  Raises if it cannot."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        _build.build_lib()
    if not _build.LIB.exists():
        raise RuntimeError(f"{_build.LIB} is missing: build it with `python -m rtiow_b200.build` (no CPU fallback exists)")
    L = C.CDLL(str(_build.LIB))
    _declare(L)
    if L.rtiow_abi_version() != ABI_VERSION:
        raise RuntimeError("librtiow_cuda.so ABI version mismatch")
    _lib = L
    return L


def _declare(L):
    P, i32, i64, u32, u64, d = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_double
    sig = {
        "rtiow_abi_version": (C.c_int, []),
        "rtiow_last_error": (C.c_char_p, []),
        "rtiow_device_count": (C.c_int, [C.POINTER(C.c_int)]),
        "rtiow_ctx_create": (C.c_int, [C.c_int, C.POINTER(P)]),
        "rtiow_ctx_create_on_device": (C.c_int, [C.c_int, C.POINTER(P)]),
        "rtiow_ctx_destroy": (None, [P]),
        "rtiow_ctx_set_scan_backend": (C.c_int, [P, C.c_int]),
        "rtiow_ctx_set_filter_bypass": (C.c_int, [P, C.c_int]),
        "rtiow_nccl_unique_id": (C.c_int, [P]),
        "rtiow_ctx_create_rank": (C.c_int, [C.c_int, C.c_int, C.c_int, P, C.POINTER(P)]),
        "rtiow_ctx_set_gather": (C.c_int, [P, C.c_int]),
        "rtiow_ctx_set_stream": (C.c_int, [P, P]),
        "rtiow_ctx_gather_info": (C.c_int, [P, C.c_char_p, C.c_size_t]),
        "rtiow_render_rank": (C.c_int, [P, C.POINTER(Camera), C.POINTER(Params), P, C.POINTER(Stats)]),
        "rtiow_render_rank_device": (C.c_int, [P, C.POINTER(Camera), C.POINTER(Params), C.POINTER(P), C.POINTER(Stats)]),
        "rtiow_scene_upload": (C.c_int, [P, C.POINTER(Spheres), C.POINTER(Materials)]),
        "rtiow_camera_new": (C.c_int, [P, P, P, d, d, d, d, C.POINTER(Camera)]),
        "rtiow_params_default": (None, [C.POINTER(Params)]),
        "rtiow_render": (C.c_int, [P, C.POINTER(Camera), C.POINTER(Params), P, C.POINTER(Stats)]),
        "rtiow_render_aov": (C.c_int, [P, C.POINTER(Camera), C.POINTER(Params), P, P, P, P, P, C.POINTER(Stats)]),
        "rtiow_render_adaptive": (C.c_int, [P, C.POINTER(Camera), C.POINTER(Params), u32, d, P, P, P, C.POINTER(Stats)]),
        "rtiow_render_views": (C.c_int, [P, C.POINTER(Camera), C.c_uint32, C.POINTER(Params), P, C.POINTER(Stats)]),
        "rtiow_render_progressive": (C.c_int, [P, C.POINTER(Camera), C.POINTER(Params), C.c_uint32, PROGRESS_FN, P, P, C.POINTER(Stats)]),
        "rtiow_render_rank_enqueue": (C.c_int, [P, C.POINTER(Camera), C.POINTER(Params), C.POINTER(C.c_void_p)]),
        "rtiow_ctx_synchronize": (C.c_int, [P, C.POINTER(Stats)]),
        "rtiow_tile_buffer_bytes": (C.c_int, [C.POINTER(Params), C.c_int, C.POINTER(C.c_size_t)]),
        "rtiow_render_tiles_device": (C.c_int, [P, C.POINTER(Camera), C.POINTER(Params), C.c_int, C.c_int, P, P, C.POINTER(Stats)]),
        "rtiow_render_to_frame_device": (C.c_int, [P, C.POINTER(Camera), C.POINTER(Params), C.c_int, C.c_int, P, P, C.POINTER(Stats)]),
        "rtiow_deinterleave_device": (C.c_int, [P, P, C.POINTER(Params), C.c_int, P, P]),
        "rtiow_sphere_hit_batch": (C.c_int, [P, C.c_int, i64] + [P] * 11),
        "rtiow_hitlist_batch": (C.c_int, [P, C.c_int, i64, P, P, d] + [P] * 6),
        "rtiow_scatter_batch": (C.c_int, [P, C.c_int, i64] + [P] * 13),
        "rtiow_get_ray_batch": (C.c_int, [P, C.c_int, C.POINTER(Camera), i64, P, P, P, P, P]),
        "rtiow_to_rgba_batch": (C.c_int, [P, C.c_int, i64, P, C.c_uint8, u64, P]),
        "rtiow_reflect_batch": (C.c_int, [P, C.c_int, i64, P, P, P]),
        "rtiow_refract_batch": (C.c_int, [P, C.c_int, i64, P, P, P, P]),
        "rtiow_ray_color_batch": (C.c_int, [P, C.c_int, i64, P, P, P, P, u64, i32, d, P, P]),
        "rtiow_ray_color_trace_batch": (C.c_int, [P, C.c_int, i64, P, P, P, P, u64, i32, d, P, P, P, P]),
        "rtiow_sampler_batch": (C.c_int, [P, C.c_int, i64, P, P, P, u64, P]),
        "rtiow_fp32_peak_probe": (C.c_int, [P, C.c_int, d, C.POINTER(d), C.POINTER(d)]),
        "rtiow_flush_l2": (C.c_int, [P]),
        "rtiow_random_scene": (C.c_int, [u64, i32, i32, u32, P, P, P, P, P, P, P, C.POINTER(u32)]),
        "rtiow_scene_save": (C.c_int, [C.c_char_p, u32, P, P, P, P, P, P, P]),
        "rtiow_scene_load": (C.c_int, [C.c_char_p, u32, P, P, P, P, P, P, P, C.POINTER(u32)]),
    }
    assert sorted(sig) == sorted(SYMBOLS)
    for name, (res, args) in sig.items():
        f = getattr(L, name)
        f.restype, f.argtypes = res, args


def device_to_host(ptr: int, nbytes: int) -> np.ndarray:
    """tests / tools: copy `nbytes` of device memory (a frame pointer returned by render_rank_device / _enqueue) to the host"""
    from cuda.bindings import runtime as cudart
    out = np.empty(nbytes, np.uint8)
    (err,) = cudart.cudaMemcpy(out.ctypes.data, ptr, nbytes, cudart.cudaMemcpyKind.cudaMemcpyDeviceToHost)
    if int(err) != 0:
        raise RuntimeError(f"cudaMemcpy D2H failed: {err}")
    return out


def _check(rc: int):
    if rc != OK:
        raise RtiowError(rc, lib().rtiow_last_error().decode("utf-8", "replace"))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a.reshape(shape) if shape is not None else a


def device_count() -> int:
    n = C.c_int(0)
    _check(lib().rtiow_device_count(C.byref(n)))
    return n.value


def camera_new(look_from, look_at, v_up, v_fov, aspect_ratio, aperture, focus_dist) -> Camera:
    """Camera::new (camera.rs:17-45)."""
    cam = Camera()
    a, b, c = _f64(look_from, (3,)), _f64(look_at, (3,)), _f64(v_up, (3,))
    _check(lib().rtiow_camera_new(_p(a), _p(b), _p(c), v_fov, aspect_ratio, aperture, focus_dist, C.byref(cam)))
    return cam


def default_params(**kw) -> Params:
    p = Params()
    lib().rtiow_params_default(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def random_scene(seed: int = 1, half_extent: int = 11, material_mode: int = 0):
    """Seeded random_scene (main.rs:59-102).  Returns dict of arrays, one material per sphere."""
    cap = (2 * half_extent + 1) ** 2 + 8
    cx, cy, cz, r = (np.zeros(cap) for _ in range(4))
    kind = np.zeros(cap, np.uint32); alb = np.zeros((cap, 3)); prm = np.zeros(cap)
    n = C.c_uint32(0)
    _check(lib().rtiow_random_scene(seed, half_extent, material_mode, cap, _p(cx), _p(cy), _p(cz), _p(r), _p(kind), _p(alb),
                                    _p(prm), C.byref(n)))
    k = n.value
    return dict(center=np.stack([cx[:k], cy[:k], cz[:k]], 1), radius=r[:k].copy(), mat_index=np.arange(k, dtype=np.uint32),
                mat_kind=kind[:k].copy(), mat_albedo=alb[:k].copy(), mat_param=prm[:k].copy())


def nccl_unique_id() -> bytes:
    """rank 0: the 128 bytes every rank passes to Context(rank=..., world=..., nccl_id=...) (MPI_Bcast / a file / torch.distributed)"""
    buf = C.create_string_buffer(NCCL_UNIQUE_ID_BYTES)
    _check(lib().rtiow_nccl_unique_id(buf))
    return buf.raw


def save_scene(path, center, radius, mat_index, mat_kind, mat_albedo, mat_param, L=None):
    """rtiow_scene_save: one line per sphere (its material resolved through mat_index), f64 exact."""
    L = L or lib()
    center = _f64(center, (-1, 3)); n = len(center)
    mi = np.asarray(mat_index, np.int64)
    cx, cy, cz = (np.ascontiguousarray(center[:, i]) for i in range(3))
    r = _f64(radius, (-1,)); kind = np.ascontiguousarray(np.asarray(mat_kind, np.uint32)[mi])
    alb = np.ascontiguousarray(_f64(mat_albedo, (-1, 3))[mi]); prm = np.ascontiguousarray(_f64(mat_param, (-1,))[mi])
    rc = L.rtiow_scene_save(str(path).encode(), n, _p(cx), _p(cy), _p(cz), _p(r), _p(kind), _p(alb), _p(prm))
    if rc != OK:
        raise RtiowError(rc, f"cannot write scene file {path}")


def load_scene(path, L=None):
    """rtiow_scene_load -> the dict of arrays random_scene returns (one material per sphere)."""
    L = L or lib()
    n = C.c_uint32(0)
    rc = L.rtiow_scene_load(str(path).encode(), 0, None, None, None, None, None, None, None, C.byref(n))
    if rc != OK:
        raise RtiowError(rc, f"cannot read scene file {path}")
    k = n.value
    cx, cy, cz, r = (np.zeros(max(k, 1)) for _ in range(4))
    kind = np.zeros(max(k, 1), np.uint32); alb = np.zeros((max(k, 1), 3)); prm = np.zeros(max(k, 1))
    rc = L.rtiow_scene_load(str(path).encode(), max(k, 1), _p(cx), _p(cy), _p(cz), _p(r), _p(kind), _p(alb), _p(prm), C.byref(n))
    if rc != OK:
        raise RtiowError(rc, f"malformed scene file {path}")
    return dict(center=np.stack([cx[:k], cy[:k], cz[:k]], 1), radius=r[:k].copy(), mat_index=np.arange(k, dtype=np.uint32),
                mat_kind=kind[:k].copy(), mat_albedo=alb[:k].copy(), mat_param=prm[:k].copy())


class Context:
    """rtiow_ctx: owns device buffers and streams.  Single caller (Send, !Sync).

    Context(n)                                  one process driving GPUs 0..n-1 (rtiow_ctx_create)
    Context(device=d)                           this process drives GPU d only; the caller owns any gather (rtiow_ctx_create_on_device)
    Context(device=d, rank=r, world=w, nccl_id) one process per GPU with the gather inside the library (rtiow_ctx_create_rank)
    """

    def __init__(self, n_gpus: int = 1, device: int | None = None, rank: int | None = None, world: int = 1, nccl_id: bytes | None = None):
        h = C.c_void_p()
        if rank is not None:
            if world > 1 and (nccl_id is None or len(nccl_id) != NCCL_UNIQUE_ID_BYTES):
                raise ValueError("nccl_id must be the 128 bytes of rank 0's nccl_unique_id()")
            _check(lib().rtiow_ctx_create_rank(0 if device is None else device, rank, world, nccl_id, C.byref(h)))
        elif device is None:
            _check(lib().rtiow_ctx_create(n_gpus, C.byref(h)))
        else:
            _check(lib().rtiow_ctx_create_on_device(device, C.byref(h)))
        self._h = h
        self.n_spheres = 0
        self.rank, self.world = (rank or 0), world

    def close(self):
        if getattr(self, "_h", None):
            lib().rtiow_ctx_destroy(self._h)
            self._h = None

    def set_scan_backend(self, backend: int):
        """SCAN_AUTO / SCAN_FP32 (FFMA2 filter on the CUDA cores) / SCAN_TENSOR (tcgen05 filter): same hits, same images."""
        _check(lib().rtiow_ctx_set_scan_backend(self._h, backend))

    def set_filter_bypass(self, on: bool):
        """testing aid: scenes uploaded while on get filter images that pass every sphere (the precise test sees all of them)"""
        _check(lib().rtiow_ctx_set_filter_bypass(self._h, int(bool(on))))

    def set_gather(self, mode: int):
        """GATHER_AUTO / GATHER_NCCL (tile buffers + ncclAllGather + de-interleave) / GATHER_FUSED (peer stores into rank 0's frame)"""
        _check(lib().rtiow_ctx_set_gather(self._h, mode))

    def set_stream(self, stream_ptr: int):
        """a one-device ctx works on this cudaStream_t from now on (0: back to its own)"""
        _check(lib().rtiow_ctx_set_stream(self._h, C.c_void_p(stream_ptr)))

    def gather_info(self) -> str:
        buf = C.create_string_buffer(512)
        _check(lib().rtiow_ctx_gather_info(self._h, buf, 512))
        return buf.value.decode()

    def render_rank(self, cam: Camera, params: Params, out: np.ndarray | None = None, want_frame: bool | None = None):
        """rtiow_render_rank (collective).  Rank 0 (or want_frame=True under the NCCL gather) receives the whole frame in host memory."""
        if want_frame is None:
            want_frame = self.rank == 0
        if want_frame and out is None:
            out = np.empty((params.height, params.width, 4), np.uint8)
        st = Stats()
        _check(lib().rtiow_render_rank(self._h, C.byref(cam), C.byref(params), _p(out) if want_frame else None, C.byref(st)))
        return (out if want_frame else None), st.as_dict()

    def render_rank_device(self, cam: Camera, params: Params):
        """rtiow_render_rank_device (collective): -> (device pointer of the whole frame or 0, stats)"""
        st = Stats(); ptr = C.c_void_p()
        _check(lib().rtiow_render_rank_device(self._h, C.byref(cam), C.byref(params), C.byref(ptr), C.byref(st)))
        return (ptr.value or 0), st.as_dict()

    def render_rank_enqueue(self, cam: Camera, params: Params) -> int:
        """rtiow_render_rank_enqueue (collective): one more frame on the ctx's stream, no host synchronisation -> device pointer or 0"""
        ptr = C.c_void_p()
        _check(lib().rtiow_render_rank_enqueue(self._h, C.byref(cam), C.byref(params), C.byref(ptr)))
        return ptr.value or 0

    def synchronize(self) -> dict:
        """rtiow_ctx_synchronize: wait for everything enqueued -> stats (mean kernel_ms of the enqueued frames)"""
        st = Stats()
        _check(lib().rtiow_ctx_synchronize(self._h, C.byref(st)))
        return st.as_dict()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---------------------------------------------------------------- scene / render
    def upload_scene(self, center, radius, mat_index, mat_kind, mat_albedo, mat_param):
        center = _f64(center, (-1, 3))
        cx, cy, cz = (np.ascontiguousarray(center[:, i]) for i in range(3))
        radius = _f64(radius, (-1,))
        mi = np.ascontiguousarray(mat_index, np.uint32)
        kind = np.ascontiguousarray(mat_kind, np.uint32)
        alb = _f64(mat_albedo, (-1, 3))
        ar, ag, ab = (np.ascontiguousarray(alb[:, i]) for i in range(3))
        prm = _f64(mat_param, (-1,))
        if not (len(cx) == len(radius) == len(mi)) or not (len(kind) == len(ar) == len(prm)):
            raise ValueError("scene arrays have inconsistent lengths")
        s = Spheres(_p(cx).value, _p(cy).value, _p(cz).value, _p(radius).value, _p(mi).value, len(radius))
        m = Materials(_p(kind).value, _p(ar).value, _p(ag).value, _p(ab).value, _p(prm).value, len(kind))
        _check(lib().rtiow_scene_upload(self._h, C.byref(s), C.byref(m)))
        self.n_spheres = len(radius)

    def render(self, cam: Camera, params: Params, out: np.ndarray | None = None):
        """rtiow_render: main.rs:122-145 -> (rgba[H,W,4] uint8 top-down, stats dict)."""
        if out is None:
            out = np.empty((params.height, params.width, 4), np.uint8)
        assert out.dtype == np.uint8 and out.size == params.height * params.width * 4 and out.flags.c_contiguous
        st = Stats()
        _check(lib().rtiow_render(self._h, C.byref(cam), C.byref(params), _p(out), C.byref(st)))
        return out, st.as_dict()

    AOVS = ("color", "albedo", "normal", "depth")

    def render_aov(self, cam: Camera, params: Params, out: np.ndarray | None = None, color=True, albedo=True, normal=True, depth=True):
        """rtiow_render_aov: the frame of render(cam, params), byte for byte, and float AOVs of it for a denoiser
        -> (rgba[H,W,4] uint8, {"color", "albedo", "normal": float32[H,W,3], "depth": float32[H,W]}, stats).
        Each AOV argument is True (allocate it), False / None (not computed: NULL, absent from the dict) or a C-contiguous
        float32 array of the right size that receives it.  Linear colour, the first hit's albedo and normal, and its depth are
        defined in include/rtiow_cuda.h."""
        h, w = params.height, params.width
        if out is None:
            out = np.empty((h, w, 4), np.uint8)
        if not isinstance(out, np.ndarray) or out.dtype != np.uint8 or out.size != h * w * 4 or not out.flags.c_contiguous:
            raise ValueError(f"out must be a C-contiguous uint8 array with {h * w * 4} elements")
        bufs = {}
        for name, arg in zip(self.AOVS, (color, albedo, normal, depth)):
            shape = (h, w) if name == "depth" else (h, w, 3)
            if arg is None or arg is False:
                continue
            if arg is True:
                arg = np.empty(shape, np.float32)
            elif (not isinstance(arg, np.ndarray) or arg.dtype != np.float32 or arg.size != int(np.prod(shape))
                  or not arg.flags.c_contiguous):
                raise ValueError(f"{name} must be a C-contiguous float32 array with {int(np.prod(shape))} elements")
            bufs[name] = arg.reshape(shape)
        st = Stats()
        ptrs = [_p(bufs[k]) if k in bufs else None for k in self.AOVS]
        _check(lib().rtiow_render_aov(self._h, C.byref(cam), C.byref(params), _p(out), *ptrs, C.byref(st)))
        return out.reshape(h, w, 4), bufs, st.as_dict()

    def render_adaptive(self, cam: Camera, params: Params, min_spp: int, tolerance: float, out: np.ndarray | None = None, spp_map=True,
                        error_map=True):
        """rtiow_render_adaptive: per-pixel sample counts in [min_spp, params.spp] driven by each pixel's own noise, every pixel
        byte-identical to render() at its own count -> (rgba[H,W,4] uint8, {"spp": uint32[H,W], "error": float32[H,W]}, stats).
        spp_map / error_map are True (allocate), False / None (not returned: NULL, absent from the dict) or a C-contiguous array
        of H*W uint32 / float32 that receives it.  Schedule, noise sums, error and rule are defined in include/rtiow_cuda.h."""
        h, w = params.height, params.width
        if out is None:
            out = np.empty((h, w, 4), np.uint8)
        if not isinstance(out, np.ndarray) or out.dtype != np.uint8 or out.size != h * w * 4 or not out.flags.c_contiguous:
            raise ValueError(f"out must be a C-contiguous uint8 array with {h * w * 4} elements")
        maps = {}
        for name, arg, dt in (("spp", spp_map, np.uint32), ("error", error_map, np.float32)):
            if arg is None or arg is False:
                continue
            if arg is True:
                arg = np.empty((h, w), dt)
            elif not isinstance(arg, np.ndarray) or arg.dtype != dt or arg.size != h * w or not arg.flags.c_contiguous:
                raise ValueError(f"{name} must be a C-contiguous {np.dtype(dt).name} array with {h * w} elements")
            maps[name] = arg.reshape(h, w)
        st = Stats()
        _check(lib().rtiow_render_adaptive(self._h, C.byref(cam), C.byref(params), min_spp, tolerance, _p(out),
                                           _p(maps["spp"]) if "spp" in maps else None, _p(maps["error"]) if "error" in maps else None,
                                           C.byref(st)))
        return out.reshape(h, w, 4), maps, st.as_dict()

    def render_views(self, cams, params: Params, out=None):
        """rtiow_render_views: many cameras of the uploaded scene in one call -> (rgba[K,H,W,4] uint8, stats of the batch).
        View v is byte-identical to render(cams[v], params).  `out` (K*H*W*4 contiguous uint8: a numpy array, or a CPU torch
        tensor such as a pin_memory() one) receives the frames."""
        cams = list(cams)
        k = len(cams)
        arr = (Camera * max(k, 1))(*cams)
        shape = (k, params.height, params.width, 4)
        if out is None:
            out = np.empty(shape, np.uint8)
        if isinstance(out, np.ndarray):
            if out.dtype != np.uint8 or out.size != int(np.prod(shape)) or not out.flags.c_contiguous:
                raise ValueError(f"out must be a C-contiguous uint8 array with {int(np.prod(shape))} elements")
            ptr = _p(out)
        else:                                 # a torch tensor (e.g. pinned host memory)
            if str(out.dtype) != "torch.uint8" or out.numel() != int(np.prod(shape)) or not out.is_contiguous() or out.device.type != "cpu":
                raise ValueError(f"out must be a contiguous CPU uint8 tensor with {int(np.prod(shape))} elements")
            ptr = C.c_void_p(out.data_ptr())
        st = Stats()
        _check(lib().rtiow_render_views(self._h, arr, k, C.byref(params), ptr, C.byref(st)))
        return out.reshape(shape), st.as_dict()

    def render_progressive(self, cam: Camera, params: Params, n_passes: int, on_pass=None, out: np.ndarray | None = None):
        """rtiow_render_progressive: the spp samples in n_passes slices; on_pass(pass_1based, n_passes, spp_done, rgba[H,W,4] view)
        is called after each (return True to cancel -> RtiowError ERR_CANCELLED).  -> (final rgba, stats summed over passes)."""
        if out is None:
            out = np.empty((params.height, params.width, 4), np.uint8)
        assert out.dtype == np.uint8 and out.size == params.height * params.width * 4 and out.flags.c_contiguous
        view = out.reshape(params.height, params.width, 4)

        def tramp(_user, k, n, done, _rgba):
            return 1 if (on_pass is not None and on_pass(int(k), int(n), int(done), view)) else 0

        st = Stats()
        cb = PROGRESS_FN(tramp)              # kept alive for the duration of the call
        _check(lib().rtiow_render_progressive(self._h, C.byref(cam), C.byref(params), n_passes, cb, None, _p(out), C.byref(st)))
        return out, st.as_dict()

    def tile_buffer_bytes(self, params: Params, world: int) -> int:
        n = C.c_size_t(0)
        _check(lib().rtiow_tile_buffer_bytes(C.byref(params), world, C.byref(n)))
        return n.value

    def render_tiles_device(self, cam, params, rank, world, d_tiles_ptr: int, stream_ptr: int = 0, want_stats=False):
        st = Stats()
        _check(lib().rtiow_render_tiles_device(self._h, C.byref(cam), C.byref(params), rank, world, C.c_void_p(d_tiles_ptr),
                                               C.c_void_p(stream_ptr), C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None

    def render_to_frame_device(self, cam, params, rank, world, d_frame_ptr: int, stream_ptr: int = 0, want_stats=False):
        """this rank's rows stored straight into the whole frame at d_frame_ptr (may be another GPU's memory): gather fused into the epilogue"""
        st = Stats()
        _check(lib().rtiow_render_to_frame_device(self._h, C.byref(cam), C.byref(params), rank, world, C.c_void_p(d_frame_ptr),
                                                  C.c_void_p(stream_ptr), C.byref(st) if want_stats else None))
        return st.as_dict() if want_stats else None

    def deinterleave_device(self, d_gathered_ptr: int, params, world, d_frame_ptr: int, stream_ptr: int = 0):
        _check(lib().rtiow_deinterleave_device(self._h, C.c_void_p(d_gathered_ptr), C.byref(params), world,
                                               C.c_void_p(d_frame_ptr), C.c_void_p(stream_ptr)))

    # ---------------------------------------------------------------- unit-level batches
    def sphere_hit_batch(self, center, radius, orig, direction, t_min, t_max, precision=F32):
        center, orig, direction = _f64(center, (-1, 3)), _f64(orig, (-1, 3)), _f64(direction, (-1, 3))
        n = len(center)
        radius = _f64(np.broadcast_to(radius, (n,))); t_min = _f64(np.broadcast_to(t_min, (n,))); t_max = _f64(np.broadcast_to(t_max, (n,)))
        hit = np.zeros(n, np.int32); t = np.zeros(n); p = np.zeros((n, 3)); nrm = np.zeros((n, 3)); ff = np.zeros(n, np.int32)
        _check(lib().rtiow_sphere_hit_batch(self._h, precision, n, _p(center), _p(radius), _p(orig), _p(direction), _p(t_min),
                                            _p(t_max), _p(hit), _p(t), _p(p), _p(nrm), _p(ff)))
        return dict(hit=hit, t=t, p=p, normal=nrm, front_face=ff)

    def hitlist_batch(self, orig, direction, t_min=1e-4, precision=F32):
        orig, direction = _f64(orig, (-1, 3)), _f64(direction, (-1, 3))
        n = len(orig)
        hit = np.zeros(n, np.int32); idx = np.zeros(n, np.int32); t = np.zeros(n); p = np.zeros((n, 3)); nrm = np.zeros((n, 3))
        ff = np.zeros(n, np.int32)
        _check(lib().rtiow_hitlist_batch(self._h, precision, n, _p(orig), _p(direction), t_min, _p(hit), _p(idx), _p(t), _p(p),
                                         _p(nrm), _p(ff)))
        return dict(hit=hit, index=idx, t=t, p=p, normal=nrm, front_face=ff)

    def scatter_batch(self, kind, albedo, param, r_orig, r_dir, p, normal, front_face, sample, precision=F32):
        kind = np.ascontiguousarray(kind, np.int32); n = len(kind)
        albedo, r_orig, r_dir = _f64(albedo, (n, 3)), _f64(r_orig, (n, 3)), _f64(r_dir, (n, 3))
        p, normal, sample = _f64(p, (n, 3)), _f64(normal, (n, 3)), _f64(sample, (n, 3))
        param = _f64(param, (n,)); front_face = np.ascontiguousarray(front_face, np.int32)
        some = np.zeros(n, np.int32); att = np.zeros((n, 3)); so = np.zeros((n, 3)); sd = np.zeros((n, 3))
        _check(lib().rtiow_scatter_batch(self._h, precision, n, _p(kind), _p(albedo), _p(param), _p(r_orig), _p(r_dir), _p(p),
                                         _p(normal), _p(front_face), _p(sample), _p(some), _p(att), _p(so), _p(sd)))
        return dict(some=some, attenuation=att, orig=so, dir=sd)

    def get_ray_batch(self, cam: Camera, s, t, disk_xy, precision=F32):
        s, t, disk_xy = _f64(s, (-1,)), _f64(t, (-1,)), _f64(disk_xy, (-1, 2))
        n = len(s); o = np.zeros((n, 3)); d = np.zeros((n, 3))
        _check(lib().rtiow_get_ray_batch(self._h, precision, C.byref(cam), n, _p(s), _p(t), _p(disk_xy), _p(o), _p(d)))
        return dict(orig=o, dir=d)

    def to_rgba_batch(self, color, alpha, spp, precision=F32):
        color = _f64(color, (-1, 3)); out = np.zeros((len(color), 4), np.uint8)
        _check(lib().rtiow_to_rgba_batch(self._h, precision, len(color), _p(color), alpha, spp, _p(out)))
        return out

    def reflect_batch(self, v, n, precision=F32):
        v, n = _f64(v, (-1, 3)), _f64(n, (-1, 3)); out = np.zeros_like(v)
        _check(lib().rtiow_reflect_batch(self._h, precision, len(v), _p(v), _p(n), _p(out)))
        return out

    def refract_batch(self, uv, n, eta, precision=F32):
        uv, n = _f64(uv, (-1, 3)), _f64(n, (-1, 3)); eta = _f64(np.broadcast_to(eta, (len(uv),))); out = np.zeros_like(uv)
        _check(lib().rtiow_refract_batch(self._h, precision, len(uv), _p(uv), _p(n), _p(eta), _p(out)))
        return out

    def ray_color_batch(self, orig, direction, pixel, sample, seed, max_depth=50, t_min=1e-4, precision=F32):
        orig, direction = _f64(orig, (-1, 3)), _f64(direction, (-1, 3)); n = len(orig)
        pixel = np.ascontiguousarray(pixel, np.uint32); sample = np.ascontiguousarray(sample, np.uint32)
        col = np.zeros((n, 3)); rays = np.zeros(n, np.uint64)
        _check(lib().rtiow_ray_color_batch(self._h, precision, n, _p(orig), _p(direction), _p(pixel), _p(sample), seed, max_depth,
                                           t_min, _p(col), _p(rays)))
        return dict(color=col, rays=rays)

    def ray_color_trace_batch(self, orig, direction, pixel, sample, seed, max_depth=50, t_min=1e-4, precision=F32):
        """ray_color_batch + every ray of every path: index[n][max_depth] (list index hit, -1 = miss / no ray), ray[n][max_depth][6]"""
        orig, direction = _f64(orig, (-1, 3)), _f64(direction, (-1, 3)); n = len(orig)
        pixel = np.ascontiguousarray(pixel, np.uint32); sample = np.ascontiguousarray(sample, np.uint32)
        col = np.zeros((n, 3)); rays = np.zeros(n, np.uint64)
        idx = np.full((n, max_depth), -1, np.int32); ray = np.zeros((n, max_depth, 6))
        _check(lib().rtiow_ray_color_trace_batch(self._h, precision, n, _p(orig), _p(direction), _p(pixel), _p(sample), seed, max_depth,
                                                 t_min, _p(col), _p(rays), _p(idx), _p(ray)))
        return dict(color=col, rays=rays, index=idx, ray=ray)

    def sampler_batch(self, pixel, sample, bounce, seed, precision=F32):
        pixel = np.ascontiguousarray(pixel, np.uint32); sample = np.ascontiguousarray(sample, np.uint32)
        bounce = np.ascontiguousarray(bounce, np.uint32); n = len(pixel); out = np.zeros((n, 12))
        _check(lib().rtiow_sampler_batch(self._h, precision, n, _p(pixel), _p(sample), _p(bounce), seed, _p(out)))
        return out

    # ---------------------------------------------------------------- measurement
    def fp32_peak_probe(self, packed=True, target_ms=200.0):
        tf, ms = C.c_double(0), C.c_double(0)
        _check(lib().rtiow_fp32_peak_probe(self._h, int(packed), target_ms, C.byref(tf), C.byref(ms)))
        return tf.value, ms.value

    def flush_l2(self):
        _check(lib().rtiow_flush_l2(self._h))
