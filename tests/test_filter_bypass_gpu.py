"""GPU suite: both sphere filters drop no hit, checked exactly against the same kernels with the filter bypassed.

The FP32 filter (7 FFMA2 per sphere pair, rt_scene.cuh) and the tensor filter (a tcgen05 contraction with an fp16 hi/lo split
and an fp16 accumulator, rt_umma*.cuh) are conservative filters in front of the same precise test: they may pass spheres the
test rejects, never drop one it accepts.  With rtiow_ctx_set_filter_bypass on, the scene upload builds a filter table and a
tensor image that pass every real sphere for every ray (and never pass padding), so the same kernels, with the same SASS and
on the same scan arm, run the precise test on every sphere.  Whatever differs between the two uploads is a hit a filter
dropped, so every comparison here is byte for byte, with no tolerance and no robustness mask:
  * hitlists (rtiow_hitlist_batch) on rays built at sphere silhouettes, inside the bands where each filter's rounding
    decides (scan_scenes.silhouette_rays; each scene asserts that several hundred rays fall inside each band), and on
    scan_scenes.rays, for every scan_scenes.SCENES entry on its AUTO and FP32 arms, the edge scenes and a scene 360 units off
    the coordinate origin;
  * paths (rtiow_ray_color_trace_batch) on the edge scenes: bounce rays start on a sphere (candidate_self beside the filter);
  * frames (rtiow_render): every edge_scenes.CASES case on the arms test_render_exact_gpu.py runs, and a small frame of
    every scan_scenes.SCENES entry.
"""
import numpy as np
import pytest

import edge_scenes as es
import scan_scenes as ss
from test_parity_unit_gpu import f32
from test_render_exact_gpu import CASES as EXACT_CASES

pytestmark = pytest.mark.gpu

AUTO, FP32 = "auto", "fp32"
EDGE_HIT = ["contact", "shells", "glass-inside", "lambert"]
EDGE_PATH = EDGE_HIT + ["mirror-box"]


def far_scene():
    """test_parity_unit_gpu's scene 360 units off the coordinate origin: R ~ 370 (no tensor image), a large FP32 slack"""
    rng = np.random.default_rng(5)
    n = 300
    c = f32(np.array([300.0, 50.0, -200.0]) + rng.uniform(-8, 8, (n, 3))); r = f32(rng.uniform(0.1, 0.8, n))
    return dict(center=c, radius=r, mat_index=np.zeros(n, np.uint32), mat_kind=[0], mat_albedo=[[1.0, 1.0, 1.0]], mat_param=[0.0])


def _arrays(name, capi):
    if name in ss.SCENES:
        return ss.build(name, capi)
    return far_scene() if name == "far-360" else es.build(name)


def _backend(capi, arm):
    return capi.SCAN_FP32 if arm == FP32 else capi.SCAN_AUTO


def _arm_cases(names):
    """(name, arm) for AUTO, and for FP32 where that selects another arm than AUTO does"""
    out = []
    for name in names:
        if name in ss.SCENES:
            arms = ss.SCENES[name][1]
            auto, fp32 = arms[ss.SCAN_AUTO], arms[ss.SCAN_FP32]
        else:
            auto, fp32 = (ss.scan_arm(_arrays(name, None), b)[0] for b in (ss.SCAN_AUTO, ss.SCAN_FP32))
        out += [(name, AUTO)] + ([(name, FP32)] if fp32 != auto else [])
    return out


HIT_CASES = _arm_cases(list(ss.SCENES) + EDGE_HIT + ["far-360"])
PATH_CASES = _arm_cases(EDGE_PATH)
FRAME_CASES = [(cid, arm) for cid, arm in EXACT_CASES if arm in (AUTO, FP32)]
SCENE_FRAME_CASES = _arm_cases(list(ss.SCENES))


@pytest.fixture()
def bypass(ctx, capi):
    """compare(arrays, arm, run) -> (run(ctx) with the filter, run(ctx) with it bypassed), each on its own upload of the
    scene; afterwards bypass is off, the backend AUTO and the last scene uploaded again without it"""
    last = {}

    def compare(arrays, arm, run):
        ctx.set_scan_backend(_backend(capi, arm))
        last["arrays"] = arrays
        out = []
        for on in (False, True):
            ctx.set_filter_bypass(on)
            ctx.upload_scene(**arrays)
            out.append(run(ctx))
        ctx.set_filter_bypass(False)
        return out

    yield compare
    ctx.set_filter_bypass(False)
    ctx.set_scan_backend(capi.SCAN_AUTO)
    if "arrays" in last:
        ctx.upload_scene(**last["arrays"])


def _differ(a, b):
    """per item along the first axis: does any byte differ"""
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    assert a.shape == b.shape and a.dtype == b.dtype
    return (a.view(np.uint8).reshape(len(a), -1) != b.view(np.uint8).reshape(len(b), -1)).any(1)


def _assert_same(got, want, keys, what, n_first=None):
    bad = np.zeros(len(want[keys[0]]), bool)
    for k in keys:
        bad |= _differ(got[k], want[k])
    if bad.any():
        i = int(np.flatnonzero(bad)[0])
        fields = [k for k in keys if _differ(got[k], want[k]).any()]
        head = f" ({int(bad[:n_first].sum())} of them silhouette rays)" if n_first is not None else ""
        raise AssertionError(f"{int(bad.sum())} of {len(bad)} {what} differ from the bypassed filter{head} in {fields}; "
                             f"first: #{i} " + ", ".join(f"{k} {got[k][i]} vs {want[k][i]}" for k in fields))


@pytest.mark.parametrize("name,arm", HIT_CASES)
def test_hitlist_drops_no_hit(bypass, capi, name, arm):
    arrays = _arrays(name, capi)
    o1, d1, target = ss.silhouette_rays(arrays)
    cov = ss.assert_band_coverage(arrays, o1, d1, target)
    print(f"\n{name} [{ss.scan_arm(arrays, _backend(capi, arm))[0]}] rays in each band: {cov}")
    o2, d2 = ss.rays(name, arrays)
    o, d = np.concatenate([o1, o2]), np.concatenate([d1, d2])
    got, want = bypass(arrays, arm, lambda ctx: ctx.hitlist_batch(o, d))
    assert 0.1 < want["hit"][:len(o1)].mean() < 1.0
    _assert_same(got, want, ("hit", "index", "t", "p", "normal", "front_face"), "rays", n_first=len(o1))


def _camera_rays(name, n, rng):
    look_from, look_at = (np.asarray(v, float) for v in es.SCENES[name][1][:2])
    o = look_from + 0.05 * rng.normal(size=(n, 3))
    d = look_at + 2.5 * rng.normal(size=(n, 3)) - o
    return f32(o), f32(d)


@pytest.mark.parametrize("name,arm", PATH_CASES)
def test_paths_drop_no_hit(bypass, capi, name, arm):
    arrays = es.build(name)
    rng = np.random.default_rng(12)
    depth, n = (200, 2000) if name == "mirror-box" else (50, 4000)
    o1, d1 = _camera_rays(name, n, rng)
    o2, d2, _ = ss.silhouette_rays(arrays)
    pick = rng.choice(len(o2), n, replace=False)
    o, d = np.concatenate([o1, o2[pick]]), np.concatenate([d1, d2[pick]])
    px = rng.integers(0, 1 << 20, len(o)).astype(np.uint32); sm = rng.integers(0, 500, len(o)).astype(np.uint32)
    got, want = bypass(arrays, arm, lambda ctx: ctx.ray_color_trace_batch(o, d, px, sm, seed=13, max_depth=depth))
    assert want["rays"].max() > 3
    _assert_same(got, want, ("color", "rays", "index", "ray"), "paths")


def _assert_same_frame(got, want):
    (a, sa), (b, sb) = got, want
    off = (a != b).any(-1)
    assert not off.any(), f"{int(off.sum())} of {off.size} pixels differ from the bypassed filter, e.g. {np.argwhere(off)[0]}"
    assert sa["rays_traced"] == sb["rays_traced"] and sa["scan_backend"] == sb["scan_backend"], (sa, sb)


@pytest.mark.parametrize("cid,arm", FRAME_CASES)
def test_edge_frames_drop_no_hit(bypass, capi, cid, arm):
    _, name, p = es.CASE[cid]
    arrays = es.build(name)
    prm = capi.default_params(width=p["W"], height=p["H"], spp=p["spp"], max_depth=p["max_depth"], t_min=p["t_min"], seed=p["seed"])
    cam = es.camera(capi, name, p)
    got, want = bypass(arrays, arm, lambda ctx: ctx.render(cam, prm))
    arm_name = ss.scan_arm(arrays, _backend(capi, arm))[0]
    assert got[1]["scan_backend"] == (capi.SCAN_TENSOR if arm_name == "Tensor" else capi.SCAN_FP32), arm_name
    _assert_same_frame(got, want)


@pytest.mark.parametrize("name,arm", SCENE_FRAME_CASES)
def test_scene_frames_drop_no_hit(bypass, capi, name, arm):
    arrays = ss.build(name, capi)
    _, mid, ext, eye = ss.framing(arrays)
    W, H = 32, 18
    cam = capi.camera_new(eye, mid, (0.0, 1.0, 0.0), 40.0, W / H, 0.0, float(np.linalg.norm(eye - mid)))
    prm = capi.default_params(width=W, height=H, spp=2, seed=5)
    got, want = bypass(arrays, arm, lambda ctx: ctx.render(cam, prm))
    arm_name = ss.scan_arm(arrays, _backend(capi, arm))[0]
    assert got[1]["scan_backend"] == (capi.SCAN_TENSOR if arm_name == "Tensor" else capi.SCAN_FP32), arm_name
    _assert_same_frame(got, want)
