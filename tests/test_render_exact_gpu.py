"""GPU suite: rtiow_render byte-identical to the f64 oracle on every robust pixel, on every scan arm, on the edge scenes and
parameter sweeps of tests/edge_scenes.py.

A pixel is robust when no ray of its paths comes near a decision an f32 render could take the other way and its exact value
is not near a quantisation step (oracle.robust_pixels, o_render_margins; tests/test_oracle_margins.py checks the margin
against f32-sized perturbations and records each case's robust fraction).  For each (case, arm):
  * rtiow_stats.scan_backend is the arm scan_scenes.scan_arm expects;
  * RGB equals the oracle's on every robust pixel, and alpha on every pixel;
  * the other pixels keep the bar of test_render_vs_oracle (at most 1 % more than 1 LSB off), and rays_traced that of
    the oracle's ray count (0.5 %).
The oracle renders once per case (lru_cache); render_views, render_progressive and the tile partitions are byte-identical to
rtiow_render (tests/test_render_views_gpu.py and others), so one render per case stands for them.
"""
from functools import lru_cache

import numpy as np
import pytest

import edge_scenes as es
import scan_scenes as ss

pytestmark = pytest.mark.gpu

AUTO, FP32, F64 = "auto", "fp32", "f64"
F64_CASES = {"final", "glass", "contact", "lambert"}
BLACK = {"mirror-box"}          # no path reaches the sky: the whole frame is black whatever the paths


def _arms(cid, name):
    if cid.startswith(("final[", "glass[")):
        return [AUTO]
    arms = [AUTO] if name in ("final-h28", "grid") else [AUTO, FP32]
    return arms + ([F64] if cid in F64_CASES else [])


CASES = [(cid, arm) for cid, name, _ in es.CASES for arm in _arms(cid, name)]


@lru_cache(maxsize=None)
def _oracle_render(cid, oracle):
    _, name, p = es.CASE[cid]
    arrays = es.build(name)
    img, acc, mg, cnt = oracle.render_margins(oracle.Scene(**arrays), es.camera(oracle, name, p), p["W"], p["H"], p["spp"],
                                              p["max_depth"], p["t_min"], p["seed"])
    rob = np.ones(mg.shape, bool) if name in BLACK else oracle.robust_pixels(acc, mg, p["spp"])
    return img, acc, rob, cnt


@pytest.fixture()
def scan(ctx, capi):
    yield ctx
    ctx.set_scan_backend(capi.SCAN_AUTO)


@pytest.mark.parametrize("cid,arm", CASES)
def test_render_exact(scan, capi, oracle, cid, arm):
    _, name, p = es.CASE[cid]
    arrays = es.build(name)
    ref, acc, rob, cnt = _oracle_render(cid, oracle)
    if name in BLACK:
        assert not acc.any()
    backend = capi.SCAN_FP32 if arm == FP32 else capi.SCAN_AUTO
    want = ss.scan_arm(arrays, backend, capi.F64 if arm == F64 else capi.F32)[0]
    scan.upload_scene(**arrays)
    scan.set_scan_backend(backend)
    prm = capi.default_params(width=p["W"], height=p["H"], spp=p["spp"], max_depth=p["max_depth"], t_min=p["t_min"],
                              seed=p["seed"], precision=capi.F64 if arm == F64 else capi.F32)
    img, st = scan.render(es.camera(capi, name, p), prm)
    if arm != F64:
        assert st["scan_backend"] == (capi.SCAN_TENSOR if want == "Tensor" else capi.SCAN_FP32), want
    if cid in ("final", "final-h28[W=40,H=24,spp=4]", "grid[W=32,H=18,spp=4]"):
        assert want == {"final": "Tensor" if arm == AUTO else "Smem" if arm == FP32 else "F64",
                        "final-h28": "Wide", "grid": "Global"}[name]
    assert (img[..., 3] == ref[..., 3]).all()
    off = (img[..., :3] != ref[..., :3]).any(-1)
    bad = np.argwhere(off & rob)
    assert len(bad) == 0, (f"{len(bad)} of {rob.sum()} robust pixels differ, e.g. row {bad[0][0]} col {bad[0][1]}: "
                           f"{img[tuple(bad[0])][:3]} vs the oracle's {ref[tuple(bad[0])][:3]}")
    diff = np.abs(img[..., :3].astype(int) - ref[..., :3].astype(int)).max(axis=2)
    assert (diff > 1).sum() <= max(1, 0.01 * diff.size), f"{(diff > 1).mean():.4%} pixels off by > 1 LSB"
    assert abs(st["rays_traced"] - cnt["rays"]) <= max(5e-3 * cnt["rays"], 2), (st["rays_traced"], cnt["rays"])
