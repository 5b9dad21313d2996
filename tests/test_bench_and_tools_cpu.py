"""CPU checks of the measurement code: every script under tools/ and the driver entry points compile, and bench.py's two rooflines
do the arithmetic DESIGN.md §1.2 / §6 state (17 algorithmic FLOP per test against the FP32 pipe; 2 MMAs x K = 16 x 2 = 64 executed
FLOP per (ray, padded sphere) against the measured dense bf16 peak; traffic from the ncu capture of the same launch)."""
import importlib.util
import json
import py_compile
import types
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("path", sorted(str(p.relative_to(ROOT)) for p in list((ROOT / "tools").glob("*.py")) + [ROOT / "bench.py", ROOT / "__graft_entry__.py"]))
def test_scripts_compile(path, tmp_path):
    py_compile.compile(str(ROOT / path), cfile=str(tmp_path / "compiled.pyc"), doraise=True)      # the byte code goes to tmp_path, not into the tree


def _bench():
    spec = importlib.util.spec_from_file_location("bench_under_test", ROOT / "bench.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)                      # guarded by __name__ == "__main__": importing runs nothing
    return mod


def test_rooflines_of_the_bench_line():
    b = _bench()
    assert b.FLOP_PER_TEST == 17 and b.TENSOR_FLOP_PER_TEST == 64
    args = types.SimpleNamespace(config="cfg2", width=1200, height=675, spp=500)
    paths = 1200 * 675 * 500
    rays = 2.6542 * paths
    kms = 76.6
    main, fp32 = b.roofline_objects(1, kms, rays, 530, 576, True, 74.3, 37.0, args, paths, "rt::render_kernel_umma<6,64>")
    assert main["bound"] == "tensor" and fp32["bound"] == "fp32"
    assert fp32["achieved"] == pytest.approx(rays * 530 * 17 / (kms * 1e-3) / 1e12) and fp32["frac"] == pytest.approx(fp32["achieved"] / 74.3)
    assert main["achieved"] == pytest.approx(rays * 576 * 64 / (kms * 1e-3) / 1e12) and main["frac"] == pytest.approx(main["achieved"] / main["peak"])
    assert 1.6 < fp32["frac"] < 1.8 and 0.3 < main["frac"] < 0.45                      # the committed bench line: 1.70 and 0.38
    side = json.loads((ROOT / "profiles" / "r2_dram_bytes.json").read_text())["cfg2:rt::render_kernel_umma<6,64>"]
    assert main["traffic"] == side["dram_bytes"] and "ncu" in main["traffic_note"]     # from the ncu capture of this exact launch
    # N ranks: per-GPU figures
    main8, fp8 = b.roofline_objects(8, kms / 8, rays, 530, 576, True, 74.3, 37.0, args, paths, "rt::render_kernel_umma<6,64>")
    assert fp8["achieved"] == pytest.approx(fp32["achieved"]) and main8["traffic"] is None
    # the FP32-filter kernel reports the FP32 roofline as its main one
    m32, f32 = b.roofline_objects(1, 3900.0, 2.8011 * 530841600, 10203, 10203, False, 74.3, 37.0, args, 530841600, "rt::render_kernel<float,true,768,1>")
    assert m32["bound"] == "fp32" and m32["achieved"] == pytest.approx(f32["achieved"]) and 0.85 < m32["frac"] < 0.92


def test_both_arms_describe_the_same_workload():
    b = _bench()
    args = types.SimpleNamespace(workload="w", width=1200, height=675, spp=500)
    cfg = b.make_config(args, 530)
    assert set(cfg) >= {"workload", "width", "height", "spp", "max_depth", "n_spheres", "cache"} and "model" not in cfg
