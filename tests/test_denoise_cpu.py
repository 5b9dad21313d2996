"""CPU suite for rtiow_denoise: the library carries exactly the three denoise kernels, the ctypes binding checks the buffers it is
handed before it calls the library, rtiow_denoise_params matches the Rust -sys struct field by field, every layer exposes the
call, and the numpy restatement the GPU tests compare against (np_denoise.denoise) equals a plain scalar loop bit for bit."""
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import np_denoise
from test_rust_header_lock import c_structs, rust_structs

ROOT = Path(__file__).resolve().parent.parent
DENOISE_KERNELS = {"denoise_prepare_kernel<256>", "denoise_level_kernel<256>", "denoise_finish_kernel<256>"}


def test_library_carries_exactly_the_denoise_kernels(capi):
    syms = subprocess.run(["cuobjdump", "-symbols", str(capi.lib_path())], capture_output=True, text=True, check=True).stdout
    names = subprocess.run(["c++filt"], input=syms, capture_output=True, text=True, check=True).stdout
    found = set(re.findall(r"rt::(denoise_\w+_kernel<[^>]*>)", names))
    assert found == DENOISE_KERNELS, f"unexpected: {sorted(found - DENOISE_KERNELS)}, missing: {sorted(DENOISE_KERNELS - found)}"


def _unbound_ctx(capi):
    ctx = object.__new__(capi.Context)         # the checks run before the library is called: no ctx handle is needed
    ctx._h = None
    return ctx


def _inputs(h=9, w=16):
    return dict(color=np.zeros((h, w, 3), np.float32), albedo=np.zeros((h, w, 3), np.float32), normal=np.zeros((h, w, 3), np.float32),
                depth=np.zeros((h, w), np.float32))


@pytest.mark.parametrize("name", ["color", "albedo", "normal", "depth"])
@pytest.mark.parametrize("bad", ["short", "long", "float64", "strided"])
def test_binding_rejects_wrongly_sized_inputs(capi, name, bad):
    ins = _inputs()
    a = ins[name]
    ins[name] = {"short": a.reshape(-1)[:-1], "long": np.zeros(a.size + 3, np.float32), "float64": a.astype(np.float64),
                 "strided": np.zeros(a.shape[:-1] + (2 * a.shape[-1],), np.float32)[..., ::2]}[bad]
    with pytest.raises(ValueError, match=name):
        _unbound_ctx(capi).denoise(**ins)


@pytest.mark.parametrize("name,shape,dtype", [("out_color", (9, 16, 3), np.float32), ("out_rgba", (9, 16, 4), np.uint8)])
@pytest.mark.parametrize("bad", ["short", "long", "dtype", "strided"])
def test_binding_rejects_wrongly_sized_outputs(capi, name, shape, dtype, bad):
    n = int(np.prod(shape))
    other = np.uint8 if dtype == np.float32 else np.float32
    arr = {"short": np.zeros(n - 1, dtype), "long": np.zeros(n + 1, dtype), "dtype": np.zeros(n, other),
           "strided": np.zeros(2 * n, dtype)[::2]}[bad]
    with pytest.raises(ValueError, match=name):
        _unbound_ctx(capi).denoise(**_inputs(), **{name: arr})


def test_binding_rejects_no_output(capi):
    with pytest.raises(ValueError, match="both"):
        _unbound_ctx(capi).denoise(**_inputs(), out_color=None, out_rgba=False)


def test_params_struct_matches_rust_in_order(capi):
    c, r = c_structs(), rust_structs()
    fields = ["levels", "sigma_color", "sigma_normal", "sigma_depth", "alpha", "reserved"]
    assert c["rtiow_denoise_params"] == r["rtiow_denoise_params"] == fields
    assert [f for f, _ in capi.DenoiseParams._fields_] == fields


def test_defaults_are_valid(capi):
    dp = capi.default_denoise_params()
    assert 0 <= dp.levels <= 10 and dp.alpha == 255
    for s in (dp.sigma_color, dp.sigma_normal, dp.sigma_depth):
        assert s >= 1e-12


def test_every_layer_exposes_the_call(capi):
    from rtiow_b200 import api
    assert callable(api.denoise) and callable(capi.Context.denoise)
    for sym in ("rtiow_denoise", "rtiow_denoise_params_default"):
        assert sym in capi.SYMBOLS and hasattr(capi.lib(), sym)
    hdr = (ROOT / "include" / "rtiow_cuda.h").read_text()
    assert re.search(r"int\s+rtiow_denoise\(rtiow_ctx\* ctx, uint32_t width, uint32_t height, const float\* color, const float\* albedo, "
                     r"const float\* normal,\s+const float\* depth, const rtiow_denoise_params\* dp, float\* out_color, uint8_t\* out_rgba, "
                     r"rtiow_stats\* stats\);", hdr)
    rs = (ROOT / "rust" / "rtiow-gpu" / "gpu.rs").read_text()
    assert re.search(r"pub fn denoise\(", rs)
    hpp = (ROOT / "rtiow_b200" / "host" / "rtiow.hpp").read_text()
    assert re.search(r"inline \S+ denoise\(", hpp)
    ex = (ROOT / "rtiow_b200" / "host" / "example_main.cpp").read_text()
    assert "--denoise" in ex and "_denoised.png" in ex


def _random_aovs(rng, h, w):
    """values across the whole valid range: colour up to 2^32, albedo 0 (the floor) to 1, unit-ish normals, depths 0, finite
    and +inf, and some exact ties"""
    color = (rng.random((h, w, 3)) * rng.choice([1.0, 4.0, 1e3, 2.0 ** 32], (h, w, 1))).astype(np.float32)
    color.reshape(-1)[::7] = 0
    albedo = rng.random((h, w, 3)).astype(np.float32)
    albedo.reshape(-1)[::5] = 0
    albedo.reshape(-1)[::11] = 1
    normal = (rng.random((h, w, 3)) * 2 - 1).astype(np.float32)
    normal.reshape(-1)[::13] = 1
    depth = (rng.random((h, w)) * 20).astype(np.float32)
    depth.reshape(-1)[::3] = np.inf
    depth.reshape(-1)[::8] = 0
    depth.reshape(-1)[1::9] = 65536
    return color, albedo, normal, depth


@pytest.mark.parametrize("h,w", [(5, 7), (9, 1), (1, 9)])
@pytest.mark.parametrize("levels", [0, 1, 2, 3])
@pytest.mark.parametrize("sigmas", [(0.5, 0.3, 0.2), (1e-12, 1e-12, 1e-12), (np.inf, np.inf, np.inf), (4.0, np.inf, 0.05)])
def test_restatement_equals_a_scalar_loop(h, w, levels, sigmas):
    rng = np.random.default_rng(h * 100 + w * 10 + levels)
    args = _random_aovs(rng, h, w)
    yv, rv = np_denoise.denoise(*args, levels, *sigmas, alpha=200)
    ys, rs = np_denoise.denoise_scalar(*args, levels, *sigmas, alpha=200)
    assert yv.dtype == ys.dtype == np.float32
    assert np.array_equal(yv.view(np.uint32), ys.view(np.uint32))
    assert np.array_equal(rv, rs) and (rv[..., 3] == 200).all()
    assert np.isfinite(yv).all()
