"""CPU suite for rtiow_render_aov: the library carries one AOV render kernel per scan-plan arm, and the ctypes binding checks
the buffers it is handed before it calls the library."""
import re
import subprocess

import numpy as np
import pytest

AOV_KERNELS = {
    "render_aov_kernel<double, false, 256, 2>",     # F64
    "render_aov_kernel<float, true, 256, 3>",       # Smem
    "render_aov_kernel<float, true, 768, 1>",       # Wide, 768 threads
    "render_aov_kernel<float, true, 512, 1>",       # Wide, 512 threads
    "render_aov_kernel<float, false, 256, 4>",      # Global
    "render_aov_kernel_umma<6, 64>",                # Tensor
}


def test_aov_kernels_are_the_plan_arms(capi):
    """one render_aov_kernel per arm of the scan plan, the same instantiations as render_kernel's, and the float epilogue"""
    syms = subprocess.run(["cuobjdump", "-symbols", str(capi.lib_path())], capture_output=True, text=True, check=True).stdout
    names = subprocess.run(["c++filt"], input=syms, capture_output=True, text=True, check=True).stdout
    found = set(re.findall(r"rt::(render_aov_kernel(?:_umma)?<[^>]*>)", names))
    assert found == AOV_KERNELS, f"unexpected: {sorted(found - AOV_KERNELS)}, missing: {sorted(AOV_KERNELS - found)}"
    frame = set(re.findall(r"rt::render_kernel((?:_umma)?<[^>]*>)", names))
    assert {n.replace("render_aov_kernel", "") for n in AOV_KERNELS} == frame
    assert "rt::finalize_aov_kernel(" in names


def _unbound_ctx(capi):
    ctx = object.__new__(capi.Context)         # the checks run before the library is called: no ctx handle is needed
    ctx._h = None
    return ctx


@pytest.mark.parametrize("name", ["color", "albedo", "normal", "depth"])
@pytest.mark.parametrize("bad", ["short", "long", "float64", "strided"])
def test_binding_rejects_wrongly_sized_buffers(capi, name, bad):
    per_px = 1 if name == "depth" else 3
    n = 9 * 16 * per_px
    arr = {"short": np.zeros(n - 1, np.float32), "long": np.zeros(n + per_px, np.float32), "float64": np.zeros(n, np.float64),
           "strided": np.zeros(2 * n, np.float32)[::2]}[bad]
    with pytest.raises(ValueError, match=name):
        _unbound_ctx(capi).render_aov(capi.Camera(), capi.default_params(width=16, height=9, spp=1), **{name: arr})


@pytest.mark.parametrize("out", [np.zeros(16 * 9 * 4 - 1, np.uint8), np.zeros(16 * 9 * 4, np.float32), np.zeros(16 * 9 * 3, np.uint8)])
def test_binding_rejects_a_wrongly_sized_frame(capi, out):
    with pytest.raises(ValueError, match="out"):
        _unbound_ctx(capi).render_aov(capi.Camera(), capi.default_params(width=16, height=9, spp=1), out=out)


def test_api_and_header_expose_the_call(capi):
    from rtiow_b200 import api
    assert callable(api.render_aov) and "rtiow_render_aov" in capi.SYMBOLS
