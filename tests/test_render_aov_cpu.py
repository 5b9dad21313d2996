"""CPU suite for rtiow_render_aov: the ctypes binding checks the buffers it is handed before it calls the library, and every layer
exposes the call.  test_kernel_inventory.py checks the library's AOV render and epilogue kernels."""
import numpy as np
import pytest


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
