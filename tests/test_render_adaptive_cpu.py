"""CPU suite for rtiow_render_adaptive: the ctypes binding checks the buffers it is handed before it calls the library, and every
layer exposes the call.  test_kernel_inventory.py checks the library's adaptive render and round kernels."""
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _unbound_ctx(capi):
    ctx = object.__new__(capi.Context)         # the checks run before the library is called: no ctx handle is needed
    ctx._h = None
    return ctx


@pytest.mark.parametrize("name,dtype", [("spp_map", np.uint32), ("error_map", np.float32)])
@pytest.mark.parametrize("bad", ["short", "long", "wrong-dtype", "strided"])
def test_binding_rejects_wrongly_sized_maps(capi, name, dtype, bad):
    n = 9 * 16
    other = np.float32 if dtype == np.uint32 else np.uint32
    arr = {"short": np.zeros(n - 1, dtype), "long": np.zeros(n + 1, dtype), "wrong-dtype": np.zeros(n, other),
           "strided": np.zeros(2 * n, dtype)[::2]}[bad]
    with pytest.raises(ValueError, match=name.split("_")[0]):
        _unbound_ctx(capi).render_adaptive(capi.Camera(), capi.default_params(width=16, height=9, spp=4), 1, 1.0, **{name: arr})


@pytest.mark.parametrize("out", [np.zeros(16 * 9 * 4 - 1, np.uint8), np.zeros(16 * 9 * 4, np.float32), np.zeros(16 * 9 * 3, np.uint8)])
def test_binding_rejects_a_wrongly_sized_frame(capi, out):
    with pytest.raises(ValueError, match="out"):
        _unbound_ctx(capi).render_adaptive(capi.Camera(), capi.default_params(width=16, height=9, spp=4), 1, 1.0, out=out)


def test_header_binding_and_api_expose_the_call(capi):
    from rtiow_b200 import api
    assert callable(api.render_adaptive) and "rtiow_render_adaptive" in capi.SYMBOLS
    assert hasattr(capi.lib(), "rtiow_render_adaptive")
    hdr = (ROOT / "include" / "rtiow_cuda.h").read_text()
    assert re.search(r"int rtiow_render_adaptive\(rtiow_ctx\* ctx, const rtiow_camera\* cam, const rtiow_params\* p, uint32_t min_spp, "
                     r"double tolerance,\s+uint8_t\* out_rgba, uint32_t\* out_spp, float\* out_error, rtiow_stats\* stats\);", hdr)
