"""CPU suite for rtiow_render_denoised: the ctypes binding checks the output buffers it is handed before it calls the library, and
the header, the ctypes symbol list, the built library, api, the Rust crates and the C++ mirror all expose the call."""
import re
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _unbound_ctx(capi):
    ctx = object.__new__(capi.Context)         # the checks run before the library is called: no ctx handle is needed
    ctx._h = None
    return ctx


def _call(capi, **kw):
    return _unbound_ctx(capi).render_denoised(capi.Camera(), capi.default_params(width=16, height=9, spp=1), **kw)


@pytest.mark.parametrize("name,shape,dtype", [("out_color", (9, 16, 3), np.float32), ("out_rgba", (9, 16, 4), np.uint8)])
@pytest.mark.parametrize("bad", ["short", "long", "dtype", "strided"])
def test_binding_rejects_wrongly_sized_outputs(capi, name, shape, dtype, bad):
    n = int(np.prod(shape))
    other = np.uint8 if dtype == np.float32 else np.float32
    arr = {"short": np.zeros(n - 1, dtype), "long": np.zeros(n + 1, dtype), "dtype": np.zeros(n, other),
           "strided": np.zeros(2 * n, dtype)[::2]}[bad]
    with pytest.raises(ValueError, match=name):
        _call(capi, **{name: arr})


def test_binding_rejects_no_output(capi):
    with pytest.raises(ValueError, match="both"):
        _call(capi, out_color=None, out_rgba=False)


def test_every_layer_exposes_the_call(capi):
    from rtiow_b200 import api
    assert callable(api.render_denoised) and callable(capi.Context.render_denoised)
    assert "rtiow_render_denoised" in capi.SYMBOLS and hasattr(capi.lib(), "rtiow_render_denoised")
    hdr = (ROOT / "include" / "rtiow_cuda.h").read_text()
    assert re.search(r"int\s+rtiow_render_denoised\(rtiow_ctx\* ctx, const rtiow_camera\* cam, const rtiow_params\* p, "
                     r"const rtiow_denoise_params\* dp,\s+float\* out_color, uint8_t\* out_rgba, rtiow_stats\* stats\);", hdr)
    sys_rs = (ROOT / "rust" / "rtiow-cuda-sys" / "src" / "lib.rs").read_text()
    assert re.search(r"pub fn rtiow_render_denoised\(ctx: \*mut rtiow_ctx, cam: \*const rtiow_camera, p: \*const rtiow_params, "
                     r"dp: \*const rtiow_denoise_params,\s+out_color: \*mut f32, out_rgba: \*mut u8, stats: \*mut rtiow_stats\) -> c_int;", sys_rs)
    rs = (ROOT / "rust" / "rtiow-gpu" / "gpu.rs").read_text()
    assert re.search(r"pub fn render_denoised\(cam: &Camera, world: &HittableList, p: &RenderParams, dp: &sys::rtiow_denoise_params\)", rs)
    hpp = (ROOT / "rtiow_b200" / "host" / "rtiow.hpp").read_text()
    assert re.search(r"inline std::vector<uint8_t> render_denoised\(const Camera& cam, const HittableList& world, const RenderParams& p, "
                     r"const rtiow_denoise_params& dp,\s+std::vector<float>\* color = nullptr, rtiow_stats\* stats = nullptr\)", hpp)
    ex = (ROOT / "rtiow_b200" / "host" / "example_main.cpp").read_text()
    assert "--render-denoised" in ex and "render_denoised(" in ex


def test_ctypes_argument_types(capi):
    f = capi.lib().rtiow_render_denoised
    assert f.argtypes[1]._type_ is capi.Camera and f.argtypes[2]._type_ is capi.Params and f.argtypes[3]._type_ is capi.DenoiseParams
    assert f.argtypes[6]._type_ is capi.Stats and len(f.argtypes) == 7
