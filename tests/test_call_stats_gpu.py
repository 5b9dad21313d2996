"""Every frame-level entry point reports the same frame and the same rtiow_stats for the same work.

One 200x113 @ 3 spp frame of the final scene goes through each entry point that renders a whole frame on one device: the
plain call, one progressive pass, a batch of one view, the three calls of a world-1 rank ctx and the two per-rank calls at
rank 0 of world 1.  The frames must be byte-identical and the counts equal; the bytes a call reports copying depend on where
its frame goes (to the host, left on the device, or into the caller's buffer).
"""
import ctypes as C

import numpy as np
import pytest

from conftest import final_camera

W, H, SPP = 200, 113, 3


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["TENSOR", "FP32"])
def test_every_entry_point_reports_the_same_frame(ctx_final, capi, final_scene, backend):
    torch = pytest.importorskip("torch")
    b = getattr(capi, "SCAN_" + backend)
    cam = final_camera(capi, W / H)
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=4)
    frame_bytes = W * H * 4
    call_h2d = C.sizeof(capi.Camera) + C.sizeof(capi.Params)
    got = {}                                    # entry point -> (frame, stats, expected h2d_bytes, expected d2h_bytes)
    ctx_final.set_scan_backend(b)
    try:
        img, st = ctx_final.render(cam, prm)
        got["render"] = (img.copy(), st, call_h2d, frame_bytes + 16)
        img, st = ctx_final.render_progressive(cam, prm, 1)
        got["render_progressive"] = (img.copy(), st, call_h2d, frame_bytes + 16)
        imgs, st = ctx_final.render_views([cam], prm)
        got["render_views"] = (imgs[0].copy(), st, call_h2d, frame_bytes + 16)
        dev = torch.zeros(ctx_final.tile_buffer_bytes(prm, 1), dtype=torch.uint8, device="cuda")
        st = ctx_final.render_tiles_device(cam, prm, 0, 1, dev.data_ptr(), 0, want_stats=True)
        got["render_tiles_device"] = (dev.cpu().numpy().reshape(H, W, 4), st, 0, 0)
        dev = torch.zeros(frame_bytes, dtype=torch.uint8, device="cuda")
        st = ctx_final.render_to_frame_device(cam, prm, 0, 1, dev.data_ptr(), 0, want_stats=True)
        got["render_to_frame_device"] = (dev.cpu().numpy().reshape(H, W, 4), st, 0, 0)
    finally:
        ctx_final.set_scan_backend(capi.SCAN_AUTO)
    with capi.Context(device=0, rank=0, world=1) as rc:
        rc.upload_scene(**final_scene[0])
        rc.set_scan_backend(b)
        img, st = rc.render_rank(cam, prm)
        got["render_rank"] = (img, st, call_h2d, frame_bytes + 16)
        ptr, st = rc.render_rank_device(cam, prm)
        got["render_rank_device"] = (capi.device_to_host(ptr, frame_bytes).reshape(H, W, 4), st, call_h2d, 16)
        ptr = rc.render_rank_enqueue(cam, prm)
        st = rc.synchronize()
        got["render_rank_enqueue"] = (capi.device_to_host(ptr, frame_bytes).reshape(H, W, 4), st, call_h2d, 16)

    ref, ref_st = got["render"][:2]
    n_spheres = len(final_scene[0]["radius"])
    for name, (img, st, h2d, d2h) in got.items():
        assert np.array_equal(img, ref), f"{name}: the frame differs from rtiow_render's"
        assert st["paths"] == W * H * SPP, name
        assert st["rays_traced"] == ref_st["rays_traced"] and st["scan_backend"] == b, name
        assert st["sphere_tests"] == st["rays_traced"] * n_spheres, name
        assert st["n_gpus"] == 1 and st["kernel_launches"] == 2 and st["kernel_ms"] > 0, name
        assert (st["h2d_bytes"], st["d2h_bytes"]) == (h2d, d2h), name
