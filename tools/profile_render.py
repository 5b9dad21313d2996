"""Short single-GPU render used under ncu (profiles/): the bench workload's frame at reduced spp.
    python tools/profile_render.py [spp] [width] [height] [half_extent]
Launch order per frame: render_kernel<…, Loop::Frame> (or render_kernel_umma<6, 64, Loop::Frame>), finalize_kernel.  Two frames: the first warms up."""
import sys
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from rtiow_b200 import capi

spp = int(sys.argv[1]) if len(sys.argv) > 1 else 20
W = int(sys.argv[2]) if len(sys.argv) > 2 else 1200
H = int(sys.argv[3]) if len(sys.argv) > 3 else 675
G = int(sys.argv[4]) if len(sys.argv) > 4 else 11
with capi.Context(1) as ctx:
    ctx.upload_scene(**capi.random_scene(1, G))
    cam = capi.camera_new((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, W / H, 0.1, 10.0)
    prm = capi.default_params(width=W, height=H, spp=spp, seed=1)
    for i in range(2):
        img, st = ctx.render(cam, prm)
        print(f"frame {i}: kernel {st['kernel_ms']:.3f} ms, {st['paths'] / st['kernel_ms'] / 1e3:.1f} Mpaths/s, rays/path {st['rays_traced'] / st['paths']:.4f}, "
              f"{st['sphere_tests'] * 17 / st['kernel_ms'] / 1e9:.2f} TFLOP/s (17 flop/test)")
