"""What the first-hit AOVs of rtiow_render_aov cost over rtiow_render (GPU box).

    python tools/aov_probe.py OUT_DIR [--reps N]

Final scene (random_scene(1)), the reference camera, max_depth 50, the scan AUTO picks (the tensor-core filter).  Two arms,
alternated in one process after a warm-up of each and repeated --reps times:
  render  rtiow_render                                  (RGBA8 frame to host memory)
  aov     rtiow_render_aov with all four float buffers  (the same frame + colour, albedo, normal, depth to host memory)
for the headline frame (1200x675 @ 500 spp) and two previews where a denoiser is used (1200x675 @ 4 spp, 400x225 @ 10 spp).
Per arm: kernel_ms (CUDA events around the render kernel and its epilogues) and wall_ms (host clock around the synchronous
call, including the copies), as median / min / max over the repetitions, and the aov arm's overhead on the medians.  The
frames of the two arms are compared byte for byte.  Host buffers are pageable numpy arrays, as a Python caller's are.  Writes
OUT_DIR/aov_probe.json with the card's name, power limit and SM clocks from a read-only nvidia-smi query.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np  # noqa: E402

from rtiow_b200 import capi  # noqa: E402

DEPTH = 50
CONFIGS = ((1200, 675, 500), (1200, 675, 4), (400, 225, 10))


def gpu_identity():
    q = "name,power.limit,clocks.sm,clocks.max.sm,driver_version"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in r.stdout.strip().split(",")))) if r.returncode == 0 else {"error": r.stderr.strip()}


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def measure(ctx, cfg, reps):
    W, H, spp = cfg
    prm = capi.default_params(width=W, height=H, spp=spp, seed=1, max_depth=DEPTH)
    cam = capi.camera_new((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, W / H, 0.1, 10.0)          # main.rs:108-118
    rgba = np.empty((H, W, 4), np.uint8)
    bufs = dict(color=np.empty((H, W, 3), np.float32), albedo=np.empty((H, W, 3), np.float32),
                normal=np.empty((H, W, 3), np.float32), depth=np.empty((H, W), np.float32))

    def render():
        t0 = time.perf_counter()
        img, st = ctx.render(cam, prm, out=rgba)
        return (time.perf_counter() - t0) * 1e3, st, img

    def aov():
        t0 = time.perf_counter()
        img, _, st = ctx.render_aov(cam, prm, out=rgba, **bufs)
        return (time.perf_counter() - t0) * 1e3, st, img

    run = {"render": render, "aov": aov}
    frames = {a: run[a]()[2].copy() for a in run}                    # warm-up of both arms; their frames are compared
    wall = {a: [] for a in run}; kern = {a: [] for a in run}; backend = None
    for _ in range(reps):
        for a in run:
            w, st, _ = run[a]()
            wall[a].append(w); kern[a].append(st["kernel_ms"]); backend = st["scan_backend"]
    res = {"width": W, "height": H, "spp": spp, "max_depth": DEPTH, "reps": reps, "paths": W * H * spp,
           "scan_backend": {capi.SCAN_TENSOR: "tensor", capi.SCAN_FP32: "fp32"}.get(backend, backend),
           "identical": bool(np.array_equal(frames["render"], frames["aov"])),
           "arms": {a: {"kernel_ms": summary(kern[a]), "wall_ms": summary(wall[a])} for a in run}}
    for m in ("kernel_ms", "wall_ms"):
        res[f"aov_overhead_{m}"] = float(np.median(kern["aov"] if m == "kernel_ms" else wall["aov"]) /
                                         np.median(kern["render"] if m == "kernel_ms" else wall["render"]) - 1.0)
    print(f"{W}x{H} @ {spp} spp ({res['scan_backend']}, {reps} reps, frames identical: {res['identical']})", flush=True)
    for a in run:
        r = res["arms"][a]
        print(f"  {a:7s} kernel {r['kernel_ms']['median']:9.3f} ms [{r['kernel_ms']['min']:.3f}, {r['kernel_ms']['max']:.3f}]"
              f"  wall {r['wall_ms']['median']:9.3f} ms [{r['wall_ms']['min']:.3f}, {r['wall_ms']['max']:.3f}]", flush=True)
    print(f"  aov overhead: kernel {100 * res['aov_overhead_kernel_ms']:+.2f} %, wall {100 * res['aov_overhead_wall_ms']:+.2f} %", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("out_dir", type=Path)
    ap.add_argument("--reps", type=int, default=9)
    args = ap.parse_args()
    args.out_dir.mkdir(parents=True, exist_ok=True)
    if capi.device_count() == 0:
        raise SystemExit("aov_probe: no CUDA device (this probe measures the GPU; there is nothing to measure without one)")
    result = {"gpu_before": gpu_identity(), "scene": "random_scene(1) (final scene)", "runs": []}
    with capi.Context(1) as ctx:
        ctx.upload_scene(**capi.random_scene(1))
        for cfg in CONFIGS:
            result["runs"].append(measure(ctx, cfg, args.reps if cfg[2] < 100 else max(5, args.reps // 2)))
    result["gpu_after"] = gpu_identity()
    (args.out_dir / "aov_probe.json").write_text(json.dumps(result, indent=1) + "\n")
    if not all(r["identical"] for r in result["runs"]):
        raise SystemExit("aov_probe: render_aov's frame differs from rtiow_render's")


if __name__ == "__main__":
    main()
