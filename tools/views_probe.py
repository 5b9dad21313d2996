"""What one rtiow_render_views launch saves over one call per view (GPU box).

    python tools/views_probe.py OUT_DIR [--reps N]

Final scene, max_depth 50.  Three ways to render the same K orbit views, alternated in one process and repeated --reps times:
  render   K x rtiow_render                                      (frame to host memory, one synchronise per frame)
  enqueue  K x rtiow_render_rank_enqueue + rtiow_ctx_synchronize on a world-1 rank ctx (frames stay in device memory)
  views    one rtiow_render_views                                (all K frames to host memory)
for cfg1 (400x225 @ 10 spp) at K = 1, 4, 16, 64, and for the headline frame (1200x675 @ 500 spp) at K = 4 (enqueue vs views)
and K = 1 (render vs views).  Per arm: kernel_ms (CUDA events of the render kernels and epilogues), wall_ms (host clock around
the calls, synchronised) and Mpaths/s of both, as median / min / max over the repetitions.  The frames of the arms are compared
byte for byte (the enqueued frames share one device buffer, so only the last of them is compared).  Writes OUT_DIR/views_probe.json
with the card's name, power limit and SM clocks from a read-only nvidia-smi query.
"""
import argparse
import json
import math
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np  # noqa: E402

from rtiow_b200 import capi  # noqa: E402

DEPTH = 50


def orbit(k, aspect):
    """the reference camera (main.rs:108-118) turned about the vertical axis through the look-at point, k steps per turn"""
    cams = []
    for i in range(k):
        a = 2 * math.pi * i / k
        c, s = math.cos(a), math.sin(a)
        cams.append(capi.camera_new((13 * c + 3 * s, 2, 3 * c - 13 * s), (0, 0, 0), (0, 1, 0), 20.0, aspect, 0.1, 10.0))
    return cams


def gpu_identity():
    q = "name,power.limit,clocks.sm,clocks.max.sm,driver_version"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in r.stdout.strip().split(",")))) if r.returncode == 0 else {"error": r.stderr.strip()}


def arm_render(ctx, cams, prm):
    frames, kms = [], 0.0
    t0 = time.perf_counter()
    for cam in cams:
        img, st = ctx.render(cam, prm)
        frames.append(img)
        kms += st["kernel_ms"]
    return (time.perf_counter() - t0) * 1e3, kms, np.stack(frames)


def arm_enqueue(rctx, cams, prm):
    t0 = time.perf_counter()
    for cam in cams:
        ptr = rctx.render_rank_enqueue(cam, prm)
    st = rctx.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    last = capi.device_to_host(ptr, prm.width * prm.height * 4).reshape(prm.height, prm.width, 4)
    return wall, st["kernel_ms"] * len(cams), last[None]          # synchronize reports the mean kernel_ms of the frames


def arm_views(ctx, cams, prm, out):
    t0 = time.perf_counter()
    imgs, st = ctx.render_views(cams, prm, out=out)
    return (time.perf_counter() - t0) * 1e3, st["kernel_ms"], imgs


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def measure(ctx, rctx, cfg, k, arms, reps):
    W, H, spp = cfg
    prm = capi.default_params(width=W, height=H, spp=spp, seed=1, max_depth=DEPTH)
    cams = orbit(k, W / H)
    out = np.empty((k, H, W, 4), np.uint8)
    run = {"render": lambda: arm_render(ctx, cams, prm), "enqueue": lambda: arm_enqueue(rctx, cams, prm),
           "views": lambda: arm_views(ctx, cams, prm, out)}
    frames = {a: run[a]()[2].copy() for a in arms}                  # warm-up pass of every arm; its frames are compared
    wall = {a: [] for a in arms}; kern = {a: [] for a in arms}
    for _ in range(reps):                                           # the arms alternate within each repetition
        for a in arms:
            w, km, _ = run[a]()
            wall[a].append(w); kern[a].append(km)
    paths = k * W * H * spp
    res = {"width": W, "height": H, "spp": spp, "max_depth": DEPTH, "views": k, "paths": paths, "reps": reps, "arms": {}}
    for a in arms:
        res["arms"][a] = {"kernel_ms": summary(kern[a]), "wall_ms": summary(wall[a]),
                          "mpaths_s_kernel": paths / float(np.median(kern[a])) / 1e3, "mpaths_s_wall": paths / float(np.median(wall[a])) / 1e3}
    ref = frames["views"]
    res["identical"] = {a: bool(np.array_equal(frames[a], ref if a != "enqueue" else ref[-1:])) for a in arms if a != "views"}
    print(json.dumps({k_: v for k_, v in res.items() if k_ != "arms"}), flush=True)
    for a in arms:
        r = res["arms"][a]
        print(f"  {a:8s} kernel {r['kernel_ms']['median']:8.3f} ms  wall {r['wall_ms']['median']:8.3f} ms  "
              f"{r['mpaths_s_kernel']:7.0f} Mpaths/s (kernel)  {r['mpaths_s_wall']:7.0f} Mpaths/s (wall)", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("out_dir", type=Path)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    args.out_dir.mkdir(parents=True, exist_ok=True)
    if capi.device_count() == 0:
        raise SystemExit("views_probe: no CUDA device (this probe measures the GPU; there is nothing to measure without one)")
    result = {"gpu_before": gpu_identity(), "scene": "random_scene(1) (final scene)", "runs": []}
    scene = capi.random_scene(1)
    with capi.Context(1) as ctx, capi.Context(device=0, rank=0, world=1) as rctx:
        ctx.upload_scene(**scene)
        rctx.upload_scene(**scene)
        for k in (1, 4, 16, 64):
            result["runs"].append(measure(ctx, rctx, (400, 225, 10), k, ("render", "enqueue", "views"), args.reps))
        result["runs"].append(measure(ctx, rctx, (1200, 675, 500), 4, ("enqueue", "views"), max(3, args.reps // 2)))
        result["runs"].append(measure(ctx, rctx, (1200, 675, 500), 1, ("render", "views"), max(3, args.reps // 2)))
    result["gpu_after"] = gpu_identity()
    (args.out_dir / "views_probe.json").write_text(json.dumps(result, indent=1) + "\n")
    bad = [(r["views"], r["width"], a) for r in result["runs"] for a, same in r["identical"].items() if not same]
    if bad:
        raise SystemExit(f"views_probe: frames differ between arms: {bad}")


if __name__ == "__main__":
    main()
