"""What rtiow_render_denoised costs against the two-call path it replaces and against the raw frame of equal quality (GPU box).

    python tools/render_denoised_probe.py OUT_DIR [--reps N]

The final scene (random_scene(1)), the reference camera (main.rs:108-118), max_depth 50, 16 spp with seed 1 and the library's
default denoise parameters, at 1200x675 and 3840x2160.  Alternated repetitions (--reps, after one warm-up of every arm) of:
  fused      rtiow_render_denoised, RGBA8 only: the AOVs stay on the GPU.
  two_call   rtiow_render_aov with all four float buffers into pageable numpy arrays, then rtiow_denoise over them (RGBA8 only).
  raw        rtiow_render at the equal-quality spp of profiles/denoise_probe.json (the smallest uniform spp whose RMSE reaches the
             denoised 16-spp frame's at 1200x675).
Each arm records kernel_ms (the calls' own, summed over the two calls of two_call), total_ms (the calls' own wall time, summed)
and wall_ms (a host clock around the arm, Python included): median, min and max.  All output arrays are allocated once, outside
the timed region.  The run also checks that fused and two_call give identical bytes, and writes OUT_DIR/render_denoised_probe.json
with the card's name, power limit and SM clocks from a read-only nvidia-smi query.
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402

from rtiow_b200 import capi  # noqa: E402

DEPTH, SPP, SEED = 50, 16, 1
SIZES = ((1200, 675), (3840, 2160))


def gpu_identity():
    q = "name,power.limit,clocks.sm,clocks.max.sm,driver_version"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in r.stdout.strip().split(",")))) if r.returncode == 0 else {"error": r.stderr.strip()}


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def params(w, h, spp):
    return capi.default_params(width=w, height=h, spp=spp, seed=SEED, max_depth=DEPTH)


def arms_of(ctx, w, h, raw_spp, dp):
    cam = capi.camera_new((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, w / h, 0.1, 10.0)
    prm, prm_raw = params(w, h, SPP), params(w, h, raw_spp)
    fused_rgba, two_rgba, raw_rgba, frame = (np.empty((h, w, 4), np.uint8) for _ in range(4))
    bufs = dict(color=np.empty((h, w, 3), np.float32), albedo=np.empty((h, w, 3), np.float32),
                normal=np.empty((h, w, 3), np.float32), depth=np.empty((h, w), np.float32))

    def fused():
        _, st = ctx.render_denoised(cam, prm, dp, out_color=False, out_rgba=fused_rgba)
        return st["kernel_ms"], st["total_ms"]

    def two_call():
        _, b, sa = ctx.render_aov(cam, prm, out=frame, **bufs)
        _, sd = ctx.denoise(b["color"], b["albedo"], b["normal"], b["depth"], dp, out_color=False, out_rgba=two_rgba)
        return sa["kernel_ms"] + sd["kernel_ms"], sa["total_ms"] + sd["total_ms"]

    def raw():
        _, st = ctx.render(cam, prm_raw, out=raw_rgba)
        return st["kernel_ms"], st["total_ms"]

    return {"fused": fused, "two_call": two_call, f"raw_{raw_spp}spp": raw}, fused_rgba, two_rgba


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("out_dir", type=Path)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    args.out_dir.mkdir(parents=True, exist_ok=True)
    if capi.device_count() == 0:
        raise SystemExit("render_denoised_probe: no CUDA device (this probe measures the GPU; there is nothing to measure without one)")
    raw_spp = json.loads((ROOT / "profiles" / "denoise_probe.json").read_text())["tuning"]["sizes"]["1200x675"]["equal_quality_spp"]
    t0 = time.perf_counter()
    dp = capi.default_denoise_params()
    result = {"gpu_before": gpu_identity(), "scene": "random_scene(1) (final scene)", "max_depth": DEPTH, "spp": SPP, "seed": SEED,
              "raw_spp": raw_spp, "reps": args.reps,
              "denoise_params": {"levels": dp.levels, "sigma_color": dp.sigma_color, "sigma_normal": dp.sigma_normal,
                                 "sigma_depth": dp.sigma_depth},
              "sizes": {}}
    with capi.Context(1) as ctx:
        ctx.upload_scene(**capi.random_scene(1))
        for w, h in SIZES:
            arms, fused_rgba, two_rgba = arms_of(ctx, w, h, raw_spp, dp)
            for f in arms.values():
                f()                                            # warm-up of every arm
            identical = bool(np.array_equal(fused_rgba, two_rgba))
            kern = {a: [] for a in arms}; total = {a: [] for a in arms}; wall = {a: [] for a in arms}
            for _ in range(args.reps):
                for a, f in arms.items():
                    t = time.perf_counter()
                    k, tt = f()
                    wall[a].append((time.perf_counter() - t) * 1e3)
                    kern[a].append(k); total[a].append(tt)
            identical = identical and bool(np.array_equal(fused_rgba, two_rgba))
            res = {"fused_equals_two_call": identical,
                   "arms": {a: {"kernel_ms": summary(kern[a]), "total_ms": summary(total[a]), "wall_ms": summary(wall[a])} for a in arms}}
            result["sizes"][f"{w}x{h}"] = res
            print(f"{w}x{h} @ {SPP} spp: fused == two-call bytes: {identical}", flush=True)
            for a in arms:
                r = res["arms"][a]
                print(f"  {a:12s} kernel {r['kernel_ms']['median']:9.3f} ms [{r['kernel_ms']['min']:.3f}, {r['kernel_ms']['max']:.3f}]"
                      f"  total {r['total_ms']['median']:9.3f} ms [{r['total_ms']['min']:.3f}, {r['total_ms']['max']:.3f}]"
                      f"  wall {r['wall_ms']['median']:9.3f} ms", flush=True)
    result["gpu_after"] = gpu_identity()
    result["seconds"] = time.perf_counter() - t0
    (args.out_dir / "render_denoised_probe.json").write_text(json.dumps(result, indent=1, default=float) + "\n")
    if not all(r["fused_equals_two_call"] for r in result["sizes"].values()):
        raise SystemExit("render_denoised_probe: the fused call and the two-call path gave different bytes")


if __name__ == "__main__":
    main()
