"""What rtiow_render_adaptive costs and what it buys on the headline frame (GPU box).

    python tools/adaptive_probe.py OUT_DIR [--reps N]

Final scene (random_scene(1)), the reference camera, 1200x675, max_depth 50, the scan AUTO picks (the tensor-core filter).
  overhead  rtiow_render at 500 spp against rtiow_render_adaptive with min_spp == spp == 500 (every pixel renders the same
            samples, through the adaptive kernel, the select kernels and one host round trip), alternated after a warm-up of
            each and repeated --reps times: kernel_ms and wall_ms as median / min / max, frames compared byte for byte.
  payoff    a reference of the same view at 4096 spp with a DIFFERENT seed (a same-seed reference shares the first n samples
            of every pixel and would flatter every image), then for each tolerance an adaptive render (min_spp 16, spp 500)
            and a uniform rtiow_render at the same total paths (the nearest whole spp), each with its RMSE against the
            reference in 8-bit display space (RGB of the RGBA8 frames) and its kernel time.  The equal-error line is the
            largest tolerance whose RMSE is at most uniform 500 spp's, with its time.
Writes OUT_DIR/adaptive_probe.json with the card's name, power limit and SM clocks from a read-only nvidia-smi query.
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

W, H, DEPTH, SPP, MIN_SPP, REF_SPP = 1200, 675, 50, 500, 16, 4096
TOLERANCES = (8.0, 4.0, 3.0, 2.0, 1.5, 1.0, 0.75, 0.5)


def gpu_identity():
    q = "name,power.limit,clocks.sm,clocks.max.sm,driver_version"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in r.stdout.strip().split(",")))) if r.returncode == 0 else {"error": r.stderr.strip()}


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def rmse(img, ref):
    return float(np.sqrt(np.mean((img[..., :3].astype(np.float64) - ref[..., :3].astype(np.float64)) ** 2)))


def overhead(ctx, cam, reps):
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=1, max_depth=DEPTH)
    rgba = np.empty((H, W, 4), np.uint8)

    def render():
        t0 = time.perf_counter()
        img, st = ctx.render(cam, prm, out=rgba)
        return (time.perf_counter() - t0) * 1e3, st, img

    def adaptive():
        t0 = time.perf_counter()
        img, _, st = ctx.render_adaptive(cam, prm, SPP, 0.0, out=rgba, spp_map=False, error_map=False)
        return (time.perf_counter() - t0) * 1e3, st, img

    run = {"render": render, "adaptive": adaptive}
    frames = {a: run[a]()[2].copy() for a in run}                    # warm-up of both arms; their frames are compared
    wall = {a: [] for a in run}; kern = {a: [] for a in run}; rays = {}
    for _ in range(reps):
        for a in run:
            w, st, _ = run[a]()
            wall[a].append(w); kern[a].append(st["kernel_ms"]); rays[a] = st["rays_traced"]
    res = {"spp": SPP, "reps": reps, "identical": bool(np.array_equal(frames["render"], frames["adaptive"])),
           "same_rays": rays["render"] == rays["adaptive"],
           "arms": {a: {"kernel_ms": summary(kern[a]), "wall_ms": summary(wall[a])} for a in run},
           "overhead_kernel_ms": float(np.median(kern["adaptive"]) / np.median(kern["render"]) - 1.0),
           "overhead_wall_ms": float(np.median(wall["adaptive"]) / np.median(wall["render"]) - 1.0)}
    print(f"overhead at {SPP} spp ({reps} reps, frames identical: {res['identical']}, same rays: {res['same_rays']})", flush=True)
    for a in run:
        r = res["arms"][a]
        print(f"  {a:9s} kernel {r['kernel_ms']['median']:9.3f} ms [{r['kernel_ms']['min']:.3f}, {r['kernel_ms']['max']:.3f}]"
              f"  wall {r['wall_ms']['median']:9.3f} ms [{r['wall_ms']['min']:.3f}, {r['wall_ms']['max']:.3f}]", flush=True)
    print(f"  kernel {100 * res['overhead_kernel_ms']:+.2f} %, wall {100 * res['overhead_wall_ms']:+.2f} %", flush=True)
    return res


def payoff(ctx, cam):
    t0 = time.perf_counter()
    ref, sref = ctx.render(cam, capi.default_params(width=W, height=H, spp=REF_SPP, seed=2, max_depth=DEPTH))
    print(f"reference: {REF_SPP} spp, seed 2, kernel {sref['kernel_ms']:.1f} ms", flush=True)
    uni500, s500 = ctx.render(cam, capi.default_params(width=W, height=H, spp=SPP, seed=1, max_depth=DEPTH))
    out = {"reference": {"spp": REF_SPP, "seed": 2, "kernel_ms": sref["kernel_ms"]},
           "uniform_500": {"rmse": rmse(uni500, ref), "kernel_ms": s500["kernel_ms"], "paths": s500["paths"]}, "tolerances": []}
    print(f"uniform {SPP}: rmse {out['uniform_500']['rmse']:.4f}, kernel {s500['kernel_ms']:.2f} ms", flush=True)
    prm = capi.default_params(width=W, height=H, spp=SPP, seed=1, max_depth=DEPTH)
    for tol in TOLERANCES:
        img, maps, st = ctx.render_adaptive(cam, prm, MIN_SPP, tol)
        mean_spp = st["paths"] / (W * H)
        u_spp = max(1, int(round(mean_spp)))
        uimg, ust = ctx.render(cam, capi.default_params(width=W, height=H, spp=u_spp, seed=1, max_depth=DEPTH))
        counts, n_px = np.unique(maps["spp"], return_counts=True)
        row = {"tolerance": tol, "mean_spp": mean_spp, "paths": st["paths"], "rmse": rmse(img, ref), "kernel_ms": st["kernel_ms"],
               "kernel_launches": st["kernel_launches"], "rays_traced": st["rays_traced"],
               "pixels_per_count": {str(int(c)): int(k) for c, k in zip(counts, n_px)},
               "uniform_same_paths": {"spp": u_spp, "rmse": rmse(uimg, ref), "kernel_ms": ust["kernel_ms"]}}
        out["tolerances"].append(row)
        print(f"tol {tol:5.2f}: mean {mean_spp:6.1f} spp, rmse {row['rmse']:.4f}, kernel {st['kernel_ms']:7.2f} ms | uniform {u_spp} spp: "
              f"rmse {row['uniform_same_paths']['rmse']:.4f}, kernel {ust['kernel_ms']:7.2f} ms", flush=True)
    ok = [r for r in out["tolerances"] if r["rmse"] <= out["uniform_500"]["rmse"]]
    if ok:
        best = max(ok, key=lambda r: r["tolerance"])
        out["equal_error"] = {"tolerance": best["tolerance"], "rmse": best["rmse"], "kernel_ms": best["kernel_ms"], "mean_spp": best["mean_spp"],
                              "uniform_500_rmse": out["uniform_500"]["rmse"], "uniform_500_kernel_ms": out["uniform_500"]["kernel_ms"],
                              "speedup": out["uniform_500"]["kernel_ms"] / best["kernel_ms"]}
        print(f"equal error: tolerance {best['tolerance']} reaches rmse {best['rmse']:.4f} <= {out['uniform_500']['rmse']:.4f} in "
              f"{best['kernel_ms']:.2f} ms against {out['uniform_500']['kernel_ms']:.2f} ms", flush=True)
    else:
        out["equal_error"] = None
        print("equal error: no tolerance reaches uniform 500 spp's rmse", flush=True)
    out["seconds"] = time.perf_counter() - t0
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("out_dir", type=Path)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    args.out_dir.mkdir(parents=True, exist_ok=True)
    if capi.device_count() == 0:
        raise SystemExit("adaptive_probe: no CUDA device (this probe measures the GPU; there is nothing to measure without one)")
    result = {"gpu_before": gpu_identity(), "scene": "random_scene(1) (final scene)", "width": W, "height": H, "max_depth": DEPTH,
              "min_spp": MIN_SPP, "spp": SPP}
    cam = capi.camera_new((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, W / H, 0.1, 10.0)          # main.rs:108-118
    with capi.Context(1) as ctx:
        ctx.upload_scene(**capi.random_scene(1))
        result["overhead"] = overhead(ctx, cam, args.reps)
        result["payoff"] = payoff(ctx, cam)
    result["gpu_after"] = gpu_identity()
    (args.out_dir / "adaptive_probe.json").write_text(json.dumps(result, indent=1) + "\n")
    if not (result["overhead"]["identical"] and result["overhead"]["same_rays"]):
        raise SystemExit("adaptive_probe: min_spp == spp differs from rtiow_render")


if __name__ == "__main__":
    main()
