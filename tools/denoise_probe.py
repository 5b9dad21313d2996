"""What rtiow_denoise buys and costs, and where its defaults come from (GPU box).

    python tools/denoise_probe.py OUT_DIR [--reps N]

Tuning scene: the final scene (random_scene(1)), the reference camera (main.rs:108-118), max_depth 50, at 400x225 and 1200x675.
  reference  4096 spp with seed 2: a same-seed reference shares the first n samples of every pixel and would flatter every image.
  grid       rtiow_render_aov at 4, 16 and 64 spp (seed 1), then every combination of LEVELS x SIGMA_COLOR x SIGMA_NORMAL x
             SIGMA_DEPTH through rtiow_denoise; RMSE against the reference in 8-bit levels on the RGB bytes.
  edges      every combination also filters the converged AOVs (the reference is rtiow_render_aov at 4096 spp) at 400x225; its
             change to the converged frame over the change of the blind a-trous blur (every sigma +inf, same levels) says how
             much the edge-stopping terms keep of what is already right.
  defaults   among the combinations whose converged change is at most EDGE_RATIO of the blind blur's, the one with the lowest
             16-spp RMSE summed over both sizes.  (Without the constraint the noisiest-frame objective alone picks a filter that
             blurs converged detail away: both are recorded.)
  raw        rtiow_render at RAW_SPP; the equal-quality spp of a size is the smallest of them whose raw RMSE is at most the
             denoised 16-spp RMSE with the defaults.
  held-out   another scene seed and camera (the GPU test's quality view), with the chosen defaults: raw and denoised 16 spp
             against a 4096-spp reference of seed 3, and on the converged 4096-spp AOVs the change the defaults make to the
             frame against the change of the blind a-trous blur (every sigma +inf).
  cost       alternated repetitions (--reps) of: the denoise call at 1200x675 and at 3840x2160 (kernel_ms, and the wall time
             of the call with its 40 B/px upload), and rtiow_render at 16 spp and at the equal-quality spp (1200x675); medians
             and min-max.
Writes OUT_DIR/denoise_probe.json with the card's name, power limit and SM clocks from a read-only nvidia-smi query.
"""
import argparse
import itertools
import json
import subprocess
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import numpy as np  # noqa: E402

from rtiow_b200 import capi  # noqa: E402

DEPTH, REF_SPP, SPPS = 50, 4096, (4, 16, 64)
SIZES = ((400, 225), (1200, 675))
LEVELS = (1, 2, 3, 4, 5)
SIGMA_COLOR = (0.02, 0.05, 0.1, 0.25, 0.5, 1.0, np.inf)
SIGMA_NORMAL = (0.03, 0.1, 0.3, 1.0, np.inf)
SIGMA_DEPTH = (0.01, 0.03, 0.1, 0.5, np.inf)
EDGE_RATIO = 0.2              # the GPU test asks for 0.25 on a held-out view: the margin keeps the choice off that edge
RAW_SPP = (16, 24, 32, 48, 64, 96, 128, 192, 256, 384, 512, 768, 1024, 1536, 2048, 4096)
HELD_OUT = dict(scene_seed=7, look_from=(-11.0, 2.5, 4.0), look_at=(0.0, 0.5, -1.0), vfov=24.0, width=400, height=225)


def gpu_identity():
    q = "name,power.limit,clocks.sm,clocks.max.sm,driver_version"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in r.stdout.strip().split(",")))) if r.returncode == 0 else {"error": r.stderr.strip()}


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def rmse(img, ref):
    return float(np.sqrt(np.mean((img[..., :3].astype(np.float64) - ref[..., :3].astype(np.float64)) ** 2)))


def camera(w, h, look_from=(13, 2, 3), look_at=(0, 0, 0), vfov=20.0):
    return capi.camera_new(look_from, look_at, (0, 1, 0), vfov, w / h, 0.1, 10.0)


def params(w, h, spp, seed):
    return capi.default_params(width=w, height=h, spp=spp, seed=seed, max_depth=DEPTH)


def aovs(ctx, cam, w, h, spp, seed=1):
    img, bufs, _ = ctx.render_aov(cam, params(w, h, spp, seed))
    return img, bufs


def denoise(ctx, b, dp):
    outs, st = ctx.denoise(b["color"], b["albedo"], b["normal"], b["depth"], dp, out_color=False)
    return outs["rgba"], st


def dparams(levels, sc, sn, sz):
    return capi.default_denoise_params(levels=levels, sigma_color=sc, sigma_normal=sn, sigma_depth=sz)


def tune(ctx):
    grid = list(itertools.product(LEVELS, SIGMA_COLOR, SIGMA_NORMAL, SIGMA_DEPTH))
    per_size, score = {}, np.zeros(len(grid))
    for w, h in SIZES:
        cam = camera(w, h)
        ref, conv, _ = ctx.render_aov(cam, params(w, h, REF_SPP, 2))
        res = {"reference": {"spp": REF_SPP, "seed": 2}, "spp": {}}
        inputs = {}
        for spp in SPPS:
            img, b = aovs(ctx, cam, w, h, spp)
            inputs[spp] = b
            res["spp"][str(spp)] = {"raw_rmse": rmse(img, ref)}
        raw = {}
        for spp in RAW_SPP:
            img, st = ctx.render(cam, params(w, h, spp, 1))
            raw[str(spp)] = {"rmse": rmse(img, ref), "kernel_ms": st["kernel_ms"]}
        res["raw"] = raw
        table = np.zeros((len(grid), len(SPPS)))
        for gi, g in enumerate(grid):
            dp = dparams(*g)
            for si, spp in enumerate(SPPS):
                table[gi, si] = rmse(denoise(ctx, inputs[spp], dp)[0], ref)
        score += table[:, SPPS.index(16)]
        if (w, h) == SIZES[0]:
            blind = {lv: rmse(denoise(ctx, conv, dparams(lv, np.inf, np.inf, np.inf))[0], ref) for lv in LEVELS}
            edge = np.array([rmse(denoise(ctx, conv, dparams(*g))[0], ref) / blind[g[0]] for g in grid])
            res["converged_blind_change"] = {str(lv): v for lv, v in blind.items()}
        for si, spp in enumerate(SPPS):
            best = int(np.argmin(table[:, si]))
            res["spp"][str(spp)]["best_of_grid"] = {"params": list(grid[best]), "rmse": float(table[best, si])}
        res["_table"] = table
        res["_ref"], res["_inputs"] = ref, inputs
        per_size[f"{w}x{h}"] = res
        print(f"{w}x{h}: grid of {len(grid)} done; raw rmse " +
              ", ".join(f"{s} spp {res['spp'][str(s)]['raw_rmse']:.3f}" for s in SPPS), flush=True)
    unconstrained = int(np.argmin(score))
    if not (edge <= EDGE_RATIO).any():
        raise SystemExit(f"denoise_probe: no combination keeps the converged change within {EDGE_RATIO} of the blind blur's")
    chosen = int(np.argmin(np.where(edge <= EDGE_RATIO, score, np.inf)))
    levels, sc, sn, sz = grid[chosen]
    out = {"grid": {"levels": LEVELS, "sigma_color": SIGMA_COLOR, "sigma_normal": SIGMA_NORMAL, "sigma_depth": SIGMA_DEPTH},
           "objective": f"lowest denoised 16-spp RMSE summed over both sizes, among converged changes <= {EDGE_RATIO} of the blind blur's",
           "defaults": {"levels": levels, "sigma_color": sc, "sigma_normal": sn, "sigma_depth": sz},
           "defaults_score": float(score[chosen]), "defaults_converged_ratio": float(edge[chosen]),
           "unconstrained": {"params": list(grid[unconstrained]), "score": float(score[unconstrained]),
                             "converged_ratio": float(edge[unconstrained])},
           "sizes": {}}
    # the ten best combinations that meet the constraint, for the record
    order = [i for i in np.argsort(score) if edge[i] <= EDGE_RATIO][:10]
    out["top10"] = [{"params": list(grid[i]), "score": float(score[i]), "converged_ratio": float(edge[i])} for i in order]
    print(f"unconstrained best {grid[unconstrained]}: score {score[unconstrained]:.3f}, converged ratio {edge[unconstrained]:.3f}; "
          f"chosen {grid[chosen]}: score {score[chosen]:.3f}, converged ratio {edge[chosen]:.3f}", flush=True)
    for key, res in per_size.items():
        table = res.pop("_table"); res.pop("_ref"); res.pop("_inputs")
        for si, spp in enumerate(SPPS):
            res["spp"][str(spp)]["denoised_rmse"] = float(table[chosen, si])
        target = res["spp"]["16"]["denoised_rmse"]
        eq = [int(s) for s, r in res["raw"].items() if r["rmse"] <= target]
        res["equal_quality_spp"] = min(eq) if eq else None
        out["sizes"][key] = res
        print(f"{key}: defaults {grid[chosen]}: " + ", ".join(
            f"{s} spp raw {res['spp'][str(s)]['raw_rmse']:.3f} -> {res['spp'][str(s)]['denoised_rmse']:.3f}" for s in SPPS)
            + f"; equal-quality spp {res['equal_quality_spp']}", flush=True)
    return out


def held_out(ctx, dp):
    ho = HELD_OUT
    w, h = ho["width"], ho["height"]
    ctx.upload_scene(**capi.random_scene(ho["scene_seed"]))
    cam = camera(w, h, ho["look_from"], ho["look_at"], ho["vfov"])
    ref, _ = ctx.render(cam, params(w, h, REF_SPP, 3))
    img16, b16 = aovs(ctx, cam, w, h, 16)
    imgc, bc = aovs(ctx, cam, w, h, REF_SPP, 1)
    blind = capi.default_denoise_params(levels=dp.levels, sigma_color=np.inf, sigma_normal=np.inf, sigma_depth=np.inf)
    res = dict(ho, raw16_rmse=rmse(img16, ref), denoised16_rmse=rmse(denoise(ctx, b16, dp)[0], ref),
               converged_change_default=rmse(denoise(ctx, bc, dp)[0], imgc), converged_change_blind=rmse(denoise(ctx, bc, blind)[0], imgc))
    print(f"held-out: raw 16 spp {res['raw16_rmse']:.3f}, denoised {res['denoised16_rmse']:.3f}; converged change: default "
          f"{res['converged_change_default']:.3f}, blind {res['converged_change_blind']:.3f}", flush=True)
    ctx.upload_scene(**capi.random_scene(1))
    return res


def cost(ctx, dp, eq_spp, reps):
    W, H = 1200, 675
    cam = camera(W, H)
    b_hd = aovs(ctx, cam, W, H, 4)[1]
    b_4k = aovs(ctx, camera(3840, 2160), 3840, 2160, 4)[1]
    rgba = np.empty((H, W, 4), np.uint8)

    def dn(b):
        def run():
            t0 = time.perf_counter()
            _, st = denoise(ctx, b, dp)
            return st["kernel_ms"], (time.perf_counter() - t0) * 1e3
        return run

    def render(spp):
        def run():
            t0 = time.perf_counter()
            _, st = ctx.render(cam, params(W, H, spp, 1), out=rgba)
            return st["kernel_ms"], (time.perf_counter() - t0) * 1e3
        return run

    arms = {"denoise_1200x675": dn(b_hd), "denoise_3840x2160": dn(b_4k), "render_16spp_1200x675": render(16)}
    if eq_spp:
        arms[f"render_{eq_spp}spp_1200x675"] = render(eq_spp)
    for f in arms.values():
        f()                                            # warm-up of every arm
    kern = {a: [] for a in arms}; wall = {a: [] for a in arms}
    for _ in range(reps):
        for a, f in arms.items():
            k, wl = f()
            kern[a].append(k); wall[a].append(wl)
    res = {"reps": reps, "arms": {a: {"kernel_ms": summary(kern[a]), "wall_ms": summary(wall[a])} for a in arms}}
    for a in arms:
        r = res["arms"][a]
        print(f"  {a:26s} kernel {r['kernel_ms']['median']:9.3f} ms [{r['kernel_ms']['min']:.3f}, {r['kernel_ms']['max']:.3f}]"
              f"  wall {r['wall_ms']['median']:9.3f} ms [{r['wall_ms']['min']:.3f}, {r['wall_ms']['max']:.3f}]", flush=True)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("out_dir", type=Path)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    args.out_dir.mkdir(parents=True, exist_ok=True)
    if capi.device_count() == 0:
        raise SystemExit("denoise_probe: no CUDA device (this probe measures the GPU; there is nothing to measure without one)")
    t0 = time.perf_counter()
    result = {"gpu_before": gpu_identity(), "scene": "random_scene(1) (final scene)", "max_depth": DEPTH, "spps": SPPS}
    with capi.Context(1) as ctx:
        ctx.upload_scene(**capi.random_scene(1))
        result["tuning"] = tune(ctx)
        d = result["tuning"]["defaults"]
        dp = dparams(d["levels"], d["sigma_color"], d["sigma_normal"], d["sigma_depth"])
        lib = capi.default_denoise_params()
        result["library_defaults"] = {"levels": lib.levels, "sigma_color": lib.sigma_color, "sigma_normal": lib.sigma_normal,
                                      "sigma_depth": lib.sigma_depth}
        result["library_defaults_match"] = result["library_defaults"] == d
        result["held_out"] = held_out(ctx, dp)
        result["cost"] = cost(ctx, dp, result["tuning"]["sizes"]["1200x675"]["equal_quality_spp"], args.reps)
    result["gpu_after"] = gpu_identity()
    result["seconds"] = time.perf_counter() - t0
    (args.out_dir / "denoise_probe.json").write_text(json.dumps(result, indent=1, default=float) + "\n")
    print(f"defaults {d}; the library's defaults match: {result['library_defaults_match']}", flush=True)


if __name__ == "__main__":
    main()
