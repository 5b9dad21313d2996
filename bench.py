#!/usr/bin/env python
"""bench.py — Mpaths/s of the rtiow render hot path on B200 (BASELINE.json metric), one JSON line.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg1|cfg2|cfg3-*|cfg4|cfg5]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

A *step* is one full frame of the workload: BASELINE.json configs[1], the RTIOW Part 1 final scene
(seeded random_scene, main.rs:59-102) at 1200x675, 500 spp, depth 50 — 405 M paths.  At N > 1 the same frame is
split into interleaved row tiles, one rank per GPU ("strong" scaling), and gathered INSIDE librtiow_cuda.so
(rtiow_ctx_create_rank + rtiow_render_rank: fused peer stores into rank 0's frame, or --gather nccl: ncclAllGather);
torch.distributed only launches, hands out the library's NCCL id, and reduces the timings.

  value     device-resident: scene already in HBM, this rank's rows + gather, frame left in HBM (rtiow_render_rank_device)
  e2e       the reference-facing call with HOST buffers: scene upload (H2D) + rtiow_render_rank + frame to host (D2H)
  roofline  the dominant kernel against the tensor pipe (executed fp16 FLOP, MEASURED_PEAKS.json) when the filter runs on
            tcgen05, else the FP32 pipe; roofline_fp32 always carries SURVEY §8(d)'s algorithmic figure
            (17 FLOP x rays x spheres) against an FFMA2 calibration kernel run in this process
  cpu_baseline  the f64 CPU oracle (a port: the Rust reference cannot be built here) on a bounded sample
  --impl reference  times that same CPU restatement, all host threads, as the reference arm (loads nothing of the product)
  --inproc  one process, N GPUs: rtiow_ctx_create(N) + rtiow_render
  --dump-outputs DIR  after the timed steps, the frame of the last one as DIR/frame.npy (float32, see dump_frame)

bench.py writes nothing into the repository: the tree may be read-only.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import signal
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True                                # no __pycache__ next to the modules imported from the tree
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # NCCL's version banner must not land on stdout: ONE JSON line there

WORKLOAD = dict(name="RTIOW Part 1 final scene (seeded random_scene), 1200x675, 500 spp, depth 50", width=1200, height=675, spp=500,
                max_depth=50, t_min=1e-4, scene_seed=1, sample_seed=1)
# BASELINE.json configs by name; the default (and the line the driver records) is cfg2 = configs[1].  The others are parity-test
# cases (tests/test_full_size_gpu.py) that can also be timed: (workload name, width, height, spp, grid half-extent, material mode)
CONFIGS = {
    "cfg1": ("RTIOW Part 1 final scene (seeded random_scene), 400x225, 10 spp, depth 50", 400, 225, 10, 11, 0),
    "cfg2": (WORKLOAD["name"], 1200, 675, 500, 11, 0),
    "cfg3-lambertian": ("material isolation: all-Lambertian, 800x450, 100 spp, depth 50", 800, 450, 100, 11, 1),
    "cfg3-metal": ("material isolation: all-Metal (fuzz), 800x450, 100 spp, depth 50", 800, 450, 100, 11, 2),
    "cfg3-dielectric": ("material isolation: all-Dialectric + hollow glass shell, 800x450, 100 spp, depth 50", 800, 450, 100, 11, 3),
    "cfg4": ("random-spheres scene scaled to 10k spheres (grid -50..=50), 1920x1080, 256 spp, depth 50", 1920, 1080, 256, 50, 0),
    "cfg5": ("RTIOW Part 1 final scene (seeded random_scene), 3840x2160, 1024 spp, depth 50", 3840, 2160, 1024, 11, 0),
}
FLOP_PER_TEST = 17.0            # SURVEY §8(d): sphere.rs:18-25 with a and r^2 hoisted
FP32_NOMINAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12
TENSOR_FLOP_PER_TEST = 2 * 16 * 2.0          # two tcgen05.mma of K = 16 per (ray, padded sphere), 2 FLOP per multiply-add
# dram__bytes_read.sum + dram__bytes_write.sum of ONE render_kernel launch of this workload on one GPU, from the ncu --set full
# capture summarised in profiles/r1_p_render_kernel_ncu_bench_size.txt (19.56 MB read + 0.72 MB written): the scene, the
# per-sphere records and the fixed-point accumulators; the 9.7 TFLOP of the launch run out of shared memory and registers.
NCU_DRAM_BYTES_PER_LAUNCH = 20_274_176


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS), help="BASELINE.json configuration (default: configs[1], the headline)")
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--spp", type=int, default=None)
    ap.add_argument("--tile-rows", type=int, default=1)
    ap.add_argument("--cpu-sample-spp", type=int, default=0, help="spp of the bounded CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--gather", default="auto", choices=["auto", "fused", "nccl"],
                    help="N > 1, inside librtiow_cuda.so: 'nccl' = tile buffers + ncclAllGather + de-interleave; 'fused' = every rank's epilogue stores its "
                         "pixels into rank 0's frame over NVLink (CUDA IPC mapping) + a 1-int NCCL all-reduce as barrier; 'auto' = fused when the mapping works")
    ap.add_argument("--scan", default="auto", choices=["auto", "fp32", "tensor"], help="sphere filter backend (rtiow_ctx_set_scan_backend)")
    ap.add_argument("--inproc", action="store_true", help="one process driving --gpus N devices through rtiow_ctx_create(N) + rtiow_render (no torchrun)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame the timed path returned in its last step to DIR/frame.npy (float32; a seeded pixel sample above 64 MB)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    name, w, h, spp, grid, mode = CONFIGS[a.config]
    a.workload = name if (a.width, a.height, a.spp) == (None, None, None) else f"{name} [overridden size]"
    a.width, a.height, a.spp = a.width or w, a.height or h, a.spp or spp
    a.grid, a.material_mode = grid, mode
    return a


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    @staticmethod
    def _die_with_parent():
        ctypes.CDLL(None).prctl(1, signal.SIGTERM)              # PR_SET_PDEATHSIG: the sampler never outlives bench.py, even when it fails

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, preexec_fn=self._die_with_parent)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.proc.wait(timeout=10)
        self.t.join(timeout=2)
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0.5 * max(sm)] if sm else []
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------- shared
def make_config(args, n_spheres):
    """the workload, identical for both arms (the driver compares it): everything else goes to `impl_detail`"""
    return {"workload": args.workload, "width": args.width, "height": args.height, "spp": args.spp, "max_depth": WORKLOAD["max_depth"],
            "n_spheres": n_spheres, "scene_seed": WORKLOAD["scene_seed"], "sample_seed": WORKLOAD["sample_seed"],
            "cache": "GPU arm: L2 flushed (160 MiB device fill) between timed steps"}


DUMP_LIMIT_BYTES = 64_000_000


def dump_frame(out_dir, frame):
    """--dump-outputs: the RGBA8 frame (top-down, [H, W, 4]) a caller of the timed path receives, as out_dir/frame.npy in float32,
    so that two builds can be compared output for output (the inputs are fixed by the seeds of WORKLOAD).  A frame whose float32
    copy exceeds DUMP_LIMIT_BYTES (cfg5) is written as a fixed, seeded sample of its pixels: frame.npy [k, 4] and, in
    frame_pixels.npy (float64), the linear index y * W + x of each sampled pixel."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    H, W, C = frame.shape
    if frame.size * 4 <= DUMP_LIMIT_BYTES:
        np.save(out / "frame.npy", frame.astype(np.float32))
        return
    k = (DUMP_LIMIT_BYTES - 4096) // (C * 4 + 8)                          # 4 KiB: the two .npy headers
    idx = np.sort(np.random.default_rng(0).choice(H * W, size=k, replace=False))
    np.save(out / "frame.npy", frame.reshape(H * W, C)[idx].astype(np.float32))
    np.save(out / "frame_pixels.npy", idx.astype(np.float64))


# ----------------------------------------------------------------------------------------------- CPU arms
def oracle_module(native=True):
    """the checker / CPU baseline: bench.py is one of the places allowed to load oracle/.  For the TIMED legs the oracle is
    rebuilt with -march=native on this box (the committed recipe targets baseline x86-64 because the .so travels)."""
    from oracle import oracle as o
    march = "native" if (native and o.use_native_build()) else "x86-64"
    return o, march


def time_oracle(o, sc, W, H, spp, seed):
    cam = o.camera_new((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, W / H, 0.1, 10.0)
    t0 = time.perf_counter()
    # n_threads explicit: torchrun exports OMP_NUM_THREADS=1, the reference arm must use every host core
    img, _, cnt = o.render(sc, cam, W, H, spp, seed=seed, sampler=o.SAMPLER_REJECTION, n_threads=o.host_threads())
    dt = time.perf_counter() - t0
    return W * H * spp / dt / 1e6, dt, cnt, img


def run_reference(args, rank):
    """Reference arm: the reference's own CPU implementation of the path, all host threads.
    rustc/cargo are absent, so this is the oracle port (oracle/rtiow_oracle.c, OpenMP rows like rayon-per-row).  Nothing of the
    product is loaded: the world comes from the host-only scene library under oracle/build/."""
    if rank != 0:
        return
    o, march = oracle_module()
    W, H = args.width, args.height
    sc = o.Scene(**o.random_scene(WORKLOAD["scene_seed"], args.grid, args.material_mode))
    spp = args.cpu_sample_spp or (4 if sc.n < 2000 else 1)
    cores = o.host_threads()
    for _ in range(args.warmup):
        time_oracle(o, sc, W, H, 1, 1)
    t0 = time.perf_counter()
    for k in range(args.steps):
        img = time_oracle(o, sc, W, H, spp, 1 + k)[3]
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_frame(args.dump_outputs, img)
    v = W * H * spp * args.steps / dt / 1e6
    sample = (f"each step renders {W}x{H} @ {spp} spp ({W * H * spp / 1e6:.2f} M paths) of the {args.spp} spp workload; Mpaths/s does not depend on spp; "
              f"f64 C restatement (gcc -O2 -march={march}, OpenMP rows), NOT `cargo run --release`: no rustc in this image")
    emit_json({
        "impl": "reference", "metric": "Mpaths/s", "value": v, "unit": "Mpaths/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": make_config(args, sc.n),
        "cpu_baseline": {"value": v, "unit": "Mpaths/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0})


# ----------------------------------------------------------------------------------------------- GPU arm
def roofline_objects(world, kms, rays_total, n_spheres, npad, backend_tensor, peak_fp32, peak_fp32_scalar, args, paths, kernel_name):
    """Two rooflines for the dominant kernel (per GPU).  The filter's work is `rays x spheres` discriminants:
      fp32  : the ALGORITHMIC figure of SURVEY §8(d), 17 FLOP per test, against the FP32 pipe (FFMA2 calibration kernel of this run).
              With the filter on the tensor cores this exceeds 1: the FP32 pipe no longer does that work.
      tensor: the FLOP the tensor cores EXECUTE: per test 2 MMAs (the 32 non-zero terms of hi.hi + hi.lo + lo.hi share two K = 16
              instructions, rt_umma.cuh ray_rows) x K = 16 x 2 = 64, padding spheres included, against the measured dense bf16/fp16
              peak of MEASURED_PEAKS.json (sustained: the kernel is the whole step).  Round 2 started at 3 MMAs (96): the fraction
              went DOWN while the kernel got faster — it is a utilisation figure of a pipe that does not bound the kernel.
    """
    tests_alg = rays_total * n_spheres / world
    fp32 = {"bound": "fp32", "achieved": tests_alg * FLOP_PER_TEST / (kms * 1e-3) / 1e12, "peak": peak_fp32, "unit": "TFLOP/s",
            "flop_per_test": FLOP_PER_TEST, "sphere_tests_per_launch": tests_alg, "peak_scalar_ffma": peak_fp32_scalar, "peak_nominal": FP32_NOMINAL_TFLOPS,
            "peak_source": "FFMA2 calibration kernel in this run (rtiow_fp32_peak_probe); MEASURED_PEAKS.json has no FP32 entry",
            "note": "algorithmic FLOP (SURVEY §8d) over the FP32-pipe peak" + ("; > 1 is expected: the filter runs on the tensor cores" if backend_tensor else "")}
    fp32["frac"] = fp32["achieved"] / peak_fp32
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except (OSError, ValueError):
        pass
    t_peak, t_src = peaks.get("bf16_tflops_sustained"), "MEASURED_PEAKS.json bf16_tflops_sustained (cuBLAS bf16 8192^3, back to back; fp16 runs at the same rate)"
    if not t_peak:
        t_peak, t_src = 1400.0, "fallback of B200_PROFILING.md (sustained ~1.4 PFLOP/s); MEASURED_PEAKS.json absent"
    traffic, t_note = None, "no ncu under bench.py; see profiles/ for the capture of this kernel"
    side = ROOT / "profiles" / "r2_dram_bytes.json"
    if side.exists():
        try:
            rec = json.loads(side.read_text()).get(f"{args.config}:{kernel_name}")
            if rec and world == 1 and (args.width, args.height, args.spp) == tuple(rec["frame"]):
                traffic, t_note = rec["dram_bytes"], rec["source"]
        except (ValueError, KeyError):
            pass
    if backend_tensor:
        flop_exec = rays_total * npad * TENSOR_FLOP_PER_TEST / world
        main = {"bound": "tensor", "achieved": flop_exec / (kms * 1e-3) / 1e12, "peak": t_peak, "unit": "TFLOP/s", "peak_source": t_src,
                "peak_burst": peaks.get("bf16_tflops"), "flop_per_test_executed": TENSOR_FLOP_PER_TEST, "spheres_padded": npad,
                "bound_note": "the sphere filter is a [rays x 11] x [11 x spheres] contraction on tcgen05 (fp16 hi/lo split, 2 MMAs of K = 16 per chunk of 64 "
                              "spheres, fp16 accumulator in TMEM: only its sign is read back, four sign bits per ALU instruction); no pipe bounds the kernel "
                              "(issue slots 70 % busy, ALU pipe 55 %, tensor pipe ~30 %): it is bound by the latency of the per-group chain ray rows -> MMA -> "
                              "TMEM load -> signs and of the per-ray code, see DESIGN.md §1.2 and profiles/"}
        main["frac"] = main["achieved"] / t_peak
    else:
        main = dict(fp32)
    main.update({"traffic": traffic, "traffic_unit": "bytes/launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)", "traffic_note": t_note,
                 "kernel": kernel_name, "kernel_ms": kms, "rays_per_path": rays_total / paths})
    return main, fp32


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from rtiow_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the render path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    nccl_id = None
    if world > 1:
        # torch.distributed is the launcher's plumbing only: rendezvous, the NCCL unique id of the LIBRARY's communicator, the
        # barrier around the timed region and the max over ranks.  Tiles never pass through torch: the gather is inside
        # librtiow_cuda.so (rtiow_render_rank*).
        dist.init_process_group("nccl", device_id=dev)
        box = [capi.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        nccl_id = box[0]
    W, H, spp = args.width, args.height, args.spp
    scene = capi.random_scene(WORKLOAD["scene_seed"], args.grid, args.material_mode)
    n_spheres = len(scene["radius"])
    ctx = capi.Context(device=local_rank, rank=rank, world=world, nccl_id=nccl_id)
    ctx.set_gather({"auto": capi.GATHER_AUTO, "fused": capi.GATHER_FUSED, "nccl": capi.GATHER_NCCL}[args.gather])
    ctx.set_scan_backend({"auto": capi.SCAN_AUTO, "fp32": capi.SCAN_FP32, "tensor": capi.SCAN_TENSOR}[args.scan])
    ctx.upload_scene(**scene)
    cam = capi.camera_new((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, W / H, 0.1, 10.0)
    prm = capi.default_params(width=W, height=H, spp=spp, max_depth=WORKLOAD["max_depth"], t_min=WORKLOAD["t_min"], seed=WORKLOAD["sample_seed"],
                              tile_rows=args.tile_rows)
    flush = torch.empty(160 * 1024 * 1024, dtype=torch.uint8, device=dev)        # > 126 MB L2
    # One stream for everything: the library works on it (rtiow_ctx_set_stream), so torch's L2-flush fills and the timing events
    # are ordered with the library's kernels and NCCL calls.
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    host_np = torch.empty((H, W, 4), dtype=torch.uint8, pin_memory=True).numpy()       # page-locked: the library DMAs the frame straight into it

    def step_device():
        """this rank's rows + the gather, frame left in HBM (rank 0)"""
        _, st = ctx.render_rank_device(cam, prm)
        return st

    def step_e2e():
        """what a caller of the C ABI does per frame, from host buffers to host buffers"""
        ctx.upload_scene(**scene)                                                  # H2D: the scene SoA
        _, st = ctx.render_rank(cam, prm, out=host_np if rank == 0 else None)      # rank 0: D2H of the frame inside the call
        return st

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def reduce(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def maxr(x):
        return reduce(x, dist.ReduceOp.MAX if world > 1 else None)

    def sumr(x):
        return reduce(x, dist.ReduceOp.SUM if world > 1 else None)

    # FP32-pipe calibration, same process, same clocks regime (a kernel of about the step's length)
    peak_tflops, _ = ctx.fp32_peak_probe(packed=True, target_ms=300.0)
    peak_scalar_tflops, _ = ctx.fp32_peak_probe(packed=False, target_ms=100.0)

    for _ in range(args.warmup):
        flush.fill_(1)
        step_device()
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms, rays = [], []
    barrier()
    e0.record(stream)
    # the K frames go onto the stream back to back (rtiow_render_rank_enqueue: kernel, epilogue / gather, frame-complete barrier; no
    # host round trip per frame — at 8 GPUs a frame is 10 ms and a stream synchronisation plus four launch latencies are 1 % of it);
    # the library times every frame's kernel with its own event pair and rtiow_ctx_synchronize returns the mean
    for k in range(args.steps):
        flush.fill_(1)                                                             # evict L2 between timed iterations
        frame_ptr = ctx.render_rank_enqueue(cam, prm)
        if (k + 1) % 512 == 0 and k + 1 < args.steps:                              # the library keeps one event pair per enqueued frame (<= 1024)
            st = ctx.synchronize()
            kernel_ms += [st["kernel_ms"]] * 512; rays.append(st["rays_traced"])
    e1.record(stream)
    st = ctx.synchronize()
    tail = args.steps % 512 or min(args.steps, 512)                                # frames since the last synchronize
    kernel_ms += [st["kernel_ms"]] * tail; rays.append(st["rays_traced"])
    barrier()
    per_step_launches = st["kernel_launches"] // tail                              # render + finalize (+ de-interleave): OUR kernels, not NCCL's
    backend_tensor = st["scan_backend"] == capi.SCAN_TENSOR
    gather_note = ctx.gather_info()
    # the last timed frame, as the caller of rtiow_render_rank_enqueue has it: rank 0 holds the whole frame in HBM
    frame = capi.device_to_host(frame_ptr, W * H * 4).reshape(H, W, 4) if args.dump_outputs and rank == 0 else None
    total_ms = maxr(e0.elapsed_time(e1))
    clk = clocks.stop() if rank == 0 else None
    ms_per_step = total_ms / args.steps
    paths = W * H * spp
    value = paths / (ms_per_step * 1e-3) / 1e6
    kms = maxr(float(np.mean(kernel_ms)))
    rays_total = sumr(float(np.mean(rays)))                                        # whole frame, all ranks

    # end-to-end through the host-facing call
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize(dev)
    e2e_ms = maxr((time.perf_counter() - t0) * 1e3) / args.steps
    barrier()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        o, march = oracle_module()
        sc = o.Scene(**scene)
        cores = o.host_threads()
        s_spp = args.cpu_sample_spp or max(1, min(spp, int(2 * cores * (1200 * 675) / (W * H) * 530 / n_spheres)))   # ~10-30 s of CPU work
        v, dt, _, _ = time_oracle(o, sc, W, H, s_spp, 1)
        cpu = {"value": v, "unit": "Mpaths/s", "cores": cores, "kind": "port",
               "sample": f"{W}x{H} @ {s_spp} spp ({W * H * s_spp / 1e6:.1f} M paths, {dt:.1f} s) of the {spp} spp workload; f64 C restatement (gcc -O2 -march={march}), OpenMP rows"}

    if rank == 0:
        # the spheres the filter sees: |r| <= 8 and |c| + |r| <= 4096 (capi.cu: the others go to the f64 list), padded to whole MMA chunks
        reach = np.linalg.norm(scene["center"], axis=1) + np.abs(scene["radius"])
        n_small = int(((np.abs(scene["radius"]) <= 8.0) & (reach <= 4096.0)).sum())
        npad = -(-max(n_small, 1) // 64) * 64 if backend_tensor else n_spheres
        kname = "rt::render_kernel_umma<6,64>" if backend_tensor else ("rt::render_kernel<float,true,256,3>" if n_spheres < 3000 else "rt::render_kernel<float,true,768,1>")
        roof, roof32 = roofline_objects(world, kms, rays_total, n_spheres, npad, backend_tensor, peak_tflops, peak_scalar_tflops, args, paths, kname)
        scene_bytes = sum(int(np.asarray(v).nbytes) for v in scene.values())
        out = {
            "metric": "Mpaths/s", "value": value, "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(args, n_spheres),
            "impl_detail": {"tile_rows": args.tile_rows, "scan_backend": "tensor (tcgen05)" if backend_tensor else "fp32 (FFMA2)",
                            "parallelism": f"interleaved row tiles x{world}; {gather_note}",
                            "l2": "160 MiB device buffer (> the 126 MB L2) rewritten between timed steps, inside the timed region (~0.03 ms)",
                            "steps": "rtiow_render_rank_enqueue x K on one stream, then rtiow_ctx_synchronize: no host synchronisation between frames"},
            "clocks": clk,
            "e2e": {"value": paths / (e2e_ms * 1e-3) / 1e6, "unit": "Mpaths/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": scene_bytes + 176 + 48, "d2h_bytes_per_step": W * H * 4 + 16,
                    "call": "rtiow_scene_upload + rtiow_render_rank (host buffers; gather inside the library)"},
            "gpu_launches": per_step_launches * args.steps,
            "roofline": roof, "roofline_fp32": roof32,
        }
        if cpu:
            out["cpu_baseline"] = cpu
        if frame is not None:
            dump_frame(args.dump_outputs, frame)
        emit_json(out)
    if world > 1:
        dist.destroy_process_group()
    ctx.close()


def run_inproc(args):
    """One process driving N GPUs through rtiow_ctx_create(N) + rtiow_render — what `render(n_gpus)` of the Rust / C++ host calls
    (INTEGRATION.md).  No torch, no torch.distributed.  Host buffers in and out; wall clock around K calls."""
    from rtiow_b200 import capi
    W, H, spp, n = args.width, args.height, args.spp, args.gpus
    scene = capi.random_scene(WORKLOAD["scene_seed"], args.grid, args.material_mode)
    ctx = capi.Context(n)
    ctx.set_gather({"auto": capi.GATHER_AUTO, "fused": capi.GATHER_FUSED, "nccl": capi.GATHER_NCCL}[args.gather])
    ctx.set_scan_backend({"auto": capi.SCAN_AUTO, "fp32": capi.SCAN_FP32, "tensor": capi.SCAN_TENSOR}[args.scan])
    ctx.upload_scene(**scene)
    cam = capi.camera_new((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, W / H, 0.1, 10.0)
    prm = capi.default_params(width=W, height=H, spp=spp, max_depth=WORKLOAD["max_depth"], t_min=WORKLOAD["t_min"], seed=WORKLOAD["sample_seed"], tile_rows=args.tile_rows)
    out = np.empty((H, W, 4), np.uint8)
    for _ in range(args.warmup):
        _, st = ctx.render(cam, prm, out=out)
    clocks = ClockSampler(0); clocks.start()
    kms = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ctx.flush_l2()
        _, st = ctx.render(cam, prm, out=out)
        kms.append(st["kernel_ms"])
    dt = (time.perf_counter() - t0) / args.steps
    clk = clocks.stop()
    if args.dump_outputs:
        dump_frame(args.dump_outputs, out)
    paths = W * H * spp
    emit_json({"impl": "ours-inproc", "metric": "Mpaths/s", "value": paths / dt / 1e6, "unit": "Mpaths/s", "n_gpus": n, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": make_config(args, len(scene["radius"])),
               "impl_detail": {"tile_rows": args.tile_rows, "parallelism": ctx.gather_info(), "timing": "host wall clock around rtiow_flush_l2 + rtiow_render (host frame out), K calls",
                               "kernel_ms_slowest_device": float(np.mean(kms)), "rays_per_path": st["rays_traced"] / paths},
               "clocks": clk, "gpu_launches": st["kernel_launches"] * args.steps,
               "e2e": {"value": paths / dt / 1e6, "unit": "Mpaths/s", "h2d_bytes_per_step": 176 + 48, "d2h_bytes_per_step": W * H * 4 + 16}})
    ctx.close()


_REAL_STDOUT = None


def claim_stdout():
    """ONE JSON line on stdout, whatever libraries print: fd 1 is pointed at stderr for the run (NCCL's version banner, torch
    warnings and the like land there) and the result line goes to the original stdout through emit_json()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_json(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, line)
    else:
        os.write(_REAL_STDOUT, line)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0")); local_rank = int(os.environ.get("LOCAL_RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.inproc:
        claim_stdout()
        return run_inproc(args)
    if args.gpus > 1 and world == 1 and args.impl == "ours":
        # convenience: relaunch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", "29517", __file__] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    claim_stdout()
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
