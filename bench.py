#!/usr/bin/env python
"""bench.py — headline benchmark of the render path (BASELINE.json: Mrays/s and 4K frame time at 1/2/4/8
B200, FP32-pipe roofline %).

A "step" = one full frame of the workload (default C3: 3840x2160, 16 spp, depth 5, 1024 spheres + plane,
the configuration the metric's "4K frame time at 1/2/4/8 B200" is quoted on), tile-partitioned over the N
GPUs of one box, frame assembled on rank 0.  A ray = one nearest-hit query (ray_color call with depth > 0).

  python bench.py --gpus 1 --steps K --warmup W          # this repo's CUDA path
  python bench.py ... --dump-outputs DIR                  # + what the last timed step computed, as DIR/<name>.npy
  python bench.py --impl reference ...                    # the reference algorithm on the host cores (oracle port)
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One JSON line on stdout (rank 0).
  value     whole-job Mrays/s, scene resident in HBM, frame left in HBM (on rank 0)
  e2e       the same through the C ABI with HOST buffers: rt_scene_create (ingest + upload) + render + the frame in
            host memory, every step
  parity    the timed frame against the oracle bands the cpu_baseline leg renders (N = 1), and frame_sha256 of the
            assembled frame at every N (the same hash at N = 1, 2, 4, 8 = the same bytes)
  roofline  FP32 pipe: algorithmic FLOPs (SURVEY Appendix C x the kernel's own counters) / CUDA-event kernel time
            against a live FFMA-chain peak; ncu figures are read from the summary file the line names
  extra     (default run, N = 1) the other BASELINE configs: C2, C4 and the C5 sweep's ends
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "ray-tracer-s8_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "Mrays/s"
UNIT = "Mrays/s"
FLUSH_BYTES = 160 << 20   # > 126 MB L2
# --dump-outputs: at most this many pixels of the frame (2 Mi: 24 MiB of float32 channels + 16 MiB of float64 indices)
DUMP_PIXELS = 1 << 21

# --------------------------------------------------------------------------------------------------------
# FLOP model (SURVEY.md Appendix C; add/sub/mul/div/sqrt = 1, FMA = 2, compares/min/max/int = 0), applied to
# the kernel's own counters.  Ray::new is counted inside "primary" (91) and "shade" (79/91), not per ray.
# --------------------------------------------------------------------------------------------------------
FLOPS = dict(primary=91, slab=12, sphere_test=24, sphere_hit=23, tri_base=20, tri_s1=10, tri_s2=16, tri_s3=6,
             tri_hit=15, shade_sphere=79, shade_tri=91, emissive=3, sky=22, pixel=9)


def algorithmic_flops(st: dict, pixels: int) -> float:
    return (st["primary"] * FLOPS["primary"] + st["slab_tests"] * FLOPS["slab"]
            + st["sphere_tests"] * FLOPS["sphere_test"] + st["sphere_hits"] * FLOPS["sphere_hit"]
            + st["tri_tests"] * FLOPS["tri_base"] + st["tri_stage"][0] * FLOPS["tri_s1"]
            + st["tri_stage"][1] * FLOPS["tri_s2"] + st["tri_stage"][2] * FLOPS["tri_s3"]
            + st["tri_hits"] * FLOPS["tri_hit"] + st["shades_sphere"] * FLOPS["shade_sphere"]
            + st["shades_tri"] * FLOPS["shade_tri"] + st["emissive"] * FLOPS["emissive"] + st["sky"] * FLOPS["sky"]
            + pixels * FLOPS["pixel"])


# --------------------------------------------------------------------------------------------------------
# clocks during the timed region (B200_PROFILING.md)
# --------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw)}


# --------------------------------------------------------------------------------------------------------
# CPU legs (the oracle: a port of the reference's algorithm — the Rust reference cannot be built here)
# --------------------------------------------------------------------------------------------------------
REF_DIVISIONS = 20  # the controller's split (ray-tracer-controller/src/main.rs:33-36): one band = one slave request


def sample_divisions(k: int):
    """k evenly spaced bands of the 20-division split: a bounded, representative sample of the frame."""
    return [int((i + 0.5) * REF_DIVISIONS / k) for i in range(k)]


def oracle_sample(O, sp, tr, cfg, divs, threads=0, keep=None):
    """Render the given divisions with the oracle, each like one reference slave request (world ingest + BVH
    build + band render, ray-tracer-slave/src/main.rs:37-83); returns (rays, seconds).  keep: dict band → pixels."""
    rays, secs = 0, 0.0
    for d in divs:
        p = O.make_params(cfg["width"], cfg["height"], REF_DIVISIONS, d, cfg["spp"], cfg["max_bounces"], 0)
        t0 = time.perf_counter()
        img, st = O.render_rows(sp, tr, p, threads=threads, want_stats=True)
        secs += time.perf_counter() - t0
        rays += st["rays"]
        if keep is not None:
            keep[d] = img
    return rays, secs


def pick_sample(O, sp, tr, cfg, target_s: float):
    """Size the sample for ~target_s seconds of CPU work from a one-band probe (the middle band)."""
    assert cfg["height"] % REF_DIVISIONS == 0
    _, s = oracle_sample(O, sp, tr, cfg, [REF_DIVISIONS // 2])
    k = 1
    for cand in (2, 4, 5, 10, 20):
        if cand * s <= target_s:
            k = cand
    return sample_divisions(k)


def describe_sample(cfg, divs):
    rows = cfg["height"] // REF_DIVISIONS
    return (f"{len(divs)} of the controller's {REF_DIVISIONS} divisions (bands {divs}, {rows} rows x {cfg['width']} px each, "
            f"{cfg['spp']} spp), each rendered like one slave request incl. BVH build")


def run_reference(args, cfg, sp, tr):
    """--impl reference: the reference's CPU algorithm (oracle port, all host threads) on the same config.
    A step is the whole frame (all 20 of the controller's divisions) whenever the run then still ends within a
    few minutes on this box's cores; otherwise an evenly spaced subset, and the line says which fraction."""
    from oracle import oracle as O

    O.build()
    cores = O.hardware_threads()
    budget_s = 170.0 / max(1, args.steps + args.warmup)        # per step
    divs = pick_sample(O, sp, tr, cfg, target_s=budget_s)
    for _ in range(args.warmup):
        oracle_sample(O, sp, tr, cfg, divs[:1])
    rays, secs = 0, 0.0
    for _ in range(args.steps):
        r, s = oracle_sample(O, sp, tr, cfg, divs)
        rays += r
        secs += s
    val = rays / secs / 1e6
    frac = len(divs) / REF_DIVISIONS
    sample = describe_sample(cfg, divs) + " per step"
    return {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, cfg),
        "frame_fraction_per_step": frac, "frame_ms_extrapolated": secs / args.steps * 1e3 / frac,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "note": "C++ oracle = operation-for-operation port of the Rust slave (reference BVH build + "
                                 "unordered traversal); omits the reference's per-ray heap allocations, so it flatters the CPU"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }


def workload_config(args, cfg):
    """The same keys and values in both arms (the driver compares them)."""
    return {"workload": f"{args.workload}: {cfg['width']}x{cfg['height']}, {cfg['spp']} spp, max_bounces {cfg['max_bounces']} "
                        f"(<= {cfg['max_bounces'] + 1} queries/sample), {cfg['n_spheres']} spheres"
                        + (" + plane (2 triangles)" if cfg["plane"] else "") + ", scene_seed 0, seed 0",
            "width": cfg["width"], "height": cfg["height"], "spp": cfg["spp"], "max_bounces": cfg["max_bounces"],
            "n_spheres": cfg["n_spheres"], "n_triangles": 2 if cfg["plane"] else 0,
            "partition": f"8x4-pixel tiles, rotating interleave over {args.gpus} GPU(s)",
            "l2": "flushed between steps: 160 MiB device memset queued in front of every frame"}


def compare_frames(a, b):
    """north_star tolerance: every channel within +-1 LSB on >= 99.9 % of pixels and PSNR >= 50 dB."""
    d = np.abs(a.astype(np.int32) - b.astype(np.int32))
    mse = float((d.astype(np.float64) ** 2).mean())
    return {"n_diff": int((d > 0).sum()), "frac_within_1lsb": float((d.reshape(-1, 3).max(axis=-1) <= 1).mean()),
            "psnr_db": None if mse == 0 else float(10.0 * np.log10(255.0 ** 2 / mse)), "max_diff": int(d.max())}


def ncu_block(path):
    """Pipe / issue figures of the dominant kernel from a committed ncu summary (profiles/); None if it is missing."""
    full = os.path.join(ROOT, path)
    if not os.path.exists(full):
        return None
    txt = open(full).read()

    def grab(name):
        m = re.search(re.escape(name) + r"\s+\S+\s+([0-9.eE+-]+)", txt)
        return float(m.group(1)) if m else None

    out = {"source": path,
           "issue_slots_pct": grab("sm__inst_issued.avg.pct_of_peak_sustained_active"),
           "fma_pipe_cycles_pct": grab("sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active"),
           "alu_pipe_pct": grab("sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active"),
           "threads_per_warp_inst": grab("smsp__thread_inst_executed_per_inst_executed.ratio"),
           "warp_inst": grab("smsp__inst_executed.sum"),
           "kernel_ms": grab("gpu__time_duration.sum")}
    rd, wr = grab("dram__bytes_read.sum"), grab("dram__bytes_write.sum")
    m = re.search(r"dram__bytes_read\.sum\s+(\S+)", txt)
    scale = {"Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "byte": 1.0}.get(m.group(1), None) if m else None
    mw = re.search(r"dram__bytes_write\.sum\s+(\S+)", txt)
    scale_w = {"Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "byte": 1.0}.get(mw.group(1), None) if mw else None
    out["dram_bytes"] = (rd * scale + wr * scale_w) if None not in (rd, wr, scale, scale_w) else None
    return out


def dump_outputs(path, frame, rays):
    """Write what one render step computed, so that two builds can be compared output for output:
    frame_pixels.npy      (n, 3) float32, the frame's 8-bit channels at n pixels, row-major order
    frame_pixel_index.npy (n,) float64, the flat index (y * width + x) of each of those pixels
    rays.npy              (1,) float64, the step's nearest-hit query count (all ranks)
    The pixels are the whole frame when it has at most DUMP_PIXELS of them, else a fixed sample (seed 0) of that many."""
    os.makedirs(path, exist_ok=True)
    h, w, _ = frame.shape
    idx = np.sort(np.random.default_rng(0).choice(h * w, size=min(h * w, DUMP_PIXELS), replace=False))
    np.save(os.path.join(path, "frame_pixels.npy"), frame.reshape(-1, 3)[idx].astype(np.float32))
    np.save(os.path.join(path, "frame_pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, "rays.npy"), np.array([rays], dtype=np.float64))


# --------------------------------------------------------------------------------------------------------
def _claim_stdout():
    """Keep fd 1 for the ONE JSON line: libraries (NCCL prints its version banner there) get stderr instead."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def extra_workloads(rt, ctx, scenes):
    """The other BASELINE configs on one GPU (default run only): kernel time, Mrays/s, e2e ms; C5 ends with ingest time."""
    out = {}
    for name in ("C2", "C4"):
        cfg = scenes.CONFIGS[name]
        sp, tr = scenes.config_scene(name)
        sc = ctx.scene(sp, tr).wait_ready()
        p = rt.make_params(cfg["width"], cfg["height"], spp=cfg["spp"], max_bounces=cfg["max_bounces"])
        host = ctx.pinned_empty((cfg["height"], cfg["width"], 3))
        ks, es = [], []
        for i in range(6):
            ctx.l2_flush(FLUSH_BYTES)
            t0 = time.perf_counter()
            _, st = ctx.render_frame(sc, p, out=host, want_stats=True)
            es.append((time.perf_counter() - t0) * 1e3)
            ks.append(st["kernel_ms"])
        out[name] = {"kernel_ms": float(np.median(ks[1:])), "mrays_per_s": st["rays"] / np.median(ks[1:]) / 1e3,
                     "render_plus_download_ms": float(np.median(es[1:])), "rays": st["rays"],
                     "frame_sha256": hashlib.sha256(host.tobytes()).hexdigest()[:16]}
        sc.close()
    for n in (64, 65536):      # BASELINE config 5: the sweep's ends, 1080p, 1 spp, depth 5
        sp = scenes.synthetic_spheres(n)
        p = rt.make_params(1920, 1080, spp=1, max_bounces=5)
        host = ctx.pinned_empty((1080, 1920, 3))
        ing, ks, es = [], [], []
        for i in range(4):
            t0 = time.perf_counter()
            sc = ctx.scene(sp, None)
            t1 = time.perf_counter()
            _, st = ctx.render_frame(sc, p, out=host, want_stats=True)
            t2 = time.perf_counter()
            sc.close()
            ing.append((t1 - t0) * 1e3); ks.append(st["kernel_ms"]); es.append((t2 - t0) * 1e3)
        out[f"C5_n{n}"] = {"scene_create_ms": float(np.median(ing[1:])), "kernel_ms": float(np.median(ks[1:])),
                           "e2e_ms": float(np.median(es[1:])), "mrays_per_s": st["rays"] / np.median(ks[1:]) / 1e3,
                           "redo_pixels": st["redo_pixels"]}
    return out


def main():
    real_stdout = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C3")
    ap.add_argument("--mode", default=os.environ.get("RT_B200_GATHER", "p2p"), choices=["p2p", "nccl", "single"])
    ap.add_argument("--intersector", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame and ray count of the last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    from rt_b200 import scenes

    cfg = scenes.CONFIGS[args.workload]
    sp, tr = scenes.config_scene(args.workload)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank == 0:
            real_stdout.write(json.dumps(run_reference(args, cfg, sp, tr)) + "\n")
            real_stdout.flush()
        return 0

    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd, stdout=real_stdout.fileno())

    import torch

    import rt_b200 as rt
    from rt_b200 import multi

    dist = None
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def allreduce(x, op):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=op)
        return float(t.item())

    torch.cuda.set_device(local_rank)
    ctx = rt.Context(local_rank)
    info = ctx.device_info()
    scene = ctx.scene(sp, tr).wait_ready()
    W, H = cfg["width"], cfg["height"]
    pixels = W * H
    params = rt.make_params(W, H, spp=cfg["spp"], max_bounces=cfg["max_bounces"], intersector=args.intersector)

    mode = args.mode if world > 1 else "single"
    sched = multi.FrameScheduler(ctx, rank, world, mode=mode if world > 1 else "p2p")
    sched.setup(W, H)

    # ---- counters for the roofline: one untimed instrumented frame (deterministic → same work as timed steps)
    pc = rt.make_params(W, H, spp=cfg["spp"], max_bounces=cfg["max_bounces"], intersector=args.intersector,
                        collect_counters=True)
    cst = sched.render(scene, pc, want_stats=True)
    fp32_peak_tflops, _ = ctx.measure_fp32_peak()
    flush_ms = ctx.l2_flush(FLUSH_BYTES, timed=True)
    flush_ms = min(flush_ms, ctx.l2_flush(FLUSH_BYTES, timed=True))

    def step():
        ctx.l2_flush(FLUSH_BYTES)                      # asynchronous, on the render stream, in front of the kernel
        return sched.render(scene, params, want_stats=True)

    for _ in range(args.warmup):
        step()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    kernel_ms, rays_step = [], 0
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        st = step()
        kernel_ms.append(st["kernel_ms"])
        rays_step = st["rays"]
    barrier()
    elapsed = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    # read back before the all-reduce below: until rank 0 joins it, no rank can start a frame into this buffer again
    last_frame = sched.download(np.empty((H, W, 3), dtype=np.uint8)) if args.dump_outputs and rank == 0 else None

    ROp = dist.ReduceOp if dist is not None else None
    elapsed_max = allreduce(elapsed, ROp.MAX if ROp else None)
    rays_total = allreduce(float(rays_step), ROp.SUM if ROp else None)
    if last_frame is not None:
        dump_outputs(args.dump_outputs, last_frame, rays_total)
    value = rays_total * args.steps / elapsed_max / 1e6
    ms_per_step = elapsed_max / args.steps * 1e3

    # ---- e2e: through the C ABI with host buffers; scene ingest + upload, render, frame in host memory, every step
    host_frame = ctx.pinned_empty((H, W, 3)) if rank == 0 else None
    scene_bytes = scene.device_bytes
    e2e_redo = 0
    phases = {"scene_create": [], "render_and_frame_to_host": [], "scene_destroy": [], "kernel": []}

    def e2e_step():
        nonlocal e2e_redo
        ta = time.perf_counter()
        ctx.l2_flush(FLUSH_BYTES)
        sc = ctx.scene(sp, tr)                       # H2D: primitive SoA + traversal tree + materials (tie tables follow)
        tb = time.perf_counter()
        if world == 1:
            _, s1 = ctx.render_frame(sc, params, out=host_frame, want_stats=True)   # kernel + D2H of the frame
        else:
            s1 = sched.render(sc, params, want_stats=True, out=host_frame)          # slabs stream to the host as they complete
        tc = time.perf_counter()
        e2e_redo = max(e2e_redo, s1["redo_pixels"])
        sc.close()
        td = time.perf_counter()
        phases["scene_create"].append((tb - ta) * 1e3); phases["render_and_frame_to_host"].append((tc - tb) * 1e3)
        phases["scene_destroy"].append((td - tc) * 1e3); phases["kernel"].append(s1["kernel_ms"])

    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_elapsed = allreduce(time.perf_counter() - t0, ROp.MAX if ROp else None)
    e2e_value = rays_total * args.steps / e2e_elapsed / 1e6
    frame_sha = hashlib.sha256(host_frame.tobytes()).hexdigest() if rank == 0 else None

    # the same with a pageable destination (what a Rust Vec<u8> is): N = 1 only, a few steps
    e2e_pageable_ms = None
    if world == 1:
        pageable = np.empty((H, W, 3), dtype=np.uint8)
        ts = []
        for _ in range(4):
            ctx.l2_flush(FLUSH_BYTES)
            t1 = time.perf_counter()
            sc = ctx.scene(sp, tr)
            ctx.render_frame(sc, params, out=pageable)
            sc.close()
            ts.append((time.perf_counter() - t1) * 1e3)
        e2e_pageable_ms = float(np.median(ts[1:]))
        assert hashlib.sha256(pageable.tobytes()).hexdigest() == frame_sha

    # ---- roofline of the render kernel on rank 0 (FP32 CUDA-core pipe; HBM traffic is negligible here)
    k_ms = float(np.mean(kernel_ms))
    flops = algorithmic_flops(cst, pixels // world)
    achieved = flops / (k_ms * 1e-3) / 1e12
    alg_bytes = scene_bytes + (pixels // world) * 3
    bvh = cst["intersector_used"] == 2
    ncu_file = ("profiles/r2_k2_lanes_c3_ncu_summary.txt" if bvh else "profiles/r1_k1_brute_final_ncu_summary.txt")
    ncu = ncu_block(ncu_file) if (args.workload in ("C3", "C2")) else None
    roofline = {
        "bound": "fp32", "kernel": "render_kernel_lanes<%s>" % ("BVH" if bvh else "BRUTE"),
        "achieved": achieved, "peak": fp32_peak_tflops, "unit": "TFLOP/s", "frac": achieved / fp32_peak_tflops,
        "peak_source": "measured live: FFMA-chain micro-benchmark (rt_measure_fp32_peak); MEASURED_PEAKS.json has no CUDA-core figure",
        # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel on C3 at one GPU, read from the
        # committed ncu summary named in "ncu" (null when the file is absent or the workload is another one)
        "traffic": ncu["dram_bytes"] if (ncu and args.workload == "C3" and world == 1) else None,
        "traffic_unit": "bytes per launch (ncu --set full, file in ncu.source)",
        "algorithmic_flops_per_launch": flops, "kernel_ms_avg": k_ms, "kernel_share_of_step": k_ms / ms_per_step,
        "flops_per_ray": flops / max(1, cst["rays"]),
        "hbm": {"algorithmic_bytes_per_launch": alg_bytes, "achieved_gbs": alg_bytes / (k_ms * 1e-3) / 1e9},
        "ncu": ncu,
        "simt_efficiency_query_level": cst["active_lane_iters"] / max(1, cst["total_lane_iters"]),
        "counters": {k: cst[k] for k in ("rays", "primary", "slab_tests", "sphere_tests", "sphere_exact", "sphere_hits",
                                         "tri_tests", "tri_stage", "tri_hits", "shades_sphere", "shades_tri",
                                         "emissive", "sky")},
        "launch": {k: st[k] for k in ("grid_ctas", "cta_threads", "ctas_per_sm", "scene_in_smem", "dyn_smem_bytes")},
    }

    cpu_baseline, parity, extra = None, None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O

        O.build()
        divs = pick_sample(O, sp, tr, cfg, target_s=15.0)
        bands = {}
        r, s = oracle_sample(O, sp, tr, cfg, divs, keep=bands)
        cpu_baseline = {"value": r / s / 1e6, "unit": UNIT, "cores": O.hardware_threads(), "kind": "port",
                        "sample": describe_sample(cfg, divs) + f": {r} rays in {s:.2f} s",
                        "note": "C++ oracle (-O2 -ffp-contract=off), std::thread row-parallel like rayon; a port of the "
                                "Rust slave, which cannot be built in this image"}
        # the timed (e2e) frame against those bands
        rows = H // REF_DIVISIONS
        got = np.concatenate([host_frame[d * rows:(d + 1) * rows] for d in sorted(bands)])
        ref = np.concatenate([bands[d] for d in sorted(bands)])
        parity = dict(compare_frames(got, ref), bands=sorted(bands), pixels=int(ref.shape[0] * ref.shape[1]),
                      against="oracle bands of the cpu_baseline leg vs the frame of the last timed e2e step")
    if rank == 0 and world == 1 and not args.no_extra and args.workload == "C3":
        extra = extra_workloads(rt, ctx, scenes)

    if dist is not None:
        barrier()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "frame_ms": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, cfg),
            "run": {"gather": mode, "intersector": int(cst["intersector_used"]), "device": info["name"],
                    "l2_flush_ms": flush_ms, "l2_flush_inside_bracket": True},
            "rays_per_step": rays_total, "mrays_per_s_per_gpu": value / world,
            "frame_sha256": frame_sha,
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_elapsed / args.steps * 1e3,
                    "h2d_bytes_per_step": int(scene_bytes * world + 72 * world),
                    "d2h_bytes_per_step": int(pixels * 3 + 128 * world),
                    "pageable_destination_ms": e2e_pageable_ms, "redo_pixels_max": e2e_redo,
                    "rank0_phases_ms_median": {k: float(np.median(v[-args.steps:])) for k, v in phases.items()},
                    "what": "rt_scene_create (ingest + upload; the reference-topology tree follows on a builder thread) + render "
                            "+ frame to pinned host memory, per step"
                            + ("; slabs stream to the host while other slabs render" if world > 1 else "")},
            "gpu_launches": args.steps * world,
            "clocks": clocks,
            "roofline": roofline,
        }
        if parity:
            line["parity"] = parity
        if cpu_baseline:
            line["cpu_baseline"] = cpu_baseline
        if extra:
            line["extra"] = extra
        real_stdout.write(json.dumps(line) + "\n")
        real_stdout.flush()
    sched.close()
    scene.close()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
