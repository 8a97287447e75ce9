"""Batched divisions: one rt_render_divisions call against one rt_render_division per band, at the reference's defaults.

C2's scene (256 spheres) at 1920x1080, 20 divisions, 100 spp, max_bounces 10 (controller main.rs:33-36, slave
main.rs:39,51).  Modes, alternated within every round:
  * div_x20          20 x rt_render_division, bands 0..19
  * divs_in_order    one rt_render_divisions of bands 0..19 (one contiguous run: the plain row-range path)
  * divs_shuffled    one rt_render_divisions of the 20 bands in a fixed shuffled order (the banded launch on the same work:
                     the cost of the band table)
  * div_x10_odd      10 x rt_render_division, bands 1, 3, ..., 19 (what one of two slaves receives)
  * divs_odd         one rt_render_divisions of bands 1, 3, ..., 19
  * worker_x20       20 x slave.Worker.render (RenderInfo in, ImageSlice out)
  * worker_many      one slave.Worker.render_many of the same 20 requests
host_ms is a host clock around the mode's calls, each of which returns when its bands are in host memory; kernel_ms is the
sum of the calls' CUDA-event kernel times.  Medians over the rounds.  Every mode's bands are compared byte for byte with
div_x20's in every round.  The scene lives in shared memory and L2 in every mode, so there is no L2 flush.  The card's name
and power limit are read in the same run.  Writes a JSON report (default profiles/r5_divisions_c2.json).

    python tests/tools/divisions_bench.py [--reps 10] [--warmup 2] [--out PATH]
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
sys.path.insert(0, os.path.join(ROOT, "ray-tracer-s8_b200"))

import rt_b200 as rt  # noqa: E402
from rt_b200 import slave, wire  # noqa: E402

W, H, DIV, SPP, MB = 1920, 1080, 20, 100, 10
SHUFFLED = [int(d) for d in np.random.default_rng(7).permutation(DIV)]
ODD = list(range(1, DIV, 2))


def gpu_facts():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return [dict(zip(("index", "name", "power_limit", "sm_clock_max"), [x.strip() for x in line.split(",")]))
                for line in out.splitlines()]
    except Exception as e:  # the numbers stay valid; the report says the facts could not be read
        return [{"nvidia_smi_error": str(e)}]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_divisions_c2.json"))
    a = ap.parse_args()

    sp, tr = rt.scenes.config_scene("C2")
    ctx = rt.Context(0)
    sc = ctx.scene(sp, tr).wait_ready()
    p = rt.make_params(W, H, divisions=DIV, spp=SPP, max_bounces=MB)
    rows = H // DIV
    wk = slave.Worker(0, spp=SPP, max_bounces=MB)
    world = wire.World(sp if sp is not None else np.zeros(0, wire.SPHERE_DTYPE),
                       tr if tr is not None else np.zeros(0, wire.TRIANGLE_DTYPE),
                       np.arange(len(sp if sp is not None else []) + len(tr if tr is not None else []), dtype=np.uint32))
    meta = wire.RenderMeta(H, W, DIV, "00000000-0000-4000-8000-0000000000c2")
    infos = [wire.RenderInfo(world, meta, d) for d in range(DIV)]
    out20 = ctx.pinned_empty((DIV, rows, W, 3))
    out10 = ctx.pinned_empty((len(ODD), rows, W, 3))

    def per_division(nos, out):
        q = rt.RtParams.from_buffer_copy(p)
        ks = 0.0
        for k, d in enumerate(nos):
            q.division_no = d
            _, st = ctx.render_division(sc, q, out=out[k], want_stats=True)
            ks += st["kernel_ms"]
        return {d: out[k] for k, d in enumerate(nos)}, ks

    def batched(nos, out):
        _, st = ctx.render_divisions(sc, p, nos, out=out, want_stats=True)
        return {d: out[k] for k, d in enumerate(nos)}, st["kernel_ms"]

    def worker_each():
        ks, got = 0.0, {}
        for i in infos:
            sl, st = wk.render(i, want_stats=True)
            got[i.division_no] = sl.image.reshape(rows, W, 3)
            ks += st["kernel_ms"]
        return got, ks

    def worker_many():
        sls, st = wk.render_many(infos, want_stats=True)
        return {s.division_no: s.image.reshape(rows, W, 3) for s in sls}, st["kernel_ms"]

    modes = {
        "div_x20": lambda: per_division(list(range(DIV)), out20),
        "divs_in_order": lambda: batched(list(range(DIV)), out20),
        "divs_shuffled": lambda: batched(SHUFFLED, out20),
        "div_x10_odd": lambda: per_division(ODD, out10),
        "divs_odd": lambda: batched(ODD, out10),
        "worker_x20": worker_each,
        "worker_many": worker_many,
    }
    ref = {}

    def run(mode):
        t0 = time.perf_counter()
        got, ks = modes[mode]()
        host = (time.perf_counter() - t0) * 1e3
        digest = {d: hashlib.sha256(np.ascontiguousarray(b).tobytes()).hexdigest() for d, b in got.items()}
        if mode == "div_x20":
            ref.update(digest)
        for d, h in digest.items():
            assert h == ref[d], (mode, d)
        return host, ks

    try:
        for _ in range(a.warmup):
            for mode in modes:
                run(mode)
        res = {mode: [] for mode in modes}
        for _ in range(a.reps):
            for mode in modes:
                res[mode].append(run(mode))
        device = ctx.device_info()["name"]
    finally:
        wk.close()
        sc.close()
        ctx.close()

    report = {
        "workload": f"C2 scene (256 spheres): {W}x{H}, {DIV} divisions of {rows} rows, {SPP} spp, max_bounces {MB}",
        "gpus": gpu_facts(),
        "device": device,
        "method": (f"{a.warmup} warm-up rounds, then {a.reps} rounds; each round runs every mode once, in order; host_ms = "
                   "host clock around the mode's calls, each returning with its bands in host memory (pinned destination "
                   "for the context's calls; the Worker's own arrays for the worker modes); kernel_ms = sum of the calls' "
                   "CUDA-event kernel times; medians over the rounds; every band's sha256 equals div_x20's in every round"),
        "shuffled_order": SHUFFLED,
        "band_sha256": [ref[d] for d in range(DIV)],
        "modes": {},
    }
    for mode, runs in res.items():
        host = [r[0] for r in runs]
        ker = [r[1] for r in runs]
        report["modes"][mode] = {
            "host_ms_median": round(statistics.median(host), 4), "host_ms_min_max": [round(min(host), 4), round(max(host), 4)],
            "kernel_ms_median": round(statistics.median(ker), 4), "kernel_ms_min_max": [round(min(ker), 4), round(max(ker), 4)],
        }
    m = report["modes"]
    for new, old in (("divs_in_order", "div_x20"), ("divs_shuffled", "div_x20"), ("divs_shuffled", "divs_in_order"),
                     ("divs_odd", "div_x10_odd"), ("worker_many", "worker_x20")):
        report.setdefault("comparisons", {})[f"{new}_vs_{old}"] = {
            "host_pct": round(100.0 * (m[new]["host_ms_median"] / m[old]["host_ms_median"] - 1), 2),
            "kernel_pct": round(100.0 * (m[new]["kernel_ms_median"] / m[old]["kernel_ms_median"] - 1), 2),
        }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    for mode, e in m.items():
        print(f"{mode:14s} host {e['host_ms_median']:9.3f} ms  kernel {e['kernel_ms_median']:9.3f} ms")
    print(json.dumps({"gpus": report["gpus"], "comparisons": report["comparisons"]}))


if __name__ == "__main__":
    main()
