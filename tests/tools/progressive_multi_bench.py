"""Progressive rendering on several GPUs: what a chunk boundary costs on C3 (4K, 16 spp, depth 5, 1024 spheres + plane).

For 1, 2, 4 and 8 GPUs (as many as the box has) renders the frame as one rt_render_frame_multi at 16 spp and as chunks of
samples with rt_render_samples_multi: 2 x 8, 4 x 4 and 16 x 1 with only the last chunk downloaded, and 4 x 4 with every
chunk downloaded (an interactive preview).  Every frame starts behind an L2 flush (rt_l2_flush, 512 MB) on every GPU;
modes alternate within each round.  Writes a JSON report (default profiles/r3_progressive_multi_c3.json) with per-chunk
kernel ms (the slowest GPU's), total kernel ms, end-to-end ms, medians over the rounds, the card's name and power limit
read in the same run, and the sha256 of every final frame, which must be the same in every mode and at every GPU count.

    python tests/tools/progressive_multi_bench.py [--reps 10] [--warmup 2] [--out PATH]
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
sys.path.insert(0, os.path.join(ROOT, "ray-tracer-s8_b200"))

import rt_b200 as rt  # noqa: E402
from rt_b200 import multi  # noqa: E402

FLUSH_BYTES = 512 << 20
MODES = {"frame_multi_16": None, "chunks_2x8": ((8,) * 2, False), "chunks_4x4": ((4,) * 4, False),
         "chunks_16x1": ((1,) * 16, False), "chunks_4x4_every_download": ((4,) * 4, True)}


def gpu_facts():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return [dict(zip(("index", "name", "power_limit", "sm_clock_max"), [x.strip() for x in line.split(",")]))
                for line in out.splitlines()]
    except Exception as e:  # the numbers stay valid; the report says the facts could not be read
        return [{"nvidia_smi_error": str(e)}]


def device_count():
    import torch

    return torch.cuda.device_count()


def bench_gpus(n_gpus, reps, warmup):
    c = rt.scenes.CONFIGS["C3"]
    w, h, spp, mb = c["width"], c["height"], c["spp"], c["max_bounces"]
    sp, tr = rt.scenes.config_scene("C3")
    m = multi.MultiDeviceRenderer(list(range(n_gpus)))
    try:
        scenes = [s.wait_ready() for s in m.scenes(sp, tr)]
        out = m.ctxs[0].pinned_empty((h, w, 3))
        accs = [ctx.accum(rt.make_params(w, h, max_bounces=mb)) for ctx in m.ctxs]
        p16 = rt.make_params(w, h, spp=spp, max_bounces=mb)

        def run(mode):
            for ctx in m.ctxs:
                ctx.l2_flush(FLUSH_BYTES)
            spec = MODES[mode]
            t0 = time.perf_counter()
            if spec is None:
                _, st = m.render(scenes, p16, out=out, want_stats=True)
                return {"kernel_ms": [st["kernel_ms"]], "e2e_ms": (time.perf_counter() - t0) * 1e3, "redo": [st["redo_pixels"]]}
            chunks, every = spec
            for a in accs:
                a.reset()
            ks, redo = [], []
            for i, n in enumerate(chunks):
                down = every or i == len(chunks) - 1
                _, st = rt.render_samples_multi(m.ctxs, scenes, accs, n, out=out, download=down, want_stats=True)
                ks.append(st["kernel_ms"])
                redo.append(st["redo_pixels"])
            e2e = (time.perf_counter() - t0) * 1e3
            assert accs[0].samples == spp
            return {"kernel_ms": ks, "e2e_ms": e2e, "redo": redo}

        for _ in range(warmup):
            for mode in MODES:
                run(mode)
        res = {mode: [] for mode in MODES}
        sha = {mode: set() for mode in MODES}
        for _ in range(reps):
            for mode in MODES:
                res[mode].append(run(mode))
                sha[mode].add(hashlib.sha256(out.tobytes()).hexdigest())
        device = m.ctxs[0].device_info()["name"]
        for a in accs:
            a.close()
        for s in scenes:
            s.close()
    finally:
        m.close()

    entry = {"n_gpus": n_gpus, "device": device, "modes": {}}
    for mode, runs in res.items():
        chunks = [spp] if MODES[mode] is None else list(MODES[mode][0])
        tot = [sum(r["kernel_ms"]) for r in runs]
        e2e = [r["e2e_ms"] for r in runs]
        entry["modes"][mode] = {
            "chunks": chunks,
            "kernel_ms_per_chunk_median": [round(statistics.median(r["kernel_ms"][i] for r in runs), 4) for i in range(len(chunks))],
            "kernel_ms_total_median": round(statistics.median(tot), 4),
            "kernel_ms_total_min_max": [round(min(tot), 4), round(max(tot), 4)],
            "e2e_ms_median": round(statistics.median(e2e), 4),
            "e2e_ms_min_max": [round(min(e2e), 4), round(max(e2e), 4)],
            "redo_pixels_max": max(max(r["redo"]) for r in runs),
            "frame_sha256": sorted(sha[mode]),
        }
    base = entry["modes"]["frame_multi_16"]
    for e in entry["modes"].values():
        e["kernel_vs_frame_multi_pct"] = round(100.0 * (e["kernel_ms_total_median"] / base["kernel_ms_total_median"] - 1), 2)
        e["e2e_vs_frame_multi_pct"] = round(100.0 * (e["e2e_ms_median"] / base["e2e_ms_median"] - 1), 2)
    return entry


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_progressive_multi_c3.json"))
    a = ap.parse_args()

    have = device_count()
    if have < 1:
        raise SystemExit("no CUDA device: this benchmark measures the GPU and has no fallback")
    counts = [n for n in (1, 2, 4, 8) if n <= have]
    c = rt.scenes.CONFIGS["C3"]
    report = {
        "workload": f"C3: {c['width']}x{c['height']}, {c['spp']} spp, max_bounces {c['max_bounces']}, 1024 spheres + plane",
        "gpus": gpu_facts(),
        "method": (f"per GPU count: {a.warmup} warm-up rounds, then {a.reps} rounds; each round runs every mode once, in "
                   f"order; every frame starts behind a {FLUSH_BYTES >> 20} MB L2 flush on every GPU; kernel_ms from CUDA "
                   "events per call (the slowest GPU's); e2e_ms = host clock around the frame's calls (each returns after "
                   "the frame is in host memory); pinned destination; medians over the rounds"),
        "runs": [bench_gpus(n, a.reps, a.warmup) for n in counts],
    }
    shas = {s for r in report["runs"] for e in r["modes"].values() for s in e["frame_sha256"]}
    report["frame_sha256"] = sorted(shas)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    for r in report["runs"]:
        for mode, e in r["modes"].items():
            print(f"{r['n_gpus']} GPU  {mode:26s} kernel {e['kernel_ms_total_median']:8.3f} ms ({e['kernel_vs_frame_multi_pct']:+.2f} %)"
                  f"  e2e {e['e2e_ms_median']:8.3f} ms ({e['e2e_vs_frame_multi_pct']:+.2f} %)")
    print(json.dumps({"gpus": report["gpus"], "frame_sha256": report["frame_sha256"]}))
    assert len(shas) == 1, shas


if __name__ == "__main__":
    main()
