"""Progressive rendering cost on C3 (4K, 16 spp, depth 5, 1024 spheres + plane), one GPU.

Renders the frame as one rt_render_frame at 16 spp and as chunks of samples (rt_render_samples): 16 x 1, 4 x 4, 2 x 8,
once with only the last chunk downloaded and once with every chunk downloaded, and as ONE chunk of 16 (the resumable
kernel against the product kernel on the same work).  Every frame starts behind an L2 flush
(rt_l2_flush, 512 MB); modes alternate within each repetition.  Writes a JSON report (default
profiles/r3_progressive_c3.json) with per-chunk kernel ms, total kernel ms, end-to-end ms, the state bytes each chunk
moves (computed from the shape) and the sha256 of every final frame, which must be the same in every mode.

    python tests/tools/progressive_bench.py [--reps 10] [--warmup 2] [--out PATH]
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

STATE_RECORD_BYTES = 48
FLUSH_BYTES = 512 << 20


def gpu_facts(index):
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"nvidia_smi_name": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as e:  # the numbers stay valid; the report says the facts could not be read
        return {"nvidia_smi_error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_progressive_c3.json"))
    a = ap.parse_args()

    c = rt.scenes.CONFIGS["C3"]
    w, h, spp, mb = c["width"], c["height"], c["spp"], c["max_bounces"]
    sp, tr = rt.scenes.config_scene("C3")
    pixels = w * h
    modes = {"frame_16": None}
    for chunks in ((16,), (1,) * 16, (4,) * 4, (8,) * 2):
        tag = f"{len(chunks)}x{chunks[0]}"
        modes[f"chunks_{tag}_last_download"] = (chunks, False)
        modes[f"chunks_{tag}_every_download"] = (chunks, True)

    with rt.Context(0) as ctx:
        sc = ctx.scene(sp, tr).wait_ready()
        out = ctx.pinned_empty((h, w, 3))
        acc = ctx.accum(rt.make_params(w, h, max_bounces=mb))
        p16 = rt.make_params(w, h, spp=spp, max_bounces=mb)

        def run(mode):
            spec = modes[mode]
            ctx.l2_flush(FLUSH_BYTES)
            t0 = time.perf_counter()
            if spec is None:
                _, st = ctx.render_frame(sc, p16, out=out, want_stats=True)
                e2e = (time.perf_counter() - t0) * 1e3
                return {"kernel_ms": [st["kernel_ms"]], "e2e_ms": e2e, "redo": [st["redo_pixels"]]}
            chunks, every = spec
            acc.reset()
            ks, redo = [], []
            for i, n in enumerate(chunks):
                last = i == len(chunks) - 1
                r = ctx.render_samples(sc, acc, n, out=out, download=every or last, want_stats=True)
                st = r[1]
                ks.append(st["kernel_ms"])
                redo.append(st["redo_pixels"])
            e2e = (time.perf_counter() - t0) * 1e3
            assert acc.samples == spp
            return {"kernel_ms": ks, "e2e_ms": e2e, "redo": redo}

        for _ in range(a.warmup):
            for m in modes:
                run(m)
        res = {m: [] for m in modes}
        sha = {m: set() for m in modes}
        for _ in range(a.reps):
            for m in modes:
                res[m].append(run(m))
                sha[m].add(hashlib.sha256(out.tobytes()).hexdigest())
        dev = ctx.device_info()
        acc.close()
        sc.close()

    report = {
        "workload": f"C3: {w}x{h}, {spp} spp, max_bounces {mb}, {len(sp)} spheres + plane, one GPU",
        "device": dev["name"], **gpu_facts(int(os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0] or 0)),
        "method": (f"{a.warmup} warm-up rounds, then {a.reps} rounds; each round runs every mode once, in order; "
                   f"every frame starts behind a {FLUSH_BYTES >> 20} MB L2 flush; kernel_ms from CUDA events (per call), "
                   "e2e_ms = host clock around the frame's calls (each returns after the device has finished); pinned "
                   "destination; medians over the rounds"),
        "state_bytes_note": ("per chunk: pixels x 48 B written, plus pixels x 48 B read from the second chunk on "
                             "(the first chunk seeds its chains); computed from the shape, not measured"),
        "modes": {},
    }
    ref_sha = None
    for m, runs in res.items():
        chunks = [1] if modes[m] is None else list(modes[m][0])
        per_chunk = [statistics.median(r["kernel_ms"][i] for r in runs) for i in range(len(chunks))]
        tot = [sum(r["kernel_ms"]) for r in runs]
        e2e = [r["e2e_ms"] for r in runs]
        entry = {
            "chunks": chunks if modes[m] else [spp],
            "kernel_ms_per_chunk_median": [round(x, 4) for x in per_chunk],
            "kernel_ms_total_median": round(statistics.median(tot), 4),
            "kernel_ms_total_min_max": [round(min(tot), 4), round(max(tot), 4)],
            "e2e_ms_median": round(statistics.median(e2e), 4),
            "e2e_ms_min_max": [round(min(e2e), 4), round(max(e2e), 4)],
            "redo_pixels_max": max(max(r["redo"]) for r in runs),
            "sha256": sorted(sha[m]),
        }
        if modes[m] is not None:
            entry["state_bytes_per_chunk"] = [pixels * STATE_RECORD_BYTES * (1 if i == 0 else 2)
                                              for i in range(len(chunks))]
        report["modes"][m] = entry
        assert len(sha[m]) == 1, (m, sha[m])
        ref_sha = ref_sha or next(iter(sha[m]))
        assert next(iter(sha[m])) == ref_sha, (m, sha[m], ref_sha)
    base = report["modes"]["frame_16"]
    for m, e in report["modes"].items():
        e["kernel_overhead_vs_frame_16_pct"] = round(100.0 * (e["kernel_ms_total_median"] / base["kernel_ms_total_median"] - 1), 2)
        e["e2e_overhead_vs_frame_16_pct"] = round(100.0 * (e["e2e_ms_median"] / base["e2e_ms_median"] - 1), 2)
    report["one_sha256_across_modes"] = ref_sha
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    for m, e in report["modes"].items():
        print(f"{m:34s} kernel {e['kernel_ms_total_median']:8.3f} ms ({e['kernel_overhead_vs_frame_16_pct']:+.2f} %)  "
              f"e2e {e['e2e_ms_median']:8.3f} ms ({e['e2e_overhead_vs_frame_16_pct']:+.2f} %)")
    print(json.dumps({"device": report["device"], "power_limit": report.get("power_limit"), "sha256": ref_sha}))


if __name__ == "__main__":
    main()
