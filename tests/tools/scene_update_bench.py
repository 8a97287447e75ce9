"""rt_scene_update against rt_scene_create, one GPU.

Worlds: C3 (1024 spheres + plane: host-built SAH traversal tree, reference tables on the builder thread) and 65,536
spheres (device-built LBVH).  For each: the wall time of a warm rt_scene_create (followed by rt_scene_destroy, untimed),
of rt_scene_update with every primitive moved, and of rt_scene_update with materials only.  Every call returns
synchronised; medians over --reps calls.  Creates and updates start with the previous call's reference tables landed
(rt_scene_wait_ready, untimed), so no call waits for an earlier builder thread.

Tree quality: the refit keeps the created topology, so a scene whose primitives have moved a long way culls worse than
a fresh one.  On C3 (3840x2160, 16 spp, depth 5), after 1, 10 and 50 cumulative jitter updates, the kernel time and the
slab_tests count of the updated scene against a scene created from the same world (frames must be identical).

Writes JSON (default profiles/r5_scene_update.json) with the card name and power limit read in the same run.

    python tests/tools/scene_update_bench.py [--reps 30] [--out PATH]
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


def gpu_facts(index):
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"nvidia_smi_name": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as e:  # the numbers stay valid; the report says the facts could not be read
        return {"nvidia_smi_error": str(e)}


def jitter(sp, tr, rng, scale):
    """Every sphere moved by up to scale x its radius per axis; triangles (the plane) stay."""
    sp = sp.copy()
    sp["center"] += (rng.uniform(-scale, scale, (len(sp), 3)) * sp["radius"][:, None]).astype(np.float32)
    return sp, tr


def recolour(sp, rng):
    sp = sp.copy()
    sp["albedo"] = rng.uniform(0.05, 0.95, (len(sp), 3)).astype(np.float32)
    return sp


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return (time.perf_counter() - t0) * 1e3, r


def ingest_times(ctx, sp, tr, reps):
    rng = np.random.default_rng(1)
    for _ in range(3):  # warm: staging buffer, retired blobs, device-build scratch, module load
        ctx.scene(sp, tr).wait_ready().close()
    create = []
    for _ in range(reps):
        ms, sc = timed(lambda: ctx.scene(sp, tr))
        create.append(ms)
        sc.wait_ready().close()
    sc = ctx.scene(sp, tr).wait_ready()
    moved, mats = [], []
    cur = sp
    for k in range(reps + 3):
        cur, _ = jitter(cur, tr, rng, 0.05)
        ms, _ = timed(lambda: sc.update(cur, tr))
        sc.wait_ready()
        if k >= 3:
            moved.append(ms)
    for k in range(reps + 3):
        cur = recolour(cur, rng)
        ms, _ = timed(lambda: sc.update(cur, tr))
        sc.wait_ready()
        if k >= 3:
            mats.append(ms)
    sc.close()
    med = lambda v: round(statistics.median(v), 4)  # noqa: E731
    return {
        "n_prims": len(sp) + len(tr),
        "create_ms_median": med(create), "create_ms_min_max": [round(min(create), 4), round(max(create), 4)],
        "update_moved_ms_median": med(moved), "update_moved_ms_min_max": [round(min(moved), 4), round(max(moved), 4)],
        "update_materials_ms_median": med(mats), "update_materials_ms_min_max": [round(min(mats), 4), round(max(mats), 4)],
    }


def tree_quality(ctx, sp, tr, checkpoints=(1, 10, 50), scale=0.2, reps=3):
    c = rt.scenes.CONFIGS["C3"]
    p = rt.make_params(c["width"], c["height"], spp=c["spp"], max_bounces=c["max_bounces"], intersector=2)
    pc = rt.make_params(c["width"], c["height"], spp=c["spp"], max_bounces=c["max_bounces"], intersector=2,
                        collect_counters=True)
    rng = np.random.default_rng(2)

    def measure(scene):
        img, st = ctx.render_frame(scene, pc, want_stats=True)
        ks = [ctx.render_frame(scene, p, want_stats=True)[1]["kernel_ms"] for _ in range(reps)]
        return hashlib.sha256(img.tobytes()).hexdigest(), st["slab_tests"], statistics.median(ks)

    sc = ctx.scene(sp, tr).wait_ready()
    cur, out = sp, []
    for k in range(1, max(checkpoints) + 1):
        cur, _ = jitter(cur, tr, rng, scale)
        sc.update(cur, tr)
        if k in checkpoints:
            sc.wait_ready()
            h_u, slab_u, ms_u = measure(sc)
            fresh = ctx.scene(cur, tr).wait_ready()
            h_f, slab_f, ms_f = measure(fresh)
            fresh.close()
            assert h_u == h_f, k
            out.append({"updates": k, "kernel_ms_updated": round(ms_u, 4), "kernel_ms_fresh": round(ms_f, 4),
                        "slab_tests_updated": slab_u, "slab_tests_fresh": slab_f,
                        "slab_tests_ratio": round(slab_u / slab_f, 4), "frame_sha256": h_u})
    sc.close()
    return {"jitter": f"every sphere moved by up to {scale} x its radius per axis per update, cumulative",
            "kernel_ms": f"median of {reps} frames, CUDA events", "points": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_scene_update.json"))
    a = ap.parse_args()

    with rt.Context(0) as ctx:
        c3 = rt.scenes.config_scene("C3")
        big = (rt.scenes.synthetic_spheres(65536), rt.scenes.no_triangles())
        report = {
            "device": ctx.device_info()["name"],
            **gpu_facts(int(os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0] or 0)),
            "method": ("host wall clock around each call (each returns synchronised), after 3 warm-up calls; medians "
                       f"over {a.reps} calls; moved = every sphere jittered by up to 0.05 x its radius per axis, "
                       "materials = new albedo for every sphere"),
            "ingest": {"C3": ingest_times(ctx, *c3, a.reps), "spheres_65536": ingest_times(ctx, *big, a.reps)},
            "tree_quality_C3": tree_quality(ctx, *c3),
        }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report, indent=1))


if __name__ == "__main__":
    main()
