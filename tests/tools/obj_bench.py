"""OBJ ingest of the controller's /upload body, host path against device path.

  * parse    a height-field mesh written by obj.write_obj (one model, one material) at about 131k, 524k and 2M triangles:
             obj.build_world on the host against Context.parse_obj (rt_obj_build_world, including the copy of the body
             to the device and the triangles back); the results are asserted byte-equal every round
  * device   for one call at each size (torch.profiler, CUDA activities, a run of its own): the kernels' device time,
             the host-to-device and device-to-host copies (and memsets), and what remains of the call's median time:
             the staging of the pageable copies, the binding's copy of the result, the host's MTL / usemtl name work,
             the stage synchronisations and launch gaps
  * upload   Controller(worker=...).upload + poll of the 524k mesh at 1920x1080 (spp 4, max_bounces 4), with the device
             parse and with the host parse; the /poll JPEG bytes are asserted equal
host_ms is a host clock around work that ends with the data in host memory.  Medians over alternated rounds.  The card's
name and power limit are read in the same run.

    python tests/tools/obj_bench.py [--reps 10] [--host-reps 3] [--out profiles/r8_obj_parse.json]
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
sys.path.insert(0, os.path.join(ROOT, "ray-tracer-s8_b200"))

from rt_b200 import controller, obj, slave  # noqa: E402

SIZES = {"131k": 256, "524k": 512, "2M": 1024}  # grid quads per side: 2 q^2 triangles
MTL = b"newmtl m\nKd 0.5 0.5 0.5\nNs 300\n"


def gpu_facts():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return [dict(zip(("index", "name", "power_limit", "sm_clock_max"), [x.strip() for x in line.split(",")]))
                for line in out.splitlines()]
    except Exception as e:  # the numbers stay valid; the report says the facts could not be read
        return [{"nvidia_smi_error": str(e)}]


def mesh_body(q):
    """(q + 1)^2 vertices of a height field 20 units in front of the camera, 2 q^2 triangles, as OBJ ++ MTL."""
    xs = np.linspace(-12, 12, q + 1, dtype=np.float32)
    V = np.stack(np.meshgrid(xs, xs, indexing="ij"), -1).reshape(-1, 2)
    V = np.concatenate([V, (np.sin(V[:, :1]) - 20).astype(np.float32)], 1)
    idx = np.arange((q + 1) ** 2).reshape(q + 1, q + 1)
    a, b, c, d = idx[:-1, :-1].ravel(), idx[1:, :-1].ravel(), idx[1:, 1:].ravel(), idx[:-1, 1:].ravel()
    F = np.concatenate([np.stack([a, b, c], 1), np.stack([a, c, d], 1)])
    o = obj.write_obj(V, F, "m")
    return o + MTL, len(o)


def device_breakdown(fn):
    """Device time of one call of fn by kind (torch.profiler): kernels, copies each way, memsets."""
    from torch.profiler import ProfilerActivity, profile

    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
        out = {"kernel_ms": 0.0, "h2d_ms": 0.0, "d2h_ms": 0.0, "memset_ms": 0.0, "kernels": {}, "copies": {}}
        for e in prof.events():
            t = e.device_time_total / 1e3
            k = re.search(r"(obj_\w+|jpeg_carry_kernel)(<\w+>)?", e.name)
            if k:
                out["kernel_ms"] += t
                out["kernels"][k.group(0)] = out["kernels"].get(k.group(0), 0.0) + t
                continue
            out["copies"][e.name] = out["copies"].get(e.name, 0.0) + t
            if "HtoD" in e.name:
                out["h2d_ms"] += t
            elif "DtoH" in e.name:
                out["d2h_ms"] += t
            elif "Memset" in e.name:
                out["memset_ms"] += t
        return out
    except Exception as e:  # the host-clock numbers stand without it
        return {"profiler_error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--upload-reps", type=int, default=3)
    ap.add_argument("--sizes", default=",".join(SIZES))
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_obj_parse.json"))
    a = ap.parse_args()
    import torch  # noqa: F401  (the profiler; imported before the timed loops so its start-up is not timed)

    facts = gpu_facts()
    rep = {"gpus": facts, "parse": {}}
    wk = slave.Worker(0, spp=4, max_bounces=4)
    ctx = wk.ctx
    try:
        for name in a.sizes.split(","):
            data, n = mesh_body(SIZES[name])
            ref = obj.build_world(data, n).tobytes()
            for _ in range(2):
                assert ctx.parse_obj(data, n).tobytes() == ref
            host, dev = [], []
            for r in range(max(a.reps, a.host_reps)):
                if r < a.host_reps:
                    t0 = time.perf_counter()
                    h = obj.build_world(data, n)
                    host.append((time.perf_counter() - t0) * 1e3)
                    assert h.tobytes() == ref
                t0 = time.perf_counter()
                d = ctx.parse_obj(data, n)
                dev.append((time.perf_counter() - t0) * 1e3)
                assert d.tobytes() == ref
            r = {"triangles": len(ref) // 56, "obj_bytes": n, "body_bytes": len(data),
                 "host_ms": statistics.median(host), "device_path_ms": statistics.median(dev),
                 "host_ms_all": host, "device_path_ms_all": dev}
            r["device"] = device_breakdown(lambda: ctx.parse_obj(data, n))
            if "kernel_ms" in r["device"]:
                busy = sum(r["device"][k] for k in ("kernel_ms", "h2d_ms", "d2h_ms", "memset_ms"))
                r["device"]["other_ms"] = r["device_path_ms"] - busy
            rep["parse"][name] = r
            print(name, {k: v for k, v in r.items() if not k.endswith("_all")}, flush=True)

        # ---- a whole upload + poll at 1080p ------------------------------------------------------------------
        data, n = mesh_body(SIZES["524k"])
        times, jpegs = {"device": [], "host": []}, {}
        for _ in range(a.upload_reps):
            for mode in ("device", "host"):
                c = controller.Controller(worker=wk)
                if mode == "host":
                    c._obj_parser = lambda: None
                t0 = time.perf_counter()
                jpeg, ok = c.poll(c.upload(data, n))
                times[mode].append((time.perf_counter() - t0) * 1e3)
                assert ok
                jpegs.setdefault(mode, jpeg)
                assert jpeg == jpegs[mode]
        assert jpegs["device"] == jpegs["host"]
        rep["upload_poll_524k_1080p"] = {"spp": 4, "max_bounces": 4, "jpeg_bytes": len(jpegs["device"]),
                                         "device_parse_ms": statistics.median(times["device"]),
                                         "host_parse_ms": statistics.median(times["host"]),
                                         "device_parse_ms_all": times["device"], "host_parse_ms_all": times["host"]}
    finally:
        wk.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rep, f, indent=2)
    print(json.dumps({k: v for k, v in rep.items() if k != "parse"}, default=str)[:2000])


if __name__ == "__main__":
    main()
