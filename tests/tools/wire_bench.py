"""The slave's wire format, host path against device path, at the reference controller's sizes.

  * parse    one RenderInfo body of a 262,144-triangle world (what the controller POSTs per division for a large OBJ):
             wire.parse_render_info on the host against Worker.parse (rt_world_parse_json, including the copy of the body
             to the device and the arrays back); the results are asserted equal every round
  * job      the 20 divisions of a 1920x1080 C2 job rendered and POSTed to a local HTTP sink: render_many + ImageSlice
             .to_json() per band against render_many_json (rt_render_divisions_json); the posted bytes are asserted equal
  * device   kernel time of the parse and of the body writer (torch.profiler, CUDA activities, a run of its own)
host_ms is a host clock around work that ends with the data in host memory.  Medians over alternated rounds.  The card's
name and power limit are read in the same run.

    python tests/tools/wire_bench.py [--reps 10] [--host-reps 3] [--out profiles/r7_wire_c2.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from http.server import BaseHTTPRequestHandler, ThreadingHTTPServer

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
sys.path.insert(0, os.path.join(ROOT, "ray-tracer-s8_b200"))

import rt_b200 as rt  # noqa: E402
from rt_b200 import scenes, slave, wire  # noqa: E402

ID = "0b5e6d0e-8f3c-4d5a-9c1b-2f9e3a4b5c6d"


def gpu_facts():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return [dict(zip(("index", "name", "power_limit", "sm_clock_max"), [x.strip() for x in line.split(",")]))
                for line in out.splitlines()]
    except Exception as e:  # the numbers stay valid; the report says the facts could not be read
        return [{"nvidia_smi_error": str(e)}]


def triangle_body(n, seed=1):
    rng = np.random.default_rng(seed)
    t = np.zeros(n, scenes.TRIANGLE_DTYPE)
    for k in ("a", "b", "c"):
        t[k] = rng.uniform(-10, 10, (n, 3)).astype(np.float32)
    t["albedo"] = rng.uniform(0, 1, (n, 3)).astype(np.float32)
    t["roughness"] = np.float32(0.25)
    return wire.render_info_to_json(None, t, wire.RenderMeta(1080, 1920, 20, ID), 3).encode()


def same(a, b):
    return all(x.tobytes() == y.tobytes() for x, y in ((a.world.spheres, b.world.spheres),
                                                       (a.world.triangles, b.world.triangles),
                                                       (a.world.world_index, b.world.world_index)))


class Sink:
    """A local /result endpoint that reads every body."""

    def __init__(self):
        self.n = 0

        class H(BaseHTTPRequestHandler):
            def do_POST(h):  # noqa: N802
                h.rfile.read(int(h.headers["Content-Length"]))
                h.send_response(200)
                h.send_header("Content-Length", "2")
                h.end_headers()
                h.wfile.write(b"ok")

            def log_message(h, *a):
                pass

        self.srv = ThreadingHTTPServer(("127.0.0.1", 0), H)
        threading.Thread(target=self.srv.serve_forever, daemon=True).start()
        self.url = f"http://127.0.0.1:{self.srv.server_address[1]}/result"


def kernel_ms(fn):
    """Device time of the wire_* kernels of one call of fn (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile

    try:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
        ev = [e for e in prof.events() if "wire_" in e.name or "jpeg_carry" in e.name]
        return sum(e.device_time_total for e in ev) / 1e3, sorted({e.name for e in ev})
    except Exception as e:  # the host-clock numbers stand without it
        return None, [f"profiler failed: {e}"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--triangles", type=int, default=262144)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_wire_c2.json"))
    a = ap.parse_args()
    import torch  # noqa: F401  (the profiler; imported before the timed loops so its start-up is not timed)

    facts = gpu_facts()
    body = triangle_body(a.triangles)
    wk = slave.Worker(0)
    rep = {"gpus": facts, "body_bytes": len(body), "triangles": a.triangles}
    try:
        # ---- parse -------------------------------------------------------------------------------------------
        ref = wire.parse_render_info(body)
        for _ in range(2):
            assert same(wk.parse(body), ref)
        host, dev = [], []
        for r in range(max(a.reps, a.host_reps)):
            if r < a.host_reps:
                t0 = time.perf_counter()
                h = wire.parse_render_info(body)
                host.append((time.perf_counter() - t0) * 1e3)
                assert same(h, ref)
            t0 = time.perf_counter()
            d = wk.parse(body)
            dev.append((time.perf_counter() - t0) * 1e3)
            assert same(d, ref)
        rep["parse"] = {"host_ms": statistics.median(host), "device_path_ms": statistics.median(dev),
                        "host_ms_all": host, "device_path_ms_all": dev}
        m = wire._WORLD_FIRST.match(body)
        rep["parse"]["kernel_ms"], rep["parse"]["kernels"] = kernel_ms(lambda: wk.ctx.parse_world_json(body, m.end()))

        # ---- a 20-division C2 job posted to a sink ----------------------------------------------------------
        c = scenes.CONFIGS["C2"]
        sp, tr = scenes.config_scene("C2")
        meta = wire.RenderMeta(c["height"], c["width"], 20, ID)
        infos = [wire.RenderInfo(wire.World(sp, tr, np.arange(len(sp) + len(tr), dtype=np.uint32)), meta, d)
                 for d in range(20)]
        wj = slave.Worker(0, spp=c["spp"], max_bounces=c["max_bounces"])
        sink = Sink()

        def host_job():
            return [sl.to_json().encode() for sl in wj.render_many(infos)]

        def device_job():
            return wj.render_many_json(infos)

        want = host_job()
        assert device_job() == want
        times = {"host": [], "device": []}
        for _ in range(a.reps):
            for mode, fn in (("host", host_job), ("device", device_job)):
                t0 = time.perf_counter()
                bodies = fn()
                for b in bodies:
                    slave._post(sink.url, b)
                times[mode].append((time.perf_counter() - t0) * 1e3)
                assert bodies == want
        rep["job_c2_20_divisions"] = {"spp": c["spp"], "max_bounces": c["max_bounces"], "body_bytes": sum(map(len, want)),
                                      "host_ms": statistics.median(times["host"]),
                                      "device_path_ms": statistics.median(times["device"]),
                                      "host_ms_all": times["host"], "device_path_ms_all": times["device"]}
        p = rt.make_params(c["width"], c["height"], divisions=20, spp=c["spp"], max_bounces=c["max_bounces"])
        sc = wj._scene_for(infos[0])
        rep["job_c2_20_divisions"]["writer_kernel_ms"], _ = kernel_ms(
            lambda: wj.ctx.render_divisions_json(sc, p, list(range(20)), ID))
        sink.srv.shutdown()
        wj.close()
    finally:
        wk.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rep, f, indent=2)
    print(json.dumps({k: v for k, v in rep.items() if k != "gpus"} | {"gpus": facts}, default=str)[:2000])


if __name__ == "__main__":
    main()
