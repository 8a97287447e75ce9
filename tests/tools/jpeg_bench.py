"""JPEG of a rendered frame: PIL on the host against the device encoder, at 1080p (C2, the controller's default size) and
at 4K (C3).  Modes, alternated within every round:
  * pil                  PIL save(format="JPEG", quality=90) of the rendered frame (host RGB in)
  * jpeg_encode          rt_jpeg_encode of the same frame (host RGB in: upload, encode, download)
  * render_pil           rt_render_frame + PIL
  * render_jpeg_1        rt_render_frame_jpeg on one GPU
  * render_jpeg_all      rt_render_frame_jpeg on every GPU of the box (only when there are several)
host_ms is a host clock around the call, which returns when the bytes are in host memory; encode_ms is the device time of
rt_jpeg_encode's kernels (CUDA events).  Medians over the rounds.  Every round asserts that every mode's bytes are PIL's.
The card's name and power limit are read in the same run.  Writes one JSON report per config
(default profiles/r6_jpeg_c2.json and profiles/r6_jpeg_c3.json).

    python tests/tools/jpeg_bench.py [--reps 10] [--warmup 2] [--configs C2,C3] [--out-dir DIR]
"""
import argparse
import io
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


def gpu_facts():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return [dict(zip(("index", "name", "power_limit", "sm_clock_max"), [x.strip() for x in line.split(",")]))
                for line in out.splitlines()]
    except Exception as e:  # the numbers stay valid; the report says the facts could not be read
        return [{"nvidia_smi_error": str(e)}]


def pil_jpeg(frame, quality=90):
    from PIL import Image

    buf = io.BytesIO()
    Image.fromarray(frame, "RGB").save(buf, format="JPEG", quality=quality)
    return buf.getvalue()


def run_config(name, reps, warmup, n_gpus):
    import torch

    cfg = rt.scenes.CONFIGS[name]
    sp, tr = rt.scenes.config_scene(name)
    ctxs = [rt.Context(d) for d in range(n_gpus)]
    try:
        scenes = [c.scene(sp, tr) for c in ctxs]
        p = rt.make_params(cfg["width"], cfg["height"], spp=cfg["spp"], max_bounces=cfg["max_bounces"])
        c0, s0 = ctxs[0], scenes[0]
        frame = c0.render_frame(s0, p)
        want = pil_jpeg(frame)
        modes = {
            "pil": lambda: pil_jpeg(frame),
            "jpeg_encode": lambda: c0.encode_jpeg(frame, 90, want_ms=True),
            "render_pil": lambda: pil_jpeg(c0.render_frame(s0, p)),
            "render_jpeg_1": lambda: c0.render_frame_jpeg(s0, p, 90),
        }
        if n_gpus > 1:
            modes["render_jpeg_all"] = lambda: rt.render_frame_jpeg(ctxs, scenes, p, 90)
        times = {m: [] for m in modes}
        enc_ms = []
        for r in range(warmup + reps):
            for m, fn in modes.items():
                t = time.perf_counter()
                out = fn()
                dt = (time.perf_counter() - t) * 1e3
                if m == "jpeg_encode":
                    out, ms = out
                    if r >= warmup:
                        enc_ms.append(ms)
                assert out == want, (name, m, r)
                if r >= warmup:
                    times[m].append(dt)
        for s in scenes:
            s.close()
        return {
            "config": name, "width": cfg["width"], "height": cfg["height"], "spp": cfg["spp"], "gpus": n_gpus,
            "jpeg_bytes": len(want), "rounds": reps, "warmup": warmup, "bytes_identical_every_round": True,
            "host_ms_median": {m: statistics.median(v) for m, v in times.items()},
            "host_ms_all": times,
            "encode_device_ms_median": statistics.median(enc_ms), "encode_device_ms_all": enc_ms,
            "device": torch.cuda.get_device_name(0), "gpu_facts": gpu_facts(),
        }
    finally:
        for c in ctxs:
            c.close()


def main():
    import torch

    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--configs", default="C2,C3")
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    a = ap.parse_args()
    n_gpus = torch.cuda.device_count()
    if n_gpus == 0:
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    os.makedirs(a.out_dir, exist_ok=True)
    for name in a.configs.split(","):
        rep = run_config(name, a.reps, a.warmup, n_gpus)
        path = os.path.join(a.out_dir, f"r6_jpeg_{name.lower()}.json")
        with open(path, "w") as f:
            json.dump(rep, f, indent=1)
        print(json.dumps({k: rep[k] for k in ("config", "gpus", "jpeg_bytes", "host_ms_median", "encode_device_ms_median",
                                              "gpu_facts")}))


if __name__ == "__main__":
    main()
