"""Dev tool (GPU box): kernel timings per workload + quick parity against the oracle.
usage: python tests/tools/kbench.py [C2 C3 ...]"""
import os, sys, time
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "ray-tracer-s8_b200"))
import numpy as np
import rt_b200 as rt
from rt_b200 import scenes
from oracle import oracle as O


def main():
    names = sys.argv[1:] or ["C2", "C3"]
    ctx = rt.Context(0)
    # parity on crops
    for name, w, h, spp, mb, n, plane in [("p1", 480, 270, 4, 5, 1024, True), ("p2", 320, 240, 2, 10, 64, False),
                                          ("p3", 101, 67, 3, 4, 32, True), ("p4", 64, 48, 2, 5, 1, False)]:
        sp = scenes.synthetic_spheres(n, 3); tr = scenes.ground_plane() if plane else None
        ref, ost = O.render_frame(sp, tr, w, h, spp, mb, want_stats=True)
        sc = ctx.scene(sp, tr).wait_ready()
        img, st = ctx.render_frame(sc, rt.make_params(w, h, spp=spp, max_bounces=mb, intersector=2), want_stats=True)
        sc.close()
        print(name, "ndiff", int((img != ref).sum()), "rays", st["rays"], ost["rays"])
    for name in names:
        cfg = scenes.CONFIGS[name]
        sp, tr = scenes.config_scene(name)
        sc = ctx.scene(sp, tr).wait_ready()
        for isect in (1, 2):
            if isect == 1 and cfg["n_spheres"] > 300:
                continue
            p = rt.make_params(cfg["width"], cfg["height"], spp=cfg["spp"], max_bounces=cfg["max_bounces"], intersector=isect)
            ms = []
            for _ in range(5):
                img, st = ctx.render_frame(sc, p, want_stats=True)
                ms.append(st["kernel_ms"])
            pc = rt.make_params(cfg["width"], cfg["height"], spp=cfg["spp"], max_bounces=cfg["max_bounces"], intersector=isect, collect_counters=True)
            _, cst = ctx.render_frame(sc, pc, want_stats=True)
            k = min(ms)
            print(f"{name} isect={isect} kernel_ms best={k:.3f} med={np.median(ms):.3f} rays={st['rays']} Mrays/s={st['rays']/k/1e3:.0f} "
                  f"phase_eff={cst['active_lane_iters']/max(1,cst['total_lane_iters']):.3f} slab/ray={cst['slab_tests']/st['rays']:.1f} "
                  f"ctas/sm={st['ctas_per_sm']} grid={st['grid_ctas']} smem={st['dyn_smem_bytes']}")
        sc.close()


if __name__ == "__main__":
    main()
