"""GPU: the CUDA path through the C ABI against the oracle on the same seeded inputs.

Bar (BASELINE.json north_star): every 8-bit channel within +-1 LSB on >= 99.9 % of pixels and PSNR >= 50 dB.
This implementation is built to be bit-exact (exact-arithmetic domain in csrc/rt_device.cuh), so the tests
additionally assert zero differing bytes wherever the oracle's BVH and brute force agree.
"""
import json
import threading
import urllib.error
import urllib.request
from http.server import BaseHTTPRequestHandler, HTTPServer

import numpy as np
import pytest

from conftest import assert_parity, frame_compare

pytestmark = pytest.mark.gpu

BOTH = [1, 2]  # RT_INTERSECT_BRUTE, RT_INTERSECT_BVH


def _render(ctx, rt, sp, tr, w, h, spp, mb, isect=0, seed=0, wi=None, **cam):
    sc = ctx.scene(sp, tr, wi)
    try:
        # counters are compared with the oracle's below: have the tie-break tables first, so that no pixel is traced a
        # second time (test_render_before_tables_land covers the path without this wait)
        sc.wait_ready()
        p = rt.make_params(w, h, spp=spp, max_bounces=mb, seed=seed, intersector=isect, **cam)
        return ctx.render_frame(sc, p, want_stats=True)
    finally:
        sc.close()


# ---------------------------------------------------------------------------------------------------
# parity against the oracle at sizes the oracle finishes in seconds
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("isect", BOTH)
def test_c1_full_size(ctx, rt, O, isect):
    """BASELINE config 1: 640x480, 1 spp, reference default depth (max_bounces 10), 64 spheres."""
    c = rt.scenes.CONFIGS["C1"]
    sp, tr = rt.scenes.config_scene("C1")
    ref, ost = O.render_frame(sp, tr, c["width"], c["height"], c["spp"], c["max_bounces"], want_stats=True)
    img, st = _render(ctx, rt, sp, tr, c["width"], c["height"], c["spp"], c["max_bounces"], isect)
    assert_parity(img, ref)
    assert st["rays"] == ost["rays"] and st["primary"] == ost["primary"]
    assert st["intersector_used"] == isect and st["kernel_launches"] == 1


@pytest.mark.parametrize("isect", BOTH)
def test_c2_scene_bands(ctx, rt, O, isect):
    """BASELINE config 2 (1920x1080, 1 spp, depth 5, 256 spheres): three of the controller's 20 bands."""
    c = rt.scenes.CONFIGS["C2"]
    sp, tr = rt.scenes.config_scene("C2")
    sc = ctx.scene(sp, tr)
    for d in (0, 9, 19):
        po = O.make_params(c["width"], c["height"], 20, d, c["spp"], c["max_bounces"])
        ref, _ = O.render_rows(sp, tr, po)
        p = rt.make_params(c["width"], c["height"], divisions=20, division_no=d, spp=c["spp"],
                           max_bounces=c["max_bounces"], intersector=isect)
        img = ctx.render_division(sc, p)
        assert img.shape == (54, 1920, 3)
        assert_parity(img, ref)
    sc.close()


def test_c3_scene_crop(ctx, rt, O):
    """BASELINE config 3 scene (1024 spheres + plane, 16 spp, depth 5) on a 4K band (rows 1080..1095)."""
    c = rt.scenes.CONFIGS["C3"]
    sp, tr = rt.scenes.config_scene("C3")
    div = c["height"] // 16
    d = 1080 // 16
    ref, ost = O.render_rows(sp, tr, O.make_params(c["width"], c["height"], div, d, c["spp"], c["max_bounces"]),
                             want_stats=True)
    sc = ctx.scene(sp, tr)
    p = rt.make_params(c["width"], c["height"], divisions=div, division_no=d, spp=c["spp"],
                       max_bounces=c["max_bounces"])
    img, st = ctx.render_division(sc, p, want_stats=True)
    sc.close()
    assert_parity(img, ref)
    assert st["rays"] == ost["rays"]


@pytest.mark.parametrize("isect", BOTH)
@pytest.mark.parametrize("case", [
    dict(n=1, plane=False, w=128, h=96, spp=2, mb=5),        # root of the BVH is a leaf
    dict(n=2, plane=False, w=64, h=64, spp=3, mb=1),
    dict(n=0, plane=True, w=128, h=96, spp=2, mb=5),         # triangles only
    dict(n=32, plane=True, w=101, h=67, spp=3, mb=4),        # ragged size: partial tiles, unaligned rows
    dict(n=300, plane=True, w=7, h=5, spp=5, mb=6),          # frame smaller than one tile
    dict(n=150, plane=False, w=256, h=8, spp=1, mb=12),
    dict(n=96, plane=True, w=64, h=64, spp=2, mb=62),        # deepest path this build supports
    dict(n=9, plane=False, w=96, h=64, spp=2, mb=5),         # packed sphere pairs: one full group + one sphere
    dict(n=23, plane=True, w=96, h=64, spp=2, mb=5),         # ... a 16-group whose second half is partial, odd count
])
def test_edge_cases(ctx, rt, O, isect, case):
    sp = rt.scenes.synthetic_spheres(case["n"], 17) if case["n"] else None
    tr = rt.scenes.ground_plane() if case["plane"] else None
    ref, ost = O.render_frame(sp, tr, case["w"], case["h"], case["spp"], case["mb"], seed=5, want_stats=True)
    img, st = _render(ctx, rt, sp, tr, case["w"], case["h"], case["spp"], case["mb"], isect, seed=5)
    assert_parity(img, ref)
    assert st["rays"] == ost["rays"]


@pytest.mark.parametrize("isect", BOTH)
def test_mixed_world_order_and_mesh(ctx, rt, O, isect):
    """Spheres and triangles interleaved in the world, plus a small closed mesh (shared edges)."""
    sc = rt.scenes
    sp = sc.synthetic_spheres(40, 21)
    # an octahedron around (0,0,-6): 8 triangles sharing edges and vertices
    v = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], dtype=np.float32) * 1.5
    v += np.array([0, 0, -6], dtype=np.float32)
    faces = [(0, 2, 4), (2, 1, 4), (1, 3, 4), (3, 0, 4), (2, 0, 5), (1, 2, 5), (3, 1, 5), (0, 3, 5)]
    tr = np.zeros(len(faces) + 2, dtype=sc.TRIANGLE_DTYPE)
    for i, (a, b, c) in enumerate(faces):
        tr[i] = (v[a], v[b], v[c], (0.8, 0.6, 0.3), 0.3 * (i % 3), 0.0)
    tr[len(faces):] = sc.ground_plane()
    wi = np.random.default_rng(3).permutation(len(sp) + len(tr)).astype(np.uint32)
    ref, ost = O.render_frame(sp, tr, 160, 120, 4, 6, seed=9, world_index=wi, want_stats=True)
    img, st = _render(ctx, rt, sp, tr, 160, 120, 4, 6, isect, seed=9, wi=wi)
    assert_parity(img, ref)
    assert st["rays"] == ost["rays"]


def test_large_scene_l2_resident_path(ctx, rt, O):
    """6000 spheres + plane: geometry and BVH (430 KB) no longer fit shared memory → the L1/L2-resident kernel variant."""
    sp, tr = rt.scenes.synthetic_spheres(6000, 12), rt.scenes.ground_plane()
    ref, ost = O.render_frame(sp, tr, 200, 120, 2, 5, seed=3, want_stats=True)
    sc = ctx.scene(sp, tr)
    img, st = ctx.render_frame(sc, rt.make_params(200, 120, spp=2, max_bounces=5, seed=3), want_stats=True)
    sc.close()
    assert st["scene_in_smem"] == 0 and st["intersector_used"] == 2
    assert_parity(img, ref)
    assert st["rays"] == ost["rays"]


def test_bvh_300_spheres_matches_oracle(ctx, rt, O):
    """300 spheres + plane with the BVH intersector, rendered straight after the upload: the product library's frame is
    the oracle's, byte for byte."""
    sp, tr = rt.scenes.synthetic_spheres(300, 5), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr)
    img = ctx.render_frame(sc, rt.make_params(160, 96, spp=3, max_bounces=5, seed=4, intersector=2))
    sc.close()
    ref, _ = O.render_frame(sp, tr, 160, 96, 3, 5, seed=4)
    assert np.array_equal(img, ref)


def test_device_built_tree_agrees(rt, O):
    """SURVEY 8f row f3: the traversal tree built on the GPU (Morton LBVH + refit, RT_B200_BUILD=device) culls
    conservatively like the host's SAH tree, so the frame is the same bytes — spheres + plane (split layout) and a
    scene large enough for the automatic switch (>= 8192 primitives)."""
    import hashlib
    import os
    import subprocess
    import sys

    code = (
        "import sys, hashlib; sys.path.insert(0, 'ray-tracer-s8_b200'); import rt_b200 as rt; from rt_b200 import scenes;"
        "ctx = rt.Context(0); out = [];\n"
        "for n, plane in ((300, True), (9000, False)):\n"
        "    sc = ctx.scene(scenes.synthetic_spheres(n, 5), scenes.ground_plane() if plane else None)\n"
        "    img = ctx.render_frame(sc, rt.make_params(160, 96, spp=2, max_bounces=5, seed=4, intersector=2))\n"
        "    out.append(hashlib.sha256(img.tobytes()).hexdigest()); sc.close()\n"
        "print(' '.join(out))"
    )
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    digests = {}
    for mode in ("host", "device", "auto"):
        env = dict(os.environ, RT_B200_BUILD=mode)
        out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, (mode, out.stderr[-500:])
        digests[mode] = out.stdout.strip().splitlines()[-1]
    assert len(set(digests.values())) == 1, digests
    ref, _ = O.render_frame(rt.scenes.synthetic_spheres(300, 5), rt.scenes.ground_plane(), 160, 96, 2, 5, seed=4)
    assert hashlib.sha256(ref.tobytes()).hexdigest() == digests["device"].split()[0]
    ref2, _ = O.render_frame(rt.scenes.synthetic_spheres(9000, 5), None, 160, 96, 2, 5, seed=4)
    assert hashlib.sha256(ref2.tobytes()).hexdigest() == digests["device"].split()[1]


def test_camera_parameters_and_seeds(ctx, rt, O):
    sp, tr = rt.scenes.synthetic_spheres(64, 2), rt.scenes.ground_plane()
    cam = dict(cam_origin=(0.5, 0.25, 1.0), aperture=0.02, focus_distance=6.0, field_of_view=1.0, focal_length=1.5)
    for seed in (0, 1, 2**63 + 12345, 2**64 - 1):
        ref, _ = O.render_frame(sp, tr, 96, 64, 3, 4, seed=seed, **cam)
        img, _ = _render(ctx, rt, sp, tr, 96, 64, 3, 4, 0, seed=seed, **cam)
        assert_parity(img, ref)


def test_reference_defaults(ctx, rt, O):
    """Zero params = the reference's literals: 100 spp, max_bounces 10, aperture 0.1, fov PI/2 (main.rs:39-51)."""
    sp = rt.scenes.synthetic_spheres(16, 4)
    ref, ost = O.render_frame(sp, None, 32, 24, 0, 0, want_stats=True)
    img, st = _render(ctx, rt, sp, None, 32, 24, 0, 0)
    assert_parity(img, ref)
    assert st["primary"] == 32 * 24 * 100 and st["rays"] == ost["rays"]


@pytest.mark.parametrize("isect", BOTH)
def test_golden_frames(ctx, rt, isect):
    import golden.make_golden as G

    for name, case in G.CASES.items():
        sp, tr = G.scene_of(rt.scenes, case)
        img, _ = _render(ctx, rt, sp, tr, case["w"], case["h"], case["spp"], case["mb"], isect, seed=case["seed"])
        assert_parity(img, G.load(name))


def test_counters_match_oracle(ctx, rt, O):
    """The instrumented kernel's path-level counters equal the oracle's for the same seed."""
    sp, tr = rt.scenes.synthetic_spheres(128, 8), rt.scenes.ground_plane()
    _, ost = O.render_frame(sp, tr, 128, 72, 4, 5, want_stats=True)
    sc = ctx.scene(sp, tr)
    for isect in BOTH:
        p = rt.make_params(128, 72, spp=4, max_bounces=5, intersector=isect, collect_counters=True)
        img, st = ctx.render_frame(sc, p, want_stats=True)
        p.collect_counters = 0
        img2, st2 = ctx.render_frame(sc, p, want_stats=True)
        assert np.array_equal(img, img2) and st["rays"] == st2["rays"] == ost["rays"]
        assert st["shades_sphere"] == ost["shades_sphere"] and st["shades_tri"] == ost["shades_tri"]
        assert st["emissive"] == ost["emissive"] and st["sky"] == ost["sky"]
        assert st["active_lane_iters"] == st["rays"] and st["total_lane_iters"] >= st["rays"]
        if isect == 1:
            assert st["sphere_tests"] == st["rays"] * 128 and st["tri_tests"] == st["rays"] * 2
        else:
            assert 0 < st["slab_tests"] and st["sphere_tests"] < st["rays"] * 128
    _, ob = O.render_frame(sp, tr, 128, 72, 4, 5, mode=1, want_stats=True)
    p = rt.make_params(128, 72, spp=4, max_bounces=5, intersector=1, collect_counters=True)
    _, st = ctx.render_frame(sc, p, want_stats=True)
    assert st["tri_tests"] == ob["tri_tests"] and st["sphere_tests"] == ob["sphere_tests"]
    assert st["tri_stage"] == [ob["tri_tests"] - ob["tri_exit"][0], ob["tri_tests"] - ob["tri_exit"][0] - ob["tri_exit"][1],
                               ob["tri_exit"][3]]
    assert st["sphere_hits"] == ob["sphere_hits"] and st["tri_hits"] == ob["tri_hits"]
    sc.close()


def test_c4_crop(ctx, rt, O):
    """BASELINE config 4 (7680x4320, 4 spp, max_bounces 8, 1024 spheres + plane): one 10-row band of the 432 the tile
    scheduler's configuration cuts the frame into, at the height where spheres, plane and sky meet."""
    c = rt.scenes.CONFIGS["C4"]
    sp, tr = rt.scenes.config_scene("C4")
    div, d = c["height"] // 10, 2400 // 10
    ref, ost = O.render_rows(sp, tr, O.make_params(c["width"], c["height"], div, d, c["spp"], c["max_bounces"]),
                             want_stats=True)
    sc = ctx.scene(sp, tr).wait_ready()
    p = rt.make_params(c["width"], c["height"], divisions=div, division_no=d, spp=c["spp"], max_bounces=c["max_bounces"])
    img, st = ctx.render_division(sc, p, want_stats=True)
    sc.close()
    assert img.shape == (10, 7680, 3)
    assert_parity(img, ref)
    assert st["rays"] == ost["rays"]


def test_c5_65536_spheres_band(ctx, rt, O):
    """BASELINE config 5's upper end: 65,536 spheres at 1080p, 1 spp, max_bounces 5 — scene read through L1/L2,
    traversal tree built on the device, reference tree built beside the upload.  One of the controller's 20 bands."""
    sp = rt.scenes.synthetic_spheres(65536)
    ref, ost = O.render_rows(sp, None, O.make_params(1920, 1080, 20, 10, 1, 5), want_stats=True)
    sc = ctx.scene(sp, None)
    p = rt.make_params(1920, 1080, divisions=20, division_no=10, spp=1, max_bounces=5)
    img, st = ctx.render_division(sc, p, want_stats=True)          # straight after the upload: tables may still be on their way
    assert_parity(img, ref)
    assert st["scene_in_smem"] == 0 and st["intersector_used"] == 2
    sc.wait_ready()
    img2, st2 = ctx.render_division(sc, p, want_stats=True)
    sc.close()
    assert np.array_equal(img, img2) and st2["rays"] == ost["rays"] and st2["redo_pixels"] == 0


AXIS_CASES = [
    # camera origin: on box planes of several spheres at once / strictly inside boxes / outside everything in x
    (0.5, 0.25, 3.0), (0.5, 1.0, 3.0), (0.0, 0.25, 3.0), (0.75, 0.3, 3.0), (-3.0, 0.25, 3.0),
]


@pytest.mark.parametrize("isect", BOTH)
@pytest.mark.parametrize("org", AXIS_CASES)
def test_axis_aligned_rays_nan_slabs(ctx, rt, O, isect, org):
    """Ray::intersects_aabb with a zero direction component (ray.rs:133-143,174-194 and the crate's min/max, ray.rs:82-112):
    1/0 = inf and 0*inf = NaN planes.  A denormal field of view and aperture make EVERY primary ray exactly
    (+0, +0, -1) from the camera origin, which sits on the min/max planes of several spheres' (and their ancestors')
    boxes; a mirror wall sends the rays back as (0, 0, +1).  The reference's traversal drops or keeps subtrees by NaN
    propagation order; the GPU path has to reproduce it (exact test on the shape's box + the ancestor chain of the
    reference tree for such rays)."""
    sc_ = rt.scenes
    sp = np.zeros(12, dtype=sc_.SPHERE_DTYPE)
    centers = [(1.5, 0.25, -4.0), (-0.5, 0.25, -6.0), (0.5, 1.25, -8.0), (0.5, -0.75, -2.0), (1.0, 0.75, -5.0),
               (0.5, 0.25, -9.0), (2.5, 0.25, -3.0), (0.25, 0.0, -7.0), (-1.5, 1.25, -4.5), (0.75, 0.5, -1.0),
               (0.5, 0.25, -12.0), (3.0, 3.0, -6.0)]
    radii = [1.0, 1.0, 1.0, 1.0, 0.5, 0.25, 2.0, 0.25, 1.0, 0.25, 0.5, 1.0]
    for i, (c, r) in enumerate(zip(centers, radii)):
        sp[i] = (c, r, (0.9, 0.6 + 0.03 * i, 0.3), [0.0, 1.0, 0.5][i % 3], 2.0 if i == 11 else 0.0)
    tr = np.zeros(2, dtype=sc_.TRIANGLE_DTYPE)   # mirror wall at z = -14 facing the camera
    tr[0] = ((-20, -20, -14), (20, -20, -14), (20, 20, -14), (0.9, 0.9, 0.9), 1.0, 0.0)
    tr[1] = ((-20, -20, -14), (20, 20, -14), (-20, 20, -14), (0.9, 0.9, 0.9), 1.0, 0.0)
    cam = dict(cam_origin=org, aperture=1e-40, field_of_view=1e-40, focus_distance=1.0)
    ref, ost = O.render_frame(sp, tr, 16, 8, 6, 6, seed=3, want_stats=True, **cam)
    img, st = _render(ctx, rt, sp, tr, 16, 8, 6, 6, isect, seed=3, **cam)
    assert_parity(img, ref)
    assert st["rays"] == ost["rays"]
    # and with the tables still on their way: every pixel depends on them, the second pass has to put it right
    sc = ctx.scene(sp, tr)
    img2 = ctx.render_frame(sc, rt.make_params(16, 8, spp=6, max_bounces=6, seed=3, intersector=isect, **cam))
    sc.close()
    assert np.array_equal(img2, ref)


def _tie_mesh(rt, n_quads=160):
    """Every triangle twice: each hit is an exact-distance tie that only the reference tree's leaf order decides
    (shapes/mod.rs:177-182); the two copies differ in colour, so a wrong winner shows."""
    rng = np.random.default_rng(5)
    tr = np.zeros(4 * n_quads, dtype=rt.scenes.TRIANGLE_DTYPE)
    for q in range(n_quads):
        c = np.array([rng.uniform(-6, 6), rng.uniform(-3.5, 3.5), rng.uniform(-14, -5)], dtype=np.float32)
        e1 = rng.normal(size=3).astype(np.float32) * 0.9
        e2 = rng.normal(size=3).astype(np.float32) * 0.9
        if q == 0:  # a wall behind everything that fills the view: no pixel without a tie
            c = np.array([-60, -40, -20], dtype=np.float32)
            e1, e2 = np.array([120, 0, 0], dtype=np.float32), np.array([0, 80, 0], dtype=np.float32)
        a, b, cc, dd = c, c + e1, c + e1 + e2, c + e2
        for k, (p0, p1, p2) in enumerate(((a, b, cc), (a, cc, dd))):
            tr[4 * q + 2 * k] = (p0, p1, p2, (0.9, 0.2, 0.2), 0.3, 0.0)
            tr[4 * q + 2 * k + 1] = (p0, p1, p2, (0.2, 0.2, 0.9), 0.3, 0.0)
    return tr


def test_render_before_tables_land(rt, O):
    """rt_scene_create returns before the reference-topology tree is built (its tables only break exact-distance ties).
    RT_B200_AUX_DELAY_MS holds the builder thread back, so the first frame is rendered without the tables for certain:
    the kernel must mark every tie pixel and the second pass must reproduce the oracle's frame — with a pixel list
    (few ties) and by repeating the launch (more tie pixels than the list holds)."""
    import os
    import subprocess
    import sys
    import hashlib

    code = (
        "import sys, hashlib, numpy as np; sys.path.insert(0, 'ray-tracer-s8_b200'); sys.path.insert(0, 'tests');"
        "import rt_b200 as rt; from test_gpu_parity import _tie_mesh;"
        "ctx = rt.Context(0); tr = _tie_mesh(rt); out = [];\n"
        "for (w, h) in ((96, 64), (512, 320)):\n"
        "    sc = ctx.scene(None, tr)\n"
        "    img, st = ctx.render_frame(sc, rt.make_params(w, h, spp=2, max_bounces=3, seed=7), want_stats=True)\n"
        "    out.append(hashlib.sha256(img.tobytes()).hexdigest() + ':' + str(st['redo_pixels'])); sc.close()\n"
        "print(' '.join(out))"
    )
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    env = dict(os.environ, RT_B200_AUX_DELAY_MS="300")
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-800:]
    got = out.stdout.strip().splitlines()[-1].split()
    tr = _tie_mesh(rt)
    for (w, h), g in zip(((96, 64), (512, 320)), got):
        ref, _ = O.render_frame(None, tr, w, h, 2, 3, seed=7)
        digest, redo = g.split(":")
        assert digest == hashlib.sha256(ref.tobytes()).hexdigest(), (w, h, redo)
        assert int(redo) > 0, "the first pass must have met ties without the tables"
    assert int(got[0].split(":")[1]) < 65536 and int(got[1].split(":")[1]) == 0xffffffff


def test_blocking_launches_do_not_deadlock(rt):
    """With CUDA_LAUNCH_BLOCKING=1 (or under Nsight Compute) every launch blocks the host.  A streamed frame whose first
    pass held pixels back (tables delayed by RT_B200_AUX_DELAY_MS) used to stop there: the owner sat in a wait for counts
    only its own second pass releases.  The frame must complete, with the same bytes as without blocking launches."""
    import os
    import subprocess
    import sys

    code = (
        "import sys, hashlib, numpy as np; sys.path.insert(0, 'ray-tracer-s8_b200'); sys.path.insert(0, 'tests');"
        "import rt_b200 as rt; from test_gpu_parity import _tie_mesh;"
        "ctx = rt.Context(0); tr = _tie_mesh(rt); sc = ctx.scene(None, tr);"
        # >= 4 MiB and >= 8 spp: the frame streams to the host slab by slab while it renders
        "img, st = ctx.render_frame(sc, rt.make_params(1408, 1024, spp=8, max_bounces=2, seed=3), want_stats=True);"
        "print(hashlib.sha256(img.tobytes()).hexdigest(), st['redo_pixels'])"
    )
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    got = {}
    for blocking in ("0", "1"):
        env = dict(os.environ, RT_B200_AUX_DELAY_MS="200", CUDA_LAUNCH_BLOCKING=blocking)
        out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, (blocking, out.stderr[-800:])
        got[blocking] = out.stdout.strip().splitlines()[-1].split()
    assert got["0"][0] == got["1"][0], got
    assert int(got["0"][1]) > 0 and int(got["1"][1]) > 0, got


def test_owner_times_out_when_a_slab_never_completes(rt):
    """A frame nobody renders into: the owner's collect must give up after the wait limit with RT_ERR_TIMEOUT — by value
    waits (the host satisfies the counters itself so the copy stream drains) and by wait kernels — and leave the
    context usable."""
    import os
    import subprocess
    import sys

    code = (
        "import sys, time, hashlib, numpy as np; sys.path.insert(0, 'ray-tracer-s8_b200');"
        "import rt_b200 as rt; from rt_b200 import scenes, _abi;"
        "ctx = rt.Context(0); p = rt.make_params(256, 192, spp=1, max_bounces=2, seed=1);"
        "dev, handle = ctx.frame_alloc(256 * 192 * 3); t0 = time.time(); status = 0\n"
        "try:\n"
        "    ctx.frame_collect(dev, p, 1, out=np.empty((192, 256, 3), np.uint8))\n"
        "except rt.RtError as e:\n"
        "    status = e.status\n"
        "dt = time.time() - t0\n"
        "sc = ctx.scene(scenes.synthetic_spheres(40, 3), scenes.ground_plane()).wait_ready()\n"
        "a = ctx.render_frame(sc, p); b = ctx.render_frame(sc, p)\n"
        "print(status, round(dt, 2), int((a == b).all()), int(a.max()))"
    )
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    for extra in ({}, {"RT_B200_NO_STREAM_WAIT": "1"}):
        env = dict(os.environ, RT_B200_WAIT_TIMEOUT_MS="400", **extra)
        out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, (extra, out.stderr[-800:])
        status, dt, same, mx = out.stdout.strip().splitlines()[-1].split()
        assert int(status) == -9, (extra, out.stdout)          # RT_ERR_TIMEOUT
        assert 0.3 <= float(dt) < 10.0, (extra, dt)
        assert same == "1" and int(mx) > 0, (extra, out.stdout)


def test_scene_sizes_around_staging_capacity(rt, O):
    """The pinned staging copy of an asynchronously built scene covers the early part of the blob only; its capacity is
    a power of two.  Worlds whose early part just fits a capacity while the late tables do not (13-14 k and 27-28 k
    spheres for 2 and 4 MiB) once had their "tables landed" flag written past the buffer.  Create, render, compare."""
    import hashlib
    import os
    import subprocess
    import sys

    code = (
        "import sys, hashlib; sys.path.insert(0, 'ray-tracer-s8_b200'); import rt_b200 as rt; from rt_b200 import scenes;"
        "ctx = rt.Context(0); out = []\n"
        "for n in (13000, 14000, 27500):\n"
        "    sc = ctx.scene(scenes.synthetic_spheres(n, 2), None)\n"
        "    img = ctx.render_frame(sc, rt.make_params(96, 64, spp=1, max_bounces=3, seed=5))\n"
        "    sc.wait_ready(); out.append(hashlib.sha256(img.tobytes()).hexdigest()); sc.close()\n"
        "print(' '.join(out))"
    )
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=dict(os.environ), capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, (out.returncode, out.stderr[-800:])
    got = out.stdout.strip().splitlines()[-1].split()
    ref, _ = O.render_frame(rt.scenes.synthetic_spheres(14000, 2), None, 96, 64, 1, 3, seed=5)
    assert got[1] == hashlib.sha256(ref.tobytes()).hexdigest()


def test_pinhole_and_zero_bounce_flags(ctx, rt, O):
    """rt_params.flags: aperture 0 = pinhole and max_bounces 0 = camera rays only, instead of the reference's literals."""
    sp, tr = rt.scenes.synthetic_spheres(40, 9), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr).wait_ready()
    a = ctx.render_frame(sc, rt.make_params(96, 64, spp=2, max_bounces=0, aperture=0.0, explicit=("max_bounces", "aperture")))
    b, sb = ctx.render_frame(sc, rt.make_params(96, 64, spp=2, max_bounces=0, aperture=0.0), want_stats=True)   # literals: 10, 0.1
    c, sc_st = ctx.render_frame(sc, rt.make_params(96, 64, spp=2, max_bounces=0, explicit=("max_bounces",)), want_stats=True)
    sc.close()
    assert sc_st["rays"] == 96 * 64 * 2 and sb["rays"] > sc_st["rays"]      # one query per sample
    ref, _ = O.render_frame(sp, tr, 96, 64, 2, 0)
    assert_parity(b, ref)
    assert not np.array_equal(a, c)                                         # pinhole vs aperture 0.1
    # every hit pixel of a camera-rays-only frame is black unless the hit emits: paths end after one query
    assert (c.reshape(-1, 3).max(axis=1) == 0).mean() > 0.05


def test_multi_context_frame_matches_single(ctx, rt, O):
    """rt_render_frame_multi: N contexts (here on one device; see the 2-device test) render interleaved tile shares
    into context 0's frame; the frame equals the single-context frame and the oracle's."""
    from rt_b200 import multi

    sp, tr = rt.scenes.synthetic_spheres(200, 6), rt.scenes.ground_plane()
    ref, ost = O.render_frame(sp, tr, 322, 181, 3, 5, seed=2, want_stats=True)
    p = rt.make_params(322, 181, spp=3, max_bounces=5, seed=2)
    m = multi.MultiDeviceRenderer([0, 0, 0])
    try:
        scenes = [s.wait_ready() for s in m.scenes(sp, tr)]
        img, st = m.render(scenes, p, want_stats=True)
        for s in scenes:
            s.close()
    finally:
        m.close()
    assert_parity(img, ref)
    assert st["rays"] == ost["rays"] and st["primary"] == 322 * 181 * 3 and st["kernel_launches"] == 3


def test_two_devices_p2p_and_nccl(rt, O):
    """Two GPUs: (a) one process, rt_render_frame_multi over peer access; (b) bench.py under torchrun, one process per
    GPU, frame assembled by peer stores (p2p) and by NCCL — all must produce the single-GPU frame (same sha256)."""
    import json
    import os
    import subprocess
    import sys

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from rt_b200 import multi

    c = rt.scenes.CONFIGS["C2"]
    sp, tr = rt.scenes.config_scene("C2")
    p = rt.make_params(c["width"], c["height"], spp=2, max_bounces=c["max_bounces"])
    with rt.Context(0) as c0:
        sc = c0.scene(sp, tr)
        one = c0.render_frame(sc, p)
        sc.close()
    m = multi.MultiDeviceRenderer([0, 1])
    try:
        scenes = m.scenes(sp, tr)
        two, st = m.render(scenes, p, want_stats=True)
        for s in scenes:
            s.close()
    finally:
        m.close()
    assert np.array_equal(one, two)
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    hashes = {}
    for mode, gpus in (("single", 1), ("p2p", 2), ("nccl", 2)):
        cmd = [sys.executable, os.path.join(root, "bench.py"), "--gpus", str(gpus), "--steps", "2", "--warmup", "3",
               "--workload", "C2", "--no-cpu-baseline"] + (["--mode", mode] if gpus > 1 else [])
        out = subprocess.run(cmd, cwd=root, capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, (mode, out.stderr[-800:])
        line = json.loads(out.stdout.strip().splitlines()[-1])
        hashes[mode] = line["frame_sha256"]
        assert line["n_gpus"] == gpus
    assert len(set(hashes.values())) == 1, hashes


# ---------------------------------------------------------------------------------------------------
# size-independent properties at BASELINE's full sizes
# ---------------------------------------------------------------------------------------------------
def test_c2_full_size_properties(ctx, rt):
    """Full 1920x1080: determinism, intersector independence, division partition == whole frame."""
    c = rt.scenes.CONFIGS["C2"]
    sp, tr = rt.scenes.config_scene("C2")
    sc = ctx.scene(sp, tr)
    kw = dict(spp=c["spp"], max_bounces=c["max_bounces"])
    a, sa = ctx.render_frame(sc, rt.make_params(c["width"], c["height"], intersector=2, **kw), want_stats=True)
    b, sb = ctx.render_frame(sc, rt.make_params(c["width"], c["height"], intersector=2, **kw), want_stats=True)
    k1, s1 = ctx.render_frame(sc, rt.make_params(c["width"], c["height"], intersector=1, **kw), want_stats=True)
    assert np.array_equal(a, b) and np.array_equal(a, k1)
    assert sa["rays"] == sb["rays"] == s1["rays"] and sa["primary"] == 1920 * 1080
    bands = [ctx.render_division(sc, rt.make_params(c["width"], c["height"], divisions=20, division_no=d, **kw))
             for d in range(20)]
    assert np.array_equal(np.concatenate(bands, axis=0), a)
    # the sky saturates the u8 cast above the horizon (main.rs:136: t = y*0.5 + 1 > 1)
    assert (a[:400] == 255).mean() > 0.9
    sc.close()


def test_c3_full_size_tile_partition(ctx, rt):
    """Full 3840x2160 (4 spp to bound the time): 3 emulated ranks rendering their tiles into one frame
    reproduce the single-rank frame; ray counts add up."""
    c = rt.scenes.CONFIGS["C3"]
    sp, tr = rt.scenes.config_scene("C3")
    sc = ctx.scene(sp, tr).wait_ready()      # ray counts are compared: no pixel may be traced twice
    p = rt.make_params(c["width"], c["height"], spp=4, max_bounces=c["max_bounces"])
    whole, sw = ctx.render_frame(sc, p, want_stats=True)
    nbytes = c["width"] * c["height"] * 3
    dev, _ = ctx.frame_alloc(nbytes)
    rays = 0
    for r in range(3):
        st = ctx.render_tiles_device(sc, p, r, 3, dev, sync=True, want_stats=True)
        rays += st["rays"]
    out = np.zeros((c["height"], c["width"], 3), dtype=np.uint8)
    ctx.frame_download(dev, out)
    ctx.frame_free(dev)
    sc.close()
    assert np.array_equal(out, whole) and rays == sw["rays"]


# ---------------------------------------------------------------------------------------------------
# boundary behaviour (include/rt_b200.h)
# ---------------------------------------------------------------------------------------------------
def test_error_codes(ctx, rt):
    sp = rt.scenes.synthetic_spheres(4)
    with pytest.raises(rt.RtError) as e:
        ctx.scene(None, None)
    assert e.value.status == -2 and "never terminates" in e.value.message
    sc = ctx.scene(sp, None)
    with pytest.raises(rt.RtError) as e:
        ctx.render_division(sc, rt.make_params(16, 9, divisions=2, spp=1, max_bounces=1))
    assert e.value.status == -1 and "multiple of divisions" in e.value.message
    with pytest.raises(rt.RtError) as e:
        ctx.render_frame(sc, rt.make_params(16, 8, spp=1, max_bounces=1), out=np.zeros((8, 16, 2), dtype=np.uint8))
    assert e.value.status == -1 and "out_len" in e.value.message
    with pytest.raises(rt.RtError) as e:
        ctx.render_frame(sc, rt.make_params(16, 8, spp=1, max_bounces=64))
    assert e.value.status == -6
    with pytest.raises(rt.RtError) as e:
        ctx.render_division(sc, rt.make_params(16, 8, divisions=2, division_no=2, spp=1, max_bounces=1))
    assert e.value.status == -1
    # more primitives than node byte offsets (31 bits / 64-byte records) or primitive ids (26 bits) can address: refused
    # before anything is read
    import ctypes as C
    h = C.c_void_p()
    for count in (2**25 + 1, 2**26 + 5):
        rc = ctx._lib.rt_scene_create(ctx._h, None, count, None, 0, None, C.byref(h))
        assert rc == -6 and b"too many primitives" in ctx._lib.rt_last_error(ctx._h), (count, rc)
    # the context stays usable after errors
    img = ctx.render_frame(sc, rt.make_params(16, 8, spp=1, max_bounces=1))
    assert img.shape == (8, 16, 3)
    sc.close()


def test_pinned_output_buffer(ctx, rt, O):
    sp = rt.scenes.synthetic_spheres(16, 4)
    buf = ctx.pinned_empty((48, 64, 3))
    sc = ctx.scene(sp, None)
    ctx.render_frame(sc, rt.make_params(64, 48, spp=2, max_bounces=3), out=buf)
    sc.close()
    ref, _ = O.render_frame(sp, None, 64, 48, 2, 3)
    assert_parity(buf, ref)


def test_fp32_peak_probe(ctx):
    tf, ms = ctx.measure_fp32_peak()
    assert 30.0 < tf < 90.0 and ms > 0       # nominal 148 SM x 128 lanes x 2 x 1.965 GHz = 74.5 TFLOP/s


# ---------------------------------------------------------------------------------------------------
# the slave's interface on top of the GPU path (ray-tracer-slave/src/main.rs:32-106,148-174)
# ---------------------------------------------------------------------------------------------------
def test_worker_render_info_to_image_slice(rt, O):
    from rt_b200 import slave, wire

    sp, tr = rt.scenes.synthetic_spheres(48, 6), rt.scenes.ground_plane()
    wi = np.random.default_rng(1).permutation(50).astype(np.uint32)
    meta = wire.RenderMeta(60, 80, 5, "123e4567-e89b-12d3-a456-426614174000")
    wk = slave.Worker(0, spp=3, max_bounces=4, seed=2)
    try:
        for d in (0, 3, 4):
            body = wire.render_info_to_json(sp, tr, meta, d, wi)
            sl = wire.ImageSlice.from_json(wk.render_json(body))
            assert sl.division_no == d and sl.id == meta.id and sl.image.size == 12 * 80 * 3
            ref, _ = O.render_rows(sp, tr, O.make_params(80, 60, 5, d, 3, 4, 2), world_index=wi)
            assert_parity(sl.image.reshape(12, 80, 3), ref)
        assert wk.scene_uploads == 1          # one upload + BVH build per job id, not per division
    finally:
        wk.close()


def test_http_shell_end_to_end(rt, O):
    """POST / → ack text → the slave POSTs the ImageSlice to the master's /result (fake master here)."""
    from rt_b200 import slave, wire

    got = {}
    done = threading.Event()

    class Master(BaseHTTPRequestHandler):
        def do_POST(self):  # noqa: N802
            n = int(self.headers["Content-Length"])
            got["path"], got["body"] = self.path, self.rfile.read(n)
            self.send_response(200)
            self.send_header("Content-Length", "2")
            self.end_headers()
            self.wfile.write(b"ok")
            done.set()

        def log_message(self, *a):
            pass

    master = HTTPServer(("127.0.0.1", 0), Master)
    threading.Thread(target=master.serve_forever, daemon=True).start()
    ready, stop = threading.Event(), threading.Event()
    wk = slave.Worker(0, spp=2, max_bounces=3)
    t = threading.Thread(target=slave.serve, kwargs=dict(
        host="127.0.0.1", port=0, result_url=f"http://127.0.0.1:{master.server_address[1]}/result", worker=wk,
        ready=ready, stop=stop), daemon=True)
    t.start()
    assert ready.wait(30)
    sp = rt.scenes.synthetic_spheres(20, 3)
    meta = wire.RenderMeta(32, 48, 4, "00000000-0000-4000-8000-000000000001")
    req = urllib.request.Request(f"http://127.0.0.1:{ready.port}/", data=wire.render_info_to_json(sp, None, meta, 2).encode(),
                                 headers={"Content-Type": "application/json"}, method="POST")
    with urllib.request.urlopen(req, timeout=30) as r:
        assert r.status == 200 and r.read().decode() == slave.ACK_TEXT
    # a malformed body is a 400, like actix's Json extractor
    bad = urllib.request.Request(f"http://127.0.0.1:{ready.port}/", data=b"{}", method="POST")
    with pytest.raises(urllib.error.HTTPError) as he:
        urllib.request.urlopen(bad, timeout=30)
    assert he.value.code == 400
    assert done.wait(60)
    stop.set()
    t.join(30)
    master.shutdown()
    wk.close()
    assert got["path"] == "/result"
    o = json.loads(got["body"])
    assert list(o.keys()) == ["division_no", "image", "id"] and o["division_no"] == 2 and o["id"] == meta.id
    ref, _ = O.render_rows(sp, None, O.make_params(48, 32, 4, 2, 2, 3))
    assert_parity(np.array(o["image"], dtype=np.uint8).reshape(8, 48, 3), ref)


def test_controller_upload_to_jpeg_on_a_mesh(rt, O):
    """f4 + f2: OBJ ++ MTL → /upload → 20 divisions on the GPU worker → /poll → JPEG; the stitched frame must be the
    oracle's frame (compared through the JPEG, and exactly through the worker)."""
    import io

    from PIL import Image

    from rt_b200 import controller, obj, slave, wire
    from test_host import mesh_scene_obj

    data, n = mesh_scene_obj()
    tris = obj.build_world(data, n)
    wk = slave.Worker(0, spp=4, max_bounces=4, seed=11)
    try:
        c = controller.Controller(worker=wk, width=320, height=180, divisions=20)
        job = c.upload(data, n)
        jpeg, is_img = c.poll(job)
        assert is_img
        assert wk.scene_uploads == 1
        ref, _ = O.render_frame(None, tris, 320, 180, 4, 4, seed=11)
        got = np.array(Image.open(io.BytesIO(jpeg)).convert("RGB"))
        mse = float(((got.astype(np.float64) - ref) ** 2).mean())
        assert 10 * np.log10(255.0 ** 2 / mse) > 30.0                       # JPEG(90) of the same frame
        meta = wire.RenderMeta(180, 320, 20, "00000000-0000-4000-8000-00000000000a")
        world = wire.World(np.zeros(0, wire.SPHERE_DTYPE), tris, np.arange(len(tris), dtype=np.uint32))
        bands = [wk.render(wire.RenderInfo(world, meta, d)).image.reshape(9, 320, 3) for d in range(20)]
        assert_parity(np.concatenate(bands, axis=0), ref)
    finally:
        wk.close()


def test_controller_concurrent_uploads_are_serialised(rt, O):
    """Two /upload requests at once against the in-process controller (a ThreadingHTTPServer gives every request its own
    thread): one rt_ctx has ONE owner at a time, so the worker serialises them; both stitched frames must be the oracle's."""
    import io

    from PIL import Image

    from rt_b200 import controller, obj, slave
    from test_host import mesh_scene_obj

    data, n = mesh_scene_obj()
    tris = obj.build_world(data, n)
    wk = slave.Worker(0, spp=3, max_bounces=4, seed=5)
    ready, stop = threading.Event(), threading.Event()
    c = controller.Controller(worker=wk, width=160, height=120, divisions=20)
    t = threading.Thread(target=controller.serve, kwargs=dict(controller=c, host="127.0.0.1", port=0, ready=ready, stop=stop), daemon=True)
    t.start()
    assert ready.wait(30)
    base = f"http://127.0.0.1:{ready.port}"
    jobs, errs = [None, None], []

    def post(i):
        try:
            req = urllib.request.Request(f"{base}/upload/{n}/", data=data, method="POST")
            with urllib.request.urlopen(req, timeout=120) as r:
                jobs[i] = r.read().decode()
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    th = [threading.Thread(target=post, args=(i,)) for i in range(2)]
    for x in th:
        x.start()
    for x in th:
        x.join(180)
    try:
        assert not errs and all(jobs) and jobs[0] != jobs[1], (errs, jobs)
        ref, _ = O.render_frame(None, tris, 160, 120, 3, 4, seed=5)
        for j in jobs:
            req = urllib.request.Request(f"{base}/poll", data=j.encode(), method="POST")
            with urllib.request.urlopen(req, timeout=60) as r:
                assert r.headers["Content-Type"] == "image/jpeg"
                got = np.array(Image.open(io.BytesIO(r.read())).convert("RGB"))
            mse = float(((got.astype(np.float64) - ref) ** 2).mean())
            assert 10 * np.log10(255.0 ** 2 / mse) > 30.0
        assert wk.scene_uploads == 2          # two jobs, one upload each (20 divisions share it)
    finally:
        stop.set()
        t.join(30)
        wk.close()


def test_controller_tile_scheduler_over_devices(rt, O):
    """f2: Controller(devices=[...]) renders the whole frame in one rt_render_frame_multi call over the listed GPUs (all
    of them when there are several, else two contexts on device 0) and cuts it into the job's divisions; /poll
    stitches them back.  The stitched frame is the oracle's (through the JPEG) and the slices are exact."""
    import io

    import torch
    from PIL import Image

    from rt_b200 import controller, obj, wire
    from test_host import mesh_scene_obj

    data, n = mesh_scene_obj()
    tris = obj.build_world(data, n)
    devs = list(range(torch.cuda.device_count())) if torch.cuda.device_count() > 1 else [0, 0]
    c = controller.Controller(devices=devs, width=320, height=180, divisions=20, spp=4, max_bounces=4, seed=11)
    try:
        ref, _ = O.render_frame(None, tris, 320, 180, 4, 4, seed=11)
        meta = wire.RenderMeta(180, 320, 20, "00000000-0000-4000-8000-00000000000b")
        slices = c._render_all_gpus(tris, meta)
        assert [s.division_no for s in slices] == list(range(20))
        assert_parity(np.concatenate([s.image.reshape(9, 320, 3) for s in slices], axis=0), ref)
        job = c.upload(data, n)
        jpeg, is_img = c.poll(job)
        assert is_img
        got = np.array(Image.open(io.BytesIO(jpeg)).convert("RGB"))
        mse = float(((got.astype(np.float64) - ref) ** 2).mean())
        assert 10 * np.log10(255.0 ** 2 / mse) > 30.0
    finally:
        c.close()
