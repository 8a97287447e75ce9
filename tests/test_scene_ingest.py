"""GPU: scene ingest (rt_scene_create) at the boundaries between its stages — split layout, host or device traversal
tree, primitive ids, node records, synchronous or threaded reference tree.  Each scene's frame is compared with the
oracle byte for byte, and the scene's reference ranks with rt_bvh_build_host's for the same world."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import assert_parity

pytestmark = pytest.mark.gpu

W, H, SPP, MB, SEED = 48, 32, 2, 4, 3


def _triangles(n, seed=0):
    """n small triangles around the spheres of synthetic_spheres(n, seed): none of them is big."""
    from rt_b200 import scenes

    sp = scenes.synthetic_spheres(n, seed)
    tr = np.zeros(n, dtype=scenes.TRIANGLE_DTYPE)
    c, r = sp["center"], sp["radius"][:, None]
    tr["a"] = c + r * np.array([1.0, 0.0, 0.0], np.float32)
    tr["b"] = c + r * np.array([0.0, 1.0, 0.0], np.float32)
    tr["c"] = c + r * np.array([0.0, 0.0, 1.0], np.float32)
    tr["albedo"], tr["roughness"], tr["emission"] = sp["albedo"], sp["roughness"], sp["emission"]
    return tr


@pytest.fixture(scope="module", params=[
    "one_sphere", "two_spheres", "plane_only", "plane_and_sphere", "triangles_only", "permuted_world",
    "255_prims", "256_prims",
])
def world(request):
    """(spheres, triangles, world_index) of one boundary scene."""
    from rt_b200 import scenes

    sp, plane, none_t = scenes.synthetic_spheres, scenes.ground_plane(), scenes.no_triangles()
    name = request.param
    if name == "one_sphere":
        return sp(1, 1), none_t, None
    if name == "two_spheres":  # small enough that neither is big: a one-node traversal tree
        s = sp(2, 1)
        s["radius"] *= 0.1
        return s, none_t, None
    if name == "plane_only":  # every primitive is big: no traversal tree
        return scenes.no_spheres(), plane, None
    if name == "plane_and_sphere":  # the traversal tree is a single leaf
        return sp(1, 2), plane, None
    if name == "triangles_only":
        return scenes.no_spheres(), _triangles(40, 3), None
    if name == "permuted_world":
        s, t = sp(60, 4), np.concatenate([_triangles(6, 5), plane])
        return s, t, np.random.default_rng(7).permutation(len(s) + len(t)).astype(np.uint32)
    if name == "255_prims":  # below 256 the reference tree is built inline
        return sp(253, 6), plane, None
    if name == "256_prims":  # from 256 on a builder thread
        return sp(254, 6), plane, None
    raise AssertionError(name)


def test_boundary_scene_matches_oracle(ctx, rt, O, world):
    sp, tr, wi = world
    ref, _ = O.render_frame(sp, tr, W, H, SPP, MB, seed=SEED, world_index=wi)
    sc = ctx.scene(sp, tr, wi)
    try:
        for isect in (1, 2):  # RT_INTERSECT_BRUTE, RT_INTERSECT_BVH
            img = ctx.render_frame(sc, rt.make_params(W, H, spp=SPP, max_bounces=MB, seed=SEED, intersector=isect))
            assert_parity(img, ref)
        info = sc.info()
    finally:
        sc.close()
    rank, n_nodes, depth = rt.api.bvh_build_host(sp, tr, wi)
    assert np.array_equal(info["rank"], rank)
    assert (info["n_prims"], info["n_nodes"], info["depth"]) == (len(sp) + len(tr), n_nodes, depth)


def test_device_tree_threshold_matches_oracle(rt, O):
    """8191 and 8192 spheres under RT_B200_BUILD=auto: the last host-built and the first device-built traversal tree."""
    code = (
        "import sys, hashlib; sys.path.insert(0, 'ray-tracer-s8_b200'); import rt_b200 as rt; from rt_b200 import scenes;"
        "ctx = rt.Context(0)\n"
        "for n in (8191, 8192):\n"
        "    sc = ctx.scene(scenes.synthetic_spheres(n, 8))\n"
        f"    img = ctx.render_frame(sc, rt.make_params({W}, {H}, spp={SPP}, max_bounces={MB}, seed={SEED}, intersector=2))\n"
        "    info = sc.info(); sc.close()\n"
        "    print(hashlib.sha256(img.tobytes()).hexdigest(), hashlib.sha256(info['rank'].tobytes()).hexdigest())"
    )
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    env = dict(os.environ, RT_B200_BUILD="auto")
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    lines = out.stdout.strip().splitlines()[-2:]
    assert len(lines) == 2, out.stdout
    for n, line in zip((8191, 8192), lines):
        sp = rt.scenes.synthetic_spheres(n, 8)
        ref, _ = O.render_frame(sp, None, W, H, SPP, MB, seed=SEED)
        rank = rt.api.bvh_build_host(sp, None)[0]
        assert line.split() == [hashlib.sha256(ref.tobytes()).hexdigest(), hashlib.sha256(rank.tobytes()).hexdigest()], n
