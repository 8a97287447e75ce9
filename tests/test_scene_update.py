"""GPU: rt_scene_update — a scene updated in place to world B renders byte-identically to a scene created from B, and
so to the oracle: moved primitives (traversal tree refitted on the device, reference tables rebuilt), material edits
(boxes unchanged: nothing but the primitive data is uploaded), updates while tables are in flight, progressive accums,
errors that leave the scene as it was, and multi-context frames."""
import ctypes as C
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import assert_parity

pytestmark = pytest.mark.gpu

W, H, SPP, MB, SEED = 48, 32, 2, 4, 3
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _moved(sp, tr, seed, materials=True, scale=0.3):
    """Copies of sp / tr with every primitive moved by a seeded random offset (a triangle's three corners together; the
    two copies of a _tie_mesh triangle, neighbours in the array, by the same offset so their ties stay exact) and, with
    `materials`, new albedo, roughness and emission."""
    rng = np.random.default_rng(seed)
    sp = None if sp is None else sp.copy()
    tr = None if tr is None else tr.copy()
    if sp is not None and len(sp):
        sp["center"] += (rng.uniform(-scale, scale, (len(sp), 3)) * sp["radius"][:, None]).astype(np.float32)
        if materials:
            _new_materials(sp, rng)
    if tr is not None and len(tr):
        off = np.repeat(rng.uniform(-scale, scale, ((len(tr) + 1) // 2, 1, 3)), 2, axis=0)[:len(tr)].astype(np.float32)
        for k in ("a", "b", "c"):
            tr[k] += off[:, 0]
        if materials:
            _new_materials(tr, rng)
    return sp, tr


def _new_materials(a, rng):
    a["albedo"] = rng.uniform(0.05, 0.95, (len(a), 3)).astype(np.float32)
    a["roughness"] = rng.uniform(0.0, 1.0, len(a)).astype(np.float32)
    a["emission"] = np.where(rng.uniform(size=len(a)) < 0.15, rng.uniform(1.0, 4.0, len(a)), 0.0).astype(np.float32)


def _params(rt, isect=2, **kw):
    return rt.make_params(W, H, spp=SPP, max_bounces=MB, seed=SEED, intersector=isect, **kw)


def _run(code, env=None, timeout=600):
    """`code` in a fresh interpreter (the test hooks are read once per process, in rt_init); its last stdout line."""
    head = ("import sys, hashlib, numpy as np; sys.path.insert(0, 'ray-tracer-s8_b200'); sys.path.insert(0, 'tests');"
            "import rt_b200 as rt; from test_scene_update import _moved\n")
    out = subprocess.run([sys.executable, "-c", head + code], cwd=ROOT, env=dict(os.environ, **(env or {})),
                         capture_output=True, text=True, timeout=timeout)
    assert out.returncode == 0, out.stderr[-1500:]
    return out.stdout.strip().splitlines()[-1]


def _sha(img):
    return hashlib.sha256(img.tobytes()).hexdigest()


# ---------------------------------------------------------------------------------------------------
# boundary worlds (those of test_scene_ingest.py): A -> B -> A
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=[
    "one_sphere", "plane_only", "plane_and_sphere", "triangles_only", "permuted_world", "255_prims", "256_prims",
])
def world(request):
    """(spheres, triangles, world_index) of one boundary scene."""
    from rt_b200 import scenes
    from test_scene_ingest import _triangles

    sp, plane, none_t = scenes.synthetic_spheres, scenes.ground_plane(), scenes.no_triangles()
    name = request.param
    if name == "one_sphere":
        return sp(1, 1), none_t, None
    if name == "plane_only":  # every primitive is big: no traversal tree
        return scenes.no_spheres(), plane, None
    if name == "plane_and_sphere":  # the traversal tree is a single leaf
        return sp(1, 2), plane, None
    if name == "triangles_only":
        return scenes.no_spheres(), _triangles(40, 3), None
    if name == "permuted_world":
        s, t = sp(60, 4), np.concatenate([_triangles(6, 5), plane])
        return s, t, np.random.default_rng(7).permutation(len(s) + len(t)).astype(np.uint32)
    if name == "255_prims":  # reference tables built inline
        return sp(253, 6), plane, None
    if name == "256_prims":  # on a builder thread
        return sp(254, 6), plane, None
    raise AssertionError(name)


def _check_world(ctx, rt, O, sc, sp, tr, wi):
    ref, _ = O.render_frame(sp, tr, W, H, SPP, MB, seed=SEED, world_index=wi)
    for isect in (1, 2):  # RT_INTERSECT_BRUTE, RT_INTERSECT_BVH
        assert_parity(ctx.render_frame(sc, _params(rt, isect)), ref)
    info = sc.info()
    rank, n_nodes, depth = rt.api.bvh_build_host(sp, tr, wi)
    assert np.array_equal(info["rank"], rank)
    assert (info["n_prims"], info["n_nodes"], info["depth"]) == (len(sp) + len(tr), n_nodes, depth)


def test_update_boundary_worlds_match_oracle(ctx, rt, O, world):
    sp, tr, wi = world
    sp_b, tr_b = _moved(sp, tr, 11)
    sc = ctx.scene(sp, tr, wi)
    try:
        bytes_a = sc.device_bytes
        assert sc.update(sp_b, tr_b) is sc
        _check_world(ctx, rt, O, sc, sp_b, tr_b, wi)
        sc.update(sp, tr)
        _check_world(ctx, rt, O, sc, sp, tr, wi)
        assert sc.device_bytes == bytes_a
    finally:
        sc.close()


# ---------------------------------------------------------------------------------------------------
# device-built traversal tree: refit_nodes reproduces the LBVH's records
# ---------------------------------------------------------------------------------------------------
def test_update_device_built_tree(rt, O):
    """RT_B200_BUILD=device at 300 and 8192 spheres: A -> B renders the oracle's B; A -> B -> A counts the same slab tests
    as a fresh scene of A (the refit's records are the build's), with the tables landed before both renders."""
    code = (
        "ctx = rt.Context(0); out = []\n"
        "for n in (300, 8192):\n"
        "    a = rt.scenes.synthetic_spheres(n, 8); b, _ = _moved(a, None, 21)\n"
        f"    p = rt.make_params({W}, {H}, spp={SPP}, max_bounces={MB}, seed={SEED}, intersector=2)\n"
        f"    pc = rt.make_params({W}, {H}, spp={SPP}, max_bounces={MB}, seed={SEED}, intersector=2, collect_counters=True)\n"
        "    sc = ctx.scene(a); sc.update(b); img = ctx.render_frame(sc, p)\n"
        "    sc.update(a); sc.wait_ready(); _, st = ctx.render_frame(sc, pc, want_stats=True); sc.close()\n"
        "    fresh = ctx.scene(a).wait_ready(); _, st2 = ctx.render_frame(fresh, pc, want_stats=True); fresh.close()\n"
        "    out.append(f\"{hashlib.sha256(img.tobytes()).hexdigest()}:{st['slab_tests']}:{st2['slab_tests']}\")\n"
        "print(' '.join(out))"
    )
    got = _run(code, {"RT_B200_BUILD": "device"}).split()
    assert len(got) == 2, got
    for n, g in zip((300, 8192), got):
        digest, slabs, slabs_fresh = g.split(":")
        b, _ = _moved(rt.scenes.synthetic_spheres(n, 8), None, 21)
        ref, _ = O.render_frame(b, None, W, H, SPP, MB, seed=SEED)
        assert digest == _sha(ref), n
        assert int(slabs) == int(slabs_fresh) > 0, (n, slabs, slabs_fresh)


# ---------------------------------------------------------------------------------------------------
# materials only
# ---------------------------------------------------------------------------------------------------
def test_update_materials_only(ctx, rt, O):
    sp, tr = rt.scenes.synthetic_spheres(64, 2), rt.scenes.ground_plane()
    sp_b, tr_b = sp.copy(), tr.copy()
    _new_materials(sp_b, np.random.default_rng(3))
    sp_b["emission"][5], sp_b["albedo"][5] = 3.0, (1.0, 0.9, 0.6)  # a sphere that becomes a light
    tr_b["albedo"] = (0.3, 0.8, 0.3)
    sc = ctx.scene(sp, tr)
    try:
        sc.update(sp_b, tr_b)
        ref, _ = O.render_frame(sp_b, tr_b, W, H, SPP, MB, seed=SEED)
        for isect in (1, 2):
            assert_parity(ctx.render_frame(sc, _params(rt, isect)), ref)
    finally:
        sc.close()


def test_materials_update_restarts_nothing(rt, O):
    """Boxes unchanged: the tables that have landed stay, so a render straight after the update needs no second pass
    although the builder thread of a new build would still be asleep (RT_B200_AUX_DELAY_MS)."""
    code = (
        "ctx = rt.Context(0); a = rt.scenes.synthetic_spheres(300, 4); tr = rt.scenes.ground_plane()\n"
        "b = a.copy(); b['albedo'] = b['albedo'][::-1].copy(); b['emission'][7] = 2.0\n"
        "sc = ctx.scene(a, tr).wait_ready(); sc.update(b, tr)\n"
        f"img, st = ctx.render_frame(sc, rt.make_params({W}, {H}, spp={SPP}, max_bounces={MB}, seed={SEED}, intersector=2),"
        " want_stats=True)\n"
        "print(hashlib.sha256(img.tobytes()).hexdigest(), st['redo_pixels'], st['kernel_launches'])"
    )
    digest, redo, launches = _run(code, {"RT_B200_AUX_DELAY_MS": "300"}).split()
    a, tr = rt.scenes.synthetic_spheres(300, 4), rt.scenes.ground_plane()
    b = a.copy()
    b["albedo"] = b["albedo"][::-1].copy()
    b["emission"][7] = 2.0
    ref, _ = O.render_frame(b, tr, W, H, SPP, MB, seed=SEED)
    assert digest == _sha(ref)
    assert (int(redo), int(launches)) == (0, 1)


# ---------------------------------------------------------------------------------------------------
# update before the new tables land
# ---------------------------------------------------------------------------------------------------
def test_update_before_tables_land(rt, O):
    """The moved tie mesh's tables are held back (RT_B200_AUX_DELAY_MS): the first pass marks every tie pixel and the
    second pass reproduces the oracle of the moved mesh — with a pixel list and by repeating the launch."""
    code = (
        "from test_gpu_parity import _tie_mesh\n"
        "ctx = rt.Context(0); tr = _tie_mesh(rt); _, trb = _moved(None, tr, 31, materials=False); out = []\n"
        "for (w, h) in ((96, 64), (512, 320)):\n"
        "    sc = ctx.scene(None, tr).wait_ready(); sc.update(None, trb)\n"
        "    img, st = ctx.render_frame(sc, rt.make_params(w, h, spp=2, max_bounces=3, seed=7), want_stats=True)\n"
        "    out.append(hashlib.sha256(img.tobytes()).hexdigest() + ':' + str(st['redo_pixels'])); sc.close()\n"
        "print(' '.join(out))"
    )
    got = _run(code, {"RT_B200_AUX_DELAY_MS": "300"}).split()
    from test_gpu_parity import _tie_mesh

    _, trb = _moved(None, _tie_mesh(rt), 31, materials=False)
    for (w, h), g in zip(((96, 64), (512, 320)), got):
        ref, _ = O.render_frame(None, trb, w, h, 2, 3, seed=7)
        digest, redo = g.split(":")
        assert digest == _sha(ref), (w, h, redo)
        assert int(redo) > 0, "the first pass must have met ties without the tables"
    assert int(got[0].split(":")[1]) < 65536 and int(got[1].split(":")[1]) == 0xffffffff


# ---------------------------------------------------------------------------------------------------
# animation: successive updates of one large scene
# ---------------------------------------------------------------------------------------------------
def test_animation_sequence_65536_spheres(ctx, rt):
    """20 updates of one 65,536-sphere scene (device-built tree, threaded tables), every fifth of them materials only:
    after each, the frame equals that of a scene created from the same world (stale flags, builder threads or arrival
    counters would show)."""
    sp = rt.scenes.synthetic_spheres(65536, 9)
    p = rt.make_params(256, 144, spp=4, max_bounces=5, seed=1, intersector=2)
    sc = ctx.scene(sp)
    try:
        for k in range(20):
            if k % 5 == 4:
                sp = sp.copy()
                _new_materials(sp, np.random.default_rng(100 + k))
            else:
                sp, _ = _moved(sp, None, 100 + k, materials=(k % 4 == 0), scale=0.2)
            sc.update(sp)
            got = _sha(ctx.render_frame(sc, p))
            fresh = ctx.scene(sp)
            want = _sha(ctx.render_frame(fresh, p))
            fresh.close()
            assert got == want, k
    finally:
        sc.close()


# ---------------------------------------------------------------------------------------------------
# progressive
# ---------------------------------------------------------------------------------------------------
def test_update_refuses_old_accum_until_reset(ctx, rt, O):
    sp, tr = rt.scenes.synthetic_spheres(64, 5), rt.scenes.ground_plane()
    sp_b, tr_b = _moved(sp, tr, 41)
    w, h, mb, seed = 64, 40, 4, 2
    sc = ctx.scene(sp, tr)
    try:
        with ctx.accum(rt.make_params(w, h, max_bounces=mb, seed=seed)) as acc:
            ctx.render_samples(sc, acc, 1)
            sc.update(sp_b, tr_b)
            with pytest.raises(rt.RtError) as e:
                ctx.render_samples(sc, acc, 1)
            assert e.value.status == rt._abi.RT_ERR_INVALID_ARG
            assert acc.samples == 1
            acc.reset()
            done = 0
            for n in (1, 1, 2):
                img = ctx.render_samples(sc, acc, n)
                done += n
                ref, _ = O.render_frame(sp_b, tr_b, w, h, done, mb, seed=seed)
                assert_parity(img, ref)
    finally:
        sc.close()


# ---------------------------------------------------------------------------------------------------
# errors leave the scene as it was
# ---------------------------------------------------------------------------------------------------
def test_update_errors(ctx, rt, O):
    from rt_b200 import _abi

    L = _abi.lib()
    sp, tr = rt.scenes.synthetic_spheres(32, 6), rt.scenes.ground_plane()
    ref, _ = O.render_frame(sp, tr, W, H, SPP, MB, seed=SEED)
    sc = ctx.scene(sp, tr)
    other = rt.Context(0)
    try:
        ptr = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        inv = _abi.RT_ERR_INVALID_ARG
        assert L.rt_scene_update(None, sc._h, ptr(sp), len(sp), ptr(tr), len(tr)) == inv
        assert L.rt_scene_update(ctx._h, None, ptr(sp), len(sp), ptr(tr), len(tr)) == inv
        assert L.rt_scene_update(ctx._h, sc._h, ptr(sp), len(sp) - 1, ptr(tr), len(tr)) == inv
        assert L.rt_scene_update(ctx._h, sc._h, ptr(sp), len(sp), ptr(tr), len(tr) + 1) == inv
        assert L.rt_scene_update(ctx._h, sc._h, None, len(sp), ptr(tr), len(tr)) == inv
        assert L.rt_scene_update(ctx._h, sc._h, ptr(sp), len(sp), None, len(tr)) == inv
        assert L.rt_scene_update(other._h, sc._h, ptr(sp), len(sp), ptr(tr), len(tr)) == inv
        with pytest.raises(rt.RtError) as e:
            sc.update(sp[:-1], tr)
        assert e.value.status == inv
        bad = _moved(sp, tr, 51)[0]
        bad["center"][17, 1] = np.nan
        with pytest.raises(rt.RtError) as e:
            sc.update(bad, tr)
        assert e.value.status == _abi.RT_ERR_BVH and "non-finite" in e.value.message
        for isect in (1, 2):
            assert np.array_equal(ctx.render_frame(sc, _params(rt, isect)), ref)
        assert np.array_equal(sc.info()["rank"], rt.api.bvh_build_host(sp, tr)[0])
    finally:
        sc.close()
        other.close()


# ---------------------------------------------------------------------------------------------------
# multi-context frame
# ---------------------------------------------------------------------------------------------------
def test_update_multi_context_frame(ctx, rt, O):
    sp, tr = rt.scenes.synthetic_spheres(200, 7), rt.scenes.ground_plane()
    sp_b, tr_b = _moved(sp, tr, 61)
    ref, _ = O.render_frame(sp_b, tr_b, W, H, SPP, MB, seed=SEED)
    c1 = rt.Context(0)
    s0, s1 = ctx.scene(sp, tr), c1.scene(sp, tr)
    try:
        s0.update(sp_b, tr_b)
        s1.update(sp_b, tr_b)
        img = rt.api.render_frame_multi([ctx, c1], [s0, s1], _params(rt))
        assert_parity(img, ref)
    finally:
        s0.close()
        s1.close()
        c1.close()
