"""Progressive rendering on several contexts (rt_render_samples_multi): accum i holds the chains of rank i's tiles, and
after every chunk the frame is byte-identical to rt_render_frame on one context at the cumulative sample count.  Three
contexts share device 0 here, as in the other multi-context tests; the last test uses two devices when there are two."""
import ctypes as C
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import assert_parity

SCHEDULE = (1, 1, 2, 4)
ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


# ---------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------
def test_entry_point_declared_and_exported(rt):
    from rt_b200 import _abi

    header = open(os.path.join(ROOT, "include", "rt_b200.h")).read()
    assert "int rt_render_samples_multi(" in header
    assert "rt_render_samples_multi" in _abi.EXPORTS and hasattr(_abi.lib(), "rt_render_samples_multi")


def test_null_handles_refused(rt):
    from rt_b200 import _abi

    L = _abi.lib()
    assert L.rt_render_samples_multi(None, None, None, 0, 1, None, 0, None) == _abi.RT_ERR_INVALID_ARG
    nul = (C.c_void_p * 1)()
    assert L.rt_render_samples_multi(nul, nul, nul, 1, 1, None, 0, None) == _abi.RT_ERR_INVALID_ARG


@pytest.mark.parametrize("lens", [(0, 0, 0), (2, 1, 2), (2, 2, 1), (1, 2, 2)])
def test_wrapper_refuses_mismatched_lists(rt, lens):
    """The lists are checked before anything reaches the library: these placeholders have no handles at all."""
    c, s, a = ([object()] * k for k in lens)
    with pytest.raises(rt.RtError) as e:
        rt.render_samples_multi(c, s, a, 1)
    assert e.value.status == -1


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def trio(rt):
    """Three contexts on device 0: three ranks that share one device."""
    cs = [rt.Context(0) for _ in range(3)]
    yield cs
    for c in cs:
        c.close()


def _chain(rt, ctxs, scenes, params, schedule):
    """(cumulative samples, frame, stats) after each chunk of `schedule`, on fresh accums."""
    accs = [c.accum(params) for c in ctxs]
    try:
        out, done = [], 0
        for n in schedule:
            img, st = rt.render_samples_multi(ctxs, scenes, accs, n, want_stats=True)
            done += n
            assert [a.samples for a in accs] == [done] * len(accs)
            out.append((done, img, st))
        return out
    finally:
        for a in accs:
            a.close()


def _one_shot(ctx, scene, params, spp):
    """rt_render_frame on one context at `spp`."""
    q = type(params).from_buffer_copy(params)
    q.spp = spp
    return ctx.render_frame(scene, q)


@pytest.mark.gpu
@pytest.mark.parametrize("case", [
    dict(id="smem_brute", n=64, w=160, h=96, isect=1, smem=1),
    dict(id="smem_bvh", n=64, w=160, h=96, isect=2, smem=1),
    dict(id="l2_bvh", n=65536, w=96, h=64, isect=2, smem=0),     # the scene does not fit shared memory
    dict(id="l2_brute", n=8000, w=64, h=40, isect=1, smem=0),
    dict(id="ragged_bvh", n=32, w=1001, h=701, isect=2, smem=1),  # two slabs; tiles and slabs do not divide the frame
    dict(id="ragged_brute", n=32, w=1001, h=701, isect=1, smem=1),
], ids=lambda c: c["id"])
def test_each_chunk_equals_one_shot(ctx, trio, rt, case):
    sp, tr = rt.scenes.synthetic_spheres(case["n"], 17), rt.scenes.ground_plane()
    p = rt.make_params(case["w"], case["h"], max_bounces=5, seed=9, intersector=case["isect"])
    scenes = [c.scene(sp, tr) for c in trio + [ctx]]
    try:
        steps = _chain(rt, trio, scenes[:3], p, SCHEDULE)
        for done, img, st in steps:
            assert np.array_equal(img, _one_shot(ctx, scenes[3], p, done)), (case["id"], done)
            assert st["scene_in_smem"] == case["smem"] and st["intersector_used"] == case["isect"]
            assert st["kernel_launches"] >= 3
    finally:
        for s in scenes:
            s.close()


@pytest.mark.gpu
def test_small_frame_matches_oracle(trio, rt, O):
    sp, tr = rt.scenes.synthetic_spheres(40, 4), rt.scenes.ground_plane()
    w, h, mb, seed = 64, 48, 4, 3
    scenes = [c.scene(sp, tr) for c in trio]
    try:
        steps = _chain(rt, trio, scenes, rt.make_params(w, h, max_bounces=mb, seed=seed), (1, 2))
    finally:
        for s in scenes:
            s.close()
    for done, img, _ in steps:
        ref, _ = O.render_frame(sp, tr, w, h, done, mb, seed=seed)
        assert_parity(img, ref)


@pytest.mark.gpu
def test_stats_match_single_context_chunks(ctx, trio, rt):
    """rays of each chunk equal rt_render_samples' on one context over the same chunk; primary = W*H*n_samples."""
    sp, tr = rt.scenes.synthetic_spheres(64, 3), rt.scenes.ground_plane()
    w, h = 128, 72
    p = rt.make_params(w, h, max_bounces=5, seed=4)
    scenes = [c.scene(sp, tr).wait_ready() for c in trio]
    one = ctx.scene(sp, tr).wait_ready()
    try:
        steps = _chain(rt, trio, scenes, p, (1, 3))
        with ctx.accum(p) as acc:
            single = [ctx.render_samples(one, acc, n, want_stats=True) for n in (1, 3)]
    finally:
        for s in scenes + [one]:
            s.close()
    for (done, img, st), (simg, sst), n in zip(steps, single, (1, 3)):
        assert np.array_equal(img, simg)
        assert st["rays"] == sst["rays"] and st["primary"] == w * h * n and st["redo_pixels"] == 0
        assert st["kernel_launches"] == 3


@pytest.mark.gpu
def test_progressive_generator(ctx, rt):
    from rt_b200 import multi

    sp, tr = rt.scenes.synthetic_spheres(64), rt.scenes.ground_plane()
    p = rt.make_params(160, 96, max_bounces=5, seed=7)
    m = multi.MultiDeviceRenderer([0, 0, 0])
    one = ctx.scene(sp, tr)
    try:
        scenes = m.scenes(sp, tr)
        got = [(n, img.copy()) for n, img in m.render_progressive(scenes, p, schedule=SCHEDULE)]
        for s in scenes:
            s.close()
        assert [n for n, _ in got] == [1, 2, 4, 8]
        for n, img in got:
            assert np.array_equal(img, _one_shot(ctx, one, p, n)), n
    finally:
        one.close()
        m.close()


@pytest.mark.gpu
def test_second_passes_under_chained_state(rt, O):
    """The tie-break tables are held back (RT_B200_AUX_DELAY_MS), so the first chunk holds every tie pixel back: at 96x64
    the host re-renders them from a pixel list, at 640x400 each of the three ranks has more than the list's 65,536 and
    repeats its whole launch.  Both passes start over from the chunk's state: a pixel advanced twice would show in the
    second chunk."""
    code = (
        "import sys, hashlib; sys.path.insert(0, 'ray-tracer-s8_b200'); sys.path.insert(0, 'tests');"
        "import rt_b200 as rt; from test_gpu_parity import _tie_mesh;"
        "cs = [rt.Context(0) for _ in range(3)]; tr = _tie_mesh(rt); out = []\n"
        "for (w, h) in ((96, 64), (640, 400)):\n"
        "    scs = [c.scene(None, tr) for c in cs]; accs = [c.accum(rt.make_params(w, h, max_bounces=3, seed=7)) for c in cs]\n"
        "    f1, st = rt.render_samples_multi(cs, scs, accs, 1, want_stats=True)\n"
        "    f2 = rt.render_samples_multi(cs, scs, accs, 1)\n"
        "    out.append(':'.join([hashlib.sha256(f1.tobytes()).hexdigest(), hashlib.sha256(f2.tobytes()).hexdigest(),\n"
        "                         str(st['redo_pixels'])]))\n"
        "    [a.close() for a in accs]; [s.close() for s in scs]\n"
        "print(' '.join(out))"
    )
    env = dict(os.environ, RT_B200_AUX_DELAY_MS="300")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-800:]
    got = out.stdout.strip().splitlines()[-1].split()
    from test_gpu_parity import _tie_mesh

    tr = _tie_mesh(rt)
    for (w, h), g in zip(((96, 64), (640, 400)), got):
        d1, d2, redo = g.split(":")
        for spp, d in ((1, d1), (2, d2)):
            ref, _ = O.render_frame(None, tr, w, h, spp, 3, seed=7)
            assert d == hashlib.sha256(ref.tobytes()).hexdigest(), (w, h, spp, redo)
    assert 0 < int(got[0].split(":")[2]) < 65536, "the first chunk must have met ties without the tables"
    assert int(got[1].split(":")[2]) == 0xffffffff, "every rank must have held back more pixels than the list holds"


@pytest.mark.gpu
def test_errors_move_no_accum(ctx, trio, rt):
    from rt_b200 import _abi

    sp, tr = rt.scenes.synthetic_spheres(48, 8), rt.scenes.ground_plane()
    w, h = 64, 48
    p = rt.make_params(w, h, max_bounces=4, seed=6)
    scenes = [c.scene(sp, tr) for c in trio]
    one = ctx.scene(sp, tr)
    accs = [c.accum(p) for c in trio]
    extra = []
    done = 0

    def step(n=1):
        nonlocal done
        img = rt.render_samples_multi(trio, scenes, accs, n)
        done += n
        assert [a.samples for a in accs] == [done] * 3
        assert np.array_equal(img, _one_shot(ctx, one, p, done)), done

    def refused(call):
        with pytest.raises(rt.RtError) as e:
            call()
        assert e.value.status == _abi.RT_ERR_INVALID_ARG
        assert [a.samples for a in accs] == [done] * 3
        step()  # the chain goes on as if nothing had been tried

    try:
        step()
        a0, a1, a2 = accs
        s0, s1, s2 = scenes
        c0, c1, c2 = trio
        refused(lambda: rt.render_samples_multi(trio, scenes, [a1, a0, a2], 1))           # accum of another context
        refused(lambda: rt.render_samples_multi([c1, c0, c2], [s1, s0, s2], [a1, a0, a2], 1))  # another rank
        refused(lambda: rt.render_samples_multi(trio[:2], scenes[:2], accs[:2], 1))       # another n
        refused(lambda: c0.render_samples(s0, a0, 1))                                     # multi-bound, used singly
        refused(lambda: a0.read_linear())                                                 # no multi-GPU readback
        refused(lambda: rt.render_samples_multi(trio, scenes, accs, 0))                   # no samples
        refused(lambda: rt.render_samples_multi(trio, scenes, accs, 0xffffffff))          # overflows 32 bits
        buf = np.zeros((h, w, 3), np.uint8)
        refused(lambda: rt.render_samples_multi(trio, scenes, accs, 1, out=buf[:-1]))     # wrong out_len
        # a singly-bound accum in a multi call
        single = c0.accum(p)
        extra.append(single)
        c0.render_samples(s0, single, done)
        refused(lambda: rt.render_samples_multi(trio, scenes, [single, a1, a2], 1))
        # another binding: a fresh accum of another seed, and one of the same params at another sample count
        other = c1.accum(rt.make_params(w, h, max_bounces=4, seed=99))
        extra.append(other)
        refused(lambda: rt.render_samples_multi(trio, scenes, [a0, other, a2], 1))
        behind = [c.accum(p) for c in trio]
        extra.extend(behind)
        rt.render_samples_multi(trio, scenes, behind, 1)
        refused(lambda: rt.render_samples_multi(trio, scenes, [a0, behind[1], a2], 1))
        # a scene updated mid-chain: refused until the accums are reset
        s1.update(sp, tr)
        with pytest.raises(rt.RtError) as e:
            rt.render_samples_multi(trio, scenes, accs, 1)
        assert e.value.status == _abi.RT_ERR_INVALID_ARG and [a.samples for a in accs] == [done] * 3
        for a in accs:
            a.reset()
        done = 0
        step(2)
    finally:
        for a in accs + extra:
            a.close()
        for s in scenes + [one]:
            s.close()


@pytest.mark.gpu
def test_reset_rebinds(ctx, trio, rt):
    """Multi to single and back: after rt_accum_reset an accum takes the share of its next chunk."""
    sp, tr = rt.scenes.synthetic_spheres(48, 2), rt.scenes.ground_plane()
    w, h = 96, 64
    p = rt.make_params(w, h, max_bounces=4, seed=5)
    scenes = [c.scene(sp, tr) for c in trio]
    one = ctx.scene(sp, tr)
    accs = [c.accum(p) for c in trio]
    c0, s0, a0 = trio[0], scenes[0], accs[0]
    try:
        rt.render_samples_multi(trio, scenes, accs, 1)
        a0.reset()
        img = c0.render_samples(s0, a0, 2)                      # now rank 0 of 1
        assert np.array_equal(img, _one_shot(ctx, one, p, 2))
        assert a0.read_linear().shape == (h, w, 3)
        with pytest.raises(rt.RtError) as e:
            rt.render_samples_multi(trio, scenes, accs, 1)      # a0 is bound singly now
        assert e.value.status == -1
        for a in accs:
            a.reset()
        for n, want in ((1, 1), (2, 3)):
            img = rt.render_samples_multi(trio, scenes, accs, n)
            assert np.array_equal(img, _one_shot(ctx, one, p, want)), want
        # and a reset with new params (a camera move) on every rank
        q = rt.make_params(w, h, max_bounces=4, seed=5, cam_origin=(0.2, 0.1, 0.0))
        for a in accs:
            a.reset(q)
        img = rt.render_samples_multi(trio, scenes, accs, 2)
        assert np.array_equal(img, _one_shot(ctx, one, q, 2))
    finally:
        for a in accs:
            a.close()
        for s in scenes + [one]:
            s.close()


@pytest.mark.gpu
def test_two_devices(rt):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from rt_b200 import multi

    sp, tr = rt.scenes.synthetic_spheres(200, 6), rt.scenes.ground_plane()
    p = rt.make_params(322, 181, max_bounces=5, seed=2)
    m = multi.MultiDeviceRenderer([0, 1])
    try:
        scenes = m.scenes(sp, tr)
        got = [(n, img.copy()) for n, img in m.render_progressive(scenes, p, schedule=SCHEDULE)]
        for n, img in got:
            q = rt.RtParams.from_buffer_copy(p)
            q.spp = n
            assert np.array_equal(img, m.render(scenes, q)), n
            assert np.array_equal(img, _one_shot(m.ctxs[0], scenes[0], p, n)), n
        for s in scenes:
            s.close()
    finally:
        m.close()
