"""Progressive rendering (rt_accum / rt_render_samples): a band rendered in chunks of samples is byte-identical at every
step to rt_render_division at the cumulative sample count, and so to the oracle."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from conftest import assert_parity

BOTH = [1, 2]  # RT_INTERSECT_BRUTE, RT_INTERSECT_BVH
NEW_EXPORTS = ["rt_accum_create", "rt_accum_destroy", "rt_accum_reset", "rt_accum_samples", "rt_render_samples",
               "rt_accum_read_linear"]


# ---------------------------------------------------------------------------------------------------
# CPU: the entry points exist and refuse missing handles before touching a device
# ---------------------------------------------------------------------------------------------------
def test_progressive_entry_points_exported(rt):
    from rt_b200 import _abi

    L = _abi.lib()
    for name in NEW_EXPORTS:
        assert name in _abi.EXPORTS and hasattr(L, name), name


def test_progressive_null_handles(rt):
    from rt_b200 import _abi

    L = _abi.lib()
    p = rt.make_params(16, 8, spp=1)
    n = C.c_uint32(7)
    h = C.c_void_p(1)
    assert L.rt_accum_create(None, C.byref(p), C.byref(h)) == _abi.RT_ERR_INVALID_ARG
    assert L.rt_accum_samples(None, C.byref(n)) == _abi.RT_ERR_INVALID_ARG and n.value == 7
    assert L.rt_accum_reset(None, None, None) == _abi.RT_ERR_INVALID_ARG
    assert L.rt_render_samples(None, None, None, 1, None, 0, None) == _abi.RT_ERR_INVALID_ARG
    assert L.rt_accum_read_linear(None, None, None, 0) == _abi.RT_ERR_INVALID_ARG
    L.rt_accum_destroy(None, None)  # a no-op


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def _chunks(ctx, sc, acc, chunks):
    """(cumulative samples, frame, stats) after each chunk."""
    out, done = [], 0
    for n in chunks:
        img, st = ctx.render_samples(sc, acc, n, want_stats=True)
        done += n
        assert acc.samples == done
        out.append((done, img, st))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("isect", BOTH)
def test_prefix_parity(ctx, rt, O, isect):
    """Chunks of 1, 2, 1, 4 samples: after each, the frame of spp = 1, 3, 4, 8 (oracle and render_frame)."""
    sp, tr = rt.scenes.synthetic_spheres(64), rt.scenes.ground_plane()
    w, h, mb, seed = 160, 96, 5, 7
    sc = ctx.scene(sp, tr).wait_ready()  # rays are compared: no pixel traced twice for want of the tie-break tables
    p = rt.make_params(w, h, max_bounces=mb, seed=seed, intersector=isect)
    with ctx.accum(p) as acc:
        assert acc.samples == 0
        steps = _chunks(ctx, sc, acc, [1, 2, 1, 4])
    rays = 0
    for done, img, st in steps:
        ref, _ = O.render_frame(sp, tr, w, h, done, mb, seed=seed)
        assert_parity(img, ref)
        full = ctx.render_frame(sc, rt.make_params(w, h, spp=done, max_bounces=mb, seed=seed, intersector=isect))
        assert np.array_equal(img, full)
        assert st["intersector_used"] == isect and st["redo_pixels"] == 0
        rays += st["rays"]
    assert [s["primary"] for _, _, s in steps] == [w * h * n for n in (1, 2, 1, 4)]
    _, ost = O.render_frame(sp, tr, w, h, 8, mb, seed=seed, want_stats=True)
    assert rays == ost["rays"]
    sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("isect", BOTH)
@pytest.mark.parametrize("case", [
    dict(n=300, plane=True, w=7, h=5, chunks=(2, 3), mb=6),      # frame smaller than one tile
    dict(n=32, plane=True, w=101, h=67, chunks=(1, 2), mb=4),    # ragged size: partial tiles, unaligned rows
    dict(n=96, plane=True, w=64, h=64, chunks=(1, 1), mb=62),    # deepest path this build supports
    dict(n=1, plane=False, w=128, h=96, chunks=(1, 1), mb=5),    # root of the BVH is a leaf
])
def test_edge_shapes_in_two_chunks(ctx, rt, O, isect, case):
    sp = rt.scenes.synthetic_spheres(case["n"], 17)
    tr = rt.scenes.ground_plane() if case["plane"] else None
    spp = sum(case["chunks"])
    ref, ost = O.render_frame(sp, tr, case["w"], case["h"], spp, case["mb"], seed=5, want_stats=True)
    sc = ctx.scene(sp, tr).wait_ready()
    with ctx.accum(rt.make_params(case["w"], case["h"], max_bounces=case["mb"], seed=5, intersector=isect)) as acc:
        steps = _chunks(ctx, sc, acc, case["chunks"])
    sc.close()
    assert_parity(steps[-1][1], ref)
    assert sum(st["rays"] for _, _, st in steps) == ost["rays"]


@pytest.mark.gpu
def test_division_band(ctx, rt, O):
    """A band of the controller's 20 (C2 scene) in chunks of 1 + 1 equals the oracle's band at spp 2."""
    c = rt.scenes.CONFIGS["C2"]
    sp, tr = rt.scenes.config_scene("C2")
    ref, _ = O.render_rows(sp, tr, O.make_params(c["width"], c["height"], 20, 9, 2, c["max_bounces"]))
    sc = ctx.scene(sp, tr)
    with ctx.accum(rt.make_params(c["width"], c["height"], divisions=20, division_no=9,
                                  max_bounces=c["max_bounces"])) as acc:
        steps = _chunks(ctx, sc, acc, [1, 1])
    sc.close()
    assert steps[-1][1].shape == (54, 1920, 3)
    assert_parity(steps[-1][1], ref)


@pytest.mark.gpu
def test_l2_resident_variant(ctx, rt, O):
    """6000 spheres + plane do not fit shared memory: the resumable form of the L1/L2-resident kernel."""
    sp, tr = rt.scenes.synthetic_spheres(6000, 12), rt.scenes.ground_plane()
    ref, _ = O.render_frame(sp, tr, 200, 120, 2, 5, seed=3)
    sc = ctx.scene(sp, tr)
    with ctx.accum(rt.make_params(200, 120, max_bounces=5, seed=3)) as acc:
        steps = _chunks(ctx, sc, acc, [1, 1])
    sc.close()
    assert all(st["scene_in_smem"] == 0 and st["intersector_used"] == 2 for _, _, st in steps)
    assert_parity(steps[-1][1], ref)


@pytest.mark.gpu
def test_chunks_before_tables_land(rt, O):
    """The first chunk renders before the scene's tie-break tables land (RT_B200_AUX_DELAY_MS): its held-back pixels are
    rendered again from the chunk's starting state by the host's pixel-list pass (96x64) and by repeating the whole
    launch (512x320: more held-back pixels than the list holds).  If that second pass advanced a pixel twice, the
    next chunk would not match the oracle at spp 2."""
    import os
    import subprocess
    import sys

    code = (
        "import sys, hashlib; sys.path.insert(0, 'ray-tracer-s8_b200'); sys.path.insert(0, 'tests');"
        "import rt_b200 as rt; from test_gpu_parity import _tie_mesh;"
        "ctx = rt.Context(0); tr = _tie_mesh(rt); out = [];\n"
        "for (w, h) in ((96, 64), (512, 320)):\n"
        "    sc = ctx.scene(None, tr); acc = ctx.accum(rt.make_params(w, h, max_bounces=3, seed=7))\n"
        "    f1, st = ctx.render_samples(sc, acc, 1, want_stats=True)\n"
        "    f2 = ctx.render_samples(sc, acc, 1)\n"
        "    out.append(':'.join([hashlib.sha256(f1.tobytes()).hexdigest(), hashlib.sha256(f2.tobytes()).hexdigest(),\n"
        "                         str(st['redo_pixels'])])); acc.close(); sc.close()\n"
        "print(' '.join(out))"
    )
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    env = dict(os.environ, RT_B200_AUX_DELAY_MS="300")
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-800:]
    got = out.stdout.strip().splitlines()[-1].split()
    from test_gpu_parity import _tie_mesh

    tr = _tie_mesh(rt)
    for (w, h), g in zip(((96, 64), (512, 320)), got):
        d1, d2, redo = g.split(":")
        for spp, d in ((1, d1), (2, d2)):
            ref, _ = O.render_frame(None, tr, w, h, spp, 3, seed=7)
            assert d == hashlib.sha256(ref.tobytes()).hexdigest(), (w, h, spp, redo)
    assert 0 < int(got[0].split(":")[2]) < 65536, "the first chunk must have met ties without the tables"
    assert int(got[1].split(":")[2]) == 0xffffffff


def _quantise(lin):
    """quantise() of rt_trace.cuh on the host: sqrt, * 255.999 in float32, truncate, saturate, NaN -> 0."""
    with np.errstate(invalid="ignore", over="ignore"):
        s = np.sqrt(lin.astype(np.float32)) * np.float32(255.999)
        s = np.nan_to_num(s, nan=0.0, posinf=255.0, neginf=0.0)
    return np.clip(np.trunc(s), 0, 255).astype(np.uint8)


@pytest.mark.gpu
def test_read_linear_quantises_to_the_frame(ctx, rt):
    sp, tr = rt.scenes.synthetic_spheres(64), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr)
    with ctx.accum(rt.make_params(160, 96, max_bounces=5, seed=7)) as acc:
        with pytest.raises(rt.RtError) as e:
            acc.read_linear()  # nothing rendered yet
        assert e.value.status == -1
        for n in (1, 3):
            img = ctx.render_samples(sc, acc, n)
            lin = acc.read_linear()
            assert lin.dtype == np.float32 and lin.shape == img.shape
            assert np.array_equal(_quantise(lin), img)
            # reading does not disturb the chain
            assert acc.samples == (1 if n == 1 else 4)
        img8 = ctx.render_samples(sc, acc, 4)
        assert np.array_equal(img8, ctx.render_frame(sc, rt.make_params(160, 96, spp=8, max_bounces=5, seed=7)))
    sc.close()


@pytest.mark.gpu
def test_reset_and_rebind(ctx, rt):
    sp, tr = rt.scenes.synthetic_spheres(64), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr)
    p = rt.make_params(128, 72, max_bounces=5, seed=7)
    with ctx.accum(p) as acc:
        first = [img for _, img, _ in _chunks(ctx, sc, acc, [1, 2])]
        acc.reset()
        assert acc.samples == 0
        again = [img for _, img, _ in _chunks(ctx, sc, acc, [1, 2])]
        assert all(np.array_equal(a, b) for a, b in zip(first, again))
        # a camera move and another seed: the same as a fresh render with those params
        q = rt.make_params(128, 72, max_bounces=5, seed=11, cam_origin=(0.3, 0.1, 0.0))
        acc.reset(q)
        img = ctx.render_samples(sc, acc, 2)
        q.spp = 2
        assert np.array_equal(img, ctx.render_frame(sc, q))
        with pytest.raises(rt.RtError) as e:
            acc.reset(rt.make_params(130, 72, max_bounces=5, seed=11))
        assert e.value.status == -1
        assert acc.samples == 2
        img3 = ctx.render_samples(sc, acc, 1)
        q.spp = 3
        assert np.array_equal(img3, ctx.render_frame(sc, q))
    sc.close()


@pytest.mark.gpu
def test_errors_leave_the_state_unchanged(ctx, rt):
    from rt_b200 import _abi

    sp, tr = rt.scenes.synthetic_spheres(64), rt.scenes.ground_plane()
    w, h, mb, seed = 96, 64, 5, 7
    sc = ctx.scene(sp, tr)
    acc = ctx.accum(rt.make_params(w, h, max_bounces=mb, seed=seed))
    ctx.render_samples(sc, acc, 1)

    def expect(status, call):
        with pytest.raises(rt.RtError) as e:
            call()
        assert e.value.status == status
        assert acc.samples == 1

    expect(-1, lambda: ctx.render_samples(sc, acc, 0))                          # no samples
    expect(-1, lambda: ctx.render_samples(sc, acc, 0xffffffff))                 # 1 + (2^32 - 1) overflows
    buf = np.zeros((h, w, 3), np.uint8)
    rc = ctx._lib.rt_render_samples(ctx._h, sc._h, acc._h, 1, buf.ctypes.data_as(C.c_void_p), buf.nbytes - 1, None)
    assert rc == _abi.RT_ERR_INVALID_ARG and acc.samples == 1                   # wrong out_len
    with rt.Context(0) as other:
        expect(-1, lambda: other.render_samples(sc, acc, 1))                    # accum of another context
    expect(-1, lambda: acc.reset(rt.make_params(w, h + 4, max_bounces=mb)))    # another size
    expect(-1, lambda: acc.reset(rt.make_params(w, h, divisions=2, max_bounces=mb)))  # another band
    # the same world, but another scene object (it may even sit at the closed one's address)
    sc.close()
    sc2 = ctx.scene(sp, tr)
    expect(-1, lambda: ctx.render_samples(sc2, acc, 1))
    # after a reset any scene is accepted again; without one, the chain goes on as if nothing had failed
    acc.reset()
    img = ctx.render_samples(sc2, acc, 2)
    assert np.array_equal(img, ctx.render_frame(sc2, rt.make_params(w, h, spp=2, max_bounces=mb, seed=seed)))
    acc.close()
    acc = ctx.accum(rt.make_params(w, h, max_bounces=mb, seed=seed))
    ctx.render_samples(sc2, acc, 1)
    expect(-1, lambda: ctx.render_samples(sc2, acc, 0))
    img = ctx.render_samples(sc2, acc, 1)
    assert np.array_equal(img, ctx.render_frame(sc2, rt.make_params(w, h, spp=2, max_bounces=mb, seed=seed)))
    acc.close()
    sc2.close()


@pytest.mark.gpu
def test_render_progressive_generator(ctx, rt):
    sp, tr = rt.scenes.synthetic_spheres(64), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr)
    p = rt.make_params(160, 96, max_bounces=5, seed=7)
    got = [(n, img.copy()) for n, img in ctx.render_progressive(sc, p, schedule=(1, 1, 2, 4))]
    assert [n for n, _ in got] == [1, 2, 4, 8]
    for n, img in got:
        q = rt.make_params(160, 96, spp=n, max_bounces=5, seed=7)
        assert np.array_equal(img, ctx.render_frame(sc, q))
    sc.close()


@pytest.mark.gpu
def test_c3_full_size_in_four_chunks(ctx, rt):
    """C3 (4K, 16 spp, depth 5) in 4 x 4 samples: the same bytes as one rt_render_frame at 16 spp."""
    c = rt.scenes.CONFIGS["C3"]
    sp, tr = rt.scenes.config_scene("C3")
    sc = ctx.scene(sp, tr)
    full = ctx.render_frame(sc, rt.make_params(c["width"], c["height"], spp=c["spp"], max_bounces=c["max_bounces"]))
    with ctx.accum(rt.make_params(c["width"], c["height"], max_bounces=c["max_bounces"])) as acc:
        for _ in range(3):
            assert ctx.render_samples(sc, acc, 4, download=False) is None
        img = ctx.render_samples(sc, acc, 4)
        assert acc.samples == c["spp"] == 16
    sc.close()
    assert hashlib.sha256(img.tobytes()).hexdigest() == hashlib.sha256(full.tobytes()).hexdigest()
