"""The render entries end to end on one GPU: the frame owner's collection (ranks emulated by one context), rt_frame_collect,
and the statistics each entry reports.  Every wait on these paths has the library's wait limit, so a frame that never
completes fails with RT_ERR_TIMEOUT instead of hanging."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H, SPP, MB = 512, 320, 2, 5
NBYTES = W * H * 3


@pytest.fixture(scope="module")
def settled(ctx, rt):
    """A scene whose tie-break tables are on the device (no second pass), its parameters and render_frame's result."""
    sc = ctx.scene(rt.scenes.synthetic_spheres(64, 3), rt.scenes.ground_plane()).wait_ready()
    p = rt.make_params(W, H, spp=SPP, max_bounces=MB, seed=4)
    ref, st = ctx.render_frame(sc, p, want_stats=True)
    yield sc, p, ref, st
    sc.close()


@pytest.mark.parametrize("dest", ["pageable", "pinned"])
def test_owner_collects_emulated_ranks(ctx, settled, dest):
    """Ranks 1 and 2 render into a frame_alloc'd buffer, then rank 0 renders its share and collects the whole frame.
    The second frame goes into the same buffer behind frame_wait_consumed: the per-slab counters are cumulative."""
    sc, p, ref, ref_st = settled
    dev, _ = ctx.frame_alloc(NBYTES)
    try:
        for seq in (1, 2):
            if seq > 1:
                ctx.frame_wait_consumed(dev, NBYTES, seq - 1)
            rays = 0
            for rank in (1, 2):
                rays += ctx.render_tiles_device(sc, p, rank, 3, dev, sync=True, want_stats=True)["rays"]
            out = np.empty((H, W, 3), np.uint8) if dest == "pageable" else ctx.pinned_empty((H, W, 3))
            st = ctx.render_tiles_collect(sc, p, 0, 3, dev, seq, out, want_stats=True)
            rays += st["rays"]
            assert np.array_equal(out, ref), (dest, seq)
            assert rays == ref_st["rays"], (dest, seq)
    finally:
        ctx.frame_free(dev)


def test_frame_collect_after_three_ranks(ctx, settled):
    sc, p, ref, _ = settled
    dev, _ = ctx.frame_alloc(NBYTES)
    try:
        for rank in range(3):
            ctx.render_tiles_device(sc, p, rank, 3, dev, sync=True)
        out = ctx.frame_collect(dev, p, 1, out=np.empty((H, W, 3), np.uint8))
    finally:
        ctx.frame_free(dev)
    assert np.array_equal(out, ref)


def test_stats_per_entry(ctx, rt, settled):
    sc, p, ref, st = settled
    assert st["primary"] == H * W * SPP and st["kernel_launches"] == 1 and st["redo_pixels"] == 0

    div = 4
    _, sd = ctx.render_division(sc, rt.make_params(W, H, divisions=div, division_no=1, spp=SPP, max_bounces=MB, seed=4),
                                want_stats=True)
    assert sd["primary"] == H // div * W * SPP and sd["kernel_launches"] == 1

    dev, _ = ctx.frame_alloc(NBYTES)
    try:
        s1 = ctx.render_tiles_device(sc, p, 1, 2, dev, sync=True, want_stats=True)
        s0 = ctx.render_tiles_collect(sc, p, 0, 2, dev, 1, np.empty((H, W, 3), np.uint8), want_stats=True)
    finally:
        ctx.frame_free(dev)
    for s in (s0, s1):
        assert s["primary"] == W * H // 2 * SPP and s["kernel_launches"] == 1
    assert s0["rays"] + s1["rays"] == st["rays"]

    with ctx.accum(rt.make_params(W, H, divisions=div, division_no=2, max_bounces=MB, seed=4)) as acc:
        _, c1 = ctx.render_samples(sc, acc, 2, want_stats=True)
        _, c2 = ctx.render_samples(sc, acc, 3, want_stats=True)
    assert c1["primary"] == H // div * W * 2 and c1["kernel_launches"] == 1
    assert c2["primary"] == H // div * W * 3 and c2["kernel_launches"] == 1


def test_multi_context_stats(rt, settled):
    from rt_b200 import multi

    _, p, ref, st = settled
    sp, tr = rt.scenes.synthetic_spheres(64, 3), rt.scenes.ground_plane()
    m = multi.MultiDeviceRenderer([0, 0, 0])
    try:
        scenes = [s.wait_ready() for s in m.scenes(sp, tr)]
        img, sm = m.render(scenes, p, want_stats=True)
        c0 = m.ctxs[0]
        dev, _ = c0.frame_alloc(NBYTES)
        try:
            s0 = c0.render_tiles_device(scenes[0], p, 0, 3, dev, sync=True, want_stats=True)
        finally:
            c0.frame_free(dev)
        for s in scenes:
            s.close()
    finally:
        m.close()
    assert np.array_equal(img, ref)
    assert sm["primary"] == W * H * SPP and sm["kernel_launches"] == 3 and sm["rays"] == st["rays"]
    for k in ("intersector_used", "grid_ctas", "cta_threads"):
        assert sm[k] == s0[k], k


def test_second_pass_is_counted(rt):
    """Tie-break tables held back (RT_B200_AUX_DELAY_MS): render_frame re-renders the tie pixels in a second launch."""
    code = (
        "import sys; sys.path.insert(0, 'ray-tracer-s8_b200'); sys.path.insert(0, 'tests');"
        "import rt_b200 as rt; from test_gpu_parity import _tie_mesh;"
        "ctx = rt.Context(0); sc = ctx.scene(None, _tie_mesh(rt));"
        "img, st = ctx.render_frame(sc, rt.make_params(96, 64, spp=2, max_bounces=3, seed=7), want_stats=True);"
        "print(st['redo_pixels'], st['kernel_launches'])"
    )
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    env = dict(os.environ, RT_B200_AUX_DELAY_MS="300")
    out = subprocess.run([sys.executable, "-c", code], cwd=root, env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-800:]
    redo, launches = (int(v) for v in out.stdout.strip().splitlines()[-1].split())
    assert redo > 0 and launches == 2, (redo, launches)
