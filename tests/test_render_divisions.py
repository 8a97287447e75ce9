"""Several divisions of one job in one call (rt_render_divisions): every band equals rt_render_division of that band byte
for byte, whether the list is one contiguous run (a plain row range) or any other list (the banded launch, bands stacked
in list order).  The slave renders the requests it finds queued together (Worker.render_many)."""
import ctypes as C
import os
import subprocess
import sys
import threading
import urllib.request
from collections import OrderedDict

import numpy as np
import pytest

from conftest import assert_parity

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


# ---------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------
def test_entry_point_declared_and_exported(rt):
    from rt_b200 import _abi

    header = open(os.path.join(ROOT, "include", "rt_b200.h")).read()
    assert "int rt_render_divisions(" in header
    assert "rt_render_divisions" in _abi.EXPORTS and hasattr(_abi.lib(), "rt_render_divisions")


def test_null_handles_refused(rt):
    from rt_b200 import _abi

    L = _abi.lib()
    nos = (C.c_uint32 * 2)(0, 1)
    buf = (C.c_uint8 * 12)()
    assert L.rt_render_divisions(None, None, None, nos, 2, buf, 12, None) == _abi.RT_ERR_INVALID_ARG
    assert L.rt_render_divisions(None, None, C.byref(rt.make_params(2, 2, divisions=2)), None, 0, None, 0, None) \
        == _abi.RT_ERR_INVALID_ARG


class _FakeCtx:
    """Stands in for the GPU context under a real Worker: render_divisions records its lists, and its first call waits
    until the test has queued every request, so what the slave finds queued is fixed."""

    def __init__(self):
        self.calls = []
        self.entered, self.gate = threading.Event(), threading.Event()

    def scene(self, *a):
        class S:
            def close(self):
                pass
        return S()

    def _band(self, p, d):
        from rt_b200 import _abi, api

        if d >= p.divisions:
            raise api.RtError(_abi.RT_ERR_INVALID_ARG, "division_no out of range")
        return np.full((p.height // p.divisions, p.width, 3), d, np.uint8)

    def render_divisions(self, scene, p, nos, want_stats=False):
        self.calls.append(list(nos))
        if len(self.calls) == 1:
            self.entered.set()
            assert self.gate.wait(30)
        return np.stack([self._band(p, d) for d in nos])

    def render_division(self, scene, p, want_stats=False):
        self.calls.append(("alone", p.division_no))
        return self._band(p, p.division_no)


def _fake_worker():
    from rt_b200 import slave

    wk = slave.Worker.__new__(slave.Worker)
    wk.ctx = _FakeCtx()
    wk.spp = wk.max_bounces = wk.seed = 0
    wk.intersector = 0
    wk._scenes, wk._cache_size, wk.scene_uploads = OrderedDict(), 4, 0
    wk.lock = threading.Lock()
    return wk


def _drain(rt, first, rest, n_posts):
    """Queues `first`, waits until the worker renders it, queues `rest` ((job id, division_no) pairs, 20 divisions
    of 8x40 each), lets the worker go on and returns (render_divisions lists, posted (id, division_no, first byte))."""
    from rt_b200 import slave, wire

    sp = rt.scenes.synthetic_spheres(4, 1)
    posts, done = [], threading.Event()

    def post(url, body):
        sl = wire.ImageSlice.from_json(body)
        posts.append((sl.id, sl.division_no, int(sl.image[0])))
        if len(posts) == n_posts:
            done.set()
        return "ok"

    wk = _fake_worker()
    ready, stop = threading.Event(), threading.Event()
    t = threading.Thread(target=slave.serve, kwargs=dict(host="127.0.0.1", port=0, result_url="http://master/result",
                                                         worker=wk, post=post, ready=ready, stop=stop), daemon=True)
    t.start()
    assert ready.wait(30)

    def send(job, d):
        meta = wire.RenderMeta(160, 40, 20, job)
        req = urllib.request.Request(f"http://127.0.0.1:{ready.port}/", data=wire.render_info_to_json(sp, None, meta, d).encode(),
                                     headers={"Content-Type": "application/json"}, method="POST")
        with urllib.request.urlopen(req, timeout=30) as r:
            assert r.read().decode() == slave.ACK_TEXT

    try:
        send(*first)
        assert wk.ctx.entered.wait(30)
        for job, d in rest:
            send(job, d)
        wk.ctx.gate.set()
        assert done.wait(30), posts
    finally:
        stop.set()
        t.join(30)
    return wk.ctx.calls, posts


A, B = "00000000-0000-4000-8000-00000000000a", "00000000-0000-4000-8000-00000000000b"


def test_slave_renders_a_queued_job_in_one_call(rt):
    calls, posts = _drain(rt, (A, 0), [(A, d) for d in range(1, 20)], 20)
    assert calls == [[0], list(range(1, 20))]
    assert sorted(posts) == [(A, d, d) for d in range(20)]


def test_slave_groups_interleaved_jobs_in_arrival_order(rt):
    rest = [(B, 5), (A, 3), (B, 1), (A, 4), (B, 2)]
    calls, posts = _drain(rt, (A, 0), rest, 6)
    assert calls == [[0], [5, 1, 2], [3, 4]]
    assert [p[:2] for p in posts[1:]] == [(B, 5), (B, 1), (B, 2), (A, 3), (A, 4)]


def test_slave_renders_a_duplicate_once_and_posts_it_twice(rt):
    calls, posts = _drain(rt, (A, 0), [(A, 7), (A, 2), (A, 7), (A, 9)], 5)
    assert calls == [[0], [7, 2, 9]]
    assert posts[1:] == [(A, 7, 7), (A, 2, 2), (A, 7, 7), (A, 9, 9)]


def test_slave_bad_request_fails_alone(rt, capfd):
    calls, posts = _drain(rt, (A, 0), [(A, 3), (A, 25), (A, 6)], 3)
    assert calls == [[0], [3, 25, 6], ("alone", 3), ("alone", 25), ("alone", 6)]
    assert posts[1:] == [(A, 3, 3), (A, 6, 6)]
    assert "[rt_b200.slave] job failed: RT_ERR_INVALID_ARG: division_no out of range" in capfd.readouterr().out


def test_controller_renders_a_job_in_one_call(rt):
    from rt_b200 import controller, wire
    from test_host import mesh_scene_obj

    calls = []

    class Many:
        def render_many(self, infos):
            calls.append([i.division_no for i in infos])
            m = infos[0].render_meta
            return [wire.ImageSlice(i.division_no, np.full(m.height // m.divisions * m.width * 3, i.division_no, np.uint8),
                                    m.id) for i in infos]

    data, n = mesh_scene_obj()
    c = controller.Controller(worker=Many(), width=64, height=40, divisions=4)
    job = c.upload(data, n)
    assert calls == [[0, 1, 2, 3]]
    assert sorted(c.jobs[job]["result"]) == [0, 1, 2, 3]


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def _params(rt, w, h, div, **kw):
    return rt.make_params(w, h, divisions=div, **kw)


def _check(ctx, sc, p, nos):
    """render_divisions of `nos` against render_division band by band; returns the call's stats and the bands' rays."""
    got, st = ctx.render_divisions(sc, p, nos, want_stats=True)
    rays = 0
    q = type(p).from_buffer_copy(p)
    for k, d in enumerate(nos):
        q.division_no = d
        ref, sd = ctx.render_division(sc, q, want_stats=True)
        assert np.array_equal(got[k], ref), (list(nos), k, d)
        rays += sd["rays"]
    return st, rays


LISTS = {
    "one": [6],
    "all_in_order": list(range(20)),
    "all_shuffled": [int(d) for d in np.random.default_rng(3).permutation(20)],
    "sparse": [19, 0, 7, 8, 3],
    "every_other": list(range(1, 20, 2)),
    "run_after_start": [4, 5, 6, 7],
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", [
    dict(id="smem_brute", n=12, w=96, h=80, isect=1, smem=1),
    dict(id="smem_bvh", n=64, w=96, h=80, isect=2, smem=1),
    dict(id="l2_bvh", n=65536, w=64, h=80, isect=2, smem=0),   # the scene does not fit shared memory
    dict(id="l2_brute", n=8000, w=40, h=40, isect=1, smem=0),
    dict(id="rows_54", n=64, w=120, h=1080, isect=2, smem=1),  # 54-row bands: tiles straddle two bands
    dict(id="ragged", n=32, w=1001, h=140, isect=2, smem=1),   # 7-row bands, a partial tile column
], ids=lambda c: c["id"])
@pytest.mark.parametrize("which", list(LISTS))
def test_each_band_equals_render_division(ctx, rt, case, which):
    sp, tr = rt.scenes.synthetic_spheres(case["n"], 11), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr).wait_ready()
    try:
        p = _params(rt, case["w"], case["h"], 20, spp=2, max_bounces=4, seed=5, intersector=case["isect"])
        st, _ = _check(ctx, sc, p, LISTS[which])
        assert st["scene_in_smem"] == case["smem"] and st["intersector_used"] == case["isect"]
        assert st["kernel_launches"] == 1
    finally:
        sc.close()


@pytest.mark.gpu
def test_streamed_and_unstreamed(ctx, rt):
    """At the reference's 1920x1080 / 20 divisions, 14 non-contiguous bands at 8 spp are 4.35 MB: the banded launch stages
    its output and streams it slab by slab.  Three bands at 8 spp and all 14 at 2 spp do not stream."""
    sp, tr = rt.scenes.synthetic_spheres(200, 2), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr).wait_ready()
    nos = [19, 17, 15, 13, 11, 9, 7, 5, 3, 1, 0, 4, 8, 12]
    try:
        for spp, lst in ((8, nos), (8, [2, 18, 10]), (2, nos)):
            _check(ctx, sc, _params(rt, 1920, 1080, 20, spp=spp, max_bounces=3, seed=1), lst)
    finally:
        sc.close()


@pytest.mark.gpu
def test_sparse_list_matches_oracle(ctx, rt, O):
    sp, tr = rt.scenes.synthetic_spheres(40, 4), rt.scenes.ground_plane()
    w, h, div, spp, mb, seed = 64, 48, 6, 2, 4, 3
    nos = [5, 0, 3]
    sc = ctx.scene(sp, tr)
    try:
        got = ctx.render_divisions(sc, _params(rt, w, h, div, spp=spp, max_bounces=mb, seed=seed), nos)
    finally:
        sc.close()
    for k, d in enumerate(nos):
        ref, _ = O.render_rows(sp, tr, O.make_params(w, h, div, d, spp, mb, seed))
        assert_parity(got[k], ref)


@pytest.mark.gpu
def test_stats(ctx, rt):
    sp, tr = rt.scenes.synthetic_spheres(64, 3), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr).wait_ready()
    w, h, div, spp = 128, 80, 20, 3
    try:
        for nos in ([9, 2, 14, 3], [4, 5, 6]):
            p = _params(rt, w, h, div, spp=spp, max_bounces=5, seed=2, collect_counters=True)
            st, rays = _check(ctx, sc, p, nos)
            assert st["rays"] == rays and st["primary"] == len(nos) * (h // div) * w * spp
            assert st["sphere_tests"] == 0 and st["redo_pixels"] == 0 and st["kernel_launches"] == 1
    finally:
        sc.close()


@pytest.mark.gpu
def test_second_passes_on_a_banded_launch(rt):
    """Tie-break tables held back (RT_B200_AUX_DELAY_MS): the first pass of a banded launch holds every tie pixel back.
    At 96x64 the host re-renders them from a pixel list, at 640x400 there are more than the list's 65,536 and it repeats
    the whole launch.  Both run the banded form with the same table: the bands equal render_division once the tables
    are there."""
    code = (
        "import sys, numpy as np; sys.path.insert(0, 'ray-tracer-s8_b200'); sys.path.insert(0, 'tests');"
        "import rt_b200 as rt; from test_gpu_parity import _tie_mesh;"
        "ctx = rt.Context(0); tr = _tie_mesh(rt); out = []\n"
        "for (w, h) in ((96, 64), (640, 400)):\n"
        "    sc = ctx.scene(None, tr); nos = [3, 0, 2]\n"
        "    p = rt.make_params(w, h, divisions=4, spp=2, max_bounces=3, seed=7)\n"
        "    got, st = ctx.render_divisions(sc, p, nos, want_stats=True)\n"
        "    sc.wait_ready(); same = True\n"
        "    for k, d in enumerate(nos):\n"
        "        p.division_no = d; same = same and np.array_equal(got[k], ctx.render_division(sc, p))\n"
        "    out.append('%d:%d:%d' % (same, st['redo_pixels'], st['kernel_launches'])); sc.close()\n"
        "print(' '.join(out))"
    )
    env = dict(os.environ, RT_B200_AUX_DELAY_MS="300")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-800:]
    (s1, r1, k1), (s2, r2, k2) = (tuple(int(v) for v in g.split(":")) for g in out.stdout.strip().splitlines()[-1].split())
    assert s1 == 1 and 0 < r1 < 65536 and k1 == 2, (s1, r1, k1)
    assert s2 == 1 and r2 == 0xffffffff and k2 == 2, (s2, r2, k2)


@pytest.mark.gpu
def test_refusals_then_a_valid_call(ctx, rt):
    from rt_b200 import _abi

    sp, tr = rt.scenes.synthetic_spheres(32, 5), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr).wait_ready()
    w, h, div = 64, 40, 10
    p = _params(rt, w, h, div, spp=2, max_bounces=3, seed=4)
    L = _abi.lib()
    band = (h // div) * w * 3

    def raw(nos, n=None, out_len=None, params=p, out=True):
        arr = (C.c_uint32 * max(1, len(nos)))(*nos)
        buf = (C.c_uint8 * max(1, len(nos) * band))()
        return L.rt_render_divisions(ctx._h, sc._h, C.byref(params), arr if nos is not None else None,
                                     len(nos) if n is None else n, buf if out else None,
                                     len(nos) * band if out_len is None else out_len, None)

    def refused(rc):
        assert rc == _abi.RT_ERR_INVALID_ARG, rc
        _check(ctx, sc, p, [7, 1, 4])  # the context renders on as if nothing had been tried

    try:
        refused(L.rt_render_divisions(ctx._h, sc._h, C.byref(p), None, 2, (C.c_uint8 * (2 * band))(), 2 * band, None))
        refused(L.rt_render_divisions(ctx._h, None, C.byref(p), (C.c_uint32 * 1)(0), 1, (C.c_uint8 * band)(), band, None))
        refused(L.rt_render_divisions(ctx._h, sc._h, None, (C.c_uint32 * 1)(0), 1, (C.c_uint8 * band)(), band, None))
        refused(raw([1, 2], out=False))                       # no destination
        refused(raw([], n=0, out_len=0))                      # n == 0
        refused(raw([3, 10]))                                 # division number >= divisions
        refused(raw([3, 5, 3]))                               # listed twice
        refused(raw([3, 5], out_len=2 * band - 3))            # wrong out_len
        refused(raw([3, 5], out_len=3 * band))
        refused(raw([0, 1], params=_params(rt, w, h, 7, spp=2, max_bounces=3, seed=4)))  # 40 rows in 7 divisions
        with pytest.raises(rt.RtError) as e:
            ctx.render_divisions(sc, p, [2, -1])
        assert e.value.status == _abi.RT_ERR_INVALID_ARG
        with pytest.raises(rt.RtError) as e:
            ctx.render_divisions(sc, p, [2, 11])
        assert e.value.status == _abi.RT_ERR_INVALID_ARG
        _check(ctx, sc, p, [9, 0])
    finally:
        sc.close()


@pytest.mark.gpu
def test_worker_render_many(rt):
    """Worker.render_many gives the slices render gives, a duplicate included, with one scene upload."""
    from rt_b200 import slave, wire

    sp, tr = rt.scenes.synthetic_spheres(48, 6), rt.scenes.ground_plane()
    world = wire.World(sp, tr, np.arange(len(sp) + len(tr), dtype=np.uint32))
    meta = wire.RenderMeta(60, 80, 5, "123e4567-e89b-12d3-a456-426614174000")
    wk = slave.Worker(0, spp=3, max_bounces=4, seed=2)
    try:
        infos = [wire.RenderInfo(world, meta, d) for d in (4, 1, 4, 2)]
        many = wk.render_many(infos)
        assert [s.division_no for s in many] == [4, 1, 4, 2] and all(s.id == meta.id for s in many)
        for s, i in zip(many, infos):
            assert np.array_equal(s.image, wk.render(i).image)
        assert wk.scene_uploads == 1
    finally:
        wk.close()
