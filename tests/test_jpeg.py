"""JPEG on the device (rt_jpeg_encode, rt_render_frame_jpeg): the bytes are libjpeg's defaults at the same quality, i.e.
what PIL's save(format="JPEG", quality=q) writes and what the controller's /poll returns.  The CPU reference
(tests/jpeg_oracle.py) is checked against PIL here first; the device encoder is checked against both."""
import ctypes as C
import glob
import io
import os

import numpy as np
import pytest

from conftest import assert_parity
from jpeg_oracle import oracle_jpeg

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))

# 1x1 .. 17x17: partial MCUs; 40x24: an odd count of luma blocks per row (right-edge dummies); 61x37: odd w and h;
# 320x180, 1920x1080: even h with h % 16 != 0 (bottom dummy blocks, repeated chroma rows); 1000x1: one row
SIZES = [(1, 1), (7, 5), (8, 8), (16, 16), (17, 17), (40, 24), (61, 37), (320, 180), (1920, 1080), (1000, 1)]
QUALITIES = [1, 10, 49, 50, 51, 75, 90, 100]
SMALL = [s for s in SIZES if s[0] * s[1] <= 320 * 180]


def pil_jpeg(frame, quality):
    from PIL import Image

    buf = io.BytesIO()
    Image.fromarray(np.ascontiguousarray(frame), "RGB").save(buf, format="JPEG", quality=quality)
    return buf.getvalue()


def contents(w, h, seed=0):
    """name → uint8 (h, w, 3): uniform noise (large coefficients, many stuffed 0xFF), flat colour (EOB-only blocks),
    gradients, pure 0 / 255 primaries."""
    rng = np.random.default_rng(seed + w * 7919 + h)
    yy, xx = np.mgrid[0:h, 0:w]
    grad = np.stack([xx * 255 // max(w - 1, 1), yy * 255 // max(h - 1, 1), (xx + 2 * yy) % 256], -1).astype(np.uint8)
    prim = np.zeros((h, w, 3), np.uint8)
    prim[:, : (w + 1) // 2, 0] = 255
    prim[h // 2:, :, 2] = 255
    prim[::3, ::5, 1] = 255
    return {
        "noise": rng.integers(0, 256, (h, w, 3), dtype=np.uint8),
        "flat": np.full((h, w, 3), (200, 30, 90), np.uint8),
        "gradient": grad,
        "primaries": prim,
    }


def golden_frames():
    return {os.path.basename(f): np.load(f) for f in sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "*.npy")))}


# ---------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h", SMALL)
def test_oracle_equals_pil(w, h):
    for q in QUALITIES:
        for name, img in contents(w, h).items():
            assert oracle_jpeg(img, w, h, q) == pil_jpeg(img, q), (w, h, q, name)


def test_oracle_equals_pil_1080p():
    for name, img in contents(1920, 1080).items():
        for q in ((90, 100) if name == "noise" else (1, 90)):
            assert oracle_jpeg(img, 1920, 1080, q) == pil_jpeg(img, q), (q, name)


def test_oracle_equals_pil_golden():
    for name, img in golden_frames().items():
        h, w = img.shape[:2]
        for q in QUALITIES:
            assert oracle_jpeg(img, w, h, q) == pil_jpeg(img, q), (name, q)


def test_bound_holds_for_noise_at_q100(rt):
    from rt_b200 import _abi

    L = _abi.lib()
    for w, h in SIZES:
        img = contents(w, h)["noise"]
        n = len(oracle_jpeg(img, w, h, 100))
        assert n <= L.rt_jpeg_bound(w, h), (w, h, n)
    # every byte 0xFF-stuffed is the worst case the bound allows for: it still leaves room
    assert L.rt_jpeg_bound(1920, 1080) == 623 + 4 + 120 * 68 * 2490


def test_entry_points_declared_and_exported(rt):
    from rt_b200 import _abi

    header = open(os.path.join(ROOT, "include", "rt_b200.h")).read()
    for name in ("rt_jpeg_bound", "rt_jpeg_encode", "rt_render_frame_jpeg"):
        assert f" {name}(" in header, name
        assert name in _abi.EXPORTS and hasattr(_abi.lib(), name), name


def test_null_handles_refused(rt):
    from rt_b200 import _abi

    L = _abi.lib()
    rgb = (C.c_uint8 * 3)()
    out = (C.c_uint8 * 4096)()
    n = C.c_size_t(0)
    assert L.rt_jpeg_encode(None, rgb, 1, 1, 90, out, 4096, C.byref(n), None) == _abi.RT_ERR_INVALID_ARG
    p = rt.make_params(8, 8)
    assert L.rt_render_frame_jpeg(None, None, 1, C.byref(p), 90, out, 4096, C.byref(n), None) == _abi.RT_ERR_INVALID_ARG
    ch = (C.c_void_p * 1)(None)
    assert L.rt_render_frame_jpeg(ch, ch, 1, C.byref(p), 90, out, 4096, C.byref(n), None) == _abi.RT_ERR_INVALID_ARG
    assert n.value == 0


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", SIZES)
def test_encode_equals_pil_and_oracle(ctx, w, h):
    for name, img in contents(w, h).items():
        for q in QUALITIES:
            got = ctx.encode_jpeg(img, q)
            assert got == pil_jpeg(img, q), (w, h, q, name)
            if (w, h) in SMALL:
                assert got == oracle_jpeg(img, w, h, q), (w, h, q, name)


@pytest.mark.gpu
def test_encode_golden_frames(ctx):
    for name, img in golden_frames().items():
        h, w = img.shape[:2]
        for q in QUALITIES:
            assert ctx.encode_jpeg(img, q) == pil_jpeg(img, q) == oracle_jpeg(img, w, h, q), (name, q)


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(3840, 2160), (7680, 4320)])
def test_encode_large_noise(ctx, w, h):
    img = np.random.default_rng(w).integers(0, 256, (h, w, 3), dtype=np.uint8)
    for q in (90, 100):
        got, ms = ctx.encode_jpeg(img, q, want_ms=True)
        assert ms > 0
        assert got == pil_jpeg(img, q), (w, h, q)


@pytest.mark.gpu
def test_sizes_grow_then_shrink(ctx):
    """The scratch grows with the frame; a smaller frame after a larger one gives the same bytes as before."""
    order = [(17, 17), (320, 180), (1920, 1080), (61, 37), (320, 180), (1, 1), (1920, 1080), (17, 17)]
    first = {}
    for w, h in order:
        img = contents(w, h)["noise"]
        got = ctx.encode_jpeg(img, 90)
        assert got == first.setdefault((w, h), got)
        assert got == pil_jpeg(img, 90), (w, h)


@pytest.mark.gpu
def test_refusals_then_valid_call(rt, ctx):
    from rt_b200 import _abi

    L = _abi.lib()
    img = contents(40, 24)["gradient"]
    want = pil_jpeg(img, 90)
    cap = L.rt_jpeg_bound(40, 24)
    out = np.zeros(cap, np.uint8)
    n = C.c_size_t(0)
    rgb = img.ctypes.data_as(C.c_void_p)
    o = out.ctypes.data_as(C.c_void_p)

    def valid():
        m = C.c_size_t(0)
        assert L.rt_jpeg_encode(ctx._h, rgb, 40, 24, 90, o, cap, C.byref(m), None) == 0
        assert out[: m.value].tobytes() == want

    bad = [
        (ctx._h, None, 40, 24, 90, o, cap, C.byref(n), None),        # NULL frame
        (ctx._h, rgb, 40, 24, 90, None, cap, C.byref(n), None),      # NULL out
        (ctx._h, rgb, 40, 24, 90, o, cap, None, None),               # NULL out_len
        (ctx._h, rgb, 0, 24, 90, o, cap, C.byref(n), None),          # width 0
        (ctx._h, rgb, 40, 0, 90, o, cap, C.byref(n), None),          # height 0
        (ctx._h, rgb, 65536, 1, 90, o, 1 << 40, C.byref(n), None),   # above the SOF field
        (ctx._h, rgb, 1, 65536, 90, o, 1 << 40, C.byref(n), None),
        (ctx._h, rgb, 40, 24, 0, o, cap, C.byref(n), None),          # quality outside 1..100
        (ctx._h, rgb, 40, 24, 101, o, cap, C.byref(n), None),
        (ctx._h, rgb, 40, 24, 90, o, cap - 1, C.byref(n), None),     # below rt_jpeg_bound
    ]
    for args in bad:
        assert L.rt_jpeg_encode(*args) == _abi.RT_ERR_INVALID_ARG, args
        valid()
    # rt_render_frame_jpeg: its own refusals and the render's
    sp, tr = rt.scenes.synthetic_spheres(16, 2), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr)
    try:
        p = rt.make_params(40, 24, spp=1, max_bounces=2)
        one = (C.c_void_p * 1)(ctx._h)
        scs = (C.c_void_p * 1)(sc._h)
        for q, c, params in [(0, cap, p), (101, cap, p), (90, cap - 1, p), (90, cap, rt.make_params(0, 24, spp=1))]:
            assert L.rt_render_frame_jpeg(one, scs, 1, C.byref(params), q, o, c, C.byref(n), None) == _abi.RT_ERR_INVALID_ARG
            valid()
        assert L.rt_render_frame_jpeg(one, scs, 1, C.byref(p), 90, None, cap, C.byref(n), None) == _abi.RT_ERR_INVALID_ARG
        assert ctx.render_frame_jpeg(sc, p) == pil_jpeg(ctx.render_frame(sc, p), 90)
    finally:
        sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("isect", ["brute", "bvh"])
def test_render_frame_jpeg_equals_pil_of_render_frame(rt, ctx, isect):
    sp, tr = rt.scenes.synthetic_spheres(64, 3), rt.scenes.ground_plane()
    sc = ctx.scene(sp, tr)
    try:
        for (w, h), spp in [((320, 180), 2), ((61, 37), 1), ((1920, 1080), 1)]:
            p = rt.make_params(w, h, spp=spp, max_bounces=4, seed=5,
                               intersector=rt.INTERSECT_BRUTE if isect == "brute" else rt.INTERSECT_BVH)
            frame = ctx.render_frame(sc, p)
            for q in (75, 90):
                got, st = ctx.render_frame_jpeg(sc, p, quality=q, want_stats=True)
                assert got == pil_jpeg(frame, q), (w, h, q)
                assert st["primary"] == w * h * spp and st["total_ms"] >= st["kernel_ms"] > 0
    finally:
        sc.close()


@pytest.mark.gpu
def test_render_frame_jpeg_multi_three_contexts(rt):
    sp, tr = rt.scenes.synthetic_spheres(48, 8), rt.scenes.ground_plane()
    cs = [rt.Context(0) for _ in range(3)]
    try:
        scs = [c.scene(sp, tr) for c in cs]
        for w, h in [(320, 180), (1920, 1080)]:
            p = rt.make_params(w, h, spp=2, max_bounces=4, seed=7)
            frame = rt.render_frame_multi(cs, scs, p)
            assert rt.render_frame_jpeg(cs, scs, p) == pil_jpeg(frame, 90)
        for s in scs:
            s.close()
    finally:
        for c in cs:
            c.close()


@pytest.mark.gpu
def test_render_frame_jpeg_two_devices(rt):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    from rt_b200 import multi

    sp, tr = rt.scenes.synthetic_spheres(64, 3), rt.scenes.ground_plane()
    m = multi.MultiDeviceRenderer([0, 1])
    try:
        scs = m.scenes(sp, tr)
        p = rt.make_params(1920, 1080, spp=2, max_bounces=4, seed=3)
        assert m.render_jpeg(scs, p) == pil_jpeg(m.render(scs, p), 90)
        for s in scs:
            s.close()
    finally:
        m.close()


@pytest.mark.gpu
def test_render_after_encode_matches_oracle(rt, ctx, O):
    """An encode overwrites the context's staging frame; the next render is still the oracle's, byte for byte."""
    sp, tr = rt.scenes.synthetic_spheres(64), rt.scenes.ground_plane()
    w, h, spp, mb = 128, 72, 2, 5
    ctx.encode_jpeg(contents(1920, 1080)["noise"], 90)
    sc = ctx.scene(sp, tr)
    try:
        ref, _ = O.render_frame(sp, tr, w, h, spp, mb)
        img = ctx.render_frame(sc, rt.make_params(w, h, spp=spp, max_bounces=mb))
        assert_parity(img, ref)
        assert ctx.render_frame_jpeg(sc, rt.make_params(w, h, spp=spp, max_bounces=mb)) == pil_jpeg(ref, 90)
    finally:
        sc.close()


@pytest.mark.gpu
def test_controller_poll_worker_and_devices_modes(rt):
    """/poll returns PIL's JPEG(90) of the stitched frame, now encoded on the GPU in both in-process modes."""
    from rt_b200 import controller, obj, slave, wire
    from test_host import mesh_scene_obj

    data, n = mesh_scene_obj()
    tris = obj.build_world(data, n)
    world = wire.World(np.zeros(0, wire.SPHERE_DTYPE), tris, np.arange(len(tris), dtype=np.uint32))
    wk = slave.Worker(0, spp=2, max_bounces=4, seed=11)
    try:
        c = controller.Controller(worker=wk, width=320, height=180, divisions=20)
        job = c.upload(data, n)
        jpeg, is_img = c.poll(job)
        meta = wire.RenderMeta(180, 320, 20, "00000000-0000-4000-8000-00000000000c")
        frame = np.concatenate([wk.render(wire.RenderInfo(world, meta, d)).image.reshape(9, 320, 3) for d in range(20)])
        assert is_img and jpeg == pil_jpeg(frame, 90)
    finally:
        wk.close()
    c = controller.Controller(devices=[0, 0], width=320, height=180, divisions=20, spp=2, max_bounces=4, seed=11)
    try:
        assert c.poll(c.upload(data, n)) == (pil_jpeg(frame, 90), True)
        meta = wire.RenderMeta(180, 320, 20, "00000000-0000-4000-8000-00000000000d")
        slices = c._render_all_gpus(tris, meta)
        assert np.array_equal(np.concatenate([s.image.reshape(9, 320, 3) for s in slices]), frame)
    finally:
        c.close()
