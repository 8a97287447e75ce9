"""OBJ ingest on the device: rt_obj_build_world turns the controller's /upload body (OBJ ++ MTL) into the triangle
array obj.build_world returns, bit for bit, or declines (and the host code decides, with its own errors)."""
import ctypes as C
import os
import random
import struct

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
NAMES = ["rt_obj_max_triangles", "rt_obj_build_world"]
MTL = b"newmtl m\nKd 0.8 0.2 0.1\nNs 250\n"


def _outcome(data, obj_size, **kw):
    """build_world's result as bytes, or its error (type, text)."""
    from rt_b200 import obj

    try:
        with np.errstate(over="ignore"):
            return ("ok", obj.build_world(data, obj_size, **kw).tobytes())
    except Exception as e:  # noqa: BLE001 - the host path's exact exception is what must be kept
        return ("error", type(e).__name__, str(e))


def _host_bodies():
    """The bodies of test_host's OBJ test, valid and invalid, as (data, obj_size)."""
    from test_host import mesh_scene_obj

    o = b"usemtl m\nv 0 0 -3\nv 1 0 -3\nv 0 1 -3\nv 1 1 -3\nf 1 2 3\nf 2/1/1 4/2/2 -2//3\n"
    q = b"usemtl m\nv 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nv 2 2 2\nv 3 3 3\nf 1 2 3 4\nf 5 6 1\n"
    bad = b"v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n"
    return [mesh_scene_obj(), (o + MTL, len(o)), (q + MTL, len(q)), (bad, 36), (o + MTL, len(o) + len(MTL) + 5),
            (o + MTL, -1)]


# ---------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------
def test_exports_declared_and_exported(rt):
    from rt_b200 import _abi

    header = open(os.path.join(ROOT, "include", "rt_b200.h")).read()
    L = _abi.lib()
    for name in NAMES:
        assert f" {name}(" in header and name in _abi.EXPORTS and hasattr(L, name), name
    assert L.rt_obj_max_triangles(0) == 0 and L.rt_obj_max_triangles(7) == 1 and L.rt_obj_max_triangles(600) == 100


def _oracle_parser(data, obj_size):
    """What a correct device parser returns: the host's array, None where the host fails."""
    from rt_b200 import obj

    try:
        with np.errstate(over="ignore"):
            return obj.build_world(data, obj_size)
    except Exception:  # noqa: BLE001
        return None


@pytest.mark.parametrize("parser", ["declining", "oracle"])
def test_build_world_unchanged_with_a_parser(rt, parser):
    p = (lambda d, n: None) if parser == "declining" else _oracle_parser
    bodies = _host_bodies() + [(b, n) for _, b, n in _edge_bodies()] + [(b, n) for b, n in DECLINED.values()]
    for data, n in bodies:
        assert _outcome(data, n, parser=p) == _outcome(data, n), (data[:80], n)


class _StandIn:
    """A worker without a GPU context: renders a slice whose bytes encode the triangle count."""

    def __init__(self):
        self.worlds = []

    def render(self, info):
        from rt_b200 import wire

        m = info.render_meta
        self.worlds.append(info.world.triangles.tobytes())
        img = np.full((m.height // m.divisions, m.width, 3), len(info.world.triangles) % 251, dtype=np.uint8)
        return wire.ImageSlice(info.division_no, img.reshape(-1), m.id)


def test_controller_upload_with_a_stand_in_worker(rt):
    from rt_b200 import controller, obj
    from test_host import mesh_scene_obj

    data, n = mesh_scene_obj()
    w = _StandIn()
    c = controller.Controller(worker=w, width=64, height=40, divisions=4)
    assert c._obj_parser() is None
    jpeg, is_img = c.poll(c.upload(data, n))
    assert is_img and jpeg == controller.encode_jpeg(np.full((40, 64, 3), 82, np.uint8), 90)
    assert w.worlds == [obj.build_world(data, n).tobytes()] * 4
    with pytest.raises(obj.ObjError):
        c.upload(b"v 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3\n", 36)


# ---------------------------------------------------------------------------------------------------
# Bodies
# ---------------------------------------------------------------------------------------------------
def _edge_bodies():
    """(name, data, obj_size): line ends, whitespace and comments the host's splitlines / split / '#' rules allow."""
    o = (b"# comment only\r\n\r\nmtllib x.mtl\rusemtl m\x0bv 0 0 -3#c\x0cv\t1 0 -3 extra tokens\x1cv 0\x1f1 -3\x1d"
         b"vt 0 1\x1evn 0 0 1\n  \t\ns off\nv 1 1 -3 # tail\nf 1 2 3#x\nf\t2/1/1  4/2/2\t-2//3 \n"
         b"g two\nf 1 2 3 4\no three\nf 3 2 1 4 1\nusemtl n\nf 4 3 2\n")
    m = (b"newmtl m\r\nKd 0.5 0.25\nKd 0.8 0.2 0.1 9\r\nNs 250 x\nnewmtl n\nKd 1 1 1\nnewmtl m\nKd .5 5. +1e-1\n"
         b"# Kd 0 0 0\nNs 7\n")
    crlf = b"usemtl m\r\nv 0 0 0\r\nv 1 0 0\r\nv 0 1 0\r\nf 1 2 3\r\n"
    lone_cr = b"usemtl m\rv 0 0 0\rv 1 0 0\rv 0 1 0\rf -3 -2 -1\r"
    two_corner_model = b"usemtl m\nv 0 0 0\nv 1 0 0\nv 0 1 0\nf 1 2 3 1 2\ng x\nf 3 2 1\n"
    return [("edges", o + m, len(o)), ("crlf", crlf + b"newmtl m\r\nKd 1 0 0\r\n", len(crlf)),
            ("lone_cr", lone_cr + b"newmtl m\rNs 10\r", len(lone_cr)),
            ("two_corner_model", two_corner_model + MTL, len(two_corner_model)),
            ("no_faces", b"usemtl m\nv 0 0 0\n" + MTL, 17), ("empty", b"", 0), ("mtl_only", MTL, 0)]


def _grid_obj(q, seed):
    """A (q + 1)^2-vertex height field, 2 q^2 triangles, in several models and materials: o / g / usemtl interleaved,
    a usemtl kept across g, f lines of 3 and 4 corners (a quad runs into the next face), several index forms."""
    rng = np.random.default_rng(seed)
    xs = np.linspace(-12, 12, q + 1, dtype=np.float32)
    V = np.stack(np.meshgrid(xs, xs, indexing="ij"), -1).reshape(-1, 2)
    V = np.concatenate([V, np.sin(V[:, :1]).astype(np.float32)], 1)
    idx = np.arange((q + 1) ** 2).reshape(q + 1, q + 1) + 1
    a, b, c, d = idx[:-1, :-1].ravel(), idx[1:, :-1].ravel(), idx[1:, 1:].ravel(), idx[:-1, 1:].ravel()
    corners = np.stack([a, b, c, a, c, d], 1).reshape(-1)
    lines = ["v %.9g %.9g %.9g" % tuple(v) for v in V.tolist()]
    i, k, n_mat = 0, 0, 5
    while i < len(corners):
        r = rng.random()
        if r < 0.3:
            lines.append("usemtl mat%d" % rng.integers(n_mat))
        elif r < 0.5:
            lines.append("g part%d" % k)
        elif r < 0.6:
            lines.append("o obj%d" % k)
        k += 1
        if k == 1:
            lines.append("usemtl mat0")
        for _ in range(int(rng.integers(1, 4000))):
            m = 4 if rng.random() < 0.1 else 3
            cs = corners[i:i + m].tolist()
            if not cs:
                break
            i += len(cs)
            form = rng.integers(3)
            cs = [str(x) if form == 0 else "%d/%d" % (x, x) if form == 1 else "%d//7" % x for x in cs]
            lines.append("f " + " ".join((cs + [cs[-1]] * 2)[:max(3, len(cs))]))  # the mesh's last face may be short
    o = ("\n".join(lines) + "\n").encode()
    m = "".join("newmtl mat%d\nKd %.6g %.6g %.6g\nNs %d\n" % (j, *rng.uniform(0, 1, 3), rng.integers(0, 1000))
                for j in range(n_mat)).encode()
    return o + m, len(o)


def _fuzz_tokens(n, seed):
    """Number tokens in the device grammar whose host value is finite: f32 halfway points written in decimal (where
    rounding to f64 first matters), 19-digit integers just off a halfway point, subnormals, signed zeros, '+', '.5',
    '5.', leading zeros, 17 to 19 digits, and FLT_MAX with half an ulp either side."""
    rng = random.Random(seed)
    toks = ["-0", "-0.0", "+0", "0e0", ".5", "5.", "+1.5", "-.25", "007.5", "+.0e-3", "1E5", "1e+5", "1e-50", "-1e-50",
            "1.401298464324817e-45", "7.006492321624085e-46", "7.006492321624087e-46", "1e-45", "-2.8e-45",
            "1.1754942e-38", "3.4028234663852886e38", "3.40282356779733e38", "-3.40282356779733e38",
            "16777217", "16777219", "33554434", "9007199254740993",
            "1.0000000596046448", "1.00000005960464477", "0.1", "0.30000000000000004", "9999999999999999999"]
    while len(toks) < n:
        r = rng.random()
        if r < 0.3:  # the midpoint of two adjacent f32 values, as the shortest f64 decimal (it is exactly a double)
            f = np.float32(rng.uniform(1, 10) * 10.0 ** rng.randint(-44, 37))
            g = np.nextafter(f, np.float32(np.inf))
            if np.isfinite(g):
                t = repr((float(f) + float(g)) / 2)
                toks.append(("-" if rng.random() < 0.5 else "") + t)
        elif r < 0.45:  # a 17..19-digit integer within a few units of an f32 midpoint above 2^53
            e = rng.randint(54, 62)
            f = (rng.getrandbits(24) | 1 << 23) << (e - 23)
            t = str(f + (1 << (e - 24)) + rng.randint(-3, 3))
            toks.append(t if rng.random() < 0.5 else "0" * rng.randint(1, 3) + t)
        elif r < 0.65:
            x = struct.unpack("<f", struct.pack("<I", rng.getrandbits(32)))[0]
            if np.isfinite(x):
                toks.append("%.*e" % (rng.randint(0, 18), x))
        elif r < 0.8:
            nd = rng.randint(1, 19)
            s = str(rng.randint(10 ** (nd - 1), 10 ** nd - 1))
            p = rng.randint(0, nd)
            toks.append(("+" if rng.random() < 0.2 else "") + s[:p] + "." + s[p:])
        else:
            toks.append("%de%d" % (rng.randint(1, 10 ** rng.randint(1, 18)), rng.randint(-60, 30)))
    with np.errstate(over="ignore"):
        return [t for t in toks if np.isfinite(np.float32(t))]


def _fuzz_body(n_tokens, seed):
    """Vertices from the fuzzed tokens, each vertex used by a face; materials whose Kd and Ns are fuzzed too."""
    toks = _fuzz_tokens(n_tokens, seed)
    mt, toks = toks[: len(toks) // 5], toks[len(toks) // 5:]
    o, n_mat = [], len(mt) // 4
    for i in range(0, len(toks) - 8, 9):
        o.append("usemtl k%d" % (i // 9 % n_mat))
        o += ["v %s %s %s" % tuple(toks[j:j + 3]) for j in range(i, i + 9, 3)]
        o.append("f -3 -2 -1")
    m = "".join("newmtl k%d\nKd %s %s %s\nNs %s\n" % (j, *mt[4 * j:4 * j + 3], mt[4 * j + 3]) for j in range(n_mat))
    o = ("\n".join(o) + "\n").encode()
    return o + m.encode(), len(o)


def _body(o, m=MTL):
    return o + m, len(o)


_TRI = b"usemtl m\nv 0 0 0\nv 1 0 0\nv 0 1 0\n"
DECLINED = {
    "non_ascii": _body(_TRI + b"f 1 2 3 # caf\xc3\xa9\n"),
    "u0085_in_comment": _body(_TRI + b"f 1 2 3 # a\xc2\x85f 1 2 3\n"),
    "inf": _body(_TRI + b"v inf 0 0\nf 1 2 4\n"),
    "nan": _body(_TRI + b"v 0 nan 0\nf 1 2 4\n"),
    "underscore": _body(_TRI + b"v 1_0 0 0\nf 1 2 4\n"),
    "twenty_digits": _body(_TRI + b"v 1.0000000000000000001 0 0\nf 1 2 4\n"),
    "overflow_to_inf": _body(_TRI + b"v 1e39 0 0\nf 1 2 4\n"),
    "flt_max_half_ulp": _body(_TRI + b"v 3.4028235677973366e38 0 0\nf 1 2 4\n"),
    "index_0": _body(_TRI + b"f 0 1 2\n"),
    "forward_reference": _body(_TRI + b"f 1 2 4\nv 1 1 1\n"),
    "index_out_of_range": _body(_TRI + b"f 1 2 -4\n"),
    "empty_index": _body(_TRI + b"f //1 2 3\n"),
    "v_two_coordinates": _body(_TRI + b"v 1 2\nf 1 2 3\n"),
    "f_two_corners": _body(_TRI + b"f 1 2\n"),
    "no_material": _body(_TRI[9:] + b"f 1 2 3\n"),
    "unknown_usemtl": _body(_TRI + b"f 1 2 3\nusemtl nope\nf 1 2 3\n"),
    "bad_kd_unused_material": _body(_TRI + b"f 1 2 3\n", MTL + b"newmtl unused\nKd 1 x 1\n"),
    "newmtl_order": _body(_TRI + b"f 1 2 3\n", MTL + b"newmtl __order__\n"),
    "usemtl_order": _body(_TRI + b"f 1 2 3\nusemtl __order__\nf 1 2 3\n"),
}


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def _parity(ctx, data, obj_size):
    from rt_b200 import obj

    got = ctx.parse_obj(data, obj_size)
    assert got is not None, ctx._lib.rt_last_error(ctx._h)
    with np.errstate(over="ignore"):
        want = obj.build_world(data, obj_size)
    assert got.dtype == want.dtype and got.tobytes() == want.tobytes()
    return got


@pytest.mark.gpu
def test_host_test_bodies(ctx):
    for data, n in _host_bodies()[:3]:
        _parity(ctx, data, n)


@pytest.mark.gpu
@pytest.mark.parametrize("name", [e[0] for e in _edge_bodies()])
def test_line_ends_whitespace_comments(ctx, name):
    _, data, n = next(e for e in _edge_bodies() if e[0] == name)
    t = _parity(ctx, data, n)
    if name == "edges":
        # the second newmtl m resets it: Kd from its own block, Ns 7; usemtl m holds across g and o
        assert len(t) == 5 and t["albedo"][3].tolist() == [0.5, 5.0, np.float32(0.1)] and t["albedo"][4].tolist() == [1] * 3
        assert t["roughness"][0] == np.float32(7) / np.float32(1000)
    if name == "two_corner_model":
        assert len(t) == 2
    if name in ("no_faces", "empty", "mtl_only"):
        assert len(t) == 0


@pytest.mark.gpu
def test_mesh_of_a_million_triangles(ctx):
    data, n = _grid_obj(724, 3)
    t = _parity(ctx, data, n)
    assert len(t) >= 1_000_000 and len(np.unique(t["roughness"])) > 1


@pytest.mark.gpu
def test_number_fuzz(ctx):
    data, n = _fuzz_body(100_000, 7)
    t = _parity(ctx, data, n)
    assert len(t) > 8000


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(DECLINED))
def test_declines_then_host_path(ctx, case):
    from rt_b200 import _abi, scenes

    data, n = DECLINED[case]
    assert ctx.parse_obj(data, n) is None
    out, cnt = np.empty(16, scenes.TRIANGLE_DTYPE), C.c_uint32()
    assert ctx._lib.rt_obj_build_world(ctx._h, data, len(data), n, out.ctypes.data, 16, C.byref(cnt)) \
        == _abi.RT_ERR_UNSUPPORTED
    assert _outcome(data, n, parser=ctx.parse_obj) == _outcome(data, n)


@pytest.mark.gpu
def test_refusals_then_valid(ctx):
    from rt_b200 import _abi, scenes

    data, n = _host_bodies()[1]
    L = ctx._lib
    cap = L.rt_obj_max_triangles(n)
    out, cnt = np.empty(cap, scenes.TRIANGLE_DTYPE), C.c_uint32()
    bad = _abi.RT_ERR_INVALID_ARG
    assert L.rt_obj_build_world(ctx._h, None, len(data), n, out.ctypes.data, cap, C.byref(cnt)) == bad
    assert L.rt_obj_build_world(ctx._h, data, len(data), n, None, cap, C.byref(cnt)) == bad
    assert L.rt_obj_build_world(ctx._h, data, len(data), n, out.ctypes.data, cap, None) == bad
    assert L.rt_obj_build_world(ctx._h, data, len(data), len(data) + 1, out.ctypes.data, 1 << 20, C.byref(cnt)) == bad
    assert L.rt_obj_build_world(ctx._h, data, len(data), n, out.ctypes.data, cap - 1, C.byref(cnt)) == bad
    assert L.rt_obj_build_world(ctx._h, data, len(data), n, out.ctypes.data, cap, C.byref(cnt)) == _abi.RT_OK
    assert cnt.value == 2
    _parity(ctx, data, n)


@pytest.mark.gpu
def test_scratch_grows_then_small_body_and_other_entries_unchanged(ctx, rt):
    """The parse's scratch grows with the body and is kept; a small body after a large one, a render and a wire parse
    after an OBJ parse on the same context give what they gave before it."""
    from rt_b200 import wire
    from test_host import mesh_scene_obj

    data, n = mesh_scene_obj()
    tris = obj_tris = _parity(ctx, data, n)
    sc = ctx.scene(None, tris)
    p = rt.make_params(96, 64, spp=2, max_bounces=4)
    before = ctx.render_frame(sc, p).copy()
    meta = wire.RenderMeta(64, 96, 4, "123e4567-e89b-12d3-a456-426614174000")
    body = wire.render_info_to_json(None, tris, meta, 1).encode()
    start = body.index(b"[")
    w0, e0 = ctx.parse_world_json(body, start)
    _parity(ctx, *_grid_obj(128, 1))
    assert np.array_equal(ctx.render_frame(sc, p), before)
    w1, e1 = ctx.parse_world_json(body, start)
    assert e1 == e0 and w1.triangles.tobytes() == w0.triangles.tobytes() == obj_tris.tobytes()
    sc.close()
    assert _parity(ctx, data, n).tobytes() == obj_tris.tobytes()
    _parity(ctx, *_host_bodies()[2])


def _poll_both_ways(monkeypatch, make_controller, data, n):
    """/poll's bytes for one upload with the device parse, then with the host parse."""
    from rt_b200 import controller

    out = []
    for device in (True, False):
        c = make_controller()
        try:
            if not device:
                monkeypatch.setattr(c, "_obj_parser", lambda: None)
            else:
                assert c._obj_parser() is not None
            out.append(c.poll(c.upload(data, n)))
        finally:
            c.close()
    assert out[0][1] and out[0] == out[1]
    return controller


@pytest.mark.gpu
def test_controller_poll_same_bytes_worker_mode(monkeypatch):
    from rt_b200 import controller, slave

    data, n = _grid_obj(48, 5)
    wk = slave.Worker(0, spp=2, max_bounces=4, seed=3)
    try:
        _poll_both_ways(monkeypatch, lambda: controller.Controller(worker=wk, width=160, height=90, divisions=10),
                        data, n)
    finally:
        wk.close()


@pytest.mark.gpu
def test_controller_poll_same_bytes_devices_mode(monkeypatch):
    import torch

    from rt_b200 import controller

    data, n = _grid_obj(48, 6)
    lists = [[0, 0, 0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for devs in lists:
        _poll_both_ways(monkeypatch, lambda: controller.Controller(devices=devs, width=160, height=90, divisions=10,
                                                                   spp=2, max_bounces=4, seed=3), data, n)
