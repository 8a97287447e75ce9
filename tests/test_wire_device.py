"""The slave's wire format on the device: rt_world_parse_json reads the world of a RenderInfo body into the arrays
wire.parse_render_info builds, bit for bit, or declines (and the host parser decides); rt_render_divisions_json writes the
ImageSlice bodies, byte for byte wire.ImageSlice(...).to_json()."""
import ctypes as C
import json
import os
import random
import struct
import threading
import urllib.request
from collections import OrderedDict

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
ID = "123e4567-e89b-12d3-a456-426614174000"
META = '{"height":40,"width":16,"divisions":4,"id":"%s"}' % ID
NAMES = ["rt_world_json_max_objects", "rt_world_parse_json", "rt_slice_json_bound", "rt_render_divisions_json"]


def _body(world_text, meta=META, division_no="0"):
    return ('{"world":%s,"render_meta":%s,"division_no":%s}' % (world_text, meta, division_no)).encode()


def _outcome(body, **kw):
    """parse_render_info's result as comparable bytes, or its error (type, text)."""
    from rt_b200 import wire

    try:
        info = wire.parse_render_info(body, **kw)
    except Exception as e:  # noqa: BLE001 - the host path's exact exception is what must be kept
        return ("error", type(e).__name__, str(e))
    w = info.world
    return ("ok", w.spheres.dtype.str, w.spheres.tobytes(), w.triangles.tobytes(), w.world_index.dtype.str,
            w.world_index.tobytes(), info.render_meta, info.division_no)


# ---------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------
def test_exports_declared_and_exported(rt):
    from rt_b200 import _abi

    header = open(os.path.join(ROOT, "include", "rt_b200.h")).read()
    L = _abi.lib()
    for name in NAMES:
        assert f" {name}(" in header and name in _abi.EXPORTS and hasattr(L, name), name


def test_pow5_table_is_generated(rt):
    """rt_wire_pow5.h is exactly what its generator writes."""
    import importlib.util

    csrc = os.path.join(ROOT, "ray-tracer-s8_b200", "csrc")
    spec = importlib.util.spec_from_file_location("gen_pow5", os.path.join(csrc, "gen_pow5.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    assert open(os.path.join(csrc, "rt_wire_pow5.h")).read() == gen.header()
    assert next(gen.entries()) == (-342, 0xeef453d6923bd65a, 0x113faa2906a13b3f)


def _oracle_parser(data, start):
    """What a correct device parser returns: the host's World of the array at data[start:] and its end, None when the
    host would fail on it."""
    from rt_b200 import wire

    text = data.decode("utf-8", "surrogatepass")  # the text up to start is ASCII: offsets agree up to there
    while start < len(text) and text[start] in " \t\n\r":
        start += 1
    try:
        objs, end = json.JSONDecoder().raw_decode(text, start)
        return wire.world_from_objects(objs), len(text[:end].encode("utf-8", "surrogatepass"))
    except Exception:  # noqa: BLE001
        return None


def _sphere_json():
    return '{"Sphere":{"radius":1.5,"center":[0,1,-3],"node_index":0,"p_albedo_at":{"r":0.5,"g":0.25,"b":1},' \
           '"p_roughness_at":0,"p_emission_at":0}}'


def _bodies():
    from test_host import test_wire_rejects_malformed_bodies as malformed

    bad = [m.args[1] for m in malformed.pytestmark if m.name == "parametrize"][0]
    s = _sphere_json()
    good = _body("[%s,%s]" % (s, s))
    return list(bad) + [
        good,
        b" \n\t" + good,                                                             # leading whitespace
        good.replace(b'{"world"', b'{ "world" '),
        ('{"render_meta":%s,"world":[%s],"division_no":0}' % (META, s)).encode(),   # a non-canonical first key
        good[:-1] + b',"world":[]}',                                                 # duplicate "world": json keeps the last
        good[:-1] + b',"world":5}',
        good[:-1] + b',"world":[%s]}' % s.encode(),
        good + b"}",                                                                 # an error after the world
        good[:-1] + b',"extra":[{"Sphere":{}}]}',                                    # an Object pattern past the world
        _body("[%s]" % s, division_no="-1"),
        _body("[%s]" % s, meta=META.replace(ID, "nope")),
        _body("[%s]" % s, meta=META.replace('"height":40,', "")),
        _body("[%s" % s),
        _body("[]"),
        _body("[ ]"),
        _body("[%s]" % s.replace("1.5", "1e999")),                                   # inf on both paths
        good.decode().encode("utf-16"),
        b'{"world":[' + s.encode() + b'],"render_meta":' + META.encode() + b',"division_no":0,"x":"\xff"}',
    ]


@pytest.mark.parametrize("parser", ["declines", "oracle"])
def test_parse_render_info_unchanged_with_a_world_parser(rt, parser):
    fake = (lambda data, start: None) if parser == "declines" else _oracle_parser
    for body in _bodies():
        for b in (body, body.decode("utf-8", "surrogateescape") if body[:2] != b"\xff\xfe" else body):
            assert _outcome(b, world_parser=fake) == _outcome(b), b[:120]


class _FakeCtx:
    """A context with or without the device wire path: renders band d as the value d everywhere."""

    def __init__(self, device_wire):
        self.calls = []
        if device_wire:
            self.parse_world_json = self._parse
            self.render_divisions_json = self._bodies

    def scene(self, *a):
        class S:
            def close(self):
                pass
        return S()

    def render_divisions(self, scene, p, nos, want_stats=False):
        self.calls.append(("rgb", list(nos)))
        return np.stack([np.full((p.height // p.divisions, p.width, 3), d, np.uint8) for d in nos])

    def _parse(self, data, start):
        self.calls.append(("parse", start))
        return _oracle_parser(data, start)

    def _bodies(self, scene, p, nos, id):
        from rt_b200 import wire

        self.calls.append(("json", list(nos)))
        return [wire.ImageSlice(d, np.full(p.height // p.divisions * p.width * 3, d, np.uint8), id).to_json().encode()
                for d in nos]


def _serve_and_send(device_wire, divisions):
    from rt_b200 import slave, wire

    wk = slave.Worker.__new__(slave.Worker)
    wk.ctx = _FakeCtx(device_wire)
    wk.spp = wk.max_bounces = wk.seed = 0
    wk.intersector = 0
    wk._scenes, wk._cache_size, wk.scene_uploads = OrderedDict(), 4, 0
    wk.lock = threading.Lock()
    posts, done = [], threading.Event()

    def post(url, body):
        posts.append(body)
        if len(posts) == len(divisions):
            done.set()
        return "ok"

    ready, stop = threading.Event(), threading.Event()
    t = threading.Thread(target=slave.serve, kwargs=dict(host="127.0.0.1", port=0, result_url="http://master/result",
                                                         worker=wk, post=post, ready=ready, stop=stop), daemon=True)
    t.start()
    assert ready.wait(30)
    meta = wire.RenderMeta(40, 16, 4, ID)
    sp = np.zeros(2, wire.SPHERE_DTYPE)
    try:
        for d in divisions:
            req = urllib.request.Request(f"http://127.0.0.1:{ready.port}/",
                                         data=wire.render_info_to_json(sp, None, meta, d).encode(), method="POST")
            with urllib.request.urlopen(req, timeout=30) as r:
                assert r.read().decode() == slave.ACK_TEXT
        assert done.wait(30)
    finally:
        stop.set()
        t.join(30)
    expect = {d: wire.ImageSlice(d, np.full(10 * 16 * 3, d, np.uint8), ID).to_json().encode() for d in divisions}
    return wk.ctx.calls, posts, expect


@pytest.mark.parametrize("device_wire", [False, True])
def test_serve_posts_the_same_bytes(rt, device_wire):
    calls, posts, expect = _serve_and_send(device_wire, [2, 0, 3])
    assert sorted(posts) == sorted(expect.values())
    assert all(isinstance(p, bytes) for p in posts)
    kinds = {c[0] for c in calls}
    assert kinds == ({"parse", "json"} if device_wire else {"rgb"})


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def _host_world(text):
    from rt_b200 import wire

    return wire.world_from_objects(json.loads(text)["world"])


def _same_world(a, b):
    return (a.spheres.tobytes() == b.spheres.tobytes() and a.triangles.tobytes() == b.triangles.tobytes()
            and a.world_index.dtype == b.world_index.dtype and a.world_index.tobytes() == b.world_index.tobytes()
            and a.spheres.dtype == b.spheres.dtype and a.triangles.dtype == b.triangles.dtype)


def _device_parity(ctx, body):
    """The device parse of body's world equals the host's, and parse_render_info through it equals the host path."""
    from rt_b200 import wire

    body = body if isinstance(body, bytes) else body.encode()
    m = wire._WORLD_FIRST.match(body)
    got = ctx.parse_world_json(body, m.end())
    assert got is not None, ctx._lib.rt_last_error(ctx._h)
    world, end = got
    assert _same_world(world, _host_world(body))
    assert body[end - 1:end] == b"]"
    assert _outcome(body, world_parser=ctx.parse_world_json) == _outcome(body)
    return world


def _random_triangles(n, seed):
    from rt_b200 import scenes

    rng = np.random.default_rng(seed)
    t = np.zeros(n, scenes.TRIANGLE_DTYPE)
    for k in ("a", "b", "c"):
        t[k] = rng.uniform(-10, 10, (n, 3)).astype(np.float32)
    t["albedo"] = rng.uniform(0, 1, (n, 3)).astype(np.float32)
    t["roughness"] = rng.uniform(0, 1, n).astype(np.float32)
    t["emission"] = np.where(rng.uniform(0, 1, n) < 0.01, 2.5, 0).astype(np.float32)
    return t


@pytest.mark.gpu
def test_parse_interleaved_worlds(ctx, rt):
    from rt_b200 import wire

    meta = wire.RenderMeta(1080, 1920, 20, ID)
    for seed, (ns, nt) in enumerate([(1, 0), (0, 1), (5, 2), (300, 41), (2000, 3000)]):
        sp = rt.scenes.synthetic_spheres(ns, seed) if ns else rt.scenes.no_spheres()
        tr = _random_triangles(nt, seed)
        wi = np.random.default_rng(seed).permutation(ns + nt).astype(np.uint32)
        w = _device_parity(ctx, wire.render_info_to_json(sp, tr, meta, 7, wi))
        assert len(w.spheres) == ns and len(w.triangles) == nt


@pytest.mark.gpu
def test_parse_262144_triangles(ctx, rt):
    from rt_b200 import wire

    tr = _random_triangles(262144, 1)
    body = wire.render_info_to_json(None, tr, wire.RenderMeta(1080, 1920, 20, ID), 3).encode()
    w = _device_parity(ctx, body)
    assert w.triangles.tobytes() == tr.tobytes()


def _fuzz_tokens(n, seed):
    """Number tokens in the device grammar: integers to 19 digits, signed zeros, subnormals, the f32 range's edges, f32
    halfway points, 17-digit f64 strings, exponents at the conversion table's edges."""
    rng = random.Random(seed)
    toks = ["-0", "-0.0", "0e0", "0", "0.0", "-0e5", "1e-46", "-1e-46", "3.4028235e38", "3.4028236e38", "-3.4028236e38",
            "1.401298464324817e-45", "7.006492321624085e-46", "7.006492321624086e-46", "1e-320", "4.9e-324",
            "2.2250738585072014e-308", "1.7976931348623157e308", "1e308", "9e308", "1e-342", "1e-300", "9999999999999999999",
            "-9999999999999999999", "16777217", "16777217.0", "33554431", "1E5", "1e+5", "0.000001", "123456789012345678e-342",
            "1234567890123456789e308", "5e-342", "0.9e-341"]
    while len(toks) < n:
        r = rng.random()
        if r < 0.25:
            nd = rng.randint(1, 19)
            toks.append(("-" if rng.random() < 0.3 else "") + str(rng.randint(10 ** (nd - 1), 10 ** nd - 1)))
        elif r < 0.5:
            x = struct.unpack("<d", struct.pack("<Q", rng.getrandbits(64)))[0]
            if np.isfinite(x):
                toks.append("%.16e" % x if rng.random() < 0.5 else repr(x))
        elif r < 0.75:
            f = np.float32(rng.uniform(-1e4, 1e4) * 10.0 ** rng.randint(-30, 30))
            g = np.nextafter(f, np.float32(np.inf))
            toks.append(repr((float(f) + float(g)) / 2))
        else:
            toks.append("%de%d" % (rng.randint(1, 10 ** rng.randint(1, 18)), rng.randint(-342, 308)))
    return toks


@pytest.mark.gpu
def test_parse_number_fuzz(ctx):
    toks = _fuzz_tokens(100_000, 5)
    objs = []
    for i in range(0, len(toks) - 9, 9):
        t = toks[i:i + 9]
        objs.append('{"Sphere":{"radius":%s,"center":[%s,%s,%s],"node_index":%d,"p_albedo_at":{"r":%s,"g":%s,"b":%s},'
                    '"p_roughness_at":%s,"p_emission_at":%s}}' % (t[0], t[1], t[2], t[3], i, t[4], t[5], t[6], t[7], t[8]))
    with np.errstate(over="ignore"):
        _device_parity(ctx, _body("[" + ",".join(objs) + "]"))


@pytest.mark.gpu
def test_parse_pretty_printed(ctx, rt):
    from rt_b200 import wire

    sp, tr = rt.scenes.synthetic_spheres(40, 2), _random_triangles(25, 2)
    wi = np.random.default_rng(4).permutation(65).astype(np.uint32)
    o = json.loads(wire.render_info_to_json(sp, tr, wire.RenderMeta(40, 16, 4, ID), 1, wi))
    for indent in (2, "\t", None):
        _device_parity(ctx, json.dumps(o, indent=indent))
    _device_parity(ctx, json.dumps(o, indent=1).replace("\n", "\r\n"))


DECLINED = {
    "backslash": ('"radius"', '"rad\\u0069us"'),
    "nan": ("1.5", "NaN"),
    "infinity": ("1.5", "-Infinity"),
    "reordered": ('"radius":1.5,"center":[0,1,-3]', '"center":[0,1,-3],"radius":1.5'),
    "extra_key": ('"p_emission_at":0', '"p_emission_at":0,"x":1'),
    "missing_key": (',"p_roughness_at":0', ""),
    "repeated_key": ('"p_emission_at":0', '"p_emission_at":0,"p_emission_at":0'),
    "20_digits": ("1.5", "15000000000000000000"),
    "leading_zero": ("1.5", "01.5"),
    "plus": ("1.5", "+1.5"),
    "bare_fraction": ("1.5", ".5"),
    "exponent_past_table": ("1.5", "1e-400"),
    "string_value": ("1.5", '"1.5"'),
    "key_with_space": ('"radius"', '"radius "'),
    "negative_node_index": ('"node_index":0', '"node_index":-1'),
    "float_node_index": ('"node_index":0', '"node_index":0.5'),
    "trailing_comma": (None, None),
    "not_an_object": (None, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(DECLINED))
def test_declines_then_host_path(ctx, case):
    from rt_b200 import _abi

    s = _sphere_json()
    old, new = DECLINED[case]
    if case == "trailing_comma":
        world = "[%s,%s,]" % (s, s)
    elif case == "not_an_object":
        world = "[%s,1]" % s
    else:
        assert old in s
        world = "[%s,%s]" % (s, s.replace(old, new, 1))
    body = _body(world)
    start = body.index(b"[")
    assert ctx.parse_world_json(body, start) is None
    sp, tr = np.empty(8, _abi_dtype("s")), np.empty(8, _abi_dtype("t"))
    wi, a, b, c = np.empty(8, np.uint32), C.c_uint32(), C.c_uint32(), C.c_size_t()
    rc = ctx._lib.rt_world_parse_json(ctx._h, body[start:], len(body) - start, sp.ctypes.data, tr.ctypes.data,
                                      wi.ctypes.data, 8, C.byref(a), C.byref(b), C.byref(c))
    assert rc == _abi.RT_ERR_UNSUPPORTED
    assert _outcome(body, world_parser=ctx.parse_world_json) == _outcome(body)


def _abi_dtype(kind):
    from rt_b200 import scenes

    return scenes.SPHERE_DTYPE if kind == "s" else scenes.TRIANGLE_DTYPE


@pytest.mark.gpu
def test_parse_refusals_then_valid(ctx):
    from rt_b200 import _abi

    body = _body("[%s]" % _sphere_json())
    L = ctx._lib
    cap = L.rt_world_json_max_objects(len(body))
    sp, tr, wi = np.empty(cap, _abi_dtype("s")), np.empty(cap, _abi_dtype("t")), np.empty(cap, np.uint32)
    a, b, c = C.c_uint32(), C.c_uint32(), C.c_size_t()
    args = [sp.ctypes.data, tr.ctypes.data, wi.ctypes.data]
    assert L.rt_world_parse_json(ctx._h, body, len(body), *args, cap - 1, C.byref(a), C.byref(b), C.byref(c)) \
        == _abi.RT_ERR_INVALID_ARG
    assert L.rt_world_parse_json(ctx._h, None, len(body), *args, cap, C.byref(a), C.byref(b), C.byref(c)) \
        == _abi.RT_ERR_INVALID_ARG
    assert L.rt_world_parse_json(ctx._h, body, len(body), *args, cap, None, C.byref(b), C.byref(c)) == _abi.RT_ERR_INVALID_ARG
    _device_parity(ctx, body)


def _slice_scene(rt):
    """A frame with values of one, two and three digits, 0 and 255 among them: a bright emitter (255), a black sphere (0),
    a nearly black one (1-9) and the sky between them, over a plane."""
    sp = np.zeros(3, rt.scenes.SPHERE_DTYPE)
    sp[0] = ((-1.5, 0.0, -4.0), 1.0, (1.0, 1.0, 1.0), 0.0, 50.0)
    sp[1] = ((1.5, 0.0, -4.0), 1.0, (0.0, 0.0, 0.0), 0.0, 0.0)
    sp[2] = ((0.0, 1.6, -4.0), 0.8, (0.0003, 0.0003, 0.0003), 0.0, 0.0)
    return sp, rt.scenes.ground_plane()


def _check_bodies(ctx, sc, p, nos):
    from rt_b200 import wire

    bodies, st = ctx.render_divisions_json(sc, p, nos, ID, want_stats=True)
    rgb = ctx.render_divisions(sc, p, nos)
    assert len(bodies) == len(nos) and st["primary"] > 0
    for k, d in enumerate(nos):
        assert bodies[k] == wire.ImageSlice(d, rgb[k].reshape(-1), ID).to_json().encode(), (list(nos), k, d)
    return rgb


@pytest.mark.gpu
@pytest.mark.parametrize("isect", [1, 2])
def test_image_slice_bytes_20_divisions(ctx, rt, isect):
    sp, tr = _slice_scene(rt)
    sc = ctx.scene(sp, tr).wait_ready()
    p = rt.make_params(96, 80, divisions=20, spp=2, max_bounces=3, intersector=isect)
    seen = set()
    for nos in (list(range(20)), [19, 0, 7, 8, 3], [11], [int(d) for d in np.random.default_rng(2).permutation(20)]):
        seen |= set(np.unique(_check_bodies(ctx, sc, p, nos)).tolist())
    assert {0, 255} <= seen and any(10 <= v < 100 for v in seen) and any(0 < v < 10 for v in seen)
    sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,div", [(1, 40, 20), (1, 7, 7), (101, 63, 9), (37, 20, 20)])
def test_image_slice_bytes_odd_sizes(ctx, rt, w, h, div):
    sp, tr = _slice_scene(rt)
    sc = ctx.scene(sp, tr)
    p = rt.make_params(w, h, divisions=div, spp=1, max_bounces=2)
    _check_bodies(ctx, sc, p, list(range(div)))
    _check_bodies(ctx, sc, p, list(range(div))[::-2])
    sc.close()


@pytest.mark.gpu
def test_image_slice_refusals_then_valid(ctx, rt):
    from rt_b200 import _abi, api

    sp, tr = _slice_scene(rt)
    sc = ctx.scene(sp, tr)
    p = rt.make_params(16, 40, divisions=4, spp=1)
    L = ctx._lib
    nos = np.array([1, 2], np.uint32)
    bound = L.rt_slice_json_bound(10, 16)
    buf, lens = np.empty(2 * bound, np.uint8), np.zeros(2, np.uintp)
    lp = lens.ctypes.data_as(C.POINTER(C.c_size_t))

    def call(id_, out_cap=2 * bound, n=2, lens_ptr=lp, nos_=nos):
        return L.rt_render_divisions_json(ctx._h, sc._h, C.byref(p), nos_.ctypes.data, n, id_, buf.ctypes.data, out_cap,
                                          lens_ptr, None)

    for rc in (call(None), call(ID.upper().encode()), call(ID[:-1].encode()), call((ID + "0").encode()),
               call(ID.replace("-", "x", 1).encode()), call(ID.encode(), out_cap=2 * bound - 1),
               call(ID.encode(), lens_ptr=None), call(ID.encode(), n=0), call(ID.encode(), nos_=np.array([1, 4], np.uint32))):
        assert rc == _abi.RT_ERR_INVALID_ARG
        _check_bodies(ctx, sc, p, [1, 2])
    with pytest.raises(api.RtError):
        ctx.render_divisions_json(sc, p, [1, 1], ID)
    _check_bodies(ctx, sc, p, [3])
    sc.close()


@pytest.mark.gpu
def test_slave_end_to_end_obj_world(rt):
    """A real serve() on the GPU worker posts, for an OBJ-built world, the bodies the host path writes."""
    from rt_b200 import obj, slave, wire
    from test_host import mesh_scene_obj

    data, n = mesh_scene_obj()
    tr = obj.build_world(data, n)
    meta = wire.RenderMeta(40, 32, 4, ID)
    wk = slave.Worker(0, spp=2, max_bounces=3)
    posts, done = [], threading.Event()

    def post(url, body):
        posts.append(body)
        if len(posts) == 4:
            done.set()
        return "ok"

    ready, stop = threading.Event(), threading.Event()
    t = threading.Thread(target=slave.serve, kwargs=dict(host="127.0.0.1", port=0, result_url="http://master/result",
                                                         worker=wk, post=post, ready=ready, stop=stop), daemon=True)
    t.start()
    try:
        assert ready.wait(30)
        bodies = [wire.render_info_to_json(None, tr, meta, d).encode() for d in (3, 0, 2, 1)]
        for b in bodies:
            req = urllib.request.Request(f"http://127.0.0.1:{ready.port}/", data=b, method="POST")
            with urllib.request.urlopen(req, timeout=30) as r:
                assert r.read().decode() == slave.ACK_TEXT
        assert done.wait(60)
        expect = sorted(wk.render(wire.parse_render_info(b)).to_json().encode() for b in bodies)
        assert sorted(posts) == expect
        assert wk.scene_uploads == 1
    finally:
        stop.set()
        t.join(30)
        wk.close()
