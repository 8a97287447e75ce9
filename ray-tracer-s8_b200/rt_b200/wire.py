"""The reference's wire types, byte-compatible with its serde_json encoding.

ray-tracer-slave/src/lib.rs:10-30 (RenderInfo / ImageSlice / RenderMeta), shapes/mod.rs:23-27 (externally
tagged `enum Object`), shapes/sphere.rs:13-20, shapes/mesh.rs:15-23, color.rs:5-10.  `Vec3A` serialises as a
3-element array (glam `serde` feature).  Field order as declared in the Rust structs.

    RenderInfo = {"world":[Object...], "render_meta":RenderMeta, "division_no":u32}
    RenderMeta = {"height":u32, "width":u32, "divisions":u32, "id":"<uuid>"}
    Object     = {"Sphere":{"radius","center":[x,y,z],"node_index","p_albedo_at":{"r","g","b"},
                            "p_roughness_at","p_emission_at"}}
               | {"Triangle":{"a","b","c","node_index","p_albedo_at","p_roughness_at","p_emission_at"}}
    ImageSlice = {"division_no":u32, "image":[u8...], "id":"<uuid>"}
"""
from __future__ import annotations

import json
import re
import uuid as _uuid
from dataclasses import dataclass, field

import numpy as np

from .scenes import SPHERE_DTYPE, TRIANGLE_DTYPE


class WireError(ValueError):
    """Malformed request body (the reference's actix Json extractor answers 400 in this case)."""


@dataclass
class RenderMeta:
    height: int
    width: int
    divisions: int
    id: str

    def to_obj(self):
        return {"height": self.height, "width": self.width, "divisions": self.divisions, "id": self.id}


@dataclass
class World:
    """`Vec<Object>` as two primitive arrays + the world position of each (spheres first, then triangles)."""
    spheres: np.ndarray
    triangles: np.ndarray
    world_index: np.ndarray

    def __len__(self):
        return len(self.spheres) + len(self.triangles)


@dataclass
class RenderInfo:
    world: World
    render_meta: RenderMeta
    division_no: int


@dataclass
class ImageSlice:
    division_no: int
    image: np.ndarray  # uint8, flat, (height/divisions)*width*3
    id: str = field(default="")

    def to_json(self) -> str:
        # serde_json writes Vec<u8> as an array of decimal numbers (lib.rs:18-22)
        img = np.asarray(self.image, dtype=np.uint8).reshape(-1)
        return '{"division_no":%d,"image":[%s],"id":"%s"}' % (
            self.division_no, ",".join(map(str, img.tolist())), self.id)

    @staticmethod
    def from_json(text: str | bytes) -> "ImageSlice":
        o = json.loads(text)
        try:
            return ImageSlice(int(o["division_no"]), np.asarray(o["image"], dtype=np.uint8), str(o["id"]))
        except (KeyError, TypeError, ValueError, OverflowError) as e:
            raise WireError(f"bad ImageSlice: {e}") from e


def _f(x) -> float:
    if isinstance(x, bool) or not isinstance(x, (int, float)):
        raise WireError(f"expected a number, got {x!r}")
    return float(x)


def _u32(x, name) -> int:
    if isinstance(x, bool) or not isinstance(x, int) or x < 0 or x > 0xFFFFFFFF:
        raise WireError(f"{name}: expected u32, got {x!r}")
    return x


def _vec3(v, name):
    if not isinstance(v, list) or len(v) != 3:
        raise WireError(f"{name}: expected [x,y,z]")
    return tuple(_f(c) for c in v)


def _color(c, name):
    if not isinstance(c, dict):
        raise WireError(f"{name}: expected {{r,g,b}}")
    try:
        return (_f(c["r"]), _f(c["g"]), _f(c["b"]))
    except KeyError as e:
        raise WireError(f"{name}: missing field {e}") from e


def world_from_objects(objs) -> World:
    if not isinstance(objs, list):
        raise WireError("world: expected an array of Object")
    sph, sph_pos, tri, tri_pos = [], [], [], []
    for pos, o in enumerate(objs):
        if not isinstance(o, dict) or len(o) != 1:
            raise WireError(f"world[{pos}]: expected an externally tagged Object")
        (tag, body), = o.items()
        try:
            if tag == "Sphere":
                sph.append((_vec3(body["center"], "center"), _f(body["radius"]), _color(body["p_albedo_at"], "p_albedo_at"),
                            _f(body["p_roughness_at"]), _f(body["p_emission_at"])))
                sph_pos.append(pos)
            elif tag == "Triangle":
                tri.append((_vec3(body["a"], "a"), _vec3(body["b"], "b"), _vec3(body["c"], "c"),
                            _color(body["p_albedo_at"], "p_albedo_at"), _f(body["p_roughness_at"]),
                            _f(body["p_emission_at"])))
                tri_pos.append(pos)
            else:
                raise WireError(f"world[{pos}]: unknown variant {tag!r}")
        except KeyError as e:
            raise WireError(f"world[{pos}]: missing field {e}") from e
        except TypeError as e:
            raise WireError(f"world[{pos}]: {e}") from e
    spheres = np.array(sph, dtype=SPHERE_DTYPE) if sph else np.zeros(0, SPHERE_DTYPE)
    triangles = np.array(tri, dtype=TRIANGLE_DTYPE) if tri else np.zeros(0, TRIANGLE_DTYPE)
    return World(spheres, triangles, np.array(sph_pos + tri_pos, dtype=np.uint32))


# serde's layout of a RenderInfo starts with its world: {"world":[
_WORLD_FIRST = re.compile(rb'[ \t\n\r]*\{[ \t\n\r]*"world"[ \t\n\r]*:')


def _device_world(body, world_parser):
    """(World, the body's other members as json parses them) when the world went through `world_parser`, else None.

    world_parser(data, start) parses the array at data[start:] and returns (World, end offset) or None (declined).  The
    rest of the body is parsed by json with [] in place of the world, so it meets exactly the host path's checks; any
    doubt (a decline, a JSON error, a second "world" key, which json resolves to the last) leaves the body to the host
    path, which then gives today's result or error text."""
    data = body.encode("utf-8", "surrogatepass") if isinstance(body, str) else bytes(body)
    m = _WORLD_FIRST.match(data)
    if m is None:
        return None
    got = world_parser(data, m.end())
    if got is None:
        return None
    world, end = got
    last_pairs = []

    def pairs(kv):
        last_pairs[:] = kv
        return dict(kv)

    try:
        o = json.loads(data[: m.end()] + b"[]" + data[end:], object_pairs_hook=pairs)  # the outermost object comes last
    except (json.JSONDecodeError, UnicodeDecodeError):
        return None
    if sum(k == "world" for k, _ in last_pairs) != 1:
        return None
    return world, o


def parse_render_info(text: str | bytes, world_parser=None) -> RenderInfo:
    """RenderInfo from a request body.  world_parser (optional, e.g. a GPU context's parse_world_json) parses the world
    array when the body starts with it; the result and every WireError are those of the host path alone."""
    device = _device_world(text, world_parser) if world_parser is not None else None
    if device is not None:
        world, o = device
    else:
        world = None
        try:
            o = json.loads(text)
        except json.JSONDecodeError as e:
            raise WireError(f"invalid JSON: {e}") from e
    if not isinstance(o, dict):
        raise WireError("RenderInfo: expected an object")
    try:
        m = o["render_meta"]
        meta = RenderMeta(_u32(m["height"], "height"), _u32(m["width"], "width"), _u32(m["divisions"], "divisions"),
                          str(_uuid.UUID(str(m["id"]))))
        return RenderInfo(world if world is not None else world_from_objects(o["world"]), meta,
                          _u32(o["division_no"], "division_no"))
    except KeyError as e:
        raise WireError(f"RenderInfo: missing field {e}") from e
    except (TypeError, ValueError) as e:
        if isinstance(e, WireError):
            raise
        raise WireError(f"RenderInfo: {e}") from e


def _num(x) -> str:
    # shortest decimal that round-trips the f32 (what serde_json's ryu prints for f32)
    s = np.format_float_positional(np.float32(x), unique=True, trim="0")
    if s.endswith("."):
        s += "0"
    return s


def objects_from_world(world: World):
    """World → list of externally tagged Objects in world order (node_index 0, rebuilt by the slave)."""
    n = len(world)
    objs = [None] * n
    ns = len(world.spheres)
    for i in range(n):
        pos = int(world.world_index[i]) if world.world_index is not None else i
        if i < ns:
            s = world.spheres[i]
            objs[pos] = ("Sphere", s)
        else:
            objs[pos] = ("Triangle", world.triangles[i - ns])
    return objs


def render_info_to_json(spheres, triangles, meta: RenderMeta, division_no: int, world_index=None) -> str:
    """Emit the body the controller POSTs to a slave (ray-tracer-controller/src/main.rs:59-66)."""
    spheres = np.zeros(0, SPHERE_DTYPE) if spheres is None else np.asarray(spheres, dtype=SPHERE_DTYPE)
    triangles = np.zeros(0, TRIANGLE_DTYPE) if triangles is None else np.asarray(triangles, dtype=TRIANGLE_DTYPE)
    n = len(spheres) + len(triangles)
    wi = np.arange(n, dtype=np.uint32) if world_index is None else np.asarray(world_index, dtype=np.uint32)
    parts = []
    for tag, p in objects_from_world(World(spheres, triangles, wi)):
        alb = '{"r":%s,"g":%s,"b":%s}' % tuple(_num(c) for c in p["albedo"])
        if tag == "Sphere":
            parts.append('{"Sphere":{"radius":%s,"center":[%s],"node_index":0,"p_albedo_at":%s,"p_roughness_at":%s,'
                         '"p_emission_at":%s}}' % (_num(p["radius"]), ",".join(_num(c) for c in p["center"]), alb,
                                                  _num(p["roughness"]), _num(p["emission"])))
        else:
            parts.append('{"Triangle":{"a":[%s],"b":[%s],"c":[%s],"node_index":0,"p_albedo_at":%s,'
                         '"p_roughness_at":%s,"p_emission_at":%s}}' % (
                             ",".join(_num(c) for c in p["a"]), ",".join(_num(c) for c in p["b"]),
                             ",".join(_num(c) for c in p["c"]), alb, _num(p["roughness"]), _num(p["emission"])))
    return '{"world":[%s],"render_meta":%s,"division_no":%d}' % (
        ",".join(parts), json.dumps(meta.to_obj(), separators=(",", ":")), division_no)
