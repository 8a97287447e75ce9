"""OBJ + MTL → world of triangles, as the controller ingests it.

Mirror of ray-tracer-controller/src/obj.rs:10-53 (tobj 3.2.4, `LoadOptions::default()`: no triangulation,
multi-index):  the request body is the OBJ bytes followed by the MTL bytes; every face of every model becomes a
`Triangle` with `roughness = Ns / 1000`, `albedo = Kd`, `emission = 0` (obj.rs:43-45), in file order.

Faithful quirks: a model is closed at every `o`, `g` or `usemtl`; inside a model the face indices are one flat list
cut into triples (obj.rs:23-26), so a polygon with more than three corners is NOT fan-triangulated — its corners
run into the next face exactly as in the reference; a model without a material makes the reference panic
(`mesh.material_id.unwrap()`, obj.rs:22) and raises ObjError here.
"""
from __future__ import annotations

import numpy as np

from .scenes import TRIANGLE_DTYPE


class ObjError(ValueError):
    """The reference would panic ("Failed to load obj or mtl file" / unwrap on None)."""


def parse_mtl(data: bytes) -> dict:
    """name → {"Kd": (r,g,b), "Ns": s}; tobj defaults: diffuse (0,0,0)... shininess 0."""
    mats: dict = {}
    order = []
    cur = None
    for raw in data.decode("utf-8", errors="replace").splitlines():
        line = raw.split("#", 1)[0].strip()
        if not line:
            continue
        key, *rest = line.split()
        if key == "newmtl":
            cur = " ".join(rest)
            if cur not in mats:
                order.append(cur)
            mats[cur] = {"Kd": (0.0, 0.0, 0.0), "Ns": 0.0}
        elif cur is not None and key == "Kd" and len(rest) >= 3:
            try:
                mats[cur]["Kd"] = tuple(float(np.float32(x)) for x in rest[:3])
            except ValueError as e:
                raise ObjError(f"bad Kd in material {cur!r}") from e
        elif cur is not None and key == "Ns" and rest:
            try:
                mats[cur]["Ns"] = float(np.float32(rest[0]))
            except ValueError as e:
                raise ObjError(f"bad Ns in material {cur!r}") from e
    mats["__order__"] = order
    return mats


def build_world(data: bytes, obj_size: int, parser=None) -> np.ndarray:
    """`data[:obj_size]` = OBJ, `data[obj_size:]` = MTL → TRIANGLE_DTYPE array in the reference's world order.

    parser: optional `parser(data, obj_size)` (e.g. `Context.parse_obj`, which builds the world on the GPU) returning
    this function's array or None when it declines; a decline falls through to the host code below, which decides
    whether the body is valid and what its error is."""
    if obj_size < 0 or obj_size > len(data):
        raise ObjError("obj_size out of range")
    if parser is not None:
        out = parser(data, obj_size)
        if out is not None:
            return out
    mats = parse_mtl(data[obj_size:])
    verts: list = []
    tris: list = []
    model_idx: list = []       # flat corner indices of the open model
    model_mat = None

    def close_model():
        nonlocal model_idx
        if model_idx:
            if model_mat is None or model_mat not in mats:
                raise ObjError("model without a material (the reference unwraps mesh.material_id)")
            m = mats[model_mat]
            rough = float(np.float32(m["Ns"]) / np.float32(1000.0))
            for i in range(len(model_idx) // 3):
                a, b, c = (verts[model_idx[3 * i + k]] for k in range(3))
                tris.append((a, b, c, m["Kd"], rough, 0.0))
        model_idx = []

    for raw in data[:obj_size].decode("utf-8", errors="replace").splitlines():
        line = raw.split("#", 1)[0].strip()
        if not line:
            continue
        key, *rest = line.split()
        if key == "v":
            if len(rest) < 3:
                raise ObjError("vertex with fewer than 3 coordinates")
            try:
                verts.append(tuple(float(np.float32(x)) for x in rest[:3]))
            except ValueError as e:
                raise ObjError("bad vertex") from e
        elif key == "f":
            if len(rest) < 3:
                raise ObjError("face with fewer than 3 corners")
            for corner in rest:
                try:
                    i = int(corner.split("/")[0])
                except ValueError as e:
                    raise ObjError(f"bad face corner {corner!r}") from e
                i = i - 1 if i > 0 else len(verts) + i      # negative indices are relative to the end
                if i < 0 or i >= len(verts):
                    raise ObjError("face index out of range")
                model_idx.append(i)
        elif key in ("o", "g"):
            close_model()
        elif key == "usemtl":
            close_model()
            model_mat = " ".join(rest)
    close_model()
    out = np.zeros(len(tris), dtype=TRIANGLE_DTYPE)
    for i, t in enumerate(tris):
        out[i] = t
    return out


def write_obj(vertices, faces, material="mat") -> bytes:
    """Tiny writer for tests/tools: one model, one material."""
    lines = [f"usemtl {material}"]
    lines += ["v %.9g %.9g %.9g" % tuple(v) for v in vertices]
    lines += ["f " + " ".join(str(i + 1) for i in f) for f in faces]
    return ("\n".join(lines) + "\n").encode()
