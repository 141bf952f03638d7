"""Indexed meshes (rt_mesh) in numpy: the rt_triangle records a mesh stands for, and the scene description with
every mesh ref replaced by those records -- the form the indexed one must render bit for bit like."""
import ctypes as C

import numpy as np

from raytracingoneweekendapplication_b200 import capi

TRI = np.dtype([("p", "<f8", 9), ("uv", "<f4", 6), ("material", "<i4"), ("xform", "<i4")])
REF = np.dtype([("type", "<i4"), ("index", "<i4")])
assert TRI.itemsize == C.sizeof(capi.rt_triangle) and REF.itemsize == C.sizeof(capi.rt_prim_ref)
RECORD = {capi.RT_PRIM_SPHERE: ("spheres", capi.rt_sphere), capi.RT_PRIM_QUAD: ("quads", capi.rt_quad),
          capi.RT_PRIM_TRIANGLE: ("triangles", capi.rt_triangle)}


def array(ptr, count, dtype):
    if count == 0:
        return np.zeros(0, dtype=dtype)
    return np.frombuffer(C.string_at(ptr, count * np.dtype(dtype).itemsize), dtype=dtype).copy()


def view(ptr, count, ctype):
    """A writable numpy view of `count` elements behind a ctypes pointer (the caller keeps the owner alive)."""
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(count,))


def refs(d, boundary=False):
    return array(d.boundary_refs if boundary else d.world, d.n_boundary_refs if boundary else d.n_world, REF)


def triangles(d):
    return array(d.triangles, d.n_triangles, TRI)


def record_bytes(d, ref):
    field, ctype = RECORD[int(ref["type"])]
    return C.string_at(C.cast(getattr(d, field), C.c_void_p).value + int(ref["index"]) * C.sizeof(ctype), C.sizeof(ctype))


def expand_mesh(m: capi.rt_mesh) -> np.ndarray:
    """positions[indices] widened to float64, uvs[uv_indices] (or the default UVs), the mesh's material and xform."""
    n = m.n_triangles
    pos = array(m.positions, 3 * m.n_vertices, np.float32).reshape(-1, 3)
    idx = array(m.indices, 3 * n, np.uint32).reshape(-1, 3)
    t = np.zeros(n, dtype=TRI)
    t["p"] = pos[idx].astype(np.float64).reshape(n, 9)
    if m.uvs:
        uv = array(m.uvs, 2 * m.n_uvs, np.float32).reshape(-1, 2)
        ui = array(m.uv_indices, 3 * n, np.uint32).reshape(-1, 3) if m.uv_indices else idx
        t["uv"] = uv[ui].reshape(n, 6)
    else:
        t["uv"] = np.array([0, 0, 1, 0, 0, 1], dtype=np.float32)
    t["material"], t["xform"] = m.material, m.xform
    return t


class Expanded:
    """The description `d` with every mesh ref replaced by rt_triangle records appended to its triangles, in place
    (same world positions, same canonical ids); n_meshes = 0.  Usable wherever capi.Context.upload takes a scene."""

    def __init__(self, d: capi.rt_scene_desc):
        e = capi.rt_scene_desc.from_buffer_copy(d)
        tris = [triangles(d)]
        world = []
        base = d.n_triangles
        for r in refs(d):
            if r["type"] == capi.RT_PRIM_MESH:
                t = expand_mesh(d.meshes[int(r["index"])])
                world += [(capi.RT_PRIM_TRIANGLE, base + k) for k in range(len(t))]
                tris.append(t)
                base += len(t)
            else:
                world.append((int(r["type"]), int(r["index"])))
        self.tris = np.ascontiguousarray(np.concatenate(tris))
        self.world = np.array(world, dtype=REF)
        e.triangles = self.tris.ctypes.data_as(C.POINTER(capi.rt_triangle))
        e.n_triangles = len(self.tris)
        e.world = self.world.ctypes.data_as(C.POINTER(capi.rt_prim_ref))
        e.n_world = len(self.world)
        e.meshes, e.n_meshes = None, 0
        self.desc = e
        self.desc_ptr = C.pointer(e)
