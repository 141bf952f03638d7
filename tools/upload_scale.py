"""How rt_upload_scene and the render kernel scale with the triangle count (SURVEY 8f rank 1): a terrain of N small
triangles (a height-field grid of shared float vertices with per-vertex UVs) + one ground sphere, built straight into
the C ABI structs with numpy, in one of two input forms of the same triangles:

  indexed  one rt_mesh: float positions, 12 bytes of indices per triangle, float UVs (ABI 4)
  soup     the same triangles expanded into rt_triangle records (104 bytes each) and one world ref per triangle

Both forms give the same device records.  With --input both the two forms are uploaded alternately, each into its own
context, and the best of three is kept.  Prints one JSON line per N and form, with the card name and power limit.

Usage: upload_scale.py [--input soup|indexed|both] [N ...]   (default soup, 10000 100000 1000000; builder from
RT_B200_BVH, default host)"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from raytracingoneweekendapplication_b200 import capi  # noqa: E402

TRI = np.dtype([("p0", "<f8", 3), ("p1", "<f8", 3), ("p2", "<f8", 3), ("uv0", "<f4", 2), ("uv1", "<f4", 2), ("uv2", "<f4", 2),
                ("material", "<i4"), ("xform", "<i4")])
REF = np.dtype([("type", "<i4"), ("index", "<i4")])
assert TRI.itemsize == C.sizeof(capi.rt_triangle) and REF.itemsize == C.sizeof(capi.rt_prim_ref)


def terrain(n_tris: int, seed: int = 1):
    """A (k x k) height-field grid, two triangles per cell, ~n_tris triangles in [-50,50]^2, as rt_triangle records
    (double positions, the default UVs)."""
    k = max(2, int(np.sqrt(n_tris / 2)) + 1)
    xs = np.linspace(-50.0, 50.0, k)
    X, Z = np.meshgrid(xs, xs, indexing="ij")
    rng = np.random.default_rng(seed)
    Y = 3.0 * np.sin(0.21 * X) * np.cos(0.17 * Z) + 0.3 * rng.standard_normal(X.shape)
    P = np.stack([X, Y, Z], axis=-1)
    a, b, c, d = P[:-1, :-1], P[1:, :-1], P[1:, 1:], P[:-1, 1:]
    t = np.zeros(2 * (k - 1) * (k - 1), dtype=TRI)
    t["p0"][0::2], t["p1"][0::2], t["p2"][0::2] = a.reshape(-1, 3), b.reshape(-1, 3), c.reshape(-1, 3)
    t["p0"][1::2], t["p1"][1::2], t["p2"][1::2] = a.reshape(-1, 3), c.reshape(-1, 3), d.reshape(-1, 3)
    t["uv1"] = [1, 0]
    t["uv2"] = [0, 1]
    t["material"] = 0
    t["xform"] = -1
    return t[:n_tris] if len(t) > n_tris else t


def indexed_terrain(n_tris: int, seed: int = 1):
    """The same grid as shared float vertices: positions (k*k, 3), indices (n, 3) in the order of terrain(), per-vertex
    UVs (k*k, 2)."""
    k = max(2, int(np.sqrt(n_tris / 2)) + 1)
    xs = np.linspace(-50.0, 50.0, k)
    X, Z = np.meshgrid(xs, xs, indexing="ij")
    rng = np.random.default_rng(seed)
    Y = 3.0 * np.sin(0.21 * X) * np.cos(0.17 * Z) + 0.3 * rng.standard_normal(X.shape)
    pos = np.ascontiguousarray(np.stack([X, Y, Z], axis=-1).reshape(-1, 3), dtype=np.float32)
    v = np.arange(k * k, dtype=np.uint32).reshape(k, k)
    a, b, c, d = v[:-1, :-1].ravel(), v[1:, :-1].ravel(), v[1:, 1:].ravel(), v[:-1, 1:].ravel()
    idx = np.empty((2 * len(a), 3), dtype=np.uint32)
    idx[0::2] = np.stack([a, b, c], axis=1)
    idx[1::2] = np.stack([a, c, d], axis=1)
    u = np.linspace(0.0, 1.0, k, dtype=np.float32)
    U, V = np.meshgrid(u, u, indexing="ij")
    uvs = np.ascontiguousarray(np.stack([U, V], axis=-1).reshape(-1, 2))
    return pos, np.ascontiguousarray(idx[:n_tris]), uvs


def expand(pos, idx, uvs):
    """The rt_triangle records an indexed mesh stands for (positions widened to double)."""
    t = np.zeros(len(idx), dtype=TRI)
    for c, (p, uv) in enumerate((("p0", "uv0"), ("p1", "uv1"), ("p2", "uv2"))):
        t[p] = pos[idx[:, c]]
        t[uv] = uvs[idx[:, c]]
    t["material"], t["xform"] = 0, -1
    return t


def scene_desc(tris=None, mesh=None):
    """The terrain -- rt_triangle records `tris`, or an indexed mesh `mesh` = (positions, indices, uvs) -- and a
    ground sphere."""
    keep = {}
    d = capi.rt_scene_desc()
    d.struct_size = C.sizeof(d)
    d.abi_version = capi.RT_B200_ABI_VERSION
    if tris is not None:
        n = len(tris)
        refs = np.zeros(n + 1, dtype=REF)
        refs["type"][:n] = capi.RT_PRIM_TRIANGLE
        refs["index"][:n] = np.arange(n)
        d.triangles = tris.ctypes.data_as(C.POINTER(capi.rt_triangle)); d.n_triangles = n
        keep["tris"] = tris
    else:
        pos, idx, uvs = mesh
        refs = np.zeros(2, dtype=REF)
        refs[0] = (capi.RT_PRIM_MESH, 0)
        m = (capi.rt_mesh * 1)()
        m[0].positions, m[0].n_vertices = pos.ctypes.data_as(C.POINTER(C.c_float)), len(pos)
        m[0].indices, m[0].n_triangles = idx.ctypes.data_as(C.POINTER(C.c_uint32)), len(idx)
        m[0].uvs, m[0].n_uvs = uvs.ctypes.data_as(C.POINTER(C.c_float)), len(uvs)
        m[0].material, m[0].xform = 0, -1
        d.meshes, d.n_meshes = m, 1
        keep.update(m=m, mesh=mesh)
    refs["type"][-1], refs["index"][-1] = capi.RT_PRIM_SPHERE, 0
    sph = (capi.rt_sphere * 1)()
    sph[0].center0[:] = [0.0, -1010.0, 0.0]
    sph[0].radius = 1000.0
    sph[0].material, sph[0].xform = 1, -1
    mats = (capi.rt_material * 2)()
    texs = (capi.rt_texture * 2)()
    for i, col in enumerate([(0.6, 0.5, 0.3), (0.3, 0.6, 0.3)]):
        mats[i].type, mats[i].texture = 0, i
        texs[i].type = 0
        texs[i].color[:] = col
    d.world = refs.ctypes.data_as(C.POINTER(capi.rt_prim_ref)); d.n_world = len(refs)
    d.spheres = sph; d.n_spheres = 1
    d.materials = mats; d.n_materials = 2
    d.textures = texs; d.n_textures = 2
    d.camera.lookfrom[:] = [0.0, 40.0, 90.0]
    d.camera.lookat[:] = [0.0, 0.0, 0.0]
    d.camera.vup[:] = [0.0, 1.0, 0.0]
    d.camera.vfov = 45.0
    d.camera.focus_dist = 10.0
    d.camera.background[:] = [0.7, 0.8, 1.0]
    keep.update(refs=refs, sph=sph, mats=mats, texs=texs)
    return d, keep


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception:
        return None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--input", choices=["soup", "indexed", "both"], default="soup")
    ap.add_argument("sizes", nargs="*", type=int, default=[10_000, 100_000, 1_000_000])
    args = ap.parse_args()
    forms = ["soup", "indexed"] if args.input == "both" else [args.input]
    mode = os.environ.get("RT_B200_BVH", "host")
    gpu, power = card()
    for n in args.sizes:
        t0 = time.perf_counter()
        mesh = indexed_terrain(n)
        scenes = {f: scene_desc(tris=expand(*mesh)) if f == "soup" else scene_desc(mesh=mesh) for f in forms}
        n_tris = len(mesh[1])
        t_gen = time.perf_counter() - t0
        ctxs = {f: capi.Context(0) for f in forms}
        best = {f: None for f in forms}
        for _ in range(3):   # the forms alternate, best of three each
            for f in forms:
                ctxs[f].set_bvh_builder(mode)
                t0 = time.perf_counter()
                ctxs[f].upload(scenes[f][0])
                ms = 1e3 * (time.perf_counter() - t0)
                st = ctxs[f].stats()
                if best[f] is None or ms < best[f][0]:
                    best[f] = (ms, st)
        w, h, spp = 1920, 1080, 4
        for f in forms:
            ctx = ctxs[f]
            ctx.render(w, h, spp, max_depth=8, seed=1)
            render = 1e30
            for _ in range(2):
                ctx.render(w, h, spp, max_depth=8, seed=1)
                render = min(render, ctx.stats()["render_ms"])
            ms, st = best[f]
            aov = ctx.aov(w, h)
            print(json.dumps({"triangles": n_tris, "input": f, "gpu": gpu, "power_limit": power, "gen_s": round(t_gen, 3),
                              "upload_ms": round(ms, 1), "upload_bytes": st["upload_bytes"], "bytes_per_triangle": round(st["upload_bytes"] / n_tris, 1),
                              "bvh_nodes": st["bvh_nodes"], "bvh_depth": st["bvh_depth"], "bvh_leaves": st["bvh_leaves"],
                              "render_ms": round(render, 2), "msamples_s": round(w * h * spp / render / 1e3, 1),
                              "primary_hit_fraction": round(float((aov["prim_id"] >= 0).mean()), 4),
                              "builder": mode, "on_device": st["bvh_on_device"], "device_build_ms": round(st["device_build_ms"], 3),
                              "device_copy_in_ms": round(st["device_copy_in_ms"], 3), "device_top_ms": round(st["device_top_ms"], 3)}), flush=True)
        for c in ctxs.values():
            c.close()


if __name__ == "__main__":
    main()
