"""Indexed meshes in the scene ABI (rt_mesh, RT_PRIM_MESH): mesh::indexed_meshes() must hand rt_upload_scene
exactly the triangles the triangle_soup path hands it -- expanding the indexed description in numpy gives the soup's
rt_triangle bytes in order, the soup's run of triangle refs is ONE mesh ref at the same world position, the media
(Q15 multiplicities) are unchanged -- and the scene fingerprint of checkpoint files covers the mesh arrays."""
import ctypes as C
import os

import numpy as np
import pytest

from mesh_expand import REF, Expanded, expand_mesh, record_bytes, refs, triangles, view
from raytracingoneweekendapplication_b200 import capi
from test_obj_fast_path import TRICKY


def check_same_scene(soup, idx):
    """idx (indexed meshes) and soup describe the same triangles, refs, media and tables."""
    ds, di = soup.desc, idx.desc
    sw, iw = refs(ds), refs(di)
    stris = triangles(ds)
    j = 0
    for r in iw:
        if r["type"] == capi.RT_PRIM_MESH:
            t = expand_mesh(di.meshes[int(r["index"])])
            run = sw[j:j + len(t)]
            assert len(run) == len(t) and np.all(run["type"] == capi.RT_PRIM_TRIANGLE)
            assert stris[run["index"]].tobytes() == t.tobytes()
            j += len(t)
        else:
            assert sw[j]["type"] == r["type"] and record_bytes(ds, sw[j]) == record_bytes(di, r)
            j += 1
    assert j == len(sw)
    sb, ib = refs(ds, boundary=True), refs(di, boundary=True)
    assert len(sb) == len(ib)
    for a, b in zip(sb, ib):
        assert a["type"] == b["type"] and record_bytes(ds, a) == record_bytes(di, b)
    for field, ctype in [("media", capi.rt_medium), ("materials", capi.rt_material), ("textures", capi.rt_texture),
                         ("xforms", capi.rt_xform), ("lights", capi.rt_point_light)]:
        n = getattr(ds, "n_" + field)
        assert n == getattr(di, "n_" + field), field
        if n:
            assert C.string_at(getattr(ds, field), n * C.sizeof(ctype)) == C.string_at(getattr(di, field), n * C.sizeof(ctype)), field
    # and the numpy expansion is a complete description of the soup's world
    e = Expanded(di)
    assert e.desc.n_world == ds.n_world


def positions(sc, mesh=0):
    m = sc.desc.meshes[mesh]
    return view(m.positions, 3 * m.n_vertices, C.c_float)


@pytest.mark.parametrize("newline,tail", [("\n", "\n"), ("\r\n", "\r\n"), ("\n", "")])
def test_tricky_obj(built, tmp_path, newline, tail):
    path = str(tmp_path / "tricky.obj")
    with open(path, "w", newline="") as f:
        f.write(TRICKY.replace("\n", newline) + tail)
    soup, idx = capi.ObjScene(path, scale=1.5), capi.ObjScene(path, scale=1.5, indexed=True)
    d = idx.desc
    assert (d.n_meshes, d.n_triangles, d.n_world) == (1, 0, 1)
    m = d.meshes[0]
    assert m.n_triangles == soup.desc.n_triangles == 9 and m.n_vertices == 6
    assert m.uv_indices and m.n_uvs == 5   # the file's four `vt` + the (0,0) of corners without a valid one
    check_same_scene(soup, idx)
    # Q5: both halves of a quad carry the UVs of the face's first three corners, without duplicated vertices
    t = expand_mesh(m)
    assert np.array_equal(t["uv"][1], t["uv"][2])


def test_blob_and_multi_piece_terrain(built, tmp_path):
    from raytracingoneweekendapplication_b200.assets import ensure_assets

    blob = os.path.join(ensure_assets(), "blob.obj")
    check_same_scene(capi.ObjScene(blob), capi.ObjScene(blob, indexed=True))
    k = 260
    xs = np.linspace(-5, 5, k)
    path = str(tmp_path / "terrain.obj")
    with open(path, "w") as f:
        for i in range(k):
            for j in range(k):
                f.write(f"v {xs[i]:.6f} {np.sin(xs[i]) * np.cos(xs[j]):.6f} {xs[j]:.6f}\nvt {i / (k - 1):.5f} {j / (k - 1):.5f}\n")
        for i in range(k - 1):
            for j in range(k - 1):
                a, b, c, d = i * k + j + 1, (i + 1) * k + j + 1, (i + 1) * k + j + 2, i * k + j + 2
                f.write(f"f {a}/{a} {b}/{b} {c}/{c} {d}/{d}\n")
    assert os.path.getsize(path) > 3 << 20   # several parser pieces
    soup, idx = capi.ObjScene(path), capi.ObjScene(path, indexed=True)
    assert idx.desc.meshes[0].n_triangles == 2 * (k - 1) ** 2 and idx.desc.meshes[0].n_vertices == k * k
    check_same_scene(soup, idx)


def test_with_media(built):
    """Q15: the indexed mesh takes part in the replayed median split with one box per triangle, like the soup."""
    from raytracingoneweekendapplication_b200.assets import ensure_assets

    blob = os.path.join(ensure_assets(), "blob.obj")
    soup, idx = capi.ObjScene(blob, with_media=True), capi.ObjScene(blob, with_media=True, indexed=True)
    assert idx.desc.n_media == 3 and idx.desc.n_meshes == 1
    check_same_scene(soup, idx)
    assert idx.hash != soup.hash


@pytest.mark.parametrize("name", ["mesh", "kitchen_sink"])
def test_baseline_scenes_built_with_indexed_meshes(built, name):
    soup, idx = capi.Scene(name), capi.Scene(name, indexed=True)
    assert idx.desc.n_meshes == (3 if name == "mesh" else 0)   # kitchen_sink loads no OBJ file
    check_same_scene(soup, idx)
    assert capi.Scene(name).desc.n_meshes == 0   # the setting does not outlive the build


def test_scene_hash_covers_the_mesh_arrays(built):
    from raytracingoneweekendapplication_b200.assets import ensure_assets

    blob = os.path.join(ensure_assets(), "blob.obj")
    a, b = capi.ObjScene(blob, indexed=True), capi.ObjScene(blob, indexed=True)
    assert a.hash == b.hash
    p = positions(b)
    p[7] += 0.25
    assert a.hash != b.hash
    p[7] -= 0.25
    assert a.hash == b.hash
    ui = view(b.desc.meshes[0].uv_indices, 3 * b.desc.meshes[0].n_triangles, C.c_uint32)
    ui[0], ui[1] = ui[1], ui[0]
    assert a.hash != b.hash


def test_loaders_are_exclusive(built, tmp_path):
    with pytest.raises(ValueError):
        capi.ObjScene(str(tmp_path / "x.obj"), per_triangle=True, indexed=True)


def test_descriptor_layout(built):
    assert C.sizeof(capi.rt_mesh) == 56 and REF.itemsize == 8
    assert capi.RT_SCENE_DESC_V3_SIZE == C.sizeof(capi.rt_scene_desc) - 16
    assert capi.load().rt_struct_size(15) == C.sizeof(capi.rt_mesh)
