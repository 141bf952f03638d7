"""Indexed meshes (rt_mesh, RT_PRIM_MESH) on the B200: the indexed form of a scene and its expansion into rt_triangle
records upload to the same device records, so they render the same bits, report the same primary hits and build the
same trees, on the host path and on the device path; malformed meshes are refused with their code (and never reach a
kernel); ABI-3 descriptions still upload; the scene cache and checkpoints see a moved vertex."""
import ctypes as C
import os
import shutil

import numpy as np
import pytest

from mesh_expand import Expanded
from raytracingoneweekendapplication_b200 import capi

W, H, SPP = 128, 72, 4


def terrain(n_tris: int, size: float = 50.0, seed: int = 1):
    """A k x k height field of float vertices, two triangles per cell, per-vertex UVs."""
    k = max(2, int(np.sqrt(n_tris / 2)) + 1)
    xs = np.linspace(-size, size, k, dtype=np.float32)
    X, Z = np.meshgrid(xs, xs, indexing="ij")
    rng = np.random.default_rng(seed)
    Y = (3.0 * np.sin(0.21 * X) * np.cos(0.17 * Z) * size / 50.0 + 0.05 * size / 50.0 * rng.standard_normal(X.shape)).astype(np.float32)
    pos = np.ascontiguousarray(np.stack([X, Y, Z], axis=-1).reshape(-1, 3))
    v = np.arange(k * k, dtype=np.uint32).reshape(k, k)
    a, b, c, d = v[:-1, :-1].ravel(), v[1:, :-1].ravel(), v[1:, 1:].ravel(), v[:-1, 1:].ravel()
    idx = np.empty((2 * len(a), 3), dtype=np.uint32)
    idx[0::2] = np.stack([a, b, c], axis=1)
    idx[1::2] = np.stack([a, c, d], axis=1)
    u = np.linspace(0, 1, k, dtype=np.float32)
    U, V = np.meshgrid(u, u, indexing="ij")
    uvs = np.ascontiguousarray(np.stack([U, V], axis=-1).reshape(-1, 2))
    return pos, np.ascontiguousarray(idx), uvs


def rot_y(deg, t):
    x = capi.rt_xform()
    c, s = np.cos(np.radians(deg)), np.sin(np.radians(deg))
    x.r[:] = [c, 0, s, 0, 1, 0, -s, 0, c]
    x.t[:] = t
    return x


class MeshScene:
    """A scene description built in numpy around indexed meshes.  arrays: [(positions, indices, uvs | None,
    uv_indices | None)]; meshes: [(array set, material, xform)]; world: [(type, index)]; spheres: [(centre, radius,
    material)].  Materials: 0 image-textured lambertian, 1 grey lambertian, 2 metal, 3 diffuse light."""

    def __init__(self, arrays, meshes, world, spheres=((0.0, -1010.0, 0.0, 1000.0, 1),), xforms=(), light=False,
                 camera=((0.0, 40.0, 90.0), (0.0, 0.0, 0.0), 45.0)):
        self.arrays = [tuple(None if a is None else np.ascontiguousarray(a) for a in s) for s in arrays]
        d = capi.rt_scene_desc()
        d.struct_size, d.abi_version = C.sizeof(d), capi.RT_B200_ABI_VERSION
        self.mesh = (capi.rt_mesh * max(1, len(meshes)))()
        for i, (s, mat, xf) in enumerate(meshes):
            pos, idx, uvs, uvi = self.arrays[s]
            m = self.mesh[i]
            m.positions = pos.ctypes.data_as(C.POINTER(C.c_float))
            m.indices = idx.ctypes.data_as(C.POINTER(C.c_uint32))
            m.n_vertices, m.n_triangles = len(pos), len(idx)
            if uvs is not None:
                m.uvs, m.n_uvs = uvs.ctypes.data_as(C.POINTER(C.c_float)), len(uvs)
            if uvi is not None:
                m.uv_indices = uvi.ctypes.data_as(C.POINTER(C.c_uint32))
            m.material, m.xform = mat, xf
        d.meshes, d.n_meshes = self.mesh, len(meshes)
        self.world = (capi.rt_prim_ref * len(world))(*[capi.rt_prim_ref(t, i) for t, i in world])
        d.world, d.n_world = self.world, len(world)
        self.sph = (capi.rt_sphere * max(1, len(spheres)))()
        for i, (x, y, z, r, mat) in enumerate(spheres):
            self.sph[i].center0[:] = [x, y, z]
            self.sph[i].radius, self.sph[i].material, self.sph[i].xform = r, mat, -1
        d.spheres, d.n_spheres = self.sph, len(spheres)
        self.quad = (capi.rt_quad * 1)()
        if light:
            q = self.quad[0]
            q.Q[:], q.u[:], q.v[:] = [-10.0, 30.0, -10.0], [20.0, 0.0, 0.0], [0.0, 0.0, 20.0]
            q.material, q.xform = 3, -1
            d.quads, d.n_quads = self.quad, 1
        self.xf = (capi.rt_xform * max(1, len(xforms)))(*xforms)
        d.xforms, d.n_xforms = self.xf, len(xforms)
        self.mats = (capi.rt_material * 4)()
        self.texs = (capi.rt_texture * 4)()
        for i, (mt, tex, col) in enumerate([(capi.RT_MAT_LAMBERTIAN, 0, None), (capi.RT_MAT_LAMBERTIAN, 1, (0.5, 0.5, 0.5)),
                                            (capi.RT_MAT_METAL, -1, None), (capi.RT_MAT_DIFFUSE_LIGHT, 2, (4.0, 4.0, 4.0))]):
            self.mats[i].type, self.mats[i].texture = mt, tex
            if col:
                self.texs[tex].type = capi.RT_TEX_SOLID
                self.texs[tex].color[:] = col
        self.mats[2].albedo[:], self.mats[2].param = [0.8, 0.7, 0.6], 0.05
        self.texels = np.random.default_rng(7).integers(0, 256, (64, 64, 3), dtype=np.uint8)
        self.img = (capi.rt_image * 1)()
        self.img[0].width, self.img[0].height = 64, 64
        self.img[0].rgb = self.texels.ctypes.data_as(C.POINTER(C.c_uint8))
        self.texs[0].type, self.texs[0].image = capi.RT_TEX_IMAGE, 0
        d.materials, d.n_materials = self.mats, 4
        d.textures, d.n_textures = self.texs, 3
        d.images, d.n_images = self.img, 1
        (f, a, vfov) = camera
        d.camera.lookfrom[:], d.camera.lookat[:], d.camera.vup[:] = f, a, [0.0, 1.0, 0.0]
        d.camera.vfov, d.camera.focus_dist = vfov, 10.0
        d.camera.background[:] = [0.7, 0.8, 1.0]
        self.desc = d
        self.desc_ptr = C.pointer(d)


def one_terrain(n_tris):
    pos, idx, uvs = terrain(n_tris)
    return MeshScene([(pos, idx, uvs, None)], [(0, 0, -1)], [(capi.RT_PRIM_SPHERE, 0), (capi.RT_PRIM_MESH, 0)])


def run(scene, builder, width=2, nee=False, device=0, aov=True):
    c = capi.Context(device)
    c.set_bvh_builder(builder)
    c.set_bvh_width(width)
    c.upload(scene)
    st = c.stats()
    c.render(W, H, SPP, max_depth=8, seed=3, nee=nee)
    out = {"acc": c.accum_download(), "st": st}
    if aov:
        out["aov"] = c.aov(W, H)
    c.close()
    return out


def check_same(indexed, builder, width=2, nee=False):
    expanded = Expanded(indexed.desc)
    a, b = run(indexed, builder, width, nee), run(expanded, builder, width, nee)
    assert a["st"]["bvh_on_device"] == (builder != "host")
    assert np.array_equal(a["acc"], b["acc"]), "accumulated sums differ"
    assert a["acc"][..., :3].sum() > 0
    for k in ("prim_id", "t", "normal", "uv"):
        assert np.array_equal(a["aov"][k], b["aov"][k]), k
    for k in ("bvh_nodes", "bvh_leaves", "bvh_depth"):
        assert a["st"][k] == b["st"][k], k
    return a


CONFIGS = [("host", 2), ("host", 8), ("device", 2), ("lbvh", 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mesh", "kitchen_sink"])
@pytest.mark.parametrize("builder,width", CONFIGS)
def test_baseline_scene_with_indexed_meshes(built, name, builder, width):
    sc = capi.Scene(name, indexed=True)
    a = check_same(sc, builder, width)
    # and the same bits as the soup form the scene builder makes by default
    assert np.array_equal(a["acc"], run(capi.Scene(name), builder, width, aov=False)["acc"])


@pytest.mark.gpu
@pytest.mark.parametrize("builder,width", CONFIGS)
def test_200k_terrain_with_an_image_texture(built, builder, width):
    sc = one_terrain(200_000)
    a = check_same(sc, builder, width)
    assert (a["aov"]["prim_id"] >= 1).mean() > 0.2   # the terrain fills much of the frame (id 0 is the ground sphere)


@pytest.mark.gpu
def test_2m_terrain_on_the_device_path(built):
    sc = one_terrain(2_000_000)
    check_same(sc, "device")


@pytest.mark.gpu
@pytest.mark.parametrize("builder,width", CONFIGS)
def test_transformed_mesh_between_spheres_and_shared_arrays(built, builder, width):
    pos, idx, uvs = terrain(20_000, size=6.0)
    uvi = np.ascontiguousarray(idx[:, ::-1])    # uv indices of their own
    xf = [rot_y(30.0, [5.0, 4.0, 0.0]), rot_y(-60.0, [-8.0, 2.0, 5.0])]
    spheres = ((0.0, -1010.0, 0.0, 1000.0, 1), (0.0, 6.0, 0.0, 5.0, 2), (12.0, 3.0, -4.0, 3.0, 1))
    # a mesh between two spheres in the world list, under translate / rotate_y
    sc = MeshScene([(pos, idx, uvs, uvi)], [(0, 0, 0)],
                   [(capi.RT_PRIM_SPHERE, 0), (capi.RT_PRIM_SPHERE, 1), (capi.RT_PRIM_MESH, 0), (capi.RT_PRIM_SPHERE, 2)],
                   spheres=spheres, xforms=xf, light=True)
    check_same(sc, builder, width)
    # two meshes sharing the same arrays, one of them without UVs
    sc2 = MeshScene([(pos, idx, uvs, uvi), (pos, idx, None, None)], [(0, 0, 0), (1, 1, 1), (0, 0, -1)],
                    [(capi.RT_PRIM_MESH, 0), (capi.RT_PRIM_SPHERE, 0), (capi.RT_PRIM_MESH, 1), (capi.RT_PRIM_MESH, 2)],
                    spheres=spheres[:1], xforms=xf)
    check_same(sc2, builder, width)


@pytest.mark.gpu
@pytest.mark.parametrize("builder", ["host", "device"])
def test_next_event_estimation(built, builder):
    pos, idx, uvs = terrain(20_000, size=20.0)
    sc = MeshScene([(pos, idx, uvs, None)], [(0, 0, -1)], [(capi.RT_PRIM_MESH, 0), (capi.RT_PRIM_SPHERE, 0)], light=True)
    check_same(sc, builder, nee=True)


# ---- malformed input --------------------------------------------------------------------------------------


def _expect(c, scene, code, *words):
    with pytest.raises(capi.RtError) as e:
        c.upload(scene)
    assert e.value.code == code, str(e.value)
    for w in words:
        assert w in str(e.value)


@pytest.mark.gpu
@pytest.mark.parametrize("builder,n_tris", [("host", 2_000), ("device", 70_000)])
def test_malformed_meshes_are_refused(built, builder, n_tris):
    pos, idx, uvs = terrain(n_tris)
    n, nv = len(idx), len(pos)
    assert builder == "host" or n >= 1 << 16
    good = MeshScene([(pos, idx, uvs, None)], [(0, 0, -1)], [(capi.RT_PRIM_SPHERE, 0), (capi.RT_PRIM_MESH, 0)])
    c = capi.Context(0)
    c.set_bvh_builder(builder)

    def with_mesh(**fields):
        s = MeshScene([(pos, fields.pop("indices", idx), uvs, fields.pop("uv_indices", None))], [(0, 0, -1)],
                      [(capi.RT_PRIM_SPHERE, 0), (capi.RT_PRIM_MESH, 0)])
        for k, v in fields.items():
            setattr(s.mesh[0], k, v)
        return s

    def index_past_end(tri, corner, value):
        bad = idx.copy()
        bad[tri, corner] = value
        return with_mesh(indices=bad)

    cases = [
        (index_past_end(0, 0, nv), capi.RT_ERR_INVALID, ["meshes[0]", "triangle 0:"]),
        (index_past_end(n // 2, 1, nv + 100), capi.RT_ERR_INVALID, ["meshes[0]", f"triangle {n // 2}:"]),
        (index_past_end(n - 1, 2, 0xFFFFFFFF), capi.RT_ERR_INVALID, ["meshes[0]", f"triangle {n - 1}:"]),
    ]
    bad_uv = idx.copy()
    bad_uv[n // 3, 0] = nv
    cases.append((with_mesh(uv_indices=bad_uv), capi.RT_ERR_INVALID, ["uv index", f"triangle {n // 3}:"]))
    cases.append((with_mesh(n_uvs=nv - 1), capi.RT_ERR_INVALID, ["n_uvs"]))
    cases.append((with_mesh(positions=None), capi.RT_ERR_INVALID, ["null"]))
    s = with_mesh()
    s.mesh[0].indices = None
    cases.append((s, capi.RT_ERR_INVALID, ["null"]))
    cases.append((with_mesh(n_triangles=-1), capi.RT_ERR_INVALID, ["negative"]))
    s = with_mesh()
    s.desc.n_meshes = -1
    cases.append((s, capi.RT_ERR_INVALID, ["negative"]))
    s = with_mesh()
    s.world[1] = capi.rt_prim_ref(capi.RT_PRIM_MESH, 1)
    cases.append((s, capi.RT_ERR_INVALID, ["world[1]", "mesh index"]))
    cases.append((with_mesh(material=99), capi.RT_ERR_INVALID, ["material"]))
    cases.append((with_mesh(xform=0), capi.RT_ERR_INVALID, ["xform"]))
    # a mesh as the boundary of a medium
    s = with_mesh()
    s.bref = (capi.rt_prim_ref * 1)(capi.rt_prim_ref(capi.RT_PRIM_MESH, 0))
    s.media = (capi.rt_medium * 1)()
    s.media[0].boundary_first, s.media[0].boundary_count, s.media[0].density = 0, 1, 0.5
    s.media[0].multiplicity, s.media[0].material, s.media[0].xform = 1, 1, -1
    s.desc.boundary_refs, s.desc.n_boundary_refs = s.bref, 1
    s.desc.media, s.desc.n_media = s.media, 1
    cases.append((s, capi.RT_ERR_UNSUPPORTED, ["boundary"]))
    # 2^25 primitives once expanded: 32768 refs to one 1024-triangle mesh
    p2, i2, _ = terrain(1100)
    i2 = np.ascontiguousarray(i2[:1024])
    s = MeshScene([(p2, i2, None, None)], [(0, 0, -1)], [(capi.RT_PRIM_MESH, 0)] * 32768)
    cases.append((s, capi.RT_ERR_UNSUPPORTED, ["2^25"]))
    for scene, code, words in cases:
        _expect(c, scene, code, *words)
        c.upload(good)   # a valid upload succeeds after every refusal
        assert c.stats()["bvh_on_device"] == (builder == "device")
    c.render(W, H, 1, max_depth=4)
    c.close()


# ---- ABI 3, scene cache, upload bytes ---------------------------------------------------------------------


@pytest.mark.gpu
def test_abi3_descriptor_renders_like_its_v4_twin(built):
    sc = capi.Scene("kitchen_sink")
    raw = bytearray(C.string_at(C.addressof(sc.desc), capi.RT_SCENE_DESC_V3_SIZE))
    raw[0:8] = np.array([capi.RT_SCENE_DESC_V3_SIZE, 3], dtype=np.uint32).tobytes()
    buf = C.create_string_buffer(bytes(raw), len(raw))
    v3 = C.cast(buf, C.POINTER(capi.rt_scene_desc))
    frames = []
    for scene in (v3, sc):
        c = capi.Context(0)
        c.upload(scene)
        c.render(W, H, SPP, max_depth=8, seed=3)
        frames.append(c.accum_download())
        c.close()
    assert np.array_equal(frames[0], frames[1])
    # any other size / version pair is refused
    c = capi.Context(0)
    for size, version in [(capi.RT_SCENE_DESC_V3_SIZE, 4), (C.sizeof(capi.rt_scene_desc), 3)]:
        raw[0:8] = np.array([size, version], dtype=np.uint32).tobytes()
        full = C.create_string_buffer(bytes(raw) + bytes(C.sizeof(capi.rt_scene_desc) - len(raw)))
        _expect(c, C.cast(full, C.POINTER(capi.rt_scene_desc)), capi.RT_ERR_INVALID, "ABI")
    c.close()


@pytest.mark.gpu
def test_scene_cache_sees_a_moved_vertex(built):
    sc = one_terrain(20_000)
    c = capi.Context(0)
    c.set_bvh_builder("host")
    c.upload(sc)
    assert c.stats()["scene_reused"] == 0
    c.render(W, H, SPP, max_depth=8, seed=3)
    first = c.accum_download()
    c.upload(sc)
    assert c.stats()["scene_reused"] == 1
    c.render(W, H, SPP, max_depth=8, seed=3)
    assert np.array_equal(c.accum_download(), first)
    pos = sc.arrays[0][0]
    pos[len(pos) // 2 + 70, 1] += 25.0    # one vertex near the middle of the terrain, moved in place
    c.upload(sc)
    assert c.stats()["scene_reused"] == 0
    c.render(W, H, SPP, max_depth=8, seed=3)
    assert not np.array_equal(c.accum_download(), first)
    # device-path scenes are not fingerprinted, so never reused
    c.set_bvh_builder("device")
    c.upload(sc)
    c.upload(sc)
    assert c.stats()["scene_reused"] == 0 and c.stats()["bvh_on_device"] == 1
    c.close()


@pytest.mark.gpu
def test_indexed_upload_copies_a_third_of_the_bytes(built):
    """Counted, not timed: at 1 M triangles with UVs the device path copies the float vertices, the UVs and 12 bytes
    of indices per triangle instead of 104-byte rt_triangle records and 8-byte refs."""
    sc = one_terrain(1_000_000)
    up = {}
    for form, scene in (("indexed", sc), ("soup", Expanded(sc.desc))):
        c = capi.Context(0)
        c.set_bvh_builder("device")
        c.upload(scene)
        st = c.stats()
        assert st["bvh_on_device"] == 1
        up[form] = st["upload_bytes"]
        c.close()
    assert up["soup"] >= 112 * sc.mesh[0].n_triangles
    assert up["indexed"] <= 0.35 * up["soup"], up


# ---- camera::render, multi-device ---------------------------------------------------------------------------


def _render_mesh(tmp_path, name, spp, asset_dir, ckpt=None, stop=0):
    s = capi.load_scenes()
    out = str(tmp_path / name)
    done, resumed = C.c_int(), C.c_int()
    with capi.indexed_meshes(True):
        rc = s.rtsc_render_resumable(b"mesh", 1, asset_dir.encode(), 96, 54, spp, 8, out.encode(), ckpt.encode() if ckpt else None,
                                     0, stop, None, C.byref(done), C.byref(resumed))
    assert rc == 0
    return open(out, "rb").read(), done.value, resumed.value


@pytest.mark.gpu
def test_checkpoint_resume_with_indexed_meshes(built, tmp_path):
    from raytracingoneweekendapplication_b200.assets import ensure_assets

    assets = ensure_assets()
    ck = str(tmp_path / "mesh.ckpt")
    ref_png, done, _ = _render_mesh(tmp_path, "ref.png", 6, assets)
    assert done == 6
    _, done, _ = _render_mesh(tmp_path, "part.png", 6, assets, ckpt=ck, stop=3)
    assert done == 3 and os.path.exists(ck)
    png, done, resumed = _render_mesh(tmp_path, "full.png", 6, assets, ckpt=ck)
    assert (done, resumed) == (6, 3) and png == ref_png
    # a checkpoint of the same scene with one vertex of one mesh moved is ignored
    moved = str(tmp_path / "assets")
    shutil.copytree(assets, moved)
    lines = open(os.path.join(moved, "knot.obj")).read().split("\n")
    k = next(i for i, ln in enumerate(lines) if ln.startswith("v "))
    x, y, z = map(float, lines[k].split()[1:4])
    lines[k] = f"v {x} {y + 0.5} {z}"
    open(os.path.join(moved, "knot.obj"), "w").write("\n".join(lines))
    _render_mesh(tmp_path, "part2.png", 6, assets, ckpt=ck, stop=3)
    _, done, resumed = _render_mesh(tmp_path, "other.png", 6, moved, ckpt=ck)
    assert (done, resumed) == (6, 0)


def _gpu_count() -> int:
    import torch

    return torch.cuda.device_count()


@pytest.mark.gpu
@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_two_device_context(built):
    sc = capi.Scene("mesh", indexed=True)
    frames = []
    for dev in (0, [0, 1]):
        c = capi.Context(dev)
        c.upload(sc)
        c.render(W, H, SPP, max_depth=8, seed=3)
        frames.append(c.download(SPP))
        c.close()
    assert np.array_equal(frames[0], frames[1])
