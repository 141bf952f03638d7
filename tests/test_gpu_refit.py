"""rt_refit_scene (csrc/bvh_refit.cuh): a changed scene of the same structure replaces the uploaded one without a tree
build.  The records are derived by the same code as an upload's (csrc/prim_derive.h) and the closest hit does not
depend on the tree, so frames are compared for EQUALITY with a fresh upload of the changed scene; the only legitimate
differences are rays that hit two primitives at exactly the same t (shared edges of the Cornell box)."""
import ctypes as C
import math

import numpy as np
import pytest

import fuzz_scenes

pytestmark = pytest.mark.gpu
from raytracingoneweekendapplication_b200 import capi  # noqa: E402

W, H, SPP = 96, 64, 2

_ARRAYS = [("world", capi.rt_prim_ref, "n_world"), ("boundary_refs", capi.rt_prim_ref, "n_boundary_refs"),
           ("spheres", capi.rt_sphere, "n_spheres"), ("quads", capi.rt_quad, "n_quads"),
           ("triangles", capi.rt_triangle, "n_triangles"), ("media", capi.rt_medium, "n_media"),
           ("xforms", capi.rt_xform, "n_xforms"), ("materials", capi.rt_material, "n_materials"),
           ("textures", capi.rt_texture, "n_textures"), ("images", capi.rt_image, "n_images"),
           ("perlins", capi.rt_perlin, "n_perlins"), ("lights", capi.rt_point_light, "n_lights"),
           ("meshes", capi.rt_mesh, "n_meshes")]


class Copy:
    """A scene description whose arrays (and mesh positions) are copies that a test may change; exposes .desc_ptr."""

    def __init__(self, scene, extra=None):
        src = scene.desc
        self._src = scene
        self._keep = []
        d = capi.rt_scene_desc()
        C.memmove(C.byref(d), C.byref(src), C.sizeof(d))
        self.arr = {}
        for field, ctype, count in _ARRAYS:
            n = getattr(d, count) + (extra or {}).get(count, 0)
            a = (ctype * max(1, n))()
            m = min(n, getattr(src, count))
            if m:
                C.memmove(a, getattr(src, field), m * C.sizeof(ctype))
            for i in range(m, n):   # grown arrays repeat their first element (or stay zero)
                if m:
                    a[i] = a[0]
            setattr(d, field, C.cast(a, C.POINTER(ctype)))
            setattr(d, count, n)
            self.arr[field] = a
            self._keep.append(a)
        self.positions = []
        for i in range(min(d.n_meshes, src.n_meshes)):
            m = src.meshes[i]
            p = np.ctypeslib.as_array(m.positions, shape=(m.n_vertices * 3,)).copy()
            self._keep.append(p)
            self.positions.append(p)
            self.arr["meshes"][i].positions = p.ctypes.data_as(C.POINTER(C.c_float))
        self.desc = d
        self.desc_ptr = C.pointer(d)


def moved(scene, k=1):
    """`scene` with every xform turned by 7k degrees about y and shifted, and every triangle and mesh vertex shifted."""
    c = Copy(scene)
    a = math.radians(7.0 * k)
    ry = np.array([[math.cos(a), 0, math.sin(a)], [0, 1, 0], [-math.sin(a), 0, math.cos(a)]])
    shift = np.array([0.05 * k, 0.02 * k, -0.03 * k])
    for x in c.arr["xforms"][:c.desc.n_xforms]:
        r = ry @ np.array(x.r[:]).reshape(3, 3)
        x.r[:] = list(r.reshape(-1))
        x.t[:] = list(ry @ np.array(x.t[:]) + shift)
    for t in c.arr["triangles"][:c.desc.n_triangles]:
        for p in (t.p0, t.p1, t.p2):
            p[:] = [p[i] + shift[i] for i in range(3)]
    for p in c.positions:
        p.reshape(-1, 3)[:] += shift.astype(np.float32)
    return c


def emitters(desc):
    """Quads of the world list with an emissive material (each one an entry of the next-event emitter list)."""
    return sum(1 for i in range(desc.n_world) if desc.world[i].type == 1
               and desc.materials[desc.quads[desc.world[i].index].material].type in (3, 4))


def frame(c, sc, nee=False, moments=False, **kw):
    c.render(W, H, SPP, max_depth=sc.depth, seed=7, nee=nee, moments=moments, **kw)
    return c.accum_download()


def fresh(scene, fn, builder="auto"):
    c = capi.Context(0)
    try:
        c.set_bvh_builder(builder)
        c.upload(scene)
        return fn(c)
    finally:
        c.close()


@pytest.fixture
def context():
    c = capi.Context(0)
    yield c
    c.close()


def _random_spheres():
    return fuzz_scenes.random_scene(11, 300, 0, 0, with_xforms=True)


@pytest.mark.parametrize("builder", ["host", "device"])
@pytest.mark.parametrize("name", ["final", "mesh", "spheres"])
def test_refit_equals_a_fresh_upload(scene_of, context, name, builder):
    sc = _random_spheres() if name == "spheres" else scene_of(name)
    depth = getattr(sc, "depth", 8)
    b = moved(sc)
    b.depth = depth
    if name == "spheres":
        sc.depth = depth
    context.set_bvh_builder(builder)
    context.upload(sc)
    st = context.stats()
    assert st["bvh_on_device"] == (1 if builder == "device" else 0)
    context.refit(b)
    after = context.stats()
    for k in ("bvh_nodes", "bvh_depth", "bvh_leaves", "bvh_on_device"):
        assert after[k] == st[k], k
    assert after["upload_bytes"] > 0 and after["scene_reused"] == 0
    got = frame(context, b, moments=True)
    got_m = context.moments_download()
    want, want_m = fresh(b, lambda c: (frame(c, b, moments=True), c.moments_download()), builder)
    assert np.array_equal(got, want)
    assert np.array_equal(got_m, want_m)
    if builder == "device" or emitters(b.desc) <= 1:   # host-built: the emitter list keeps the uploaded leaf order
        assert np.array_equal(frame(context, b, nee=True), fresh(b, lambda c: frame(c, b, nee=True), builder))


@pytest.mark.parametrize("name", ["book1", "final", "mesh", "kitchen_sink", "quads", "cornell", "cornell_smoke", "mixed"])
def test_refit_primary_hits_match_a_fresh_upload(scene_of, context, name):
    sc = scene_of(name)
    b = moved(sc)
    w, h = 160, 120
    context.upload(sc)
    context.refit(b)
    got = context.aov(w, h)
    want = fresh(b, lambda c: c.aov(w, h))
    assert np.array_equal(got["t"], want["t"]), f"{name}: primary t differs"
    tie = got["prim_id"] != want["prim_id"]
    assert tie.mean() <= 0.01, f"{name}: primary ids differ on {tie.sum()} pixels"
    if name not in ("kitchen_sink", "cornell"):
        assert not tie.any()
    assert np.array_equal(got["normal"][~tie], want["normal"][~tie])


def test_animation_sequence_and_return(scene_of, context):
    sc = scene_of("final")
    context.upload(sc)
    for k in range(1, 9):
        b = moved(sc, k)
        b.depth = sc.depth
        context.refit(b)
        assert np.array_equal(frame(context, b), fresh(b, lambda c: frame(c, b))), k
    context.refit(sc)
    a_frame = fresh(sc, lambda c: frame(c, sc))
    assert np.array_equal(frame(context, sc), a_frame)
    # upload(A), refit(B), upload(A): A (the staged arena of A may be reused); then upload(B): B
    b = moved(sc, 3)
    b.depth = sc.depth
    context.upload(sc)
    context.refit(b)
    context.upload(sc)
    assert np.array_equal(frame(context, sc), a_frame)
    context.upload(b)
    assert np.array_equal(frame(context, b), fresh(b, lambda c: frame(c, b)))


def test_materials_camera_and_lights_follow(scene_of, context):
    # the geometry stays: the refitted tree is the tree a fresh upload builds, so even the coincident faces of
    # kitchen_sink resolve alike
    sc = scene_of("kitchen_sink")
    b = Copy(sc)
    b.depth = sc.depth
    for m in b.arr["materials"][:b.desc.n_materials]:
        m.albedo[:] = [0.9 * v for v in m.albedo]
    b.desc.camera.lookfrom[0] += 0.5
    b.desc.camera.vfov *= 1.1
    for lt in b.arr["lights"][:b.desc.n_lights]:
        lt.intensity[:] = [2.0 * v for v in lt.intensity]
    context.upload(sc)
    context.refit(b)
    assert np.array_equal(frame(context, b, shadowed_point_lights=True), fresh(b, lambda c: frame(c, b, shadowed_point_lights=True)))


def test_a_new_specular_material_switches_the_instance(scene_of, context):
    sc = scene_of("book1")
    b = moved(sc)
    b.depth = sc.depth
    mats = b.arr["materials"]
    for i in range(b.desc.n_materials):
        if mats[i].type == 0:
            mats[i].type = 6   # RT_MAT_SPECULAR
            break
    context.upload(sc)
    context.refit(b)
    assert np.array_equal(frame(context, b), fresh(b, lambda c: frame(c, b)))


def test_refit_is_ordered_after_passes_in_flight(scene_of, context):
    sc = scene_of("final")
    b = moved(sc)
    b.depth = sc.depth
    want_a = fresh(sc, lambda c: frame(c, sc, accumulate=False))
    context.upload(sc)
    context.render(W, H, SPP, max_depth=sc.depth, seed=7, blocking=False)
    context.refit(b)
    assert np.array_equal(context.accum_download(), want_a)
    assert np.array_equal(frame(context, b), fresh(b, lambda c: frame(c, b)))
    # overlapped accumulate passes of A in flight
    def passes(c, s):
        c.render(W, H, 1, max_depth=s.depth, seed=7, blocking=False)
        for i in (1, 2):
            c.render(W, H, 1, max_depth=s.depth, seed=7, spp_begin=i, accumulate=True, blocking=False, overlap=True)
    context.upload(sc)
    passes(context, sc)
    context.refit(b)
    want = fresh(sc, lambda c: (passes(c, sc), c.sync(), c.accum_download())[2])
    assert np.array_equal(context.accum_download(), want)


def test_two_device_context_after_refit(scene_of, monkeypatch):
    monkeypatch.setenv("RT_B200_ALLOW_DUPLICATE_DEVICES", "1")
    sc = scene_of("final")
    b = moved(sc)
    b.depth = sc.depth

    def one(c1, s):
        c1.render(W, H, SPP, max_depth=s.depth, seed=7)
        return c1.download(SPP)

    c = capi.Context([0, 0])
    try:
        c.upload(sc)
        c.render(W, H, SPP, max_depth=sc.depth, seed=7)
        with pytest.raises(capi.RtError):   # a refused refit keeps the frame the devices hold
            c.refit(_changes(sc)[-1][1])
        assert np.array_equal(c.download(SPP), fresh(sc, lambda c1: one(c1, sc)))
        c.refit(b)
        got = one(c, b)
    finally:
        c.close()
    assert np.array_equal(got, fresh(b, lambda c1: one(c1, b)))


def test_device_built_emitter_follows_its_source_quad(scene_of, context):
    """A device-built tree numbers the next-event emitters by source quad.  The world ref of the light and the world ref
    of a ground quad trade their quads: the emitter list is the same, but the light now sits in the other slot."""
    sc = scene_of("final")
    d = sc.desc
    light = next(i for i in range(d.n_world) if d.world[i].type == 1 and d.materials[d.quads[d.world[i].index].material].type == 3)
    other = next(i for i in range(d.n_world) if d.world[i].type == 1 and i != light)
    b = Copy(sc)
    b.depth = sc.depth
    wl = b.arr["world"]
    wl[light].index, wl[other].index = d.world[other].index, d.world[light].index
    context.set_bvh_builder("device")
    context.upload(sc)
    context.refit(b)
    for nee in (False, True):
        assert np.array_equal(frame(context, b, nee=nee), fresh(b, lambda c: frame(c, b, nee=nee), "device")), nee
    # a host-built tree numbers them by canonical primitive: the light moved to another primitive, the list changed
    host = capi.Context(0)
    try:
        host.set_bvh_builder("host")
        host.upload(sc)
        with pytest.raises(capi.RtError) as e:
            host.refit(b)
        assert e.value.code == capi.RT_ERR_INVALID and "emitter" in str(e.value)
    finally:
        host.close()


def test_refit_after_a_refused_upload(scene_of, context):
    """An upload that fails validation leaves the uploaded scene in place; it still refits like that scene."""
    sc = scene_of("final")
    b = moved(sc)
    b.depth = sc.depth
    context.upload(sc)
    with pytest.raises(capi.RtError):
        context.upload(_changes(sc)[-1][1])   # an out-of-range index
    context.refit(b)
    assert np.array_equal(frame(context, b), fresh(b, lambda c: frame(c, b)))


def test_views_after_refit(scene_of, context):
    sc = scene_of("final")
    b = moved(sc)
    cam2 = capi.rt_camera()
    C.memmove(C.byref(cam2), C.byref(b.desc.camera), C.sizeof(cam2))
    cam2.lookfrom[0] += 30.0
    cams = [b.desc.camera, cam2]

    def views(c):
        c.render_views(cams, W, H, SPP, max_depth=sc.depth, seed=3)
        return c.download_views(SPP)

    context.upload(sc)
    context.refit(b)
    assert np.array_equal(views(context), fresh(b, views))


def _changes(sc):
    """(label, description, expected code): each a refit `sc` must refuse."""
    out = []
    d = sc.desc
    for _, _, count in _ARRAYS:
        if getattr(d, count) > 0:
            out.append((count, Copy(sc, {count: 1}), capi.RT_ERR_INVALID))
    mov = Copy(sc)   # a static sphere starts moving and the moving one stops: same counts, two kinds change
    sph = mov.arr["spheres"]
    moving = [i for i in range(d.n_spheres) if any(sph[i].center_vec[k] for k in range(3))]
    static = [i for i in range(d.n_spheres) if i not in moving]
    sph[static[0]].center_vec[:] = [0.0, 0.1, 0.0]
    sph[moving[0]].center_vec[:] = [0.0, 0.0, 0.0]
    out.append(("sphere starts moving", mov, capi.RT_ERR_INVALID))
    one = Copy(sc)   # only one sphere starts moving: the world's counts of each kind change
    one.arr["spheres"][static[1]].center_vec[:] = [0.1, 0.0, 0.0]
    out.append(("counts of a kind", one, capi.RT_ERR_INVALID))
    swap = Copy(sc)  # a sphere ref and a quad ref trade places: same counts, two world refs change type
    wl = swap.arr["world"]
    i = next(k for k in range(d.n_world) if wl[k].type == 0)
    j = next(k for k in range(d.n_world) if wl[k].type == 1)
    wl[i], wl[j] = capi.rt_prim_ref(wl[j].type, wl[j].index), capi.rt_prim_ref(wl[i].type, wl[i].index)
    out.append(("world ref changes type", swap, capi.RT_ERR_INVALID))
    dark = Copy(sc)  # the light quad's material stops emitting
    for m in dark.arr["materials"][:d.n_materials]:
        if m.type == 3:
            m.type = 0
    out.append(("emitter loses its light", dark, capi.RT_ERR_INVALID))
    bad = Copy(sc)
    bad.arr["world"][0].index = d.n_spheres + d.n_quads + 100
    out.append(("index out of range", bad, capi.RT_ERR_INVALID))
    return out


def test_refused_refits_leave_the_scene_intact(scene_of, context):
    sc = scene_of("final")
    want = fresh(sc, lambda c: frame(c, sc))
    with pytest.raises(capi.RtError) as e:
        context.refit(sc)
    assert e.value.code == capi.RT_ERR_STATE
    context.upload(sc)
    st = context.stats()
    for label, desc, code in _changes(sc):
        with pytest.raises(capi.RtError) as e:
            context.refit(desc)
        assert e.value.code == code, label
        assert "rt_refit_scene" in str(e.value), label
        assert np.array_equal(frame(context, sc), want), label
    for k in ("bvh_nodes", "bvh_depth", "bvh_leaves"):
        assert context.stats()[k] == st[k]


def test_wide_tree_is_unsupported(scene_of, context):
    sc = scene_of("book1")
    context.set_bvh_width(4)
    context.upload(sc)
    assert context.stats()["bvh_width"] == 4
    want = frame(context, sc)
    with pytest.raises(capi.RtError) as e:
        context.refit(moved(sc))
    assert e.value.code == capi.RT_ERR_UNSUPPORTED
    assert np.array_equal(frame(context, sc), want)
