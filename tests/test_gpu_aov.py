"""Auxiliary render outputs (RT_FLAG_AOV): antialiased first-hit albedo, normal and depth, and the coverage of the hits.

They are exact integer sums over the same camera samples as the radiance, so the image must not change, every way of
scheduling the samples must give the same floats bit for bit, and on simple geometry the resolved values are known."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import fuzz_scenes
from raytracingoneweekendapplication_b200 import capi

pytestmark = pytest.mark.gpu

W, H = 64, 48


def _all(d):
    """The (H, W, 8) array behind the views download_aov returns."""
    return d["albedo"].base


def _code(fn, *a, **kw):
    with pytest.raises(capi.RtError) as e:
        fn(*a, **kw)
    return e.value.code


@pytest.mark.parametrize("name", ["book1", "cornell", "cornell_smoke", "mesh", "final"])
@pytest.mark.parametrize("nee", [False, True])
def test_aov_leaves_the_image_unchanged(ctx, scene_of, name, nee):
    ctx.upload(scene_of(name))
    ctx.render(W, H, 6, seed=3, nee=nee)
    plain = ctx.accum_download()
    ctx.render(W, H, 6, seed=3, nee=nee, aov=True)
    assert np.array_equal(ctx.accum_download(), plain)
    a = ctx.download_aov(6)
    assert _all(a).shape == (H, W, 8) and a["coverage"].max() <= 1.0 and np.any(a["coverage"] > 0)
    assert np.all(np.abs(a["normal"]) <= 1.0) and np.all(a["depth"] >= 0)


def test_aov_does_not_depend_on_scheduling(ctx, scene_of, monkeypatch):
    sc, n, w, h = scene_of("cornell_smoke"), 12, 96, 80
    ctx.upload(sc)
    ctx.render(w, h, n, seed=5, aov=True)
    ref = _all(ctx.download_aov(n)).copy()
    sums = ctx.accum_download()

    def same():
        assert np.array_equal(_all(ctx.download_aov(n)), ref)
        assert np.array_equal(ctx.accum_download(), sums)

    for split in ([5, 4, 3], [1, 11]):  # accumulating passes
        begin = 0
        for k, s in enumerate(split):
            ctx.render(w, h, s, seed=5, spp_begin=begin, aov=True, accumulate=k > 0)
            begin += s
        same()
    ctx.render(w, h, 6, seed=5, aov=True, blocking=False)  # asynchronous passes
    ctx.render(w, h, 6, seed=5, spp_begin=6, aov=True, accumulate=True, blocking=False)
    same()
    ctx.render(w, h, 4, seed=5, aov=True)  # overlapped passes
    for begin in (4, 8):
        ctx.render(w, h, 4, seed=5, spp_begin=begin, aov=True, accumulate=True, blocking=False, overlap=True)
    ctx.sync()
    same()
    for tile in (8, 16, 32):
        ctx.render(w, h, n, seed=5, aov=True, tile_size=tile)
        same()

    # compact tile shards: the shard's own tiles, exactly zero elsewhere
    for count in (2, 4):
        for r in range(count):
            ctx.render(w, h, n, seed=5, aov=True, shard_rank=r, shard_count=count, shard_mode=capi.RT_SHARD_TILES, tile_size=16,
                       compact=True)
            got = _all(ctx.download_aov(n))
            own = _own_mask(w, h, 16, r, count)
            assert np.array_equal(got[own], ref[own]) and not np.any(got[~own])

    # two devices in one context (the same GPU twice where only one is visible)
    monkeypatch.setenv("RT_B200_ALLOW_DUPLICATE_DEVICES", "1")
    import torch
    md = capi.Context([0, 1] if torch.cuda.device_count() >= 2 else [0, 0])
    try:
        md.upload(sc)
        md.render(w, h, 5, seed=5, aov=True, shard_mode=capi.RT_SHARD_TILES, tile_size=16)
        md.render(w, h, 7, seed=5, spp_begin=5, aov=True, accumulate=True, shard_mode=capi.RT_SHARD_TILES, tile_size=16)
        assert np.array_equal(_all(md.download_aov(n)), ref)
        md.render(w, h, n, seed=5, aov=True, shard_mode=capi.RT_SHARD_SAMPLES)  # sample shards: no per-device AOVs
        assert _code(md.download_aov, n) == capi.RT_ERR_UNSUPPORTED
    finally:
        md.close()


def _own_mask(w, h, tile, rank, count):
    y, x = np.mgrid[0:h, 0:w]
    return ((y // tile) * ((w + tile - 1) // tile) + x // tile) % count == rank


# ---- known answers ---------------------------------------------------------------------------------------------------
EPS = 2.0 ** -27


def test_a_solid_quad_facing_a_pinhole_camera(built):
    colour, bg, D, half = (0.3, 0.6, 0.9), (0.5, 0.7, 1.0), 10.0, 2.0
    tex = capi.rt_texture()
    tex.type, tex.even, tex.odd, tex.image, tex.perlin = capi.RT_TEX_SOLID, -1, -1, -1, -1
    tex.color = fuzz_scenes.d3(colour)
    lam = capi.rt_material()
    lam.type, lam.texture = capi.RT_MAT_LAMBERTIAN, 0
    q = capi.rt_quad()  # u x v points back at the camera: the normal facing the rays is the quad's own, (0, 0, -1)
    q.Q, q.u, q.v = fuzz_scenes.d3((-half, -half, D)), fuzz_scenes.d3((0, 2 * half, 0)), fuzz_scenes.d3((2 * half, 0, 0))
    q.material, q.xform = 0, -1
    cam = capi.rt_camera()
    cam.lookfrom, cam.lookat, cam.vup = fuzz_scenes.d3((0, 0, 0)), fuzz_scenes.d3((0, 0, 1)), fuzz_scenes.d3((0, 1, 0))
    cam.vfov, cam.defocus_angle, cam.focus_dist = 40.0, 0.0, D
    cam.background = fuzz_scenes.d3(bg)
    sc = fuzz_scenes.PyScene([], [q], [], [], [lam], [tex], camera=cam)
    c = capi.Context(0)
    try:
        c.upload(sc)
        c.render(W, H, 16, max_depth=8, seed=2, aov=True)
        a = c.download_aov(16)
    finally:
        c.close()
    # the footprint of pixel (i, j) on the viewport, which lies in the quad's plane (focus_dist = D): x in
    # [-vw / 2 + i p, -vw / 2 + (i + 1) p], y likewise; lo / hi: the least and the largest |x| (|y|) over it
    vh = 2.0 * math.tan(math.radians(20.0)) * D
    vw, pw = vh * W / H, vh / H

    def extent(n, size):
        e0 = -size / 2 + np.arange(n) * pw
        e1 = e0 + pw
        return np.where(e0 * e1 <= 0, 0.0, np.minimum(np.abs(e0), np.abs(e1))), np.maximum(np.abs(e0), np.abs(e1))

    xlo, xhi = extent(W, vw)
    ylo, yhi = extent(H, vh)
    inside = (yhi[:, None] < half * 0.999) & (xhi[None, :] < half * 0.999)
    outside = (ylo[:, None] > half * 1.001) | (xlo[None, :] > half * 1.001)
    assert inside.sum() > 200 and outside.sum() > 1000
    cov, alb, nrm, dep = a["coverage"], a["albedo"].astype(np.float64), a["normal"].astype(np.float64), a["depth"].astype(np.float64)
    assert np.all(cov[inside] == 1.0)
    assert np.all(np.abs(alb[inside] - np.array(colour, dtype=np.float32)) <= EPS)
    assert np.all(np.abs(nrm[inside] - np.array([0.0, 0.0, -1.0])) <= EPS)
    r2lo = (xlo[None, :] ** 2 + ylo[:, None] ** 2) / D ** 2
    r2hi = (xhi[None, :] ** 2 + yhi[:, None] ** 2) / D ** 2
    lo, hi = D * np.sqrt(1 + r2lo), D * np.sqrt(1 + r2hi)
    assert np.all(dep[inside] >= lo[inside] * (1 - 1e-6)) and np.all(dep[inside] <= hi[inside] * (1 + 1e-6))
    assert np.all(cov[outside] == 0) and np.all(dep[outside] == 0) and np.all(nrm[outside] == 0)
    assert np.all(np.abs(alb[outside] - np.array(bg, dtype=np.float32)) <= EPS)


def test_a_dense_medium_and_a_grazing_fuzzy_metal(built):
    """The medium row: the isotropic albedo, a zero normal and the distance to the scatter event, which lies past the
    boundary.  And a metal of fuzz 1 seen at grazing angles, where about half the samples are absorbed (the fuzzed
    direction points into the surface): its albedo is still the metal's."""
    iso_colour, metal_albedo, centre, radius, density = (0.3, 0.5, 0.7), (0.8, 0.6, 0.4), np.array([0.0, 2.0, 12.0]), 1.5, 10.0
    w, h, n = 96, 64, 64
    tex = capi.rt_texture()
    tex.type, tex.even, tex.odd, tex.image, tex.perlin = capi.RT_TEX_SOLID, -1, -1, -1, -1
    tex.color = fuzz_scenes.d3(iso_colour)
    metal, iso = capi.rt_material(), capi.rt_material()
    metal.type, metal.texture, metal.albedo, metal.param = capi.RT_MAT_METAL, -1, fuzz_scenes.d3(metal_albedo), 1.0
    iso.type, iso.texture = capi.RT_MAT_ISOTROPIC, 0
    floor = capi.rt_quad()
    floor.Q, floor.u, floor.v = fuzz_scenes.d3((-60, -1, 0.5)), fuzz_scenes.d3((120, 0, 0)), fuzz_scenes.d3((0, 0, 120))
    floor.material, floor.xform = 0, -1
    ball = capi.rt_sphere()
    ball.center0, ball.center_vec, ball.radius, ball.material, ball.xform = fuzz_scenes.d3(centre), fuzz_scenes.d3((0, 0, 0)), radius, 1, -1
    cam = capi.rt_camera()
    cam.lookfrom, cam.lookat, cam.vup = fuzz_scenes.d3((0, 0, 0)), fuzz_scenes.d3((0, 0, 1)), fuzz_scenes.d3((0, 1, 0))
    cam.vfov, cam.defocus_angle, cam.focus_dist = 40.0, 0.0, 10.0
    cam.background = fuzz_scenes.d3((0.5, 0.7, 1.0))
    sc = fuzz_scenes.PyScene([ball], [floor], [], [], [metal, iso], [tex], camera=cam)
    d = sc.desc
    world = (capi.rt_prim_ref * 1)(capi.rt_prim_ref(capi.RT_PRIM_QUAD, 0))
    refs = (capi.rt_prim_ref * 1)(capi.rt_prim_ref(capi.RT_PRIM_SPHERE, 0))
    med = (capi.rt_medium * 1)()
    med[0].boundary_first, med[0].boundary_count = 0, 1
    med[0].density, med[0].multiplicity, med[0].material, med[0].xform = density, 1, 1, -1
    sc._keep += [world, refs, med]
    d.world, d.n_world = world, 1
    d.boundary_refs, d.n_boundary_refs = refs, 1
    d.media, d.n_media = med, 1
    c = capi.Context(0)
    try:
        c.upload(sc)
        c.render(w, h, n, max_depth=8, seed=6, aov=True)
        a = c.download_aov(n)
    finally:
        c.close()
    alb, nrm, dep, cov = (a[k].astype(np.float64) for k in ("albedo", "normal", "depth", "coverage"))
    # pixel-centre directions: the viewport at distance 10, x to the left (u = -x) and rows downwards
    vh = 2.0 * math.tan(math.radians(20.0)) * 10.0
    pw = vh / h
    x = -(-pw * w / 2 + (np.arange(w) + 0.5) * pw)
    y = vh / 2 - (np.arange(h) + 0.5) * pw
    dirs = np.stack(np.broadcast_arrays(x[None, :], y[:, None], np.full((h, w), 10.0)), axis=-1)
    dirs /= np.linalg.norm(dirs, axis=-1, keepdims=True)
    along = dirs @ centre
    impact = np.sqrt(np.maximum(centre @ centre - along ** 2, 0.0))
    medium = impact < 0.5 * radius                     # chords of >= 2.6 units at density 10: no sample gets through
    entry = along - np.sqrt(radius ** 2 - np.minimum(impact, radius) ** 2)   # the boundary, along the pixel-centre ray
    assert medium.sum() > 30
    assert np.all(cov[medium] == 1.0) and np.all(nrm[medium] == 0.0)
    assert np.all(np.abs(alb[medium] - np.array(iso_colour, dtype=np.float32)) <= EPS)
    past = dep[medium] - entry[medium]                 # exponential free flights of mean 1 / density past the boundary
    assert np.all(past > 0.04) and 0.08 < past.mean() < 0.12, (past.min(), past.mean())
    floor_px = (cov == 1.0) & (np.arange(h)[:, None] >= h // 2)
    assert floor_px.sum() > 500
    assert np.all(np.abs(alb[floor_px] - np.array(metal_albedo, dtype=np.float32)) <= EPS)
    assert np.all(np.abs(nrm[floor_px] - np.array([0.0, 1.0, 0.0])) <= EPS)


def _material_of(desc, prim_id):
    r = desc.world[int(prim_id)]
    return desc.materials[(desc.quads if r.type == capi.RT_PRIM_QUAD else desc.spheres)[r.index].material]


def _interior(prim_id, w, h):
    """Pixels whose 3x3 neighbourhood of pixel-centre rays hits one primitive."""
    p = prim_id.reshape(h, w)
    ok = np.zeros((h, w), dtype=bool)
    ok[1:-1, 1:-1] = p[1:-1, 1:-1] >= 0
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            ok[1:-1, 1:-1] &= p[1 + dy:h - 1 + dy, 1 + dx:w - 1 + dx] == p[1:-1, 1:-1]
    return ok, p


def test_cornell_walls_and_light(ctx, scene_of):
    sc, w, h, n = scene_of("cornell"), 128, 128, 16
    d = sc.desc
    ctx.upload(sc)
    centre = ctx.aov(w, h)
    ok, p = _interior(centre["prim_id"], w, h)
    geo = centre["normal"].reshape(h, w, 3)
    ctx.render(w, h, n, seed=4, aov=True)
    a = ctx.download_aov(n)
    walls = lights = 0
    for pid in np.unique(p[ok]):
        m = _material_of(d, pid)
        px = ok & (p == pid)
        assert np.all(a["coverage"][px] == 1.0)
        if m.type == capi.RT_MAT_DIFFUSE_LIGHT:
            assert np.all(a["albedo"][px] == 1.0)
            lights += 1
            continue
        nrm = geo[px]
        if m.type != capi.RT_MAT_LAMBERTIAN or not np.all(np.abs(nrm).max(axis=1) == 1.0):
            continue  # the walls: axis-aligned lambertian quads of one colour
        colour = np.array(list(d.textures[m.texture].color), dtype=np.float32).astype(np.float64)
        assert np.all(np.abs(a["albedo"][px] - colour) <= EPS), pid
        assert np.all(np.abs(a["normal"][px] - nrm) <= EPS), pid
        walls += 1
    assert walls >= 5 and lights == 1, (walls, lights)


def test_final_glass_sphere_is_white(ctx, scene_of):
    sc, w, h, n = scene_of("final"), 200, 200, 8
    d = sc.desc
    ctx.upload(sc)
    ok, p = _interior(ctx.aov(w, h)["prim_id"], w, h)
    glass = np.zeros_like(ok)
    for pid in np.unique(p[ok]):
        if d.world[int(pid)].type == capi.RT_PRIM_SPHERE and _material_of(d, pid).type == capi.RT_MAT_DIELECTRIC:
            glass |= ok & (p == pid)
    assert glass.sum() > 50
    ctx.render(w, h, n, seed=4, aov=True)
    a = ctx.download_aov(n)
    assert np.all(a["albedo"][glass] == 1.0) and np.all(a["coverage"][glass] == 1.0)


# ---- rules -----------------------------------------------------------------------------------------------------------
def test_state_and_argument_errors(built, scene_of):
    c = capi.Context(0)
    try:
        c.upload(scene_of("cornell"))
        c.render(W, H, 2, seed=1)
        assert _code(c.download_aov, 2) == capi.RT_ERR_STATE  # no AOV pass yet
        assert _code(c.render, W, H, 2, seed=1, spp_begin=2, accumulate=True, aov=True) == capi.RT_ERR_STATE
        assert _code(c.render, W, H, 2, seed=1, stats=True, aov=True) == capi.RT_ERR_UNSUPPORTED
        assert _code(c.render, W, H, 2, seed=1, moments=True, aov=True) == capi.RT_ERR_UNSUPPORTED
        p = capi.rt_render_params()
        p.struct_size, p.width, p.height, p.samples_per_pixel, p.max_depth, p.seed = C.sizeof(p), W, H, 2, 8, 1
        p.flags = capi.RT_FLAG_AOV
        cam = scene_of("cornell").desc.camera
        assert c.lib.rt_render_views(c._h, C.byref(p), C.byref(cam), None, 1) == capi.RT_ERR_UNSUPPORTED
        c.render(W, H, 2, seed=1, aov=True)
        assert _code(c.download_aov, 0) == capi.RT_ERR_INVALID
        c.download_aov(2)
        c.render(W, H, 2, seed=1, spp_begin=2, accumulate=True)  # a pass without the flag leaves the frame without AOVs
        assert _code(c.download_aov, 4) == capi.RT_ERR_STATE
        c.render(W, H, 2, seed=1, aov=True)
        c.accum_upload(c.accum_download())  # sums restored without AOV sums
        assert _code(c.download_aov, 2) == capi.RT_ERR_STATE
        assert _code(c.render, W, H, 2, seed=1, spp_begin=2, accumulate=True, aov=True) == capi.RT_ERR_STATE
    finally:
        c.close()


def test_an_untile_hand_out_is_unchanged_by_an_aov_download(built, scene_of):
    """rt_untile_begin copies out of frame_scratch after it returns; rt_download_aov resolves into frame_scratch, so it
    must wait for that copy.  frame_scratch is grown first, so that the download reuses it instead of reallocating."""
    import torch

    c, sc = capi.Context(0), scene_of("final")
    try:
        w, h, spp, count, tile = 960, 540, 4, 2, 16
        c.upload(sc)
        c.render(w, h, spp, seed=7, aov=True)
        want = c.download(spp, linear=True)
        want_aov = _all(c.download_aov(spp)).copy()  # frame_scratch now holds w * h * 32 bytes
        cap = max(capi.load().rt_shard_pixels(w, h, tile, r, count) for r in range(count))
        glin = torch.zeros((count, cap * 3), dtype=torch.float32, device="cuda:0")
        torch.cuda.synchronize()
        for r in range(count):
            c.render(w, h, spp, seed=7, shard_rank=r, shard_count=count, shard_mode=capi.RT_SHARD_TILES, tile_size=tile, compact=True)
            c.resolve_tiles(spp, None, cap, dev_linear=glin[r].data_ptr())
        c.render(w, h, spp, seed=7, aov=True)
        c.untile_begin(glin.data_ptr(), cap * 12, 12, count, w, h, tile)  # the untiled frame in frame_scratch, copy queued
        got_aov = _all(c.download_aov(spp))                                # resolves over the same bytes of frame_scratch
        lin, _ = c.frame_end()
        assert np.array_equal(lin, want)
        assert np.array_equal(got_aov, want_aov)
    finally:
        c.close()


# ---- host mirror: camera::render with --aov (apps/rtow_b200) ------------------------------------------------------------
def test_camera_writes_the_aov_files(built, scene_of, tmp_path):
    from helpers import ROOT
    from test_frame_io import read_pfm
    from raytracingoneweekendapplication_b200.assets import ensure_assets

    sc, spp = scene_of("cornell"), 96
    c = capi.Context(0)
    try:
        c.upload(sc)
        c.render(80, 80, spp, max_depth=sc.depth, seed=1, aov=True)
        a = c.download_aov(spp)
    finally:
        c.close()
    exe = os.path.join(ROOT, "apps", "rtow_b200")
    out = str(tmp_path / "x.pfm")
    r = subprocess.run([exe, "cornell", str(tmp_path / "x.png"), ensure_assets(), "80", "80", str(spp), "--aov", out],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(read_pfm(str(tmp_path / "x_albedo.pfm")), a["albedo"])
    assert np.array_equal(read_pfm(str(tmp_path / "x_normal.pfm")), a["normal"])
    depth = read_pfm(str(tmp_path / "x_depth.pfm"))
    assert all(np.array_equal(depth[..., k], a["depth"]) for k in range(3))
    r = subprocess.run([exe, "cornell", str(tmp_path / "y.png"), ensure_assets(), "80", "80", "8", "--aov", out, "--turntable", "3"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 2 and "AOV" in r.stderr
