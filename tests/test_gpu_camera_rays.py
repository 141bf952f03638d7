"""Caller-defined cameras (rt_set_camera_rays, RT_FLAG_CAMERA_RAYS): the primary ray of every sample comes from a record
per pixel instead of the uploaded camera.

Only ray generation changes, so a rays frame is summed exactly like a camera frame: every way of scheduling its samples
gives the same integers, AOVs leave it unchanged, and rays without a pixel footprint give known values.  The pinhole
rays of the uploaded camera render the camera's image in expectation, though not bit for bit."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from raytracingoneweekendapplication_b200 import capi

pytestmark = pytest.mark.gpu

W, H = 64, 48


def _code(fn, *a, **kw):
    with pytest.raises(capi.RtError) as e:
        fn(*a, **kw)
    return e.value.code


def _pinhole_rays(cam, w, h):
    """The uploaded camera's pixel-centre rays as (h, w, 12) records: origin = lookfrom, direction = dir00 + i du + j dv
    in double (dir00 = pixel00 - lookfrom, Camera.txt:136-168), dx = du, dy = dv."""
    lookfrom, lookat, vup = (np.array(list(v), dtype=np.float64) for v in (cam.lookfrom, cam.lookat, cam.vup))
    vh = 2 * math.tan(math.radians(cam.vfov) / 2) * cam.focus_dist
    vw = vh * (w / h)
    ww = (lookfrom - lookat) / np.linalg.norm(lookfrom - lookat)
    u = np.cross(vup, ww)
    u /= np.linalg.norm(u)
    v = np.cross(ww, u)
    du, dv = vw * u / w, -vh * v / h
    dir00 = -cam.focus_dist * ww - 0.5 * vw * u + 0.5 * vh * v + 0.5 * (du + dv)
    jj, ii = np.mgrid[0:h, 0:w]
    rec = np.zeros((h, w, 12), dtype=np.float64)
    rec[..., 0:3] = lookfrom
    rec[..., 3:6] = dir00 + ii[..., None] * du + jj[..., None] * dv
    rec[..., 6:9] = du
    rec[..., 9:12] = dv
    return rec.astype(np.float32)


def _probe(ctx, rec):
    """rt_probe_hit on the records' directions (their rays when dx = dy = 0), as the render kernels would trace them."""
    h, w = rec.shape[:2]
    rays = np.zeros((h * w, 9), dtype=np.float32)
    rays[:, 0:6] = rec.reshape(-1, 12)[:, 0:6]
    rays[:, 7], rays[:, 8] = 0.001, np.inf
    return ctx.probe_hit(rays)


def _material_of(desc, prim_id):
    r = desc.world[int(prim_id)]
    return desc.materials[(desc.quads if r.type == capi.RT_PRIM_QUAD else desc.spheres)[r.index].material]


# ---- known values ------------------------------------------------------------------------------------------------------
def test_exact_rays_give_the_first_vertex_emission(ctx, scene_of):
    """Depth 1 and no pixel footprint: every sample of a pixel is the same ray, so the mean is exactly what its first
    vertex emits (the quad light), 0 on the walls and the background on a miss."""
    sc, n = scene_of("cornell"), 16
    d = sc.desc
    ctx.upload(sc)
    rec = _pinhole_rays(d.camera, W, H)
    rec[..., 6:12] = 0.0
    # a few rays into the open side of the box and past it: misses
    rec[0, :4, 3:6] = rec[0, :4, 3:6] * np.float32(-1.0)
    ctx.set_camera_rays(rec)
    ctx.render(W, H, n, max_depth=1, seed=3, camera_rays=True)
    got = ctx.download(n).reshape(-1, 3)
    pid = _probe(ctx, rec)["prim_id"]
    want = np.zeros_like(got)
    lights = 0
    for k in range(W * H):
        if pid[k] < 0:
            want[k] = np.array(list(d.camera.background), dtype=np.float32)
            continue
        m = _material_of(d, pid[k])
        if m.type == capi.RT_MAT_DIFFUSE_LIGHT:
            want[k] = np.array(list(d.textures[m.texture].color), dtype=np.float32)
            lights += 1
    assert lights >= 8 and (pid < 0).sum() >= 4
    assert np.array_equal(got, want)


def test_exact_rays_give_the_probed_aov(ctx, scene_of):
    sc, n = scene_of("cornell"), 8
    ctx.upload(sc)
    rec = _pinhole_rays(sc.desc.camera, W, H)
    rec[..., 6:12] = 0.0
    rec[0, :4, 3:6] = rec[0, :4, 3:6] * np.float32(-1.0)
    ctx.set_camera_rays(rec)
    ctx.render(W, H, n, max_depth=4, seed=3, aov=True, camera_rays=True)
    a = ctx.download_aov(n)
    pr = _probe(ctx, rec)
    hit = pr["prim_id"] >= 0
    cov, nrm, dep = a["coverage"].reshape(-1), a["normal"].reshape(-1, 3), a["depth"].reshape(-1)
    assert np.all(cov[hit] == 1.0) and np.all(cov[~hit] == 0.0) and hit.sum() > W * H // 2
    d = rec.reshape(-1, 12)[:, 3:6]
    pn = pr["normal"]
    facing = np.where((np.sum(pn.astype(np.float64) * d, axis=1) < 0)[:, None], pn, -pn)
    q = (np.rint(np.clip(facing, -1, 1).astype(np.float64) * 2.0 ** 28) / 2.0 ** 28).astype(np.float32)
    assert np.array_equal(nrm[hit], q[hit])
    assert np.all(nrm[~hit] == 0)
    dd = d.astype(np.float64)
    want = (pr["t"].astype(np.float64) * np.sqrt(np.sum(dd * dd, axis=1))).astype(np.float32)
    assert np.all(np.abs(dep[hit] - want[hit]) <= np.spacing(want[hit]))


# ---- the pinhole rays render the camera's image in expectation -----------------------------------------------------------
@pytest.mark.parametrize("name", ["cornell", "cornell_smoke", "final"])
def test_pinhole_rays_have_the_cameras_expectation(ctx, scene_of, name):
    """Per-pixel means within 5 sigma of the difference, sigma from the moments of two camera renders: one with another
    seed, and one with the rays pass's seed, whose moments describe nearly the same samples as that pass.  (The variance
    of one render alone misses the rare bright paths of a pixel it happened not to sample.)"""
    sc, w, h, n = scene_of(name), 48, 32, 2048
    assert sc.desc.camera.defocus_angle == 0
    ctx.upload(sc)
    ctx.render(w, h, n, max_depth=50, seed=11, moments=True)
    cam = ctx.download(n).astype(np.float64)
    var = ctx.download_variance(n).astype(np.float64)
    ctx.render(w, h, n, max_depth=50, seed=12, moments=True)
    var += ctx.download_variance(n).astype(np.float64)
    ctx.set_camera_rays(_pinhole_rays(sc.desc.camera, w, h))
    ctx.render(w, h, n, max_depth=50, seed=12, camera_rays=True)
    rays = ctx.download(n).astype(np.float64)
    sigma = np.sqrt(var / n)  # of the difference of the two means
    ok = (np.abs(rays - cam) <= 5 * sigma).all(axis=2)
    assert ok.mean() >= 0.995, (ok.mean(), np.argwhere(~ok)[:5])
    # the frame means: the pixels are independent, a pixel's channels bounded by the sum of their deviations
    frame_sigma = math.sqrt(np.sum(np.sum(sigma, axis=2) ** 2)) / (3 * w * h)
    assert abs(rays.mean() - cam.mean()) <= 3 * frame_sigma, (rays.mean(), cam.mean(), frame_sigma)


# ---- bit-identical however it is scheduled ---------------------------------------------------------------------------------
def _own_mask(w, h, tile, rank, count):
    y, x = np.mgrid[0:h, 0:w]
    return ((y // tile) * ((w + tile - 1) // tile) + x // tile) % count == rank


def test_rays_frames_do_not_depend_on_scheduling(ctx, scene_of, monkeypatch):
    sc, n, w, h = scene_of("cornell_smoke"), 12, 96, 80
    rec = _pinhole_rays(sc.desc.camera, w, h)
    rec[..., 3:6] += 0.05 * np.sin(np.arange(w * h * 3, dtype=np.float32)).reshape(h, w, 3)  # not a pinhole
    ctx.upload(sc)
    ctx.set_camera_rays(rec)
    ctx.render(w, h, n, seed=5, aov=True, camera_rays=True)
    ref_aov = ctx.download_aov(n)["albedo"].base.copy()
    ref = ctx.accum_download()

    def same(aov=True):
        assert np.array_equal(ctx.accum_download(), ref)
        if aov:
            assert np.array_equal(ctx.download_aov(n)["albedo"].base, ref_aov)

    for split in ([5, 4, 3], [1, 11]):
        begin = 0
        for k, s in enumerate(split):
            ctx.render(w, h, s, seed=5, spp_begin=begin, aov=True, accumulate=k > 0, camera_rays=True)
            begin += s
        same()
    ctx.render(w, h, 6, seed=5, aov=True, blocking=False, camera_rays=True)
    ctx.render(w, h, 6, seed=5, spp_begin=6, aov=True, accumulate=True, blocking=False, camera_rays=True)
    same()
    ctx.render(w, h, 4, seed=5, aov=True, camera_rays=True)
    for begin in (4, 8):
        ctx.render(w, h, 4, seed=5, spp_begin=begin, aov=True, accumulate=True, blocking=False, overlap=True, camera_rays=True)
    ctx.sync()
    same()
    for tile in (8, 32):
        ctx.render(w, h, n, seed=5, aov=True, tile_size=tile, camera_rays=True)
        same()

    # shards, summed: tiles, samples, compact tiles
    for mode, compact in ((capi.RT_SHARD_TILES, False), (capi.RT_SHARD_SAMPLES, False), (capi.RT_SHARD_TILES, True)):
        total = np.zeros_like(ref)
        for r in range(3):
            ctx.render(w, h, n, seed=5, shard_rank=r, shard_count=3, shard_mode=mode, tile_size=16, compact=compact, camera_rays=True)
            total += ctx.accum_download()
        assert np.array_equal(total, ref), (mode, compact)
    for r in range(2):  # the AOVs of compact tile shards: the shard's own tiles, zero elsewhere
        ctx.render(w, h, n, seed=5, aov=True, shard_rank=r, shard_count=2, shard_mode=capi.RT_SHARD_TILES, tile_size=16,
                   compact=True, camera_rays=True)
        got = ctx.download_aov(n)["albedo"].base
        own = _own_mask(w, h, 16, r, 2)
        assert np.array_equal(got[own], ref_aov[own]) and not np.any(got[~own])

    # NEE: one pass against a split
    ctx.render(w, h, n, seed=5, nee=True, camera_rays=True)
    nee = ctx.accum_download()
    ctx.render(w, h, 7, seed=5, nee=True, camera_rays=True)
    ctx.render(w, h, 5, seed=5, spp_begin=7, nee=True, accumulate=True, camera_rays=True)
    assert np.array_equal(ctx.accum_download(), nee) and not np.array_equal(nee, ref)

    # a render stopped, saved and resumed in a new context
    ctx.render(w, h, 5, seed=5, camera_rays=True)
    saved = ctx.accum_download()
    with capi.Context(0) as c2:
        c2.upload(sc)
        c2.set_camera_rays(rec)
        c2.accum_upload(saved)
        c2.render(w, h, 7, seed=5, spp_begin=5, accumulate=True, camera_rays=True)
        assert np.array_equal(c2.accum_download(), ref)

    # two devices in one context (the same GPU twice where only one is visible)
    monkeypatch.setenv("RT_B200_ALLOW_DUPLICATE_DEVICES", "1")
    import torch
    md = capi.Context([0, 1] if torch.cuda.device_count() >= 2 else [0, 0])
    try:
        md.upload(sc)
        md.set_camera_rays(rec)
        md.render(w, h, 5, seed=5, aov=True, shard_mode=capi.RT_SHARD_TILES, tile_size=16, camera_rays=True)
        md.render(w, h, 7, seed=5, spp_begin=5, aov=True, accumulate=True, shard_mode=capi.RT_SHARD_TILES, tile_size=16,
                  camera_rays=True)
        assert np.array_equal(md.accum_download(), ref)
        assert np.array_equal(md.download_aov(n)["albedo"].base, ref_aov)
        md.render(w, h, n, seed=5, shard_mode=capi.RT_SHARD_SAMPLES, camera_rays=True)
        assert np.array_equal(md.accum_download(), ref)
    finally:
        md.close()


@pytest.mark.parametrize("name", ["book1", "cornell", "cornell_smoke", "mesh", "final"])
@pytest.mark.parametrize("nee", [False, True])
def test_aov_leaves_the_rays_image_unchanged(ctx, scene_of, name, nee):
    sc = scene_of(name)
    ctx.upload(sc)
    ctx.set_camera_rays(_pinhole_rays(sc.desc.camera, W, H))
    ctx.render(W, H, 6, seed=3, nee=nee, camera_rays=True)
    plain = ctx.accum_download()
    ctx.render(W, H, 6, seed=3, nee=nee, aov=True, camera_rays=True)
    assert np.array_equal(ctx.accum_download(), plain)
    assert np.any(ctx.download_aov(6)["coverage"] > 0)


# ---- rules ---------------------------------------------------------------------------------------------------------------
def test_errors_and_frame_sources(built, scene_of):
    lib = capi.load()
    assert lib.rt_struct_size(16) == 48 == C.sizeof(capi.rt_camera_ray)
    sc = scene_of("cornell")
    rec = _pinhole_rays(sc.desc.camera, W, H)
    c = capi.Context(0)
    try:
        c.upload(sc)
        assert _code(c.render, W, H, 2, seed=1, camera_rays=True) == capi.RT_ERR_STATE  # no rays
        c.set_camera_rays(rec)
        assert _code(c.render, W + 8, H, 2, seed=1, camera_rays=True) == capi.RT_ERR_INVALID
        assert _code(c.render, W, H, 2, seed=1, stats=True, camera_rays=True) == capi.RT_ERR_UNSUPPORTED
        assert _code(c.render, W, H, 2, seed=1, moments=True, camera_rays=True) == capi.RT_ERR_UNSUPPORTED
        p = capi.rt_render_params()
        p.struct_size, p.width, p.height, p.samples_per_pixel, p.max_depth, p.seed = C.sizeof(p), W, H, 2, 8, 1
        p.flags = capi.RT_FLAG_CAMERA_RAYS
        cam = sc.desc.camera
        assert c.lib.rt_render_views(c._h, C.byref(p), C.byref(cam), None, 1) == capi.RT_ERR_UNSUPPORTED

        c.render(W, H, 2, seed=1, camera_rays=True)
        good = c.accum_download()
        for k, bad in ((5, np.nan), (W + 3, np.inf)):  # non-finite values: refused, nothing changes
            b = rec.copy()
            b.reshape(-1, 12)[k, 7] = bad
            with pytest.raises(capi.RtError) as e:
                c.set_camera_rays(b)
            assert e.value.code == capi.RT_ERR_INVALID and f"record {k} " in str(e.value)
        b = rec.copy()
        b[1, 2, 3:6] = 0.0
        with pytest.raises(capi.RtError) as e:
            c.set_camera_rays(b)
        assert e.value.code == capi.RT_ERR_INVALID and f"record {W + 2} " in str(e.value) and "zero direction" in str(e.value)
        assert _code(c.set_camera_rays, np.zeros((0, 4, 12), np.float32)) == capi.RT_ERR_INVALID
        c.render(W, H, 2, seed=1, spp_begin=2, accumulate=True, camera_rays=True)  # the previous rays still render
        c.render(W, H, 2, seed=1, camera_rays=True)
        assert np.array_equal(c.accum_download(), good)

        # one source per frame
        assert _code(c.render, W, H, 2, seed=1, spp_begin=2, accumulate=True) == capi.RT_ERR_STATE
        c.render(W, H, 2, seed=1)
        assert _code(c.render, W, H, 2, seed=1, spp_begin=2, accumulate=True, camera_rays=True) == capi.RT_ERR_STATE
        c.render(W, H, 2, seed=1, spp_begin=2, accumulate=True)  # camera passes are as before
        c.render(W, H, 2, seed=1, camera_rays=True)
        c.set_camera_rays(rec)  # the same records again: a new source
        assert _code(c.render, W, H, 2, seed=1, spp_begin=2, accumulate=True, camera_rays=True) == capi.RT_ERR_STATE
        c.accum_upload(good)  # a restored frame takes either source
        c.render(W, H, 2, seed=1, spp_begin=2, accumulate=True, camera_rays=True)
        c.set_camera_rays(None)
        assert _code(c.render, W, H, 2, seed=1, camera_rays=True) == capi.RT_ERR_STATE
    finally:
        c.close()


# ---- host mirror: camera::render with --panorama (apps/rtow_b200) -----------------------------------------------------------
def test_mirror_panorama(built, scene_of, tmp_path):
    from helpers import ROOT
    from test_gpu_views import _read_png
    from raytracingoneweekendapplication_b200.assets import ensure_assets

    s = capi.load_scenes()
    sc, w, h, spp = scene_of("cornell_smoke"), 96, 48, 80
    buf = (capi.rt_camera_ray * (w * h))()
    assert s.rtsc_panorama_rays(b"cornell_smoke", 1, ensure_assets().encode(), w, h, buf) == 0
    rec = np.frombuffer(buf, dtype=np.float32).reshape(h, w, 12)
    c = capi.Context(0)
    try:
        c.upload(sc)
        c.set_camera_rays(rec)
        c.render(w, h, spp, max_depth=sc.depth, seed=1, camera_rays=True)
        want = c.download(spp, linear=False, rgb8=True)
    finally:
        c.close()
    exe = os.path.join(ROOT, "apps", "rtow_b200")
    out = tmp_path / "pano.png"
    r = subprocess.run([exe, "cornell_smoke", str(out), ensure_assets(), str(w), str(h), str(spp), "--panorama"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(_read_png(str(out)), want)
    r = subprocess.run([exe, "cornell_smoke", str(tmp_path / "t.png"), ensure_assets(), str(w), str(h), "4", "--panorama",
                        "--turntable", "3"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 2 and "panorama" in r.stderr
