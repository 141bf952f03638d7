"""Environment lighting (rt_set_environment): an equirectangular map seen by every ray that leaves the scene.

A map whose texels all equal the background renders the background's frame bit for bit on every render path, so the
environment instances keep their twins' arithmetic.  Rays without a pixel footprint in an empty scene see known values:
a float64 restatement of the lookup of include/rt_b200.h.  A panorama at the map's size gives the map back."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from raytracingoneweekendapplication_b200 import capi

pytestmark = pytest.mark.gpu

W, H = 64, 48


@pytest.fixture
def ectx(built):
    """A context of its own: the environment is context state, and the session context must not keep one."""
    c = capi.Context(0)
    yield c
    c.close()


def _code(fn, *a, **kw):
    with pytest.raises(capi.RtError) as e:
        fn(*a, **kw)
    return e.value.code


def lookup(env, rot, d):
    """The lookup of include/rt_b200.h in float64: env (h, w, 3), rot map -> world, d (n, 3) world directions."""
    h, w, _ = env.shape
    m = np.asarray(d, np.float64).reshape(-1, 3) @ np.asarray(rot, np.float64)  # R^T d, row vectors
    phi = np.arctan2(m[:, 0], -m[:, 2])
    theta = np.arctan2(m[:, 1], np.hypot(m[:, 0], m[:, 2]))
    tx = (phi / (2 * np.pi) + 0.5) * w - 0.5
    ty = (0.5 - theta / np.pi) * h - 0.5
    x0, y0 = np.floor(tx), np.floor(ty)
    fx, fy = (tx - x0)[:, None], (ty - y0)[:, None]
    x0, y0 = x0.astype(np.int64), y0.astype(np.int64)
    xa, xb = x0 % w, (x0 + 1) % w
    ya, yb = np.clip(y0, 0, h - 1), np.clip(y0 + 1, 0, h - 1)
    e = env.astype(np.float64)
    top = e[ya, xa] + fx * (e[ya, xb] - e[ya, xa])
    bot = e[yb, xa] + fx * (e[yb, xb] - e[yb, xa])
    return top + fy * (bot - top)


def rot_y(deg):
    """A turn of deg degrees about +y, computed as camera::environment_rotation does."""
    a = deg * 3.1415926535897932385 / 180.0
    c, s = math.cos(a), math.sin(a)
    return np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]])


def random_rotation(seed):
    q, r = np.linalg.qr(np.random.default_rng(seed).standard_normal((3, 3)))
    q = q * np.sign(np.diag(r))
    return q if np.linalg.det(q) > 0 else -q


def sky(w=256, h=128, sun=40.0):
    """A smooth sky gradient with a small sun of radiance about `sun`: non-uniform, finite, >= 0."""
    j, i = np.mgrid[0:h, 0:w]
    theta = np.pi * (0.5 - (j + 0.5) / h)
    phi = 2 * np.pi * ((i + 0.5) / w - 0.5)
    m = np.empty((h, w, 3), np.float32)
    up = np.clip(np.sin(theta), 0, 1)
    m[..., 0] = 0.3 + 0.5 * up
    m[..., 1] = 0.4 + 0.4 * up + 0.1 * np.cos(phi)
    m[..., 2] = 0.9 - 0.2 * up
    disc = np.hypot(theta - 0.6, phi - 0.8) < 0.08
    m[disc] = (sun, 0.9 * sun, 0.75 * sun)
    return m


def panorama_records(w, h):
    """Zero-footprint records of camera::panorama_rays for lookfrom 0, lookat (0, 0, -1), vup +y (the map frame)."""
    j, i = np.mgrid[0:h, 0:w]
    th = np.pi * (0.5 - (j + 0.5) / h)
    ph = 2 * np.pi * ((i + 0.5) / w - 0.5)
    rec = np.zeros((h, w, 12), np.float32)
    rec[..., 3:6] = np.stack([np.cos(th) * np.sin(ph), np.sin(th), -np.cos(th) * np.cos(ph)], -1)
    return rec


def empty_scene(background=(0.2, 0.3, 0.4)):
    from fuzz_scenes import PyScene, d3

    tex = capi.rt_texture()
    tex.type, tex.even, tex.odd, tex.image, tex.perlin = capi.RT_TEX_SOLID, -1, -1, -1, -1
    tex.color = d3((0.5, 0.5, 0.5))
    mat = capi.rt_material()
    mat.type, mat.texture = capi.RT_MAT_LAMBERTIAN, 0
    sc = PyScene([], [], [], [], [mat], [tex])
    sc.desc.camera.background = d3(background)
    assert sc.desc.n_world == 0
    return sc


def uniform_map(sc):
    return np.broadcast_to(np.array(list(sc.desc.camera.background), dtype=np.float32), (8, 16, 3)).copy()


# ---- a uniform map is the background, bit for bit --------------------------------------------------------------------------
def _passes(c, sc):
    """Every render path once: what it leaves in the context (sums, moments, AOV sums, views)."""
    from test_gpu_camera_rays import _pinhole_rays
    from test_gpu_views import _orbit

    d, n, out = sc.depth, 4, {}
    c.render(W, H, n, max_depth=d, seed=3)
    out["plain"] = c.accum_download()
    c.render(W, H, n, max_depth=d, seed=3, nee=True)
    out["nee"] = c.accum_download()
    c.render(W, H, n, max_depth=d, seed=3, nee=True, shadowed_point_lights=True)
    out["nee_shadowed"] = c.accum_download()
    c.render(W, H, n, max_depth=d, seed=3, moments=True)
    out["moments"] = (c.accum_download(), c.moments_download())
    c.render(W, H, n, max_depth=d, seed=3, aov=True)
    out["aov"] = (c.accum_download(), c.download_aov(n)["albedo"].base.copy())
    c.set_camera_rays(_pinhole_rays(sc.desc.camera, W, H))
    c.render(W, H, n, max_depth=d, seed=3, camera_rays=True)
    out["camera_rays"] = c.accum_download()
    c.render(W, H, n, max_depth=d, seed=3, shard_rank=1, shard_count=3, shard_mode=capi.RT_SHARD_TILES, tile_size=16, compact=True)
    out["compact_shard"] = c.accum_download()
    c.render(W, H, 2, max_depth=d, seed=3)
    for begin in (2, 4):
        c.render(W, H, 2, max_depth=d, seed=3, spp_begin=begin, accumulate=True, blocking=False, overlap=True)
    c.sync()
    out["overlap"] = c.accum_download()
    cams = _orbit(sc.desc.camera, 3)
    c.render_views(cams, W, H, n, max_depth=d, seed=3)
    out["views"] = c.download_views(n)
    return out


@pytest.mark.parametrize("name", ["book1", "mesh", "cornell_smoke", "final", "kitchen_sink"])
def test_uniform_map_is_the_background(ectx, scene_of, name):
    sc = scene_of(name)
    ectx.upload(sc)
    plain = _passes(ectx, sc)
    ectx.set_environment(uniform_map(sc))
    env = _passes(ectx, sc)
    for k in plain:
        a, b = (plain[k], env[k]) if isinstance(plain[k], tuple) else ((plain[k],), (env[k],))
        for x, y in zip(a, b):
            assert np.array_equal(x, y), k
    assert np.any(plain["plain"]) and np.any(plain["views"])


def test_two_devices_render_the_environment_of_one(built, scene_of, monkeypatch):
    """The map is copied to every device: a multi-device frame equals the single-device one (the same GPU listed twice
    where only one is visible)."""
    import torch

    sc, env, n = scene_of("cornell_smoke"), sky(), 6
    with capi.Context(0) as one:
        one.upload(sc)
        one.set_environment(env, rot_y(40))
        one.render(W, H, n, seed=5, aov=True)
        want, want_aov = one.accum_download(), one.download_aov(n)["albedo"].base.copy()
    monkeypatch.setenv("RT_B200_ALLOW_DUPLICATE_DEVICES", "1")
    md = capi.Context([0, 1] if torch.cuda.device_count() >= 2 else [0, 0])
    try:
        md.upload(sc)
        md.set_environment(env, rot_y(40))
        md.render(W, H, n, seed=5, aov=True, shard_mode=capi.RT_SHARD_TILES, tile_size=16)
        assert np.array_equal(md.accum_download(), want)
        assert np.array_equal(md.download_aov(n)["albedo"].base, want_aov)
        md.render(W, H, n, seed=5, shard_mode=capi.RT_SHARD_SAMPLES)
        assert np.array_equal(md.accum_download(), want)
    finally:
        md.close()


# ---- known values --------------------------------------------------------------------------------------------------------
def test_known_values(ectx):
    rng = np.random.default_rng(17)
    mw, mh = 64, 32
    env = rng.uniform(0.0, 4.0, (mh, mw, 3)).astype(np.float32)
    env[0] = env[0, 0]    # the pole rows are uniform, as in any map continuous at the poles: a pole ray's longitude
    env[-1] = env[-1, 0]  # is whatever the rounding of R^T d makes it
    rot = random_rotation(5)
    dm = [rng.standard_normal((150, 3)), [[0, 1, 0], [0, -1, 0]]]                    # random, both poles
    ys = np.linspace(-0.9, 0.9, 7)
    dm.append(np.stack([np.zeros_like(ys), ys, np.sqrt(1 - ys ** 2)], -1))           # the +-pi seam (straight behind)
    j, i = rng.integers(0, mh, 33), rng.integers(0, mw, 33)
    th, ph = np.pi * (0.5 - (j + 0.5) / mh), 2 * np.pi * ((i + 0.5) / mw - 0.5)
    dm.append(np.stack([np.cos(th) * np.sin(ph), np.sin(th), -np.cos(th) * np.cos(ph)], -1))  # texel centres
    d = (np.concatenate(dm) @ rot.T).astype(np.float32)  # world = R map
    w = 16
    h = (len(d) + w - 1) // w
    rec = np.zeros((h, w, 12), np.float32)
    rec.reshape(-1, 12)[: len(d), 3:6] = d
    rec.reshape(-1, 12)[len(d):, 3:6] = d[0]
    sc = empty_scene()
    ectx.upload(sc)
    ectx.set_environment(env, rot)
    ectx.set_camera_rays(rec)
    ectx.render(w, h, 4, max_depth=8, seed=2, camera_rays=True, aov=True)
    want = lookup(env, rot, rec.reshape(-1, 12)[:, 3:6])
    got = ectx.download(4).reshape(-1, 3)
    assert np.abs(got - want).max() <= 1e-3, np.abs(got - want).max()
    a = ectx.download_aov(4)
    assert np.abs(a["albedo"].reshape(-1, 3) - np.clip(want, 0, 1)).max() <= 1e-3
    assert not np.any(a["coverage"]) and not np.any(a["normal"]) and not np.any(a["depth"])
    assert want[:, 0].max() > 1.0  # the clamp was exercised


def test_panorama_round_trip(ectx):
    mw, mh = 64, 32
    env = np.random.default_rng(3).uniform(0.0, 4.0, (mh, mw, 3)).astype(np.float32)
    ectx.upload(empty_scene())
    ectx.set_camera_rays(panorama_records(mw, mh))
    ectx.set_environment(env)
    ectx.render(mw, mh, 2, max_depth=4, seed=1, camera_rays=True)
    assert np.abs(ectx.download(2) - env).max() <= 1e-3
    ectx.set_environment(env, rot_y(90))
    ectx.render(mw, mh, 2, max_depth=4, seed=1, camera_rays=True)
    assert np.abs(ectx.download(2) - np.roll(env, -mw // 4, axis=1)).max() <= 1e-3


# ---- the estimate: NEE leaves the environment to the BSDF samples -----------------------------------------------------------
def test_nee_and_plain_agree_in_expectation(ectx, scene_of):
    """Cornell's open side lets paths out into the map.  Per-pixel means within 5 sigma of the difference, sigma from the
    moments of both renders, as in test_gpu_camera_rays."""
    sc, w, h, n = scene_of("cornell"), 48, 32, 2048
    ectx.upload(sc)
    ectx.set_environment(sky(sun=3.0), rot_y(180))  # a dim sun: the rare paths that find it stay within the moments
    ectx.render(w, h, n, max_depth=50, seed=11, moments=True)
    plain, var = ectx.download(n).astype(np.float64), ectx.download_variance(n).astype(np.float64)
    ectx.render(w, h, n, max_depth=50, seed=12, moments=True, nee=True)
    nee = ectx.download(n).astype(np.float64)
    var += ectx.download_variance(n).astype(np.float64)
    ectx.set_environment(None)
    ectx.render(w, h, 64, max_depth=50, seed=11)
    assert abs(plain.mean() - ectx.download(64).mean()) > 0.01  # the map is seen
    sigma = np.sqrt(var / n)
    ok = (np.abs(nee - plain) <= 5 * sigma).all(axis=2)
    assert ok.mean() >= 0.995, (ok.mean(), np.argwhere(~ok)[:5])
    frame_sigma = math.sqrt(np.sum(np.sum(sigma, axis=2) ** 2)) / (3 * w * h)
    assert abs(nee.mean() - plain.mean()) <= 3 * frame_sigma, (nee.mean(), plain.mean(), frame_sigma)


# ---- state ---------------------------------------------------------------------------------------------------------------
def test_state_rules(ectx, scene_of):
    sc, n = scene_of("cornell_smoke"), 4
    env, other = sky(), sky()[:, ::-1].copy()

    def frame(**kw):
        ectx.render(W, H, n, seed=7, **kw)
        return ectx.accum_download()

    ectx.upload(sc)
    background = frame()
    ectx.set_environment(env, rot_y(25))
    lit = frame()
    assert not np.array_equal(lit, background)
    ectx.upload(sc)
    assert np.array_equal(frame(), lit)  # an upload keeps the map
    ectx.refit(sc)
    assert np.array_equal(frame(), lit)  # and so does a refit

    # refused maps change nothing
    good = rot_y(25)
    bad_maps = [env[:0], env * np.float32(-1), np.where(np.arange(W)[None, :, None] == 3, np.float32(np.nan), env[:, :W]).astype(np.float32)]
    for m in bad_maps:
        assert _code(ectx.set_environment, m, good) == capi.RT_ERR_INVALID
    for r in (good * 1.01, good @ np.diag([1.0, 1.0, -1.0]), np.full((3, 3), np.nan)):
        assert _code(ectx.set_environment, env, r) == capi.RT_ERR_INVALID
    e = capi.rt_environment()
    e.rgb, e.width, e.height = None, 4, 4
    e.rotation = (C.c_double * 9)(1, 0, 0, 0, 1, 0, 0, 0, 1)
    assert ectx.lib.rt_set_environment(ectx._h, C.byref(e)) == capi.RT_ERR_INVALID
    assert np.array_equal(frame(), lit)
    with pytest.raises(capi.RtError) as err:
        ectx.set_environment(np.where(np.arange(16)[None, :, None] == 5, np.float32(-1), env[:8, :16]).astype(np.float32))
    assert "texel 5 " in str(err.value)

    assert _code(ectx.render, W, H, n, seed=7, stats=True) == capi.RT_ERR_UNSUPPORTED

    # a map set after passes in flight applies to the passes after it: the frame of the blocking sequence
    ectx.set_environment(env, rot_y(25))
    ectx.render(W, H, n, seed=7)
    ectx.set_environment(other)
    ectx.render(W, H, n, seed=7, spp_begin=n, accumulate=True)
    want = ectx.accum_download()
    ectx.set_environment(env, rot_y(25))
    ectx.render(W, H, n, seed=7, blocking=False)
    ectx.set_environment(other)
    ectx.render(W, H, n, seed=7, spp_begin=n, accumulate=True)
    assert np.array_equal(ectx.accum_download(), want)
    ectx.set_environment(env, rot_y(25))
    ectx.render(W, H, 2, seed=7)
    ectx.render(W, H, 2, seed=7, spp_begin=2, accumulate=True, blocking=False, overlap=True)
    ectx.set_environment(other)
    ectx.render(W, H, n, seed=7, spp_begin=n, accumulate=True)
    assert np.array_equal(ectx.accum_download(), want)

    ectx.set_environment(None)
    assert np.array_equal(frame(), background)
    ectx.render(W, H, 2, seed=7, stats=True)


@pytest.mark.parametrize("name", ["book1", "cornell_smoke"])
def test_each_view_is_its_own_render(ectx, scene_of, name):
    from test_gpu_views import _orbit, _with_camera

    sc, n = scene_of(name), 6
    cams = _orbit(sc.desc.camera, 3)
    ectx.upload(sc)
    ectx.set_environment(sky(), rot_y(70))
    ectx.render_views(cams, W, H, n, max_depth=sc.depth, seed=4, nee=True)
    views = ectx.download_views(n)
    for v, cam in enumerate(cams):
        ectx.upload(_with_camera(sc, cam))
        ectx.render(W, H, n, max_depth=sc.depth, seed=4, nee=True)
        assert np.array_equal(ectx.download(n), views[v]), v


# ---- host mirror: rtow_b200 --env --------------------------------------------------------------------------------------
def test_mirror_environment(built, scene_of, tmp_path):
    from helpers import ROOT
    from test_environment_io import _write_pfm
    from test_gpu_views import _read_png
    from raytracingoneweekendapplication_b200.assets import ensure_assets

    s = capi.load_scenes()
    sc, w, h, spp = scene_of("book1"), 96, 48, 24
    env = sky()
    pfm = tmp_path / "sky.pfm"
    _write_pfm(pfm, env, little=True)
    buf = (capi.rt_camera_ray * (w * h))()
    assert s.rtsc_panorama_rays(b"book1", 1, ensure_assets().encode(), w, h, buf) == 0
    with capi.Context(0) as c:
        c.upload(sc)
        c.set_camera_rays(np.frombuffer(buf, dtype=np.float32).reshape(h, w, 12))
        c.set_environment(env, rot_y(30))
        c.render(w, h, spp, max_depth=sc.depth, seed=1, camera_rays=True)
        want = c.download(spp, linear=False, rgb8=True)
    exe = os.path.join(ROOT, "apps", "rtow_b200")
    out = tmp_path / "pano.png"
    r = subprocess.run([exe, "book1", str(out), ensure_assets(), str(w), str(h), str(spp), "--panorama", "--env", str(pfm),
                        "--env-rotate", "30"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert np.array_equal(_read_png(str(out)), want)

    # a checkpoint resumes under its own map only
    other = tmp_path / "other.pfm"
    _write_pfm(other, env[::-1].copy(), little=False)
    ck = tmp_path / "ck.bin"
    base = [exe, "book1", str(tmp_path / "c.png"), ensure_assets(), "48", "32", "8", "--checkpoint", str(ck)]
    r = subprocess.run(base + ["--stop-after", "4", "--env", str(pfm)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and ck.exists(), r.stderr
    r = subprocess.run(base + ["--stop-after", "6", "--env", str(other)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "Ignoring" in r.stderr and "Resuming" not in r.stderr, r.stderr
    r = subprocess.run(base + ["--env", str(other)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "Resuming" in r.stderr, r.stderr
