"""Multi-view batches (rt_render_views / rt_download_views).

A view of a batch must equal, bit for bit, an ordinary render of the scene uploaded with that view's camera: the image
is a pure function of (scene, camera, frame, sample range, depth, seed) and the sums are integers.  So every check here
is np.array_equal against that oracle, never a tolerance."""
import ctypes as C
import math
import os
import struct
import zlib

import numpy as np
import pytest

from raytracingoneweekendapplication_b200 import capi

pytestmark = pytest.mark.gpu

W, H = 48, 32
SPP, DEPTH = 8, 50


def _orbit(cam, n, defocus_view=None):
    """n rt_cameras: `cam` with lookfrom turned about the vertical axis through lookat, a slightly different vfov each."""
    out = []
    for k in range(n):
        c = capi.rt_camera.from_buffer_copy(cam)
        a = 0.35 * k
        rx, rz = c.lookfrom[0] - c.lookat[0], c.lookfrom[2] - c.lookat[2]
        c.lookfrom[0] = c.lookat[0] + rx * math.cos(a) - rz * math.sin(a)
        c.lookfrom[2] = c.lookat[2] + rx * math.sin(a) + rz * math.cos(a)
        c.lookfrom[1] += 0.1 * k
        c.vfov = cam.vfov * (1.0 + 0.03 * k)
        if k == defocus_view:
            c.defocus_angle, c.focus_dist = 2.0, math.dist(list(c.lookfrom), list(c.lookat))
        out.append(c)
    return out


def _with_camera(sc, cam):
    d = capi.rt_scene_desc.from_buffer_copy(sc.desc)
    d.camera = cam
    return d


def _single(ctx, sc, cam, w=W, h=H, spp=SPP, seed=1, **kw):
    ctx.upload(_with_camera(sc, cam))
    ctx.render(w, h, spp, max_depth=DEPTH, seed=seed, **kw)
    return ctx.download(spp, linear=True, rgb8=True)


def _batch(ctx, sc, cams, w=W, h=H, spp=SPP, **kw):
    ctx.upload(sc)
    ctx.render_views(cams, w, h, spp, max_depth=DEPTH, **kw)
    return ctx.download_views(spp, linear=True, rgb8=True)


def _assert_views_equal(ctx, sc, cams, w=W, h=H, seeds=None, **kw):
    lin, b8 = _batch(ctx, sc, cams, w, h, seeds=seeds, **kw)
    assert lin.shape == (len(cams), h, w, 3) and b8.shape == (len(cams), h, w, 3)
    for v, cam in enumerate(cams):
        ref_lin, ref_b8 = _single(ctx, sc, cam, w, h, seed=seeds[v] if seeds else kw.get("seed", 1),
                                  **{k: x for k, x in kw.items() if k != "seed"})
        assert np.array_equal(lin[v], ref_lin), f"view {v}: linear planes differ"
        assert np.array_equal(b8[v], ref_b8), f"view {v}: RGB8 planes differ"
    assert np.any(b8)


@pytest.mark.parametrize("name", ["book1", "cornell", "cornell_smoke", "mesh", "final"])
def test_each_view_is_its_own_render(ctx, scene_of, name):
    sc = scene_of(name)
    w, h = (96, 54) if name == "final" else (W, H)
    _assert_views_equal(ctx, sc, _orbit(sc.desc.camera, 5), w, h)


def test_a_defocused_view_of_a_lite_scene(ctx, scene_of):
    sc = scene_of("cornell")  # LITE: no triangles, point lights or defocus; one view needs the defocus code
    assert sc.desc.camera.defocus_angle == 0
    _assert_views_equal(ctx, sc, _orbit(sc.desc.camera, 4, defocus_view=2))


@pytest.mark.parametrize("name", ["cornell", "cornell_smoke", "final"])
def test_views_with_nee(ctx, scene_of, name):
    sc = scene_of(name)
    _assert_views_equal(ctx, sc, _orbit(sc.desc.camera, 3), nee=True)


def test_views_with_shadowed_point_lights(ctx, scene_of):
    sc = scene_of("mesh")
    assert sc.desc.n_lights > 0
    _assert_views_equal(ctx, sc, _orbit(sc.desc.camera, 3), shadowed_point_lights=True)


def test_per_view_seeds(ctx, scene_of):
    sc = scene_of("cornell_smoke")
    cams = _orbit(sc.desc.camera, 3)
    _assert_views_equal(ctx, sc, cams, seeds=[7, 2**40 + 3, 7])
    # without seeds every view uses `seed`
    _assert_views_equal(ctx, sc, cams, seed=9)
    ctx.upload(sc)
    same = [cams[0]] * 3
    ctx.render_views(same, W, H, 4, max_depth=DEPTH, seeds=[1, 2, 1])
    v = ctx.download_views(4)
    assert np.array_equal(v[0], v[2]) and not np.array_equal(v[0], v[1])


def test_progressive_async_and_tiles_give_the_same_bits(ctx, scene_of):
    sc = scene_of("final")
    cams = _orbit(sc.desc.camera, 3)
    ctx.upload(sc)
    ctx.render_views(cams, W, H, 8, max_depth=DEPTH)
    ref = ctx.download_views(8, rgb8=True)
    ctx.render_views(cams, W, H, 3, max_depth=DEPTH)
    ctx.render_views(cams, W, H, 5, max_depth=DEPTH, spp_begin=3, accumulate=True)
    got = ctx.download_views(8, rgb8=True)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    ctx.render_views(cams, W, H, 8, max_depth=DEPTH, blocking=False)
    got = ctx.download_views(8, rgb8=True)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    for tile in (8, 32):
        ctx.render_views(cams, W, H, 8, max_depth=DEPTH, tile_size=tile)
        got = ctx.download_views(8, rgb8=True)
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), f"tile_size {tile}"
    # a sub-range of the views
    part = ctx.download_views(8, first=1, count=2, rgb8=True)
    assert np.array_equal(part[0], ref[0][1:]) and np.array_equal(part[1], ref[1][1:])


def test_views_and_the_single_frame_are_independent(ctx, scene_of):
    sc = scene_of("cornell")
    cams = _orbit(sc.desc.camera, 2)
    ctx.upload(sc)
    ctx.render(W, H, 4, max_depth=DEPTH, seed=5)
    frame = ctx.download(4, rgb8=True)
    up = ctx.stats()
    ctx.render_views(cams, W, H, 4, max_depth=DEPTH)
    views = ctx.download_views(4, rgb8=True)
    st = ctx.stats()
    assert st["upload_ms"] == up["upload_ms"] and st["bvh_nodes"] == up["bvh_nodes"] and st["upload_bytes"] == up["upload_bytes"]
    # a views render between a render and its download leaves that frame alone
    ctx.render(W, H, 4, max_depth=DEPTH, seed=5)
    ctx.render_views(cams[::-1], 40, 24, 2, max_depth=DEPTH)
    got = ctx.download(4, rgb8=True)
    assert np.array_equal(got[0], frame[0]) and np.array_equal(got[1], frame[1])
    # and the other way round
    ctx.render_views(cams, W, H, 4, max_depth=DEPTH)
    ctx.render(64, 40, 3, max_depth=DEPTH, seed=8)
    got = ctx.download_views(4, rgb8=True)
    assert np.array_equal(got[0], views[0]) and np.array_equal(got[1], views[1])


def test_stats_of_a_views_pass(ctx, scene_of):
    sc = scene_of("cornell")
    ctx.upload(sc)
    ctx.render_views(_orbit(sc.desc.camera, 3), W, H, 5, max_depth=DEPTH)
    st = ctx.stats()
    assert st["samples"] == 3 * W * H * 5 and st["kernel_launches"] == 1 and st["render_ms"] > 0


def _code(fn):
    with pytest.raises(capi.RtError) as e:
        fn()
    return e.value.code


def _raw_views(ctx, cams, n, flags=0, shard_count=0, w=W, h=H, spp=2, seeds=None):
    p = capi.rt_render_params()
    p.struct_size = C.sizeof(capi.rt_render_params)
    p.width, p.height, p.samples_per_pixel, p.max_depth, p.seed = w, h, spp, DEPTH, 1
    p.flags, p.shard_count = flags, shard_count
    arr = (capi.rt_camera * max(1, len(cams)))(*cams) if cams is not None else None
    return ctx.lib.rt_render_views(ctx._h, C.byref(p), arr, seeds, n)


def test_errors(built, scene_of):
    sc = scene_of("cornell")
    cams = _orbit(sc.desc.camera, 2)
    with capi.Context(0) as c:
        # nothing uploaded, nothing rendered
        assert _raw_views(c, cams, 2) == capi.RT_ERR_STATE
        assert _code(lambda: c.download_views(2)) == capi.RT_ERR_STATE
        c.upload(sc)
        assert _code(lambda: c.download_views(2)) == capi.RT_ERR_STATE  # no views render yet
        # invalid arguments
        assert _raw_views(c, cams, 0) == capi.RT_ERR_INVALID
        assert _raw_views(c, None, 2) == capi.RT_ERR_INVALID
        assert _raw_views(c, cams, 2, w=0) == capi.RT_ERR_INVALID
        bad = capi.rt_camera.from_buffer_copy(cams[1])
        bad.background[1] += 0.25
        assert _code(lambda: c.render_views([cams[0], bad], W, H, 2)) == capi.RT_ERR_INVALID
        # unsupported flags and shards
        for f in (capi.RT_FLAG_STATS, capi.RT_FLAG_MOMENTS, capi.RT_FLAG_COMPACT_TILES, capi.RT_FLAG_OVERLAP | capi.RT_FLAG_ASYNC | capi.RT_FLAG_ACCUMULATE):
            assert _raw_views(c, cams, 2, flags=f) == capi.RT_ERR_UNSUPPORTED, f
        assert _raw_views(c, cams, 2, shard_count=2) == capi.RT_ERR_UNSUPPORTED
        # the slot limit: 2^31 slots or more (checked before anything is allocated)
        assert _raw_views(c, cams[:1] * 2, 2, w=32768, h=32768) == capi.RT_ERR_UNSUPPORTED
        # accumulating before any views render
        assert _code(lambda: c.render_views(cams, W, H, 2, accumulate=True)) == capi.RT_ERR_STATE
        c.render_views(cams, W, H, 2, seeds=[3, 4])
        # accumulate mismatches: views, size, cameras, seeds
        assert _code(lambda: c.render_views(cams + cams[:1], W, H, 2, spp_begin=2, accumulate=True, seeds=[3, 4, 5])) == capi.RT_ERR_STATE
        assert _code(lambda: c.render_views(cams, W + 8, H, 2, spp_begin=2, accumulate=True, seeds=[3, 4])) == capi.RT_ERR_STATE
        assert _code(lambda: c.render_views(cams[::-1], W, H, 2, spp_begin=2, accumulate=True, seeds=[3, 4])) == capi.RT_ERR_STATE
        assert _code(lambda: c.render_views(cams, W, H, 2, spp_begin=2, accumulate=True, seeds=[3, 5])) == capi.RT_ERR_STATE
        assert _code(lambda: c.render_views(cams, W, H, 2, spp_begin=2, accumulate=True)) == capi.RT_ERR_STATE
        c.render_views(cams, W, H, 2, spp_begin=2, accumulate=True, seeds=[3, 4])  # the matching pass still continues
        # out-of-range views
        for first, count in ((-1, 1), (0, 3), (2, 1), (1, 0)):
            out = np.empty((max(count, 1), H, W, 3), np.float32)
            assert c.lib.rt_download_views(c._h, 4, first, count, out.ctypes.data, None) == capi.RT_ERR_INVALID, (first, count)
        assert c.download_views(4).shape == (2, H, W, 3)


def test_multi_device_context_is_unsupported(built, scene_of, monkeypatch):
    monkeypatch.setenv("RT_B200_ALLOW_DUPLICATE_DEVICES", "1")
    sc = scene_of("cornell")
    with capi.Context([0, 0]) as c:
        c.upload(sc)
        assert _code(lambda: c.render_views(_orbit(sc.desc.camera, 2), W, H, 2)) == capi.RT_ERR_UNSUPPORTED
        assert _code(lambda: c.download_views(2, count=1)) == capi.RT_ERR_UNSUPPORTED


def _read_png(path):
    """The mirror's PNG writer stores filter-0 scanlines in stored deflate blocks."""
    data = open(path, "rb").read()
    pos, idat, w, h = 8, b"", 0, 0
    while pos < len(data):
        n, tag = struct.unpack(">I4s", data[pos:pos + 8])
        body = data[pos + 8:pos + 8 + n]
        if tag == b"IHDR":
            w, h = struct.unpack(">II", body[:8])
        elif tag == b"IDAT":
            idat += body
        pos += 12 + n
    raw = np.frombuffer(zlib.decompress(idat), np.uint8).reshape(h, 1 + 3 * w)
    assert not raw[:, 0].any()
    return raw[:, 1:].reshape(h, w, 3)


def test_mirror_turntable(built, ctx, scene_of, tmp_path):
    s = capi.load_scenes()
    from raytracingoneweekendapplication_b200.assets import ensure_assets

    assets = ensure_assets(None).encode()
    w, h, spp, depth, n = 64, 36, 6, 12, 4
    s.rtsc_render_turntable(b"cornell_smoke", 1, assets, w, h, spp, depth, str(tmp_path / "tt.png").encode(), n, 0, 0)
    s.rtsc_render_png(b"cornell_smoke", 1, assets, w, h, spp, depth, str(tmp_path / "plain.png").encode())
    assert sorted(os.listdir(tmp_path)) == ["plain.png"] + [f"tt_{k:03d}.png" for k in range(n)]
    assert (tmp_path / "tt_000.png").read_bytes() == (tmp_path / "plain.png").read_bytes()
    sc = scene_of("cornell_smoke")
    for k in (1, 3):
        cam = capi.rt_camera()
        assert s.rtsc_turntable_camera(b"cornell_smoke", 1, assets, n, k, C.byref(cam)) == 0
        assert cam.lookat[:] == sc.desc.camera.lookat[:] and cam.lookfrom[:] != sc.desc.camera.lookfrom[:]
        _, ref = _single_depth(ctx, sc, cam, w, h, spp, depth)
        assert np.array_equal(_read_png(tmp_path / f"tt_{k:03d}.png"), ref), f"frame {k}"


def _single_depth(ctx, sc, cam, w, h, spp, depth):
    ctx.upload(_with_camera(sc, cam))
    ctx.render(w, h, spp, max_depth=depth, seed=1)
    return ctx.download(spp, linear=True, rgb8=True)
