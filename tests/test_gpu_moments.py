"""Per-pixel second moments (RT_FLAG_MOMENTS), the sample variance and the frame noise built on them.

The moments are exact integer sums of x^2, x being the integer a sample adds to its radiance word, so everything here
is compared for EQUALITY: against Python big-integer sums of single-sample frames, and across every way the samples of
a frame can be scheduled (passes, overlapped passes, tile and sample shards, two devices in one context, resume)."""
import math
import os
import re
import subprocess

import numpy as np
import pytest

from raytracingoneweekendapplication_b200 import capi

pytestmark = pytest.mark.gpu

W, H = 64, 48


def _s2(m):
    """S2 = m0 + m1 * 2^48 per channel, as Python integers (H, W, 3)."""
    m = m.astype(object)
    return m[..., 0::2] + m[..., 1::2] * (1 << 48)


def _d(sums, m, n):
    s1 = sums[..., :3].astype(object)
    return n * _s2(m) - s1 * s1


def _variance_ref(sums, m, n):
    d = _d(sums, m, n)
    return np.vectorize(lambda v: float(v) / float(n * (n - 1)) * 2.0 ** -56, otypes=[np.float64])(d).astype(np.float32)


def _noise_ref(sums, m, n, pixels):
    """The documented definition of rt_frame_noise: sum S1 and sum round(s^2 / n * 2^32), divided once."""
    d = _d(sums, m, n)
    q = np.vectorize(lambda v: min(round(float(v) / (float(n) * float(n) * float(n - 1)) * 2.0 ** -24), (1 << 64) - 1), otypes=[object])(d)
    s1 = int(sums[..., :3].astype(object).sum())
    values = 3.0 * pixels
    return float(s1) / (2.0 ** 28 * n * values), math.sqrt(math.ldexp(float(int(q.sum())), -32) / values)


def _ulps(a, b):
    return np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64)).max()


def _moments_frame(ctx, sc, spp, seed=3, nee=False, w=W, h=H):
    ctx.upload(sc)
    ctx.render(w, h, spp, seed=seed, nee=nee, moments=True)
    return ctx.accum_download(), ctx.moments_download()


@pytest.mark.parametrize("name", ["cornell", "cornell_smoke", "final", "mesh"])
@pytest.mark.parametrize("nee", [False, True])
def test_moments_leave_the_image_unchanged(ctx, scene_of, name, nee):
    ctx.upload(scene_of(name))
    ctx.render(W, H, 6, seed=3, nee=nee)
    plain = ctx.accum_download()
    ctx.render(W, H, 6, seed=3, nee=nee, moments=True)
    assert np.array_equal(ctx.accum_download(), plain)
    m = ctx.moments_download()
    assert m.shape == (H, W, 6) and m[..., 1::2].max() < (1 << 48) * 6 and np.any(m)


@pytest.mark.parametrize("nee", [False, True])
def test_moments_are_the_exact_sums_of_squared_samples(ctx, scene_of, nee):
    sc, n = scene_of("cornell"), 6
    ctx.upload(sc)
    frames = []
    for k in range(n):  # sample k alone: each radiance word is that sample's x
        ctx.render(W, H, 1, seed=3, spp_begin=k, nee=nee)
        frames.append(ctx.accum_download()[..., :3].astype(object))
    sq = sum(f * f for f in frames)
    sums, m = _moments_frame(ctx, sc, n, nee=nee)
    assert np.array_equal(sums[..., :3].astype(object), sum(frames))
    assert np.array_equal(_s2(m), sq)
    # the same samples in three accumulating passes
    ctx.render(W, H, 2, seed=3, nee=nee, moments=True)
    ctx.render(W, H, 3, seed=3, spp_begin=2, nee=nee, moments=True, accumulate=True)
    ctx.render(W, H, 1, seed=3, spp_begin=5, nee=nee, moments=True, accumulate=True)
    assert np.array_equal(ctx.moments_download(), m)

    var = ctx.download_variance(n)
    assert var.shape == (H, W, 3) and var.dtype == np.float32
    assert _ulps(var, _variance_ref(sums, m, n)) <= 1
    x = np.stack([f.astype(np.float64) for f in frames]) * 2.0 ** -28
    ref = x.var(axis=0, ddof=1)
    assert np.allclose(var, ref, rtol=2e-7, atol=1e-12 * max(float((x * x).max()), 1.0))
    assert ctx.lib.rt_download_variance(ctx._h, 1, var.ctypes.data) == capi.RT_ERR_INVALID


def test_variance_noise_and_moments_do_not_depend_on_scheduling(ctx, scene_of, monkeypatch):
    sc, n, w, h, tile = scene_of("cornell_smoke"), 12, 96, 80, 16
    ctx.upload(sc)
    ctx.render(w, h, n, seed=5, moments=True)
    sums, m, var, noise = ctx.accum_download(), ctx.moments_download(), ctx.download_variance(n), ctx.frame_noise(n)
    mean, rms = _noise_ref(sums, m, n, w * h)
    assert math.isclose(noise[0], mean, rel_tol=1e-15) and math.isclose(noise[1], rms, rel_tol=1e-15)

    def same_frame():
        assert np.array_equal(ctx.accum_download(), sums)
        assert np.array_equal(ctx.moments_download(), m)
        assert np.array_equal(ctx.download_variance(n), var)
        assert ctx.frame_noise(n) == noise

    for split in ([5, 4, 3], [1, 11]):  # accumulating passes
        begin = 0
        for k, s in enumerate(split):
            ctx.render(w, h, s, seed=5, spp_begin=begin, moments=True, accumulate=k > 0)
            begin += s
        same_frame()
    ctx.render(w, h, 4, seed=5, moments=True)  # overlapped passes
    for begin in (4, 8):
        ctx.render(w, h, 4, seed=5, spp_begin=begin, moments=True, accumulate=True, blocking=False, overlap=True)
    ctx.sync()
    same_frame()

    # tile shards (compact buffers) and sample shards, downloaded as full frames and added on the host
    for mode, compact in ((capi.RT_SHARD_TILES, True), (capi.RT_SHARD_TILES, False), (capi.RT_SHARD_SAMPLES, False)):
        tot_s, tot_m, tot_v = 0, 0, 0
        for r in range(3):
            ctx.render(w, h, n, seed=5, moments=True, shard_rank=r, shard_count=3, shard_mode=mode, tile_size=tile, compact=compact)
            s_r, m_r = ctx.accum_download(), ctx.moments_download()
            tot_s, tot_m = tot_s + s_r, tot_m + m_r
            if mode == capi.RT_SHARD_TILES:
                tot_v = tot_v + ctx.download_variance(n)  # zero outside the shard's tiles
            if compact:  # the noise of the pixels this context holds: the shard's own tiles
                got = ctx.frame_noise(n)
                ref = _noise_ref(s_r, m_r, n, _own_pixels(w, h, tile, r, 3))
                assert math.isclose(got[0], ref[0], rel_tol=1e-15) and math.isclose(got[1], ref[1], rel_tol=1e-15)
        assert np.array_equal(tot_s, sums) and np.array_equal(tot_m, m)
        if mode == capi.RT_SHARD_TILES:
            assert np.array_equal(tot_v, var)

    # two devices in one context (the same GPU twice where only one is visible)
    monkeypatch.setenv("RT_B200_ALLOW_DUPLICATE_DEVICES", "1")
    import torch
    ids = [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]
    md = capi.Context(ids)
    try:
        md.upload(sc)
        md.render(w, h, 5, seed=5, moments=True, shard_mode=capi.RT_SHARD_TILES, tile_size=tile)
        md.render(w, h, 7, seed=5, spp_begin=5, moments=True, accumulate=True, shard_mode=capi.RT_SHARD_TILES, tile_size=tile)
        assert np.array_equal(md.accum_download(), sums)
        assert np.array_equal(md.download_variance(n), var)
        assert md.frame_noise(n) == noise
        with pytest.raises(capi.RtError) as e:
            md.moments_download()
        assert e.value.code == capi.RT_ERR_UNSUPPORTED
    finally:
        md.close()


def _own_pixels(w, h, tile, rank, count):
    tx, ty = (w + tile - 1) // tile, (h + tile - 1) // tile
    return sum(min(tile, w - (t % tx) * tile) * min(tile, h - (t // tx) * tile) for t in range(rank, tx * ty, count))


def test_resume_restores_sums_and_moments(ctx, scene_of):
    sc, n, split = scene_of("final"), 10, 4
    sums, m = _moments_frame(ctx, sc, n, seed=9)
    var, noise = ctx.download_variance(n), ctx.frame_noise(n)
    ctx.render(W, H, split, seed=9, moments=True)
    part_s, part_m = ctx.accum_download(), ctx.moments_download()
    other = capi.Context(0)
    try:
        other.upload(sc)
        other.accum_upload(part_s)
        other.moments_upload(part_m)
        other.render(W, H, n - split, seed=9, spp_begin=split, moments=True, accumulate=True)
        assert np.array_equal(other.accum_download(), sums)
        assert np.array_equal(other.moments_download(), m)
        assert np.array_equal(other.download_variance(n), var)
        assert other.frame_noise(n) == noise
    finally:
        other.close()


def _code(fn, *a, **kw):
    with pytest.raises(capi.RtError) as e:
        fn(*a, **kw)
    return e.value.code


def test_state_and_argument_errors(ctx, scene_of):
    ctx.upload(scene_of("cornell"))
    ctx.render(W, H, 2, seed=1)
    assert _code(ctx.render, W, H, 2, seed=1, spp_begin=2, accumulate=True, moments=True) == capi.RT_ERR_STATE
    assert _code(ctx.download_variance, 2) == capi.RT_ERR_STATE
    assert _code(ctx.frame_noise, 2) == capi.RT_ERR_STATE
    assert _code(ctx.render, W, H, 2, seed=1, stats=True, moments=True) == capi.RT_ERR_UNSUPPORTED
    ctx.render(W, H, 2, seed=1, moments=True)
    m = ctx.moments_download()
    assert ctx.lib.rt_moments_download(ctx._h, m.ctypes.data, m.nbytes - 8) == capi.RT_ERR_INVALID
    assert ctx.lib.rt_moments_upload(ctx._h, m.ctypes.data, m.nbytes - 8, W, H) == capi.RT_ERR_INVALID
    ctx.accum_upload(ctx.accum_download())  # sums restored without their moments
    assert _code(ctx.render, W, H, 2, seed=1, spp_begin=2, accumulate=True, moments=True) == capi.RT_ERR_STATE
    assert _code(ctx.download_variance, 2) == capi.RT_ERR_STATE
    ctx.render(W, H, 2, seed=1, moments=True)
    ctx.render(W, H, 2, seed=1, spp_begin=2, accumulate=True)  # a pass without the flag leaves the frame without moments
    assert _code(ctx.download_variance, 4) == capi.RT_ERR_STATE


def test_frame_noise_falls_as_one_over_root_spp_and_nee_halves_the_variance(ctx, scene_of):
    sc, w, h = scene_of("cornell"), 96, 96
    ctx.upload(sc)
    rel = {}
    for n in (64, 256):
        ctx.render(w, h, n, seed=2, moments=True)
        mean, rms = ctx.frame_noise(n)
        ref = _noise_ref(ctx.accum_download(), ctx.moments_download(), n, w * h)
        assert math.isclose(mean, ref[0], rel_tol=1e-15) and math.isclose(rms, ref[1], rel_tol=1e-15)
        rel[n] = rms / mean
    assert 1.6 < rel[64] / rel[256] < 2.5, rel
    ctx.render(w, h, 64, seed=2, moments=True)
    plain = ctx.download_variance(64).mean()
    ctx.render(w, h, 64, seed=2, moments=True, nee=True)
    nee = ctx.download_variance(64).mean()
    assert nee < 0.5 * plain, (nee, plain)


# ---- host mirror: camera::render with a noise target (apps/rtow_b200) ----------------------------------------------
def _app(tmp_path, out, spp, *opts):
    from helpers import ROOT
    from raytracingoneweekendapplication_b200.assets import ensure_assets

    exe = os.path.join(ROOT, "apps", "rtow_b200")
    p = subprocess.run([exe, "cornell", str(tmp_path / out), ensure_assets(), "80", "80", str(spp), *map(str, opts)],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    reached = re.search(r"reached at (\d+) samples per pixel", p.stdout)
    return open(tmp_path / out, "rb").read(), int(reached.group(1)) if reached else None


def test_camera_stops_at_a_noise_target(built, scene_of, tmp_path):
    from test_frame_io import read_pfm

    sc = scene_of("cornell")
    c = capi.Context(0)
    try:
        c.upload(sc)
        rel = {}
        for s in (64, 128, 192):
            c.render(80, 80, s, max_depth=sc.depth, seed=1, moments=True)
            mean, rms = c.frame_noise(s)
            rel[s] = rms / mean
        c.render(80, 80, 128, max_depth=sc.depth, seed=1, moments=True)
        var128 = c.download_variance(128)
    finally:
        c.close()
    target = rel[192]
    stop = min(s for s in rel if rel[s] <= target)
    png, reached = _app(tmp_path, "noise.png", 1024, "--noise", repr(target), "--noise-every", 64)
    assert reached == stop < 1024
    fixed, none = _app(tmp_path, "fixed.png", stop)
    assert none is None and fixed == png
    # per-pixel variance output
    _app(tmp_path, "v.png", 128, "--variance", str(tmp_path / "v.pfm"))
    assert np.array_equal(read_pfm(str(tmp_path / "v.pfm")), var128)
    # a version-2 checkpoint resumed under the noise target
    ck = str(tmp_path / "n.ckpt")
    _, r = _app(tmp_path, "part.png", 1024, "--noise", repr(target), "--noise-every", 64, "--checkpoint", ck, "--stop-after", 64)
    assert (r is None) == (stop > 64)
    if stop > 64:
        assert os.path.getsize(ck) == 48 + 80 * 80 * 80
        assert int.from_bytes(open(ck, "rb").read(12)[8:12], "little") == 2
    resumed, reached = _app(tmp_path, "resumed.png", 1024, "--noise", repr(target), "--noise-every", 64, "--checkpoint", ck)
    assert reached == stop and resumed == png
    assert not os.path.exists(ck)
