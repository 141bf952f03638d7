"""Readbacks of a frame to host memory: every plane equals the frame it was taken of.

A hand-out (rt_download_begin / rt_untile_begin) copies out of the context's device staging buffers while the call has
long returned; the synchronous readbacks that follow it write those same buffers.  rt_frame_end must still return the
frame as of its begin.  Each sequence below runs once: the check is of the ordering the library promises, and the
frames are compared for EQUALITY (integer sums, a pure function of the Philox counter)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
from raytracingoneweekendapplication_b200 import capi  # noqa: E402


@pytest.fixture
def fresh_ctx(built):
    """A context of its own on cuda:0, so that no staging buffer or outstanding frame of another test is involved."""
    c = capi.Context(0)
    yield c
    c.close()


@pytest.fixture
def two_device_ctx(built, monkeypatch):
    """Device 0 listed twice: the multi-device gather and hand-out on one GPU."""
    monkeypatch.setenv("RT_B200_ALLOW_DUPLICATE_DEVICES", "1")
    c = capi.Context([0, 0])
    yield c
    c.close()


def _own_mask(w, h, tile, rank, count):
    """The pixels of the tiles of shard `rank` of `count` (tile t belongs to shard t mod count)."""
    y, x = np.mgrid[0:h, 0:w]
    return ((y // tile) * ((w + tile - 1) // tile) + x // tile) % count == rank


def test_hand_out_is_unchanged_by_later_readbacks(fresh_ctx, scene_of):
    c, sc = fresh_ctx, scene_of("final")
    w, h, spp = 1920, 1080, 4
    c.upload(sc)
    c.render(w, h, spp, seed=7, moments=True)
    want_lin, want_b8 = c.download(spp, linear=True, rgb8=True)
    c.download_begin(spp, linear=True, rgb8=True)
    # every one of these writes the device buffers the hand-out is copying from, or renders over the frame
    c.download(spp + 3, linear=True, rgb8=True)
    c.download_variance(spp)
    c.accum_download()
    c.render_views([sc.desc.camera, sc.desc.camera], 320, 180, 2, seeds=[1, 2])
    c.download_views(2, linear=True, rgb8=True)
    c.render(w, h, spp, seed=8, moments=True)
    lin, b8 = c.frame_end()
    assert np.array_equal(lin, want_lin)
    assert np.array_equal(b8, want_b8)


def test_untile_hand_out_is_unchanged_by_a_compact_checkpoint(fresh_ctx, scene_of):
    import torch

    c, sc = fresh_ctx, scene_of("final")
    w, h, spp, count, tile = 480, 270, 4, 2, 16
    c.upload(sc)
    c.render(w, h, spp, seed=7)
    want = c.download(spp, linear=True)
    cap = max(capi.load().rt_shard_pixels(w, h, tile, r, count) for r in range(count))
    glin = torch.zeros((count, cap * 3), dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    for r in range(count):
        c.render(w, h, spp, seed=7, shard_rank=r, shard_count=count, shard_mode=capi.RT_SHARD_TILES, tile_size=tile, compact=True)
        c.resolve_tiles(spp, None, cap, dev_linear=glin[r].data_ptr())
    sums = c.accum_download()        # the last shard's tiles in a zeroed full frame
    c.untile_begin(glin.data_ptr(), cap * 12, 12, count, w, h, tile)
    assert np.array_equal(c.accum_download(), sums)
    lin, _ = c.frame_end()
    assert np.array_equal(lin, want)


def test_multi_device_hand_out_is_unchanged_by_later_readbacks(two_device_ctx, scene_of):
    c, sc = two_device_ctx, scene_of("final")
    w, h, spp = 1280, 720, 4         # 3600 tiles: tile-sharded
    ref = capi.Context(0)
    try:
        ref.upload(sc)
        ref.render(w, h, spp, seed=7, moments=True)
        want_b8 = ref.download(spp, linear=False, rgb8=True)
        want_sums, want_var = ref.accum_download(), ref.download_variance(spp)
    finally:
        ref.close()
    c.upload(sc)
    c.render(w, h, spp, seed=7, moments=True)
    assert np.array_equal(c.accum_download(), want_sums)
    c.download_begin(spp, linear=False, rgb8=True)
    assert np.array_equal(c.accum_download(), want_sums)
    assert np.array_equal(c.download_variance(spp), want_var)
    c.render(w, h, spp, seed=8, moments=True)
    _, b8 = c.frame_end()
    assert np.array_equal(b8, want_b8)


def test_compact_shard_download_is_its_tiles_in_a_black_frame(fresh_ctx, scene_of):
    c, sc = fresh_ctx, scene_of("final")
    w, h, spp, rank, count, tile = 200, 136, 4, 1, 3, 16   # partial edge tiles on both axes
    c.upload(sc)
    c.render(w, h, spp, seed=7)
    want_lin, want_b8 = c.download(spp, linear=True, rgb8=True)
    c.render(w, h, spp, seed=7, shard_rank=rank, shard_count=count, shard_mode=capi.RT_SHARD_TILES, tile_size=tile, compact=True)
    lin, b8 = c.download(spp, linear=True, rgb8=True)
    own = _own_mask(w, h, tile, rank, count)
    assert own.any() and not own.all()
    assert np.array_equal(lin[own], want_lin[own]) and np.array_equal(b8[own], want_b8[own])
    assert not lin[~own].any() and not b8[~own].any()
