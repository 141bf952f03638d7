"""The state rules of a frame and the planes that carry per-pixel data of the same samples (moments, AOV sums), where
no other test asserts them: a bound frame, a frame restored on a multi-device context, and rt_moments_upload after a
render."""
import numpy as np
import pytest

from raytracingoneweekendapplication_b200 import capi

pytestmark = pytest.mark.gpu

W, H = 64, 48


def _code(fn, *a, **kw):
    with pytest.raises(capi.RtError) as e:
        fn(*a, **kw)
    return e.value.code


def _rays(cam, w, h):
    """Valid camera rays: from the camera towards the look-at point, fanned out a little per pixel."""
    rec = np.zeros((h, w, 12), dtype=np.float32)
    jj, ii = np.mgrid[0:h, 0:w]
    rec[..., 0:3] = list(cam.lookfrom)
    rec[..., 3:6] = np.array(list(cam.lookat)) - np.array(list(cam.lookfrom))
    rec[..., 3] += (ii - w / 2) * 0.01
    rec[..., 4] += (h / 2 - jj) * 0.01
    rec[..., 6] = 0.01
    rec[..., 10] = -0.01
    return rec


def test_a_bound_frame_has_no_companions(built, scene_of):
    import torch

    c = capi.Context(0)
    try:
        c.upload(scene_of("cornell"))
        buf = torch.zeros(W * H * 4, dtype=torch.int64, device="cuda")
        c.render(W, H, 2, seed=1, moments=True)
        c.bind_accum(buf.data_ptr(), buf.numel() * 8, W, H)
        assert _code(c.render, W, H, 2, seed=1, spp_begin=2, accumulate=True, moments=True) == capi.RT_ERR_STATE
        assert _code(c.download_variance, 2) == capi.RT_ERR_STATE
        c.bind_accum(None, 0, 0, 0)
        c.render(W, H, 2, seed=1, aov=True)
        c.bind_accum(buf.data_ptr(), buf.numel() * 8, W, H)
        assert _code(c.render, W, H, 2, seed=1, spp_begin=2, accumulate=True, aov=True) == capi.RT_ERR_STATE
        assert _code(c.download_aov, 2) == capi.RT_ERR_STATE
        c.bind_accum(None, 0, 0, 0)
    finally:
        c.close()


@pytest.mark.parametrize("camera_rays", [False, True])
def test_a_bound_frame_takes_either_source(built, scene_of, camera_rays):
    """Sums of the first passes bound as the frame, then resumed: the uninterrupted render's sums, from the camera or
    from rays set after those passes."""
    import torch

    sc = scene_of("cornell")
    c = capi.Context(0)
    try:
        c.upload(sc)
        c.set_camera_rays(_rays(sc.desc.camera, W, H))
        c.render(W, H, 4, seed=3, camera_rays=camera_rays)
        whole = c.accum_download()
        c.render(W, H, 2, seed=3, camera_rays=not camera_rays)
        c.render(W, H, 2, seed=3, camera_rays=camera_rays)
        first = c.accum_download()
        c.set_camera_rays(_rays(sc.desc.camera, W, H))  # the same rays again: a new source for a rendered frame
        buf = torch.from_numpy(first.view(np.int64).reshape(-1)).cuda()
        c.bind_accum(buf.data_ptr(), buf.numel() * 8, W, H)
        c.render(W, H, 2, seed=3, spp_begin=2, accumulate=True, camera_rays=camera_rays)
        torch.cuda.synchronize()
        assert np.array_equal(buf.cpu().numpy().view(np.uint64).reshape(H, W, 4), whole)
        c.bind_accum(None, 0, 0, 0)
    finally:
        c.close()


def test_a_restored_multi_device_frame_has_no_companions(built, scene_of, monkeypatch):
    monkeypatch.setenv("RT_B200_ALLOW_DUPLICATE_DEVICES", "1")
    c = capi.Context([0, 0])
    try:
        c.upload(scene_of("cornell"))
        c.render(W, H, 2, seed=1, moments=True)
        c.render(W, H, 2, seed=1, spp_begin=2, accumulate=True, moments=True)  # accepted before the upload
        c.accum_upload(c.accum_download())
        assert _code(c.render, W, H, 2, seed=1, spp_begin=4, accumulate=True, moments=True) == capi.RT_ERR_STATE
        c.render(W, H, 2, seed=1, aov=True)
        c.accum_upload(c.accum_download())
        assert _code(c.render, W, H, 2, seed=1, spp_begin=2, accumulate=True, aov=True) == capi.RT_ERR_STATE
        c.render(W, H, 2, seed=1, spp_begin=2, accumulate=True)  # the restored sums themselves resume
    finally:
        c.close()


def test_moments_upload_follows_an_accum_upload(built, scene_of):
    c = capi.Context(0)
    try:
        c.upload(scene_of("cornell"))
        c.render(W, H, 2, seed=1, moments=True)
        sums, m = c.accum_download(), c.moments_download()
        assert _code(c.moments_upload, m) == capi.RT_ERR_STATE
        c.accum_upload(sums)
        c.render(W, H, 2, seed=1, spp_begin=2, accumulate=True)
        assert _code(c.moments_upload, m) == capi.RT_ERR_STATE
        c.accum_upload(sums)
        c.moments_upload(m)
        c.render(W, H, 2, seed=1, spp_begin=2, accumulate=True, moments=True)
    finally:
        c.close()
