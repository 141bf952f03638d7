"""Parity gate (b): converged images.  The device render must reach >= 40 dB PSNR after gamma
against the reference's converged render, with per-channel mean linear radiance within 3 sigma
of Monte Carlo noise; plus the determinism properties the multi-GPU path relies on
(bit-identical under sharding, progressive passes and re-runs)."""
import numpy as np
import pytest
import torch

import helpers
from raytracingoneweekendapplication_b200 import capi

pytestmark = pytest.mark.gpu

CONVERGED = ["book1", "cornell", "cornell_smoke", "mesh", "final", "quads", "emissive", "specular", "mixed", "kitchen_sink", "monkey",
             # C1-C3 at a quarter of the BASELINE frame (200x112, 300x300, 300x300), reference at 8192 / 32768 / 32768 spp
             "book1_quarter", "cornell_quarter", "cornell_smoke_quarter"]
GPU_SPP = 32768


_bound = {}


def accum_of(ctx):
    """The frame's accumulation buffer (uint64 fixed-point sums) as a host array.  The tests
    render into a torch tensor bound with rt_bind_accum, which is also what bench.py does."""
    key = (ctx.width, ctx.height)
    torch.cuda.synchronize()
    return _bound[key].cpu().numpy().copy()


def bind(ctx, w, h):
    key = (w, h)
    if key not in _bound:
        _bound[key] = torch.zeros(w * h * 4, dtype=torch.int64, device="cuda")
    buf = _bound[key]
    ctx.bind_accum(buf.data_ptr(), buf.numel() * 8, w, h)
    return buf


@pytest.fixture(autouse=True)
def _unbind(ctx):
    yield
    ctx.bind_accum(None, 0, 0, 0)


@pytest.mark.parametrize("name", CONVERGED)
def test_converged_image_matches_reference(ctx, scene_of, name):
    """Against tests/golden/image_*.npz: float radiance rendered by the unmodified reference
    (get_ray + ray_color of Camera.txt) at 2048-32768 spp, with its per-pixel sample variance."""
    sc = scene_of(name.replace("_quarter", ""))
    ctx.upload(sc)
    g = helpers.golden("image", name)
    if g is None:
        pytest.skip(f"tests/golden/image_{name}.npz has not been generated")
    ref, ref_var, ref_spp, depth = g["image"].astype(np.float64), g["var"].astype(np.float64), int(g["spp"]), int(g["depth"])
    h, w, _ = ref.shape
    half = GPU_SPP // 2
    ctx.render(w, h, half, max_depth=depth, seed=101)
    a = ctx.download(half).astype(np.float64)
    ctx.render(w, h, half, max_depth=depth, seed=202)
    b = ctx.download(half).astype(np.float64)
    dev = 0.5 * (a + b)
    n = h * w
    # Monte Carlo error bars: the reference's from its sample variance, the device's from the
    # difference of two independent halves
    sigma_ref = np.sqrt((ref_var / ref_spp).sum(axis=(0, 1))) / n
    sigma_dev = 0.5 * np.sqrt(((a - b) ** 2).sum(axis=(0, 1))) / n
    sigma = np.sqrt(sigma_ref ** 2 + sigma_dev ** 2)
    diff = np.abs(dev.mean(axis=(0, 1)) - ref.mean(axis=(0, 1)))
    assert np.all(diff <= 3 * sigma + 1e-7), (name, diff, sigma, diff / sigma)
    psnr = helpers.psnr_after_gamma(dev, ref)
    assert psnr >= 40.0, (name, psnr)


@pytest.mark.parametrize("name,w,h", [("book1", 100, 56), ("cornell", 64, 64), ("cornell_smoke", 64, 64), ("final", 96, 54),
                                      ("kitchen_sink", 96, 54), ("mesh", 96, 54)])
def test_same_samples_as_the_oracle(ctx, scene_of, name, w, h):
    """The restatement draws from the same Philox stream as the device, so a 2-spp image is the
    SAME estimate pixel by pixel except where FP32 rounding sends a path through a different
    branch.  Much sharper than a statistical comparison."""
    from oracle import port

    sc = scene_of(name)
    ctx.upload(sc)
    depth, spp = 50, 2
    ref = port.render(sc, w, h, spp, depth=depth, seed=5)
    ctx.render(w, h, spp, max_depth=depth, seed=5)
    dev = ctx.download(spp).astype(np.float64)
    err = np.abs(dev - ref).max(axis=2)
    scale = np.maximum(np.abs(ref).max(axis=2), 1e-3)
    close = (err / scale) <= 2e-3
    assert close.mean() >= 0.93, (name, close.mean())
    # and the pixels that diverged do not bias the image
    assert abs(dev.mean() - ref.mean()) <= 0.05 * max(ref.mean(), 1e-3), (dev.mean(), ref.mean())


def test_rerun_is_bit_identical(ctx, scene_of):
    ctx.upload(scene_of("kitchen_sink"))
    bind(ctx, 160, 90)
    ctx.render(160, 90, 8, seed=3)
    a = accum_of(ctx)
    ctx.render(160, 90, 8, seed=3)
    assert np.array_equal(a, accum_of(ctx))
    ctx.render(160, 90, 8, seed=4)
    assert not np.array_equal(a, accum_of(ctx))


@pytest.mark.parametrize("count", [2, 4, 8])
@pytest.mark.parametrize("mode", [1, 2])
def test_sharded_render_is_bit_identical(ctx, scene_of, count, mode):
    """1/2/4/8-way tile or sample sharding summed into one buffer == the unsharded frame, bit
    for bit (64-bit fixed-point sums; Philox keyed on pixel, sample, bounce)."""
    ctx.upload(scene_of("final"))
    w, h, spp = 208, 117, 12
    bind(ctx, w, h)
    ctx.render(w, h, spp, seed=9)
    whole = accum_of(ctx)
    for rank in range(count):
        ctx.render(w, h, spp, seed=9, shard_rank=rank, shard_count=count, shard_mode=mode, accumulate=rank > 0)
    assert np.array_equal(whole, accum_of(ctx))


def test_progressive_passes_equal_one_pass(ctx, scene_of):
    ctx.upload(scene_of("cornell_smoke"))
    w, h = 120, 120
    bind(ctx, w, h)
    ctx.render(w, h, 24, seed=2)
    whole = accum_of(ctx)
    ctx.render(w, h, 10, seed=2)
    ctx.render(w, h, 14, seed=2, spp_begin=10, accumulate=True)
    assert np.array_equal(whole, accum_of(ctx))


def test_rgb8_is_the_reference_quantisation(ctx, scene_of):
    """Camera.txt:77-89: sqrt, clamp [0, 0.999], int(255.999 x)."""
    ctx.upload(scene_of("book1"))
    ctx.render(200, 112, 16, seed=1)
    lin, b8 = ctx.download(16, linear=True, rgb8=True)
    expect = (255.999 * np.clip(np.sqrt(np.maximum(lin.astype(np.float64), 0)), 0, 0.999)).astype(np.int64)
    assert np.abs(b8.astype(np.int64) - expect).max() <= 1
    assert (b8.astype(np.int64) == expect).mean() > 0.999


def test_full_4k_frame_properties(ctx, scene_of):
    """BASELINE's full C5 frame (3840x2160): too big for the CPU oracle, so size-independent
    properties: every pixel gets exactly its samples (accumulate linearity), nothing is dropped,
    and the tile-sharded halves add up to the whole."""
    ctx.upload(scene_of("final"))
    w, h = 3840, 2160
    bind(ctx, w, h)
    ctx.render(w, h, 2, seed=1, stats=True)
    st = ctx.stats()
    assert st["samples"] == w * h * 2 and st["nonfinite_samples"] == 0
    assert st["rays"] >= st["samples"]
    whole = accum_of(ctx)
    ctx.render(w, h, 1, seed=1)
    ctx.render(w, h, 1, seed=1, spp_begin=1, accumulate=True)
    assert np.array_equal(whole, accum_of(ctx))
    ctx.render(w, h, 2, seed=1, shard_rank=0, shard_count=2, shard_mode=1)
    ctx.render(w, h, 2, seed=1, shard_rank=1, shard_count=2, shard_mode=1, accumulate=True)
    assert np.array_equal(whole, accum_of(ctx))
    img = whole.reshape(h, w, 4)
    assert (img[..., 3] == 0).all()
    assert img[:200, 1200:2200, :3].mean() > img[:200, :400, :3].mean()   # the ceiling light is up there


def test_only_render_kernel_v2_is_accepted(built, monkeypatch):
    """The alternatives to render_kernel_v2 were removed: RT_B200_KERNEL=v1 | v3 | wf, left over from an old script,
    fails loudly instead of reporting v2's numbers under another name; v2 is accepted."""
    for version in ("v1", "v3", "wf"):
        monkeypatch.setenv("RT_B200_KERNEL", version)
        with pytest.raises(capi.RtError) as e:
            capi.Context(0).close()
        assert e.value.code == capi.RT_ERR_UNSUPPORTED and "removed" in str(e.value), version
    monkeypatch.setenv("RT_B200_KERNEL", "v2")
    capi.Context(0).close()


def test_lite_kernel_instance_renders_the_same_bits(ctx, scene_of):
    """Scenes without triangles, point lights and defocus run an instance of the kernel compiled
    without those features (smaller, faster); it must be the same function of the samples."""
    import os

    ctx.upload(scene_of("final"))
    bind(ctx, 200, 112)
    ctx.render(200, 112, 6, seed=4)
    lite = accum_of(ctx)
    os.environ["RT_B200_NO_LITE"] = "1"
    try:
        ctx.render(200, 112, 6, seed=4)
    finally:
        os.environ.pop("RT_B200_NO_LITE", None)
    assert np.array_equal(lite, accum_of(ctx))


def test_box_bounded_media_take_the_slab_test(built, scene_of, monkeypatch):
    """A constant_medium whose boundary is one box() (both smoke volumes of C3) is intersected with ONE three-slab test
    instead of 2 x 6 quad tests (boundary_pair_box).  Same entry/exit distances up to FP32 rounding: the counted
    boundary tests drop to one per query, the image statistics stay, and RT_B200_NO_BOX_MEDIA=1 restores the quad path."""
    sc = scene_of("cornell_smoke")
    w, h, spp = 200, 200, 64
    out = {}
    for mode in ("slabs", "quads"):
        if mode == "quads":
            monkeypatch.setenv("RT_B200_NO_BOX_MEDIA", "1")
        else:
            monkeypatch.delenv("RT_B200_NO_BOX_MEDIA", raising=False)
        c = capi.Context(0)
        try:
            c.upload(sc)
            c.render(w, h, spp, max_depth=sc.depth, seed=3, stats=True)
            st = c.stats()
            out[mode] = (c.download(spp).astype(np.float64), st["medium_queries"], st["boundary_tests"])
        finally:
            c.close()
    (a, qa, ba), (b, qb, bb) = out["slabs"], out["quads"]
    assert qa > 0 and ba == qa           # one slab test per (ray, medium)
    assert bb == 12 * qb                 # two passes over six quads
    assert abs(qa - qb) <= 0.001 * qb    # the same rays ask
    # the same estimator: almost every sample takes the same decisions (entry/exit distances differ in the last bits)
    same = np.isclose(a, b, rtol=1e-4, atol=1e-6).all(axis=2).mean()
    assert same >= 0.98, same
    assert np.allclose(a.mean(axis=(0, 1)), b.mean(axis=(0, 1)), rtol=2e-3)


@pytest.mark.parametrize("name", ["book1", "cornell", "cornell_smoke", "mesh", "final", "kitchen_sink"])
def test_the_feature_instances_render_the_same_bits(built, scene_of, monkeypatch, name):
    """A scene runs the instance of render_kernel_v2 that carries only the code it can reach (kInstances in rt_b200.cu:
    one per BASELINE config; kitchen_sink needs the general one); RT_B200_GENERAL_INSTANCE=1 forces the general
    instance: same sums."""
    sc = scene_of(name)
    out = []
    for forced in (False, True):
        if forced:
            monkeypatch.setenv("RT_B200_GENERAL_INSTANCE", "1")
        else:
            monkeypatch.delenv("RT_B200_GENERAL_INSTANCE", raising=False)
        c = capi.Context(0)
        try:
            c.upload(sc)
            c.render(192, 108, 6, max_depth=sc.depth, seed=11)
            out.append(c.accum_download())
        finally:
            c.close()
    assert np.array_equal(out[0], out[1])
