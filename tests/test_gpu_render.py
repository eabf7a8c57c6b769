"""K1 + K8..K12 (wavefront path tracer) through the C ABI vs the oracle's restatement of
RandomSampler::sample_image + Naive/Mis integrators, and vs the reference's documented known answers.

Oracle and device share the counter-based RNG (same seed -> same sample set), so images agree far more tightly
than Monte-Carlo noise; the remaining differences come from libm (sinf/cosf/acosf/atan2f/powf) rounding.
Tolerances are on LINEAR radiance, per channel.
"""
import numpy as np
import pytest

from conftest import furnace_scene

pytestmark = pytest.mark.gpu


def rmse(a, b):
    return float(np.sqrt(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)))


def render_both(ptb, orc, ctx, scene, w, h, spp, method, seed=3):
    s = ptb.Scene(scene, ctx=ctx)
    opts = ptb.RenderOptions(samples_per_pixel=spp, render_method=method, width=w, height=h, seed=seed)
    g = s.render(opts)
    o = orc.OracleScene(scene)
    acc, counts, _ = o.render(w, h, spp, method, seed=seed)
    return g, acc / spp, ctx.stats(), counts


@pytest.mark.parametrize("method", [0, 1])
def test_rtweekend1_matches_oracle(ptb, orc, gpu_ctx, rtweekend1, method):
    gpu_ctx.stats_reset()
    g, o, st, counts = render_both(ptb, orc, gpu_ctx, rtweekend1, 160, 90, 32, method)
    assert g.shape == (90, 160, 3) and np.all(np.isfinite(g))
    # same RNG, same paths: per-channel RMSE well below the Monte-Carlo noise floor (~0.03 at 32 spp)
    assert rmse(g, o) < 5e-3
    assert abs(g.mean() - o.mean()) < 1e-3
    # ray accounting: identical definitions on both sides (SURVEY.md §8d, Q7)
    assert st.rays_camera == counts["camera"] == 160 * 90 * 32
    for a, b in ((st.rays_bounce, counts["bounce"]), (st.rays_shadow_sky, counts["shadow_sky"]),
                 (st.rays_reference, counts["reference"])):
        assert abs(a - b) <= 2e-3 * max(b, 1)
    assert st.paths == 160 * 90 * 32


def test_rtweekend1_miss_pixels_are_lerp(ptb, gpu_ctx, rtweekend1):
    """SURVEY.md appendix B: a camera ray that misses returns exactly the Lerp sky colour (both integrators)."""
    w, h = 64, 36
    for method in (0, 1):
        s = ptb.Scene(rtweekend1, ctx=gpu_ctx)
        img = s.render(ptb.RenderOptions(samples_per_pixel=4, render_method=method, width=w, height=h, seed=1))
        top = img[0]  # top row looks above the horizon: sky only
        assert np.all(top[:, 2] >= top[:, 0]) and np.all(top[:, 2] > 0.95)  # (0.5,0.7,1.0)*t + 1*(1-t), t in (0.5,1]
        assert np.all(top[:, 0] >= 0.5 - 1e-6) and np.all(top[:, 0] <= 1.0 + 1e-6)


@pytest.mark.parametrize("method", [0, 1])
def test_overshadowed_matches_oracle(ptb, orc, gpu_ctx, overshadowed, method):
    g, o, st, counts = render_both(ptb, orc, gpu_ctx, overshadowed, 160, 90, 32, method)
    assert np.all(np.isfinite(g))
    assert rmse(g, o) < 2e-2          # emitter scene: high-variance fireflies, a few decision flips move energy
    assert abs(g.mean() - o.mean()) < 5e-3 + 0.02 * o.mean()
    if method == 1:
        assert st.rays_shadow_light > 0 and st.rays_shadow_sky > 0
        assert abs(int(st.rays_shadow_light) - counts["shadow_light"]) <= 5e-3 * counts["shadow_light"]


def test_glass_and_metal_match_oracle_naive(ptb, orc, gpu_ctx):
    """Reflect + Refract (naive: quirk Q4 makes them black under MIS in the reference)."""
    s = ptb.meshgen.c3_scene(0.04)
    t = s.add_texture(ptb.TEX_SOLID, (0.8, 0.6, 0.2))
    m = s.add_material(ptb.MAT_REFLECT, t, 0.0)
    s.add_sphere((1.6, 3.5, 0.9), 0.6, m)
    s.add_sphere((-1.6, 3.5, 0.9), 0.6, 1)  # analytic glass sphere next to the tessellated one
    g, o, st, counts = render_both(ptb, orc, gpu_ctx, s, 160, 90, 16, 0)
    assert np.all(np.isfinite(g))
    assert rmse(g, o) < 3e-2
    assert abs(g.mean() - o.mean()) < 5e-3


def test_mis_strict_quirks(ptb, orc, gpu_ctx):
    """Q4: delta materials under MIS produce inf/NaN throughput and the sample is zeroed — device == oracle."""
    s = ptb.meshgen.c3_scene(0.03)
    g, o, st, counts = render_both(ptb, orc, gpu_ctx, s, 96, 54, 8, 1)
    assert np.all(np.isfinite(g))
    assert rmse(g, o) < 3e-2


@pytest.mark.parametrize("res,method", [((0, 0), 0), ((0, 0), 1), ((10, 10), 1)])
def test_furnace(ptb, gpu_ctx, res, method):
    """implementations/tests/sampling.rs:239-297: radiance (0.25,0.25,0.25) +- 0.001 seen along (0,0,3)->(0,0,-1).
    Rendered as a 64x36 image with a 0.0001-degree field of view: every pixel is that ray."""
    f = furnace_scene(ptb, res)
    f.set_camera((0, 0, 3), (0, 0, 0), (0, 1, 0), 1e-4)
    s = ptb.Scene(f, ctx=gpu_ctx)
    img = s.render(ptb.RenderOptions(samples_per_pixel=512, render_method=method, width=64, height=36, seed=9))
    val = img.reshape(-1, 3).mean(axis=0)
    assert np.linalg.norm(val - 0.25) < 1e-3, val


def test_mis_equals_naive(ptb, gpu_ctx, overshadowed):
    """implementations/tests/sampling.rs:181-207 (MIS == naive), on the shipped emitter scene with sky sampling off
    (with it on the black sky poisons MIS samples with NaN: quirk Q3)."""
    import copy
    s = copy.deepcopy(overshadowed)
    s.set_sky(int(s.sky["texture"][0]), (0, 0))
    sc = ptb.Scene(s, ctx=gpu_ctx)
    a = sc.render(ptb.RenderOptions(samples_per_pixel=256, render_method=0, width=96, height=54, seed=2))
    b = sc.render(ptb.RenderOptions(samples_per_pixel=256, render_method=1, width=96, height=54, seed=2))
    assert abs(a.mean() - b.mean()) < 0.01 * max(a.mean(), 1e-3) + 1e-3


def test_sample_offset_sharding_is_exact(ptb, gpu_ctx, rtweekend1):
    """§8e: rendering [0,8) then [8,16) into one accumulator == rendering [0,16): same sample set, f32 sum order aside."""
    sc = ptb.Scene(rtweekend1, ctx=gpu_ctx)
    full = sc.render(ptb.RenderOptions(samples_per_pixel=16, render_method=1, width=128, height=72, seed=5))
    ctx = gpu_ctx
    ctx.accum_clear()
    for off in (0, 8):
        ctx.render(ptb.RenderOptions(samples_per_pixel=8, sample_offset=off, render_method=1, width=128, height=72, seed=5))
    parts = ctx.accum_read(128, 72, normalise=True)
    assert np.max(np.abs(full - parts)) < 1e-5


def test_determinism_and_pool_size_independence(ptb, gpu_ctx, rtweekend1, monkeypatch):
    """The image does not depend on the pool size: one chunk vs 4096-path slots (18 chunks of the window wavefront)."""
    sc = ptb.Scene(rtweekend1, ctx=gpu_ctx)
    o = ptb.RenderOptions(samples_per_pixel=8, render_method=1, width=128, height=72, seed=5)
    a = sc.render(o)
    monkeypatch.setenv("PTB_POOL_PATHS", "4096")
    b = sc.render(o)
    monkeypatch.delenv("PTB_POOL_PATHS")
    assert np.max(np.abs(a - b)) < 1e-5


def test_progress_callback_and_abort(ptb, gpu_ctx, rtweekend1):
    """The progress callback ends at the call's spp; a non-zero return aborts a render of many small chunks
    (PTB_POOL_PATHS=1024 rounds up to one 4096-slot window per chunk)."""
    sc = ptb.Scene(rtweekend1, ctx=gpu_ctx)
    seen = []
    sc.render(ptb.RenderOptions(samples_per_pixel=4, render_method=0, width=64, height=36), update=lambda s, r: seen.append((s, r)) or False)
    assert seen and seen[-1][0] == 4
    with pytest.raises(ptb.PtbError) as e:
        import os
        os.environ["PTB_POOL_PATHS"] = "1024"
        try:
            sc.render(ptb.RenderOptions(samples_per_pixel=64, render_method=0, width=64, height=36), update=lambda s, r: True)
        finally:
            del os.environ["PTB_POOL_PATHS"]
    assert e.value.code == 7  # PTB_ERR_ABORTED


def test_errors(ptb, gpu_ctx, rtweekend1):
    c = ptb.Context(0)
    with pytest.raises(ptb.PtbError):
        c.render(ptb.RenderOptions(width=16, height=16, samples_per_pixel=1))   # not committed
    c.upload(rtweekend1)
    c.commit()
    with pytest.raises(ptb.PtbError):
        c.render(ptb.RenderOptions(width=1, height=16, samples_per_pixel=1))    # W-1 == 0 divides by zero in the reference
    c.close()


def test_per_pass_presentation_callback(ptb, gpu_ctx, rtweekend1):
    """SURVEY.md §8(f) N4 — random_sampler.rs:82-98: the closure sees the single-sample image of every pass exactly once,
    numbered 1..spp, and the TUI's running mean of those images (src/main.rs:179-185) equals the accumulator."""
    sc = ptb.Scene(rtweekend1, ctx=gpu_ctx)
    o = ptb.RenderOptions(samples_per_pixel=6, render_method=1, width=96, height=54, seed=8)
    one_call = sc.render(o)
    seen, mean = [], np.zeros((54, 96, 3), np.float64)

    def closure(img, i, rays):
        nonlocal mean
        seen.append((i, rays))
        mean += (img.astype(np.float64) - mean) / i          # `*pres += (acc - *pres) / i`
        return False

    passes = sc.render(o, presentation_update=closure)
    assert [i for i, _ in seen] == [1, 2, 3, 4, 5, 6] and all(r > 0 for _, r in seen)
    assert np.max(np.abs(passes - one_call)) < 1e-5          # same absolute sample indices -> same image
    assert np.max(np.abs(mean - passes)) < 1e-5
    # returning true stops the render like the reference's `return` (random_sampler.rs:84-86)
    calls = []
    with pytest.raises(ptb.PtbError) as e:
        sc.render(o, presentation_update=lambda img, i, r: calls.append(i) or i == 2)
    assert e.value.code == 7 and calls == [1, 2]


def test_render_multi_c_abi(ptb, gpu_ctx, rtweekend1):
    """SURVEY.md §8b/§8e: ptb_render_multi — one context per GPU, spp split inside the library, one ncclReduce to ctxs[0].
    With a single GPU it must equal Scene.render; with two or more the union of the shards is the same sample set."""
    import ctypes as C
    o = ptb.RenderOptions(samples_per_pixel=10, render_method=1, width=128, height=72, seed=6)
    sc = ptb.Scene(rtweekend1, ctx=gpu_ctx)
    want = sc.render(o)
    assert np.max(np.abs(ptb.render_multi([gpu_ctx], o) - want)) < 1e-6
    n = C.c_int32()
    ptb._lib.lib.ptb_device_count(C.byref(n))
    if n.value >= 2:
        ctxs = [ptb.Context(d) for d in range(min(n.value, 4))]
        for c in ctxs:
            c.upload(rtweekend1)
            c.commit()
        got = ptb.render_multi(ctxs, o)
        assert np.max(np.abs(got - want)) < 1e-5
        for c in ctxs:
            c.close()


def test_converged_images_agree_with_independent_samples(ptb, orc, gpu_ctx, rtweekend1):
    """North star: converged renders match the CPU render at equal spp within a per-channel RMSE of 1e-2 at 1024 spp. Here
    the two sides use DIFFERENT seeds (independent sample sets), so agreement is statistical, not path-for-path."""
    w, h, spp = 64, 36, 1024
    for method in (0, 1):
        sc = ptb.Scene(rtweekend1, ctx=gpu_ctx)
        g = sc.render(ptb.RenderOptions(samples_per_pixel=spp, render_method=method, width=w, height=h, seed=101))
        acc, _, _ = orc.OracleScene(rtweekend1).render(w, h, spp, method, seed=202)
        assert rmse(g, acc / spp) < 1e-2, (method, rmse(g, acc / spp))


@pytest.mark.parametrize("method", [0, 1])
def test_chunked_window_wavefront_agrees(ptb, gpu_ctx, overshadowed, method, monkeypatch):
    """The window wavefront in one chunk (every path resident, slot = generation index) and in 8 chunks trace the same
    paths: same image (f32 summation order aside), same ray counters."""
    sc = ptb.Scene(overshadowed, ctx=gpu_ctx)
    o = ptb.RenderOptions(samples_per_pixel=12, render_method=method, width=96, height=54, seed=9)

    def run():
        gpu_ctx.stats_reset()
        img = sc.render(o)
        st = gpu_ctx.stats()
        return img, (st.rays_camera, st.rays_bounce, st.rays_shadow_light, st.rays_shadow_sky, st.rays_reference, st.paths)

    a, ca = run()
    monkeypatch.setenv("PTB_POOL_PATHS", "8192")  # 62 208 paths -> 8 chunks
    b, cb = run()
    monkeypatch.delenv("PTB_POOL_PATHS")
    assert ca[0] == 96 * 54 * 12 and ca[5] == 96 * 54 * 12
    assert ca == cb
    assert np.allclose(a, b, rtol=1e-5, atol=1e-5)


def test_abort_between_chunks_in_window_mode(ptb, gpu_ctx, rtweekend1, monkeypatch):
    """Window mode calls the progress callback after each chunk; a non-zero return aborts the render (PTB_ERR_ABORTED),
    as `true` from the reference's per-pass closure does (random_sampler.rs:82-88)."""
    sc = ptb.Scene(rtweekend1, ctx=gpu_ctx)
    monkeypatch.setenv("PTB_POOL_PATHS", "8192")
    seen = []
    with pytest.raises(ptb.PtbError) as e:
        sc.render(ptb.RenderOptions(samples_per_pixel=16, render_method=0, width=64, height=36),
                  update=lambda s, r: seen.append(s) or len(seen) >= 2)
    monkeypatch.delenv("PTB_POOL_PATHS")
    assert e.value.code == 7 and len(seen) == 2 and seen[0] < seen[1] < 16
    # the context stays usable
    img = sc.render(ptb.RenderOptions(samples_per_pixel=2, render_method=0, width=64, height=36))
    assert np.all(np.isfinite(img))


def test_abort_clears_the_accumulator(ptb, gpu_ctx, rtweekend1, monkeypatch):
    """ptb200.h: an aborted ptb_render clears the accumulator, so a later read / render on the same context is not
    normalised by a stale sample count (pixels finished before the abort used to come out over-bright)."""
    ctx = gpu_ctx
    ctx.upload(rtweekend1)
    ctx.commit()
    o = ptb.RenderOptions(samples_per_pixel=16, render_method=0, width=64, height=36, seed=2)
    ctx.accum_clear()
    ctx.render(o)
    want = ctx.accum_read(64, 36, normalise=True).copy()
    monkeypatch.setenv("PTB_POOL_PATHS", "8192")
    ctx.accum_clear()
    with pytest.raises(ptb.PtbError) as e:
        ctx.render(o, progress=lambda s, r: True)
    assert e.value.code == 7
    monkeypatch.delenv("PTB_POOL_PATHS")
    assert not np.any(ctx.accum_read(64, 36, normalise=False))      # nothing left behind
    ctx.render(o)                                                     # no accum_clear in between: starts from zero
    got = ctx.accum_read(64, 36, normalise=True)
    assert np.allclose(got, want, rtol=1e-5, atol=1e-5)


def test_out_of_range_material_index_is_an_error_not_a_fault(ptb, rtweekend1):
    """ADVICE r1: a primitive whose material index is out of range must fail the commit with PTB_ERR_INVALID (the
    primitives go straight to device memory, so the device validates) and leave the process and the context usable."""
    import copy
    bad = copy.deepcopy(rtweekend1)
    bad.spheres = bad.spheres.copy()
    bad.spheres["material"][0] = 0xFFFFFFFF
    c = ptb.Context(0)
    c.upload(bad)
    with pytest.raises(ptb.PtbError) as e:
        c.commit()
    assert e.value.code == 1 and "material index" in str(e.value)
    c.upload(rtweekend1)      # same context, valid scene: no sticky CUDA error
    c.commit()
    c.render(ptb.RenderOptions(samples_per_pixel=1, render_method=0, width=32, height=18))
    assert np.all(np.isfinite(c.accum_read(32, 18)))
    c.close()


def test_image_tiles_add_up_to_the_image(ptb, gpu_ctx, overshadowed):
    """ptb_render_opts::row_begin / row_count (the image-tile axis of the multi-GPU split): bands of rows rendered one after
    the other into the same accumulator are the whole image — pixels keep their coordinates, RNG keys and camera rays."""
    ctx = gpu_ctx
    ctx.upload(overshadowed)
    ctx.commit()
    w, h = 96, 54
    base = dict(samples_per_pixel=6, render_method=1, width=w, height=h, seed=12)
    ctx.accum_clear()
    ctx.render(ptb.RenderOptions(**base))
    whole = ctx.accum_read(w, h, normalise=False).copy()
    ctx.accum_clear()
    for r0, rc in ((0, 20), (20, 1), (21, 0)):                  # 0 = every remaining row
        ctx.render(ptb.RenderOptions(row_begin=r0, row_count=rc, **base))
    tiles = ctx.accum_read(w, h, normalise=False)
    assert np.allclose(tiles, whole, rtol=1e-5, atol=1e-5)
    ctx.accum_clear()
    ctx.render(ptb.RenderOptions(row_begin=20, row_count=10, **base))
    band = ctx.accum_read(w, h, normalise=False)
    assert not np.any(band[:20]) and not np.any(band[30:]) and np.allclose(band[20:30], whole[20:30], rtol=1e-5, atol=1e-5)
    with pytest.raises(ptb.PtbError):
        ctx.render(ptb.RenderOptions(row_begin=50, row_count=10, **base))
    ctx.accum_clear()


def test_render_multi_fewer_samples_than_gpus(ptb, gpu_ctx, rtweekend1):
    """ptb_render_multi splits by image rows when samples_per_pixel < GPUs (north star: 'by samples-per-pixel and image
    tiles'). Needs >= 2 GPUs; on a single-GPU box only the n = 1 path is exercised."""
    import ctypes as C
    n = C.c_int32()
    ptb._lib.lib.ptb_device_count(C.byref(n))
    o = ptb.RenderOptions(samples_per_pixel=1, render_method=0, width=128, height=72, seed=6)
    want = ptb.Scene(rtweekend1, ctx=gpu_ctx).render(o)
    if n.value < 2:
        assert np.max(np.abs(ptb.render_multi([gpu_ctx], o) - want)) < 1e-6
        return
    ctxs = [ptb.Context(d) for d in range(min(n.value, 4))]
    for c in ctxs:
        c.upload(rtweekend1)
        c.commit()
    got = ptb.render_multi(ctxs, o)
    assert np.max(np.abs(got - want)) < 1e-6
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("method", [0, 1])
def test_fused_tail_hand_over_does_not_change_the_result(ptb, gpu_ctx, overshadowed, method, monkeypatch):
    """The last live paths of a chunk are finished by ONE k_tail launch on a side stream (closest hit -> shade -> NEE per
    lane) instead of ~45 nearly empty wavefront iterations. Same functions, same records, same RNG counters: the image and
    every ray counter are independent of where the hand-over happens (PTB_TAIL_PATHS: 0 = never, default 65 536, and a
    hand-over forced right after the first bounce)."""
    # overshadowed (14 primitives) takes the tail's lane walk, the 50 000-triangle mesh its warp-cooperative walk
    # (closest hit for both methods, any-hit for the NEE rays of MIS)
    scenes = [overshadowed, ptb.meshgen.c3_scene(0.05)]
    for scene in scenes:
        sc = ptb.Scene(scene, ctx=gpu_ctx)
        o = ptb.RenderOptions(samples_per_pixel=16, render_method=method, width=160, height=90, seed=4)

        def run():
            gpu_ctx.stats_reset()
            img = sc.render(o)
            st = gpu_ctx.stats()
            return img, (st.rays_camera, st.rays_bounce, st.rays_shadow_light, st.rays_shadow_sky, st.rays_reference, st.paths)

        monkeypatch.setenv("PTB_TAIL_PATHS", "0")
        a, ca = run()
        monkeypatch.delenv("PTB_TAIL_PATHS")
        b, cb = run()                                      # 230 400 paths: handed over once <= 65 536 are alive
        monkeypatch.setenv("PTB_TAIL_PATHS", str(1 << 24))
        c, cc = run()                                      # handed over after the first bounce
        monkeypatch.setenv("PTB_POOL_PATHS", "32768")      # 8 chunks alternating between the two slots, tails overlapping
        monkeypatch.setenv("PTB_TAIL_PATHS", "8192")
        d, cd = run()
        for k in ("PTB_TAIL_PATHS", "PTB_POOL_PATHS"):
            monkeypatch.delenv(k)
        assert ca == cb == cc == cd, (ca, cb, cc, cd)
        assert ca[5] == 160 * 90 * 16
        for other in (b, c, d):
            assert np.allclose(a, other, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("spp", [4, 32])
def test_camera_packets_are_the_same_rays(ptb, gpu_ctx, spp, monkeypatch):
    """The first iteration of a window-mode chunk walks the binary tree in packets (32 camera rays of a warp, one shared
    stack, per-lane participation masks — ptb_packet.cuh) when a warp's work items are samples of one pixel; forced on and
    off here, with one pixel per warp (32 spp) and eight (4 spp): same image, same ray counters, and the same hits as the
    per-ray walk down to the traversal statistics' primitive ids (the image is a function of the hits)."""
    sc = ptb.Scene(ptb.meshgen.c3_scene(0.05), ctx=gpu_ctx)
    o = ptb.RenderOptions(samples_per_pixel=spp, render_method=0, width=160, height=96, seed=9)
    out = []
    for packet in ("0", "1"):
        monkeypatch.setenv("PTB_CAMERA_PACKET", packet)
        gpu_ctx.stats_reset()
        img = sc.render(o)
        st = gpu_ctx.stats()
        out.append((img, (st.rays_camera, st.rays_bounce, st.rays_reference, st.paths)))
    monkeypatch.delenv("PTB_CAMERA_PACKET")
    assert out[0][1] == out[1][1]
    assert np.allclose(out[0][0], out[1][0], rtol=1e-5, atol=1e-5)
