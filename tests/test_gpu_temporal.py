"""GPU: the temporal denoiser (ptb_denoise_temporal): the device against the oracle (oracle/temporal_api.cpp) frame by
frame over sequences with camera and object motion, exactly ptb_denoise's image whenever there is no usable history,
lower error than the spatial filter on a static scene, no ghosting behind a moving emitter, determinism, untouched
accumulators and the error rules."""
import copy
import ctypes as C
import os

import numpy as np
import pytest

from temporal_oracle import denoise_temporal as oracle_temporal
from test_gpu_aov import sums
from test_gpu_denoise import close, expect_kw, rel_mse
from test_temporal_oracle import moved_camera, plane_scene

pytestmark = pytest.mark.gpu


def opts(ptb, w, h, spp, seed=3, offset=0):
    return ptb.RenderOptions(samples_per_pixel=spp, render_method=ptb.METHOD_MIS, width=w, height=h, seed=seed,
                             sample_offset=offset)


def frame(ctx, o):
    ctx.accum_clear()
    ctx.render(o)
    ctx.aov_clear()
    ctx.render_aov(o)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def motion_sums(ctx, w, h):
    """Motion sums with the same means as the device's: (mean, count 1) where a sample was valid (t' > 0), else 0."""
    m = ctx.motion_read(w, h)
    out = np.zeros((h, w, 4), np.float32)
    valid = m[..., 2] > 0
    out[..., 0:3] = m
    out[..., 3] = valid
    return out


def sequence(ptb, which):
    """scene(k): frame k of a short animation, the camera and one sphere moving."""
    if which == "plane":
        base = plane_scene(ptb)

        def scene(k):
            s = moved_camera(base, (0.04 * k, 0.0, 0.0))
            s.spheres = s.spheres.copy()
            s.spheres["center"][0] += np.float32([0.08 * k, 0.05 * k, 0.0])
            return s
        return scene
    rt = ptb.load_file(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "scenes", "rtweekend1.ssml"))

    def scene(k):
        s = moved_camera(rt, (0.05 * k, 0.01 * k, 0.0))
        s.spheres = s.spheres.copy()
        s.spheres["center"][len(s.spheres) - 1] += np.float32([0.05 * k, 0.0, 0.0])
        return s
    return scene


# ------------------------------------------------------------------------------------------------- 4. device == oracle
@pytest.mark.parametrize("which,w,h,o", [("plane", 37, 23, {}), ("plane", 160, 90, {"iterations": 1}),
                                         ("rtweekend1", 96, 54, {"iterations": 3, "alpha_color": 0.1, "max_history": 3}),
                                         ("rtweekend1", 1920, 1080, {})])
def test_device_equals_oracle_over_a_sequence(ptb, gpu_ctx, which, w, h, o):
    """Five frames, the oracle carrying its own history: |d - o| <= 1e-4 |o| + 1e-5. As for ptb_denoise, the two differ
    only in exp2f / log2f; the tap tests read guides and motion that are bit-identical on both sides, so history reaches
    the same pixels and only the weights' last bits differ."""
    scene = sequence(ptb, which)
    hist = None
    gpu_ctx.denoise_temporal_reset()
    for k in range(5):
        gpu_ctx.upload(scene(k))
        gpu_ctx.commit()
        frame(gpu_ctx, opts(ptb, w, h, 2, seed=11, offset=2 * k))
        d = gpu_ctx.denoise_temporal(w, h, **o)
        b = gpu_ctx.accum_read(w, h, normalise=False)
        ref, hist = oracle_temporal(b, sums(ptb, gpu_ctx, w, h), motion_sums(gpu_ctx, w, h), 2, 2, hist, **o)
        gpu_ctx.motion_mark()
        assert np.all(np.isfinite(d))
        excess = np.abs(d - ref) - 1e-4 * np.abs(ref)
        assert close(d, ref, 1e-4, 1e-5), (k, float(excess.max()))
        if k > 0:
            assert np.mean(hist["m"][..., 2] > 1) > 0.3  # history is in use


# ------------------------------------------------------------------------------- 5. no usable history == ptb_denoise
def test_no_history_is_ptb_denoise(ptb, gpu_ctx, rtweekend1):
    w, h = 96, 54
    o = {"iterations": 4}
    gpu_ctx.upload(rtweekend1)
    gpu_ctx.commit()
    gpu_ctx.denoise_temporal_reset()
    for k, case in enumerate(["first", "history", "reset", "size", "cut"]):
        if case == "reset":
            gpu_ctx.denoise_temporal_reset()
        if case == "size":
            w, h = 80, 45
        if case == "cut":  # the camera turns around: every point is behind the marked camera, no valid motion
            s = copy.deepcopy(rtweekend1)
            s.camera["lower_left"] = 2 * s.camera["origin"] - s.camera["lower_left"]
            s.camera["horizontal"] = -s.camera["horizontal"]
            gpu_ctx.upload(s)
            gpu_ctx.commit()
        frame(gpu_ctx, opts(ptb, w, h, 2, offset=2 * k))
        t = gpu_ctx.denoise_temporal(w, h, **o)
        s_only = gpu_ctx.denoise(w, h, **o)
        gpu_ctx.motion_mark()
        if case == "history":
            assert not np.array_equal(bits(t), bits(s_only))
        else:
            assert np.array_equal(bits(t), bits(s_only)), case


# -------------------------------------------------------------------------------------------------- 6. it accumulates
def test_static_rtweekend1_beats_the_spatial_filter(ptb, gpu_ctx, rtweekend1):
    """rtweekend1 at 160 x 90, 12 frames of 1 spp with advancing sample_offset against a 4096-spp render: on the last frame
    the temporal output's relative MSE is at most half the spatial filter's (measured on a B200: 0.00336 against 0.00816,
    2.4x)."""
    w, h = 160, 90
    gpu_ctx.upload(rtweekend1)
    gpu_ctx.commit()
    gpu_ctx.accum_clear()
    gpu_ctx.render(opts(ptb, w, h, 4096, seed=21))
    ref = gpu_ctx.accum_read(w, h).copy()
    gpu_ctx.denoise_temporal_reset()
    for k in range(12):
        frame(gpu_ctx, opts(ptb, w, h, 1, seed=21, offset=10000 + k))
        t = gpu_ctx.denoise_temporal(w, h)
        gpu_ctx.motion_mark()
    sp = gpu_ctx.denoise(w, h)
    print(f"rel MSE: spatial {rel_mse(sp, ref):.5f} temporal {rel_mse(t, ref):.5f}")
    assert rel_mse(t, ref) * 2 <= rel_mse(sp, ref), (rel_mse(sp, ref), rel_mse(t, ref))


# ---------------------------------------------------------------------------------------------------- 7. no ghosting
def emitter_scene(ptb, x):
    s = ptb.HostScene()
    tp = s.add_texture(ptb.TEX_SOLID, (0.5, 0.5, 0.5))
    te = s.add_texture(ptb.TEX_SOLID, (1.0, 1.0, 1.0))
    sky = s.add_texture(ptb.TEX_SOLID, (0.3, 0.3, 0.3))
    s.add_sphere((x, 0.0, -4.0), 0.6, s.add_material(ptb.MAT_EMIT, te, 4.0))
    s.add_sphere((0.0, 0.0, -1005.0), 1000.0, s.add_material(ptb.MAT_LAMBERTIAN, tp, 1.0))
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 60.0)
    s.set_sky(sky, (0, 0))
    return s


def test_moving_emitter_leaves_no_ghost(ptb, gpu_ctx):
    """Six frames with the emitter at x = -1, then it jumps to x = +1: on the pixels it uncovered (emitter in the previous
    frame, plane now) the depth test rejects the emitter's history, so the output stays within 0.2 of the spatial-only
    output, far from the emitter's irradiance of 4 a ghost would carry (measured on a B200: 0.123 at most, where the
    spatial output is about 0.19; what is left is the lagging history of the neighbouring plane, whose lighting changed)."""
    w, h = 128, 72
    gpu_ctx.denoise_temporal_reset()
    alb = None
    for k in range(7):
        gpu_ctx.upload(emitter_scene(ptb, -1.0 if k < 6 else 1.0))
        gpu_ctx.commit()
        frame(gpu_ctx, opts(ptb, w, h, 4, offset=4 * k))
        prev_alb = alb
        alb = gpu_ctx.aov_read(w, h, ptb.PTB_AOV_ALBEDO).copy()
        t = gpu_ctx.denoise_temporal(w, h)
        gpu_ctx.motion_mark()
    s_only = gpu_ctx.denoise(w, h)
    uncovered = np.all(prev_alb > 0.99, axis=-1) & np.all(np.abs(alb - 0.5) < 1e-6, axis=-1)
    assert uncovered.sum() > 50
    diff = np.abs(t - s_only)[uncovered]
    assert diff.max() <= 0.2, float(diff.max())


# ------------------------------------------------------------------------------------- 8. determinism and the contract
def test_determinism_untouched_sums_and_launches(ptb, gpu_ctx):
    import torch
    w, h = 96, 54
    scene = sequence(ptb, "plane")
    ctxs = [gpu_ctx, ptb.Context(0)]
    try:
        outs = [[], []]
        for c, out in zip(ctxs, outs):
            c.denoise_temporal_reset()
            for k in range(4):
                c.upload(scene(k))
                c.commit()
                frame(c, opts(ptb, w, h, 2, offset=2 * k))
                before = (bits(c.accum_read(w, h, normalise=False)), bits(sums(ptb, c, w, h)), bits(c.motion_read(w, h)))
                c.stats_reset()
                out.append(c.denoise_temporal(w, h, iterations=3))
                st = c.stats()
                assert st.kernel_launches == 3 + 3 and st.trace_launches == 0 and st.rays_total == 0
                after = (bits(c.accum_read(w, h, normalise=False)), bits(sums(ptb, c, w, h)), bits(c.motion_read(w, h)))
                assert all(np.array_equal(a, b) for a, b in zip(before, after))
                c.motion_mark()
        for a, b in zip(*outs):
            assert np.array_equal(bits(a), bits(b))
        # the device variant continues the same history: equal to the host variant of a third context
        c3 = ptb.Context(0)
        try:
            for c in (gpu_ctx, c3):
                if c is c3:
                    for k in range(4):
                        c.upload(scene(k))
                        c.commit()
                        frame(c, opts(ptb, w, h, 2, offset=2 * k))
                        c.denoise_temporal(w, h, iterations=3)
                        c.motion_mark()
                c.upload(scene(4))
                c.commit()
                frame(c, opts(ptb, w, h, 2, offset=8))
            tt = torch.full((w * h * 3,), float("nan"), dtype=torch.float32, device="cuda:0")
            torch.cuda.synchronize()
            gpu_ctx.stats_reset()
            gpu_ctx.denoise_temporal_device(tt.data_ptr(), iterations=1)
            gpu_ctx.synchronize()
            assert gpu_ctx.stats().kernel_launches == 3 + 1 + 1
            host = c3.denoise_temporal(w, h, iterations=1)
            assert np.array_equal(bits(tt.cpu().numpy().reshape(h, w, 3)), bits(host))
        finally:
            c3.close()
    finally:
        ctxs[1].close()


def test_scene_render_denoised_temporal_equals_the_manual_sequence(ptb, gpu_ctx, overshadowed):
    w, h = 96, 54
    sc = ptb.Scene(overshadowed, ctx=gpu_ctx)
    gpu_ctx.denoise_temporal_reset()
    a = [sc.render_denoised_temporal(opts(ptb, w, h, 2, offset=2 * k), iterations=3) for k in range(2)]
    gpu_ctx.denoise_temporal_reset()
    b = []
    for k in range(2):
        frame(gpu_ctx, opts(ptb, w, h, 2, offset=2 * k))
        b.append(gpu_ctx.denoise_temporal(w, h, iterations=3))
        gpu_ctx.motion_mark()
    for x, y in zip(a, b):
        assert x.shape == (h, w, 3) and close(x, y, 1e-4, 1e-5)


def test_error_rules(ptb, rtweekend1):
    L = ptb._lib
    c = ptb.Context(0)
    try:
        dn = c.denoise_temporal
        expect_kw(ptb, dn, 16, 16, match="nothing rendered yet")
        c.upload(rtweekend1)
        c.commit()
        frame(c, opts(ptb, 16, 16, 1))
        dn(16, 16)
        expect_kw(ptb, dn, 16, 16, iterations=11, match="iterations must be <= 10 (got 11)")
        expect_kw(ptb, dn, 16, 16, sigma_depth=-1.0, match="sigma_depth must be finite and >= 0")
        expect_kw(ptb, dn, 16, 16, flags=1, match="temporal flags must be 0")
        for name in ("alpha_color", "alpha_moments"):
            for bad in (-0.1, 1.5, float("nan"), float("inf")):
                expect_kw(ptb, dn, 16, 16, match=f"{name} must be in (0, 1] or 0", **{name: bad})
        dn(16, 16, alpha_color=1.0, alpha_moments=0.5, max_history=255)
        expect_kw(ptb, dn, 16, 16, max_history=256, match="max_history must be <= 255 (got 256)")
        c.stats_reset()
        buf = np.zeros(16 * 16 * 3, np.float32)
        assert L.lib.ptb_denoise_temporal(c._h, None, L.ptr(buf), buf.size) == 1
        assert b"null temporal opts" in L.lib.ptb_last_error(c._h)
        o = C.byref(ptb.temporal_opts())
        for p, n in ((None, buf.size), (L.ptr(buf), buf.size - 1)):
            assert L.lib.ptb_denoise_temporal(c._h, o, p, n) == 1 and b"denoise expects 768 floats" in L.lib.ptb_last_error(c._h)
        assert L.lib.ptb_denoise_temporal_device(c._h, o, None) == 1 and b"null device output" in L.lib.ptb_last_error(c._h)
        assert c.stats().kernel_launches == 0
        assert L.lib.ptb_denoise_temporal(None, o, L.ptr(buf), buf.size) == 1
        assert L.lib.ptb_denoise_temporal_reset(None) == 1
    finally:
        c.close()
