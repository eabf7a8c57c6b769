"""GPU: the denoiser (ptb_denoise / ptb_denoise_device): the device's spatial SVGF filter against the oracle
(oracle/denoise_api.cpp) on the sums of real renders, noise-free input passing through, noise reduction on the furnace
and on rtweekend1 against a converged render, determinism and the API's contract, every error rule, and the CLI."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import furnace_scene
from denoise_oracle import denoise as oracle_denoise
from test_gpu_aov import emitters_only_scene, sums
from test_gpu_materials import showcase_scene
from test_gpu_mesh import expect

pytestmark = pytest.mark.gpu


@pytest.fixture()
def dctx(ptb):
    c = ptb.Context(0)
    yield c
    c.close()


def opts(ptb, w, h, spp, seed=3, method=None):
    return ptb.RenderOptions(samples_per_pixel=spp, render_method=ptb.METHOD_MIS if method is None else method, width=w,
                             height=h, seed=seed)


def render_both(ctx, o):
    """Beauty and AOV sums of the same samples, from cleared accumulators."""
    ctx.accum_clear()
    ctx.render(o)
    ctx.aov_clear()
    ctx.render_aov(o)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def close(d, o, rtol, atol):
    return np.all(np.abs(d - o) <= rtol * np.abs(o) + atol)


SCENES = {
    "rtweekend1": lambda ptb, f: f["rtweekend1"],
    "overshadowed": lambda ptb, f: f["overshadowed"],  # its own sky settings: MIS samples hit quirk Q3 and are zeroed
    "showcase_lerp": lambda ptb, f: showcase_scene(ptb, sky="lerp"),
    "showcase_image": lambda ptb, f: showcase_scene(ptb, sky="image"),
    "c3_small": lambda ptb, f: ptb.meshgen.c3_scene(0.05),
    "furnace": lambda ptb, f: furnace_scene(ptb),
}
OPTION_SETS = [
    {},
    {"iterations": 1},
    {"iterations": 10, "sigma_luminance": 2.0},
    {"iterations": 3, "sigma_luminance": 8.0, "sigma_normal": 32.0, "sigma_depth": 0.25},
]
SIZES = [(2, 2), (37, 23), (3, 200), (1920, 1080)]


# ------------------------------------------------------------------------------------------------- 1. device == oracle
@pytest.mark.parametrize("which", list(SCENES))
def test_device_equals_oracle(ptb, gpu_ctx, rtweekend1, overshadowed, which):
    """|d - o| <= 1e-4 |o| + 1e-6 on the sums read back from the same context, up to five levels; at ten levels the
    absolute term is 1e-5. The two differ only in exp2f / log2f, whose last-bit differences in the tap weights build up over
    the levels: on overshadowed at 1080p with ten levels they reached 6.7e-6 (image peak 1.5), while every case up to five
    levels held the 1e-6 bound."""
    scene = SCENES[which](ptb, {"rtweekend1": rtweekend1, "overshadowed": overshadowed})
    gpu_ctx.upload(scene)
    gpu_ctx.commit()
    spp = 4
    for w, h in SIZES:
        render_both(gpu_ctx, opts(ptb, w, h, spp))
        b = gpu_ctx.accum_read(w, h, normalise=False).copy()
        a = sums(ptb, gpu_ctx, w, h)
        assert np.all(np.isfinite(b)) and np.all(np.isfinite(a))
        for o in OPTION_SETS:
            d = gpu_ctx.denoise(w, h, **o)
            ref = oracle_denoise(b, a, spp, spp, **o)
            assert np.all(np.isfinite(d)) and np.all(np.isfinite(ref))
            atol = 1e-5 if o.get("iterations", 5) > 5 else 1e-6
            excess = np.abs(d - ref) - 1e-4 * np.abs(ref)
            assert close(d, ref, 1e-4, atol), (w, h, o, float(excess.max()))


# ------------------------------------------------------------------------------------ 2. noise-free input comes through
def test_noise_free_input_comes_through(ptb, gpu_ctx):
    """An emitter-only scene's beauty is its albedo: the irradiance is 1 everywhere, edges included, so the filter returns
    the beauty."""
    gpu_ctx.upload(emitters_only_scene(ptb))
    gpu_ctx.commit()
    w, h = 96, 54
    render_both(gpu_ctx, opts(ptb, w, h, 8, seed=5, method=ptb.METHOD_NAIVE))
    beauty = gpu_ctx.accum_read(w, h)
    for o in OPTION_SETS:
        d = gpu_ctx.denoise(w, h, **o)
        assert np.abs(d - beauty).max() <= 1e-5, (o, float(np.abs(d - beauty).max()))


# ---------------------------------------------------------------------------------------------------- 3./4. it denoises
def rmse(a, b):
    return float(np.sqrt(np.mean((a.astype(np.float64) - b) ** 2)))


def rel_mse(a, ref):
    a, ref = a.astype(np.float64), ref.astype(np.float64)
    return float(np.mean((a - ref) ** 2 / (ref ** 2 + 1e-2)))


def test_furnace_noise_drops(ptb, gpu_ctx):
    """The furnace (64 x 36, a 1e-4 degree field of view: every pixel sees the grey sphere, analytic radiance 0.25) at
    4 spp: the denoised RMSE against 0.25 is at most a tenth of the noisy image's (measured on a B200: 0.00101 against
    0.0209, 20.7x; the bar asked for at first was 3x)."""
    f = furnace_scene(ptb)
    f.set_camera((0, 0, 3), (0, 0, 0), (0, 1, 0), 1e-4)
    gpu_ctx.upload(f)
    gpu_ctx.commit()
    render_both(gpu_ctx, opts(ptb, 64, 36, 4, seed=9))
    noisy = gpu_ctx.accum_read(64, 36)
    den = gpu_ctx.denoise(64, 36)
    assert rmse(den, 0.25) * 10 <= rmse(noisy, 0.25), (rmse(noisy, 0.25), rmse(den, 0.25))


def test_rtweekend1_relative_mse_drops(ptb, gpu_ctx, rtweekend1):
    """rtweekend1 at 160 x 90: 4 spp against a 4096-spp render of the same seed: the denoised relative MSE
    (mean of (x - ref)^2 / (ref^2 + 1e-2)) is at most a quarter of the noisy one's (measured on a B200: 0.00236 against
    0.0184, 7.8x; the bar asked for at first was 2x)."""
    gpu_ctx.upload(rtweekend1)
    gpu_ctx.commit()
    w, h = 160, 90
    gpu_ctx.accum_clear()
    gpu_ctx.render(opts(ptb, w, h, 4096, seed=21))
    ref = gpu_ctx.accum_read(w, h).copy()
    render_both(gpu_ctx, opts(ptb, w, h, 4, seed=21))
    noisy = gpu_ctx.accum_read(w, h)
    den = gpu_ctx.denoise(w, h)
    assert rel_mse(den, ref) * 4 <= rel_mse(noisy, ref), (rel_mse(noisy, ref), rel_mse(den, ref))


# ---------------------------------------------------------------------------------------- 5. determinism and contract
def test_determinism_device_variant_and_untouched_accumulators(ptb, gpu_ctx, rtweekend1):
    import torch
    L = ptb._lib
    gpu_ctx.upload(rtweekend1)
    gpu_ctx.commit()
    w, h = 160, 90
    render_both(gpu_ctx, opts(ptb, w, h, 4))
    b0 = gpu_ctx.accum_read(w, h, normalise=False).copy()
    m0 = gpu_ctx.accum_read(w, h).copy()
    a0 = sums(ptb, gpu_ctx, w, h)
    an0 = gpu_ctx.aov_read(w, h, L.PTB_AOV_ALBEDO).copy()
    o = {"iterations": 4, "sigma_luminance": 3.0}
    gpu_ctx.stats_reset()
    d1 = gpu_ctx.denoise(w, h, **o)
    st = gpu_ctx.stats()
    assert st.kernel_launches == 2 + 4 and st.trace_launches == 0 and st.rays_total == 0 and st.rays_reference == 0
    d2 = gpu_ctx.denoise(w, h, **o)
    assert np.array_equal(bits(d1), bits(d2))
    t = torch.full((w * h * 3,), float("nan"), dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    gpu_ctx.stats_reset()
    gpu_ctx.denoise_device(t.data_ptr(), **o)
    gpu_ctx.synchronize()
    assert gpu_ctx.stats().kernel_launches == 6
    assert np.array_equal(bits(t.cpu().numpy().reshape(h, w, 3)), bits(d1))
    gpu_ctx.stats_reset()
    gpu_ctx.denoise(w, h)
    assert gpu_ctx.stats().kernel_launches == 2 + 5
    # both accumulators and their sample counts are unchanged
    assert np.array_equal(bits(gpu_ctx.accum_read(w, h, normalise=False)), bits(b0))
    assert np.array_equal(bits(gpu_ctx.accum_read(w, h)), bits(m0))
    assert np.array_equal(bits(sums(ptb, gpu_ctx, w, h)), bits(a0))
    assert np.array_equal(bits(gpu_ctx.aov_read(w, h, L.PTB_AOV_ALBEDO)), bits(an0))


def test_scene_render_denoised_equals_the_manual_sequence(ptb, gpu_ctx, overshadowed):
    w, h = 96, 54
    o = opts(ptb, w, h, 6, seed=4)
    sc = ptb.Scene(overshadowed, ctx=gpu_ctx)
    got = sc.render_denoised(o, iterations=4)
    render_both(gpu_ctx, o)
    want = gpu_ctx.denoise(w, h, iterations=4)
    assert got.shape == (h, w, 3) and close(got, want, 1e-4, 1e-5), float(np.abs(got - want).max())


# ------------------------------------------------------------------------------------------------------- 6. error rules
def test_error_rules(ptb, dctx, rtweekend1):
    L = ptb._lib
    dn = dctx.denoise
    expect(ptb, dn, 16, 16, match="nothing rendered yet")
    dctx.upload(rtweekend1)
    dctx.commit()
    dctx.render(opts(ptb, 16, 16, 1))
    expect(ptb, dn, 16, 16, match="no AOV rendered yet")
    dctx.render_aov(opts(ptb, 24, 16, 1))
    expect(ptb, dn, 16, 16, match="the beauty image is 16x16 but the AOVs are 24x16")
    dctx.render_aov(opts(ptb, 16, 16, 1))
    dn(16, 16)  # the sizes agree now
    dctx.accum_clear()
    expect(ptb, dn, 16, 16, match="the beauty accumulator holds no samples")
    dctx.render(opts(ptb, 16, 16, 1))
    dctx.aov_clear()
    expect(ptb, dn, 16, 16, match="the AOV accumulator holds no samples")
    dctx.render_aov(opts(ptb, 16, 16, 1))
    dctx.stats_reset()
    expect_kw(ptb, dn, 16, 16, iterations=11, match="iterations must be <= 10 (got 11)")
    for name in ("sigma_luminance", "sigma_normal", "sigma_depth"):
        for bad in (-1.0, float("nan"), float("inf"), float("-inf")):
            expect_kw(ptb, dn, 16, 16, match=f"{name} must be finite and >= 0", **{name: bad})
    expect_kw(ptb, dn, 16, 16, flags=1, match="denoise flags must be 0")
    buf = np.zeros(16 * 16 * 3, np.float32)
    rc = L.lib.ptb_denoise(dctx._h, None, L.ptr(buf), buf.size)
    assert rc == 1 and b"null denoise opts" in L.lib.ptb_last_error(dctx._h)
    o = C.byref(ptb.denoise_opts())
    for ptr, n in ((None, buf.size), (L.ptr(buf), buf.size - 1), (L.ptr(buf), 16 * 16)):
        rc = L.lib.ptb_denoise(dctx._h, o, ptr, n)
        assert rc == 1 and b"denoise expects 768 floats" in L.lib.ptb_last_error(dctx._h)
    assert L.lib.ptb_denoise_device(dctx._h, None, None) == 1
    assert L.lib.ptb_denoise_device(dctx._h, o, None) == 1 and b"null device output" in L.lib.ptb_last_error(dctx._h)
    assert dctx.stats().kernel_launches == 0  # nothing was enqueued by a failing call
    assert L.lib.ptb_denoise(None, o, L.ptr(buf), buf.size) == 1


def expect_kw(ptb, fn, *args, match=None, **kw):
    with pytest.raises(ptb.PtbError) as e:
        fn(*args, **kw)
    assert e.value.code == 1 and match in str(e.value), str(e.value)


# ------------------------------------------------------------------------------------------------------------- 7. the CLI
def read_pfm(path, w, h):
    raw = path.read_bytes()
    hdr_end = raw.index(b"-1.0\n") + 5
    return np.frombuffer(raw[hdr_end:], np.float32).reshape(h, w, 3)[::-1]  # PFM stores rows bottom-up


def test_cli_denoise_matches_the_binding(ptb, gpu_ctx, root, tmp_path):
    cli = os.path.join(root, "raytracing-rust_b200", "ptb200-cli")
    assert os.path.exists(cli), "build the frontend with `make cli`"
    scene_path = os.path.join(root, "scenes", "rtweekend1.ssml")
    w, h = 96, 54
    out = tmp_path / "den.pfm"
    r = subprocess.run([cli, "-f", scene_path, "-s", "4", "-x", str(w), "-y", str(h), "-r", "mis", "-o", out.name, "--seed",
                        "5", "--denoise"], capture_output=True, text=True, timeout=300, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    img = read_pfm(out, w, h)
    gpu_ctx.upload(ptb.load_file(scene_path))
    gpu_ctx.commit()
    render_both(gpu_ctx, opts(ptb, w, h, 4, seed=5))
    want = gpu_ctx.denoise(w, h)
    assert close(img, want, 1e-4, 1e-5), float(np.abs(img - want).max())
    assert not close(img, gpu_ctx.accum_read(w, h), 1e-4, 1e-5)  # the denoised image, not the noisy one
