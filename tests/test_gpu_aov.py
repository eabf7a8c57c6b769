"""GPU: denoiser feature buffers (ptb_render_aov / ptb_aov_clear / ptb_aov_read). The device's first-hit albedo, normal,
depth and coverage of the render's camera rays against the oracle (oracle/aov_api.cpp), against the render itself and
ptb_closest_hit on the same rays, split into sample ranges and row tiles, over every tree builder, refit, mesh and
instanced scenes, and the API's contract."""
import copy

import numpy as np
import pytest

from aov_oracle import AovOracle
from test_aov_oracle import camera_rays
from test_gpu_instances import flat_of
from test_gpu_materials import showcase_scene
from test_gpu_mesh import expect, flag

pytestmark = pytest.mark.gpu
MISS = 0xFFFFFFFF
AOVS = ("albedo", "normal", "depth", "coverage")


@pytest.fixture()
def ctx2(ptb):
    c = ptb.Context(0)
    yield c
    c.close()


def opts(ptb, w, h, spp, seed=7, **kw):
    return ptb.RenderOptions(samples_per_pixel=spp, render_method=ptb.METHOD_MIS, width=w, height=h, seed=seed, **kw)


def sums(ptb, ctx, w, h):
    """The raw AOV sums as the oracle lays them out: (H, W, 8) = albedo.rgb, coverage, normal.xyz, depth."""
    L = ptb._lib
    out = np.zeros((h, w, 8), np.float32)
    out[..., 0:3] = ctx.aov_read(w, h, L.PTB_AOV_ALBEDO, normalise=False)
    out[..., 3] = ctx.aov_read(w, h, L.PTB_AOV_COVERAGE, normalise=False)
    out[..., 4:7] = ctx.aov_read(w, h, L.PTB_AOV_NORMAL, normalise=False)
    out[..., 7] = ctx.aov_read(w, h, L.PTB_AOV_DEPTH, normalise=False)
    return out


def device_sums(ptb, ctx, o):
    ctx.aov_clear()
    ctx.render_aov(o)
    return sums(ptb, ctx, o.width, o.height)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def c3_small(ptb):
    return ptb.meshgen.c3_scene(0.05)


SCENES = {
    "rtweekend1": lambda ptb, f: f["rtweekend1"],
    "overshadowed": lambda ptb, f: f["overshadowed"],
    "showcase_lerp": lambda ptb, f: showcase_scene(ptb, sky="lerp"),
    "showcase_image": lambda ptb, f: showcase_scene(ptb, sky="image"),
    "c3_small": lambda ptb, f: c3_small(ptb),
}


# ------------------------------------------------------------------------------------------------- 1. device == oracle
@pytest.mark.parametrize("which", list(SCENES))
def test_device_equals_oracle(ptb, orc, gpu_ctx, rtweekend1, overshadowed, which):
    """Coverage bit for bit; depth and normal bit for bit wherever every sample of the pixel hits the same primitive on the
    device and in the oracle (near-ties may pick another primitive: at most 0.1 % of the pixels); albedo there within
    |d - o| <= 1e-5 |o| + 1e-6 (sinf / atan2f / acosf of the checkered, image and perlin textures are the device's libm)."""
    scene = SCENES[which](ptb, {"rtweekend1": rtweekend1, "overshadowed": overshadowed})
    w, h, spp, seed = 48, 27, 3, 11
    gpu_ctx.upload(scene)
    gpu_ctx.commit()
    d = device_sums(ptb, gpu_ctx, opts(ptb, w, h, spp, seed, sample_offset=2))
    o, o_prims = AovOracle(scene).render_aov(w, h, spp, seed=seed, sample_offset=2)
    d_prims = np.stack([gpu_ctx.closest_hit(camera_rays(ptb, orc, scene, w, h, seed, 2 + s))["prim"] for s in range(spp)], 1)
    same = (d_prims == o_prims).all(axis=1).reshape(h, w)
    assert same.mean() >= 0.999, same.mean()
    assert np.array_equal(bits(d[..., 3]), bits(o[..., 3]))
    assert np.array_equal(bits(d[same][:, 4:8]), bits(o[same][:, 4:8]))
    da, oa = d[same][:, 0:3], o[same][:, 0:3]
    assert np.all(np.abs(da - oa) <= 1e-5 * np.abs(oa) + 1e-6), np.abs(da - oa).max()
    assert 0.0 < d[..., 3].mean() and np.all((d[..., 0:3] >= 0) & (d[..., 0:3] <= spp))


# ------------------------------------------------------------------------------------------- 2. same rays as the render
def emitters_only_scene(ptb):
    """Only emitters of strength <= 1 and a sky <= 1: a sample's radiance is the emission of its first hit (or the sky's),
    which is its albedo, unclamped but already in [0, 1]."""
    s = ptb.HostScene()
    t_chk = s.add_texture(ptb.TEX_CHECKERED, (0.9, 0.6, 0.3), (0.2, 0.4, 1.0))
    t_warm = s.add_texture(ptb.TEX_SOLID, (1.0, 0.8, 0.5))
    sky = s.add_texture(ptb.TEX_LERP, (0.3, 0.5, 0.9), (1.0, 1.0, 1.0))
    s.add_sphere((0, 0, -100.5), 100.0, s.add_material(ptb.MAT_EMIT, t_chk, 0.7))
    s.add_sphere((0, 0, 0), 0.5, s.add_material(ptb.MAT_EMIT, t_warm, 1.0))
    s.add_sphere((1.1, 0.3, 0), 0.4, s.add_material(ptb.MAT_EMIT, t_chk, 0.5))
    s.set_camera((0, -3, 0.8), (0, 0, 0), (0, 0, 1), 60)
    s.set_sky(sky, (16, 8))
    return s


def test_albedo_is_the_radiance_of_an_emitter_only_scene(ptb, gpu_ctx):
    scene = emitters_only_scene(ptb)
    gpu_ctx.upload(scene)
    gpu_ctx.commit()
    o = ptb.RenderOptions(samples_per_pixel=8, render_method=ptb.METHOD_NAIVE, width=96, height=54, seed=5)
    gpu_ctx.accum_clear()
    gpu_ctx.render(o)
    beauty = gpu_ctx.accum_read(96, 54)
    gpu_ctx.aov_clear()
    gpu_ctx.render_aov(o)
    albedo = gpu_ctx.aov_read(96, 54, ptb._lib.PTB_AOV_ALBEDO)
    cov = gpu_ctx.aov_read(96, 54, ptb._lib.PTB_AOV_COVERAGE)
    assert 0.0 < cov.mean() < 1.0  # the sky is seen
    assert np.allclose(albedo, beauty, rtol=1e-6, atol=1e-6), np.abs(albedo - beauty).max()


def test_depth_equals_closest_hit_on_the_camera_rays(ptb, orc, gpu_ctx, rtweekend1):
    w, h, seed = 64, 36, 0xDEADBEEF12
    gpu_ctx.upload(rtweekend1)
    gpu_ctx.commit()
    gpu_ctx.aov_clear()
    gpu_ctx.render_aov(opts(ptb, w, h, 1, seed, sample_offset=3))
    hits = gpu_ctx.closest_hit(camera_rays(ptb, orc, rtweekend1, w, h, seed, 3))
    hit = hits["prim"] != MISS
    assert hit.any() and not hit.all()
    depth = gpu_ctx.aov_read(w, h, ptb._lib.PTB_AOV_DEPTH).reshape(-1)
    assert np.array_equal(bits(depth), bits(np.where(hit, hits["t"], 0)))
    assert np.array_equal(gpu_ctx.aov_read(w, h, ptb._lib.PTB_AOV_COVERAGE).reshape(-1), hit.astype(np.float32))


# --------------------------------------------------------------------------------------------- 3. decomposition is exact
def test_sample_ranges_and_row_tiles_add_up_bit_for_bit(ptb, gpu_ctx):
    scene = showcase_scene(ptb, sky="image")
    gpu_ctx.upload(scene)
    gpu_ctx.commit()
    w, h = 64, 27
    whole = device_sums(ptb, gpu_ctx, opts(ptb, w, h, 6))
    gpu_ctx.aov_clear()
    gpu_ctx.render_aov(opts(ptb, w, h, 2))
    gpu_ctx.render_aov(opts(ptb, w, h, 4, sample_offset=2))
    assert np.array_equal(bits(sums(ptb, gpu_ctx, w, h)), bits(whole))
    gpu_ctx.aov_clear()
    for rb, rc in ((0, 8), (8, 6), (14, 0)):  # 8 x 4 tiles, 16 x 2 tiles, rows
        gpu_ctx.render_aov(opts(ptb, w, h, 6, row_begin=rb, row_count=rc))
    assert np.array_equal(bits(sums(ptb, gpu_ctx, w, h)), bits(whole))


# -------------------------------------------------------------------------------------------------- 4. tree independence
@pytest.mark.parametrize("which", ["rtweekend1", "c3_small"])
def test_every_builder_gives_the_same_bits(ptb, gpu_ctx, rtweekend1, which):
    scene = rtweekend1 if which == "rtweekend1" else c3_small(ptb)
    o = opts(ptb, 80, 45, 2)
    res = []
    for builder in ("lbvh", "sah", "wide"):
        gpu_ctx.upload(scene)
        gpu_ctx.commit(flag(ptb, builder))
        res.append(device_sums(ptb, gpu_ctx, o))
    assert np.array_equal(bits(res[0]), bits(res[1])) and np.array_equal(bits(res[0]), bits(res[2]))


def test_refit_equals_a_fresh_commit(ptb, gpu_ctx, ctx2, overshadowed):
    gpu_ctx.upload(overshadowed)
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    moved = copy.deepcopy(overshadowed)
    moved.spheres["center"][:, 0] += np.float32(0.05)
    moved.triangles["p"][: len(moved.triangles) // 2, :, 2] += np.float32(0.02)
    gpu_ctx.update_spheres(0, moved.spheres)
    gpu_ctx.update_triangles(0, moved.triangles)
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    ctx2.upload(moved)
    ctx2.commit(ptb._lib.BUILD_SAH)
    o = opts(ptb, 80, 45, 2)
    assert np.array_equal(bits(device_sums(ptb, gpu_ctx, o)), bits(device_sums(ptb, ctx2, o)))


@pytest.mark.parametrize("kind", ["mesh", "instanced"])
def test_mesh_and_instanced_scenes_equal_their_flat_expansion(ptb, gpu_ctx, ctx2, kind):
    if kind == "mesh":
        scene, mesh = ptb.meshgen.c3_indexed(0.05)
        gpu_ctx.upload(scene, mesh=mesh)
        flat = copy.copy(scene)
        flat.triangles = mesh.expand()
    else:
        scene, mesh, inst, xf = ptb.meshgen.c3_instanced(0.05)
        gpu_ctx.upload(scene, mesh=mesh, instances=(inst, xf))
        flat = flat_of(scene, mesh, inst, xf)
    gpu_ctx.commit()
    ctx2.upload(flat)
    ctx2.commit()
    o = opts(ptb, 80, 45, 2)
    a = device_sums(ptb, gpu_ctx, o)
    assert a[..., 3].mean() > 0.1
    assert np.array_equal(bits(a), bits(device_sums(ptb, ctx2, o)))


# ------------------------------------------------------------------------------------------------------------ 5. contract
def test_normalisation(ptb, gpu_ctx, rtweekend1):
    L = ptb._lib
    gpu_ctx.upload(rtweekend1)
    gpu_ctx.commit()
    w, h, n = 40, 24, 5
    s = device_sums(ptb, gpu_ctx, opts(ptb, w, h, n))
    nf = np.float32(n)
    assert np.array_equal(bits(gpu_ctx.aov_read(w, h, L.PTB_AOV_ALBEDO)), bits(s[..., 0:3] / nf))
    assert np.array_equal(bits(gpu_ctx.aov_read(w, h, L.PTB_AOV_NORMAL)), bits(s[..., 4:7] / nf))
    assert np.array_equal(bits(gpu_ctx.aov_read(w, h, L.PTB_AOV_COVERAGE)), bits(s[..., 3] / nf))
    cov = s[..., 3]
    partial = (cov > 0) & (cov < n)
    assert partial.any() and (cov == 0).any()
    want = np.where(cov > 0, s[..., 7] / np.where(cov > 0, cov, np.float32(1)), np.float32(0))
    assert np.array_equal(bits(gpu_ctx.aov_read(w, h, L.PTB_AOV_DEPTH)), bits(want))


def test_empty_scene_gives_sky_albedo_and_zeros(ptb, gpu_ctx, rtweekend1):
    L = ptb._lib
    s = copy.deepcopy(rtweekend1)
    s.spheres, s.triangles = s.spheres[:0], s.triangles[:0]
    sky = s.add_texture(ptb.TEX_SOLID, (1.5, 0.25, 0.75))
    s.set_sky(sky, (0, 0))
    gpu_ctx.upload(s)
    gpu_ctx.commit()
    gpu_ctx.aov_clear()
    gpu_ctx.render_aov(opts(ptb, 32, 18, 3))
    assert np.all(gpu_ctx.aov_read(32, 18, L.PTB_AOV_ALBEDO) == np.float32([1.0, 0.25, 0.75]))
    for a in (L.PTB_AOV_NORMAL, L.PTB_AOV_DEPTH, L.PTB_AOV_COVERAGE):
        assert not gpu_ctx.aov_read(32, 18, a).any()


def test_size_change_resets_and_clear_zeroes(ptb, gpu_ctx, rtweekend1):
    L = ptb._lib
    gpu_ctx.upload(rtweekend1)
    gpu_ctx.commit()
    gpu_ctx.aov_clear()
    gpu_ctx.render_aov(opts(ptb, 40, 24, 2))
    gpu_ctx.render_aov(opts(ptb, 48, 24, 1))  # another size: the 40 x 24 sums are dropped
    one = device_sums(ptb, gpu_ctx, opts(ptb, 48, 24, 1))
    gpu_ctx.aov_clear()
    gpu_ctx.render_aov(opts(ptb, 40, 24, 2))
    gpu_ctx.render_aov(opts(ptb, 48, 24, 1))
    assert np.array_equal(bits(sums(ptb, gpu_ctx, 48, 24)), bits(one))
    assert np.array_equal(bits(gpu_ctx.aov_read(48, 24, L.PTB_AOV_COVERAGE)), bits(one[..., 3]))  # divided by 1 sample
    gpu_ctx.aov_clear()
    assert not sums(ptb, gpu_ctx, 48, 24).any()
    expect(ptb, gpu_ctx.aov_read, 40, 24, L.PTB_AOV_DEPTH)  # the buffers are 48 x 24 now


def test_beauty_accumulator_is_untouched_and_stats_count_launches(ptb, gpu_ctx, rtweekend1):
    gpu_ctx.upload(rtweekend1)
    gpu_ctx.commit()
    o = opts(ptb, 64, 36, 4)
    gpu_ctx.accum_clear()
    gpu_ctx.render(o)
    before = gpu_ctx.accum_read(64, 36, normalise=False).copy()
    mean_before = gpu_ctx.accum_read(64, 36).copy()
    gpu_ctx.stats_reset()
    gpu_ctx.aov_clear()
    gpu_ctx.render_aov(o)
    gpu_ctx.synchronize()
    st = gpu_ctx.stats()
    assert st.kernel_launches == 4 and st.trace_launches == 4
    assert st.rays_total == 0 and st.rays_reference == 0 and st.paths == 0
    assert np.array_equal(bits(gpu_ctx.accum_read(64, 36, normalise=False)), bits(before))
    assert np.array_equal(bits(gpu_ctx.accum_read(64, 36)), bits(mean_before))  # sample count unchanged
    # and Scene.render_aov returns the four normalised buffers of the same samples
    sc = ptb.Scene(rtweekend1, ctx=gpu_ctx)
    d = sc.render_aov(o)
    assert set(d) == set(AOVS) and d["albedo"].shape == (36, 64, 3) and d["depth"].shape == (36, 64)
    assert np.array_equal(bits(d["coverage"]), bits(gpu_ctx.aov_read(64, 36, ptb._lib.PTB_AOV_COVERAGE)))


def test_error_rules(ptb, gpu_ctx, ctx2, rtweekend1):
    L = ptb._lib
    expect(ptb, ctx2.render_aov, opts(ptb, 16, 16, 1), match="scene not committed")
    expect(ptb, ctx2.aov_read, 16, 16, L.PTB_AOV_ALBEDO, match="no AOV rendered yet")  # read before any AOV render
    ctx2.upload(rtweekend1)
    ctx2.commit()
    expect(ptb, ctx2.aov_read, 16, 16, L.PTB_AOV_ALBEDO, match="no AOV rendered yet")
    expect(ptb, ctx2.render_aov, opts(ptb, 1, 16, 1), match="width and height must be >= 2")
    expect(ptb, ctx2.render_aov, opts(ptb, 16, 1, 1), match="width and height must be >= 2")
    expect(ptb, ctx2.render_aov, opts(ptb, 65536, 65536, 1), match="image too large")
    expect(ptb, ctx2.render_aov, opts(ptb, 16, 16, 1, row_begin=16), match="image tile rows")
    expect(ptb, ctx2.render_aov, opts(ptb, 16, 16, 1, row_begin=10, row_count=7), match="image tile rows")
    o = opts(ptb, 16, 16, 1)
    o.render_method = 7  # not read: no error
    ctx2.render_aov(o)
    with pytest.raises(ptb.PtbError):  # ... while ptb_render rejects it
        ctx2.render(o)
    expect(ptb, ctx2.aov_read, 16, 16, 4, match="unknown AOV")
    buf = np.zeros(16 * 16 * 3, np.float32)
    for aov, n in ((L.PTB_AOV_ALBEDO, 16 * 16), (L.PTB_AOV_NORMAL, 16 * 16 * 3 + 1), (L.PTB_AOV_DEPTH, 16 * 16 * 3),
                   (L.PTB_AOV_COVERAGE, 16 * 16 - 1)):
        rc = L.lib.ptb_aov_read(ctx2._h, aov, L.ptr(buf), n, 1)
        assert rc == 1 and b"aov_read expects" in L.lib.ptb_last_error(ctx2._h)
