"""Parity at the sizes BASELINE.json states (VERDICT r1, next #1): the render and closest-hit paths against the oracle at
C2 / C3 / C5 size, the converged-image bar of the north star on the emitter scene and on a mesh, and the independent f64
intersector (oracle.closest_hit_f64, Moller-Trumbore / quadratic over every primitive).

Sizes are chosen so that the oracle side of the whole file costs ~2 minutes on the GPU box's host cores (the SAH build
of the 10 M-triangle heightfield alone is ~35 s, single threaded as in the reference).
Tolerances are on LINEAR radiance, per channel; closest hit is id-exact and t-bit-exact.
"""
import numpy as np
import pytest

from conftest import random_rays

pytestmark = pytest.mark.gpu

MISS = 0xFFFFFFFF


def rmse(a, b):
    return float(np.sqrt(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)))


def q1_region(rays, ratio):
    """Quirk Q1 (rt_core/ray.rs:16-37, primitives/mod.rs:72-82): Y-dominant rays are permuted x<->z, so the shear divides
    by dir.x; for |dir.x| << |dir.y| the f32 error bound delta_t of triangle.rs:160-177 grows like (dir.y/dir.x)^2 and the
    reference REJECTS genuine hits. `ratio` bounds |dir.x| / |dir.y|."""
    d = rays["d"] / np.linalg.norm(rays["d"], axis=1, keepdims=True)
    ax, ay, az = np.abs(d[:, 0]), np.abs(d[:, 1]), np.abs(d[:, 2])
    ydom = ~((ax > ay) & (ax > az)) & (ay > az)
    return ydom & (ax < ratio * ay)


def exact_or_tied(g, r):
    """Device answers == oracle answers: same primitive and bit-identical t, u, v — except exact-t ties between two
    primitives (quirk Q2: the reference keeps the first found in ITS tree order, the device the lower id)."""
    tie = (g["prim"] != r["prim"]) & (g["t"] == r["t"]) & (g["prim"] != MISS) & (r["prim"] != MISS)
    ok = ~tie
    assert tie.mean() < 1e-3
    assert np.array_equal(g["prim"][ok], r["prim"][ok]), f"{int((g['prim'][ok] != r['prim'][ok]).sum())} id mismatches"
    for f in ("t", "u", "v"):
        assert np.array_equal(g[f][ok].view(np.uint32), r[f][ok].view(np.uint32)), f
    return ok


# ------------------------------------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def c3_full(ptb):
    return ptb.meshgen.c3_scene(1.0)


@pytest.fixture(scope="module")
def c3_full_oracle(orc, c3_full):
    return orc.OracleScene(c3_full)  # the reference's SAH tree over 1 000 000 triangles (~3 s)


# ------------------------------------------------------------------------------------------------ (i) C2 at 1920 x 1080
@pytest.mark.parametrize("method", [0, 1])
def test_c2_overshadowed_1080p_matches_oracle(ptb, orc, gpu_ctx, overshadowed, method):
    """BASELINE configs[1] at its stated resolution, 4 spp, naive and strict-reference MIS (quirk Q3 kept), same seed on
    both sides: same sample set, so the images agree far below the Monte-Carlo noise (sigma ~ 0.3 per pixel at 4 spp)."""
    w, h, spp = 1920, 1080, 4
    sc = ptb.Scene(overshadowed, ctx=gpu_ctx)
    gpu_ctx.stats_reset()
    g = sc.render(ptb.RenderOptions(samples_per_pixel=spp, render_method=method, width=w, height=h, seed=21))
    st = gpu_ctx.stats()
    acc, counts, _ = orc.OracleScene(overshadowed).render(w, h, spp, method, seed=21)
    o = acc / spp
    assert np.all(np.isfinite(g))
    assert rmse(g, o) < 1e-2, rmse(g, o)
    assert abs(float(g.mean()) - float(o.mean())) < 5e-4
    # a decision flip (libm last-ulp differences in sinf / cosf / acosf) changes a whole path: such pixels must be rare
    assert float(np.mean(np.abs(g - o).max(axis=2) > 1e-3)) < 5e-3
    assert st.rays_camera == counts["camera"] == w * h * spp and st.paths == w * h * spp
    for a, b in ((st.rays_bounce, counts["bounce"]), (st.rays_shadow_light, counts["shadow_light"]),
                 (st.rays_shadow_sky, counts["shadow_sky"]), (st.rays_reference, counts["reference"])):
        assert abs(a - b) <= 2e-3 * max(b, 1), (a, b)


# ------------------------------------------------------------------------------------------------ (ii) C3 render, full size
def test_c3_full_size_render_matches_oracle(ptb, gpu_ctx, c3_full, c3_full_oracle):
    """BASELINE configs[2]: the 1 000 000-triangle mesh at 1920 x 1080, naive (quirk Q4), 2 spp, same seed vs the oracle's
    SAH-tree render — the bench workload itself, through the window-mode wavefront the bench uses."""
    w, h, spp = 1920, 1080, 2
    sc = ptb.Scene(c3_full, ctx=gpu_ctx)
    gpu_ctx.stats_reset()
    g = sc.render(ptb.RenderOptions(samples_per_pixel=spp, render_method=0, width=w, height=h, seed=22))
    st = gpu_ctx.stats()
    acc, counts, _ = c3_full_oracle.render(w, h, spp, 0, seed=22)
    o = acc / spp
    assert np.all(np.isfinite(g))
    assert rmse(g, o) < 1e-2, rmse(g, o)
    assert abs(float(g.mean()) - float(o.mean())) < 5e-4
    assert float(np.mean(np.abs(g - o).max(axis=2) > 1e-3)) < 1e-2
    assert st.rays_camera == counts["camera"] == w * h * spp and st.paths == w * h * spp
    assert abs(st.rays_bounce - counts["bounce"]) <= 2e-3 * counts["bounce"]
    assert st.rays_reference == st.rays_camera + st.rays_bounce   # naive: 1 per check_hit (integrators/mod.rs:34)


def test_c3_bench_chunking_is_the_same_image(ptb, gpu_ctx, c3_full, monkeypatch):
    """The bench renders 256 spp per call and the path pool splits such a call into chunks; chunking may only change the
    f32 summation order. 1080p x 8 spp in one chunk vs forced 2 Mi-path chunks."""
    w, h, spp = 1920, 1080, 8
    sc = ptb.Scene(c3_full, ctx=gpu_ctx)
    o = ptb.RenderOptions(samples_per_pixel=spp, render_method=0, width=w, height=h, seed=23)
    a = sc.render(o)
    monkeypatch.setenv("PTB_POOL_PATHS", str(1 << 21))
    b = sc.render(o)
    monkeypatch.delenv("PTB_POOL_PATHS")
    assert np.max(np.abs(a - b)) < 1e-5


# ------------------------------------------------------------------------------------------------ (iii) C3 closest hit vs SAH
def test_c3_full_size_closest_hit_matches_sah_oracle(ptb, gpu_ctx, c3_full, c3_full_oracle):
    """Full-size C3, 256 Ki incoherent rays + the 1080p camera rays of every 5th pixel, against the REFERENCE-SEMANTICS
    oracle (SAH tree, BFS un-culled candidates, test-all: acceleration/mod.rs:199-224, 265-298), not the LBVH one."""
    rays = random_rays(ptb, 1 << 18, 78, centre=(0, 4, 1), radius=6.0)
    cam = np.zeros((1080 // 5) * (1920 // 5), ptb.ray_dtype)
    k = 0
    for y in range(0, 1080 - 4, 5):
        for x in range(0, 1920 - 4, 5):
            org, d = c3_full_oracle.camera_ray((x + 0.5) / 1919, 1 - (y + 0.5) / 1079)
            cam["o"][k], cam["d"][k] = org, d
            k += 1
    rays = np.concatenate([rays, cam[:k]])
    gpu_ctx.upload(c3_full)
    gpu_ctx.commit()
    g = gpu_ctx.closest_hit(rays)
    r = c3_full_oracle.closest_hit(rays)
    exact_or_tied(g, r)
    assert 0.2 < float((g["prim"] != MISS).mean()) < 0.95


# ------------------------------------------------------------------------------------------------ (iv) C5 at 10 M triangles
def test_c5_full_size_matches_lbvh_and_sah_oracles(ptb, orc, gpu_ctx):
    """BASELINE configs[4] geometry (10 000 000-triangle heightfield), the first 2^20 rays of the bench's own Philox stream:
    bit-exact against the CPU traversal of the same LBVH; the first 2^16 also against the reference-semantics SAH oracle."""
    s = ptb.meshgen.heightfield_scene(2500, 2000)
    assert len(s.triangles) == 10_000_000
    gpu_ctx.upload(s)
    gpu_ctx.commit()
    rays = ptb.meshgen.philox_rays(1 << 20, first=0)
    g = gpu_ctx.closest_hit(rays)
    o = orc.OracleScene(s, split_type=-1)
    h, nodes, prims = o.lbvh_closest_hit(rays)
    assert np.array_equal(g["prim"], h["prim"])
    for f in ("t", "u", "v"):
        assert np.array_equal(g[f].view(np.uint32), h[f].view(np.uint32)), f
    del o
    sah = orc.OracleScene(s)   # ~35 s: the reference's top-down SAH build is single threaded
    n = 1 << 16
    r = sah.closest_hit(rays[:n])
    exact_or_tied(g[:n], r)
    assert 0.05 < float((g["prim"] != MISS).mean()) < 0.95


# ------------------------------------------------------------------------------------------------ (v) converged images
def test_converged_overshadowed_naive_1024spp(ptb, orc, gpu_ctx, overshadowed):
    """North star: converged renders match the CPU render at equal spp within RMSE 1e-2 at 1024 spp. INDEPENDENT sample
    sets (different seeds) on the scene with an emitter; two oracle renders of this kind differ by 4.5e-3."""
    w, h, spp = 64, 36, 1024
    g = ptb.Scene(overshadowed, ctx=gpu_ctx).render(
        ptb.RenderOptions(samples_per_pixel=spp, render_method=0, width=w, height=h, seed=101))
    acc, _, _ = orc.OracleScene(overshadowed).render(w, h, spp, 0, seed=202)
    assert rmse(g, acc / spp) < 1e-2, rmse(g, acc / spp)


def test_converged_c3_mesh_1024spp(ptb, orc, gpu_ctx):
    """Same bar on the C3 mesh (0.1 scale: 8 000 terrain + 2 000 glass triangles), naive, independent seeds."""
    w, h, spp = 64, 36, 1024
    s = ptb.meshgen.c3_scene(0.1)
    g = ptb.Scene(s, ctx=gpu_ctx).render(ptb.RenderOptions(samples_per_pixel=spp, render_method=0, width=w, height=h, seed=101))
    acc, _, _ = orc.OracleScene(s).render(w, h, spp, 0, seed=202)
    assert rmse(g, acc / spp) < 1e-2, rmse(g, acc / spp)


# ------------------------------------------------------------------------------------------------ (vi) independent intersector
def check_against_f64(ptb, g, f, margin, rays, scale, bary_tol=1e-4):
    """Device (f32 watertight, reference arithmetic) vs f64 Moller-Trumbore over every primitive.
    Outside the Q1 region and away from grazing / near-tie decisions (margin > 1e-4): ids equal and
    |dt| <= 1e-5 t + 2e-6 scale / min(margin, 1): a sphere hit at grazing margin m = sqrt(discriminant) / radius is
    conditioned like 1 / m (rounding the f32 INPUTS alone moves t by eps * scale / m), `scale` = |origin - centre| + radius.
    Inside the Q1 region the reference's conservative t bound may only LOSE hits: the device's answer is a miss or a hit at
    least as far as the true closest one."""
    q1 = q1_region(rays, 0.25)
    sure = ~q1 & (margin > 1e-4)
    assert sure.mean() > 0.8
    assert np.array_equal(g["prim"][sure], f["prim"][sure]), int((g["prim"][sure] != f["prim"][sure]).sum())
    hit = sure & (f["prim"] != MISS)
    tol = 1e-5 * np.abs(f["t"][hit]) + 2e-6 * scale[hit] / np.minimum(margin[hit], 1.0)
    assert np.all(np.abs(g["t"][hit] - f["t"][hit]) <= tol)
    # barycentrics: an f32 position error of ~t * 1e-6 relative to the triangle's size (2e-2 at 1 M triangles, t ~ 5)
    tri = hit & (f["u"] + f["v"] > 0)
    assert np.all(np.abs(g["u"][tri] - f["u"][tri]) < bary_tol) and np.all(np.abs(g["v"][tri] - f["v"][tri]) < bary_tol)
    inq = q1 & (g["prim"] != f["prim"]) & (margin > 1e-4)
    lost = (g["prim"][inq] == MISS) | (g["t"][inq] >= f["t"][inq] * (1 - 1e-5))
    assert np.all(lost)
    return float(inq.mean())


def test_f64_intersector_shipped_scenes(ptb, orc, gpu_ctx, rtweekend1, overshadowed):
    for scene, centre, radius in ((rtweekend1, (0, 1, 0), 3.0), (overshadowed, (-0.3, 0.3, -0.3), 1.5)):
        rays = random_rays(ptb, 100_000, 41, centre=centre, radius=radius)
        gpu_ctx.upload(scene)
        gpu_ctx.commit()
        g = gpu_ctx.closest_hit(rays)
        f, margin = orc.OracleScene(scene, split_type=-1).closest_hit_f64(rays)
        # f32 error of the sphere quadratic is relative to |origin - centre| + radius, not to t (radius-100 / -1000 ground)
        big = float(np.max(scene.spheres["radius"])) if len(scene.spheres) else 1.0
        check_against_f64(ptb, g, f, margin, rays, np.full(len(rays), big + radius + 2.0, np.float32))


def test_f64_intersector_c3_full_size(ptb, gpu_ctx, c3_full, c3_full_oracle):
    """2 048 rays x 1 000 000 triangles, brute force in double precision (~10 s of host work)."""
    rays = random_rays(ptb, 2048, 42, centre=(0, 4, 1), radius=6.0)
    gpu_ctx.upload(c3_full)
    gpu_ctx.commit()
    g = gpu_ctx.closest_hit(rays)
    f, margin = c3_full_oracle.closest_hit_f64(rays)
    frac_q1_lost = check_against_f64(ptb, g, f, margin, rays, np.full(len(rays), 12.0, np.float32), bary_tol=2e-3)
    assert frac_q1_lost < 0.02
