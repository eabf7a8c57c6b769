"""CPU: the motion-vector oracle (oracle/motion_api.cpp) and the temporal denoiser's oracle (oracle/temporal_api.cpp),
which ptb_render_aov's motion sums and ptb_denoise_temporal are compared against: a step without history is the spatial
filter bit for bit, a static frame has exactly zero motion, and a sideways camera translation in front of a plane
perpendicular to the view gives the analytic, uniform Δx."""
import numpy as np
import pytest

from aov_oracle import AovOracle, split
from denoise_oracle import denoise
from motion_oracle import MotionOracle, mean
from temporal_oracle import denoise_temporal, empty_history
from test_denoise_oracle import make_sums, quadrants


def plane_scene(ptb, depth=5.0, sphere=True):
    """A Lambertian square (two triangles, normal +z) at z = -depth filling the view of a camera at the origin looking
    down -z, and a sphere in front of it."""
    s = ptb.HostScene()
    t = s.add_texture(ptb.TEX_SOLID, (0.6, 0.5, 0.4))
    ts = s.add_texture(ptb.TEX_SOLID, (0.2, 0.7, 0.3))
    sky = s.add_texture(ptb.TEX_SOLID, (0.5, 0.6, 0.9))
    m = s.add_material(ptb.MAT_LAMBERTIAN, t, 1.0)
    ms = s.add_material(ptb.MAT_LAMBERTIAN, ts, 1.0)
    if sphere:
        s.add_sphere((0.4, -0.2, -depth * 0.6), 0.5, ms)
    tri = np.zeros(2, ptb._lib.triangle_dtype)
    a, z = 100.0, -depth
    tri[0]["p"] = [(-a, -a, z), (a, -a, z), (a, a, z)]
    tri[1]["p"] = [(-a, -a, z), (a, a, z), (-a, a, z)]
    tri["n"] = (0, 0, 1)
    tri["material"] = m
    s.triangles = tri
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 60.0)
    s.set_sky(sky, (0, 0))
    return s


def moved_camera(scene, shift):
    """A copy of `scene` whose whole camera (origin and image plane) is translated by `shift`."""
    import copy
    s = copy.deepcopy(scene)
    for k in ("origin", "lower_left"):
        s.camera[k] = s.camera[k] + np.float32(shift)
    return s


def noisy_sums(seed, h=36, w=52):
    rng = np.random.default_rng(seed)
    _, n, z, a, irr = quadrants(h, w)
    c = (irr[..., None] * a * rng.uniform(0.3, 1.7, (h, w, 3))).astype(np.float32)
    b, aov, s_b, s_a = make_sums(c, a, n, z, np.ones((h, w), np.float32))
    mot = np.zeros((h, w, 4), np.float32)
    mot[..., 0:2] = rng.uniform(-3, 3, (h, w, 2))
    mot[..., 2] = z
    mot[..., 3] = 1
    return b, aov, mot, s_b, s_a


@pytest.mark.parametrize("opts", [{}, {"iterations": 1}, {"iterations": 2, "sigma_luminance": 2.0},
                                  {"iterations": 10, "sigma_normal": 32.0, "sigma_depth": 0.25}])
def test_no_history_is_the_spatial_filter_bit_for_bit(opts):
    b, aov, mot, s_b, s_a = noisy_sums(1)
    want = denoise(b, aov, s_b, s_a, **opts)
    got, hist = denoise_temporal(b, aov, mot, s_b, s_a, None, **opts)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.all(hist["m"][..., 2] == 1)
    # a history all of whose taps are rejected (no coverage there) changes nothing either
    h2 = dict(hist, alpha=np.zeros_like(hist["alpha"]))
    got2, hist2 = denoise_temporal(b, aov, mot, s_b, s_a, h2, alpha_color=0.5, **opts)
    assert np.array_equal(got2.view(np.uint32), want.view(np.uint32))
    assert np.all(hist2["m"][..., 2] == 1)


def test_static_history_accumulates_and_lowers_the_noise():
    """Zero motion over a static image: the history length grows to the cap and the output's error against the clean
    image falls below the spatial filter's on the same frame."""
    h, w = 36, 52
    _, n, z, a, irr = quadrants(h, w)
    clean = (irr[..., None] * a).astype(np.float32)
    hist, errs = None, []
    for f in range(8):
        b, aov, mot, s_b, s_a = noisy_sums(10 + f, h, w)
        mot[..., 0:2] = 0
        out, hist = denoise_temporal(b, aov, mot, s_b, s_a, hist, max_history=6)
        errs.append((float(np.mean((out - clean) ** 2)), float(np.mean((denoise(b, aov, s_b, s_a) - clean) ** 2))))
    assert np.all(hist["m"][..., 2] == 6)
    assert errs[-1][0] < errs[-1][1], errs


def test_static_frame_has_zero_motion(ptb, rtweekend1):
    w, h, spp = 48, 27, 3
    mo = MotionOracle(rtweekend1)
    sums = mo.render_motion(rtweekend1, w, h, spp, seed=4)
    assert np.all(sums[..., 0:2] == 0)
    aov, _ = AovOracle(rtweekend1).render_aov(w, h, spp, seed=4)
    assert np.array_equal(sums[..., 3], aov[..., 3])  # every hit counts: the marked camera sees it in front
    depth = split(aov, spp)["depth"]
    t = mean(sums)[..., 2]
    assert np.all(np.abs(t - depth) <= 1e-5 * depth)


def test_sideways_camera_translation_gives_the_analytic_dx(ptb):
    """Camera moved by +s along its image-plane x between the marked frame and now, in front of a plane perpendicular to
    the view at distance D: every plane point moves by Δx = s * f * (W - 1) / (D * |h|) pixels (f: the image plane's
    distance along the view), and Δy = 0."""
    D, s, w, h = 5.0, 0.3, 64, 36
    scene = plane_scene(ptb, D, sphere=False)
    cam = scene.camera[0]
    hz = cam["horizontal"].astype(np.float64)
    prev = moved_camera(scene, -s * hz / np.linalg.norm(hz))
    sums = MotionOracle(scene).render_motion(prev, w, h, 2, seed=1)
    m = mean(sums)
    assert np.all(sums[..., 3] == 2)
    f = -(cam["lower_left"].astype(np.float64) - cam["origin"])[2]
    want = s * f * (w - 1) / (D * np.linalg.norm(hz))
    assert np.allclose(m[..., 0], want, rtol=1e-4, atol=1e-4), (float(m[..., 0].min()), float(m[..., 0].max()), want)
    assert np.all(np.abs(m[..., 1]) <= 1e-4)
    assert np.all(m[..., 2] >= D * (1 - 1e-6))  # t' = |P' - o'| along the marked camera's rays
