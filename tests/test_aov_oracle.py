"""CPU: the oracle's denoiser feature buffers (oracle/aov_api.cpp), which the device's ptb_render_aov is compared against,
agree with the oracle's own closest hit on its camera rays, with the furnace scene's known albedo, and clamp a bright
sky."""
import numpy as np

from aov_oracle import AovOracle, split
from conftest import furnace_scene

MISS = 0xFFFFFFFF


def camera_rays(ptb, orc, scene, width, height, seed, sample, rows=None):
    """The camera ray of (pixel, sample) for every pixel of `rows` (default: all), rebuilt on the host as the reference's
    sample_pixel forms it (random_sampler.rs:50-61, camera.rs:57-63): jitter from Philox (pixel, sample, RNG_JITTER), the
    un-normalised direction lower_left + horizontal * u + vertical * v - origin in f32. Each direction's normalisation is
    checked against orc.OracleScene.camera_ray. Returns ray records (ray_dtype) in row-major pixel order."""
    o = orc.OracleScene(scene, split_type=-1)
    cam = scene.camera[0]
    f = np.float32
    origin, ll, hor, ver = (np.asarray(cam[k], np.float32) for k in ("origin", "lower_left", "horizontal", "vertical"))
    rows = range(height) if rows is None else rows
    out = np.zeros(len(rows) * width, ptb.ray_dtype)
    k = 0
    for y in rows:
        for x in range(width):
            r = orc.philox([y * width + x, sample, 0, 0], [seed & 0xFFFFFFFF, seed >> 32])
            u = (f(r[0] >> 8) * f(1.0 / 16777216.0) + f(x)) / f(width - 1)
            v = f(1) - (f(r[1] >> 8) * f(1.0 / 16777216.0) + f(y)) / f(height - 1)
            d = ll + hor * u + ver * v - origin
            n = d / np.sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2])
            o_ref, d_ref = o.camera_ray(u, v)
            assert np.array_equal(d_ref.view(np.uint32), n.view(np.uint32)) and np.array_equal(o_ref, origin)
            out[k]["o"], out[k]["d"] = origin, d
            k += 1
    return out


def test_depth_and_coverage_equal_closest_hit_on_camera_rays(ptb, orc, rtweekend1):
    w, h, seed = 24, 14, 0x1234_5678_9ABC
    sums, prims = AovOracle(rtweekend1).render_aov(w, h, 1, seed=seed, sample_offset=5)
    hits = orc.OracleScene(rtweekend1).closest_hit(camera_rays(ptb, orc, rtweekend1, w, h, seed, 5))
    assert np.array_equal(prims[:, 0], hits["prim"])
    hit = hits["prim"] != MISS
    assert 0 < hit.sum() < hit.size  # both cases occur
    assert np.array_equal(sums[..., 3].reshape(-1), hit.astype(np.float32))
    assert np.array_equal(sums[..., 7].reshape(-1).view(np.uint32), np.where(hit, hits["t"], 0).astype(np.float32).view(np.uint32))


def test_furnace_centre_albedo_is_grey_sphere(ptb):
    s = furnace_scene(ptb)
    w = h = 33
    sums, prims = AovOracle(s).render_aov(w, h, 4, seed=3)
    c = h // 2 * w + w // 2
    assert np.all(prims[c] == 0)  # the r = 0.5 grey Lambertian sphere
    b = split(sums, 4)
    assert np.array_equal(b["albedo"][h // 2, w // 2], np.full(3, 0.5 * 0.5, np.float32))
    assert b["coverage"][h // 2, w // 2] == 1.0
    n = b["normal"][h // 2, w // 2]
    assert abs(np.linalg.norm(n) - 1) < 1e-3 and n[2] > 0.99  # facing the camera at +z
    assert abs(b["depth"][h // 2, w // 2] - 2.5) < 1e-2  # camera at z = 3, nearest sphere point at z = 0.5


def test_bright_sky_albedo_is_clamped(ptb):
    s = ptb.HostScene()
    tg = s.add_texture(ptb.TEX_SOLID, (0.5, 0.5, 0.5))
    sky = s.add_texture(ptb.TEX_SOLID, (2.0, 0.5, -1.0))
    s.add_sphere((0, 0, 0), 0.5, s.add_material(ptb.MAT_LAMBERTIAN, tg, 0.5))
    s.set_camera((0, 0, 3), (0, 0, 0), (0, 1, 0), 40)
    s.set_sky(sky, (0, 0))
    sums, prims = AovOracle(s).render_aov(16, 9, 2, seed=1)
    b = split(sums, 2)
    miss = (prims == MISS).all(axis=1).reshape(9, 16)
    assert miss[0, 0] and not miss.all()
    assert np.array_equal(b["albedo"][miss], np.tile(np.float32([1.0, 0.5, 0.0]), (int(miss.sum()), 1)))
    assert np.all(b["coverage"][miss] == 0) and np.all(b["depth"][miss] == 0) and np.all(b["normal"][miss] == 0)


def test_sample_ranges_and_row_tiles_add_up(ptb, rtweekend1):
    o = AovOracle(rtweekend1)
    w, h = 20, 12
    whole, _ = o.render_aov(w, h, 3, seed=9)
    parts, _ = o.render_aov(w, h, 1, seed=9)
    o.render_aov(w, h, 2, seed=9, sample_offset=1, sums=parts)
    assert np.array_equal(whole.view(np.uint32), parts.view(np.uint32))
    tiles = np.zeros_like(whole)
    o.render_aov(w, h, 3, seed=9, row_begin=0, row_count=5, sums=tiles)
    o.render_aov(w, h, 3, seed=9, row_begin=5, sums=tiles)
    assert np.array_equal(whole.view(np.uint32), tiles.view(np.uint32))
