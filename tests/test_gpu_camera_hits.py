"""Camera-ray hits inside a render, sample by sample, over a sweep of cameras, scenes, image shapes and trees.

Every primitive of the scenes is an emitter whose colour is a function of its id (test_camera_hits_oracle.id_coded), and
the integrator is the naive one: a camera sample's radiance is exactly the colour of its first hit, so the accumulator
of a render is a checksum of its first hits. For each configuration:
1. the lists forced on (k_cam_candidates + the list path of k_trace_camera), forced off (the packet walk) and
   PTB_CAMERA_PACKET=0 (the persistent per-lane walk) give the same ray counters and the same image: bit for bit at 32
   samples per pixel (each pixel's 32 samples are one warp, summed by shuffles and added with one atomic per channel
   into a cleared accumulator), within 1e-6 relative with more samples (several atomics per pixel, in any order);
2. each image equals the sum over the pixel's samples of the colour of closest_hit (k_trace, a separate kernel) on the
   same rays, rebuilt on the host, within 1e-6 * spp + 1e-6 per channel, far below one wrong sample's PALETTE_STEP;
3. closest_hit's primitive ids on those rays equal the oracle's closest_hit_brute, except for the rays
   test_gpu_closest_hit.degenerate excludes (quirk Q1, exact-t ties);
4. the lists were used: a counted render fetches fewer nodes with them, and the CPU statement of the lists
   (scripts/camcand_ref.py) overflows in fewer than half of the image's pixels (only reported for the scene far from the origin,
   where the margins that scale with |origin| make most pixels overflow, for shortened lists and for images of a few
   pixels, whose footprints are large; at 2 x 2 every pixel overflows and the walk answers every sample);
5. inside the watertight shell only samples in the band quirk Q1 affects reach the sky, and the oracle agrees on them."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "scripts"))
import camcand_ref  # noqa: E402

from test_camera_hits_oracle import (C3_SWEEP, MISS, PALETTE_STEP, axis_cameras, c3, camera_rays_np, colours,  # noqa: E402
                                     hard_geometry, id_coded, in_leaf_camera, moved, q1_band, shell, spheres_and_ground,
                                     with_camera)
from test_gpu_closest_hit import degenerate  # noqa: E402

pytestmark = pytest.mark.gpu

SEED = 0x5EED_CA3E_0001
BRUTE_RAYS = 40000  # rays per configuration checked against closest_hit_brute (a fixed subsample above that)


def tolerance(spp):
    return 1e-6 * spp + 1e-6


def test_one_wrong_sample_is_visible():
    """The tolerance of assertion 2 at the largest spp used stays far below one wrong sample's change of a pixel sum."""
    assert PALETTE_STEP >= 0.05 and tolerance(96) < PALETTE_STEP / 100


def counters(st):
    return (st.rays_camera, st.rays_bounce, st.rays_shadow_light, st.rays_shadow_sky, st.rays_reference, st.paths,
            st.rays_total)


def _env(monkeypatch, env):
    for k in ("PTB_CAMERA_CAND", "PTB_CAMERA_PACKET", "PTB_CAMERA_CAND_K"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, str(v))


def render(ptb, ctx, o, monkeypatch, env, count=False):
    _env(monkeypatch, env)
    if count:
        ctx.set_option(ptb._lib.OPT_COUNT_TRAVERSAL, 1)
    try:
        ctx.accum_clear()
        ctx.stats_reset()
        ctx.render(o)
        st = ctx.stats()
        img = ctx.accum_read(o.width, o.height, normalise=False).copy()
    finally:
        if count:
            ctx.set_option(ptb._lib.OPT_COUNT_TRAVERSAL, 0)
        _env(monkeypatch, {})
    return img, counters(st), st.kernel_launches, st.nodes_fetched


def check(ptb, orc, ctx, scene, monkeypatch, W=33, H=17, spp=32, sample_offset=0, row_begin=0, row_count=0, k=None,
          build=None, refit=None, far_scene=False, watertight=False):
    """Assertions 1-5 of the module docstring for one configuration; returns what the report needs."""
    build = ptb._lib.BUILD_SAH if build is None else build
    ctx.upload(scene)
    ctx.commit(build)
    if refit is not None:  # the same counts, moved: keep the tree, refit its boxes
        ctx.update_triangles(0, refit.triangles)
        ctx.commit(ptb._lib.BUILD_REFIT)
        scene = refit
    wide = build == ptb._lib.BUILD_WIDE
    o = ptb.RenderOptions(samples_per_pixel=spp, render_method=ptb.METHOD_NAIVE, width=W, height=H, seed=SEED,
                          sample_offset=sample_offset, row_begin=row_begin, row_count=row_count)
    kenv = {} if k is None else {"PTB_CAMERA_CAND_K": k}
    on, off, lane = (render(ptb, ctx, o, monkeypatch, dict(kenv, **e))
                     for e in ({"PTB_CAMERA_CAND": 1}, {"PTB_CAMERA_CAND": 0}, {"PTB_CAMERA_PACKET": 0}))
    rows = np.arange(row_begin, row_begin + (row_count or H - row_begin))
    # 1. the three walks agree
    assert on[1] == off[1] == lane[1], (on[1], off[1], lane[1])
    assert on[1][0] == W * len(rows) * spp
    for other in (off, lane):
        if spp == 32:
            assert np.array_equal(on[0].view(np.uint32), other[0].view(np.uint32))
        else:
            assert np.allclose(on[0], other[0], rtol=1e-6, atol=0), float(np.abs(on[0] - other[0]).max())
    assert on[2] == off[2] + (0 if wide else 1)  # k_cam_candidates runs, except on the wide tree
    # 2. the image is the checksum of closest_hit on the same rays
    rays = camera_rays_np(ptb, scene, W, H, SEED, np.arange(sample_offset, sample_offset + spp), rows=rows).reshape(-1)
    g = ctx.closest_hit(rays)
    expected = colours(g["prim"]).reshape(len(rows), W, spp, 3).sum(axis=2)
    tol = tolerance(spp)
    for img in (on[0], off[0], lane[0]):
        assert np.all(img[:row_begin] == 0) and np.all(img[rows[-1] + 1:] == 0)
        err = np.abs(img[rows].astype(np.float64) - expected)
        assert err.max() <= tol, (float(err.max()), np.unravel_index(int(err.argmax()), err.shape))
    # 3. closest_hit against the oracle's test-all closest hit
    pick = np.arange(len(rays))
    if len(rays) > BRUTE_RAYS:
        pick = np.sort(np.random.default_rng(1).choice(len(rays), BRUTE_RAYS, replace=False))
    r = orc.OracleScene(scene).closest_hit_brute(rays[pick])
    excl = degenerate(rays[pick], g[pick], r)
    same = g["prim"][pick] == r["prim"]
    assert np.all(same[~excl]), int((~same & ~excl).sum())
    # 4. the lists were used
    rep = {"q1_excluded": int(excl.sum()), "bit_exact": [bool(np.array_equal(on[0].view(np.uint32), x[0].view(np.uint32)))
                                                         for x in (off, lane)]}
    if not wide:
        L = camcand_ref.CamCandScene(scene).lists(W, H, k or 16, row_begin=row_begin, rows=len(rows))
        rep["overflow"] = float(L.overflowed.mean())
        # a listed ray fetches no node, while the beam walk costs each pixel about one packet walk: on a small tile that
        # fixed cost hides the saving unless the pixels take more samples (8x: the same rays and more)
        oc = o if W * len(rows) >= 33 * 17 else ptb.RenderOptions(**{**o.__dict__, "samples_per_pixel": 8 * spp})
        cnt_on = render(ptb, ctx, oc, monkeypatch, dict(kenv, PTB_CAMERA_CAND=1), count=True)
        cnt_off = render(ptb, ctx, oc, monkeypatch, dict(kenv, PTB_CAMERA_CAND=0), count=True)
        assert cnt_on[1] == cnt_off[1]
        if rep["overflow"] < 1.0:  # tiny images (2 x 2): every pixel's footprint overflows, all samples take the walk
            assert cnt_on[3] < cnt_off[3], (cnt_on[3], cnt_off[3])
        if not far_scene and k is None and W * H >= 33 * 5:
            # over the whole image: a tile of a few rows can lie where most pixels see many leaves (the 7 middle rows
            # of C3's camera at 33 x 17 overflow in 51 % of their pixels); the counted render above proves the tile's
            # own rays took the lists
            full = L if len(rows) == H else camcand_ref.CamCandScene(scene).lists(W, H, 16)
            rep["overflow_image"] = float(full.overflowed.mean())
            assert rep["overflow_image"] < 0.5, rep
    # 5. inside a watertight shell, only Q1 lets a sample through to the sky
    if watertight:
        sky = g["prim"] == MISS
        assert np.all(q1_band(rays[sky]))
        rb = orc.OracleScene(scene).closest_hit_brute(rays[sky])
        assert np.all(rb["prim"] == MISS)
        rep["sky_samples_q1"] = int(sky.sum())
    print(rep)
    return rep


@pytest.fixture(scope="module")
def c3_small(ptb):
    return c3(ptb, 0.05)


@pytest.mark.parametrize("scale", [0.05, 0.25])
def test_c3(ptb, orc, gpu_ctx, monkeypatch, scale):
    check(ptb, orc, gpu_ctx, c3(ptb, scale), monkeypatch, W=64, H=36)


@pytest.mark.parametrize("cam", sorted(C3_SWEEP) + ["in_leaf"])
def test_c3_camera_sweep(ptb, orc, gpu_ctx, monkeypatch, c3_small, cam):
    s = with_camera(c3_small, in_leaf_camera(c3_small) if cam == "in_leaf" else C3_SWEEP[cam])
    check(ptb, orc, gpu_ctx, s, monkeypatch)


def test_aperture_changes_nothing(ptb, gpu_ctx, monkeypatch, c3_small):
    """The device camera is a pinhole: a lens radius given to set_camera leaves the camera record and the image alone."""
    pin, lens = with_camera(c3_small, C3_SWEEP["aperture"][:5] + (0.0, 3.0)), with_camera(c3_small, C3_SWEEP["aperture"])
    assert pin.camera.tobytes() == lens.camera.tobytes()


@pytest.mark.parametrize("cfg", [
    dict(W=2, H=2), dict(W=157, H=91), dict(W=33, H=17, row_begin=5, row_count=7), dict(W=157, H=91, row_begin=40, row_count=9),
    dict(sample_offset=96), dict(spp=96), dict(spp=96, sample_offset=17), dict(k=1), dict(k=3), dict(k=16)])
@pytest.mark.parametrize("cam", ["c3", "-z", "+x"])
def test_image_and_call_parameters(ptb, orc, gpu_ctx, monkeypatch, c3_small, cfg, cam):
    check(ptb, orc, gpu_ctx, with_camera(c3_small, C3_SWEEP[cam]), monkeypatch, **cfg)


@pytest.mark.parametrize("shift,scale", [((1e4, -3e3, 5e3), 1.0), ((0.0, 0.0, 0.0), 1e-3), ((0.0, 0.0, 0.0), 1e3)])
@pytest.mark.parametrize("cam", ["c3", "-z", "fov0.5"])
def test_moved_and_scaled(ptb, orc, gpu_ctx, monkeypatch, c3_small, shift, scale, cam):
    far = shift != (0.0, 0.0, 0.0)
    rep = check(ptb, orc, gpu_ctx, with_camera(moved(ptb, c3_small, shift, scale), C3_SWEEP[cam]), monkeypatch, far_scene=far)
    print(f"overflow fraction {rep['overflow']:.2f} at shift {shift}, scale {scale}")


def _scene_cams(scene):
    return [("own", scene)] + [(k, with_camera(scene, c)) for k, c in axis_cameras(scene.camera[0]["origin"]).items()]


@pytest.fixture(scope="module")
def extra_scenes(ptb):
    return {"shell": shell(ptb), "spheres_and_ground": spheres_and_ground(ptb), "hard_geometry": hard_geometry(ptb)}


@pytest.mark.parametrize("name", ["shell", "spheres_and_ground", "hard_geometry"])
def test_scenes(ptb, orc, gpu_ctx, monkeypatch, extra_scenes, name):
    """(b) the watertight shell, (c) spheres over a triangle ground with a radius-1000 sphere, (e) duplicates, zero-area
    triangles, slivers seen edge-on and planes through the apex (fewer than 4096 primitives: the lists are forced)."""
    for cam, s in _scene_cams(extra_scenes[name]):
        for W, H in ((65, 33), (9, 5)):
            print(name, cam, W, H)
            check(ptb, orc, gpu_ctx, s, monkeypatch, W=W, H=H, watertight=name == "shell")


@pytest.mark.parametrize("cam", ["c3", "-z", "+y"])
def test_lbvh(ptb, orc, gpu_ctx, monkeypatch, c3_small, cam):
    check(ptb, orc, gpu_ctx, with_camera(c3_small, C3_SWEEP[cam]), monkeypatch, build=ptb._lib.BUILD_BINARY)


@pytest.mark.parametrize("build", ["sah", "lbvh"])
def test_refit(ptb, orc, gpu_ctx, monkeypatch, build):
    base = c3(ptb, 0.25)
    new = id_coded(ptb, ptb.meshgen.c3_deform(ptb.meshgen.c3_scene(0.25), 0.5, 1.0))
    b = ptb._lib.BUILD_SAH if build == "sah" else ptb._lib.BUILD_BINARY
    check(ptb, orc, gpu_ctx, base, monkeypatch, W=64, H=36, build=b, refit=new)


def test_wide_tree_takes_no_lists(ptb, orc, gpu_ctx, monkeypatch, c3_small):
    """The wide tree has no packet walk and so no list path: forcing the lists adds no launch, the image still holds."""
    check(ptb, orc, gpu_ctx, c3(ptb, 0.25), monkeypatch, W=64, H=36, build=ptb._lib.BUILD_WIDE)
    check(ptb, orc, gpu_ctx, with_camera(c3_small, C3_SWEEP["-z"]), monkeypatch, build=ptb._lib.BUILD_WIDE)
