"""GPU: motion vectors (ptb_motion_mark, the motion sums of ptb_render_aov, ptb_motion_read): exactly zero on a static
frame with t' equal to the depth AOV, the device against the oracle (oracle/motion_api.cpp) for a moved camera, a moved
instance and a moved sphere, static background exactly zero when only an object moves, split invariance, a mark of other
counts, and the error rules."""
import copy

import numpy as np
import pytest

from aov_oracle import AovOracle
from motion_oracle import MotionOracle, mean
from test_gpu_aov import sums
from test_temporal_oracle import moved_camera, plane_scene

pytestmark = pytest.mark.gpu


def opts(ptb, w, h, spp, seed=3, offset=0, **kw):
    return ptb.RenderOptions(samples_per_pixel=spp, width=w, height=h, seed=seed, sample_offset=offset, **kw)


def aov_frame(ctx, o):
    ctx.aov_clear()
    ctx.render_aov(o)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("which", ["rtweekend1", "c3_small", "plane"])
def test_static_frame_is_exactly_zero(ptb, gpu_ctx, rtweekend1, which):
    scene = {"rtweekend1": lambda: rtweekend1, "c3_small": lambda: ptb.meshgen.c3_scene(0.05),
             "plane": lambda: plane_scene(ptb)}[which]()
    gpu_ctx.upload(scene)
    gpu_ctx.commit()
    gpu_ctx.motion_mark()
    w, h, spp = 96, 54, 4
    aov_frame(gpu_ctx, opts(ptb, w, h, spp))
    m = gpu_ctx.motion_read(w, h)
    assert np.all(m[..., 0:2] == 0)
    depth = gpu_ctx.aov_read(w, h, ptb.PTB_AOV_DEPTH)
    cov = gpu_ctx.aov_read(w, h, ptb.PTB_AOV_COVERAGE)
    assert np.array_equal(m[..., 2] > 0, cov > 0)
    assert np.all(np.abs(m[..., 2] - depth) <= 1e-5 * depth)


def same_hits_mask(ptb, ctx, scene, w, h, spp, seed):
    """Pixels whose AOV sums are bit-identical on device and oracle: the same hit, sample by sample."""
    a, _ = AovOracle(scene).render_aov(w, h, spp, seed=seed)
    return np.all(bits(sums(ptb, ctx, w, h)) == bits(a), axis=-1)


def compare(ptb, ctx, cur, prev, w, h, spp, seed):
    """Device motion against the oracle's on the pixels with the same hits. Both evaluate the same expressions without
    contraction on bit-identical hit records, so they agree to a few ulps of the projection's divisions:
    |d - o| <= 1e-4 |o| + 1e-4 pixels (t' alike)."""
    d = ctx.motion_read(w, h)
    o = mean(MotionOracle(cur).render_motion(prev, w, h, spp, seed=seed))
    same = same_hits_mask(ptb, ctx, cur, w, h, spp, seed)
    assert same.mean() > 0.95, same.mean()
    err = np.abs(d - o) - 1e-4 * np.abs(o)
    assert np.all(err[same] <= 1e-4), float(err[same].max())
    return d, o


def test_camera_moved(ptb, gpu_ctx, rtweekend1):
    w, h, spp, seed = 96, 54, 3, 7
    prev = rtweekend1
    cur = moved_camera(rtweekend1, (0.15, -0.05, 0.1))
    gpu_ctx.upload(prev)
    gpu_ctx.commit()
    gpu_ctx.motion_mark()
    gpu_ctx.upload(cur)  # a full rebuild with the same counts keeps the primitive ids
    gpu_ctx.commit()
    aov_frame(gpu_ctx, opts(ptb, w, h, spp, seed))
    d, o = compare(ptb, gpu_ctx, cur, prev, w, h, spp, seed)
    assert np.abs(d[..., 0]).max() > 1.0  # the camera did move


def test_sphere_moved_background_stays_zero(ptb, gpu_ctx):
    L = ptb._lib
    w, h, spp, seed = 96, 54, 4, 2
    prev = plane_scene(ptb)
    cur = copy.deepcopy(prev)
    cur.spheres["center"][0] += np.float32([0.6, 0.2, -0.3])
    cur.spheres["radius"][0] *= np.float32(1.2)
    gpu_ctx.upload(prev)
    gpu_ctx.commit()
    gpu_ctx.motion_mark()
    gpu_ctx.update_spheres(0, cur.spheres)
    gpu_ctx.commit(L.BUILD_REFIT)
    aov_frame(gpu_ctx, opts(ptb, w, h, spp, seed))
    d, o = compare(ptb, gpu_ctx, cur, prev, w, h, spp, seed)
    # pixels whose samples all hit the static plane (ids 1, 2) move by exactly 0
    _, prims = AovOracle(cur).render_aov(w, h, spp, seed=seed)
    plane = np.all((prims >= 1) & (prims != ptb.PTB_MISS), axis=1).reshape(h, w) & same_hits_mask(ptb, gpu_ctx, cur, w, h, spp, seed)
    assert plane.mean() > 0.5 and np.all(d[plane][:, 0:2] == 0)
    assert np.abs(d[~plane][:, 0:2]).max() > 0.5  # the sphere's pixels moved


def test_instance_moved(ptb, gpu_ctx):
    L = ptb._lib
    w, h, spp, seed = 96, 54, 2, 5
    scene, mesh, inst, xf = ptb.meshgen.c3_instanced(0.05)
    xf2 = xf.copy()
    xf2[1] = ptb.meshgen.c3_instanced_frame(1.5)
    gpu_ctx.upload(scene, mesh=mesh, instances=(inst, xf))
    gpu_ctx.commit()
    gpu_ctx.motion_mark()
    gpu_ctx.update_instance_xforms(1, xf2[1:2])
    gpu_ctx.commit(L.BUILD_REFIT)
    aov_frame(gpu_ctx, opts(ptb, w, h, spp, seed))
    prev, cur = copy.deepcopy(scene), copy.deepcopy(scene)
    prev.triangles = mesh.expand_instances(inst, xf)
    cur.triangles = mesh.expand_instances(inst, xf2)
    d, _ = compare(ptb, gpu_ctx, cur, prev, w, h, spp, seed)
    assert np.abs(d[..., 0:2]).max() > 0.5
    # terrain pixels (the first instance does not move, nor does the camera) stay exactly 0
    _, prims = AovOracle(cur).render_aov(w, h, spp, seed=seed)
    ns = len(scene.spheres)
    terrain = np.all((prims >= ns) & (prims < ns + int(inst[0]["n_triangles"])), axis=1).reshape(h, w)
    assert terrain.mean() > 0.3 and np.all(d[terrain][:, 0:2] == 0)


def test_split_invariance_counts_and_errors(ptb, dctx, rtweekend1):
    L = ptb._lib
    with pytest.raises(ptb.PtbError, match="scene not committed"):
        dctx.motion_mark()
    with pytest.raises(ptb.PtbError, match="no AOV rendered yet"):
        dctx.motion_read(16, 16)
    w, h = 64, 36
    cur = moved_camera(rtweekend1, (0.1, 0.0, 0.05))
    dctx.upload(rtweekend1)
    dctx.commit()
    dctx.motion_mark()
    dctx.upload(cur)
    dctx.commit()
    aov_frame(dctx, opts(ptb, w, h, 4))
    whole = dctx.motion_read(w, h).copy()
    dctx.aov_clear()
    dctx.render_aov(opts(ptb, w, h, 2))
    dctx.render_aov(opts(ptb, w, h, 2, offset=2))
    assert np.array_equal(bits(dctx.motion_read(w, h)), bits(whole))
    dctx.aov_clear()
    for r0, rc in ((0, 10), (10, 26)):
        dctx.render_aov(opts(ptb, w, h, 4, row_begin=r0, row_count=rc))
    assert np.array_equal(bits(dctx.motion_read(w, h)), bits(whole))
    # a size change reallocates and zeroes the motion sums with the AOV sums
    aov_frame(dctx, opts(ptb, 32, 18, 1))
    assert dctx.motion_read(32, 18).shape == (18, 32, 3)
    # read errors
    buf = np.zeros(32 * 18 * 3, np.float32)
    for p, n in ((None, buf.size), (L.ptr(buf), buf.size - 1)):
        assert L.lib.ptb_motion_read(dctx._h, p, n) == 1 and b"motion_read expects 1728 floats" in L.lib.ptb_last_error(dctx._h)
    assert L.lib.ptb_motion_read(None, L.ptr(buf), buf.size) == 1 and L.lib.ptb_motion_mark(None) == 1
    # a mark whose counts differ from the committed scene's: no valid samples, no error
    s2 = copy.deepcopy(cur)
    s2.add_sphere((0, 100, 0), 0.1, 0)
    dctx.upload(s2)
    dctx.commit()
    aov_frame(dctx, opts(ptb, w, h, 2))
    assert np.all(dctx.motion_read(w, h) == 0)
    assert dctx.aov_read(w, h, ptb.PTB_AOV_COVERAGE).max() > 0


@pytest.fixture()
def dctx(ptb):
    c = ptb.Context(0)
    yield c
    c.close()
