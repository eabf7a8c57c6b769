"""Camera samples answered from per-pixel candidate lists (ptb_camcand.cuh: k_cam_candidates + the list path of
k_trace_camera) against the packet walk: PTB_CAMERA_CAND forced off and on, same ray counters and the same image (the
image is a function of the hits, which the list path must reproduce bit for bit; the tolerance is that of
test_camera_packets_are_the_same_rays)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H = 160, 96


def counters(st):
    return (st.rays_camera, st.rays_bounce, st.rays_shadow_light, st.rays_shadow_sky, st.rays_reference, st.paths,
            st.rays_total)


def render_pair(ctx, opts, monkeypatch, k=None):
    """Render twice, lists off then on (k: PTB_CAMERA_CAND_K): same counters, same image, one launch more."""
    if k is not None:
        monkeypatch.setenv("PTB_CAMERA_CAND_K", str(k))
    out = []
    for cand in ("0", "1"):
        monkeypatch.setenv("PTB_CAMERA_CAND", cand)
        ctx.accum_clear()
        ctx.stats_reset()
        ctx.render(opts)
        st = ctx.stats()
        out.append((ctx.accum_read(opts.width, opts.height).copy(), counters(st), st.kernel_launches))
    monkeypatch.delenv("PTB_CAMERA_CAND")
    if k is not None:
        monkeypatch.delenv("PTB_CAMERA_CAND_K")
    (a, ca, la), (b, cb, lb) = out
    assert ca == cb, (ca, cb)
    assert np.allclose(a, b, rtol=1e-5, atol=1e-5), float(np.abs(a - b).max())
    assert lb == la + 1  # k_cam_candidates: one launch per call
    assert a.max() > 0


def opts(ptb, **kw):
    base = dict(samples_per_pixel=64, render_method=0, width=W, height=H, seed=7)
    base.update(kw)
    return ptb.RenderOptions(**base)


@pytest.mark.parametrize("scale", [0.05, 0.25])
@pytest.mark.parametrize("method", [0, 1])
def test_c3(ptb, gpu_ctx, scale, method, monkeypatch):
    gpu_ctx.upload(ptb.meshgen.c3_scene(scale))
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    render_pair(gpu_ctx, opts(ptb, render_method=method), monkeypatch)


def test_odd_image_tile_and_sample_offset(ptb, gpu_ctx, monkeypatch):
    gpu_ctx.upload(ptb.meshgen.c3_scene(0.25))
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    render_pair(gpu_ctx, opts(ptb, width=157, height=91), monkeypatch)
    render_pair(gpu_ctx, opts(ptb, row_begin=37, row_count=29), monkeypatch)
    render_pair(gpu_ctx, opts(ptb, samples_per_pixel=32, sample_offset=96), monkeypatch)


def test_overflow_falls_back_to_the_packet_walk(ptb, gpu_ctx, monkeypatch):
    gpu_ctx.upload(ptb.meshgen.c3_scene(0.25))
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    for k in (1, 3):
        render_pair(gpu_ctx, opts(ptb), monkeypatch, k=k)


def test_mesh_and_instances(ptb, gpu_ctx, monkeypatch):
    scene, mesh = ptb.meshgen.c3_indexed(0.25)
    gpu_ctx.upload(scene, mesh=mesh)
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    render_pair(gpu_ctx, opts(ptb), monkeypatch)
    scene, mesh, inst, xf = ptb.meshgen.c3_instanced(0.25)
    gpu_ctx.upload(scene, mesh=mesh, instances=(inst, xf))
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    render_pair(gpu_ctx, opts(ptb), monkeypatch)


def test_deformed_and_refitted(ptb, gpu_ctx, monkeypatch):
    base = ptb.meshgen.c3_scene(0.25)
    new = ptb.meshgen.c3_deform(base, 0.5, 1.0)
    gpu_ctx.upload(base)
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    gpu_ctx.update_triangles(0, new.triangles)
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    render_pair(gpu_ctx, opts(ptb), monkeypatch)


def test_default_choice(ptb, gpu_ctx, monkeypatch):
    """Lists by default on C3 at 62 500 triangles; not below 4096 primitives, nor with fewer than 32 samples per pixel."""
    launches = {}
    for scale in (0.05, 0.25):
        gpu_ctx.upload(ptb.meshgen.c3_scene(scale))
        gpu_ctx.commit(ptb._lib.BUILD_SAH)
        for name, spp in (("32", 32), ("4", 4)):
            runs = []
            for env in ("0", None):
                if env is None:
                    monkeypatch.delenv("PTB_CAMERA_CAND", raising=False)
                else:
                    monkeypatch.setenv("PTB_CAMERA_CAND", env)
                gpu_ctx.stats_reset()
                gpu_ctx.render(opts(ptb, samples_per_pixel=spp))
                runs.append(gpu_ctx.stats().kernel_launches)
            launches[(scale, name)] = runs[1] - runs[0]
    monkeypatch.delenv("PTB_CAMERA_CAND", raising=False)
    assert launches == {(0.05, "32"): 0, (0.05, "4"): 0, (0.25, "32"): 1, (0.25, "4"): 0}, launches


def test_counted_render_takes_the_list_path(ptb, gpu_ctx, monkeypatch):
    """Traversal statistics prove that warps were answered from lists: with them, a camera ray costs no node visits (the
    beam walk's are counted once per pixel), so far fewer nodes are fetched for the same rays, hits and image."""
    gpu_ctx.upload(ptb.meshgen.c3_scene(0.25))
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    o = opts(ptb)
    gpu_ctx.set_option(ptb._lib.OPT_COUNT_TRAVERSAL, 1)
    try:
        res = {}
        for cand in ("0", "1"):
            monkeypatch.setenv("PTB_CAMERA_CAND", cand)
            gpu_ctx.accum_clear()
            gpu_ctx.stats_reset()
            gpu_ctx.render(o)
            st = gpu_ctx.stats()
            res[cand] = (gpu_ctx.accum_read(W, H).copy(), counters(st), st.rays_counted, st.nodes_fetched, st.prims_tested)
    finally:
        gpu_ctx.set_option(ptb._lib.OPT_COUNT_TRAVERSAL, 0)
        monkeypatch.delenv("PTB_CAMERA_CAND", raising=False)
    (a, ca, ra, na, pa), (b, cb, rb, nb, pb) = res["0"], res["1"]
    assert ca == cb and ra == rb
    assert np.allclose(a, b, rtol=1e-5, atol=1e-5)
    camera_rays = ca[0]
    # the packet walk fetches well over 10 nodes per camera ray on this scene; the lists save most of them
    assert na - nb > 3 * camera_rays, (na, nb, camera_rays)
    assert pb > 0
