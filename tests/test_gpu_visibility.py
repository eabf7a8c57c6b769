"""Batch visibility through the C ABI (ptb_check_hit_index / ptb_occluded: k_visibility_api, the any-hit walk k_shadow
runs) against the oracle's check_hit_index / occlusion query (oracle/visibility_api.cpp, reference semantics: SAH tree + BFS
candidates + blocker scan), and
against the device's own closest hit at full size."""
import copy

import numpy as np
import pytest

from conftest import random_rays
from test_gpu_closest_hit import degenerate
from test_visibility_oracle import MISS, occlusion_rays, target_rays, target_t
from visibility_oracle import VisibilityOracle

pytestmark = pytest.mark.gpu


def commit(ctx, scene, flags=0):
    ctx.upload(scene)
    ctx.commit(flags)


def same_bits(a, b):
    return all(np.array_equal(a[f].view(np.uint32), b[f].view(np.uint32)) for f in ("t", "prim", "u", "v"))


@pytest.fixture(scope="module")
def c3_full(ptb):
    return ptb.meshgen.c3_scene(1.0)


@pytest.fixture(scope="module")
def c5_full(ptb):
    return ptb.meshgen.heightfield_scene(2500, 2000)


def _scene(ptb, request, name):
    if name.startswith("c3_"):
        return ptb.meshgen.c3_scene(float(name[3:]))
    return request.getfixturevalue(name)


SCENES = [("rtweekend1", (0, 1, 0), 3.0), ("overshadowed", (-0.3, 0.3, -0.3), 1.5), ("c3_0.03", (0, 4, 1), 4.0),
          ("c3_0.1", (0, 4, 1), 4.0)]


@pytest.mark.parametrize("name,centre,radius", SCENES)
def test_check_hit_index_vs_oracle(ptb, orc, gpu_ctx, request, name, centre, radius):
    s = _scene(ptb, request, name)
    commit(gpu_ctx, s)
    rays, ids = target_rays(ptb, s, 60_000, 21, centre=centre, radius=radius)
    g = gpu_ctx.check_hit_index(rays, ids)
    r = VisibilityOracle(s).check_hit_index(rays, ids)
    c = orc.OracleScene(s).closest_hit(rays)
    # exact-t ties between the target and a blocker: the target's t (whichever side saw it) equals the closest hit's
    t_vis = np.where(g["prim"] != MISS, g["t"], r["t"])
    tie = (c["t"] == t_vis) & (c["prim"] != ids) & (t_vis > 0)
    ok = ~(degenerate(rays, c, c) | tie)
    gv, rv = g["prim"][ok] != MISS, r["prim"][ok] != MISS
    assert np.array_equal(gv, rv), f"{int((gv != rv).sum())} visibility mismatches on {int(ok.sum())} rays"
    assert same_bits(g[ok], r[ok])
    vis = g["prim"] != MISS
    assert np.array_equal(g["prim"][vis], ids[vis])
    assert np.all(g["t"][~vis] == 0) and np.all(g["u"][~vis] == 0) and np.all(g["v"][~vis] == 0)
    missed = np.isnan(target_t(ptb, s, rays, ids))
    blocked = ~vis & ~missed
    assert vis.mean() > 0.1 and blocked.mean() > 0.05 and missed.mean() > 0.2, (vis.mean(), blocked.mean(), missed.mean())


@pytest.mark.parametrize("name,centre,radius", SCENES)
def test_occluded_vs_oracle(ptb, orc, gpu_ctx, request, name, centre, radius):
    s = _scene(ptb, request, name)
    commit(gpu_ctx, s)
    rays = random_rays(ptb, 60_000, 22, centre=centre, radius=radius)
    c = orc.OracleScene(s).closest_hit(rays)
    rng = np.random.default_rng(5)
    n = len(rays)
    tmax = np.choose(rng.integers(0, 5, n), [np.full(n, np.inf), rng.uniform(0, 2 * radius, n), np.zeros(n),
                                            -rng.uniform(0, 1, n), np.full(n, np.nan)]).astype(np.float32)
    exclude = np.choose(rng.integers(0, 4, n), [np.full(n, MISS, np.int64), rng.integers(0, s.n_primitives, n),
                                                c["prim"].astype(np.int64), s.n_primitives + rng.integers(0, 1000, n)])
    q = occlusion_rays(ptb, rays, tmax, exclude.astype(np.uint32))
    g = gpu_ctx.occluded(q)
    r = VisibilityOracle(s).occluded(q)
    ok = ~degenerate(rays, c, c) & (c["t"] != tmax)
    assert g.dtype == bool and np.array_equal(g[ok], r[ok]), int((g[ok] != r[ok]).sum())
    assert 0.02 < g.mean() < 0.9
    assert not g[~(tmax > 0)].any()


@pytest.mark.parametrize("which", ["c3", "c5"])
def test_agrees_with_closest_hit_at_full_size(ptb, gpu_ctx, request, which):
    if which == "c3":
        s, rays = request.getfixturevalue("c3_full"), random_rays(ptb, 1 << 20, 77, centre=(0, 4, 1), radius=6.0)
    else:
        s, rays = request.getfixturevalue("c5_full"), ptb.meshgen.philox_rays(1 << 22, first=0)
    commit(gpu_ctx, s)
    h = gpu_ctx.closest_hit(rays)
    hit = h["prim"] != MISS
    assert 0.05 < hit.mean() < 0.95
    tc = h["t"]
    for tmax in (np.full(len(rays), np.inf, np.float32), tc, np.nextafter(tc, np.float32(np.inf)), np.float32(0.5) * tc):
        occ = gpu_ctx.occluded(occlusion_rays(ptb, rays, tmax, MISS))
        assert np.array_equal(occ, hit & (tc < tmax))
    chi = gpu_ctx.check_hit_index(rays[hit], h["prim"][hit])
    assert same_bits(chi, h[hit])


def test_builders_agree(ptb, gpu_ctx):
    s = ptb.meshgen.c3_scene(0.1)
    rays, ids = target_rays(ptb, s, 100_000, 23, centre=(0, 4, 1), radius=4.0)
    q = occlusion_rays(ptb, rays, np.random.default_rng(1).uniform(0, 8, len(rays)).astype(np.float32), ids)
    out = []
    for flags in (ptb._lib.BUILD_SAH, ptb._lib.BUILD_BINARY, ptb._lib.BUILD_WIDE):
        commit(gpu_ctx, s, flags)
        out.append((gpu_ctx.check_hit_index(rays, ids), gpu_ctx.occluded(q)))
    assert gpu_ctx.bvh_builder()[0] == ptb._lib.BUILD_WIDE
    for chi, occ in out[1:]:
        assert same_bits(chi, out[0][0]) and np.array_equal(occ, out[0][1])
    assert 0.05 < (out[0][0]["prim"] != MISS).mean() < 0.95 and 0.05 < out[0][1].mean() < 0.95


def test_ordering_and_staging_do_not_change_results(ptb, gpu_ctx, monkeypatch):
    s = ptb.meshgen.c3_scene(0.1)
    commit(gpu_ctx, s)
    rays, ids = target_rays(ptb, s, 150_001, 24, centre=(0, 4, 1), radius=6.0)
    q = occlusion_rays(ptb, rays, np.inf, ids)
    a_chi, a_occ = gpu_ctx.check_hit_index(rays, ids), gpu_ctx.occluded(q)
    monkeypatch.setenv("PTB_HIT_SORT", "0")
    b_chi, b_occ = gpu_ctx.check_hit_index(rays, ids), gpu_ctx.occluded(q)
    monkeypatch.delenv("PTB_HIT_SORT")
    monkeypatch.setenv("PTB_HIT_BATCH", "4096")
    out_chi, out_occ = np.zeros(len(rays), ptb.hit_dtype), np.zeros(len(rays), bool)
    c_chi, c_occ = gpu_ctx.check_hit_index(rays, ids, out=out_chi), gpu_ctx.occluded(q, out=out_occ)
    assert c_chi is out_chi and c_occ is out_occ
    for chi, occ in ((b_chi, b_occ), (c_chi, c_occ)):
        assert same_bits(chi, a_chi) and np.array_equal(occ, a_occ)
    assert 0.05 < (a_chi["prim"] != MISS).mean() < 0.95 and 0.05 < a_occ.mean() < 0.95


def test_device_variants_match_host_variants(ptb, gpu_ctx):
    import torch
    s = ptb.meshgen.c3_scene(0.1)
    commit(gpu_ctx, s)
    rays, ids = target_rays(ptb, s, 100_000, 25, centre=(0, 4, 1), radius=4.0)
    q = occlusion_rays(ptb, rays, np.random.default_rng(2).uniform(0, 8, len(rays)).astype(np.float32), ids)
    dev = torch.device("cuda", 0)
    t_rays = torch.from_numpy(rays.view(np.uint8).copy()).to(dev)
    t_ids = torch.from_numpy(ids.view(np.int32).copy()).to(dev)
    t_q = torch.from_numpy(q.view(np.uint8).copy()).to(dev)
    t_hits = torch.zeros(len(rays) * 16, dtype=torch.uint8, device=dev)
    t_occ = torch.full((len(rays),), 7, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    gpu_ctx.check_hit_index_device(t_rays.data_ptr(), t_ids.data_ptr(), len(rays), t_hits.data_ptr())
    gpu_ctx.occluded_device(t_q.data_ptr(), len(rays), t_occ.data_ptr())
    gpu_ctx.synchronize()
    chi = t_hits.cpu().numpy().view(ptb.hit_dtype)
    occ = t_occ.cpu().numpy()
    assert same_bits(chi, gpu_ctx.check_hit_index(rays, ids))
    assert set(np.unique(occ)) <= {0, 1} and np.array_equal(occ.view(bool), gpu_ctx.occluded(q))


def test_edge_inputs(ptb, gpu_ctx, rtweekend1):
    L = ptb._lib
    fresh = ptb.Context(0)
    try:
        with pytest.raises(ptb.PtbError) as e:
            fresh.occluded(occlusion_rays(ptb, random_rays(ptb, 4, 1), np.inf, MISS))
        assert e.value.code == 1
        with pytest.raises(ptb.PtbError) as e:
            fresh.check_hit_index(random_rays(ptb, 4, 1), np.zeros(4, np.uint32))
        assert e.value.code == 1
    finally:
        fresh.close()
    commit(gpu_ctx, rtweekend1)
    h = gpu_ctx._h
    assert len(gpu_ctx.check_hit_index(np.zeros(0, ptb.ray_dtype), np.zeros(0, np.uint32))) == 0       # empty batch
    assert len(gpu_ctx.occluded(np.zeros(0, ptb.occlusion_ray_dtype))) == 0
    assert L.lib.ptb_occluded(h, None, 0, None) == 0 and L.lib.ptb_check_hit_index(h, None, None, 0, None) == 0
    assert L.lib.ptb_occluded_device(h, None, 0, None) == 0 and L.lib.ptb_check_hit_index_device(h, None, None, 0, None) == 0
    buf = np.zeros(64, np.uint8)
    for rc in (L.lib.ptb_occluded(h, None, 3, L.ptr(buf)), L.lib.ptb_occluded(h, L.ptr(buf), 1, None),
               L.lib.ptb_check_hit_index(h, L.ptr(buf), None, 1, L.ptr(buf)),
               L.lib.ptb_occluded_device(h, None, 3, None), L.lib.ptb_check_hit_index_device(h, None, None, 3, None)):
        assert rc == 1
    for n in (1, 31, 32, 33, 255, 257, 1025):                                                            # ragged sizes
        rays, ids = target_rays(ptb, rtweekend1, n, n, centre=(0, 1, 0))
        assert len(gpu_ctx.check_hit_index(rays, ids)) == n and len(gpu_ctx.occluded(occlusion_rays(ptb, rays, 1.0, ids))) == n
    rays = random_rays(ptb, 1000, 3, centre=(0, 1, 0), radius=3.0)                                       # out-of-range target
    for bad in (rtweekend1.n_primitives, MISS):
        out = gpu_ctx.check_hit_index(rays, np.full(len(rays), bad, np.uint32))
        assert np.all(out["prim"] == MISS) and np.all(out["t"] == 0)
    s = copy.deepcopy(rtweekend1)                                                                         # empty scene
    s.spheres = s.spheres[:0].copy()
    commit(gpu_ctx, s)
    out = gpu_ctx.check_hit_index(rays, np.zeros(len(rays), np.uint32))
    assert np.all(out["prim"] == MISS) and np.all(out["t"] == 0)
    assert not gpu_ctx.occluded(occlusion_rays(ptb, rays, np.inf, MISS)).any()
