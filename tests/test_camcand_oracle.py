"""CPU: the statement of the per-pixel camera candidate lists (scripts/camcand_ref.cpp, restating csrc/ptb_camcand.cuh) on
the device SAH tree's CPU definition. Every jittered camera ray answered from its pixel's list gets the ordered walk's
hit bit for bit (t and primitive); pixels with more candidates than the list holds are reported as overflowed."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "scripts"))
import camcand_ref  # noqa: E402


@pytest.fixture(scope="module", params=[0.05, 0.25])
def scene(request, ptb):
    return camcand_ref.CamCandScene(ptb.meshgen.c3_scene(request.param))


@pytest.mark.parametrize("W,H,row_begin,rows", [(64, 36, 0, None), (97, 55, 0, None), (160, 90, 31, 17)])
def test_list_hits_equal_the_ordered_walk(scene, W, H, row_begin, rows):
    L = scene.lists(W, H, 16, row_begin=row_begin, rows=rows)
    r = scene.check(L, spp=24, sample_offset=5, seed=11)
    assert r["rays"] == W * L.rows * 24
    assert r["list_rays"] >= 0.5 * r["rays"]  # small images: large pixel footprints, more overflow
    assert r["mismatches"] == 0, r
    assert r["box_rejected_hits"] == 0, r
    assert r["key_above_tkey"] == 0, r  # every key is a lower bound on the cull key of every ray of its pixel
    # the lists hold the nearest candidates in key order, the rest of each entry row is empty
    n = np.minimum(L.count, L.K)
    keys = L.keys.reshape(-1, L.K)
    filled = np.arange(L.K)[None, :] < n[:, None]
    assert np.all(np.isinf(keys[~filled]))
    assert np.all(np.diff(np.where(filled, keys, np.inf), axis=1)[filled[:, 1:]] >= 0)


def test_overflow(scene):
    W, H = 97, 55
    L16, L1 = scene.lists(W, H, 16), scene.lists(W, H, 1)
    assert np.array_equal(L16.count, L1.count)
    assert L1.overflowed.mean() > 0.5
    assert L16.overflowed.mean() < L1.overflowed.mean()
    r = scene.check(L1, spp=8)
    assert r["list_rays"] == 8 * int(np.count_nonzero(~L1.overflowed)) and r["mismatches"] == 0
