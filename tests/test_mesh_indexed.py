"""Indexed triangle meshes on the host: mesh_triangle_dtype, IndexedMesh.expand(), index_triangles() and the indexed
generators of meshgen. Every indexed scene must expand to its flat counterpart byte for byte: that identity is what the
device tests (test_gpu_mesh.py) compare against."""
import numpy as np
import pytest


def test_mesh_triangle_layout(ptb):
    L = ptb._lib
    assert L.mesh_triangle_dtype.itemsize == 28
    assert [L.mesh_triangle_dtype.fields[f][1] for f in ("p", "n", "material")] == [0, 12, 24]


@pytest.mark.parametrize("scale", [0.05, 0.3, 1.0])
def test_c3_indexed_expands_to_c3(ptb, scale):
    flat = ptb.meshgen.c3_scene(scale)
    scene, mesh = ptb.meshgen.c3_indexed(scale)
    assert len(scene.triangles) == 0 and scene.camera.tobytes() == flat.camera.tobytes()
    assert mesh.expand().tobytes() == flat.triangles.tobytes()
    if scale == 1.0:  # 1001 x 401 terrain points + 202 x 501 sphere points
        assert len(mesh.vertices) == len(mesh.normals) == 502_603 and len(mesh.triangles) == 1_000_000
        assert mesh.nbytes() == 502_603 * 24 + 1_000_000 * 28


@pytest.mark.parametrize("rows, cols", [(7, 5), (60, 41), (2500, 2000)])
def test_heightfield_indexed_expands_to_heightfield(ptb, rows, cols):
    flat = ptb.meshgen.heightfield_scene(rows, cols)
    _, mesh = ptb.meshgen.heightfield_indexed(rows, cols)
    assert len(mesh.vertices) == (rows + 1) * (cols + 1)
    assert mesh.expand().tobytes() == flat.triangles.tobytes()


def test_index_triangles_round_trips(ptb, overshadowed):
    for tri in (overshadowed.triangles, ptb.meshgen.c3_scene(0.3).triangles):
        mesh = ptb.index_triangles(tri)
        assert mesh.expand().tobytes() == tri.tobytes()
        assert len(mesh.vertices) < 3 * len(tri)
        assert len(np.unique(mesh.vertices.view(np.dtype((np.void, 12))))) == len(mesh.vertices)


def test_index_triangles_keeps_signed_zero_and_nan_bits(ptb):
    tri = np.zeros(2, ptb._lib.triangle_dtype)
    tri["p"][0, 0] = [0.0, 1.0, 2.0]
    tri["p"][1, 0] = [-0.0, 1.0, 2.0]
    tri["n"][0, 1, 0] = np.frombuffer(np.uint32(0x7FC00001).tobytes(), np.float32)[0]
    mesh = ptb.index_triangles(tri)
    assert mesh.expand().tobytes() == tri.tobytes()


def test_expand_rejects_an_index_out_of_range(ptb):
    mesh = ptb.index_triangles(ptb.meshgen.c3_scene(0.05).triangles)
    mesh.triangles["p"][3, 1] = len(mesh.vertices)
    with pytest.raises(IndexError):
        mesh.expand()


def test_c3_deform_vertices_keeps_counts_and_indices(ptb):
    _, mesh = ptb.meshgen.c3_indexed(0.05)
    moved = ptb.meshgen.c3_deform_vertices(mesh, 0.5, 1.0)
    assert moved.vertices.shape == mesh.vertices.shape
    assert moved.triangles.tobytes() == mesh.triangles.tobytes() and moved.normals.tobytes() == mesh.normals.tobytes()
    changed = np.any(moved.vertices != mesh.vertices, axis=1)
    assert changed.any() and not changed.all()
    # the same motion as c3_deform: positions agree to rounding, normals and materials are untouched
    flat = ptb.meshgen.c3_deform(ptb.meshgen.c3_scene(0.05), 0.5, 1.0).triangles
    e = moved.expand()
    assert np.allclose(e["p"], flat["p"], rtol=1e-6, atol=1e-6)
    assert e[["n", "material"]].tobytes() == flat[["n", "material"]].tobytes()
