"""Mesh instances on the host: the record layouts of include/ptb200.h, instance_xform, the generators and
IndexedMesh.expand_instances (the definition the device expansion is compared against), checked with independent
arithmetic."""
import numpy as np
import pytest

F = np.float32


def test_record_layouts(ptb):
    i, x = ptb.mesh_instance_dtype, ptb.instance_xform_dtype
    assert i.itemsize == 12 and x.itemsize == 84
    assert [i.fields[k][1] for k in ("first_triangle", "n_triangles", "material")] == [0, 4, 8]
    assert x.fields["m"][1] == 0 and x.fields["n"][1] == 48
    r = np.zeros(1, x)
    r["m"][0] = np.arange(12, dtype=F).reshape(3, 4)
    assert np.array_equal(r.view(F)[:12], np.arange(12, dtype=F))  # row-major m[0..11], then n


def small_mesh(ptb):
    return ptb.index_triangles(ptb.meshgen.c3_scene(0.02).triangles)


def as_value(a):
    """Bytes of a float32 array with -0.0 folded into +0.0: an identity transform may turn -0.0 into +0.0
    (1 * -0 + 0 * y is +0 for y >= 0), so such cases compare by value."""
    return (np.asarray(a, F) + F(0)).tobytes()


def one(ptb, first, n, material=None):
    inst = np.zeros(1, ptb.mesh_instance_dtype)
    inst[0] = (first, n, ptb.PTB_MISS if material is None else material)
    return inst


def test_identity_translation_and_rotation_against_expand(ptb):
    mesh = small_mesh(ptb)
    flat = mesh.expand()
    n = len(flat)
    out = mesh.expand_instances(one(ptb, 0, n), ptb.instance_xform())
    assert as_value(out["p"]) == as_value(flat["p"]) and as_value(out["n"]) == as_value(flat["n"])
    assert np.array_equal(out["material"], flat["material"])
    t = F([0.25, -3.0, 1.5])
    out = mesh.expand_instances(one(ptb, 0, n), ptb.instance_xform(translation=t))
    assert as_value(out["p"]) == as_value(flat["p"] + t) and as_value(out["n"]) == as_value(flat["n"])
    # a quarter turn about z given as an exact matrix: (x, y, z) -> (-y, x, z)
    out = mesh.expand_instances(one(ptb, 0, n), ptb.instance_xform(rotation=[[0, -1, 0], [1, 0, 0], [0, 0, 1]]))
    turned = np.stack([-flat["p"][..., 1], flat["p"][..., 0], flat["p"][..., 2]], -1)
    assert as_value(out["p"]) == as_value(turned)


def test_statement_order_and_no_fma(ptb):
    """x' = ((m0 x + m1 y) + m2 z) + m3 in float32, each operation rounded, recomputed here one scalar at a time."""
    mesh = small_mesh(ptb)
    xf = ptb.instance_xform(rotation=(0.9, 0.1, -0.3, 0.2), scale=1.7, translation=(0.1, 0.2, 0.3))
    xf["n"][0] = F([[0.3, 1.1, -0.7], [2.0, 0.5, 0.25], [-1.5, 0.9, 0.1]])  # a caller-supplied normal map
    out = mesh.expand_instances(one(ptb, 5, 7), xf)
    src = mesh.expand()[5:12]
    m, nm = xf["m"][0], xf["n"][0]
    for t in range(7):
        for k in range(3):
            x, y, z = (F(v) for v in src["p"][t, k])
            a, b, c = (F(v) for v in src["n"][t, k])
            for r in range(3):
                want = F(F(F(F(m[r, 0] * x) + F(m[r, 1] * y)) + F(m[r, 2] * z)) + m[r, 3])
                assert out["p"][t, k, r].tobytes() == want.tobytes()
                want = F(F(F(nm[r, 0] * a) + F(nm[r, 1] * b)) + F(nm[r, 2] * c))
                assert out["n"][t, k, r].tobytes() == want.tobytes()


def test_instance_xform_is_sR_t_and_R(ptb):
    from scipy.spatial.transform import Rotation
    q = np.array([0.3, -0.5, 0.7, 0.2])  # (w, x, y, z), not normalised
    R = Rotation.from_quat([q[1], q[2], q[3], q[0]]).as_matrix()
    xf = ptb.instance_xform(rotation=q, scale=2.5, translation=(1, 2, 3))
    assert np.allclose(xf["n"][0], R, atol=1e-6)
    assert np.allclose(xf["m"][0, :, :3], 2.5 * R, atol=1e-6)
    assert np.array_equal(xf["m"][0, :, 3], F([1, 2, 3]))
    n = xf["n"][0].astype(np.float64)
    assert np.allclose(n @ n.T, np.eye(3), atol=1e-6)
    by_matrix = ptb.instance_xform(rotation=R, scale=2.5, translation=(1, 2, 3))
    assert np.allclose(by_matrix["m"], xf["m"], atol=1e-6) and np.allclose(by_matrix["n"], xf["n"], atol=1e-6)
    ident = ptb.instance_xform()
    assert np.array_equal(ident["m"][0], np.eye(3, 4, dtype=F)) and np.array_equal(ident["n"][0], np.eye(3, dtype=F))
    # unit normals stay unit up to rounding
    mesh = small_mesh(ptb)
    out = mesh.expand_instances(one(ptb, 0, len(mesh.triangles)), ptb.instance_xform(rotation=q))
    assert np.allclose(np.linalg.norm(out["n"], axis=-1), 1.0, atol=1e-5)


def test_ids_order_overlap_repeat_empty_and_materials(ptb):
    mesh = small_mesh(ptb)
    flat = mesh.expand()
    inst = np.zeros(6, ptb.mesh_instance_dtype)
    inst[:] = [(10, 5, ptb.PTB_MISS), (0, 0, 7), (12, 6, 1), (10, 5, ptb.PTB_MISS), (len(flat) - 1, 1, 0), (3, 0, ptb.PTB_MISS)]
    shifts = [F([i, 2 * i, -i]) for i in range(6)]
    xf = np.concatenate([ptb.instance_xform(translation=s) for s in shifts])
    out = mesh.expand_instances(inst, xf)
    assert len(out) == 5 + 0 + 6 + 5 + 1 + 0
    tid = 0
    for i, (first, n, material) in enumerate(inst.tolist()):
        for k in range(n):  # triangle id = earlier instances' n_triangles + position in the range
            src = flat[first + k]
            assert as_value(out["p"][tid]) == as_value(src["p"] + shifts[i])
            assert out["material"][tid] == (src["material"] if material == ptb.PTB_MISS else material)
            tid += 1
    assert tid == len(out)
    assert len(mesh.expand_instances(np.zeros(0, ptb.mesh_instance_dtype), np.zeros(0, ptb.instance_xform_dtype))) == 0
    with pytest.raises(ValueError):
        mesh.expand_instances(inst, xf[:2])


def test_generators(ptb):
    scene, mesh, inst, xf = ptb.meshgen.c3_instanced(0.05)
    assert len(inst) == 2 and inst["n_triangles"].sum() == len(mesh.triangles)
    flat = ptb.meshgen.c3_scene(0.05).triangles
    out = mesh.expand_instances(inst, xf)
    assert as_value(out["p"]) == as_value(flat["p"]) and np.array_equal(out["material"], flat["material"])
    # the sphere instance moved as c3_deform moves the glass sphere
    moved = ptb.meshgen.c3_deform(ptb.meshgen.c3_scene(0.05), 0.0, 0.7).triangles
    xf[1] = ptb.meshgen.c3_instanced_frame(0.7)[0]
    out = mesh.expand_instances(inst, xf)
    glass = flat["material"] == 1
    assert as_value(out["p"][glass]) == as_value(moved["p"][glass])
    rock = ptb.meshgen.rock()
    assert len(rock.triangles) == 1000
    s, m, i, x = ptb.meshgen.scatter_instances(rock, 50, seed=3)
    assert len(i) == 51 and np.all(i["n_triangles"][1:] == 1000)
    s2, m2, i2, x2 = ptb.meshgen.scatter_instances(rock, 50, seed=3)
    assert x.tobytes() == x2.tobytes() and m.triangles.tobytes() == m2.triangles.tobytes()
    out = m.expand_instances(i, x)
    assert len(out) == i["n_triangles"].sum() and np.all(np.isfinite(out["p"]))
