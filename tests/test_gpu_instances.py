"""Mesh instances through the C ABI: ptb_scene_set_mesh_instances, ptb_scene_update_instance_xforms(_device) and the
device expansion (lbvh_build.cu k_expand_instances) that runs at commit.

An instanced scene must behave bit for bit as the flat scene IndexedMesh.expand_instances() gives, so every test uploads
the instanced scene in one context and that flat expansion in a second one and compares them:
  * full commits over the LBVH, SAH and wide builders: tree exports, SAH cost, closest hit, check_hit_index, occlusion;
  * renders (naive and MIS), including a scene whose only lights are instances with an emissive material override;
  * transform updates (host, device from a torch tensor, partial ranges) and mesh vertex updates, with refit;
  * the error rules, and build_ms / kernel_launches including the expansion.
"""
import copy

import numpy as np
import pytest

from test_gpu_mesh import expect, flag, render_both, same_export, same_queries

pytestmark = pytest.mark.gpu

INVALID = 1


@pytest.fixture()
def ctx2(ptb):
    """The flat scene's context, beside the instanced one."""
    c = ptb.Context(0)
    yield c
    c.close()


def flat_of(scene, mesh, inst, xf):
    s = copy.copy(scene)
    s.triangles = mesh.expand_instances(inst, xf)
    return s


def emissive_scene(ptb):
    """c3_instanced with a third instance, a rotated, smaller copy of the glass sphere whose triangles all get an emissive
    material: the scene's only lights are those instanced triangles."""
    scene, mesh, inst, xf = ptb.meshgen.c3_instanced(0.05)
    scene = copy.deepcopy(scene)
    lamp = scene.add_material(ptb.MAT_EMIT, scene.add_texture(ptb.TEX_SOLID, (1.0, 0.9, 0.7)), 6.0)
    extra = np.zeros(1, ptb.mesh_instance_dtype)
    extra[0] = (inst["first_triangle"][1], inst["n_triangles"][1], lamp)
    lamp_xf = ptb.instance_xform(rotation=(0.8, 0.2, 0.1, 0.3), scale=0.4, translation=(-1.0, -2.2, 0.9))
    return scene, mesh, np.concatenate([inst, extra]), np.concatenate([xf, lamp_xf])


def instanced(ptb, which):
    if which == "c3":
        return ptb.meshgen.c3_instanced(0.05)
    if which == "scatter":
        return ptb.meshgen.scatter_instances(ptb.meshgen.rock(8, 5), 1000, seed=11, terrain=(40, 16))
    return emissive_scene(ptb)


def commit_pair(ptb, ctx_i, ctx_f, scene, mesh, inst, xf, builder):
    ctx_i.upload(scene, mesh=mesh, instances=(inst, xf))
    ctx_i.commit(flag(ptb, builder))
    ctx_f.upload(flat_of(scene, mesh, inst, xf))
    ctx_f.commit(flag(ptb, builder))


# ------------------------------------------------------------------------------------------------------- full commit
@pytest.mark.parametrize("builder", ["lbvh", "sah", "wide"])
@pytest.mark.parametrize("which", ["c3", "scatter", "emissive"])
def test_full_commit_equals_the_flat_scene(ptb, gpu_ctx, ctx2, builder, which):
    scene, mesh, inst, xf = instanced(ptb, which)
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, inst, xf, builder)
    n = len(scene.spheres) + int(inst["n_triangles"].sum())
    assert gpu_ctx.bvh_info() == ctx2.bvh_info() and gpu_ctx.bvh_info()[0] == n
    same_export(gpu_ctx, ctx2, builder)
    g = same_queries(ptb, gpu_ctx, ctx2, "c3")
    assert (g["prim"] != ptb.PTB_MISS).any()


@pytest.mark.parametrize("shift", [0.0, 1.0])
def test_full_size_c3(ptb, gpu_ctx, ctx2, shift):
    scene, mesh, inst, xf = ptb.meshgen.c3_instanced(1.0)
    gpu_ctx.upload(scene, mesh=mesh, instances=(inst, xf))
    gpu_ctx.commit(ptb._lib.BUILD_SAH)
    if shift:  # the moved frame: one transform update, then a full commit
        xf = xf.copy()
        xf[1] = ptb.meshgen.c3_instanced_frame(shift)[0]
        gpu_ctx.update_instance_xforms(1, xf[1:])
        gpu_ctx.commit(ptb._lib.BUILD_SAH)
    ctx2.upload(flat_of(scene, mesh, inst, xf))
    ctx2.commit(ptb._lib.BUILD_SAH)
    assert gpu_ctx.bvh_info()[0] == 1_000_000
    same_export(gpu_ctx, ctx2, "sah")
    same_queries(ptb, gpu_ctx, ctx2, "c3", n=400_000)


# ------------------------------------------------------------------------------------------------------------ render
@pytest.mark.parametrize("method", [0, 1])
@pytest.mark.parametrize("which", ["c3", "emissive"])
def test_render_equals_the_flat_scene(ptb, gpu_ctx, ctx2, which, method):
    scene, mesh, inst, xf = instanced(ptb, which)
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, inst, xf, "sah")
    img = render_both(ptb, gpu_ctx, ctx2, method)
    assert img.max() > 0
    if which == "emissive" and method == 1:  # the MIS render samples the instanced emitters as lights
        assert gpu_ctx.stats().rays_shadow_light > 0


# --------------------------------------------------------------------------------------------------------- animation
def moved_xforms(ptb, xf, step):
    """Every instance but the terrain turned a little about z and shifted along x."""
    out = xf.copy()
    c, s = np.cos(0.2 * step), np.sin(0.2 * step)
    turn = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]], np.float32)
    out["m"][1:, :, :3] = np.einsum("ij,njk->nik", turn, out["m"][1:, :, :3]).astype(np.float32)
    out["n"][1:] = np.einsum("ij,njk->nik", turn, out["n"][1:]).astype(np.float32)
    out["m"][1:, 0, 3] += np.float32(0.3 * step)
    return out


@pytest.mark.parametrize("builder", ["lbvh", "sah"])
@pytest.mark.parametrize("path", ["host", "device", "partial"])
def test_xform_update_and_refit_equal_the_flat_update(ptb, gpu_ctx, ctx2, builder, path):
    import torch
    scene, mesh, inst, xf = ptb.meshgen.scatter_instances(ptb.meshgen.rock(8, 5), 60, seed=5, terrain=(40, 16))
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, inst, xf, builder)
    new = moved_xforms(ptb, xf, 1)
    if path == "host":
        gpu_ctx.update_instance_xforms(0, new)
    elif path == "device":
        d = torch.from_numpy(new.view(np.float32).copy()).cuda()
        torch.cuda.synchronize()  # the tensor is ready before the context's stream copies it
        gpu_ctx.update_instance_xforms_device(0, d.data_ptr(), len(new))
    else:  # three ranges, host and device mixed; an empty update in between
        a, b = len(new) // 3, 2 * len(new) // 3
        d = torch.from_numpy(new[a:b].view(np.float32).copy()).cuda()
        torch.cuda.synchronize()
        gpu_ctx.update_instance_xforms(b, new[b:])
        gpu_ctx.update_instance_xforms_device(a, d.data_ptr(), b - a)
        gpu_ctx.update_instance_xforms(0, new[:0])
        gpu_ctx.update_instance_xforms(0, new[:a])
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    ctx2.update_triangles(0, mesh.expand_instances(inst, new))
    ctx2.commit(ptb._lib.BUILD_REFIT)
    same_export(gpu_ctx, ctx2, builder)
    same_queries(ptb, gpu_ctx, ctx2, "c3", seed=33)
    # hits of the refitted instanced scene = a fresh full commit of the moved scene
    ctx2.upload(flat_of(scene, mesh, inst, new))
    ctx2.commit(flag(ptb, builder))
    same_queries(ptb, gpu_ctx, ctx2, "c3", seed=34)


def test_mesh_vertex_update_moves_every_instance(ptb, gpu_ctx, ctx2):
    scene, mesh, inst, xf = ptb.meshgen.scatter_instances(ptb.meshgen.rock(8, 5), 40, seed=6, terrain=(40, 16))
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, inst, xf, "sah")
    k = len(mesh.vertices) - len(ptb.meshgen.rock(8, 5).vertices)  # the rock's vertices follow the terrain's
    grown = mesh.vertices[k:] * np.float32(1.3)
    gpu_ctx.update_mesh_vertices(k, grown)
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    moved = ptb.IndexedMesh(np.concatenate([mesh.vertices[:k], grown]), mesh.normals, mesh.triangles)
    after = moved.expand_instances(inst, xf)
    assert not np.array_equal(after["p"], mesh.expand_instances(inst, xf)["p"])
    ctx2.update_triangles(0, after)
    ctx2.commit(ptb._lib.BUILD_REFIT)
    same_export(gpu_ctx, ctx2, "sah")
    same_queries(ptb, gpu_ctx, ctx2, "c3", seed=35)


# ------------------------------------------------------------------------------------------------------------ errors
def test_instances_need_a_mesh_scene_and_valid_ranges(ptb, gpu_ctx, overshadowed):
    scene, mesh, inst, xf = ptb.meshgen.c3_instanced(0.05)
    gpu_ctx.upload(overshadowed)
    expect(ptb, gpu_ctx.set_mesh_instances, inst, xf, match="not an indexed mesh")
    gpu_ctx.upload(scene, mesh=mesh)
    bad = inst.copy()
    bad[1]["n_triangles"] += 1  # one past the end of the mesh
    expect(ptb, gpu_ctx.set_mesh_instances, bad, xf, match="mesh instance 1:")
    bad = inst.copy()
    bad[0]["first_triangle"] = 0xFFFFFFFF  # first + n overflows 32 bits
    expect(ptb, gpu_ctx.set_mesh_instances, bad, xf, match="mesh instance 0:")
    lib, h = ptb._lib.lib, gpu_ctx._h
    assert lib.ptb_scene_set_mesh_instances(h, None, ptb._lib.ptr(xf), 1) == INVALID
    assert lib.ptb_scene_set_mesh_instances(h, ptb._lib.ptr(inst), None, 1) == INVALID
    assert lib.ptb_scene_set_mesh_instances(h, None, None, 0) == 0  # zero instances: zero triangles
    gpu_ctx.commit()
    assert gpu_ctx.bvh_info()[0] == 0


def test_more_than_2_32_triangles_fail_before_allocating(ptb, gpu_ctx):
    scene, mesh = ptb.meshgen.heightfield_indexed(128, 256)
    assert len(mesh.triangles) == 65536
    gpu_ctx.upload(scene, mesh=mesh)
    inst = np.zeros(65537, ptb.mesh_instance_dtype)
    inst["n_triangles"], inst["material"] = 65536, ptb.PTB_MISS
    xf = np.repeat(ptb.instance_xform(), len(inst))
    # 2^32 + 65536 triangles would be 326 GB of records: INVALID (not out of memory) shows nothing was allocated
    expect(ptb, gpu_ctx.set_mesh_instances, inst, xf, match="mesh instance 65535: the instances place more than 2^32 - 1")
    gpu_ctx.set_mesh_instances(inst[:2], xf[:2])
    gpu_ctx.commit()
    assert gpu_ctx.bvh_info()[0] == 2 * 65536


def test_xform_update_ranges_and_modes(ptb, gpu_ctx, overshadowed):
    import torch
    scene, mesh, inst, xf = ptb.meshgen.c3_instanced(0.05)
    gpu_ctx.upload(scene, mesh=mesh)
    expect(ptb, gpu_ctx.update_instance_xforms, 0, xf[:1], match="no instance list")
    gpu_ctx.set_mesh_instances(inst, xf)
    lib, h, p = ptb._lib.lib, gpu_ctx._h, ptb._lib.ptr(xf)
    big = 2**64 - 1
    for fn in (lib.ptb_scene_update_instance_xforms, lib.ptb_scene_update_instance_xforms_device):
        assert fn(h, 1, p, 2) == INVALID             # one past the end
        assert fn(h, 3, p, 0) == INVALID             # first beyond the end, even with n == 0
        assert fn(h, big, p, 2) == INVALID and fn(h, 1, p, big) == INVALID
        assert fn(h, 0, None, 1) == INVALID
        assert fn(h, 0, None, 0) == 0 and fn(h, 2, p, 0) == 0
    # set_mesh drops the instance list: the scene's triangles are the mesh's own again
    gpu_ctx.set_mesh(mesh)
    expect(ptb, gpu_ctx.update_instance_xforms, 0, xf[:1], match="no instance list")
    gpu_ctx.set_mesh_instances(inst[:1], xf[:1])
    gpu_ctx.commit()
    assert gpu_ctx.bvh_info()[0] == inst["n_triangles"][0]
    gpu_ctx.set_mesh(mesh)
    gpu_ctx.commit()
    assert gpu_ctx.bvh_info()[0] == len(mesh.triangles)
    # set_triangles drops the mesh and the instances
    gpu_ctx.set_mesh_instances(inst, xf)
    expect(ptb, gpu_ctx.update_triangles, 0, mesh.expand()[:1], match="indexed mesh")
    gpu_ctx.upload(overshadowed)
    d = torch.zeros(84, dtype=torch.uint8, device="cuda")
    expect(ptb, gpu_ctx.update_instance_xforms, 0, xf[:1], match="no instance list")
    expect(ptb, gpu_ctx.update_instance_xforms_device, 0, d.data_ptr(), 1, match="no instance list")
    expect(ptb, gpu_ctx.update_mesh_vertices, 0, mesh.vertices[:1], match="not an indexed mesh")
    expect(ptb, gpu_ctx.set_mesh_instances, inst, xf, match="not an indexed mesh")
    gpu_ctx.commit()
    assert gpu_ctx.bvh_info()[0] == len(overshadowed.spheres) + len(overshadowed.triangles)


def test_refit_after_the_instance_count_changed(ptb, gpu_ctx, ctx2):
    scene, mesh, inst, xf = ptb.meshgen.c3_instanced(0.05)
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, inst, xf, "lbvh")
    # the same triangles as three instances (the terrain's range split in two): the refit keeps the tree
    half = int(inst["n_triangles"][0]) // 2
    split = np.concatenate([inst[:1], inst[:1], inst[1:]])
    split[0]["n_triangles"], split[1]["first_triangle"], split[1]["n_triangles"] = half, half, inst["n_triangles"][0] - half
    gpu_ctx.set_mesh_instances(split, np.concatenate([xf[:1], xf]))
    gpu_ctx.commit(ptb._lib.BUILD_REFIT)
    same_export(gpu_ctx, ctx2, "lbvh")
    same_queries(ptb, gpu_ctx, ctx2, "c3", n=20_000)
    # a different total: the refit is refused, a full commit works
    gpu_ctx.set_mesh_instances(inst[1:], xf[1:])
    expect(ptb, gpu_ctx.commit, ptb._lib.BUILD_REFIT, match="PTB_BUILD_REFIT keeps the tree")
    gpu_ctx.commit(ptb._lib.BUILD_BINARY)
    assert gpu_ctx.bvh_info()[0] == inst["n_triangles"][1]


@pytest.mark.parametrize("refit", [False, True])
def test_a_bad_index_in_a_placed_triangle_names_the_mesh_triangle(ptb, gpu_ctx, ctx2, refit):
    scene, mesh, inst, xf = ptb.meshgen.c3_instanced(0.05)
    n_terrain = int(inst["n_triangles"][0])
    # place the sphere twice and the terrain not at all: terrain triangles are never expanded, so never checked
    place = np.concatenate([inst[1:], inst[1:]])
    two = np.concatenate([xf[1:], ptb.instance_xform(translation=(0.0, 0.0, 2.0))])
    commit_pair(ptb, gpu_ctx, ctx2, scene, mesh, place, two, "sah")
    bad = mesh.triangles[[3, n_terrain + 7]].copy()
    bad["p"][:, 1] = len(mesh.vertices)
    gpu_ctx.update_mesh_triangles(3, bad[:1])  # an unplaced triangle: still commits
    gpu_ctx.commit(ptb._lib.BUILD_REFIT if refit else ptb._lib.BUILD_SAH)
    gpu_ctx.update_mesh_triangles(n_terrain + 7, bad[1:])
    commit = (lambda: gpu_ctx.commit(ptb._lib.BUILD_REFIT)) if refit else (lambda: gpu_ctx.commit(ptb._lib.BUILD_SAH))
    expect(ptb, commit, match=f"mesh triangle {n_terrain + 7}: vertex index out of range")
    gpu_ctx.update_mesh_triangles(n_terrain + 7, mesh.triangles[n_terrain + 7:n_terrain + 8])
    commit()
    same_export(gpu_ctx, ctx2, "sah")
    same_queries(ptb, gpu_ctx, ctx2, "c3", n=20_000)


# ------------------------------------------------------------------------------------------------------------- stats
def test_build_stats_include_the_expansion(ptb, gpu_ctx, ctx2):
    scene, mesh, inst, xf = ptb.meshgen.c3_instanced(0.05)
    gpu_ctx.upload(scene, mesh=mesh, instances=(inst, xf))
    ctx2.upload(flat_of(scene, mesh, inst, xf))

    def launches(ctx, flags):
        ctx.stats_reset()
        ctx.commit(flags)
        st = ctx.stats()
        assert st.build_ms > 0
        return st.kernel_launches

    B, R = ptb._lib.BUILD_BINARY, ptb._lib.BUILD_REFIT
    assert launches(gpu_ctx, B) == launches(ctx2, B) + 1        # the expansion: one kernel
    assert launches(gpu_ctx, B) == launches(ctx2, B)            # nothing changed: not expanded again
    assert launches(gpu_ctx, R) == launches(ctx2, R)
    gpu_ctx.update_instance_xforms(1, ptb.meshgen.c3_instanced_frame(0.5))
    assert launches(gpu_ctx, R) == launches(ctx2, R) + 1        # a transform update makes the next commit expand
    gpu_ctx.update_mesh_vertices(0, mesh.vertices[:3])
    assert launches(gpu_ctx, R) == launches(ctx2, R) + 1        # and so does a mesh update
