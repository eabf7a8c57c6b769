#!/usr/bin/env python
"""Mesh instances (ptb_scene_set_mesh_instances, ptb_scene_update_instance_xforms, k_expand_instances) against indexed
meshes and flat triangles, on the GPU only (no device: it fails).

  python scripts/instance_bench.py [--reps 11] [--warmup 3] [--phases kernel,frame,assembly] [--json FILE]

  kernel    k_expand_instances and k_expand_mesh under torch.profiler (kernel device time; a refit commit after a one-record
            update re-expands everything): C3 as two instances (meshgen.c3_instanced) and as its indexed mesh, C5
            (heightfield_indexed) as one instance and as its mesh, and 10 000 instances of the 1 000-triangle meshgen.rock()
            over a small terrain (meshgen.scatter_instances, 10.03 M triangles). Bytes model, per placed triangle: 28 B of
            indices read + 76 B of record written, plus the mesh's vertex and normal arrays read once (12 B an entry); the
            instance records and transforms are cached. Achieved GB/s against 7.7 TB/s: about 100 flops per triangle
            against over 100 bytes moved is far below the card's f32 rate per byte, so HBM bandwidth is the bound.
  frame     one C3 animation frame end to end, the glass sphere moved by c3_deform's translation three ways: one 84-byte
            transform (update_instance_xforms), the whole 6 MB vertex array (update_mesh_vertices) and all 1 M flat
            triangles (76 MB, update_triangles), each from pinned host memory and from a CUDA tensor (_device twins),
            followed by a PTB_BUILD_REFIT commit. Host wall time from the update call to the end of the commit, and build_ms.
  assembly  upload + SAH commit of the 10 M-triangle scattered scene as instances (mesh + instance list, 2.3 MB) against
            the same scene uploaded flat (760 MB of ptb_triangle), host wall time and build_ms.
Hits are checked after every phase: closest hit of the instanced context against the flat one on 2^20 Philox rays (prim
and t bit for bit; an identity transform may turn a -0.0 coordinate into +0.0, which changes no hit). Reported: median
and range over --reps repetitions after --warmup.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import re
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from mesh_bench import HBM_TBPS, device_identity, fmt, stat  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=11)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--phases", default="kernel,frame,assembly")
    ap.add_argument("--json", default="", help="also write the results to this file")
    args = ap.parse_args()
    assert args.reps >= 11, "at least 11 timed repetitions"
    phases = set(args.phases.split(","))

    import torch
    if not torch.cuda.is_available():
        sys.exit("instance_bench.py measures on the GPU and found no CUDA device")
    from torch.profiler import ProfilerActivity, profile
    import ptb200
    L = ptb200._lib
    mg = ptb200.meshgen
    R, W = args.reps, args.warmup
    name, power = device_identity(torch)
    print(f"device: {name}, power limit {power}, library {L.LIB_PATH}", flush=True)
    out = dict(device=name, power_limit=power, library=os.path.basename(L.LIB_PATH), reps=R, warmup=W, checks=[])
    rays = mg.philox_rays(1 << 20, seed=9, centre=(0.0, 4.0, 1.0), radius=5.0)
    ctx_f, ctx_m, ctx_i = ptb200.Context(0), ptb200.Context(0), ptb200.Context(0)

    def check(tag, a, b, rays=rays):
        ha, hb = a.closest_hit(rays), b.closest_hit(rays)
        same = ha["prim"].tobytes() == hb["prim"].tobytes() and ha["t"].tobytes() == hb["t"].tobytes()
        out["checks"].append(dict(what=tag, hits_bit_identical=same))
        if not same:
            sys.exit(f"closest hits differ ({tag}): nothing is reported")

    def kernel_ms(ctx, kernel, touch):
        """Device time of `kernel` in R refit commits, each after `touch()` (a one-record update)."""
        for _ in range(W):
            touch()
            ctx.commit(L.BUILD_REFIT)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(R):
                touch()
                ctx.commit(L.BUILD_REFIT)
            torch.cuda.synchronize()
        times = [e.device_time / 1e3 for e in prof.events() if re.search(rf"(^|::){kernel}(\(|<|$)", e.name)]
        if len(times) != R:
            sys.exit(f"found {len(times)} {kernel} launches in the profile, expected {R}")
        return stat(times)

    # ---------------------------------------------------------------- 1. the expansion kernels
    if "kernel" in phases:
        kern = {}
        workloads = [("C3", lambda: mg.c3_instanced(1.0)), ("C5", None), ("scatter", lambda: mg.scatter_instances(mg.rock(), 10_000, seed=1))]
        for wl, make in workloads:
            if wl == "C5":
                scene, mesh = mg.heightfield_indexed(2500, 2000)
                inst = np.zeros(1, L.mesh_instance_dtype)
                inst[0] = (0, len(mesh.triangles), L.PTB_MISS)
                xf = ptb200.instance_xform()
            else:
                scene, mesh, inst, xf = make()
            res = {}
            arms = [("k_expand_instances", True)] + ([("k_expand_mesh", False)] if wl != "scatter" else [])
            for kernel, use_inst in arms:
                ctx = ctx_i if use_inst else ctx_m
                ctx.upload(scene, mesh=mesh, instances=(inst, xf) if use_inst else None)
                ctx.commit(L.BUILD_BINARY)
                touch = (lambda: ctx.update_instance_xforms(0, xf[:1])) if use_inst else (lambda: ctx.update_mesh_vertices(0, mesh.vertices[:1]))
                s = kernel_ms(ctx, kernel, touch)
                nt = int(inst["n_triangles"].sum()) if use_inst else len(mesh.triangles)
                nbytes = nt * (28 + 76) + (len(mesh.vertices) + len(mesh.normals)) * 12
                gbs = nbytes / (s["median"] * 1e-3) / 1e9
                res[kernel] = dict(kernel_ms=s, triangles=nt, bytes=nbytes, GBps=gbs, fraction_of_hbm=gbs / (HBM_TBPS * 1e3))
                print(f"{wl} {kernel}: {fmt(s, 4)} ms, {nt} triangles, {nbytes / 1e6:.1f} MB -> {gbs:.0f} GB/s = "
                      f"{100 * gbs / (HBM_TBPS * 1e3):.0f} % of {HBM_TBPS} TB/s", flush=True)
            if wl != "scatter":
                check(f"{wl} instanced vs mesh after the kernel phase", ctx_i, ctx_m,
                      rays if wl == "C3" else mg.philox_rays(1 << 20, seed=9, centre=(0.0, 0.0, 0.0), radius=2.0))
            kern[wl] = res
            del scene, mesh, inst, xf
        out["kernel"] = kern

    # ---------------------------------------------------------------- 2. one C3 animation frame, three ways
    if "frame" in phases:
        scene_i, mesh, inst, xf = mg.c3_instanced(1.0)
        scene_m, _ = mg.c3_indexed(1.0)
        flat = mg.c3_scene(1.0)
        ctx_f.upload(flat)
        ctx_m.upload(scene_m, mesh=mesh)
        ctx_i.upload(scene_i, mesh=mesh, instances=(inst, xf))
        for ctx in (ctx_f, ctx_m, ctx_i):
            ctx.commit(L.BUILD_SAH)
        nt, nv = len(flat.triangles), len(mesh.vertices)
        pin_t = torch.empty(nt * 76, dtype=torch.uint8, pin_memory=True).numpy().view(L.triangle_dtype)
        pin_v = torch.empty(nv * 12, dtype=torch.uint8, pin_memory=True).numpy().view(np.float32).reshape(nv, 3)
        pin_x = torch.empty(84, dtype=torch.uint8, pin_memory=True).numpy().view(L.instance_xform_dtype)
        arms = (("instances", ctx_i), ("vertices", ctx_m), ("triangles", ctx_f))
        frames = {}
        for twin in ("host", "device"):
            res = {a: dict(wall=[], dev=[]) for a, _ in arms}
            for k in range(W + R):
                shift = 2.0 * (k + 1) / (W + R)
                pin_t[:] = mg.c3_deform(flat, 0.0, shift).triangles
                pin_v[:] = mg.c3_deform_vertices(mesh, 0.0, shift).vertices
                pin_x[:] = mg.c3_instanced_frame(shift)
                if twin == "device":
                    d = {a: torch.from_numpy(p.view(np.uint8).reshape(-1)).cuda() for a, p in
                         (("instances", pin_x), ("vertices", pin_v), ("triangles", pin_t))}
                    torch.cuda.synchronize()  # produced before the contexts' streams copy them
                for arm, ctx in arms:
                    t0 = time.perf_counter()
                    if twin == "host":
                        {"instances": lambda: ctx.update_instance_xforms(1, pin_x), "vertices": lambda: ctx.update_mesh_vertices(0, pin_v),
                         "triangles": lambda: ctx.update_triangles(0, pin_t)}[arm]()
                    else:
                        {"instances": lambda: ctx.update_instance_xforms_device(1, d[arm].data_ptr(), 1),
                         "vertices": lambda: ctx.update_mesh_vertices_device(0, d[arm].data_ptr(), nv),
                         "triangles": lambda: ctx.update_triangles_device(0, d[arm].data_ptr(), nt)}[arm]()
                    ctx.commit(L.BUILD_REFIT)
                    t1 = time.perf_counter()
                    if k >= W:
                        res[arm]["wall"].append((t1 - t0) * 1e3)
                        res[arm]["dev"].append(ctx.stats().build_ms)
                check(f"C3 frame {k} ({twin}): instances vs triangles", ctx_i, ctx_f)
                check(f"C3 frame {k} ({twin}): vertices vs triangles", ctx_m, ctx_f)
            frames[twin] = {a: dict(wall_ms=stat(v["wall"]), build_ms=stat(v["dev"])) for a, v in res.items()}
            print(f"C3 frame, {twin} update + refit: " + "; ".join(
                f"{a} {fmt(frames[twin][a]['wall_ms'])} ms wall ({fmt(frames[twin][a]['build_ms'])} build)" for a, _ in arms), flush=True)
        out["frame"] = frames
        out["frame_bytes"] = dict(instances=84, vertices=nv * 12, triangles=nt * 76)
        del scene_i, scene_m, mesh, flat

    # ---------------------------------------------------------------- 3. scene assembly of the 10 M scattered scene
    if "assembly" in phases:
        scene, mesh, inst, xf = mg.scatter_instances(mg.rock(), 10_000, seed=1)
        flat = copy.copy(scene)
        flat.triangles = mesh.expand_instances(inst, xf)
        res = {}
        for arm, ctx, op, nbytes in (
                ("flat", ctx_f, lambda: ctx_f.upload(flat), flat.triangles.nbytes),
                ("instances", ctx_i, lambda: ctx_i.upload(scene, mesh=mesh, instances=(inst, xf)), mesh.nbytes() + inst.nbytes + xf.nbytes)):
            wall, dev = [], []
            for k in range(W + R):
                t0 = time.perf_counter()
                op()
                ctx.commit(L.BUILD_SAH)
                t1 = time.perf_counter()
                if k >= W:
                    wall.append((t1 - t0) * 1e3)
                    dev.append(ctx.stats().build_ms)
            res[arm] = dict(wall_ms=stat(wall), build_ms=stat(dev), bytes=int(nbytes))
        check("scattered 10 M scene: instances vs flat", ctx_i, ctx_f)
        out["assembly"] = dict(triangles=len(flat.triangles), **res)
        print(f"scatter {len(flat.triangles)} triangles, upload + SAH commit: flat {fmt(res['flat']['wall_ms'])} ms wall "
              f"({res['flat']['bytes'] / 1e6:.0f} MB), instances {fmt(res['instances']['wall_ms'])} ms wall "
              f"({res['instances']['bytes'] / 1e6:.2f} MB); build {fmt(res['flat']['build_ms'])} vs {fmt(res['instances']['build_ms'])} ms",
              flush=True)

    for c in (ctx_f, ctx_m, ctx_i):
        c.close()
    print(f"all {len(out['checks'])} hit checks bit-identical")
    print(json.dumps(out))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
