#!/usr/bin/env python
"""Indexed meshes (ptb_scene_set_mesh, ptb_scene_update_mesh_*, k_expand_mesh) against flat triangles, on the GPU only (no
device: it fails).

  python scripts/mesh_bench.py [--reps 11] [--warmup 3] [--phases upload,frame,kernel] [--json FILE]

Two contexts hold the same scene: one as flat 76-byte triangles, one as an indexed mesh (meshgen.c3_indexed /
heightfield_indexed, whose expand() is byte-identical to the flat scene). Before anything is reported, closest hits of
the two contexts are compared bit for bit on 2^20 Philox rays, after every timed frame and after each upload workload.
  upload  full upload + SAH commit of C3 (1 M triangles) and C5 (10 M): host wall time of Context.upload + commit (pageable
          numpy arrays, as the Python interface passes them) and the commit's device time (ptb_stats.build_ms).
  frame   one C3 animation frame end to end (meshgen.c3_deform_vertices, a new wave / shift each frame): host
          update_triangles of all 1 M triangles (76 MB) + PTB_BUILD_REFIT against host update_mesh_vertices of the
          502 603 vertices (6 MB) + refit, from pinned host buffers; then the same with the _device twins from CUDA
          tensors. Host wall time from the update call to the end of the commit, and build_ms.
  kernel  k_expand_mesh alone under torch.profiler (a refit commit after a one-vertex update expands the whole mesh) on C3
          and C5: bytes the expansion must move (28 B of indices read + 76 B written per triangle + 12 B per vertex and
          per normal read once), achieved bandwidth and its fraction of 7.7 TB/s. C3's ~116 MB is about the size of the
          126 MB L2, so part of it may be served from L2; C5's ~1.2 GB is not.
Reported: median and range over --reps repetitions after --warmup.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_TBPS = 7.7  # HGX B200 data sheet, one GPU


def device_identity(torch):
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def stat(xs):
    xs = sorted(xs)
    return dict(median=float(np.median(xs)), min=float(xs[0]), max=float(xs[-1]), reps=len(xs))


def fmt(s, d=3):
    return f"{s['median']:.{d}f} ({s['min']:.{d}f} - {s['max']:.{d}f})"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=11)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--phases", default="upload,frame,kernel")
    ap.add_argument("--json", default="", help="also write the results to this file")
    args = ap.parse_args()
    assert args.reps >= 11, "at least 11 timed repetitions"
    phases = set(args.phases.split(","))

    import torch
    if not torch.cuda.is_available():
        sys.exit("mesh_bench.py measures on the GPU and found no CUDA device")
    import ptb200
    L = ptb200._lib
    mg = ptb200.meshgen
    R, W = args.reps, args.warmup
    name, power = device_identity(torch)
    print(f"device: {name}, power limit {power}, library {L.LIB_PATH}", flush=True)
    out = dict(device=name, power_limit=power, library=os.path.basename(L.LIB_PATH), reps=R, warmup=W, checks=[])
    rays = mg.philox_rays(1 << 20, seed=9, centre=(0.0, 4.0, 1.0), radius=5.0)
    ctx_f, ctx_m = ptb200.Context(0), ptb200.Context(0)

    def check(tag, rays=rays):
        same = ctx_f.closest_hit(rays).tobytes() == ctx_m.closest_hit(rays).tobytes()
        out["checks"].append(dict(what=tag, hits_bit_identical=same))
        if not same:
            sys.exit(f"closest hits of the mesh scene differ from the flat scene's ({tag}): nothing is reported")

    # ---------------------------------------------------------------- 1. full upload + commit
    if "upload" in phases:
        up = {}
        for wl in ("C3", "C5"):
            scene, mesh = mg.c3_indexed(1.0) if wl == "C3" else mg.heightfield_indexed(2500, 2000)
            flat = mg.c3_scene(1.0) if wl == "C3" else mg.heightfield_scene(2500, 2000)
            assert mesh.expand().tobytes() == flat.triangles.tobytes()
            res = {}
            for arm, ctx, op in (("flat", ctx_f, lambda: ctx_f.upload(flat)), ("indexed", ctx_m, lambda: ctx_m.upload(scene, mesh=mesh))):
                wall, dev = [], []
                for k in range(W + R):
                    t0 = time.perf_counter()
                    op()
                    ctx.commit(L.BUILD_SAH)
                    t1 = time.perf_counter()
                    if k >= W:
                        wall.append((t1 - t0) * 1e3)
                        dev.append(ctx.stats().build_ms)
                res[arm] = dict(wall_ms=stat(wall), build_ms=stat(dev),
                                bytes=int(flat.triangles.nbytes if arm == "flat" else mesh.nbytes()))
            wr = rays if wl == "C3" else mg.philox_rays(1 << 20, seed=9, centre=(0.0, 0.0, 0.0), radius=2.0)
            check(f"{wl} full commit", wr)
            up[wl] = res
            print(f"{wl} upload+commit: flat {fmt(res['flat']['wall_ms'])} ms wall, {fmt(res['flat']['build_ms'])} ms build; "
                  f"indexed {fmt(res['indexed']['wall_ms'])} ms wall, {fmt(res['indexed']['build_ms'])} ms build", flush=True)
            del scene, mesh, flat
        out["upload"] = up

    # ---------------------------------------------------------------- 2. one C3 animation frame
    if "frame" in phases:
        scene, mesh = mg.c3_indexed(1.0)
        ctx_f.upload(mg.c3_scene(1.0))
        ctx_f.commit(L.BUILD_SAH)
        ctx_m.upload(scene, mesh=mesh)
        ctx_m.commit(L.BUILD_SAH)
        nt, nv = len(mesh.triangles), len(mesh.vertices)
        pin_t = torch.empty(nt * 76, dtype=torch.uint8, pin_memory=True).numpy().view(L.triangle_dtype)
        pin_v = torch.empty(nv * 12, dtype=torch.uint8, pin_memory=True).numpy().view(np.float32).reshape(nv, 3)
        frames = {}
        for twin in ("host", "device"):
            res = {"flat": dict(wall=[], dev=[]), "indexed": dict(wall=[], dev=[])}
            for k in range(W + R):
                moved = mg.c3_deform_vertices(mesh, 0.05 + 0.4 * k / (W + R), 2.0 * k / (W + R))
                pin_t[:] = moved.expand()
                pin_v[:] = moved.vertices
                if twin == "device":
                    d_t = torch.from_numpy(pin_t.view(np.uint8)).cuda()
                    d_v = torch.from_numpy(pin_v.view(np.uint8).reshape(-1)).cuda()
                    torch.cuda.synchronize()  # produced before the contexts' streams copy them
                for arm, ctx in (("flat", ctx_f), ("indexed", ctx_m)):
                    t0 = time.perf_counter()
                    if twin == "host":
                        if arm == "flat":
                            ctx.update_triangles(0, pin_t)
                        else:
                            ctx.update_mesh_vertices(0, pin_v)
                    elif arm == "flat":
                        ctx.update_triangles_device(0, d_t.data_ptr(), nt)
                    else:
                        ctx.update_mesh_vertices_device(0, d_v.data_ptr(), nv)
                    ctx.commit(L.BUILD_REFIT)
                    t1 = time.perf_counter()
                    if k >= W:
                        res[arm]["wall"].append((t1 - t0) * 1e3)
                        res[arm]["dev"].append(ctx.stats().build_ms)
                check(f"C3 frame {k} ({twin} update)")
            frames[twin] = {arm: dict(wall_ms=stat(v["wall"]), build_ms=stat(v["dev"])) for arm, v in res.items()}
            f, m = frames[twin]["flat"], frames[twin]["indexed"]
            print(f"C3 frame, {twin} update + refit: flat {fmt(f['wall_ms'])} ms wall ({fmt(f['build_ms'])} build), indexed "
                  f"{fmt(m['wall_ms'])} ms wall ({fmt(m['build_ms'])} build): {f['wall_ms']['median'] / m['wall_ms']['median']:.2f}x",
                  flush=True)
        out["frame"] = frames
        out["frame_bytes"] = dict(flat=nt * 76, indexed=nv * 12)

    # ---------------------------------------------------------------- 3. k_expand_mesh alone
    if "kernel" in phases:
        from torch.profiler import ProfilerActivity, profile
        kern = {}
        for wl in ("C3", "C5"):
            scene, mesh = mg.c3_indexed(1.0) if wl == "C3" else mg.heightfield_indexed(2500, 2000)
            ctx_m.upload(scene, mesh=mesh)
            ctx_m.commit(L.BUILD_BINARY)
            one = mesh.vertices[:1].copy()
            for _ in range(W):
                ctx_m.update_mesh_vertices(0, one)
                ctx_m.commit(L.BUILD_REFIT)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(R):
                    ctx_m.update_mesh_vertices(0, one)
                    ctx_m.commit(L.BUILD_REFIT)
                torch.cuda.synchronize()
            times = [e.device_time / 1e3 for e in prof.events() if re.search(r"(^|::)k_expand_mesh(\(|<|$)", e.name)]
            refit_ms = [ctx_m.stats().build_ms]
            nt, nvn = len(mesh.triangles), len(mesh.vertices) + len(mesh.normals)
            nbytes = nt * (28 + 76) + nvn * 12
            if len(times) != R:
                sys.exit(f"{wl}: found {len(times)} k_expand_mesh launches in the profile, expected {R}")
            s = stat(times)  # device_time: microseconds
            gbs = nbytes / (s["median"] * 1e-3) / 1e9
            kern[wl] = dict(kernel_ms=s, bytes=nbytes, triangles=nt, GBps=gbs, fraction_of_hbm=gbs / (HBM_TBPS * 1e3),
                            last_refit_build_ms=refit_ms[0])
            print(f"{wl} k_expand_mesh: {fmt(s, 4)} ms for {nbytes / 1e6:.1f} MB -> {gbs:.0f} GB/s = "
                  f"{100 * gbs / (HBM_TBPS * 1e3):.0f} % of {HBM_TBPS} TB/s (refit commit {refit_ms[0]:.3f} ms)", flush=True)
            if wl == "C3":
                ctx_f.upload(mg.c3_scene(1.0))
                ctx_f.commit(L.BUILD_BINARY)
                ctx_m.commit(L.BUILD_BINARY)
                check("C3 after the kernel phase")
            del scene, mesh
        out["kernel"] = kern

    ctx_f.close()
    ctx_m.close()
    print(f"all {len(out['checks'])} hit checks bit-identical")
    print(json.dumps(out))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
