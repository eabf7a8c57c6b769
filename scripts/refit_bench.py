#!/usr/bin/env python
"""Cost and payoff of PTB_BUILD_REFIT (keep the binary tree, refit its boxes) against full commits, on the GPU only (no
device: it fails).

  python scripts/refit_bench.py [--reps 11] [--warmup 3] [--json FILE]

C3 (1 M triangles), per operation: device time (ptb_stats.build_ms: first to last event of the commit on the context's
    stream) and host wall time of the call, for a full SAH commit, a full LBVH commit, a refit of unchanged primitives, a
    refit after ptb_scene_update_triangles_device of the whole array, and a host ptb_scene_update_triangles of the 200 k
    glass triangles + refit, timed end to end (upload included).
Deformation sequence (meshgen.c3_deform): terrain height scaled by a growing wave, glass sphere moved by 0, 0.5, 1, 2 and 4
    radii into the terrain. The tree of the undeformed SAH commit is refitted to each frame and compared with a fresh SAH
    commit of the same frame: SAH cost (ptb_bvh_sah_cost), nodes fetched / primitives tested per ray (V / T,
    PTB_OPT_COUNT_TRAVERSAL), closest-hit rays/s on 2^22 Philox rays (device buffers), and Mrays/s of a 32-spp 1920x1080
    MIS render.
C5 (10 M triangles): refit time against the SAH and LBVH commit times.
Kernels: one LBVH commit and one refit of C3 under torch.profiler: the fused refit kernel against the three kernels of the
    commit that do the same job (k_prim_bounds, k_refit, k_gather).
Outputs are checked before anything is reported: on every frame, the refitted tree's hits equal the fresh commit's bit for
bit on the timed rays. Reported: median and range over the repetitions, after warm-up.
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


def time_op(ctx, op, reps, warmup):
    """op() ends in a commit (which synchronises): (device ms = build_ms, host wall ms) per repetition."""
    dev, wall = [], []
    for k in range(warmup + reps):
        t0 = time.perf_counter()
        op()
        t1 = time.perf_counter()
        if k >= warmup:
            dev.append(ctx.stats().build_ms)
            wall.append((t1 - t0) * 1e3)
    return dict(device_ms=stat(dev), wall_ms=stat(wall))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=11)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--json", default="", help="also write the results to this file")
    args = ap.parse_args()
    assert args.reps >= 5, "at least 5 timed repetitions"

    import torch
    if not torch.cuda.is_available():
        sys.exit("refit_bench.py measures on the GPU and found no CUDA device")
    import ptb200
    L = ptb200._lib
    mg = ptb200.meshgen

    name, power = device_identity(torch)
    print(f"device: {name}, power limit {power}", flush=True)
    R, W = args.reps, args.warmup
    out = dict(device=name, power_limit=power)

    # ---------------------------------------------------------------- C3 operations
    base = mg.c3_scene(1.0)
    frame = mg.c3_deform(base, 0.5, 1.0)
    glass = np.nonzero(base.triangles["material"] == 1)[0]
    g0, g1 = int(glass[0]), int(glass[-1]) + 1
    ctx = ptb200.Context(0)
    ctx.upload(base)
    ops = {}
    ops["full SAH commit"] = time_op(ctx, lambda: ctx.commit(L.BUILD_SAH), R, W)
    ops["full LBVH commit"] = time_op(ctx, lambda: ctx.commit(L.BUILD_BINARY), R, W)
    ctx.commit(L.BUILD_SAH)
    ops["refit, primitives unchanged"] = time_op(ctx, lambda: ctx.commit(L.BUILD_REFIT), R, W)
    d_frame = torch.from_numpy(np.ascontiguousarray(frame.triangles).view(np.uint8)).cuda()
    torch.cuda.synchronize()
    n_tri = len(base.triangles)

    def device_update():
        ctx.update_triangles_device(0, d_frame.data_ptr(), n_tri)
        ctx.commit(L.BUILD_REFIT)
    ops["update_triangles_device (all 1 M) + refit"] = time_op(ctx, device_update, R, W)
    glass_moved = np.ascontiguousarray(frame.triangles[g0:g1])

    def host_update():
        ctx.update_triangles(g0, glass_moved)
        ctx.commit(L.BUILD_REFIT)
    ops[f"update_triangles host ({g1 - g0} glass) + refit, end to end"] = time_op(ctx, host_update, R, W)
    out["c3_ops"] = ops
    refit_ms = ops["refit, primitives unchanged"]["device_ms"]["median"]
    lbvh_ms = ops["full LBVH commit"]["device_ms"]["median"]
    sah_ms = ops["full SAH commit"]["device_ms"]["median"]
    verdict = (f"C3 refit {refit_ms:.3f} ms vs full LBVH commit {lbvh_ms:.3f} ms ({lbvh_ms / refit_ms:.1f}x) and full SAH commit "
               f"{sah_ms:.3f} ms ({sah_ms / refit_ms:.1f}x), device time, same run")
    out["c3_verdict"] = verdict
    print(verdict, flush=True)
    del d_frame

    # ---------------------------------------------------------------- deformation sequence
    n_rays = 1 << 22
    rays_np = mg.philox_rays(n_rays, seed=0x5EED, centre=(0.0, 4.0, 1.0), radius=5.0)
    rays = torch.from_numpy(rays_np.view(np.float32).reshape(n_rays, 8)).cuda()
    hits_r = torch.zeros((n_rays, 4), dtype=torch.float32, device="cuda")
    hits_f = torch.zeros((n_rays, 4), dtype=torch.float32, device="cuda")
    fresh = ptb200.Context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    fresh.set_stream(stream.cuda_stream)
    ctx.upload(base)
    ctx.commit(L.BUILD_SAH)
    opts = ptb200.RenderOptions(samples_per_pixel=32, render_method=L.METHOD_MIS, width=1920, height=1080, seed=1)

    def hit_rate(c, hits):
        for _ in range(W):
            c.closest_hit_device(rays.data_ptr(), n_rays, hits.data_ptr())
        ms = []
        for _ in range(R):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            c.closest_hit_device(rays.data_ptr(), n_rays, hits.data_ptr())
            e1.record(stream)
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return stat([n_rays / (m * 1e-3) for m in ms])

    def counts(c):
        c.set_option(L.OPT_COUNT_TRAVERSAL, 1)
        c.stats_reset()
        c.closest_hit_device(rays.data_ptr(), n_rays, hits_r.data_ptr() if c is ctx else hits_f.data_ptr())
        c.synchronize()
        st = c.stats()
        c.set_option(L.OPT_COUNT_TRAVERSAL, 0)
        return st.nodes_fetched / st.rays_counted, st.prims_tested / st.rays_counted

    def render_rate(c):
        rates = []
        for k in range(1 + 3):
            c.accum_clear()
            c.stats_reset()
            c.render(opts)
            st = c.stats()
            if k >= 1:
                rates.append(st.rays_total / (st.render_ms * 1e-3) / 1e6)
        return stat(rates)

    seq = []
    for wave, shift in ((0.0, 0.0), (0.25, 0.5), (0.5, 1.0), (1.0, 2.0), (2.0, 4.0)):
        fr = mg.c3_deform(base, wave, shift)
        ctx.update_triangles(0, fr.triangles)
        ctx.commit(L.BUILD_REFIT)
        fresh.upload(fr)
        fresh.commit(L.BUILD_SAH)
        rec = dict(wave=wave, shift_radii=shift, refit_ms=ctx.stats().build_ms, fresh_sah_ms=fresh.stats().build_ms,
                   sah_cost_refit=ctx.bvh_sah_cost(), sah_cost_fresh=fresh.bvh_sah_cost())
        rec["rays_per_s_refit"] = hit_rate(ctx, hits_r)
        rec["rays_per_s_fresh"] = hit_rate(fresh, hits_f)
        torch.cuda.synchronize()
        diff = int((hits_r.view(torch.int32) != hits_f.view(torch.int32)).any(1).sum())
        assert diff == 0, f"frame wave={wave} shift={shift}: refitted tree's hits differ from the fresh commit's on {diff} rays"
        rec["VT_refit"] = counts(ctx)
        rec["VT_fresh"] = counts(fresh)
        rec["render_mrays_refit"] = render_rate(ctx)
        rec["render_mrays_fresh"] = render_rate(fresh)
        seq.append(rec)
        print(f"frame wave={wave} shift={shift}r: hits identical on {n_rays} rays; SAH cost {rec['sah_cost_refit']:.2f} refit vs "
              f"{rec['sah_cost_fresh']:.2f} fresh; V/T {rec['VT_refit'][0]:.1f}/{rec['VT_refit'][1]:.2f} vs "
              f"{rec['VT_fresh'][0]:.1f}/{rec['VT_fresh'][1]:.2f}; {rec['rays_per_s_refit']['median'] / 1e9:.3f} vs "
              f"{rec['rays_per_s_fresh']['median'] / 1e9:.3f} G rays/s; render {rec['render_mrays_refit']['median']:.0f} vs "
              f"{rec['render_mrays_fresh']['median']:.0f} Mrays/s", flush=True)
    out["deformation"] = seq
    fresh.close()
    del rays, hits_r, hits_f

    # ---------------------------------------------------------------- kernels: fused refit vs the commit's three kernels
    from torch.profiler import ProfilerActivity, profile
    ctx.upload(base)
    ctx.commit(L.BUILD_BINARY)
    ctx.commit(L.BUILD_REFIT)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            ctx.commit(L.BUILD_BINARY)
            ctx.commit(L.BUILD_REFIT)
        torch.cuda.synchronize()
    kms = {}
    for ev in prof.key_averages():
        for k in ("k_refit_slots", "k_prim_bounds", "k_refit", "k_gather"):
            if re.search(rf"(^|::){k}(\(|<|$)", ev.key) and ev.count:
                kms[k] = dict(mean=ev.device_time_total / ev.count / 1e3, launches=ev.count)   # us -> ms
    out["c3_kernels_ms"] = kms
    if all(k in kms for k in ("k_refit_slots", "k_prim_bounds", "k_refit", "k_gather")):
        three = kms["k_prim_bounds"]["mean"] + kms["k_refit"]["mean"] + kms["k_gather"]["mean"]
        kv = (f"C3 kernels (mean of 5 launches each): k_refit_slots {kms['k_refit_slots']['mean']:.3f} ms vs k_prim_bounds + "
              f"k_refit + k_gather {three:.3f} ms ({three / kms['k_refit_slots']['mean']:.2f}x)")
    else:
        kv = f"C3 kernels: not all kernels found in the profile ({sorted(kms)})"
    out["kernel_verdict"] = kv
    print(kv, flush=True)

    # ---------------------------------------------------------------- C5
    c5 = mg.heightfield_scene(2500, 2000)
    ctx.upload(c5)
    del c5
    c5ops = {}
    c5ops["full SAH commit"] = time_op(ctx, lambda: ctx.commit(L.BUILD_SAH), R, W)
    c5ops["full LBVH commit"] = time_op(ctx, lambda: ctx.commit(L.BUILD_BINARY), R, W)
    ctx.commit(L.BUILD_SAH)
    c5ops["refit, primitives unchanged"] = time_op(ctx, lambda: ctx.commit(L.BUILD_REFIT), R, W)
    out["c5_ops"] = c5ops
    ctx.close()

    print(f"\n| workload | operation | device ms (median, range) | host wall ms (median, range) |  ({name}, power limit {power})")
    print("|---|---|---:|---:|")
    for wl, table in (("C3", ops), ("C5", c5ops)):
        for k, v in table.items():
            d, w = v["device_ms"], v["wall_ms"]
            print(f"| {wl} | {k} | {d['median']:.3f} ({d['min']:.3f} - {d['max']:.3f}) | {w['median']:.3f} ({w['min']:.3f} - {w['max']:.3f}) |")
    print("\n| wave | shift (radii) | SAH cost refit / fresh | V refit / fresh | T refit / fresh | closest hit G rays/s refit / fresh | render Mrays/s refit / fresh |")
    print("|---:|---:|---:|---:|---:|---:|---:|")
    for r in seq:
        print(f"| {r['wave']} | {r['shift_radii']} | {r['sah_cost_refit']:.2f} / {r['sah_cost_fresh']:.2f} | {r['VT_refit'][0]:.1f} / "
              f"{r['VT_fresh'][0]:.1f} | {r['VT_refit'][1]:.2f} / {r['VT_fresh'][1]:.2f} | {r['rays_per_s_refit']['median'] / 1e9:.3f} / "
              f"{r['rays_per_s_fresh']['median'] / 1e9:.3f} | {r['render_mrays_refit']['median']:.0f} / {r['render_mrays_fresh']['median']:.0f} |")
    print(verdict)
    print(kv)
    print(json.dumps(out))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
