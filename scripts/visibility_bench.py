#!/usr/bin/env python
"""Rays/s of the batch visibility queries (ptb_occluded_device, ptb_check_hit_index_device: k_visibility_api) beside closest
hit (ptb_closest_hit_device) on the same rays, on the GPU only (no device: it fails).

  python scripts/visibility_bench.py [--reps 7] [--warmup 2] [--json FILE]

C5: the 10 M-triangle heightfield, the first 2^24 rays of the Philox stream (meshgen.philox_rays, generated on the device):
    closest hit; occlusion at tmax = +inf (the walk stops at the first blocker); occlusion at tmax = 0.5 t_closest (nothing
    can block: the full walk up to tmax); check_hit_index towards each ray's closest primitive over the rays that hit (all
    visible), with closest hit timed on the same subset.
C3: the 1 M-triangle mesh; shadow rays from the terrain hit points of 2^22 camera rays towards random points on the glass
    sphere, through occlusion (tmax = distance to the point, the terrain triangle excluded) and check_hit_index (the
    glass triangle the point lies on).
Inputs are seeded and resident on the device (512 MiB of C5 rays, more than L2); every launch is timed alone with CUDA events
after warm-up launches; reported: median and range over the repetitions. Outputs are checked before anything is reported:
occlusion at +inf must equal "closest hit found something" on every C5 ray, occlusion at 0.5 t_closest must be all clear,
and check_hit_index must reproduce the closest-hit records bit for bit.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MISS = 0xFFFFFFFF


def device_identity(torch):
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def timed(torch, stream, fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


def row(workload, case, n, ms):
    rates = sorted(n / (m * 1e-3) for m in ms)
    return dict(workload=workload, case=case, rays=n, reps=len(ms), median_rays_per_s=float(np.median(rates)),
                min_rays_per_s=rates[0], max_rays_per_s=rates[-1], median_ms=float(np.median(ms)))


def occlusion_records(torch, rays8, tmax, exclude):
    """(n, 8) float32 ray records -> ptb_occlusion_ray records (tmax in .w of the origin, exclude bits in .w of the direction)."""
    q = rays8.clone()
    q[:, 3] = tmax
    q.view(torch.int32)[:, 7] = exclude.to(torch.int32) if torch.is_tensor(exclude) else (exclude ^ 0x80000000) - 0x80000000
    return q


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--json", default="", help="also write the result rows to this file")
    args = ap.parse_args()
    assert args.reps >= 5, "at least 5 timed repetitions"

    import torch
    if not torch.cuda.is_available():
        sys.exit("visibility_bench.py measures on the GPU and found no CUDA device")
    import ptb200
    from bench import philox_rays_device

    name, power = device_identity(torch)
    print(f"device: {name}, power limit {power}", flush=True)
    ctx = ptb200.Context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    rows = []
    R, W = args.reps, args.warmup

    # ---- C5
    scene = ptb200.meshgen.heightfield_scene(2500, 2000)
    ctx.upload(scene)
    ctx.commit()
    del scene
    n = 1 << 24
    rays = philox_rays_device(n, 0, "cuda")
    chk = ptb200.meshgen.philox_rays(4096)
    got = rays[:4096].cpu().numpy()
    assert max(np.max(np.abs(got[:, 0:3] - chk["o"])), np.max(np.abs(got[:, 4:7] - chk["d"]))) < 1e-5, "ray stream"
    hits = torch.zeros((n, 4), dtype=torch.float32, device="cuda")
    occ = torch.zeros(n, dtype=torch.uint8, device="cuda")
    rows.append(row("c5", "closest_hit", n, timed(torch, stream, lambda: ctx.closest_hit_device(rays.data_ptr(), n, hits.data_ptr()), R, W)))
    t_c = hits[:, 0].clone()
    prim = hits[:, 1].view(torch.int32).clone()
    hit = prim != -1
    q_inf = occlusion_records(torch, rays, float("inf"), MISS)
    rows.append(row("c5", "occluded tmax=+inf", n, timed(torch, stream, lambda: ctx.occluded_device(q_inf.data_ptr(), n, occ.data_ptr()), R, W)))
    mism = int(((occ != 0) != hit).sum())
    assert mism == 0, f"occluded(+inf) differs from closest hit on {mism} of {n} C5 rays"
    print(f"check: occluded(+inf) == (closest.prim != PTB_MISS) on all {n} C5 rays ({float(hit.float().mean()):.4f} hit)", flush=True)
    del q_inf
    q_half = occlusion_records(torch, rays, 0.5 * t_c, MISS)
    rows.append(row("c5", "occluded tmax=0.5*t_closest", n, timed(torch, stream, lambda: ctx.occluded_device(q_half.data_ptr(), n, occ.data_ptr()), R, W)))
    assert int(occ.sum()) == 0, "occluded(0.5 t_closest) found a blocker before the closest hit"
    print("check: occluded(0.5 * t_closest) is clear on every C5 ray", flush=True)
    del q_half
    sub = rays[hit].contiguous()
    idx = prim[hit].contiguous()
    m = sub.shape[0]
    sub_hits = torch.zeros((m, 4), dtype=torch.float32, device="cuda")
    chi = torch.zeros((m, 4), dtype=torch.float32, device="cuda")
    rows.append(row("c5", "closest_hit (rays that hit)", m, timed(torch, stream, lambda: ctx.closest_hit_device(sub.data_ptr(), m, sub_hits.data_ptr()), R, W)))
    rows.append(row("c5", "check_hit_index -> closest prim (all visible)", m,
                    timed(torch, stream, lambda: ctx.check_hit_index_device(sub.data_ptr(), idx.data_ptr(), m, chi.data_ptr()), R, W)))
    assert torch.equal(chi.view(torch.int32), hits[hit].view(torch.int32)), "check_hit_index differs from the closest-hit records"
    print(f"check: check_hit_index(closest.prim) reproduces the closest-hit records bit for bit on {m} C5 rays", flush=True)
    del rays, hits, occ, sub, idx, sub_hits, chi, t_c, prim, hit

    # ---- C3
    scene = ptb200.meshgen.c3_scene(1.0)
    ctx.upload(scene)
    ctx.commit()
    tri_p = torch.from_numpy(np.ascontiguousarray(scene.triangles["p"])).cuda()       # (T, 3, 3)
    glass = np.nonzero(scene.triangles["material"] == 1)[0]
    n_terrain = int(glass[0])
    cam = scene.camera[0]
    g = torch.Generator(device="cuda").manual_seed(7)
    n = 1 << 22
    uv = torch.rand((n, 2), generator=g, device="cuda")
    o = torch.tensor(cam["origin"], device="cuda")
    d = (torch.tensor(cam["lower_left"], device="cuda") + uv[:, :1] * torch.tensor(cam["horizontal"], device="cuda")
         + uv[:, 1:] * torch.tensor(cam["vertical"], device="cuda") - o)
    cam_rays = torch.zeros((n, 8), dtype=torch.float32, device="cuda")
    cam_rays[:, 0:3] = o
    cam_rays[:, 4:7] = d
    cam_hits = torch.zeros((n, 4), dtype=torch.float32, device="cuda")
    ctx.closest_hit_device(cam_rays.data_ptr(), n, cam_hits.data_ptr())
    torch.cuda.synchronize()
    cprim = cam_hits[:, 1].view(torch.int32).to(torch.int64)
    on_terrain = (cprim >= 0) & (cprim < n_terrain)
    dn = d / torch.linalg.norm(d, dim=1, keepdim=True)
    p = o + dn * cam_hits[:, :1]
    p, dn, terrain_prim = p[on_terrain], dn[on_terrain], cprim[on_terrain]
    m = p.shape[0]
    target = torch.randint(int(glass[0]), int(glass[-1]) + 1, (m,), generator=g, device="cuda")
    ab = torch.rand((m, 2), generator=g, device="cuda")
    flip = ab.sum(1, keepdim=True) > 1
    ab = torch.where(flip, 1 - ab, ab)
    tp = tri_p[target]
    pt = tp[:, 0] + ab[:, :1] * (tp[:, 1] - tp[:, 0]) + ab[:, 1:] * (tp[:, 2] - tp[:, 0])
    org = p - 1e-4 * dn
    sd = pt - org
    shadow = torch.zeros((m, 8), dtype=torch.float32, device="cuda")
    shadow[:, 0:3] = org
    shadow[:, 4:7] = sd
    q = occlusion_records(torch, shadow, torch.linalg.norm(sd, dim=1), terrain_prim)
    idx = target.to(torch.int32).contiguous()
    occ = torch.zeros(m, dtype=torch.uint8, device="cuda")
    chi = torch.zeros((m, 4), dtype=torch.float32, device="cuda")
    rows.append(row("c3", "shadow rays: occluded", m, timed(torch, stream, lambda: ctx.occluded_device(q.data_ptr(), m, occ.data_ptr()), R, W)))
    rows.append(row("c3", "shadow rays: check_hit_index", m,
                    timed(torch, stream, lambda: ctx.check_hit_index_device(shadow.data_ptr(), idx.data_ptr(), m, chi.data_ptr()), R, W)))
    vis = chi[:, 1].view(torch.int32) != -1
    assert torch.equal(chi[vis][:, 1].view(torch.int32), idx[vis]), "check_hit_index reports another primitive"
    print(f"c3: {m} shadow rays from terrain hits, {float((occ != 0).float().mean()):.4f} occluded, "
          f"{float(vis.float().mean()):.4f} of the targets visible", flush=True)

    print(f"\n| workload | case | rays | median rays/s | range (min - max) |  ({name}, power limit {power})")
    print("|---|---|---:|---:|---|")
    for r in rows:
        print(f"| {r['workload']} | {r['case']} | {r['rays']} | {r['median_rays_per_s'] / 1e9:.3f} G | "
              f"{r['min_rays_per_s'] / 1e9:.3f} - {r['max_rays_per_s'] / 1e9:.3f} G |")
    for r in rows:
        print(json.dumps(dict(r, device=name, power_limit=power)))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(device=name, power_limit=power, rows=rows), f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
