#!/usr/bin/env python
"""Rays/s of the denoiser feature buffers (ptb_render_aov: k_aov) beside closest hit (ptb_closest_hit_device:
k_closest_hit_api) on the same camera rays, on the GPU only (no device: it fails).

  python scripts/aov_bench.py [--reps 20] [--warmup 3] [--json FILE] [--md FILE]

Workloads: C3 (the 1 M-triangle mesh, meshgen.c3_scene) and C5 (the 10 M-triangle heightfield, meshgen.heightfield_scene)
at 1920 x 1080, on the library's default tree. One AOV sample = one ptb_render_aov call of samples_per_pixel = 1 (a 4-byte
memset of its work cursor and one k_aov launch over the 2 073 600 pixels), each call timed alone with CUDA events after
warm-up calls; successive calls take successive samples (sample_offset) and keep adding into the AOV sums. Closest hit is
timed on the camera rays of sample 0, built on the host with the render's jitter (Philox) and camera arithmetic and
resident on the device before timing; its time includes its own ray ordering (batches of >= 65 536 rays are sorted).
Before anything is reported, the AOV depth of sample 0 must equal the closest-hit t of those rays bit for bit on every
pixel (and its coverage the hit mask). Reported: median and range over the repetitions; the card's name and power limit
are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from visibility_bench import device_identity, row, timed  # noqa: E402

W, H = 1920, 1080


def camera_rays(ptb, scene, seed, sample):
    """The render's camera rays of `sample` for every pixel (row-major), as (W*H, 8) float32 ray records with the
    un-normalised direction (the library normalises it once, as the render does)."""
    cam = scene.camera[0]
    f = np.float32
    pix = np.arange(W * H, dtype=np.uint64)
    r0, r1, _, _ = ptb.meshgen.philox4x32_10(pix, np.full_like(pix, sample), np.zeros_like(pix), np.zeros_like(pix),
                                             seed & 0xFFFFFFFF, seed >> 32)
    x = (pix % W).astype(np.float32)
    y = (pix // W).astype(np.float32)
    unit = f(1.0 / 16777216.0)
    u = ((np.asarray(r0, np.uint32) >> 8).astype(np.float32) * unit + x) / f(W - 1)
    v = f(1) - ((np.asarray(r1, np.uint32) >> 8).astype(np.float32) * unit + y) / f(H - 1)
    o = np.asarray(cam["origin"], np.float32)
    d = (np.asarray(cam["lower_left"], np.float32) + np.asarray(cam["horizontal"], np.float32) * u[:, None]
         + np.asarray(cam["vertical"], np.float32) * v[:, None] - o)
    rays = np.zeros((W * H, 8), np.float32)
    rays[:, 0:3] = o
    rays[:, 4:7] = d
    return rays


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--json", default="", help="also write the result rows to this file")
    ap.add_argument("--md", default="", help="also write the table to this file")
    args = ap.parse_args()
    assert args.reps >= 5, "at least 5 timed repetitions"

    import torch
    if not torch.cuda.is_available():
        sys.exit("aov_bench.py measures on the GPU and found no CUDA device")
    import ptb200
    L = ptb200._lib

    name, power = device_identity(torch)
    print(f"device: {name}, power limit {power}", flush=True)
    ctx = ptb200.Context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    rows = []
    seed = 0x5EED
    n = W * H
    for wl, make in (("c3", lambda: ptb200.meshgen.c3_scene(1.0)), ("c5", lambda: ptb200.meshgen.heightfield_scene(2500, 2000))):
        scene = make()
        ctx.upload(scene)
        ctx.commit()
        rays = torch.from_numpy(camera_rays(ptb200, scene, seed, 0)).cuda()
        hits = torch.zeros((n, 4), dtype=torch.float32, device="cuda")
        rows.append(row(wl, "closest_hit (camera rays of one sample)", n,
                        timed(torch, stream, lambda: ctx.closest_hit_device(rays.data_ptr(), n, hits.data_ptr()), args.reps, args.warmup)))
        ctx.aov_clear()
        ctx.render_aov(ptb200.RenderOptions(samples_per_pixel=1, width=W, height=H, seed=seed))
        depth = torch.from_numpy(ctx.aov_read(W, H, L.PTB_AOV_DEPTH).reshape(-1)).cuda()
        cov = torch.from_numpy(ctx.aov_read(W, H, L.PTB_AOV_COVERAGE).reshape(-1)).cuda()
        hit = hits[:, 1].view(torch.int32) != -1
        want = torch.where(hit, hits[:, 0], torch.zeros_like(hits[:, 0]))
        assert torch.equal(depth.view(torch.int32), want.view(torch.int32)), f"{wl}: AOV depth differs from closest-hit t"
        assert torch.equal(cov, hit.float()), f"{wl}: AOV coverage differs from the closest-hit mask"
        print(f"check: {wl} AOV depth == closest-hit t bit for bit on all {n} camera rays ({float(hit.float().mean()):.4f} hit)",
              flush=True)
        k = [1]

        def one_sample():
            ctx.render_aov(ptb200.RenderOptions(samples_per_pixel=1, sample_offset=k[0], width=W, height=H, seed=seed))
            k[0] += 1

        rows.append(row(wl, "render_aov (one sample)", n, timed(torch, stream, one_sample, args.reps, args.warmup)))
        del rays, hits, depth, cov, scene

    lines = [f"| workload | case | rays | median rays/s | range (min - max) | median ms |",
             "|---|---|---:|---:|---|---:|"]
    for r in rows:
        lines.append(f"| {r['workload']} | {r['case']} | {r['rays']} | {r['median_rays_per_s'] / 1e9:.3f} G | "
                     f"{r['min_rays_per_s'] / 1e9:.3f} - {r['max_rays_per_s'] / 1e9:.3f} G | {r['median_ms']:.3f} |")
    print(f"\n({name}, power limit {power})")
    print("\n".join(lines))
    for r in rows:
        print(json.dumps(dict(r, device=name, power_limit=power)))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(device=name, power_limit=power, width=W, height=H, rows=rows), f, indent=1)
    if args.md:
        with open(args.md, "w") as f:
            f.write(f"Measured on {name}, power limit {power}, with `scripts/aov_bench.py --reps {args.reps} --warmup {args.warmup}`.\n\n")
            f.write("\n".join(lines) + "\n")
    ctx.close()


if __name__ == "__main__":
    main()
