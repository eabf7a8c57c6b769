#!/usr/bin/env python
"""Cost and quality of motion vectors and the temporal denoiser, on the GPU only (no device: it fails).

  python scripts/temporal_bench.py [--reps 10] [--warmup 2] [--json FILE] [--md FILE]

Time, with CUDA events around each call alone after warm-up calls (the same inputs every call):
  ptb_render_aov at C3 (meshgen.c3_scene(1.0)) 1920 x 1080, 4 spp per call, reported per sample: without a mark (k_aov)
  and with a mark of a slightly moved camera (k_aov_motion: every hit computes its motion);
  ptb_denoise_temporal_device against ptb_denoise_device on C3's sums at 1920 x 1080 and 3840 x 2160, 5 levels, with a
  history in place (every pixel reprojects).
Quality: rtweekend1 at 160 x 90, a static camera, 16 frames of 1 spp with advancing sample_offset: relative MSE (mean of
(x - ref)^2 / (ref^2 + 1e-2)) of the noisy frame, the spatial filter and the temporal filter against a 4096-spp render.
The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from denoise_bench import rel_mse  # noqa: E402
from visibility_bench import device_identity, timed  # noqa: E402


def med(ms):
    return float(np.median(ms))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--json", default="", help="also write the results to this file")
    ap.add_argument("--md", default="", help="also write the tables to this file")
    args = ap.parse_args()
    assert args.reps >= 5, "at least 5 timed repetitions"

    import torch
    if not torch.cuda.is_available():
        sys.exit("temporal_bench.py measures on the GPU and found no CUDA device")
    import ptb200

    name, power = device_identity(torch)
    print(f"device: {name}, power limit {power}", flush=True)
    ctx = ptb200.Context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    res = {"device": name, "power_limit": power, "render_aov": [], "denoise": [], "quality": []}

    # ---- ptb_render_aov with and without motion
    c3 = ptb200.meshgen.c3_scene(1.0)
    moved = copy.deepcopy(c3)
    for k in ("origin", "lower_left"):
        moved.camera[k] = moved.camera[k] + np.float32([0.05, 0.0, 0.02])
    w, h, spp = 1920, 1080, 4
    o = ptb200.RenderOptions(samples_per_pixel=spp, width=w, height=h, seed=11)
    for mark in (False, True):
        c = ptb200.Context(0)
        c.set_stream(stream.cuda_stream)
        c.upload(moved if mark else c3)
        c.commit()
        if mark:
            c.motion_mark()
            c.upload(c3)
            c.commit()
        ms = timed(torch, stream, lambda: c.render_aov(o), args.reps, args.warmup)
        valid = float(np.mean(c.motion_read(w, h)[..., 2] > 0)) if mark else 0.0
        res["render_aov"].append({"mark": mark, "ms_per_call": med(ms), "ms_per_sample": med(ms) / spp,
                                  "pixels_with_motion": valid})
        print(f"render_aov C3 {w}x{h} mark={mark}: {med(ms) / spp:.3f} ms per sample", flush=True)
        c.close()

    # ---- ptb_denoise_temporal against ptb_denoise
    ctx.upload(c3)
    ctx.commit()
    for w, h in ((1920, 1080), (3840, 2160)):
        o = ptb200.RenderOptions(samples_per_pixel=4, width=w, height=h, seed=11)
        ctx.accum_clear()
        ctx.render(o)
        ctx.aov_clear()
        ctx.motion_mark()
        ctx.render_aov(o)
        out = torch.empty(w * h * 3, dtype=torch.float32, device="cuda")
        ctx.denoise_temporal_reset()
        ctx.denoise_temporal(w, h)  # the history every timed call reprojects from
        ms_s = timed(torch, stream, lambda: ctx.denoise_device(out.data_ptr()), args.reps, args.warmup)
        ms_t = timed(torch, stream, lambda: ctx.denoise_temporal_device(out.data_ptr()), args.reps, args.warmup)
        res["denoise"].append({"width": w, "height": h, "ms_spatial": med(ms_s), "ms_temporal": med(ms_t)})
        print(f"denoise {w}x{h}: spatial {med(ms_s):.3f} ms, temporal {med(ms_t):.3f} ms", flush=True)

    # ---- quality over a static sequence
    rt = ptb200.load_file(os.path.join(ROOT, "scenes", "rtweekend1.ssml"))
    ctx.upload(rt)
    ctx.commit()
    w, h = 160, 90
    ctx.accum_clear()
    ctx.render(ptb200.RenderOptions(samples_per_pixel=4096, width=w, height=h, seed=21))
    ref = ctx.accum_read(w, h).copy()
    ctx.denoise_temporal_reset()
    for k in range(16):
        o = ptb200.RenderOptions(samples_per_pixel=1, width=w, height=h, seed=21, sample_offset=10000 + k)
        ctx.accum_clear()
        ctx.render(o)
        ctx.aov_clear()
        ctx.render_aov(o)
        t = ctx.denoise_temporal(w, h)
        ctx.motion_mark()
        q = {"frame": k + 1, "noisy": rel_mse(ctx.accum_read(w, h), ref), "spatial": rel_mse(ctx.denoise(w, h), ref),
             "temporal": rel_mse(t, ref)}
        res["quality"].append(q)
        print(f"frame {k + 1}: rel MSE noisy {q['noisy']:.5f} spatial {q['spatial']:.5f} temporal {q['temporal']:.5f}",
              flush=True)
    ctx.close()

    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)
    if args.md:
        with open(args.md, "w") as f:
            f.write("# Motion vectors and the temporal denoiser on the B200\n\n")
            f.write(f"Measured by `scripts/temporal_bench.py` on {name}, power limit {power}. Median of {args.reps} calls, "
                    "CUDA events around each call alone after warm-up.\n\n")
            f.write("## ptb_render_aov, C3 at 1920 x 1080, 4 spp per call\n\n| mark | ms per sample | pixels with motion |\n|---|---|---|\n")
            for r in res["render_aov"]:
                f.write(f"| {'yes (k_aov_motion)' if r['mark'] else 'no (k_aov)'} | {r['ms_per_sample']:.3f} | "
                        f"{r['pixels_with_motion']:.3f} |\n")
            f.write("\n## ptb_denoise_temporal against ptb_denoise, C3 4 spp sums, 5 levels\n\n"
                    "| size | spatial ms | temporal ms |\n|---|---|---|\n")
            for r in res["denoise"]:
                f.write(f"| {r['width']} x {r['height']} | {r['ms_spatial']:.3f} | {r['ms_temporal']:.3f} |\n")
            f.write("\n## Quality: rtweekend1 160 x 90, static camera, 1 spp per frame, relative MSE against 4096 spp\n\n"
                    "| frame | noisy | spatial | temporal |\n|---|---|---|---|\n")
            for q in res["quality"]:
                f.write(f"| {q['frame']} | {q['noisy']:.5f} | {q['spatial']:.5f} | {q['temporal']:.5f} |\n")


if __name__ == "__main__":
    main()
