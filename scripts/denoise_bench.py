#!/usr/bin/env python
"""Time and quality of the denoiser (ptb_denoise_device: k_denoise_prepare, k_denoise_variance, k_denoise_atrous), on the
GPU only (no device: it fails).

  python scripts/denoise_bench.py [--reps 20] [--warmup 3] [--json FILE] [--md FILE]

Time: C3 (meshgen.c3_scene(1.0)) rendered at 4 spp with its feature buffers at 1920 x 1080 and 3840 x 2160, then
ptb_denoise_device into a torch tensor on the context's stream, each call timed alone with CUDA events after warm-up calls
(the inputs are the same every call, so they stay in L2 as far as they fit). Levels L = 1 .. 5 are timed separately; the
difference of successive L is one à-trous level, and L = 1 less one level is prepare + variance. The bytes model counts
each kernel's compulsory DRAM traffic (every record read and written once; the taps' re-reads are assumed to hit in
L1 / L2) against 7.7 TB/s.
Quality: relative MSE (mean of (x - ref)^2 / (ref^2 + 1e-2)) of the noisy and the denoised image against a 4096-spp render
of the same seed at 1, 4 and 16 spp, on rtweekend1, overshadowed and C3 at 320 x 180; and the two ratios the tests bound
(the furnace's RMSE at 64 x 36 and rtweekend1's relative MSE at 160 x 90, both at 4 spp). The card's name and power limit
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

from visibility_bench import device_identity, timed  # noqa: E402

PEAK_BPS = 7.7e12
# compulsory bytes per pixel of each launch: prepare reads beauty (12) + AOV records (32) and writes e (16), [n | z] (16),
# α (4), gradient (8); variance and a level read [e | var], [n | z], α, gradient (44) and write [e | var] (16); the last
# level reads the albedo record (16) and writes RGB (12) instead
BYTES = {"prepare": 44 + 44, "variance": 44 + 16, "level": 44 + 16, "last_level": 44 + 16 + 12}


def rel_mse(a, ref):
    a, ref = a.astype(np.float64), ref.astype(np.float64)
    return float(np.mean((a - ref) ** 2 / (ref ** 2 + 1e-2)))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--json", default="", help="also write the results to this file")
    ap.add_argument("--md", default="", help="also write the tables to this file")
    args = ap.parse_args()
    assert args.reps >= 5, "at least 5 timed repetitions"

    import torch
    if not torch.cuda.is_available():
        sys.exit("denoise_bench.py measures on the GPU and found no CUDA device")
    import ptb200
    from conftest import furnace_scene

    name, power = device_identity(torch)
    print(f"device: {name}, power limit {power}", flush=True)
    ctx = ptb200.Context(0)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)

    # ---- time
    timing = []
    c3 = ptb200.meshgen.c3_scene(1.0)
    ctx.upload(c3)
    ctx.commit()
    for w, h in ((1920, 1080), (3840, 2160)):
        o = ptb200.RenderOptions(samples_per_pixel=4, width=w, height=h, seed=11)
        ctx.accum_clear()
        ctx.render(o)
        ctx.aov_clear()
        ctx.render_aov(o)
        out = torch.empty(w * h * 3, dtype=torch.float32, device="cuda")
        host = ctx.denoise(w, h)
        ctx.denoise_device(out.data_ptr())
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy().view(np.uint32), host.reshape(-1).view(np.uint32))
        med = {}
        for levels in range(1, 6):
            ms = timed(torch, stream, lambda: ctx.denoise_device(out.data_ptr(), iterations=levels), args.reps, args.warmup)
            med[levels] = float(np.median(ms))
            npx = w * h
            model = (BYTES["prepare"] + BYTES["variance"] + BYTES["level"] * (levels - 1) + BYTES["last_level"]) * npx
            timing.append(dict(width=w, height=h, levels=levels, median_ms=med[levels], min_ms=float(min(ms)),
                               max_ms=float(max(ms)), model_bytes=model, model_ms=model / PEAK_BPS * 1e3))
            print(json.dumps(timing[-1]), flush=True)
        del out

    # ---- quality
    quality = []
    scenes = {"rtweekend1": ptb200.load_file(os.path.join(ROOT, "scenes", "rtweekend1.ssml")),
              "overshadowed": ptb200.load_file(os.path.join(ROOT, "scenes", "overshadowed.ssml")),
              "c3": ptb200.meshgen.c3_scene(1.0)}
    w, h = 320, 180
    for sname, scene in scenes.items():
        ctx.upload(scene)
        ctx.commit()
        ctx.accum_clear()
        ctx.render(ptb200.RenderOptions(samples_per_pixel=4096, width=w, height=h, seed=31))
        ref = ctx.accum_read(w, h).copy()
        for spp in (1, 4, 16):
            o = ptb200.RenderOptions(samples_per_pixel=spp, width=w, height=h, seed=31)
            ctx.accum_clear()
            ctx.render(o)
            ctx.aov_clear()
            ctx.render_aov(o)
            sc_noisy = ctx.accum_read(w, h)
            den = ctx.denoise(w, h)
            quality.append(dict(scene=sname, spp=spp, rel_mse_noisy=rel_mse(sc_noisy, ref), rel_mse_denoised=rel_mse(den, ref)))
            print(json.dumps(quality[-1]), flush=True)

    # ---- the two ratios the tests bound
    f = furnace_scene(ptb200)
    f.set_camera((0, 0, 3), (0, 0, 0), (0, 1, 0), 1e-4)
    ctx.upload(f)
    ctx.commit()
    o = ptb200.RenderOptions(samples_per_pixel=4, width=64, height=36, seed=9)
    ctx.accum_clear()
    ctx.render(o)
    ctx.aov_clear()
    ctx.render_aov(o)
    rm = lambda a: float(np.sqrt(np.mean((a.astype(np.float64) - 0.25) ** 2)))  # noqa: E731
    furnace = dict(rmse_noisy=rm(ctx.accum_read(64, 36)), rmse_denoised=rm(ctx.denoise(64, 36)))
    ctx.upload(scenes["rtweekend1"])
    ctx.commit()
    ctx.accum_clear()
    ctx.render(ptb200.RenderOptions(samples_per_pixel=4096, width=160, height=90, seed=21))
    ref = ctx.accum_read(160, 90).copy()
    o = ptb200.RenderOptions(samples_per_pixel=4, width=160, height=90, seed=21)
    ctx.accum_clear()
    ctx.render(o)
    ctx.aov_clear()
    ctx.render_aov(o)
    rt1 = dict(rel_mse_noisy=rel_mse(ctx.accum_read(160, 90), ref), rel_mse_denoised=rel_mse(ctx.denoise(160, 90), ref))
    print(json.dumps(dict(furnace=furnace, rtweekend1_160x90=rt1)), flush=True)
    ctx.close()

    lines = [f"Measured on {name}, power limit {power}, with `scripts/denoise_bench.py --reps {args.reps} --warmup {args.warmup}`.",
             "", "| image | levels | median ms | range (min - max) ms | model bytes | model ms at 7.7 TB/s | share of the bound |",
             "|---|---:|---:|---|---:|---:|---:|"]
    for t in timing:
        lines.append(f"| {t['width']} x {t['height']} | {t['levels']} | {t['median_ms']:.3f} | {t['min_ms']:.3f} - {t['max_ms']:.3f} | "
                     f"{t['model_bytes'] / 1e6:.0f} MB | {t['model_ms']:.3f} | {t['model_ms'] / t['median_ms'] * 100:.0f} % |")
    lines += ["", "| scene (320 x 180) | spp | rel. MSE noisy | rel. MSE denoised | ratio |", "|---|---:|---:|---:|---:|"]
    for q in quality:
        lines.append(f"| {q['scene']} | {q['spp']} | {q['rel_mse_noisy']:.4g} | {q['rel_mse_denoised']:.4g} | "
                     f"{q['rel_mse_noisy'] / q['rel_mse_denoised']:.2f} x |")
    lines += ["", f"Furnace 64 x 36, 4 spp: RMSE against 0.25 {furnace['rmse_noisy']:.4g} noisy, {furnace['rmse_denoised']:.4g} "
              f"denoised ({furnace['rmse_noisy'] / furnace['rmse_denoised']:.2f} x).",
              f"rtweekend1 160 x 90, 4 spp against 4096 spp: relative MSE {rt1['rel_mse_noisy']:.4g} noisy, "
              f"{rt1['rel_mse_denoised']:.4g} denoised ({rt1['rel_mse_noisy'] / rt1['rel_mse_denoised']:.2f} x)."]
    print("\n".join(lines))
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(dict(device=name, power_limit=power, timing=timing, quality=quality, furnace=furnace,
                           rtweekend1_160x90=rt1), fh, indent=1)
    if args.md:
        with open(args.md, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
