"""GPU only: camera candidate lists (csrc/ptb_camcand.cuh) against the parent build, on the card this runs on.

    python scripts/camcand_bench.py --base DIR [--reps 3] [--md profiles/camcand_b200.md] [--json profiles/camcand_b200.json]

DIR is a built checkout of the parent commit. Alternating the two builds, `reps` times each:
  * `bench.py --gpus 1 --no-cpu` (the default C3 line: 1920 x 1080, 256 spp per step, naive; with extra.c1_mis, c2_mis, c5)
  * `bench.py --gpus 1 --no-cpu --no-c5-leg --spp-per-step 32` (a rank's share of the default at N = 8)
then `bench.py --dump-outputs` once per build (the images must agree within the float summation order), and one C3 call
of each config per build under torch.profiler: time of the camera launches (k_trace_camera) and of k_cam_candidates.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def device_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return q


def bench(tree, extra_args, env=None):
    cmd = [sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--no-cpu"] + extra_args
    r = subprocess.run(cmd, cwd=tree, capture_output=True, text=True, env=env)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode != 0 or not lines:
        raise RuntimeError(f"{cmd} failed ({r.returncode}):\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}")
    return json.loads(lines[-1])


def profile_child(spp, reps):
    """Runs in a subprocess whose PTB200_LIB names the build: kernel times of one C3 call of `spp` samples per pixel."""
    sys.path.insert(0, ROOT)
    import torch
    from torch.profiler import ProfilerActivity, profile
    import ptb200
    L = ptb200._lib
    ctx = ptb200.Context(0)
    ctx.upload(ptb200.meshgen.c3_scene(1.0))
    ctx.commit(L.BUILD_SAH)
    o = ptb200.RenderOptions(samples_per_pixel=spp, render_method=ptb200.METHOD_NAIVE, width=1920, height=1080, seed=1)
    for _ in range(2):
        ctx.render(o)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ctx.render(o)
        torch.cuda.synchronize()
    out = {}
    for name in ("k_trace_camera", "k_cam_candidates", "k_trace", "k_shade"):
        ts = [e.device_time / 1e3 for e in prof.events() if re.search(rf"(^|::){name}(\(|<|$)", e.name)]
        out[name] = {"ms_per_call": sum(ts) / reps, "launches_per_call": len(ts) / reps}
    ctx.close()
    print(json.dumps(out))


def profile_build(tree, spp, reps):
    env = dict(os.environ, PTB200_LIB=os.path.join(tree, "raytracing-rust_b200", "libptb200.so"))
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--profile-child", str(spp), "--reps", str(reps)], cwd=ROOT,
                       capture_output=True, text=True, env=env)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode != 0 or not lines:
        raise RuntimeError(f"profile of {tree} failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}")
    return json.loads(lines[-1])


def stats(xs):
    a = np.asarray(xs, float)
    return {"mean": float(a.mean()), "min": float(a.min()), "max": float(a.max()), "values": [float(x) for x in a]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", default="")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--md", default="")
    ap.add_argument("--json", default="")
    ap.add_argument("--profile-child", type=int, default=0)
    a = ap.parse_args()
    if a.profile_child:
        profile_child(a.profile_child, a.reps)
        return
    builds = {"parent": os.path.abspath(a.base), "lists": ROOT}
    dev = device_identity()
    print(f"device: {dev}", flush=True)
    configs = {"default": [], "spp32": ["--no-c5-leg", "--spp-per-step", "32"]}
    res = {b: {c: [] for c in configs} for b in builds}
    for rep in range(a.reps):
        for b, tree in builds.items():
            for c, args in configs.items():
                line = bench(tree, args)
                res[b][c].append(line)
                print(f"rep {rep} {b:6s} {c:7s} {line['value']:.1f} Mrays/s", flush=True)
    summary = {}
    for b in builds:
        summary[b] = {c: stats([l["value"] for l in res[b][c]]) for c in configs}
        for k in ("c1_mis", "c2_mis", "c5"):
            summary[b][k] = stats([l["extra"][k]["value"] for l in res[b]["default"]])
    # outputs of the two builds
    diffs = {}
    with tempfile.TemporaryDirectory() as td:
        for b, tree in builds.items():
            bench(tree, ["--no-c5-leg", "--steps", "1", "--warmup", "1", "--no-e2e", "--dump-outputs", os.path.join(td, b)])
        for f in sorted(os.listdir(os.path.join(td, "parent"))):
            x, y = np.load(os.path.join(td, "parent", f)), np.load(os.path.join(td, "lists", f))
            diffs[f] = {"shape": list(x.shape), "max_abs_diff": float(np.abs(x.astype(np.float64) - y).max()),
                        "allclose_1e-5": bool(np.allclose(x, y, rtol=1e-5, atol=1e-5))}
    prof = {b: {spp: profile_build(tree, spp, 3) for spp in (256, 32)} for b, tree in builds.items()}
    out = {"device": dev, "reps": a.reps, "summary": summary, "outputs": diffs, "kernels": prof,
           "lines": {b: {c: res[b][c] for c in configs} for b in builds}}
    print(json.dumps({"summary": summary, "outputs": diffs, "kernels": prof}, indent=1))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)
    if a.md:
        def row(name, key):
            p, n = summary["parent"][key], summary["lists"][key]
            return (f"| {name} | {p['mean']:.1f} ({p['min']:.1f} – {p['max']:.1f}) | {n['mean']:.1f} ({n['min']:.1f} – {n['max']:.1f}) "
                    f"| {100.0 * (n['mean'] / p['mean'] - 1.0):+.1f} % |")
        lines = [f"# Camera candidate lists on B200\n",
                 f"Measured on {dev} (name, power limit, max SM clock) with `scripts/camcand_bench.py --reps {a.reps}`: the parent "
                 "build and this one alternated, each line `bench.py --gpus 1 --no-cpu` (the CPU baseline leg skipped).\n",
                 "| line | parent: mean (min – max) | lists: mean (min – max) | change |", "|---|---|---|---|",
                 row("default C3 (256 spp per step), Mrays/s", "default"), row("C3 `--spp-per-step 32`, Mrays/s", "spp32"),
                 row("extra.c1_mis", "c1_mis"), row("extra.c2_mis", "c2_mis"), row("extra.c5", "c5"), "",
                 "## Kernel times per 1920 x 1080 C3 call (torch.profiler, 3 calls after 2 warm-up calls)\n",
                 "| build | spp | k_trace_camera ms (launches) | k_cam_candidates ms (launches) | k_trace ms | k_shade ms |",
                 "|---|---|---|---|---|---|"]
        for b in builds:
            for spp in (256, 32):
                k = prof[b][spp]
                lines.append(f"| {b} | {spp} | {k['k_trace_camera']['ms_per_call']:.2f} ({k['k_trace_camera']['launches_per_call']:.0f}) "
                             f"| {k['k_cam_candidates']['ms_per_call']:.2f} ({k['k_cam_candidates']['launches_per_call']:.0f}) "
                             f"| {k['k_trace']['ms_per_call']:.2f} | {k['k_shade']['ms_per_call']:.2f} |")
        lines += ["", "## Outputs (`bench.py --dump-outputs`, one step each)\n", "| array | max abs diff | allclose 1e-5 |", "|---|---|---|"]
        for f, d in diffs.items():
            lines.append(f"| {f} {d['shape']} | {d['max_abs_diff']:.3g} | {d['allclose_1e-5']} |")
        with open(a.md, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
