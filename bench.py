#!/usr/bin/env python
"""bench.py — Mrays/s of the path-tracing hot path (BVH traversal + closest hit + scatter loop) on B200.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA backend (one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU algorithm (oracle port) on host cores

Workload (default, BASELINE.json configs[2]): procedurally tessellated 1 000 000-triangle mesh (800k Lambertian
terrain + 200k dielectric UV sphere), 1920x1080, naive integrator (quirk Q4: dielectrics are black under the
reference's MIS), max depth 50. One STEP renders the configuration as BASELINE.json states it: `--spp-per-step` = 256
samples of every pixel IN TOTAL. With N ranks the 256 samples are split N ways (rank r renders absolute samples
[r*256/N, (r+1)*256/N) of every pixel — the reference's only parallel axis splits one image as well,
samplers/random_sampler.rs:41-79) and the per-rank accumulators are combined by ONE reduce(SUM) to rank 0 per step (NCCL
over NVLink): STRONG scaling. `--scaling weak` gives every rank its own 256 spp instead.

A ray = one BVH traversal launched (camera, bounce, light-shadow, sky-shadow each count 1) — SURVEY.md §8(d).

At N = 1 the default run also carries `extra.c5`: BASELINE.json configs[4] (closest-hit microbenchmark, 10 M-triangle
heightfield, 2 x 2^24 incoherent Philox rays) with its own roofline block — the one config where the HBM roofline binds.

`--dump-outputs DIR` writes what the last timed step computed (rank 0) as DIR/<name>.npy, so that two builds run with the
same arguments can be compared output for output: a render workload's mean image (`image`, H x W x 3 float32; above 2^21
pixels a fixed seeded sample of them, `image` N x 3 at `pixel_index`); for closest_hit the hits of the step's rays, above
2^21 rays a fixed seeded sample (`ray_index`, `t`, `prim`, `uv`; a miss is prim 2^32 - 1). 56 MiB at most.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DEFAULT_SPP = {"c3": 256, "rtweekend1": 4096, "overshadowed": 256}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=["c3", "rtweekend1", "overshadowed", "closest_hit"])
    ap.add_argument("--spp-per-step", type=int, default=0,
                    help="samples per pixel one step renders, summed over all ranks (default: the config's own: c3 256, "
                         "rtweekend1 4096, overshadowed 256)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default): the step's spp are split across the ranks; weak: every rank renders them all")
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--method", default="", choices=["", "naive", "mis"])
    ap.add_argument("--rays", type=int, default=100_000_000, help="closest_hit workload: rays in the stream")
    ap.add_argument("--tris", type=int, default=10_000_000, help="closest_hit workload: triangles in the heightfield")
    ap.add_argument("--cpu-spp", type=int, default=0, help="cpu_baseline sample size in spp (0 = auto)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-c5-leg", action="store_true", help="skip extra.c5 (N = 1 default workload only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed to DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


# ---------------------------------------------------------------------------------------------- workloads
def build_workload(args):
    import ptb200

    name = args.workload
    if name == "c3":
        scene = ptb200.meshgen.c3_scene(1.0)
        w, h, method = 1920, 1080, ptb200.METHOD_NAIVE
        label = "c3: 1M-triangle mesh (800k lambertian terrain + 200k dielectric sphere), 1920x1080, naive, depth 50"
    elif name == "rtweekend1":
        scene = ptb200.load_file(os.path.join(ROOT, "scenes", "rtweekend1.ssml"))
        w, h, method = 3840, 2160, ptb200.METHOD_MIS
        label = "c4: scenes/rtweekend1.ssml, 3840x2160, mis, depth 50"
    elif name == "overshadowed":
        scene = ptb200.load_file(os.path.join(ROOT, "scenes", "overshadowed.ssml"))
        w, h, method = 1920, 1080, ptb200.METHOD_MIS
        label = "c2: scenes/overshadowed.ssml, 1920x1080, mis (strict reference semantics, quirk Q3), depth 50"
    else:
        raise SystemExit("closest_hit is handled separately")
    if args.width:
        w = args.width
    if args.height:
        h = args.height
    if args.method:
        method = ptb200.METHOD_NAIVE if args.method == "naive" else ptb200.METHOD_MIS
        label += f" [method overridden: {args.method}]"
    return scene, w, h, method, label


def workload_config(args, scene, w, h, method, label):
    """`config` of the JSON line: what the workload IS. Identical for the CUDA arm and the reference arm (the bounded
    sample the reference arm times per step is described in its cpu_baseline.sample, not here)."""
    spp = args.spp_per_step or DEFAULT_SPP[args.workload]
    return {"workload": label, "width": w, "height": h, "spp_per_step": spp, "method": "naive" if method == 0 else "mis",
            "max_depth": 50, "primitives": int(scene.n_primitives), "n_gpus": args.gpus,
            "parallelism": (f"spp-split x{args.gpus} ({args.scaling} scaling), scene + BVH replicated per GPU, one "
                            "reduce(SUM) of the accumulators per step"),
            "l2": "scene + BVH (1M triangles: 168 MB) plus the resident path state exceed the 126 MB L2; no explicit flush",
            "ray_definition": "one BVH traversal launched (camera + bounce + shadow)"}


def closest_hit_config(args, n_tris):
    return {"workload": f"c5: closest hit, incoherent Philox rays (seed 0x5EED, origin in the radius-2 ball, direction on S^2) "
                        f"vs a {n_tris}-triangle heightfield BVH, intersection only",
            "primitives": int(n_tris), "n_gpus": args.gpus, "parallelism": f"rays sharded x{args.gpus}, BVH replicated",
            "l2": "BVH + triangles (> 1 GB at 10M triangles) and the ray batches exceed the 126 MB L2; no explicit flush"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_evidence(key):
    """What the committed ncu captures say limits a kernel (profiles/ncu_evidence.json, written from the .ncu-rep files by
    scripts/ncu_summary.py). NOT measured by this run — the run only checks that the kernel's share of the step agrees."""
    p = os.path.join(ROOT, "profiles", "ncu_evidence.json")
    try:
        with open(p) as f:
            return json.load(f).get(key)
    except Exception:
        return None


DUMP_ROWS = 1 << 21   # pixels / rays --dump-outputs writes at most: <= 56 MiB in all; a 1920 x 1080 image fits whole


def dump_outputs(out_dir, **arrays):
    """--dump-outputs: every array as out_dir/<name>.npy; float32 stays float32, anything else is written as float64."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def dump_index(n):
    """The rows of an n-row output that --dump-outputs writes: all of them, or a fixed seeded sample of DUMP_ROWS."""
    import numpy as np
    return np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))


def dump_image(out_dir, img):
    """The mean image (H, W, 3) whole, or the pixels of dump_index (`pixel_index` into the row-major H * W pixels)."""
    index = dump_index(img.shape[0] * img.shape[1])
    if len(index) == img.shape[0] * img.shape[1]:
        dump_outputs(out_dir, image=img)
    else:
        dump_outputs(out_dir, pixel_index=index, image=img.reshape(-1, 3)[index])


def dump_hits(out_dir, n, hits_of):
    """The hits of the rays of dump_index(n) in an n-ray step; `hits_of(index)` returns their hit_dtype records."""
    import numpy as np
    index = dump_index(n)
    h = hits_of(index)
    dump_outputs(out_dir, ray_index=index, t=h["t"], prim=h["prim"], uv=np.stack([h["u"], h["v"]], 1))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- CPU legs
def import_oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    return O


def cpu_render_leg(scene, w, h, method, spp, seed=0):
    """The reference's algorithm (oracle port: SAH BVH, BFS candidates, test-all, pass-per-sample driver) on every host
    core, traversal counters off. Returns (rays, seconds, threads, build_seconds)."""
    O = import_oracle()
    o = O.OracleScene(scene)
    _, counts, secs = o.render(w, h, spp, method, seed=seed)
    rays = counts["camera"] + counts["bounce"] + counts["shadow_light"] + counts["shadow_sky"]
    return rays, secs, O.hardware_threads(), o.build_seconds()


def run_reference(args):
    """--impl reference: rank 0 times the oracle port on the host cores; other ranks exit 0 without work.
    The process maps oracle/liboracle.so only: the scene generators are numpy, and SimpleCamera::new is taken from the
    oracle's restatement instead of libptb200.so's host side (asserted below for the default workload)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    O = import_oracle()
    import numpy as np
    import ptb200

    def camera_from_oracle(origin, lookat, vup, hfov_deg, aspect, aperture, focus_dist):
        c = O.camera_make(origin, lookat, vup, hfov_deg, aspect, aperture, focus_dist)
        cam = np.zeros(1, ptb200._lib.camera_dtype)
        for k in ("origin", "lower_left", "horizontal", "vertical"):
            cam[k] = c[k]
        return cam

    ptb200.scene.CAMERA_MAKE = camera_from_oracle
    if args.workload == "closest_hit":
        return run_reference_closest_hit(args, O)
    scene, w, h, method, label = build_workload(args)
    if args.workload == "c3":
        assert not ptb200._lib.is_loaded(), "the reference arm must not map libptb200.so"
    o = O.OracleScene(scene)
    # one step = a bounded sample of the workload: 1 spp of the full-resolution image
    total_rays, total_s = 0, 0.0
    for i in range(args.warmup + args.steps):
        acc, counts, secs = o.render(w, h, 1, method, seed=0, sample_offset=i)
        if i >= args.warmup:
            total_rays += counts["camera"] + counts["bounce"] + counts["shadow_light"] + counts["shadow_sky"]
            total_s += secs
    if args.dump_outputs:
        dump_image(args.dump_outputs, acc)   # the sum of one sample per pixel is its mean
    v = total_rays / total_s / 1e6
    sample = (f"{w}x{h} x 1 spp per step on all host threads; reference SAH BVH (built once in {o.build_seconds():.2f} s, not "
              "timed), BFS un-culled candidates, test-all closest hit")
    print(json.dumps({
        "impl": "reference", "metric": "Mrays/s", "value": v, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_s / args.steps, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, scene, w, h, method, label),
        "cpu_baseline": {"value": v, "unit": "Mrays/s", "cores": O.hardware_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "libptb200_mapped": ptb200._lib.is_loaded(),
    }))


def heightfield_dims(tris):
    rows = max(2, int(round((tris / 2 / 1.25) ** 0.5 * 1.25)))
    cols = max(2, tris // (2 * rows))
    return rows, cols


def run_reference_closest_hit(args, O):
    import ptb200

    rows, cols = heightfield_dims(args.tris)
    scene = ptb200.meshgen.heightfield_scene(rows, cols)
    o = O.OracleScene(scene)
    n = 1 << 18
    total, secs = 0, 0.0
    for i in range(args.warmup + args.steps):
        rays = ptb200.meshgen.philox_rays(n, first=i * n)
        t0 = time.perf_counter()
        hits = o.closest_hit(rays)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            total += n; secs += dt
    if args.dump_outputs:
        dump_hits(args.dump_outputs, n, lambda index: hits[index])
    v = total / secs / 1e6
    sample = f"{n} rays per step on all host threads, reference SAH BVH + BFS candidates"
    print(json.dumps({"impl": "reference", "metric": "Mrays/s", "value": v, "unit": "Mrays/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": closest_hit_config(args, len(scene.triangles)),
                      "cpu_baseline": {"value": v, "unit": "Mrays/s", "cores": O.hardware_threads(), "kind": "port", "sample": sample},
                      "e2e": {"value": v, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


# ---------------------------------------------------------------------------------------------- device ray stream
def philox_rays_device(n, first, device, seed=0x5EED, radius=2.0):
    """The C5 ray stream (meshgen.philox_rays) generated on the device with torch integer ops: same Philox4x32-10 counters
    and the same uniform floats bit for bit; sqrt / cos / sin / cbrt are torch's (<= 2 ulp from the numpy stream, checked on
    the first rays by the caller). Returns an (n, 8) float32 tensor: o.xyz 0 d.xyz 0."""
    import torch

    M32 = 0xFFFFFFFF

    def mulhilo(a: int, b):  # 32 x 32 -> (hi, lo) without overflowing int64
        a0, a1 = a & 0xFFFF, a >> 16
        t = b * a0
        u = b * a1 + (t >> 16)
        return u >> 16, ((u & 0xFFFF) << 16) | (t & 0xFFFF)

    def philox(c0, c1, c2, c3, k0, k1):
        for _ in range(10):
            hi0, lo0 = mulhilo(0xD2511F53, c0)
            hi1, lo1 = mulhilo(0xCD9E8D57, c2)
            c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
            k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
        return c0, c1, c2, c3

    idx = torch.arange(first, first + n, dtype=torch.int64, device=device)
    lo, hi = idx & M32, idx >> 32
    zero = torch.zeros_like(idx)
    a = philox(lo, hi, zero, zero, seed, 0)
    b = philox(lo, hi, zero, zero + 1, seed, 0)
    unit = lambda u: (u >> 8).to(torch.float32) * (1.0 / 16777216.0)

    def sphere(u, v):
        z = 1.0 - 2.0 * u
        r = torch.sqrt(torch.clamp(1.0 - z * z, min=0.0))
        ph = 6.2831855 * v
        return torch.stack([r * torch.cos(ph), r * torch.sin(ph), z], -1)

    out = torch.zeros((n, 8), dtype=torch.float32, device=device)
    rad = radius * torch.pow(unit(a[2]), 1.0 / 3.0)
    out[:, 0:3] = sphere(unit(a[0]), unit(a[1])) * rad[:, None]
    out[:, 4:7] = sphere(unit(b[0]), unit(b[1]))
    return out


# ---------------------------------------------------------------------------------------------- CUDA arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import ptb200

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA arm has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    args.gpus = world

    if args.workload == "closest_hit":
        out = run_closest_hit(args, rank, world, local, args.tris, args.rays, cpu=not args.no_cpu, dump_dir=args.dump_outputs)
        if rank == 0:
            print(json.dumps(out))
        if world > 1:
            dist.destroy_process_group()
        return

    scene, w, h, method, label = build_workload(args)
    S = args.spp_per_step or DEFAULT_SPP[args.workload]
    strong = args.scaling == "strong"
    K, W = args.steps, args.warmup
    ctx = ptb200.Context(local)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.upload(scene)
    ctx.commit()
    build_ms = ctx.stats().build_ms
    n_prims, n_nodes = ctx.bvh_info()
    n_wide, wide_leaf = ctx.bvh_wide_info()
    tree_label = binary_tree_label(ctx)
    if strong:
        my_off, my_spp = ptb200.shard_samples(S, rank, world)
        step_span = S
    else:
        my_off, my_spp = rank * S, S
        step_span = S * world
    if my_spp == 0:
        raise SystemExit(f"bench.py: {S} spp cannot be split over {world} ranks (the image-tile axis is ptb_render_multi's)")

    def step(i, reduce=True, spp=None, w_=w, h_=h):
        """One step: this rank's share of the step's samples of every pixel + the reduce to rank 0."""
        ctx.accum_clear()
        ctx.render(ptb200.RenderOptions(samples_per_pixel=spp or my_spp, sample_offset=i * step_span + my_off,
                                        render_method=method, width=w_, height=h_, seed=0))
        if world > 1 and reduce:
            acc = ptb200.accumulator_tensor(ctx)
            dist.reduce(acc, dst=0, op=dist.ReduceOp.SUM)

    for i in range(W):
        step(i)
    torch.cuda.synchronize()

    # ---- timed region: device time with CUDA events on the launching stream; max over ranks
    ctx.set_option(ptb200._lib.OPT_TIME_KERNELS, 1)
    ctx.stats_reset()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record(stream)
    for i in range(K):
        step(W + i)
    e1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = e0.elapsed_time(e1)
    st = ctx.stats()
    ctx.set_option(ptb200._lib.OPT_TIME_KERNELS, 0)
    if args.dump_outputs and rank == 0:   # rank 0's accumulator holds the reduced sums of all step_span samples
        ctx.accum_set_samples(step_span)
        dump_image(args.dump_outputs, ctx.accum_read(w, h, normalise=True))
    t = torch.tensor([dev_ms, float(st.rays_total), float(st.kernel_launches)], dtype=torch.float64, device="cuda")
    tmax = t.clone()
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    total_ms = float(tmax[0])
    total_rays = float(t[1])
    value = total_rays / (total_ms * 1e-3) / 1e6

    # ---- V and T of the closest-hit kernel (k_trace): one untimed counted step
    ctx.set_option(ptb200._lib.OPT_COUNT_TRAVERSAL, 1)
    ctx.stats_reset()
    step(W + K, reduce=False, spp=min(my_spp, 16))
    torch.cuda.synchronize()
    sc = ctx.stats()
    ctx.set_option(ptb200._lib.OPT_COUNT_TRAVERSAL, 0)
    V = sc.nodes_fetched / max(sc.rays_counted, 1)
    T = sc.prims_tested / max(sc.rays_counted, 1)

    # ---- N-GPU == 1-GPU, on the hardware the scaling run uses: a small image of the same scene rendered (a) sharded over
    # all ranks + reduce and (b) by rank 0 alone with the same absolute sample set
    multi_diff = None
    if world > 1:
        sw, sh, sspp = 480, 270, 2 * world
        o0, n0 = ptb200.shard_samples(sspp, rank, world)
        ctx.accum_clear()
        ctx.render(ptb200.RenderOptions(samples_per_pixel=n0, sample_offset=o0, render_method=method, width=sw, height=sh, seed=7))
        acc = ptb200.accumulator_tensor(ctx)
        dist.reduce(acc, dst=0, op=dist.ReduceOp.SUM)
        torch.cuda.synchronize()
        if rank == 0:
            ctx.accum_set_samples(sspp)
            sharded = ctx.accum_read(sw, sh, normalise=True).copy()
            ctx.accum_clear()
            ctx.render(ptb200.RenderOptions(samples_per_pixel=sspp, sample_offset=0, render_method=method, width=sw, height=sh, seed=7))
            alone = ctx.accum_read(sw, sh, normalise=True)
            multi_diff = float(np.max(np.abs(sharded - alone)))
        dist.barrier()

    # ---- e2e: the public API with HOST buffers, every step: scene upload + BVH build + render + reduce + read-back
    e2e = None
    if not args.no_e2e:
        import copy

        pins = []

        def pinned_like(a):
            t_ = torch.empty(max(a.nbytes, 1), dtype=torch.uint8, pin_memory=True)
            v = np.frombuffer(t_.numpy().data, dtype=a.dtype, count=len(a))
            v[...] = a
            pins.append(t_)
            return v

        hscene = copy.copy(scene)      # the step's inputs live in pinned host memory
        hscene.spheres, hscene.triangles = pinned_like(scene.spheres), pinned_like(scene.triangles)
        himg_t = torch.empty(w * h * 3, dtype=torch.float32, pin_memory=True)
        himg = himg_t.numpy()
        k2 = max(1, min(K, 4))
        rays2 = 0
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        phase = [0.0, 0.0, 0.0, 0.0, 0.0]  # host wall clock per phase (no extra synchronisation: a phase ends where its call returns)
        for i in range(k2):
            ta = time.perf_counter()
            ctx.stats_reset()
            ctx.upload(hscene)   # same context: ptb_scene_set_* + commit rebuild everything device-side
            tb = time.perf_counter()
            ctx.commit()
            tc = time.perf_counter()
            step(W + K + 1 + i)
            if rank == 0:
                td = time.perf_counter()
                ctx.accum_read(w, h, normalise=False, out=himg)
            else:
                ctx.synchronize()
                td = time.perf_counter()
            te = time.perf_counter()
            st2 = ctx.stats()
            rays2 += st2.rays_total
            for k_, (a_, b_) in enumerate(((ta, tb), (tb, tc), (tc, td), (td, te))):
                phase[k_] += b_ - a_
            phase[4] += 1e-3 * st2.render_ms   # ptb_render alone, CUDA events inside the library
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt, float(rays2)], dtype=torch.float64, device="cuda")
        tm = torch.tensor([dt] + phase, dtype=torch.float64, device="cuda")
        t_rank0 = tm.clone()
        if world > 1:
            dist.broadcast(t_rank0, src=0)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        e2e = {"value": float(tt[1]) / float(tm[0]) / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": scene.nbytes(),
               "d2h_bytes_per_step": w * h * 3 * 4, "steps": k2,
               "includes": "ptb_scene_set_* (pinned host arrays) + ptb_scene_commit (BVH build) + ptb_render + reduce + ptb_accum_read",
               "ms_per_step_by_phase": {n_: {"rank0": 1e3 * float(t_rank0[1 + k_]) / k2, "max_over_ranks": 1e3 * float(tm[1 + k_]) / k2}
                                        for k_, n_ in enumerate(("scene_set", "commit", "render_and_reduce" if world > 1 else "render",
                                                                 "accum_read_or_sync", "ptb_render_device"))}}

    ctx.close()
    del ctx

    # ---- CPU baseline (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        spp_cpu = args.cpu_spp or max(1, int(round(32.0e6 / (w * h))))  # ~10 s of host work on C3
        rays_c, secs_c, cores, build_s = cpu_render_leg(scene, w, h, method, spp_cpu)
        cpu = {"value": rays_c / secs_c / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
               "sample": f"{w}x{h} x {spp_cpu} spp, reference SAH BVH (built in {build_s:.2f} s, not timed), {secs_c:.1f} s, "
                         "traversal counters off"}

    # ---- extra.c5 (N = 1, default workload): the config where the HBM roofline applies, driver-run
    extra = {}
    if world == 1 and args.workload == "c3" and not args.no_c5_leg:
        try:
            extra["c5"] = run_closest_hit(args, rank, world, local, 10_000_000, 2 << 24, cpu=False, steps=2, warmup=3)
        except Exception as exc:  # the leg must not take the headline down with it
            extra["c5"] = {"error": repr(exc)}

    # ---- extra.c1_mis / extra.c2_mis (N = 1, default workload): BASELINE configs[0] and [1], the MIS integrator on the two
    # shipped scenes, bounded (a fraction of a second each) so that they are driver-run beside the headline
    if world == 1 and args.workload == "c3" and not args.no_c5_leg:
        for key, leg in (("c1_mis", ("rtweekend1", 800, 450, 64, 1)), ("c2_mis", ("overshadowed", 1920, 1080, 256, 1))):
            try:
                extra[key] = run_render_leg(local, *leg)
            except Exception as exc:  # a leg must not take the headline down with it
                extra[key] = {"error": repr(exc)}

    if rank == 0:
        peak, peak_src = measured_peaks()
        # Algorithmic bytes of a closest-hit traversal (SURVEY.md §8d): 32 B ray in + 16 B hit out + V nodes + T primitives
        node_bytes = 96.0 if n_wide else 64.0   # compressed 8-wide node / binary node holding both children's boxes
        b_ray = 48.0 + V * node_bytes + T * 48.0
        traced = st.rays_camera + st.rays_bounce
        ms_by_kernel = {"k_trace": st.ms_trace, "k_shade": st.ms_shade, "k_shadow": st.ms_shadow, "bookkeeping": st.ms_generate,
                        "k_tail": st.ms_tail}
        dominant = max(("k_trace", "k_shade"), key=lambda k: ms_by_kernel[k])
        ev = ncu_evidence(f"{args.workload}:{dominant}") or {}
        alg_gbs = traced * b_ray / (st.ms_trace * 1e-3) / 1e9 if st.ms_trace > 0 else 0.0
        roofline = {
            # The binding resource is NOT hbm on this workload: the 1M-triangle scene is L1/L2 resident (ncu: DRAM at a few
            # per cent of peak). What binds is named by the committed ncu capture and reported as measured THERE; this run
            # contributes the live kernel times, the kernel's share of the step and V / T.
            "kernel": dominant, "bound": ev.get("bound", "unprofiled"), "achieved": ev.get("achieved"), "peak": ev.get("peak"),
            "unit": ev.get("unit"), "frac": ev.get("frac"), "frac_source": ev.get("source", "no ncu capture committed for this workload"),
            "traffic": ev.get("dram_bytes_per_launch"), "traffic_source": ev.get("traffic_source"),
            "limiter": ev.get("limiter"),
            # secondary, live: algorithmic bytes of k_trace against the HBM peak (> 1 means served from cache; not a fraction)
            "hbm_algorithmic_ratio": alg_gbs / peak, "hbm_algorithmic_gbs": alg_gbs, "hbm_peak_gbs": peak, "peak_source": peak_src,
            "bytes_per_ray": b_ray, "nodes_per_ray": V, "prims_per_ray": T,
            "ms_by_kernel": ms_by_kernel, "dominant_kernel_share_of_step": ms_by_kernel[dominant] / dev_ms if dev_ms else None,
            "k_trace_launches": int(st.trace_launches), "rays_traced": int(traced)}
        cfg = workload_config(args, scene, w, h, method, label)
        out = {
            "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "e2e": e2e, "gpu_launches": int(st.kernel_launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "run": {"spp_this_rank": my_spp, "bvh": (f"compressed 8-wide, {n_wide} nodes x 96 B, leaf groups <= {wide_leaf}" if n_wide
                                                     else f"binary, {tree_label}, {n_nodes} nodes x 64 B"),
                    "bvh_nodes": n_wide or n_nodes, "node_bytes": node_bytes, "bvh_build_ms": build_ms, "rays_reference_style": st.rays_reference,
                    "wall_s": t_wall, "wavefront_iterations": int(st.wavefront_iterations)},
        }
        if multi_diff is not None:
            out["multi_gpu_image_max_abs_diff"] = multi_diff
            out["multi_gpu_image_check"] = f"480x270 x {2 * world} spp of the same scene: {world} ranks + reduce vs rank 0 alone, normalised radiance"
        if extra:
            out["extra"] = extra
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def run_render_leg(local, workload, w, h, spp, method, steps=3, warmup=3):
    """A bounded device-timed leg of another BASELINE render config inside the default run (extra.c1_mis / extra.c2_mis):
    the same measurement as the headline (CUDA events around `steps` renders of `spp` samples per pixel, inputs resident),
    with the roofline block of ITS dominant kernel. N = 1 only; no CPU leg, no e2e."""
    import torch
    import ptb200
    path = os.path.join(ROOT, "scenes", workload + ".ssml")
    scene = ptb200.load_file(path)
    ctx = ptb200.Context(local)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.upload(scene)
    ctx.commit()

    def step(i):
        ctx.accum_clear()
        ctx.render(ptb200.RenderOptions(samples_per_pixel=spp, sample_offset=i * spp, render_method=method, width=w, height=h, seed=0))

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    ctx.set_option(ptb200._lib.OPT_TIME_KERNELS, 1)
    ctx.stats_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        step(warmup + i)
    e1.record(stream)
    torch.cuda.synchronize()
    dev_ms = e0.elapsed_time(e1)
    st = ctx.stats()
    ctx.set_option(ptb200._lib.OPT_TIME_KERNELS, 0)
    ms_by_kernel = {"k_trace": st.ms_trace, "k_shade": st.ms_shade, "k_shadow": st.ms_shadow, "bookkeeping": st.ms_generate,
                    "k_tail": st.ms_tail}
    dominant = max(("k_trace", "k_shade", "k_shadow"), key=lambda k: ms_by_kernel[k])
    ev = ncu_evidence(f"rtweekend1:{dominant}") or {}   # the sphere scenes share one capture (rtweekend1 3840x2160 MIS)
    out = {"metric": "Mrays/s", "value": st.rays_total / (dev_ms * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": 1, "steps": steps,
           "warmup": warmup, "ms_per_step": dev_ms / steps, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{workload}.ssml, {w}x{h}, {'mis' if method == 1 else 'naive'}, depth 50", "width": w, "height": h,
                      "spp_per_step": spp, "primitives": int(scene.n_primitives)},
           "gpu_launches": int(st.kernel_launches),
           "roofline": {"kernel": dominant, "bound": ev.get("bound", "unprofiled"), "achieved": ev.get("achieved"), "peak": ev.get("peak"),
                        "unit": ev.get("unit"), "frac": ev.get("frac"),
                        "frac_source": ev.get("source", "no ncu capture committed for this kernel"),
                        "traffic": ev.get("dram_bytes_per_launch"), "traffic_source": ev.get("traffic_source"),
                        "ms_by_kernel": ms_by_kernel, "dominant_kernel_share_of_step": ms_by_kernel[dominant] / dev_ms if dev_ms else None}}
    ctx.close()
    return out


def binary_tree_label(ctx):
    """Which builder made the committed binary tree (ptb_bvh_builder): the device SAH builder or the Karras LBVH."""
    builder, levels = ctx.bvh_builder()
    return f"device SAH builder ({levels} levels of binned splits + per-warp sweeps)" if builder == 4 else "Karras LBVH"


def run_closest_hit(args, rank, world, local, n_tris, n_rays, cpu=True, steps=None, warmup=None, dump_dir=""):
    """C5: incoherent Philox rays vs a synthetic heightfield BVH, intersection only (rays sharded across ranks).
    Returns the JSON object (rank 0) — also used as the `extra.c5` leg of the default run. `dump_dir`: --dump-outputs."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import ptb200

    rows, cols = heightfield_dims(n_tris)
    scene = ptb200.meshgen.heightfield_scene(rows, cols)
    ctx = ptb200.Context(local)
    stream = torch.cuda.current_stream()
    ctx.set_stream(stream.cuda_stream)
    ctx.upload(scene)
    ctx.commit()
    n_prims, n_nodes = ctx.bvh_info()
    n_wide, wide_leaf = ctx.bvh_wide_info()
    tree_label = binary_tree_label(ctx)
    node_bytes = 96.0 if n_wide else 64.0
    ctx_build_ms = ctx.stats().build_ms
    K = steps if steps is not None else args.steps
    W = warmup if warmup is not None else args.warmup
    batch = min(max(1, n_rays // max(K, 1)), 1 << 24)   # rays per step per rank
    # resident input: the stream is generated on the device before the timed region (untimed)
    first = lambda i: (rank * (K + W) + i) * batch
    d_rays = [philox_rays_device(batch, first(i), "cuda") for i in range(W + K)]
    chk = ptb200.meshgen.philox_rays(4096, first=first(0))
    got = d_rays[0][:4096].cpu().numpy()
    stream_err = float(max(np.max(np.abs(got[:, 0:3] - chk["o"])), np.max(np.abs(got[:, 4:7] - chk["d"]))))
    assert stream_err < 1e-5, f"device ray stream deviates from meshgen.philox_rays by {stream_err}"
    d_hits = torch.empty((batch, 4), dtype=torch.float32, device="cuda")
    for i in range(W):
        ctx.closest_hit_device(d_rays[i].data_ptr(), batch, d_hits.data_ptr())
    torch.cuda.synchronize()
    ctx.stats_reset()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(K):
        ctx.closest_hit_device(d_rays[W + i].data_ptr(), batch, d_hits.data_ptr())
    e1.record(stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = e0.elapsed_time(e1)
    launches = ctx.stats().kernel_launches
    tm = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    total_ms = float(tm[0])
    value = batch * K * world / (total_ms * 1e-3) / 1e6
    hit_frac = float((d_hits[:, 1].view(torch.int32) != -1).float().mean())
    if dump_dir and rank == 0:   # d_hits still holds the last timed step's hits
        dump_hits(dump_dir, batch, lambda index: d_hits[torch.from_numpy(index).cuda()].cpu().numpy()
                  .view(ptb200.hit_dtype).reshape(-1))
    # V, T on one batch (untimed)
    ctx.set_option(ptb200._lib.OPT_COUNT_TRAVERSAL, 1)
    ctx.stats_reset()
    ctx.closest_hit_device(d_rays[W].data_ptr(), batch, d_hits.data_ptr())
    sc = ctx.stats()
    ctx.set_option(ptb200._lib.OPT_COUNT_TRAVERSAL, 0)
    V, T = sc.nodes_fetched / batch, sc.prims_tested / batch
    b_ray = 32.0 + 16.0 + V * node_bytes + T * 48.0
    achieved = batch * K * b_ray / (ms * 1e-3) / 1e9
    peak, peak_src = measured_peaks()
    ev = ncu_evidence("c5:k_closest_hit_api") or {}
    # e2e: ptb_closest_hit with PINNED host rays in, pinned host hits out (upload | traverse | read-back pipelined inside)
    e2e = None
    if not args.no_e2e:
        nb = min(batch, 1 << 22)
        h_rays = ptb200.meshgen.philox_rays(nb, first=0)
        pin_r = torch.empty(nb * 32, dtype=torch.uint8, pin_memory=True)
        pin_h = torch.empty(nb * 16, dtype=torch.uint8, pin_memory=True)
        p_rays = np.frombuffer(pin_r.numpy().data, dtype=h_rays.dtype, count=nb)
        p_rays[...] = h_rays
        p_hits = np.frombuffer(pin_h.numpy().data, dtype=ptb200.hit_dtype, count=nb)
        ctx.closest_hit(p_rays, out=p_hits)  # warm: staging buffers, copy streams
        k2 = max(1, min(K, 4))
        t0 = time.perf_counter()
        for _ in range(k2):
            ctx.closest_hit(p_rays, out=p_hits)
        dt = time.perf_counter() - t0
        e2e = {"value": nb * k2 * world / dt / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": nb * 32, "d2h_bytes_per_step": nb * 16,
               "host_buffers": "pinned", "rays_per_step": nb}
    cpu_b = None
    if rank == 0 and world == 1 and cpu:
        O = import_oracle()
        o = O.OracleScene(scene)
        n = 1 << 18
        h_rays = ptb200.meshgen.philox_rays(n, first=0)
        t0 = time.perf_counter()
        o.closest_hit(h_rays)
        dtc = time.perf_counter() - t0
        cpu_b = {"value": n / dtc / 1e6, "unit": "Mrays/s", "cores": O.hardware_threads(), "kind": "port",
                 "sample": f"first {n} rays, reference SAH BVH + BFS candidates"}
    ctx.close()
    if rank != 0:
        return None
    cfg = closest_hit_config(args, n_prims)
    return {
        "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": cfg,
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "k_closest_hit_api (+ ray ordering passes, timed together)", "achieved": achieved,
                     "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                     "traffic": ev.get("dram_bytes_per_launch"), "traffic_source": ev.get("traffic_source"),
                     "algorithmic_bytes_per_launch": b_ray * batch, "bytes_per_ray": b_ray, "nodes_per_ray": V, "prims_per_ray": T,
                     "limiter": ev.get("limiter")},
        "cpu_baseline": cpu_b,
        "run": {"rays_per_step_per_gpu": batch, "rays_timed": batch * K * world, "bvh_nodes": n_wide or n_nodes, "node_bytes": node_bytes,
                "bvh": "compressed 8-wide" if n_wide else "binary, " + tree_label, "build_ms": ctx_build_ms, "hit_fraction": hit_frac,
                "ray_stream_max_abs_dev_vs_numpy": stream_err},
    }


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
