"""CPU only: per-pixel camera candidate lists on the full C3 mesh (1 M triangles) at 1920 x 1080, on the device SAH tree's
CPU definition (scripts/camcand_ref.cpp): the distribution of the candidate count per pixel, the fraction of pixels that
overflow a list of K entries, the entries / primitive tests per camera ray of the list path against the ordered walk's
nodes and primitive tests, and the bit-for-bit check of list hits against the walk over one jittered sample per pixel.

    python scripts/camcand_probe.py [--scale 1.0] [--width 1920] [--height 1080] [--spp 1] [--md profiles/camcand_probe.md]
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import ptb200  # noqa: E402
import camcand_ref  # noqa: E402


def hist_percentile(h, p):
    """p-th percentile of the values counted in histogram h (bin i: value i; the last bin: that value or more)."""
    cum = np.cumsum(h.astype(np.float64))
    return int(np.searchsorted(cum, cum[-1] * p / 100.0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--spp", type=int, default=1)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--md", default=None)
    a = ap.parse_args()
    W, H = a.width, a.height
    scene = ptb200.meshgen.c3_scene(a.scale)
    s = camcand_ref.CamCandScene(scene)
    L = s.lists(W, H, a.k)
    r = s.check(L, a.spp, seed=1)
    c = L.count
    q = {p: float(np.percentile(c, p)) for p in (50, 90, 99)}
    lines = [f"# Camera candidate lists on C3: CPU probe\n",
             f"`python scripts/camcand_probe.py --scale {a.scale} --width {W} --height {H} --spp {a.spp} --k {a.k}` "
             f"({len(scene.triangles)} triangles, the device SAH tree's CPU definition).\n",
             "Frustum test of `csrc/ptb_camcand.cuh` (f64, pixel square widened by 2^-20, boxes grown by 2^-16), no "
             "occluder culling.\n",
             "## Candidates per pixel\n",
             "| median | p90 | p99 | max | mean | beam-walk nodes per pixel (mean) |", "|---|---|---|---|---|---|",
             f"| {q[50]:.0f} | {q[90]:.0f} | {q[99]:.0f} | {int(c.max())} | {c.mean():.2f} | {L.visits.mean():.1f} |\n",
             "## Pixels that overflow a list of K entries\n", "| K | overflowed |", "|---|---|"]
    for k in (4, 8, 16, 32):
        lines.append(f"| {k} | {100.0 * float(np.mean(c > k)):.2f} % |")
    lr = max(r["list_rays"], 1)
    lines += ["", f"## Work per camera ray (K = {a.k}, rays of pixels that did not overflow: {r['list_rays']} of {r['rays']})\n",
              "| path | nodes | entries (leaf box tests) | primitive tests |", "|---|---|---|---|",
              f"| ordered walk | {r['walk_nodes'] / lr:.2f} | | {r['walk_prims'] / lr:.2f} |",
              f"| list, nearest first, stop at key > best t | | {r['list_entries'] / lr:.2f} | {r['list_prim_tests'] / lr:.2f} |",
              "", "Per listed camera ray (the go / no-go compares the list path's p90 with the walk's):\n",
              "| count per ray | p50 | p90 | p99 |", "|---|---|---|---|"]
    for name, key in (("ordered walk: nodes", "walk_nodes"), ("list: entries tested", "list_entries"),
                      ("list: primitive tests", "list_prim_tests")):
        lines.append(f"| {name} | " + " | ".join(str(hist_percentile(r["hist"][key], p)) for p in (50, 90, 99)) + " |")
    lines += ["", "## Exactness\n",
              f"{r['list_rays']} jittered camera rays answered from their pixel's list: {r['mismatches']} differ from the "
              f"ordered walk's hit in t bits or primitive; {r['box_rejected_hits']} list entries were hit by the primitive "
              f"test although box_entry rejects their leaf box; {r['key_above_tkey']} list keys exceed the cull key "
              "box_entry computes on their leaf box for a ray of the pixel (the key must be a lower bound).\n",
              "## Occluder culling\n",
              f"Not built: without it {100.0 * float(np.mean(c > 16)):.2f} % of the pixels overflow a 16-entry list, below the "
              "10 % the design allows, and a listed ray already tests few primitives.\n"]
    text = "\n".join(lines)
    print(text)
    if a.md:
        with open(a.md, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
