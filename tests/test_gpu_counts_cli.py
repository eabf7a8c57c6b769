"""(1) The V / T of the algorithmic-bytes-per-ray figure: the device's instrumented traversal vs the CPU LBVH oracle's
ordered, t-culled traversal of the same (bit-exact) tree. The device walks speculatively (a lane holding a postponed leaf
keeps descending before its best-t is updated), so it may fetch slightly MORE nodes than the sequential oracle — never
fewer primitives' worth of work than needed, and the hits are identical.
(2) The C++ frontend (ptb200-cli) end to end against the Python binding."""
import os
import subprocess

import numpy as np
import pytest

from conftest import random_rays

pytestmark = pytest.mark.gpu


def test_traversal_counts_match_lbvh_oracle(ptb, orc, gpu_ctx):
    s = ptb.meshgen.c3_scene(0.1)
    rays = random_rays(ptb, 200_000, 21, centre=(0, 4, 1), radius=5.0)
    gpu_ctx.upload(s)
    gpu_ctx.commit(ptb._lib.BUILD_BINARY)   # the binary walk's counts (the wide tree's are EQUAL to its own CPU statement: test_gpu_wide.py)
    gpu_ctx.set_option(ptb._lib.OPT_COUNT_TRAVERSAL, 1)
    gpu_ctx.stats_reset()
    g = gpu_ctx.closest_hit(rays)
    st = gpu_ctx.stats()
    gpu_ctx.set_option(ptb._lib.OPT_COUNT_TRAVERSAL, 0)
    o = orc.OracleScene(s, split_type=-1)
    h, nodes, prims = o.lbvh_closest_hit(rays)
    assert np.array_equal(g["prim"], h["prim"]) and np.array_equal(g["t"].view(np.uint32), h["t"].view(np.uint32))
    assert st.rays_counted == len(rays)
    v_dev, v_cpu = st.nodes_fetched / len(rays), nodes / len(rays)
    t_dev, t_cpu = st.prims_tested / len(rays), prims / len(rays)
    assert v_cpu <= v_dev <= 1.10 * v_cpu, (v_dev, v_cpu)     # speculation costs a few percent of extra node fetches
    assert t_cpu <= t_dev <= 1.25 * t_cpu, (t_dev, t_cpu)


def test_stats_kernel_timers(ptb, gpu_ctx, rtweekend1):
    sc = ptb.Scene(rtweekend1, ctx=gpu_ctx)
    gpu_ctx.set_option(ptb._lib.OPT_TIME_KERNELS, 1)
    gpu_ctx.stats_reset()
    sc.render(ptb.RenderOptions(samples_per_pixel=8, render_method=1, width=320, height=180))
    st = gpu_ctx.stats()
    gpu_ctx.set_option(ptb._lib.OPT_TIME_KERNELS, 0)
    assert st.ms_trace > 0 and st.ms_shade > 0 and st.ms_generate > 0 and st.ms_shadow > 0
    assert st.ms_trace + st.ms_shade + st.ms_generate + st.ms_shadow <= st.render_ms * 1.05
    assert st.trace_launches == st.wavefront_iterations and st.kernel_launches >= 6 * st.wavefront_iterations


def test_cli_matches_binding(ptb, gpu_ctx, root, tmp_path):
    cli = os.path.join(root, "raytracing-rust_b200", "ptb200-cli")
    assert os.path.exists(cli), "build the frontend with `make cli`"
    out = tmp_path / "img.pfm"
    scene_path = os.path.join(root, "scenes", "overshadowed.ssml")
    # -o takes exactly one '.' in the whole path (output/src/lib.rs:81-85): a relative name, run inside tmp_path
    r = subprocess.run([cli, "-f", scene_path, "-s", "8", "-x", "96", "-y", "54", "-r", "naive", "-o", out.name, "--seed", "5"],
                       capture_output=True, text=True, timeout=300, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    assert "Render started:" in r.stderr and "Rays shot:" in r.stderr and "Mray/s" in r.stderr
    raw = out.read_bytes()
    hdr_end = raw.index(b"-1.0\n") + 5
    img = np.frombuffer(raw[hdr_end:], np.float32).reshape(54, 96, 3)[::-1]     # PFM stores rows bottom-up
    sc = ptb.Scene(ptb.load_file(scene_path), ctx=gpu_ctx)
    ref = sc.render(ptb.RenderOptions(samples_per_pixel=8, render_method=0, width=96, height=54, seed=5))
    assert np.max(np.abs(img - ref)) < 1e-5
    # argument errors mirror clap's behaviour: usage + non-zero exit, and the gui flag answers like the reference
    assert subprocess.run([cli], capture_output=True).returncode != 0
    g = subprocess.run([cli, "-g", "-f", scene_path], capture_output=True, text=True)
    assert g.returncode == 0 and "feature: gui not enabled" in g.stdout


def test_cli_gpus_flag_and_exr_output(ptb, gpu_ctx, root, tmp_path):
    """VERDICT r1 #8: `--gpus N -o x.exr` — the multi-GPU render from the product boundary, written as linear f32 EXR
    (output/src/lib.rs:98-104), equals the single-GPU image. With one GPU in the box N = 1 still goes through the flag."""
    import ctypes as C
    import struct
    n = C.c_int32()
    ptb._lib.lib.ptb_device_count(C.byref(n))
    gpus = 2 if n.value >= 2 else 1
    cli = os.path.join(root, "raytracing-rust_b200", "ptb200-cli")
    out = tmp_path / "img.exr"
    scene_path = os.path.join(root, "scenes", "rtweekend1.ssml")
    r = subprocess.run([cli, "-f", scene_path, "-s", "6", "-x", "96", "-y", "54", "-r", "mis", "-o", out.name, "--seed", "9",
                        "--gpus", str(gpus)], capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert r.returncode == 0, r.stderr
    assert f"{gpus} GPU(s)" in r.stderr and f"Image {out.name} saved" in r.stderr
    raw = out.read_bytes()
    assert struct.unpack_from("<I", raw, 0)[0] == 20000630
    w, h = 96, 54
    data = raw[len(raw) - h * (8 + 12 * w):]                    # uncompressed scanline chunks at the end of the file
    img = np.zeros((h, w, 3), np.float32)
    for y in range(h):
        row = np.frombuffer(data, np.float32, 3 * w, y * (8 + 12 * w) + 8).reshape(3, w)
        img[y] = row[::-1].T
    sc = ptb.Scene(ptb.load_file(scene_path), ctx=gpu_ctx)
    ref = sc.render(ptb.RenderOptions(samples_per_pixel=6, render_method=1, width=96, height=54, seed=9))
    assert np.max(np.abs(img - ref)) < 1e-5
    assert subprocess.run([cli, "-f", scene_path, "--gpus", "0"], capture_output=True).returncode != 0


def test_cli_bvh_type(ptb, root, tmp_path):
    """`-b / --bvh-type` (parameters.rs:35-36): sah = the device SAH builder, middle = the Karras LBVH (spatial-middle splits),
    equal-counts = the LBVH with a warning. The image does not depend on the tree; an unknown value is a usage error."""
    cli = os.path.join(root, "raytracing-rust_b200", "ptb200-cli")
    scene_path = os.path.join(root, "scenes", "overshadowed.ssml")
    imgs = {}
    for bvh in ("sah", "middle", "equal-counts"):
        out = tmp_path / f"img_{bvh}.pfm"
        r = subprocess.run([cli, "-f", scene_path, "-s", "4", "-x", "64", "-y", "36", "-r", "mis", "-o", out.name, "--seed", "3", "-b", bvh],
                           capture_output=True, text=True, timeout=300, cwd=tmp_path)
        assert r.returncode == 0, r.stderr
        assert ("no equal-counts builder" in r.stderr) == (bvh == "equal-counts")
        raw = out.read_bytes()
        imgs[bvh] = np.frombuffer(raw[raw.index(b"-1.0\n") + 5:], np.float32)
    # (two renders agree to the f32 summation order of the accumulator's atomic adds, not bit for bit: ptb200.h)
    assert np.allclose(imgs["sah"], imgs["middle"], rtol=1e-5, atol=1e-5) and np.allclose(imgs["middle"], imgs["equal-counts"], rtol=1e-5, atol=1e-5)
    assert subprocess.run([cli, "-f", scene_path, "-b", "octree"], capture_output=True).returncode != 0
