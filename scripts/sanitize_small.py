"""Tiny end-to-end workload for compute-sanitizer (memcheck / racecheck / initcheck): every kernel, small sizes."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import ptb200

root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ctx = ptb200.Context(0)
for name, scene in (("overshadowed", ptb200.load_file(os.path.join(root, "scenes/overshadowed.ssml"))),
                    ("c3_small", ptb200.meshgen.c3_scene(0.02))):
    sc = ptb200.Scene(scene, ctx=ctx)
    rays = ptb200.meshgen.philox_rays(5000, seed=1, centre=(0, 1, 0), radius=3.0)
    h = sc.acceleration.check_hit(rays)
    for pool in ("", "1024"):  # one chunk, many chunks
        os.environ.pop("PTB_POOL_PATHS", None)
        if pool:
            os.environ["PTB_POOL_PATHS"] = pool
        for method in (0, 1):
            img = sc.render(ptb200.RenderOptions(samples_per_pixel=3, render_method=method, width=61, height=35, seed=1))
            assert np.isfinite(img).all()
    os.environ.pop("PTB_POOL_PATHS", None)
    print(name, "ok", int((h["prim"] != ptb200.PTB_MISS).sum()), "hits")
ctx.close()
print("done")
