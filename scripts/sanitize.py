"""Small renders of every kernel family for compute-sanitizer (memcheck / racecheck):
    compute-sanitizer --tool memcheck python scripts/sanitize.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import gen_scene
import rtb200
root = os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "scenes")
cx = rtb200.load_scene(os.path.join(root, "complex.txt"))
big = rtb200.Scene(*gen_scene.generate(1500, 5, 0.2, 0.8))
for label, scene, kw, sizes in [("tables/smem", cx, {}, [(97, 61, 4), (160, 90, 5)]), ("bvh", cx, {"accel": 2}, [(97, 61, 4)]),
                                ("stream", big, {"accel": 1}, [(96, 54, 3)]), ("bvh-large", big, {}, [(96, 54, 3)]), ("exact", cx, {"mode": "exact"}, [(64, 36, 3)])]:
    with rtb200.Renderer(0, **kw) as r:
        r.upload(scene)
        for (W, H, D) in sizes:
            rgb, hit, mask, st = r.render_debug(W, H, D)
            print(label, W, H, D, "rays", st.closest_queries + st.shadow_queries, "viol", st.filter_violations)
        if kw.get("mode") != "exact":
            # production launch sequence (no stats: programmatic dependent launch)
            r.render(160, 90, 5, want_stats=False)
            r.render(160, 90, 5, want_stats=False)
            r.set_option("antialias", 1)
            r.render(50, 30, 3)
            r.set_option("antialias", 0)
            import torch
            fb = torch.zeros((40, 70, 3), dtype=torch.float32, device="cuda:0")
            torch.cuda.synchronize()
            r.render_tile_device(70, 40, 3, (5, 7, 33, 21), fb.data_ptr())
            fr = torch.zeros((40, 70, 3), dtype=torch.uint8, device="cuda:0")
            torch.cuda.synchronize()
            r.render_bands_frame(70, 40, 3, 16, 1, 2, fr.data_ptr())
            torch.cuda.synchronize()
with rtb200.MultiRenderer(3) as m:                       # rt_create_multi: three ranks (sharing devices on a 1-GPU box)
    m.upload(cx)
    m.render(97, 61, 4, band_h=8)
print("done")
