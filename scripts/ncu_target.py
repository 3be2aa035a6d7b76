"""Target for ncu captures: a few production frames (no stats) of one configuration.
usage: ncu_target.py scene W H D frames"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import rtb200
name, W, H, D, frames = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5])
if name.startswith("synth"):
    import gen_scene
    p = name.split(":")
    sc = rtb200.Scene(*gen_scene.generate(int(p[1]), int(p[2])))
else:
    sc = rtb200.load_scene(os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "scenes", name + ".txt"))
r = rtb200.Renderer(0)
r.upload(sc)
out = np.empty((H, W, 3), dtype=np.uint8)
for _ in range(frames):
    r.render(W, H, D, out=out, want_stats=False)
print("ok", int(out.sum()))
