"""Reflection level 1 of the headline frame (complex.txt, 1920x1080): per-kernel device times, level-1 bundle counters,
and ms per frame of two builds of the library, alternated in one run.  Needs a B200.

  python scripts/probe_level1.py [--old LIB] [--new LIB] [--runs 3] [--out FILE]

Each build is measured in its own process (RTB200_LIB).  A build outside the tree is made with
  make -C cs420-ray-tracer_b200 BUILD=DIR LIB=DIR/librt_b200.so EXTRA_NVFLAGS=... DIR/librt_b200.so
Per-kernel times come from torch.profiler with CUDA activities (a separate render loop of the same process; also for
simple.txt at 1280x720 d10, the workload whose tail consumes the level-0 queue directly); ms per frame from bench.py
(profiler off).

Level-1 counters = those of a depth-2 render minus a depth-1 render, wave_levels 2, one context, three renders each.
k_closest1 and k_shadow add into the same bundle_* counters; they are told apart with the same scene WITHOUT lights,
which has the same closest hits and reflected rays but no shadow walks: its level-1 counters are k_closest1's, the
difference to the lit scene is the level-1 k_shadow's.  The lightless scene's fp64_intersections are k_closest1's alone.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def child():
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    import rtb200
    sc = rtb200.load_scene(os.path.join(ROOT, "tests", "golden", "scenes", "complex.txt"))
    W, H = 1920, 1080
    res = {"nspheres": sc.nspheres}
    dark = rtb200.Scene(sc.spheres, np.zeros((0, 7)), sc.ambient, sc.camera)
    keys = ("bundle_walks", "bundle_candidates", "fp64_intersections", "closest_queries")
    for tag, scene in (("lit", sc), ("dark", dark)):
        with rtb200.Renderer(0) as r:
            r.set_option("wave_levels", 2)
            r.upload(scene)
            runs = []
            for _ in range(3):
                c = {}
                for D in (1, 2):
                    _, st = r.render(W, H, D)
                    c[D] = {k: int(getattr(st, k)) for k in keys}
                runs.append({k: c[2][k] - c[1][k] for k in keys})
            res[tag] = runs
    from torch.profiler import ProfilerActivity, profile
    simple = rtb200.load_scene(os.path.join(ROOT, "tests", "golden", "scenes", "simple.txt"))
    for tag, scene, W, H, D in (("complex", sc, 1920, 1080, 5), ("simple", simple, 1280, 720, 10)):
        with rtb200.Renderer(0) as r:
            r.upload(scene)
            buf = torch.empty(H * W * 3 + 16, dtype=torch.uint8, device="cuda:0")
            for _ in range(20):
                r.render_bands_device(W, H, D, 16, 0, 1, buf.data_ptr())
            torch.cuda.synchronize()
            n = 50
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(n):
                    r.render_bands_device(W, H, D, 16, 0, 1, buf.data_ptr())
                torch.cuda.synchronize()
            k = {}
            for ev in prof.events():
                if ev.device_type == torch.autograd.DeviceType.CUDA and "rtf::" in ev.name:
                    name = ev.name.split("(")[0].replace("void ", "")
                    k.setdefault(name, []).append(ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total)
            # launch order within a frame: the same kernel appears at level 0 and level 1 (k_shadow, k_shade)
            res["kernels_us_" + tag] = {name: [round(float(np.mean(v[i::len(v) // n])), 2) for i in range(len(v) // n)]
                                        for name, v in k.items()}
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--old", default=os.path.join(ROOT, "cs420-ray-tracer_b200", "build", "parent", "librt_b200.so"))
    ap.add_argument("--new", default=os.path.join(ROOT, "cs420-ray-tracer_b200", "librt_b200.so"))
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--child", action="store_true")
    a = ap.parse_args()
    if a.child:
        return child()
    lines = []
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    lines.append("GPU: %s" % q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "GPU: (nvidia-smi unavailable)")
    builds = {"old": a.old, "new": a.new}
    for tag, lib in builds.items():
        env = dict(os.environ, RTB200_LIB=lib)
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--child"], env=env, capture_output=True, text=True)
        if p.returncode != 0:
            raise SystemExit("%s failed:\n%s" % (tag, p.stderr[-3000:]))
        d = json.loads(p.stdout.strip().splitlines()[-1])
        for tag2, what in (("lit", "k_closest1 + k_shadow"), ("dark", "k_closest1 (scene without lights)")):
            for i, l1 in enumerate(d[tag2]):
                lines.append("%s: level-1 %-34s render %d: bundle_walks %7d bundle_candidates %8d (%5.1f per walk), fp64 %d, closest %d" % (
                    tag, what, i, l1["bundle_walks"], l1["bundle_candidates"], l1["bundle_candidates"] / max(1, l1["bundle_walks"]),
                    l1["fp64_intersections"], l1["closest_queries"]))
        lit, dark = d["lit"][0], d["dark"][0]
        w, c = lit["bundle_walks"] - dark["bundle_walks"], lit["bundle_candidates"] - dark["bundle_candidates"]
        lines.append("%s: level-1 k_shadow (lit - dark): bundle_walks %d bundle_candidates %d (%.1f per walk)" % (tag, w, c, c / max(1, w)))
        lines.append("%s: level-1 k_closest1: %d of %d 64-ray chunks culled, %.1f of %d spheres kept per culled walk (a kept pair counts 2)" % (
            tag, dark["bundle_walks"], (dark["closest_queries"] + 63) // 64, dark["bundle_candidates"] / max(1, dark["bundle_walks"]),
            d["nspheres"]))
        for wl in ("complex", "simple"):
            for name, us in sorted(d["kernels_us_" + wl].items()):
                lines.append("%s: %-7s %-40s %s us (per launch of a frame, in launch order)" % (tag, wl, name, us))
    ms = {t: [] for t in builds}
    for _ in range(a.runs):
        for tag, lib in builds.items():
            env = dict(os.environ, RTB200_LIB=lib)
            p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "300", "--warmup", "30",
                                "--no-cpu-baseline"], env=env, capture_output=True, text=True, cwd=ROOT)
            line = [x for x in p.stdout.splitlines() if x.startswith("{")]
            if p.returncode != 0 or not line:
                raise SystemExit("bench %s failed:\n%s" % (tag, p.stdout[-2000:] + p.stderr[-2000:]))
            ms[tag].append(json.loads(line[-1])["ms_per_step"])
    for tag in builds:
        v = sorted(ms[tag])
        lines.append("%s: bench ms_per_step %s median %.4f" % (tag, ["%.4f" % x for x in ms[tag]], v[len(v) // 2]))
    txt = "\n".join(lines)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
