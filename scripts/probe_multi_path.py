"""Camera paths on several GPUs: whole frames to ranks (rt_multi_render_path) against row bands of every frame.

Workloads: complex.txt 1920x1080 depth 5, a 240-frame orbit; config 4 (synthetic 10k spheres, seed 420, LBVH)
3840x2160 depth 5, a 60-frame orbit.  The orbit circles the look-at point at the scene camera's distance.  For n ranks
(default 1, 2, 4, 8; with more ranks than devices the ranks share devices and the line says so):
  path      MultiRenderer.render_path: ms/frame, host clock around the call plus a synchronise; its speed-up over the
            1-GPU Renderer.render_path (measured the same way in the same run)
  enqueue   host time until the call returns, per frame per rank (call time / ceil(K / n)): over the whole path, where a
            full launch queue makes the host wait for the device, and over a short path of 8 frames per rank
  bands     rt_multi_set_camera + rt_multi_render (16-row bands, host frame) per frame: ms/frame
  frames    byte-for-byte against the 1-GPU Renderer.render_path
Every variant is warmed up at its size first, then timed twice, alternating.

    python scripts/probe_multi_path.py [--ranks 1,2,4,8] [--out FILE]
"""
import argparse
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gen_scene  # noqa: E402
import rtb200  # noqa: E402


def orbit(cam, K):
    look = cam[3:6]
    d = cam[0:3] - look
    r, a0 = math.hypot(d[0], d[2]), math.atan2(d[0], d[2])
    return np.array([[look[0] + r * math.sin(a0 + 2 * math.pi * k / K), cam[1], look[2] + r * math.cos(a0 + 2 * math.pi * k / K),
                      look[0], look[1], look[2], cam[6]] for k in range(K)])


def sync_all():
    for d in range(torch.cuda.device_count()):
        torch.cuda.synchronize(d)


def timed_path(r, cams, W, H, D, out):
    """(ms/frame to the synchronise, ms until the call returned)"""
    sync_all()
    t0 = time.perf_counter()
    r.render_path(cams, W, H, D, out=out)
    t1 = time.perf_counter()
    torch.cuda.synchronize(0)            # the current stream of device 0 waits for every rank's frames
    t2 = time.perf_counter()
    return (t2 - t0) * 1e3 / len(cams), (t1 - t0) * 1e3


def timed_bands(m, cams, W, H, D, host):
    sync_all()
    t0 = time.perf_counter()
    for c in cams:
        m.set_camera(c[0:3], c[3:6], c[6])
        m.render(W, H, D, band_h=16, out=host, want_stats=False)
    return (time.perf_counter() - t0) * 1e3 / len(cams)


def probe(name, scene, W, H, D, K, ranks, log):
    ndev = torch.cuda.device_count()
    cams = orbit(np.asarray(scene.camera, dtype=np.float64), K)
    dev = torch.device("cuda", 0)
    ref = torch.empty((K, H, W, 3), dtype=torch.uint8, device=dev)
    out = torch.empty_like(ref)
    host = np.empty((H, W, 3), dtype=np.uint8)
    log("%s: %d spheres, %d lights, %dx%d depth %d, %d-frame orbit" % (name, scene.nspheres, scene.nlights, W, H, D, K))
    ok = True
    with rtb200.Renderer(0) as r:
        r.upload(scene)
        timed_path(r, cams[:4], W, H, D, ref[:4])
        one = [timed_path(r, cams, W, H, D, ref)[0] for _ in range(2)]
    log("  1-GPU Renderer.render_path: %s ms/frame" % " / ".join("%.3f" % x for x in one))
    base = min(one)
    for n in ranks:
        with rtb200.MultiRenderer(n) as m:
            m.upload(scene)
            w = min(K, 8 * n)
            timed_path(m, cams[:w], W, H, D, out[:w])     # warm-up: every rank's buffers and tables at this size
            timed_bands(m, cams[:w], W, H, D, host)
            short = timed_path(m, cams[:w], W, H, D, out[:w])[1] / math.ceil(w / n)
            path, bands = [], []
            for _ in range(2):
                path.append(timed_path(m, cams, W, H, D, out))
                bands.append(timed_bands(m, cams, W, H, D, host))
            same = bool(torch.equal(out, ref))
        ok &= same
        per_rank = math.ceil(K / n)
        shared = "" if n <= ndev else "  [%d ranks share %d device%s: no speed-up expected]" % (n, ndev, "s" if ndev > 1 else "")
        log("  n=%d  path %s ms/frame (%.2fx)  enqueue %s ms/frame/rank (short path %.3f)  bands %s ms/frame  frames %s%s" % (
            n, " / ".join("%.3f" % p[0] for p in path), base / min(p[0] for p in path),
            " / ".join("%.3f" % (p[1] / per_rank) for p in path), short, " / ".join("%.3f" % b for b in bands),
            "byte-identical" if same else "DIFFERENT", shared))
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ranks", default="1,2,4,8")
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    ranks = [int(x) for x in args.ranks.split(",")]
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log("GPU: %s, %d visible" % (torch.cuda.get_device_name(0), torch.cuda.device_count()))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip().splitlines()
        log("power limit, max SM clock: %s" % ("; ".join(sorted(set(q))) if q else "not available"))
    except (OSError, subprocess.SubprocessError):
        log("power limit: not available")
    ok = probe("complex.txt", rtb200.load_scene(os.path.join(ROOT, "tests", "golden", "scenes", "complex.txt")), 1920, 1080, 5,
               240, ranks, log)
    ok &= probe("config 4 (synth 10k, seed 420, LBVH)", rtb200.Scene(*gen_scene.generate(10000, 420)), 3840, 2160, 5, 60,
                ranks, log)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
