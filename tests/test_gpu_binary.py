"""The process-level drop-in contract (SURVEY 8b level 1): the `ray_cuda` binary run the way the reference's own
smoke test runs its binaries (scripts/test.sh:22-70, 205-256) -- from a directory holding scenes/, default scene
scenes/simple.txt, exit code 0, output_gpu.ppm larger than 1000 bytes, a line matching `time:|seconds`, and the image
compared with ray_serial's output_serial.ppm by the rule of scripts/compare_ppm.py at tolerance 0.5 (1 LSB).
That image is the oracle's, checked against the md5 recorded from the UNMODIFIED ray_serial.  Needs a B200: run with -m gpu."""
import hashlib
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

pytestmark = pytest.mark.gpu
PKG = os.path.join(ROOT, "cs420-ray-tracer_b200")
REF = os.path.join(ROOT, "oracle", "_ref")
REF_COMPARE = "/root/reference/scripts/compare_ppm.py"      # only in the build container; the rule is pinned by tests/test_host.py


@pytest.fixture(scope="module")
def workdir(tmp_path_factory):
    d = tmp_path_factory.mktemp("dropin")
    os.makedirs(d / "scenes")
    for n in ("simple", "medium", "complex"):
        shutil.copy(os.path.join(GOLDEN, "scenes", n + ".txt"), d / "scenes" / (n + ".txt"))
    return d


def run(cmd, cwd):
    p = subprocess.run(cmd, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    return p.returncode, p.stdout


def compare(rt, a, b, tol=0.5):
    if os.path.exists(REF_COMPARE):                     # the reference's own script when it is there
        p = subprocess.run([sys.executable, REF_COMPARE, str(a), str(b), str(tol)], stdout=subprocess.PIPE, text=True)
        assert p.returncode == 0, p.stdout
    Wa, Ha, _, ia = rt.read_ppm(str(a))
    Wb, Hb, _, ib = rt.read_ppm(str(b))
    assert (Wa, Ha) == (Wb, Hb)
    ok, pct, mx = rt.compare_rgb(ia, ib, tol)
    assert ok and mx <= 2, (pct, mx)


# the scene line ray_serial prints for each fixture (include/scene_loader.h:131-132; SURVEY F4)
SERIAL_LOADED = {"simple": "Loaded scene: 5 spheres, 2 lights", "medium": "Loaded scene: 44 spheres, 3 lights",
                 "complex": "Loaded scene: 154 spheres, 5 lights"}


@pytest.mark.parametrize("args", [[], ["scenes/medium.txt"], ["scenes/complex.txt"]])
def test_ray_cuda_is_a_drop_in_for_ray_serial(rt, oracle, scenes, golden, workdir, args):
    """ray_serial's output_serial.ppm at its built-in 1280x720 depth 10 is stood in for by the oracle's image, which must
    carry the md5 recorded from the unmodified ray_serial (tests/golden/golden.json)."""
    name = os.path.basename(args[0])[:-len(".txt")] if args else "simple"
    for f in ("output_gpu.ppm", "output_serial.ppm"):
        if os.path.exists(workdir / f):
            os.remove(workdir / f)
    rc, out = run([os.path.join(PKG, "ray_cuda")] + args, workdir)
    assert rc == 0, out
    # scripts/test.sh:49-62: output exists, > 1000 bytes, a timing line
    assert os.path.getsize(workdir / "output_gpu.ppm") > 1000
    timing = [l for l in out.splitlines() if re.search(r"(time:|seconds)", l)]
    assert timing and re.search(r"time: [0-9.eE+-]+ seconds", timing[0]), out
    # announces the scene the way ray_serial does
    loaded = [l for l in out.splitlines() if l.startswith("Loaded scene:")]
    assert loaded == [SERIAL_LOADED[name]], out
    oracle.write_ppm(str(workdir / "output_serial.ppm"), oracle.render(scenes[name], 1280, 720, 10)["rgb"])
    want = [g["md5"] for g in golden["images"] if g["by"].startswith("ray_serial") and g["scene"] == name]
    assert want and hashlib.md5((workdir / "output_serial.ppm").read_bytes()).hexdigest() == want[0]
    compare(rt, workdir / "output_serial.ppm", workdir / "output_gpu.ppm", 0.5)


def test_ray_cuda_flags_and_multi_gpu_bands(rt, workdir):
    """--width/--height/--depth/--output, -a, and --gpus N --band H (all ranks in ONE process through rt_create_multi;
    with fewer physical GPUs the ranks share devices, the frame is the same)."""
    rc, out = run([os.path.join(PKG, "ray_cuda"), "--width", "320", "--height", "180", "--depth", "5", "--output", "one.ppm",
                   "scenes/complex.txt"], workdir)
    assert rc == 0, out
    rc, out = run([os.path.join(PKG, "ray_cuda"), "--width", "320", "--height", "180", "--depth", "5", "--output", "four.ppm",
                   "--gpus", "4", "--band", "8", "scenes/complex.txt"], workdir)
    assert rc == 0, out
    assert (workdir / "one.ppm").read_bytes() == (workdir / "four.ppm").read_bytes()
    rc, out = run([os.path.join(PKG, "ray_cuda"), "scenes/missing.txt"], workdir)
    assert rc != 0 and "Could not open scene file" in out


@pytest.mark.parametrize("flags", [[], ["-p"], ["-t", "32", "scenes/medium.txt"]])
def test_reference_hybrid_links_against_the_kernel_shim(rt, oracle, workdir, flags):
    """The reference's OWN hybrid renderer (src/main_hybrid.cpp, unmodified, built by oracle/Makefile where it lies)
    linked against libkernel_shim.so in place of its kernel.o: launch_gpu_kernel / upload_lights_and_ambience keep the
    signatures of src/kernel.cu:185-207, so the tile scheduler, the three-stream launch loop and the bulk download of
    src/main_hybrid.cpp:373-706 run unchanged.  Its image (CPU tiles: the reference's FP64 code; GPU tiles: this library
    on the FP32 scene structs the caller uploads) must pass the compare_ppm.py gate against the serial renderer at
    ray_hybrid's own size (1080x720, depth 3: src/main_hybrid.cpp:42-43,715)."""
    exe = os.path.join(REF, "ray_hybrid_shim")
    if not os.path.exists(exe) or not oracle.ref_available():
        pytest.skip("oracle/_ref/ray_hybrid_shim was not built (needs /root/reference at build time)")
    out = workdir / "output_hybrid.ppm"
    if os.path.exists(out):
        os.remove(out)
    rc, log = run([exe] + flags, workdir)
    assert rc == 0, log
    assert "Hybrid rendering time:" in log and os.path.getsize(out) > 1000
    scene = [f for f in flags if f.endswith(".txt")] or ["scenes/simple.txt"]
    oracle.ref_harness("render", scene[0], 1080, 720, 3, "serial_1080.ppm", cwd=str(workdir))
    compare(rt, workdir / "serial_1080.ppm", out, 0.5)
    dist = [l for l in log.splitlines() if l.startswith("Distribution:")]
    assert dist and " tiles to GPU" in dist[0] or "GPU" in dist[0], log       # (src/main_hybrid.cpp:426: some tiles did go to the GPU)


def test_benchmark_csv_has_the_reference_format(workdir):
    """scripts/benchmark_csv.py = the reference's scripts/benchmark.sh report for this binary: same CSV header
    (scripts/benchmark.sh:29), one row per (implementation, scene, threads, iteration), the time cut from the program's
    own `time:` line the way extract_time() does (scripts/benchmark.sh:32-34), and the summary table of :193-236."""
    out = workdir / "bench_csv"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "benchmark_csv.py"), "--iterations", "1", "--threads", "4",
                        "--out", str(out)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert p.returncode == 0, p.stdout
    assert "Average Execution Times (seconds):" in p.stdout
    csvs = [f for f in os.listdir(out) if f.startswith("benchmark_") and f.endswith(".csv")]
    assert len(csvs) == 1
    lines = (out / csvs[0]).read_text().strip().split("\n")
    assert lines[0] == "Implementation,Scene,Threads,Iteration,Time(s),Pixels/s,Speedup"
    rows = [l.split(",") for l in lines[1:]]
    cuda = [r for r in rows if r[0] == "CUDA"]
    assert sorted(r[1] for r in cuda) == ["complex.txt", "medium.txt", "simple.txt"]
    for r in rows:
        assert len(r) == 7 and float(r[4]) > 0 and abs(float(r[5]) - 1280 * 720 / float(r[4])) <= 1.0 + 1e-4 * float(r[5])   # (Time(s) is printed with 6 decimals)
    if os.path.exists(os.path.join(REF, "ray_serial")):
        assert {r[0] for r in rows} == {"Serial", "OpenMP", "CUDA"}
        assert all(float(r[6]) > 10.0 for r in cuda)         # the reference's own bar for its CUDA build: >= 10x serial (scripts/benchmark.sh:298)
