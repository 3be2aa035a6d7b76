#!/usr/bin/env python3
"""bench.py -- headline benchmark: Mrays/s & ms/frame, complex.txt at 1920x1080 depth 5.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one full frame of the hot path (camera rays -> closest hit -> Phong + shadow rays
-> reflection bounces -> 8-bit RGB).  The ray count of a frame is a property of (scene, W, H,
depth) -- R_c + R_s in the oracle's definition (SURVEY 8d) -- so Mrays/s = rays / time.

  value     frame already scheduled from device-resident scene tables, output into HBM; at N > 1
            each rank renders its interleaved 16-row bands and its kernels store them straight
            into rank 0's frame over NVLink (peer memory, rt_render_bands_frame; completion flags
            inside the timed step; --gather nccl = the NCCL gather instead).  CUDA events per
            step, L2 flushed between steps.
  e2e       the same through the public C ABI with HOST buffers every step: rt_upload_scene
            (host -> device) + render + frame copy into pinned host memory (device -> host).
  roofline  FP32 FMA bound (BASELINE.md section 3): algorithmic flops = 16 x N_spheres x rays.
  cpu_baseline / --impl reference   the reference's own serial/OpenMP renderer (oracle/_ref,
            built from the unmodified sources) on the host cores of the same box.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# NCCL prints its version banner to STDOUT at NCCL_DEBUG=VERSION; stdout carries exactly one JSON line here
if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"

SCENE = os.path.join(ROOT, "tests", "golden", "scenes", "complex.txt")
W, H, DEPTH, BAND_H = 1920, 1080, 5, 16
WORKLOAD = "complex.txt (154 spheres, 5 lights) 1920x1080 depth 5"
FLOP_PER_TEST = 16          # SURVEY 8(d): reduced form of include/sphere.h:29-34
# the other BASELINE.json configs (parity-test cases; --workload runs them for profiles/, the driver never does)
WORKLOADS = {
    "complex": ("complex", 1920, 1080, 5, "complex.txt (154 spheres, 5 lights) 1920x1080 depth 5"),
    "medium": ("medium", 1920, 1080, 5, "medium.txt (44 spheres, 3 lights) 1920x1080 depth 5"),
    "simple": ("simple", 1280, 720, 10, "simple.txt (5 spheres, 2 lights) 1280x720 depth 10"),
    "synth10k": ("synth:10000:420", 3840, 2160, 5, "synthetic 10k spheres (scripts/gen_scene.py seed 420), 4 lights, 3840x2160 depth 5"),
    "synth100k": ("synth:100000:421", 7680, 4320, 8, "synthetic 100k spheres (scripts/gen_scene.py seed 421), 4 lights, 7680x4320 depth 8, device-built LBVH"),
}


def load_workload(name):
    import rtb200
    sc = WORKLOADS[name][0]
    if sc.startswith("synth:"):
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import gen_scene
        _, n, seed = sc.split(":")
        return rtb200.Scene(*gen_scene.generate(int(n), int(seed)))
    return rtb200.load_scene(os.path.join(ROOT, "tests", "golden", "scenes", sc + ".txt"))


class _PlainScene:
    """Scene arrays for the reference arm / cpu baseline WITHOUT the product library: that arm must not load
    librt_b200.so (the driver records which .so files each arm loads)."""

    def __init__(self, spheres, lights, ambient, camera):
        import numpy as np
        self.spheres = np.asarray(spheres, dtype=np.float64).reshape(-1, 10)
        self.lights = np.asarray(lights, dtype=np.float64).reshape(-1, 7)
        self.ambient = np.asarray(ambient, dtype=np.float64).reshape(3)
        self.camera = np.asarray(camera, dtype=np.float64).reshape(7)


def load_workload_plain(name):
    """The same scenes as load_workload, parsed in Python (the fixtures are plain directive lines in the grammar of
    include/scene_loader.h:15-21; defaults as include/scene.h:22,31)."""
    sc = WORKLOADS[name][0]
    if sc.startswith("synth:"):
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import gen_scene
        _, n, seed = sc.split(":")
        return _PlainScene(*gen_scene.generate(int(n), int(seed)))
    sph, lig, amb, cam = [], [], [0.0, 0.0, 0.0], [0.0, 0.0, 0.0, 0.0, 0.0, -1.0, 60.0]
    with open(os.path.join(ROOT, "tests", "golden", "scenes", sc + ".txt")) as f:
        for line in f:
            t = line.split("#")[0].split()
            if not t:
                continue
            v = [float(x) for x in t[1:]]
            if t[0] == "sphere" and len(v) >= 10:
                sph.append(v[:10])
            elif t[0] == "light" and len(v) >= 7:
                lig.append(v[:7])
            elif t[0] == "ambient" and len(v) >= 3:
                amb = v[:3]
            elif t[0] == "camera" and len(v) >= 7:
                cam = v[:7]
    return _PlainScene(sph, lig, amb, cam)


class ClockSampler(threading.Thread):
    """Samples SM clock and clock-event (throttle) reasons of one GPU through NVML while the
    timed regions run."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self.stop_flag = False
        self.err = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonGpuIdle", 0x1): "gpu_idle",
                getattr(nv, "nvmlClocksEventReasonApplicationsClocksSetting", 0x2): "applications_clocks_setting",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonSyncBoost", 0x10): "sync_boost",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
                getattr(nv, "nvmlClocksEventReasonDisplayClockSetting", 0x100): "display_clock_setting",
            }
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                bits = get_reasons(h)
                for b, n in names.items():
                    if bits & b and n != "gpu_idle":
                        self.reasons.add(n)
                time.sleep(self.period)
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def summary(self):
        s = sorted(self.samples)
        # "under load": the upper half of the samples (idle gaps between regions pull clocks down)
        load = s[len(s) // 2:] if s else []
        med = load[len(load) // 2] if load else None
        out = {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}
        if self.err:
            out["error"] = self.err
        return out


def ncu_traffic(workload="complex"):
    """DRAM bytes (read + write) of ONE FRAME -- all launches of a step, summed -- from the committed `ncu --set full` capture
    of this workload (profiles/r02_executed_<workload>.json, dram__bytes_read.sum + dram__bytes_write.sum per launch)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_executed_%s.json" % workload)) as f:
            d = json.load(f)
        return int(sum((k.get("dram_read_mb") or 0) + (k.get("dram_write_mb") or 0) for k in d["kernels"]) * 1e6)
    except Exception:  # noqa: BLE001
        return None


def ncu_executed(workload="complex"):
    """EXECUTED FP32 work of one frame from the committed ncu capture of this workload (profiles/r02_executed_<workload>.json,
    written by scripts/ncu_opcodes.py from an `ncu --set full --import-source on` run of scripts/ncu_target.py): executed
    flops, their fraction of the FFMA peak over the serialised kernel times, and per kernel the FMA-pipe / issue-slot /
    occupancy / L1 / instruction-cache figures the north star names."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_executed_%s.json" % workload)) as f:
            d = json.load(f)
        return {"fp32_flops_executed_per_frame": d["fp32_flops_executed"], "fp64_flops_executed_per_frame": d["fp64_flops_executed"],
                "executed_frac": round(d["executed_fp32_frac_of_peak"], 4), "sum_kernel_us_under_ncu": round(d["sum_us"], 1),
                "kernels": [{"name": k["name"], "us": round(k["us"], 1), "executed_frac": round(k["executed_fp32_frac_of_peak"] or 0, 4),
                             "fma_pipe_active_pct": k["fma_pipe_pct"], "issue_slots_active_pct": k["issue_pct"],
                             "achieved_occupancy_pct": k["occupancy_pct"], "l1_hit_pct": k["l1_hit_pct"], "icache_hit_pct": k["icache_hit_pct"],
                             "smem_wavefronts": k["smem_wavefronts"], "registers_per_thread": k["regs"]} for k in d["kernels"]],
                "source": "profiles/r02_executed_%s.json (ncu --set full --import-source on, scripts/ncu_opcodes.py)" % workload}
    except Exception:  # noqa: BLE001
        return None


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except (ValueError, IndexError):
            return local_rank
    return local_rank


# -------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own CPU renderer on this box's host cores
def run_reference_frames(steps, warmup, budget_s=150.0, workload="complex"):
    """Times `steps` renders with oracle/_ref/ref_harness (the unmodified reference sources, OpenMP
    loop of src/main.cpp:185 on all host threads).  Each step is a bounded sample of the frame
    (every `pix_step`-th pixel) sized so the run fits the budget.  Falls back to the C port."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py
    scene = load_workload_plain(workload)
    scene_file = SCENE
    if WORKLOADS[workload][0].startswith("synth:"):
        # the reference reads scene FILES: write the synthetic scene in its text grammar (%.6f = the same doubles)
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import gen_scene
        import tempfile
        _, nn, seed = WORKLOADS[workload][0].split(":")
        scene_file = os.path.join(tempfile.gettempdir(), "rtb200_%s.txt" % workload)
        with open(scene_file, "w") as f:
            f.write(gen_scene.to_text(*gen_scene.generate(int(nn), int(seed))))
    elif workload != "complex":
        scene_file = os.path.join(ROOT, "tests", "golden", "scenes", WORKLOADS[workload][0] + ".txt")
    cores = os.cpu_count() or 1
    kind = "reference" if oracle_py.ref_available() else "port"

    def one(pix_step):
        if kind == "reference":
            out = oracle_py.ref_harness("render", scene_file, W, H, DEPTH, "-", "omp", pix_step,
                                        env={"OMP_NUM_THREADS": str(cores)})
            return float([l for l in out.splitlines() if "time:" in l][0].split()[2])
        t0 = time.perf_counter()
        oracle_py.render(scene, W, H, DEPTH, pix_step=pix_step, nthreads=0)
        return time.perf_counter() - t0

    probe_step = 16 if workload in ("complex", "medium", "simple") else 4096
    t_probe = one(probe_step) * probe_step       # estimate of a full frame
    total = max(1, steps + warmup)
    pix_step = 1
    while t_probe / pix_step * total > budget_s and pix_step < 65536:
        pix_step *= 2
    rays = oracle_py.render(scene, W, H, DEPTH, pix_step=pix_step, nthreads=0)["counters"]["rays"]
    for _ in range(warmup):
        one(pix_step)
    times = [one(pix_step) for _ in range(steps)]
    sec = sum(times) / len(times)
    return {"mrays_s": rays / sec * 1e-6, "ms_per_step": sec * 1e3, "cores": cores, "kind": kind,
            "sample": "every %d-th pixel of the %s frame (%d rays/step), OpenMP schedule(dynamic) on %d threads, mean of %d"
                      % (pix_step, WORKLOAD, rays, cores, steps),
            "best_ms": min(times) * 1e3}


def main_reference(args, rank):
    if rank != 0:
        return 0
    steps = max(1, args.steps)
    r = run_reference_frames(steps, args.warmup)
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": round(r["mrays_s"], 3), "unit": "Mrays/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": round(r["ms_per_step"], 3),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "reference scene file (fixture)",
        "config": {"workload": WORKLOAD, "parallelism": "openmp x%d host threads" % r["cores"]},
        "cpu_baseline": {"value": round(r["mrays_s"], 3), "unit": "Mrays/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": round(r["mrays_s"], 3), "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


DUMP_BYTES = 64 << 20


def dump_frame(out_dir, frame):
    """Writes the [H, W, 3] frame of the last timed step as <out_dir>/rgb.npy (float32).  A frame larger than
    DUMP_BYTES is cut to a fixed, seeded sample of whole rows; their indices go to <out_dir>/rgb_rows.npy (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    a = frame.cpu().numpy().astype(np.float32)
    h, w, _ = a.shape
    if a.nbytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(h, DUMP_BYTES // (w * 3 * 4 + 8), replace=False))
        np.save(os.path.join(out_dir, "rgb_rows.npy"), rows.astype(np.float64))
        a = a[rows]
    np.save(os.path.join(out_dir, "rgb.npy"), a)


# -------------------------------------------------------------------------------------------------
def measure_extra(torch, dist, rtb200, local_rank, rank, n, workload, gather, steps=8, warmup=3):
    """N > 1: a short device-timed run of ANOTHER BASELINE config in the same process group (the 8-GPU config the
    north star names is config 4: synthetic 10 k spheres at 3840x2160), so that the driver's scaling record carries it.
    Same method as the headline: CUDA events per step, L2 flushed between steps, max over ranks, assembled frame checked
    against rank 0's own full-frame render."""
    import numpy as np
    _, w_, h_, d_, label = WORKLOADS[workload]
    dev = torch.device("cuda", local_rank)
    scene = load_workload(workload)
    r = rtb200.Renderer(local_rank, mode="fast")
    r.upload(scene)
    stream = torch.cuda.current_stream(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    if gather == "peer":
        pf = rtb200.PeerFrame(r, w_, h_, BAND_H, rank, n, dist)
        full = pf.frame() if rank == 0 else None

        def step():
            pf.render(d_, stream.cuda_stream)
            pf.release(stream.cuda_stream)
    else:
        bands = rtb200.BandGather(w_, h_, BAND_H, rank, n, dev, dist)
        full = bands.full

        def step():
            r.render_bands_device(w_, h_, d_, BAND_H, rank, n, bands.part.data_ptr(), stream.cuda_stream)
            bands.gather()
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        flush.fill_(k & 0xff)
        ev[k][0].record(stream)
        step()
        ev[k][1].record(stream)
    torch.cuda.synchronize()
    dist.barrier()
    t = torch.tensor([sum(a.elapsed_time(b) for a, b in ev) / steps], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out = {"workload": label, "gather": gather, "n_gpus": n, "steps": steps, "ms_per_step": round(float(t.item()), 4)}
    if rank == 0:
        full.zero_()
    torch.cuda.synchronize()
    dist.barrier()
    step()
    torch.cuda.synchronize()
    dist.barrier()
    if rank == 0:
        own, st = r.render(w_, h_, d_)
        rays = int(st.closest_queries + st.shadow_queries)
        out.update({"rays_per_frame": rays, "value": round(rays / (out["ms_per_step"] * 1e-3) * 1e-6, 1), "unit": "Mrays/s",
                    "frame_check": "identical" if np.array_equal(own, full.cpu().numpy()) else "DIFFERENT"})
    torch.cuda.synchronize()
    dist.barrier()
    if gather == "peer":
        pf.close()
    r.close()
    del flush
    return out


def main_b200(args, rank, local_rank, world):
    import torch
    import rtb200

    n = world
    dist = None
    if n > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)

    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()

    scene = load_workload(args.workload)
    r = rtb200.Renderer(local_rank, mode="fast", accel=args.accel)
    r.upload(scene)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
    # a real (non-default) stream: the library launches on the stream it is handed, and the
    # CUDA events below are recorded on that same stream
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    peer = n > 1 and args.gather == "peer"
    if peer:
        # rank 0 owns the assembled frame; everybody's kernels write their rows into it (CUDA IPC + NVLink)
        pf = rtb200.PeerFrame(r, W, H, BAND_H, rank, n, dist)
        full = pf.frame() if rank == 0 else None

        def step_device():
            pf.render(DEPTH, stream.cuda_stream)
            pf.release(stream.cuda_stream)          # `value`: the frame stays in rank 0's HBM, nothing consumes it
    else:
        bands = rtb200.BandGather(W, H, BAND_H, rank, n, dev, dist)
        part, full = bands.part, bands.full

        def step_device():
            r.render_bands_device(W, H, DEPTH, BAND_H, rank, n, part.data_ptr(), stream.cuda_stream)
            if n > 1:
                bands.gather()                      # NCCL gather of the 8-bit bands to rank 0 + row scatter

    # ray counts of the frame (one counted render on rank 0's full frame, outside the timed region)
    _, st = r.render(W, H, DEPTH)
    rays = int(st.closest_queries + st.shadow_queries)
    assert st.filter_violations == 0

    for _ in range(max(3, args.warmup)):
        step_device()
    torch.cuda.synchronize()
    if n > 1:
        dist.barrier()
    K = max(1, args.steps)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    torch.cuda.synchronize()
    for k in range(K):
        flush.fill_(k & 0xff)                     # evict L2 between timed iterations (untimed)
        ev[k][0].record(stream)
        step_device()
        ev[k][1].record(stream)
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        # before the barrier: in peer mode the other ranks may render into rank 0's frame once they pass it
        dump_frame(args.dump_outputs, full if n > 1 else part[:H * W * 3].view(H, W, 3))
    if n > 1:
        dist.barrier()
    # kernels per frame, counted in the steady state the timed loop ran in (the library picks the number of wavefront
    # levels from the previous frame's ray counts, so the very first frame of a scene may launch more)
    if n == 1:
        _, st_l = r.render(W, H, DEPTH)
    elif peer:
        st_l = pf.render(DEPTH, stream.cuda_stream, want_stats=True)
        pf.release(stream.cuda_stream)
    else:
        st_l = r.render_bands_device(W, H, DEPTH, BAND_H, rank, n, part.data_ptr(), stream.cuda_stream, want_stats=True)
    launches_per_step = int(st_l.kernel_launches)
    torch.cuda.synchronize()
    if n > 1:
        dist.barrier()
    # ---- N > 1: the assembled frame of one more sharded step must be rank 0's own full-frame render, byte for byte
    frame_check = None
    if n > 1:
        if rank == 0:
            full.zero_()                                # (stale pixels of the timed frames must not pass the check)
        torch.cuda.synchronize()
        dist.barrier()
        step_device()
        torch.cuda.synchronize()
        dist.barrier()
        if rank == 0:
            own, _ = r.render(W, H, DEPTH)
            import numpy as np
            frame_check = "identical" if np.array_equal(own, full.cpu().numpy()) else "DIFFERENT"
        torch.cuda.synchronize()
        dist.barrier()
    ms_total = sum(a.elapsed_time(b) for a, b in ev)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if n > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item()) / K

    # ---- e2e: public API with host buffers; scene upload (H2D) + render + frame to pinned host (D2H)
    if n == 1:
        host_frame = r.pinned_frame(W, H)

        def step_e2e():
            r.upload(scene)
            r.render(W, H, DEPTH, out=host_frame, want_stats=False)
        d2h = W * H * 3
    else:
        # N > 1: ONE host frame in shared memory (POSIX shm, page-locked by every rank's process); every rank renders its
        # bands and copies them over ITS OWN host link straight to their image positions (rt_render_bands_host) -- the
        # N downloads run concurrently and nothing crosses between the GPUs.  "Frame complete" = a sequence flag per rank
        # in the same shared segment, back-pressure = rank 0's acknowledge word.
        from multiprocessing import shared_memory
        import numpy as np
        nbytes = H * W * 3
        box = [None]
        if rank == 0:
            shm = shared_memory.SharedMemory(create=True, size=nbytes + 4096)
            box = [shm.name]
        dist.broadcast_object_list(box, src=0)
        if rank != 0:
            shm = shared_memory.SharedMemory(name=box[0])
        host_frame = np.ndarray((H, W, 3), dtype=np.uint8, buffer=shm.buf)
        words = np.ndarray((256,), dtype=np.uint32, buffer=shm.buf, offset=nbytes + (-nbytes) % 1024)
        if rank == 0:
            host_frame[:] = 0
            words[:] = 0
        dist.barrier()
        frame_ptr = host_frame.ctypes.data
        rtb200.host_register(frame_ptr, nbytes)
        seq = [0]

        def step_e2e():
            seq[0] += 1
            k = seq[0]
            r.upload(scene)
            while int(words[128]) < k - 1:              # frame k-1 consumed by rank 0?
                pass
            r.render_bands_host(W, H, DEPTH, BAND_H, rank, n, frame_ptr)   # returns when this rank's rows are in host memory
            words[rank] = k
            if rank == 0:
                while any(int(words[j]) < k for j in range(n)):           # the whole frame is in host memory
                    pass
                words[128] = k
        d2h = W * H * 3
    h2d = r.scene_bytes()
    Ke = max(1, min(K, 200))
    for _ in range(3):
        step_e2e()
    torch.cuda.synchronize()
    if n > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        step_e2e()
    torch.cuda.synchronize()
    if n > 1:
        dist.barrier()
    te = torch.tensor([(time.perf_counter() - t0) / Ke], dtype=torch.float64, device=dev)
    if n > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_s = float(te.item())
    e2e_check = None
    if n > 1:
        # the host frame the ranks assembled must be rank 0's own full-frame render, byte for byte
        if rank == 0:
            host_frame[:] = 0
        dist.barrier()
        step_e2e()
        dist.barrier()
        if rank == 0:
            own, _ = r.render(W, H, DEPTH)
            e2e_check = "identical" if np.array_equal(own, host_frame) else "DIFFERENT"
        dist.barrier()
        rtb200.host_unregister(frame_ptr)
        del host_frame, words
        shm.close()
        if rank == 0:
            shm.unlink()

    # ---- dominant kernel (level-0 k_shadow) timed alone with the library's CUDA events
    k_ms, lvl0_ms, frame_ms, k_rays = None, None, None, None
    if rank == 0 and n == 1:
        msk, ms0, msf = [], [], []
        r.set_option("level_timing", 1)                     # events between the level-0 kernels (PDL off for these renders)
        for _ in range(30):
            flush.fill_(1)
            _, s2 = r.render(W, H, DEPTH)
            msk.append(s2.ms_shadow0); ms0.append(s2.ms_level0); msf.append(s2.ms_device)
        k_ms, lvl0_ms, frame_ms = sum(msk) / len(msk), sum(ms0) / len(ms0), sum(msf) / len(msf)
        r.set_option("level_timing", 0)
        _, s1 = r.render(W, H, 1)                           # level 0 only: pixels + L x primary hits
        k_rays = int(s1.shadow_queries)                     # the shadow queries k_shadow(level 0) answers

    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- N > 1 on the headline workload: carry BASELINE config 4 (the one the north star names for 8 GPUs) in the same record
    extra = []
    if n > 1 and args.workload == "complex" and not args.no_extra:
        for g in ("peer", "nccl"):
            try:
                extra.append(measure_extra(torch, dist, rtb200, local_rank, rank, n, "synth10k", g))
            except Exception as e:  # noqa: BLE001
                extra.append({"workload": "synth10k", "gather": g, "error": repr(e)})

    if rank == 0:
        peak, peak_mhz = rtb200.measure_fp32_peak(local_rank)
        nsph = scene.nspheres
        frame_flops = FLOP_PER_TEST * nsph * rays
        line = {
            "metric": "Mrays/s", "value": round(rays / (ms_per_step * 1e-3) * 1e-6, 1), "unit": "Mrays/s",
            "n_gpus": n, "steps": K, "warmup": max(3, args.warmup), "ms_per_step": round(ms_per_step, 5),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 filter / f64 decide",
            "data": ("reference scene file %s.txt (tests/golden fixture, identical doubles); no dataset involved" % args.workload)
                    if not WORKLOADS[args.workload][0].startswith("synth") else "synthetic scene, scripts/gen_scene.py (SURVEY 8d spec)",
            "config": {"workload": WORKLOAD, "rays_per_frame": rays, "parallelism": "interleaved %d-row bands x %d GPU%s"
                       % (BAND_H, n, "" if n == 1 else ("s, rows stored into rank 0's frame over NVLink peer memory + completion flags"
                                                         if peer else "s, NCCL gather to rank 0")), "band_h": BAND_H,
                       "l2": "flushed between timed steps (256 MiB write, untimed)"},
            "e2e": {"value": round(rays / e2e_s * 1e-6, 1), "unit": "Mrays/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": round(e2e_s * 1e3, 4), "steps": Ke,
                    "path": "rt_upload_scene + rt_render into pinned host memory" if n == 1 else
                            "rt_upload_scene + rt_render_bands_host on every rank: bands copied over each GPU's own host link into one "
                            "shared page-locked host frame (POSIX shm), completion flags in the same segment"},
            "gpu_launches": launches_per_step * K,
            "clocks": sampler.summary(),
        }
        ach = frame_flops / (ms_per_step * 1e-3) * 1e-12
        bundle = {"walks": int(st.bundle_walks), "candidates_per_walk": round(st.bundle_candidates / max(1, st.bundle_walks), 2),
                  "note": "a culled warp-level table walk tests only the spheres its ray bundle's cone can touch"}
        lbvh = scene.nspheres >= 1024 or args.accel == 2
        # `frac` = WHOLE-FRAME algorithmic fraction: the reference's brute-force work (16 flop x spheres x rays) retired per
        # second over the measured FFMA issue peak.  It is NOT pipe utilisation: culling / early-out skip most of those
        # tests.  What the FP32 pipe really executed is `executed` (ncu capture of this command, profiles/).
        roof = {"bound": "fp32", "unit": "TFLOP/s", "peak": round(peak * 1e-12, 2), "achieved": round(ach, 2),
                "frac": None if lbvh else round(ach / (peak * 1e-12), 4),
                "kernel": "whole frame: all %d launches of a step" % launches_per_step, "flops": frame_flops, "flop_per_test": FLOP_PER_TEST,
                "note": "achieved = ALGORITHMIC flops (16 x spheres x rays: the reference's brute force, SURVEY 8d) / frame time; "
                        "frac = achieved / measured FFMA peak for the whole frame; executed.* = what the kernels really issued "
                        "(ncu per-opcode thread-instruction counts: FFMA 2, FFMA2 4, FMUL/FADD 1, FMUL2/FADD2 2 flop)",
                "peak_source": "measured live: FFMA issue peak of this GPU (rt_measure_fp32_peak, SM clock %.0f MHz); "
                               "MEASURED_PEAKS.json has no FP32 entry (nominal 148 x 128 x 2 x 1.965 GHz = 74.5)" % peak_mhz,
                "bundle_culling": bundle, "traffic": ncu_traffic(args.workload), "executed": ncu_executed(args.workload)}
        if lbvh:
            roof["note_lbvh"] = ("LBVH workload: a brute-force-based fraction is meaningless here (SURVEY 8d), frac is null; "
                                 "candidates_per_walk / fp64 counts are the executed-work figures")
            roof["lbvh"] = {"bundle_walks": int(st.bundle_walks), "candidates_per_bundle_walk": bundle["candidates_per_walk"],
                            "bundle_fallbacks": int(st.bundle_fallbacks), "fp64_sphere_evaluations_per_ray": round(st.fp64_intersections / max(1, rays), 4)}
        if k_ms:
            a0 = FLOP_PER_TEST * nsph * k_rays / (k_ms * 1e-3) * 1e-12
            roof["dominant_kernel"] = {"kernel": "k_shadow, reflection level 0 (one any-hit query per light per camera-ray hit)",
                                       "kernel_ms": round(k_ms, 5), "kernel_rays": k_rays, "kernel_flops_algorithmic": FLOP_PER_TEST * nsph * k_rays,
                                       "kernel_share_of_frame": round(k_ms / frame_ms, 4), "level0_ms": round(lvl0_ms, 5),
                                       "algorithmic_speedup": round(a0 / (peak * 1e-12), 4),
                                       "algorithmic_speedup_note": "algorithmic flops of this kernel's rays / its time / FFMA peak; > 1 means "
                                                                   "the kernel does not execute the brute-force work it is charged with (bundle culling)"}
        line["roofline"] = roof
        if n == 1 and not args.no_cpu_baseline:
            try:
                cb = run_reference_frames(3, 1, budget_s=30.0, workload=args.workload)
                line["cpu_baseline"] = {"value": round(cb["mrays_s"], 3), "unit": "Mrays/s", "cores": cb["cores"],
                                        "kind": cb["kind"], "sample": cb["sample"]}
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"value": None, "unit": "Mrays/s", "cores": os.cpu_count(), "kind": "reference",
                                        "sample": "failed: %r" % (e,)}
        if extra:
            line["extra_workloads"] = extra
        if frame_check is not None:
            line["frame_check"] = frame_check
            line["e2e"]["frame_check"] = e2e_check
            if e2e_check == "DIFFERENT":
                frame_check = "DIFFERENT"
        print(json.dumps(line), flush=True)
        if frame_check == "DIFFERENT":
            raise RuntimeError("the frame assembled from %d ranks differs from rank 0's own full-frame render" % n)
    if peer:
        torch.cuda.synchronize()
        err = pf.error()
        dist.barrier()
        pf.close()
        if err:
            raise RuntimeError("peer frame: a completion wait timed out (flag %d)" % (err - 1))
    r.close()
    if n > 1:
        dist.destroy_process_group()
    return 0


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be >= 1")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=300, help="timed steps (frames)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="complex", choices=sorted(WORKLOADS))
    ap.add_argument("--accel", type=int, default=None, help="0 auto, 1 table walks, 2 LBVH (rt_set_option accel)")
    ap.add_argument("--no-extra", action="store_true", help="N > 1: skip the extra_workloads block (config 4)")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"], help="N > 1: how the bands reach rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step to DIR/rgb.npy (float32), for comparing two builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm keeps no frame")
    global SCENE, W, H, DEPTH, WORKLOAD
    _, W, H, DEPTH, WORKLOAD = WORKLOADS[args.workload]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return main_reference(args, rank)
    if world == 1 and args.gpus > 1:
        # convenience: re-launch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(29500 + os.getpid() % 1000), os.path.abspath(__file__),
               "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup), "--workload", args.workload]
        if args.accel is not None:
            cmd += ["--accel", str(args.accel)]
        cmd += ["--gather", args.gather]
        if args.no_extra:
            cmd += ["--no-extra"]
        if args.no_cpu_baseline:
            cmd += ["--no-cpu-baseline"]
        if args.dump_outputs:
            cmd += ["--dump-outputs", os.path.abspath(args.dump_outputs)]
        return subprocess.call(cmd)
    return main_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    sys.exit(main())
