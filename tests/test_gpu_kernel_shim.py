"""libkernel_shim.so -- the reference's tile-launch C ABI (launch_gpu_kernel / upload_lights_and_ambience) -- driven
through ctypes the way the reference's ray_hybrid drives it, without the reference's sources: its structs built from the
layouts the shim asserts (ShimSphere 36 B, ShimLight 28 B, ShimCamera 88 B) in torch device memory, ragged 64x64 tiles on
three streams in turn with no sync between them.  The frame must be byte-identical to rt_render_tile of a Renderer that
uploaded the FP32-rounded scene directly, and within the colour bound (tests/colour_bound.py) of the oracle's colour of
that scene.  The scene cache (read back once per sphere pointer, camera pointer, sphere count and light count) is
checked against fresh renders.  Needs a B200: run with -m gpu."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
if TESTS not in sys.path:
    sys.path.insert(0, TESTS)

from colour_bound import colour_bound  # noqa: E402
from conftest import scene_path  # noqa: E402

pytestmark = pytest.mark.gpu

SHIM = os.path.join(ROOT, "cs420-ray-tracer_b200", "libkernel_shim.so")
SPHERE = np.dtype([("center", "<f4", 3), ("radius", "<f4"), ("albedo", "<f4", 3), ("metallic", "<f4"), ("shininess", "<f4")])
LIGHT = np.dtype([("position", "<f4", 3), ("color", "<f4", 3), ("intensity", "<f4")])
CAMERA = np.dtype([("origin", "<f4", 3), ("lower_left", "<f4", 3), ("horizontal", "<f4", 3), ("vertical", "<f4", 3),
                   ("forward", "<f4", 3), ("right", "<f4", 3), ("up", "<f4", 3), ("fov", "<f4")])
W, H, D, T = 200, 120, 5, 64


class Float3(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]


def test_struct_layouts():
    assert (SPHERE.itemsize, LIGHT.itemsize, CAMERA.itemsize) == (36, 28, 88)


def load_shim(path=SHIM):
    import rtb200
    rtb200.load_library()
    if not os.path.exists(path):
        rtb200.build_library()
    lib = C.CDLL(path)
    vp, i = C.c_void_p, C.c_int
    lib.upload_lights_and_ambience.argtypes = [vp, i, Float3]
    lib.upload_lights_and_ambience.restype = None
    lib.launch_gpu_kernel.argtypes = [vp, vp, i, i, vp, i, i, i, i, i, i, i, vp]
    lib.launch_gpu_kernel.restype = None
    lib.kernel_shim_invalidate.argtypes = []
    lib.kernel_shim_invalidate.restype = None
    return lib


@pytest.fixture(scope="module")
def shim(rt):
    return load_shim()


def shim_structs(sc):
    """The reference's GPUSphere / GPULight / GPUCamera arrays of a scene (FP32)."""
    sp = np.zeros(sc.nspheres, SPHERE)
    sp["center"], sp["radius"], sp["albedo"] = sc.spheres[:, 0:3], sc.spheres[:, 3], sc.spheres[:, 4:7]
    sp["metallic"], sp["shininess"] = sc.spheres[:, 7], sc.spheres[:, 9]
    li = np.zeros(sc.nlights, LIGHT)
    li["position"], li["color"], li["intensity"] = sc.lights[:, 0:3], sc.lights[:, 3:6], sc.lights[:, 6]
    cam = np.zeros(1, CAMERA)
    pos, look = sc.camera[0:3], sc.camera[3:6]
    cam["origin"] = pos
    cam["forward"] = (look - pos) / np.linalg.norm(look - pos)
    cam["fov"] = sc.camera[6]
    return sp, li, cam


def fp32_scene(rt, sp, li, amb, cam):
    """The scene as the shim hands it to rt_upload_scene: FP32 values widened to double, look = origin + forward
    (kernel_shim.cu), roughness column 1 - metallic."""
    s = np.zeros((len(sp), 10))
    s[:, 0:3], s[:, 3], s[:, 4:7] = sp["center"], sp["radius"], sp["albedo"]
    s[:, 7], s[:, 8], s[:, 9] = sp["metallic"], 1.0 - sp["metallic"].astype(np.float64), sp["shininess"]
    lights = np.zeros((len(li), 7))
    if len(li):
        lights[:, 0:3], lights[:, 3:6], lights[:, 6] = li["position"], li["color"], li["intensity"]
    pos = cam["origin"][0].astype(np.float64)
    camera = np.concatenate([pos, pos + cam["forward"][0].astype(np.float64), [float(cam["fov"][0])]])
    return rt.Scene(s, lights, np.asarray(amb, dtype=np.float32).astype(np.float64), camera)


def device(a):
    """A structured array copied to torch device memory (uint8 tensor; keep it alive while the pointer is used)."""
    import torch
    t = torch.from_numpy(np.frombuffer(a.tobytes(), dtype=np.uint8).copy() if a.nbytes else np.zeros(16, np.uint8)).cuda()
    torch.cuda.synchronize()
    return t


def upload_lights(shim, li, amb):
    li = np.ascontiguousarray(li)
    shim.upload_lights_and_ambience(li.ctypes.data if len(li) else None, len(li), Float3(*[float(x) for x in amb]))


def shim_frame(shim, sph_dev, n, nl, cam_dev, tiles=False):
    """One frame through launch_gpu_kernel: whole or in ragged TxT tiles on three streams in turn, one sync at the end."""
    import torch
    fb = torch.full((H, W, 3), -7.0, dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    if tiles:
        streams = [torch.cuda.Stream() for _ in range(3)]
        k = 0
        for y in range(0, H, T):
            for x in range(0, W, T):
                shim.launch_gpu_kernel(fb.data_ptr(), sph_dev.data_ptr(), n, nl, cam_dev.data_ptr(), x, y, min(T, W - x),
                                       min(T, H - y), W, H, D, streams[k % 3].cuda_stream)
                k += 1
    else:
        shim.launch_gpu_kernel(fb.data_ptr(), sph_dev.data_ptr(), n, nl, cam_dev.data_ptr(), 0, 0, W, H, W, H, D, None)
    torch.cuda.synchronize()
    return fb


def direct_frame(rt, sc):
    """rt_render_tile of a Renderer that uploaded `sc` itself."""
    import torch
    fb = torch.full((H, W, 3), -7.0, dtype=torch.float32, device="cuda:0")
    with rt.Renderer(0) as r:
        r.upload(sc)
        torch.cuda.synchronize()
        r.render_tile_device(W, H, D, (0, 0, W, H), fb.data_ptr())
        torch.cuda.synchronize()
    return fb


def test_tiles_on_three_streams_equal_the_direct_render(rt, oracle, shim):
    import torch
    sc = rt.load_scene(scene_path("complex"))
    sp, li, cam = shim_structs(sc)
    amb = np.asarray(sc.ambient, dtype=np.float32)
    upload_lights(shim, li, amb)
    sph_dev, cam_dev = device(sp), device(cam)
    shim.kernel_shim_invalidate()
    got = shim_frame(shim, sph_dev, len(sp), len(li), cam_dev, tiles=True)
    sc32 = fp32_scene(rt, sp, li, amb, cam)
    assert torch.equal(got, direct_frame(rt, sc32))
    o = oracle.render(sc32, W, H, D, want_fb=True, want_idx=True)
    bound = colour_bound(sc32, o["hit_idx"], W, H, D, o["shadow_mask"])
    err = np.abs(got.cpu().numpy().astype(np.float64) - o["fb"])
    assert (err <= bound).all(), (err / bound).max()


def test_scene_cache(rt, shim):
    """Every input the shim reads back is part of its cache key, or needs kernel_shim_invalidate() (in-place edits)."""
    import torch
    base = rt.load_scene(scene_path("medium"))
    sp, li, cam = shim_structs(base)
    amb = np.asarray(base.ambient, dtype=np.float32)
    cam_dev = device(cam)

    def check(sph_dev, spn, n, lights, nl, what):
        got = shim_frame(shim, sph_dev, n, nl, cam_dev)
        want = direct_frame(rt, fp32_scene(rt, spn[:n], lights[:nl], amb, cam))
        assert torch.equal(got, want), what
        return got

    upload_lights(shim, li, amb)
    a = device(sp)
    check(a, sp, len(sp), li, len(li), "first frame")
    # a new sphere pointer: another scene
    sp2, _, _ = shim_structs(rt.load_scene(scene_path("simple")))
    b = device(sp2)
    check(b, sp2, len(sp2), li, len(li), "new sphere pointer")
    # a new count at the same pointer
    check(a, sp, 20, li, len(li), "new sphere count")
    check(a, sp, len(sp), li, len(li), "count restored")
    # an in-place edit: stale until kernel_shim_invalidate()
    sp3 = sp.copy()
    sp3["albedo"] = sp3["albedo"][:, ::-1]
    sp3["metallic"] *= 0.5
    old = shim_frame(shim, a, len(sp), len(li), cam_dev)
    a.copy_(device(sp3))
    torch.cuda.synchronize()
    assert torch.equal(shim_frame(shim, a, len(sp), len(li), cam_dev), old), "an in-place edit is seen without invalidate"
    shim.kernel_shim_invalidate()
    check(a, sp3, len(sp3), li, len(li), "after kernel_shim_invalidate")
    # new lights and ambient
    li2 = li[::-1].copy()
    li2["color"] *= 0.5
    upload_lights(shim, li2, amb)
    check(a, sp3, len(sp3), li2, len(li2), "new upload_lights_and_ambience")
    # num_lights below the uploaded count (first launch after an upload), then changed between two launches with nothing
    # else changed (the light count is part of the cache key)
    upload_lights(shim, li2, amb)
    check(a, sp3, len(sp3), li2, 1, "num_lights 1 of 3")
    check(a, sp3, len(sp3), li2, 2, "num_lights 1 -> 2, nothing else changed")
    check(a, sp3, len(sp3), li2, 0, "num_lights 2 -> 0")
    check(a, sp3, len(sp3), li2, len(li2), "num_lights 0 -> 3")
    # zero spheres; zero lights uploaded
    check(a, sp3, 0, li2, len(li2), "no spheres")
    upload_lights(shim, li2[:0], amb)
    check(a, sp3, len(sp3), li2, 0, "no lights uploaded (the caller's count is larger)")
    check(a, sp3, len(sp3), li2[:0], 3, "no lights uploaded")


_CHILD = r"""
import ctypes as C, sys
sys.path[:0] = [%r, %r]
import numpy as np, torch
import test_gpu_kernel_shim as t, rtb200
from conftest import scene_path
shim = t.load_shim()
sc = rtb200.load_scene(scene_path("simple"))
sp, li, cam = t.shim_structs(sc)
t.upload_lights(shim, li, np.asarray(sc.ambient, dtype=np.float32))
a, c = t.device(sp), t.device(cam)
fb = torch.zeros((t.H, t.W, 3), dtype=torch.float32, device="cuda:0")
torch.cuda.synchronize()
x, y, w, h, depth = %s
shim.launch_gpu_kernel(fb.data_ptr(), a.data_ptr(), len(sp), len(li), c.data_ptr(), x, y, w, h, t.W, t.H, depth, None)
torch.cuda.synchronize()
print("returned")
"""


@pytest.mark.parametrize("args", [(150, 0, 64, 64, 5), (0, 0, 64, 64, 33), (0, 0, 0, 64, 5)],
                         ids=["tile_outside_the_image", "depth_33", "empty_tile"])
def test_errors_exit_like_cuda_check(rt, args):
    """launch_gpu_kernel returns void: an argument rt_render_tile rejects is printed and the process exits with status 1,
    as the reference's CUDA_CHECK does.  Run in a child process; every case is rejected on the host before any launch."""
    p = subprocess.run([sys.executable, "-c", _CHILD % (TESTS, ROOT, repr(args))], capture_output=True, text=True, timeout=300)
    assert p.returncode == 1, (p.returncode, p.stdout[-2000:], p.stderr[-2000:])
    assert "kernel_shim: rt_render_tile" in p.stderr and "returned" not in p.stdout
