"""Camera paths rendered frame-parallel over the ranks of a MultiRenderer (rt_multi_render_path).

Rank k % n renders frame k with rt_set_camera semantics, so every frame must be byte-identical to Renderer.render_path
on one context with the same options, and to the render of a context that uploaded the scene with that camera.  With
more ranks than devices the ranks share devices, so the n-rank code path also runs on a box with one GPU.
Tests marked gpu need a B200: run with -m gpu."""
import math

import numpy as np
import pytest

gpu = pytest.mark.gpu
W, H, D = 320, 180, 5
RT_ERR_ARG, RT_ERR_STATE = -1, -3


def with_camera(rt, scene, cam):
    return rt.Scene(scene.spheres, scene.lights, scene.ambient, np.asarray(cam, dtype=np.float64))


def orbit(cam, K, turn=2 * math.pi, lift=0.0):
    """K cameras on a circle about the look-at point at the scene camera's distance (a full turn by default)."""
    cam = np.asarray(cam, dtype=np.float64)
    look = cam[3:6]
    d = cam[0:3] - look
    r, a0 = math.hypot(d[0], d[2]), math.atan2(d[0], d[2])
    return np.array([[look[0] + r * math.sin(a0 + turn * k / K), look[1] + d[1] + lift * k / K, look[2] + r * math.cos(a0 + turn * k / K),
                      look[0], look[1], look[2], cam[6]] for k in range(K)])


def synth(rt, n, seed=7):
    import gen_scene
    return rt.Scene(*gen_scene.generate(n, seed))


def configure(r, opts):
    for k, v in (opts or {}).items():
        r.set_option(k, v)
    return r


def fresh(rt, scene, cam, mode="fast", accel=None, opts=None, size=(W, H, D)):
    """The frame of a newly created context that uploaded `scene` with camera `cam`."""
    with configure(rt.Renderer(0, mode=mode, accel=accel), opts) as r:
        r.upload(with_camera(rt, scene, cam))
        return r.render(*size, want_stats=False)[0]


def single_path(rt, scene, cams, mode="fast", accel=None, opts=None, size=(W, H, D)):
    with configure(rt.Renderer(0, mode=mode, accel=accel), opts) as r:
        r.upload(scene)
        return r.render_path(cams, *size).cpu().numpy()


def check_path(rt, n, scene, cams, mode="fast", accel=None, opts=None, size=(W, H, D), fresh_every=3):
    """rt_multi_render_path on n ranks against Renderer.render_path and against fresh uploads; then the ranks' camera."""
    with configure(rt.MultiRenderer(n, mode=mode, accel=accel), opts) as m:
        m.upload(scene)
        got = m.render_path(cams, *size).cpu().numpy()
        after, _ = m.render(*size, band_h=8, want_stats=False)
    want = single_path(rt, scene, cams, mode, accel, opts, size)
    assert got.shape == want.shape == (len(cams), size[1], size[0], 3)
    for k in range(len(cams)):
        assert np.array_equal(got[k], want[k]), "frame %d (rank %d of %d): %d bytes differ" % (
            k, k % n, n, int((got[k] != want[k]).sum()))
    for k in range(0, len(cams), fresh_every):
        assert np.array_equal(got[k], fresh(rt, scene, cams[k], mode, accel, opts, size)), "frame %d against a fresh upload" % k
    # every rank is left on the last camera: the banded render equals the last frame
    assert np.array_equal(after, want[-1]), "render after the path"
    return got


# ---- 1. ranks x modes ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("n", [1, 2, 3])
def test_path_equals_single_context_path(rt, scenes, n, mode):
    sc = scenes["complex"]
    cams = orbit(sc.camera, 7, lift=1.0)
    cams[3, 6] = 40.0                                      # a fov change inside the path; K = 7 is no multiple of 2 or 3
    check_path(rt, n, sc, cams, mode)


@gpu
def test_fewer_frames_than_ranks(rt, scenes):
    sc = scenes["complex"]
    check_path(rt, 3, sc, orbit(sc.camera, 2, turn=1.0), fresh_every=1)


# ---- 2. options and edges ------------------------------------------------------------------------------------------
CASES = {
    "antialias": dict(scene="complex", n=3, K=5, opts={"antialias": 1}, size=(160, 90, 4)),
    "tables_600": dict(scene=600, n=2, K=5, accel=1),
    "lbvh_2100": dict(scene=2100, n=2, K=4),
    "unaligned_99x41": dict(scene="complex", n=3, K=5, size=(99, 41, 3)),
    "depth0": dict(scene="complex", n=2, K=3, size=(W, H, 0)),
    "depth1": dict(scene="complex", n=3, K=4, size=(W, H, 1)),
    "wave_levels": dict(scene="complex", n=2, K=4, opts={"wave_levels": 3}),
}


@gpu
@pytest.mark.parametrize("case", list(CASES))
def test_options_and_edges(rt, scenes, case):
    c = CASES[case]
    sc = scenes[c["scene"]] if isinstance(c["scene"], str) else synth(rt, c["scene"])
    cams = orbit(sc.camera, c["K"], turn=1.5, lift=1.0)
    got = check_path(rt, c["n"], sc, cams, accel=c.get("accel"), opts=c.get("opts"), size=c.get("size", (W, H, D)))
    if c.get("size", (W, H, D))[2] == 0:
        assert not got.any(), "depth 0 is black"


# ---- 3. a camera beyond the scene: the synchronous full rebuild on one rank ----------------------------------------------
@gpu
@pytest.mark.parametrize("mode", ["fast", "bvh"])
def test_camera_beyond_the_scene_inside_the_path(rt, scenes, mode):
    sc = scenes["complex"]
    cams = orbit(sc.camera, 7, turn=1.0)
    look = cams[0, 3:6]
    cams[3] = [0, 3, 400, look[0], look[1], look[2], 40]   # rank 0 of 3 rebuilds here and again at frame 6 (back inside)
    check_path(rt, 3, sc, cams, mode, fresh_every=1)


# ---- 4. ordering on the caller's stream ---------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("which", ["side", "legacy_default"])
def test_frames_are_ordered_on_the_current_stream(rt, scenes, which):
    """Work already on the stream (a long sleep, then fill_(7)) happens before any frame is written; a reduction
    enqueued after the call, without a synchronise, sees the finished frames."""
    import torch
    dev = torch.device("cuda", 0)
    sc = scenes["complex"]
    cams = orbit(sc.camera, 6, turn=1.0)
    want = single_path(rt, sc, cams)
    s = torch.cuda.Stream(dev) if which == "side" else torch.cuda.default_stream(dev)
    with rt.MultiRenderer(3) as m:
        m.upload(sc)
        out = torch.zeros((len(cams), H, W, 3), dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        with torch.cuda.stream(s):
            torch.cuda._sleep(200_000_000)                 # ~0.1 s of device time before the fill
            out.fill_(7)
            m.render_path(cams, W, H, D, out=out)
            sums = out.view(len(cams), -1).sum(dim=1, dtype=torch.int64)
        s.synchronize()
        assert sums.cpu().tolist() == [int(f.sum(dtype=np.int64)) for f in want]
        assert np.array_equal(out.cpu().numpy(), want)


# ---- 5. frames that cross devices ---------------------------------------------------------------------------------------
@gpu
def test_frames_from_other_devices(rt, scenes):
    n = rt.load_library().rt_device_count()
    if n < 2:
        pytest.skip("needs at least 2 visible GPUs (the ranks share device 0 in the tests above)")
    sc = scenes["complex"]
    check_path(rt, n, sc, orbit(sc.camera, 2 * n + 1, lift=1.0), fresh_every=n)


# ---- 6. errors ----------------------------------------------------------------------------------------------------------
@gpu
def test_errors_through_the_library(rt, scenes):
    import torch
    lib = rt.load_library()
    cams = orbit(scenes["complex"].camera, 3)
    out = torch.empty((3, H, W, 3), dtype=torch.uint8, device="cuda:0")
    host = np.zeros((3, H, W, 3), dtype=np.uint8)
    with rt.MultiRenderer(2) as m:
        assert lib.rt_multi_render_path(m._h, cams.ctypes.data, 3, W, H, D, out.data_ptr(), None) == RT_ERR_STATE
        m.upload(scenes["complex"])
        assert lib.rt_multi_render_path(m._h, cams.ctypes.data, 3, W, H, D, host.ctypes.data, None) == RT_ERR_ARG
        for K, w, h, d in ((0, W, H, D), (3, 0, H, D), (3, W, 0, D), (3, W, H, -1)):
            assert lib.rt_multi_render_path(m._h, cams.ctypes.data, K, w, h, d, out.data_ptr(), None) == RT_ERR_ARG
        with pytest.raises(rt.RtError):
            m.render_path(cams, W, H, D, out=out[:2])
        torch.cuda.synchronize()
        assert np.array_equal(m.render_path(cams, W, H, D).cpu().numpy(), single_path(rt, scenes["complex"], cams))


# ---- 7. without a GPU ---------------------------------------------------------------------------------------------------
def test_argument_errors(rt):
    lib = rt.load_library()
    cams = np.zeros((3, 7))
    buf = np.zeros(64, dtype=np.uint8)
    assert lib.rt_multi_render_path(None, cams.ctypes.data, 3, 8, 8, 1, buf.ctypes.data, None) == RT_ERR_ARG
    assert lib.rt_multi_render_path(None, cams.ctypes.data, 0, 8, 8, 1, buf.ctypes.data, None) == RT_ERR_ARG
    assert lib.rt_multi_render_path(None, None, 3, 8, 8, 1, buf.ctypes.data, None) == RT_ERR_ARG
    assert lib.rt_multi_render_path(None, cams.ctypes.data, 3, 8, 8, 1, None, None) == RT_ERR_ARG
