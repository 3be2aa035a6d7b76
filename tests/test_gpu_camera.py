"""Camera moves without a re-upload (rt_set_camera, Renderer.render_path, ray_cuda --camera-path).

The contract: after rt_set_camera every render entry point produces exactly what a fresh rt_upload_scene of the same
spheres, lights and ambient with that camera produces.  Each comparison below therefore renders the same frame twice --
once on the moved context, once on a newly created context that uploaded the scene with that camera -- and requires equal
8-bit RGB, equal hit-index and shadow-mask buffers and equal ray counters.  Equal fp64_intersections and bundle counters
are the evidence that the camera table rebuilt on the device is the table the upload builds on the host.
Tests marked gpu need a B200: run with -m gpu."""
import math
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

gpu = pytest.mark.gpu
W, H, D = 320, 180, 5
COUNTERS = ("closest_queries", "hits", "shadow_queries", "occluded", "fp64_intersections", "sphere_tests", "bundle_walks",
            "bundle_candidates", "bundle_fallbacks")


def with_camera(rt, scene, cam):
    return rt.Scene(scene.spheres, scene.lights, scene.ambient, np.asarray(cam, dtype=np.float64))


def orbit(cam, K, turn=2 * math.pi, lift=0.0, fov=None):
    """K cameras on a circle about the look-at point at the scene camera's distance (a full turn by default)."""
    cam = np.asarray(cam, dtype=np.float64)
    look = cam[3:6]
    d = cam[0:3] - look
    r, a0 = math.hypot(d[0], d[2]), math.atan2(d[0], d[2])
    rows = []
    for k in range(K):
        a = a0 + turn * k / K
        rows.append([look[0] + r * math.sin(a), look[1] + d[1] + lift * k / K, look[2] + r * math.cos(a),
                     look[0], look[1], look[2], cam[6] if fov is None else fov])
    return np.array(rows)


def make_renderer(rt, mode, accel, opts):
    r = rt.Renderer(0, mode=mode, accel=accel)
    for k, v in opts.items():
        r.set_option(k, v)
    return r


def assert_same(got, want, what, counters=COUNTERS):
    rgb, hit, mask, st = got
    rgb0, hit0, mask0, st0 = want
    assert np.array_equal(hit, hit0), "%s: hit indices differ at %s" % (what, np.argwhere(hit != hit0)[:5].tolist())
    assert np.array_equal(mask, mask0), "%s: shadow masks differ" % what
    assert np.array_equal(rgb, rgb0), "%s: rgb differs in %d samples" % (what, int((rgb != rgb0).sum()))
    for k in counters:
        assert getattr(st, k) == getattr(st0, k), "%s: %s %d != %d" % (what, k, getattr(st, k), getattr(st0, k))
    assert list(st.alive) == list(st0.alive), what
    assert st.filter_violations == 0 and st0.filter_violations == 0, what


def fresh_debug(rt, scene, cam, mode="fast", accel=None, opts=None, size=(W, H, D)):
    """render_debug of a newly created context that uploaded `scene` with camera `cam`."""
    with make_renderer(rt, mode, accel, opts or {}) as r:
        r.upload(with_camera(rt, scene, cam))
        return r.render_debug(*size)


def follow(rt, scene, cams, mode="fast", accel=None, opts=None, size=(W, H, D), counters=COUNTERS):
    """Moves one context along `cams` and compares every frame with a fresh upload."""
    with make_renderer(rt, mode, accel, opts or {}) as r:
        r.upload(scene)
        for k, cam in enumerate(cams):
            r.set_camera(cam[0:3], cam[3:6], cam[6])
            assert_same(r.render_debug(*size), fresh_debug(rt, scene, cam, mode, accel, opts, size), "camera %d %s" % (k, list(cam)),
                        counters)


def synth(rt, n, seed=7):
    import gen_scene
    return rt.Scene(*gen_scene.generate(n, seed))


# ---- 1. orbit paths --------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", ["fast", "bvh", "exact"])
@pytest.mark.parametrize("name", ["simple", "medium", "complex"])
def test_orbit_matches_fresh_upload(rt, scenes, name, mode):
    follow(rt, scenes[name], orbit(scenes[name].camera, 12, lift=2.0), mode)


@gpu
@pytest.mark.parametrize("n", [600, 2500])        # camera table staged in shared memory / streamed through TMA tiles
def test_orbit_sorted_tables_of_synthetic_scenes(rt, n):
    sc = synth(rt, n)
    follow(rt, sc, orbit(sc.camera, 10, turn=1.5), accel=1)


@gpu
@pytest.mark.parametrize("n", [1500, 2100])       # LBVH scenes: lookup tables built on the host / on the device (>= 2048)
def test_orbit_lookup_tables_of_lbvh_scenes(rt, n):
    sc = synth(rt, n)
    follow(rt, sc, orbit(sc.camera, 8, turn=1.0))


# ---- 2. oracle parity along a path -----------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", ["fast", "bvh"])
def test_oracle_parity_along_a_path(rt, oracle, scenes, mode):
    sc = scenes["complex"]
    with rt.Renderer(0, mode=mode) as r:
        r.upload(sc)
        for cam in orbit(sc.camera, 4, turn=math.pi, lift=3.0):
            r.set_camera(cam[0:3], cam[3:6], cam[6])
            rgb, hit, mask, st = r.render_debug(160, 90, 5)
            o = oracle.render(with_camera(rt, sc, cam), 160, 90, 5, want_idx=True)
            assert np.array_equal(hit, o["hit_idx"]) and np.array_equal(mask, o["shadow_mask"])
            ok, pct, mx = rt.compare_rgb(o["rgb"], rgb, 0.5)
            assert ok and mx <= 2, (pct, mx)
            for k in ("closest_queries", "hits", "shadow_queries", "occluded"):
                assert getattr(st, k) == o["counters"][k], k
            assert st.filter_violations == 0


# ---- 3. edge cameras ---------------------------------------------------------------------------------------------------
def edge_path(scene):
    cam = np.asarray(scene.camera, dtype=np.float64)
    s = scene.spheres[np.argmax(scene.spheres[:, 3] * (scene.spheres[:, 3] < 50))]     # the largest sphere but the ground
    c, r = s[0:3], s[3]
    look = cam[3:6]
    return np.array([
        list(cam[0:3]) + [look[0] + 3, look[1] + 1, look[2]] + [cam[6]],                # only the look-at changes
        list(cam[0:3]) + [look[0] + 3, look[1] + 1, look[2]] + [cam[6] * 0.5],          # only the fov changes
        list(c + [0.3 * r, 0.2 * r, 0.1 * r]) + list(look) + [cam[6]],                    # inside a sphere (bit 30, never culled)
        list(cam[0:3] + [1, 0.5, 0]) + list(look) + [cam[6]],                             # ... and out again
        [0, 3, 400, look[0], look[1], look[2], 40],                                       # beyond the scene: delta64 changes
        list(cam),                                                                        # ... and back
        list(c) + list(look) + [cam[6]],                                                  # exactly on a sphere centre
        list(c) + list(look) + [cam[6]],                                                  # the same camera again
    ])


@gpu
@pytest.mark.parametrize("mode", ["fast", "bvh"])
def test_edge_cameras(rt, scenes, mode):
    sc = scenes["complex"]
    follow(rt, sc, edge_path(sc), mode)


@gpu
def test_edge_cameras_sorted_streamed_tables(rt):
    sc = synth(rt, 2500)
    follow(rt, sc, edge_path(sc), accel=1)


@gpu
def test_set_camera_keeps_the_layout_of_the_last_upload(rt, scenes):
    """A new accel option takes effect at the next upload only -- also through the full-rebuild path."""
    sc = scenes["complex"]
    far = [0, 3, 400, 0, 0, -20, 40]
    with rt.Renderer(0, mode="fast", accel=2) as r:
        r.upload(sc)
        r.set_option("accel", 1)
        for cam in (orbit(sc.camera, 3)[1], far):
            r.set_camera(cam[0:3], cam[3:6], cam[6])
            assert_same(r.render_debug(W, H, D), fresh_debug(rt, sc, cam, accel=2), str(cam))


# ---- 4. other render paths ---------------------------------------------------------------------------------------------
@gpu
def test_supersampling(rt, scenes):
    sc = scenes["medium"]
    follow(rt, sc, orbit(sc.camera, 4, turn=1.0)[1:], opts={"antialias": 1}, size=(160, 90, 4))


@gpu
@pytest.mark.parametrize("mode", ["fast", "bvh"])
def test_bands_frame_and_tiles(rt, scenes, mode):
    import torch
    sc = scenes["complex"]
    band_h, n = 8, 3
    dev = torch.device("cuda", 0)
    with rt.Renderer(0, mode=mode) as r:
        r.upload(sc)
        for cam in orbit(sc.camera, 4, turn=1.2)[1:]:
            r.set_camera(cam[0:3], cam[3:6], cam[6])
            want = fresh_debug(rt, sc, cam, mode)[0]
            bands = []
            for rank in range(n):
                buf = torch.zeros((rt.band_rows(H, band_h, rank, n), W, 3), dtype=torch.uint8, device=dev)
                r.render_bands_device(W, H, D, band_h, rank, n, buf.data_ptr())
                bands.append((rt.band_row_list(H, band_h, rank, n), buf))
            frame = torch.zeros((H, W, 3), dtype=torch.uint8, device=dev)
            for rank in range(n):
                r.render_bands_frame(W, H, D, band_h, rank, n, frame.data_ptr())
            fb = torch.zeros((H, W, 3), dtype=torch.float32, device=dev)
            for tile in ((0, 0, 100, 64), (100, 0, 220, 64), (0, 64, 320, 116)):
                r.render_tile_device(W, H, D, tile, fb.data_ptr())
            torch.cuda.synchronize()
            got = np.zeros_like(want)
            for rows, buf in bands:
                got[rows] = buf.cpu().numpy()
            assert np.array_equal(got, want)
            assert np.array_equal(frame.cpu().numpy(), want)
            q = (255.99 * np.minimum(1.0, fb.cpu().numpy())).astype(np.int32).astype(np.uint8)
            with rt.Renderer(0, mode=mode) as f:
                f.upload(with_camera(rt, sc, cam))
                fb0 = torch.zeros_like(fb)
                f.render_tile_device(W, H, D, (0, 0, W, H), fb0.data_ptr())
                torch.cuda.synchronize()
            assert torch.equal(fb, fb0)
            assert np.abs(q.astype(int) - want.astype(int)).max() <= 1


@gpu
@pytest.mark.parametrize("n", [1, 2, 3])
def test_multi_renderer(rt, scenes, n):
    sc = scenes["complex"]
    with rt.MultiRenderer(n) as m:
        m.upload(sc)
        for cam in orbit(sc.camera, 4, turn=1.0)[1:]:
            m.set_camera(cam[0:3], cam[3:6], cam[6])
            rgb, st = m.render(W, H, D, band_h=8)
            rgb0, _, _, st0 = fresh_debug(rt, sc, cam)
            assert np.array_equal(rgb, rgb0)
            for k in COUNTERS:
                assert getattr(st, k) == getattr(st0, k), k


# ---- 5. concurrency ----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", ["fast", "bvh"])
def test_render_path_equals_a_synchronous_loop(rt, scenes, mode):
    sc = scenes["complex"]
    cams = orbit(sc.camera, 8, lift=1.0)
    cams[3, 6] = 40.0                                      # a fov change inside the path
    with rt.Renderer(0, mode=mode) as r:
        r.upload(sc)
        frames = r.render_path(cams, W, H, D).cpu().numpy()
        r.upload(sc)
        for k, cam in enumerate(cams):
            r.set_camera(cam[0:3], cam[3:6], cam[6])
            own, _ = r.render(W, H, D)
            assert np.array_equal(frames[k], own), k
            if k % 3 == 0:
                assert np.array_equal(frames[k], fresh_debug(rt, sc, cam, mode)[0]), k
        odd = r.render_path(cams[:3], 99, 41, 3).cpu().numpy()    # frames that do not start 16-byte aligned
        for k, cam in enumerate(cams[:3]):
            assert np.array_equal(odd[k], fresh_debug(rt, sc, cam, mode, size=(99, 41, 3))[0]), k


@gpu
def test_set_camera_on_another_stream_than_a_pending_render(rt, scenes):
    import torch
    sc = scenes["complex"]
    dev = torch.device("cuda", 0)
    a, b = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    cams = orbit(sc.camera, 6, turn=1.0)
    with rt.Renderer(0, mode="fast") as r:
        r.upload(sc)
        out = torch.empty((len(cams), H, W, 3), dtype=torch.uint8, device=dev)
        for k, cam in enumerate(cams):
            render_s, cam_s = (a, b) if k % 2 == 0 else (b, a)
            r.set_camera(cam[0:3], cam[3:6], cam[6], cam_s.cuda_stream)
            r.render_bands_device(W, H, D, H, 0, 1, out[k].data_ptr(), render_s.cuda_stream)
        torch.cuda.synchronize()
        for k, cam in enumerate(cams):
            assert np.array_equal(out[k].cpu().numpy(), fresh_debug(rt, sc, cam)[0]), k


@gpu
def test_two_contexts_follow_different_paths_on_one_device(rt, scenes):
    """The constant bank changes hands between two contexts every frame."""
    import torch
    dev = torch.device("cuda", 0)
    s1, s2 = scenes["complex"], scenes["medium"]
    p1, p2 = orbit(s1.camera, 6), orbit(s2.camera, 6, turn=-2.0, lift=1.0)
    with rt.Renderer(0, mode="fast") as r1, rt.Renderer(0, mode="bvh") as r2:
        r1.upload(s1)
        r2.upload(s2)
        o1 = torch.empty((6, H, W, 3), dtype=torch.uint8, device=dev)
        o2 = torch.empty_like(o1)
        for k in range(6):
            r1.set_camera(p1[k, 0:3], p1[k, 3:6], p1[k, 6])
            r1.render_bands_device(W, H, D, H, 0, 1, o1[k].data_ptr())
            r2.set_camera(p2[k, 0:3], p2[k, 3:6], p2[k, 6])
            r2.render_bands_device(W, H, D, H, 0, 1, o2[k].data_ptr())
        torch.cuda.synchronize()
        for k in range(6):
            assert np.array_equal(o1[k].cpu().numpy(), fresh_debug(rt, s1, p1[k])[0]), k
            assert np.array_equal(o2[k].cpu().numpy(), fresh_debug(rt, s2, p2[k], "bvh")[0]), k


@gpu
def test_set_camera_does_not_wait_for_a_long_render(rt):
    import torch
    dev = torch.device("cuda", 0)
    sc = synth(rt, 10000)
    BW, BH = 3840, 2160
    a, b = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    cam = orbit(sc.camera, 8)[1]
    with rt.Renderer(0, mode="fast") as r:
        r.upload(sc)
        big = torch.empty((BH, BW, 3), dtype=torch.uint8, device=dev)
        r.render_bands_device(BW, BH, 5, BH, 0, 1, big.data_ptr(), a.cuda_stream)
        done = torch.cuda.Event()
        done.record(a)
        r.set_camera(cam[0:3], cam[3:6], cam[6], b.cuda_stream)
        still_running = not done.query()
        small = torch.empty((H, W, 3), dtype=torch.uint8, device=dev)
        r.render_bands_device(W, H, D, H, 0, 1, small.data_ptr(), b.cuda_stream)
        torch.cuda.synchronize()
        assert still_running, "rt_set_camera waited for the render in flight"
        assert np.array_equal(small.cpu().numpy(), fresh_debug(rt, sc, cam)[0])


# ---- 6. the drop-in binary ---------------------------------------------------------------------------------------------
BIN = os.path.join(ROOT, "cs420-ray-tracer_b200", "ray_cuda")


@gpu
def test_ray_cuda_camera_path(rt, scenes, tmp_path):
    sc = scenes["complex"]
    cams = orbit(sc.camera, 5, turn=1.0, lift=1.0)
    path = tmp_path / "path.txt"
    path.write_text("# orbit\n\n" + "".join("camera " + " ".join("%.17g" % v for v in c) + "\n" for c in cams))
    p = subprocess.run([BIN, os.path.join(GOLDEN, "scenes", "complex.txt"), "--width", str(W), "--height", str(H), "--depth",
                        str(D), "--camera-path", str(path), "--output", str(tmp_path / "orbit.ppm")],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert p.returncode == 0, p.stdout
    with rt.Renderer(0) as r:
        r.upload(sc)
        frames = r.render_path(cams, W, H, D).cpu().numpy()
    for k in range(len(cams)):
        w, h, _, img = rt.read_ppm(str(tmp_path / ("orbit_%04d.ppm" % k)))
        assert (w, h) == (W, H)
        assert np.array_equal(img[::-1], frames[k]), k          # (the file is top row first)
    assert not (tmp_path / "orbit.ppm").exists()


# ---- 7. without a GPU --------------------------------------------------------------------------------------------------
def test_set_camera_argument_errors(rt):
    lib = rt.load_library()
    v = (np.zeros(3), np.array([0.0, 0.0, -1.0]))
    assert lib.rt_set_camera(None, v[0].ctypes.data, v[1].ctypes.data, 60.0, None) == -1     # RT_ERR_ARG
    assert lib.rt_multi_set_camera(None, v[0].ctypes.data, v[1].ctypes.data, 60.0) == -1


@pytest.mark.parametrize("line", ["camera 0 0 5 0 0 -1", "camera 0 0 5 0 0 -1 60 7", "camrea 0 0 5 0 0 -1 60",
                                  "camera 0 0 five 0 0 -1 60"])
def test_ray_cuda_rejects_a_malformed_camera_path(rt, tmp_path, line):
    if not os.path.exists(BIN):
        rt.build_library()
    path = tmp_path / "path.txt"
    path.write_text("# ok\ncamera 0 2 5 0 0 -20 60\n" + line + "\n")
    p = subprocess.run([BIN, os.path.join(GOLDEN, "scenes", "simple.txt"), "--camera-path", str(path)],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60, cwd=tmp_path)
    assert p.returncode == 1, p.stdout
    assert "path.txt:3" in p.stdout
