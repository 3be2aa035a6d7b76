"""ctypes mirror of include/rt_b200.h.

Mirrors the reference's own surface for this path: ``load_scene`` (include/scene_loader.h:27),
``Scene`` (include/scene.h:27-38: spheres, lights, ambient_light, camera), a ``Renderer`` that
plays the role of the pixel loop + ``trace_ray`` (src/main.cpp:16-58,146-157) and ``write_ppm``
(src/main.cpp:69-91).  Everything is computed by librt_b200.so on a B200; nothing here renders.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
RT_MAX_LEVELS = 32

# every symbol include/rt_b200.h declares (tests check the .so exports each one)
ABI_SYMBOLS = [
    "rt_abi_version", "rt_last_error", "rt_device_count",
    "rt_scene_load", "rt_scene_counts", "rt_scene_data", "rt_scene_free",
    "rt_create", "rt_destroy", "rt_set_option", "rt_upload_scene", "rt_render_tile", "rt_render_bands_frame",
    "rt_dev_alloc", "rt_dev_free", "rt_ipc_export", "rt_ipc_open", "rt_ipc_close", "rt_peer_signal", "rt_peer_wait",
    "rt_render", "rt_render_debug", "rt_render_bands", "rt_band_rows", "rt_band_row_list",
    "rt_host_alloc", "rt_host_free", "rt_write_ppm", "rt_measure_fp32_peak",
    "rt_create_multi", "rt_multi_destroy", "rt_multi_ranks", "rt_multi_ctx", "rt_multi_set_option", "rt_multi_upload_scene",
    "rt_multi_render", "rt_render_bands_host", "rt_host_register", "rt_host_unregister",
    "rt_set_camera", "rt_multi_set_camera", "rt_multi_render_path",
]


class RtError(RuntimeError):
    pass


class RtStats(C.Structure):
    _fields_ = [
        ("ms_device", C.c_double), ("ms_host", C.c_double), ("ms_level0", C.c_double), ("ms_closest0", C.c_double), ("ms_shadow0", C.c_double),
        ("closest_queries", C.c_uint64), ("hits", C.c_uint64),
        ("shadow_queries", C.c_uint64), ("occluded", C.c_uint64),
        ("alive", C.c_uint64 * RT_MAX_LEVELS),
        ("fp64_intersections", C.c_uint64), ("sphere_tests", C.c_uint64),
        ("filter_violations", C.c_uint64),
        ("kernel_launches", C.c_int32), ("rows_rendered", C.c_int32),
        ("bundle_walks", C.c_uint64), ("bundle_candidates", C.c_uint64), ("bundle_fallbacks", C.c_uint64),
    ]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if k != "alive"}
        d["alive"] = [int(x) for x in self.alive]
        d["rays"] = int(self.closest_queries + self.shadow_queries)
        return d


_lib = None


def library_path():
    # RTB200_LIB: A/B testing of alternative builds of the same library (never a different backend)
    return os.environ.get("RTB200_LIB") or os.path.join(HERE, "librt_b200.so")


def load_library():
    """Loads librt_b200.so from the package directory.  Fails loudly if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise RtError("%s not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(there is no CPU fallback)" % path)
    lib = C.CDLL(path)
    vp, i, dp = C.c_void_p, C.c_int, C.POINTER(C.c_double)
    lib.rt_abi_version.restype = i
    lib.rt_last_error.restype = C.c_char_p
    lib.rt_device_count.restype = i
    lib.rt_scene_load.argtypes = [C.c_char_p, i, C.POINTER(vp)]
    lib.rt_scene_counts.argtypes = [vp, C.POINTER(i), C.POINTER(i), C.POINTER(i)]
    lib.rt_scene_data.argtypes = [vp, C.POINTER(dp), C.POINTER(dp), C.POINTER(dp), C.POINTER(dp)]
    lib.rt_scene_free.argtypes = [vp]
    lib.rt_scene_free.restype = None
    lib.rt_create.argtypes = [i, C.POINTER(vp)]
    lib.rt_destroy.argtypes = [vp]
    lib.rt_destroy.restype = None
    lib.rt_set_option.argtypes = [vp, C.c_char_p, C.c_longlong]
    lib.rt_render_tile.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    lib.rt_render_bands_frame.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, C.POINTER(RtStats)]
    lib.rt_dev_alloc.argtypes = [vp, C.c_size_t, C.POINTER(vp)]
    lib.rt_dev_free.argtypes = [vp, vp]
    lib.rt_ipc_export.argtypes = [vp, vp, C.c_char_p]
    lib.rt_ipc_open.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
    lib.rt_ipc_close.argtypes = [vp, vp]
    lib.rt_peer_signal.argtypes = [vp, vp, C.c_uint32, vp]
    lib.rt_peer_wait.argtypes = [vp, vp, C.c_int, C.c_uint32, vp, vp]
    lib.rt_upload_scene.argtypes = [vp, vp, i, vp, i, vp, vp, vp, C.c_double]
    lib.rt_set_camera.argtypes = [vp, vp, vp, C.c_double, vp]
    lib.rt_multi_set_camera.argtypes = [vp, vp, vp, C.c_double]
    lib.rt_render.argtypes = [vp, i, i, i, vp, C.POINTER(RtStats)]
    lib.rt_render_debug.argtypes = [vp, i, i, i, vp, vp, vp, C.POINTER(RtStats)]
    lib.rt_render_bands.argtypes = [vp, i, i, i, i, i, i, vp, vp, C.POINTER(RtStats)]
    lib.rt_band_rows.argtypes = [i, i, i, i]
    lib.rt_band_row_list.argtypes = [i, i, i, i, vp]
    lib.rt_host_alloc.argtypes = [C.c_size_t, C.POINTER(vp)]
    lib.rt_host_free.argtypes = [vp]
    lib.rt_host_free.restype = None
    lib.rt_write_ppm.argtypes = [C.c_char_p, vp, i, i]
    lib.rt_measure_fp32_peak.argtypes = [i, dp, dp]
    lib.rt_create_multi.argtypes = [i, C.POINTER(vp)]
    lib.rt_multi_destroy.argtypes = [vp]
    lib.rt_multi_destroy.restype = None
    lib.rt_multi_ranks.argtypes = [vp]
    lib.rt_multi_ctx.argtypes = [vp, i]
    lib.rt_multi_ctx.restype = vp
    lib.rt_multi_set_option.argtypes = [vp, C.c_char_p, C.c_longlong]
    lib.rt_multi_upload_scene.argtypes = [vp, vp, i, vp, i, vp, vp, vp, C.c_double]
    lib.rt_multi_render.argtypes = [vp, i, i, i, i, vp, C.POINTER(RtStats)]
    lib.rt_multi_render_path.argtypes = [vp, vp, i, i, i, i, vp, vp]
    lib.rt_render_bands_host.argtypes = [vp, i, i, i, i, i, i, vp, C.POINTER(RtStats)]
    lib.rt_host_register.argtypes = [vp, C.c_size_t]
    lib.rt_host_unregister.argtypes = [vp]
    for name in ABI_SYMBOLS:
        getattr(lib, name)
    _lib = lib
    return lib


def _check(rc, what):
    if rc < 0:
        raise RtError("%s failed (%d): %s" % (what, rc, load_library().rt_last_error().decode()))
    return rc


def _vec3(v):
    return np.ascontiguousarray(v, dtype=np.float64).reshape(3)


class Scene:
    """include/scene.h:27-38 as flat float64 arrays in scene-file column order."""

    def __init__(self, spheres, lights, ambient, camera, has_camera=True):
        self.spheres = np.ascontiguousarray(spheres, dtype=np.float64).reshape(-1, 10)
        self.lights = np.ascontiguousarray(lights, dtype=np.float64).reshape(-1, 7)
        self.ambient = np.ascontiguousarray(ambient, dtype=np.float64).reshape(3)
        self.camera = np.ascontiguousarray(camera, dtype=np.float64).reshape(7)
        self.has_camera = bool(has_camera)

    @property
    def nspheres(self):
        return self.spheres.shape[0]

    @property
    def nlights(self):
        return self.lights.shape[0]

    def to_text(self, fmt="%.17g"):
        """Serialises in the loader's grammar (include/scene_loader.h:15-21)."""
        out = []
        for s in self.spheres:
            out.append("sphere " + " ".join(fmt % v for v in s))
        for li in self.lights:
            out.append("light " + " ".join(fmt % v for v in li))
        out.append("ambient " + " ".join(fmt % v for v in self.ambient))
        out.append("camera " + " ".join(fmt % v for v in self.camera))
        return "\n".join(out) + "\n"


def load_scene(path, verbose=False):
    """include/scene_loader.h:27-135 through the library's parser (rt_scene_load)."""
    lib = load_library()
    h = C.c_void_p()
    _check(lib.rt_scene_load(os.fsencode(path), int(verbose), C.byref(h)), "rt_scene_load")
    try:
        n, l, hc = C.c_int(), C.c_int(), C.c_int()
        _check(lib.rt_scene_counts(h, C.byref(n), C.byref(l), C.byref(hc)), "rt_scene_counts")
        ps, pl, pa, pc = (C.POINTER(C.c_double)() for _ in range(4))
        _check(lib.rt_scene_data(h, C.byref(ps), C.byref(pl), C.byref(pa), C.byref(pc)), "rt_scene_data")
        sph = np.ctypeslib.as_array(ps, shape=(n.value * 10,)).copy() if n.value else np.zeros(0)
        lig = np.ctypeslib.as_array(pl, shape=(l.value * 7,)).copy() if l.value else np.zeros(0)
        amb = np.ctypeslib.as_array(pa, shape=(3,)).copy()
        cam = np.ctypeslib.as_array(pc, shape=(7,)).copy()
    finally:
        lib.rt_scene_free(h)
    return Scene(sph, lig, amb, cam, bool(hc.value))


def write_ppm(path, rgb_bottom_first):
    a = np.ascontiguousarray(rgb_bottom_first, dtype=np.uint8)
    H, W, _ = a.shape
    _check(load_library().rt_write_ppm(os.fsencode(path), a.ctypes.data, W, H), "rt_write_ppm")


def measure_fp32_peak(device=0):
    """(FLOP/s, SM MHz) of the FFMA issue peak, measured live by the library."""
    f, m = C.c_double(), C.c_double()
    _check(load_library().rt_measure_fp32_peak(int(device), C.byref(f), C.byref(m)), "rt_measure_fp32_peak")
    return f.value, m.value


def host_register(ptr, nbytes):
    _check(load_library().rt_host_register(C.c_void_p(ptr), nbytes), "rt_host_register")


def host_unregister(ptr):
    _check(load_library().rt_host_unregister(C.c_void_p(ptr)), "rt_host_unregister")


def _path_args(cameras, W, H, device, out):
    """(cameras as K x 7 float64, the uint8 [K, H, W, 3] output on cuda:device, torch's current stream there) of a
    camera-path render."""
    import torch
    cams = np.ascontiguousarray(cameras, dtype=np.float64).reshape(-1, 7)
    dev = torch.device("cuda", device)
    K = cams.shape[0]
    if out is None:
        out = torch.empty((K, H, W, 3), dtype=torch.uint8, device=dev)
    if tuple(out.shape) != (K, H, W, 3) or out.dtype != torch.uint8 or out.device != dev or not out.is_contiguous():
        raise RtError("render_path: out must be a contiguous uint8 [%d, %d, %d, 3] tensor on %s" % (K, H, W, dev))
    # (torch's legacy default stream is handle 0, which the library reads as "the ctx stream": pass cudaStreamLegacy)
    stream = torch.cuda.current_stream(dev).cuda_stream or 1
    return cams, out, stream


def band_rows(H, band_h, rank, nranks):
    return _check(load_library().rt_band_rows(H, band_h, rank, nranks), "rt_band_rows")


def band_row_list(H, band_h, rank, nranks):
    n = band_rows(H, band_h, rank, nranks)
    rows = np.zeros(max(n, 1), dtype=np.int32)
    _check(load_library().rt_band_row_list(H, band_h, rank, nranks, rows.ctypes.data), "rt_band_row_list")
    return rows[:n]


class Renderer:
    """One rt_ctx.  ``render`` returns uint8 [H, W, 3] with row 0 = bottom of the image
    (the reference's framebuffer convention, src/main.cpp:153-154)."""

    def __init__(self, device=0, mode="fast", accel=None):
        """mode: "fast" (FP32 filter / FP64 decide), "exact" (FP64 brute force, diagnostic) or "bvh"
        (= fast with the LBVH forced for every scene size); accel overrides: 0 auto, 1 tables, 2 LBVH."""
        self._lib = load_library()
        self._h = C.c_void_p()
        _check(self._lib.rt_create(int(device), C.byref(self._h)), "rt_create")
        self.device = int(device)
        if mode == "bvh":
            mode, accel = "fast", 2
        self.antialias = False
        self.set_mode(mode)
        if accel is not None:
            self.set_option("accel", accel)
        self._pinned = None
        self._pinned_bytes = 0

    def close(self):
        if getattr(self, "_h", None):
            if self._pinned:
                self._lib.rt_host_free(self._pinned)
                self._pinned = None
            self._lib.rt_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_mode(self, mode):
        v = {"fast": 0, "exact": 1}[mode]
        _check(self._lib.rt_set_option(self._h, b"mode", v), "rt_set_option")
        self.mode = mode

    def set_counters(self, on):
        _check(self._lib.rt_set_option(self._h, b"counters", int(bool(on))), "rt_set_option")

    def set_option(self, key, value):
        _check(self._lib.rt_set_option(self._h, key.encode(), int(value)), "rt_set_option")
        if key == "antialias":
            self.antialias = bool(value)

    def render_bands_frame(self, W, H, depth, band_h, rank, nranks, dev_frame_ptr, stream_ptr=None, want_stats=False):
        """rt_render_bands_frame: this rank's rows at their image positions of an assembled frame (local or peer memory)."""
        st = RtStats()
        _check(self._lib.rt_render_bands_frame(self._h, W, H, depth, band_h, rank, nranks, C.c_void_p(dev_frame_ptr),
                                               C.c_void_p(stream_ptr) if stream_ptr else None,
                                               C.byref(st) if want_stats else None), "rt_render_bands_frame")
        return st

    # ---- device memory shared between the processes of one box, completion flags (rt_b200.h) ----
    def dev_alloc(self, nbytes):
        p = C.c_void_p()
        _check(self._lib.rt_dev_alloc(self._h, nbytes, C.byref(p)), "rt_dev_alloc")
        return p.value

    def dev_free(self, ptr):
        _check(self._lib.rt_dev_free(self._h, C.c_void_p(ptr)), "rt_dev_free")

    def ipc_export(self, ptr):
        buf = C.create_string_buffer(64)
        _check(self._lib.rt_ipc_export(self._h, C.c_void_p(ptr), buf), "rt_ipc_export")
        return buf.raw

    def ipc_open(self, handle):
        p = C.c_void_p()
        _check(self._lib.rt_ipc_open(self._h, handle, C.byref(p)), "rt_ipc_open")
        return p.value

    def ipc_close(self, ptr):
        _check(self._lib.rt_ipc_close(self._h, C.c_void_p(ptr)), "rt_ipc_close")

    def peer_signal(self, flag_ptr, value, stream_ptr=None):
        _check(self._lib.rt_peer_signal(self._h, C.c_void_p(flag_ptr), value & 0xffffffff,
                                        C.c_void_p(stream_ptr) if stream_ptr else None), "rt_peer_signal")

    def peer_wait(self, flags_ptr, n, value, err_ptr, stream_ptr=None):
        _check(self._lib.rt_peer_wait(self._h, C.c_void_p(flags_ptr), n, value & 0xffffffff, C.c_void_p(err_ptr),
                                      C.c_void_p(stream_ptr) if stream_ptr else None), "rt_peer_wait")

    def render_tile_device(self, W, H, depth, tile, dev_fb_ptr, stream_ptr=None):
        """rt_render_tile: tile = (x, y, w, h); dev_fb_ptr = device pointer of a W*H*3 float32 framebuffer."""
        x, y, w, h = tile
        _check(self._lib.rt_render_tile(self._h, W, H, depth, x, y, w, h, C.c_void_p(dev_fb_ptr),
                                        C.c_void_p(stream_ptr) if stream_ptr else None), "rt_render_tile")

    def upload(self, scene):
        self.scene = scene
        cam = scene.camera
        pos = np.ascontiguousarray(cam[0:3]); look = np.ascontiguousarray(cam[3:6])
        _check(self._lib.rt_upload_scene(
            self._h, scene.spheres.ctypes.data, scene.nspheres, scene.lights.ctypes.data, scene.nlights,
            scene.ambient.ctypes.data, pos.ctypes.data, look.ctypes.data, float(cam[6])), "rt_upload_scene")

    def set_camera(self, pos, look, fov, stream_ptr=None):
        """rt_set_camera: moves the camera of the uploaded scene; asynchronous on stream_ptr (None = the ctx stream)."""
        p, q = _vec3(pos), _vec3(look)
        _check(self._lib.rt_set_camera(self._h, p.ctypes.data, q.ctypes.data, float(fov),
                                       C.c_void_p(stream_ptr) if stream_ptr else None), "rt_set_camera")

    def render_path(self, cameras, W, H, depth, out=None):
        """One frame per camera row (px py pz lx ly lz fov, the scene file's order) as a torch uint8 [K, H, W, 3] tensor
        on this renderer's device, row 0 = bottom.  Every frame is rt_set_camera + rt_render_bands on torch's current
        stream, with no host synchronisation between frames; the camera of the last row stays set."""
        import torch
        cams, out, stream = _path_args(cameras, W, H, self.device, out)
        dev = out.device
        K = cams.shape[0]
        # the kernels store 16-byte row segments: a frame that does not start 16-byte aligned goes through a staging frame
        stage = None if (H * W * 3) % 16 == 0 else torch.empty((H, W, 3), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            for k in range(K):
                self.set_camera(cams[k, 0:3], cams[k, 3:6], cams[k, 6], stream)
                dst = out[k] if stage is None else stage
                self.render_bands_device(W, H, depth, H, 0, 1, dst.data_ptr(), stream)
                if stage is not None:
                    out[k].copy_(stage)
        return out

    def scene_bytes(self):
        s = self.scene
        return int(s.spheres.nbytes + s.lights.nbytes + s.ambient.nbytes + s.camera.nbytes)

    def pinned_frame(self, W, H):
        """A page-locked uint8 [H, W, 3] buffer owned by this renderer (rt_host_alloc)."""
        need = W * H * 3
        if self._pinned is None or self._pinned_bytes < need:
            if self._pinned:
                self._lib.rt_host_free(self._pinned)
            p = C.c_void_p()
            _check(self._lib.rt_host_alloc(need, C.byref(p)), "rt_host_alloc")
            self._pinned, self._pinned_bytes = p, need
        buf = (C.c_uint8 * need).from_address(self._pinned.value)
        return np.frombuffer(buf, dtype=np.uint8).reshape(H, W, 3)

    def render(self, W, H, depth, out=None, want_stats=True):
        if out is None:
            out = np.empty((H, W, 3), dtype=np.uint8)
        st = RtStats()
        _check(self._lib.rt_render(self._h, W, H, depth, out.ctypes.data, C.byref(st) if want_stats else None), "rt_render")
        return out, st

    def render_debug(self, W, H, depth, want_stats=True):
        out = np.empty((H, W, 3), dtype=np.uint8)
        m = 2 if self.antialias else 1          # supersampling: debug buffers are per sample, [2H][2W][depth]
        hit = np.empty((H * m, W * m, max(depth, 1)), dtype=np.int32)
        mask = np.empty((H * m, W * m, max(depth, 1)), dtype=np.uint32)
        st = RtStats()
        _check(self._lib.rt_render_debug(self._h, W, H, depth, out.ctypes.data, hit.ctypes.data, mask.ctypes.data,
                                         C.byref(st) if want_stats else None), "rt_render_debug")
        return out, hit, mask, st

    def render_bands_host(self, W, H, depth, band_h, rank, nranks, host_ptr, want_stats=False):
        """rt_render_bands_host: this rank's bands rendered and copied to their image positions of a (shared, pinned)
        host frame over this GPU's own host link; returns when they have landed."""
        st = RtStats()
        _check(self._lib.rt_render_bands_host(self._h, W, H, depth, band_h, rank, nranks, C.c_void_p(host_ptr),
                                              C.byref(st) if want_stats else None), "rt_render_bands_host")
        return st

    def render_bands_device(self, W, H, depth, band_h, rank, nranks, dev_ptr, stream_ptr=None, want_stats=False):
        """Asynchronous banded render into device memory (e.g. a torch tensor's data_ptr())."""
        st = RtStats()
        _check(self._lib.rt_render_bands(self._h, W, H, depth, band_h, rank, nranks, C.c_void_p(dev_ptr),
                                         C.c_void_p(stream_ptr) if stream_ptr else None,
                                         C.byref(st) if want_stats else None), "rt_render_bands")
        return st


class MultiRenderer:
    """rt_create_multi: one frame sharded by interleaved row bands over `ngpus` ranks inside this process; every rank
    copies its bands to the host frame over its own link.  render_path instead gives whole frames of a camera path to
    the ranks."""

    def __init__(self, ngpus, mode="fast", accel=None):
        self._lib = load_library()
        self._h = C.c_void_p()
        _check(self._lib.rt_create_multi(int(ngpus), C.byref(self._h)), "rt_create_multi")
        self.n = int(ngpus)
        if mode == "bvh":
            mode, accel = "fast", 2
        self.set_option("mode", {"fast": 0, "exact": 1}[mode])
        if accel is not None:
            self.set_option("accel", accel)

    def set_option(self, key, value):
        _check(self._lib.rt_multi_set_option(self._h, key.encode(), int(value)), "rt_multi_set_option")

    def upload(self, scene):
        self.scene = scene
        cam = scene.camera
        pos = np.ascontiguousarray(cam[0:3]); look = np.ascontiguousarray(cam[3:6])
        _check(self._lib.rt_multi_upload_scene(
            self._h, scene.spheres.ctypes.data, scene.nspheres, scene.lights.ctypes.data, scene.nlights,
            scene.ambient.ctypes.data, pos.ctypes.data, look.ctypes.data, float(cam[6])), "rt_multi_upload_scene")

    def set_camera(self, pos, look, fov):
        """rt_multi_set_camera: rt_set_camera on every rank."""
        p, q = _vec3(pos), _vec3(look)
        _check(self._lib.rt_multi_set_camera(self._h, p.ctypes.data, q.ctypes.data, float(fov)), "rt_multi_set_camera")

    def render(self, W, H, depth, band_h=16, out=None, want_stats=True):
        if out is None:
            out = np.empty((H, W, 3), dtype=np.uint8)
        st = RtStats()
        _check(self._lib.rt_multi_render(self._h, W, H, depth, band_h, out.ctypes.data, C.byref(st) if want_stats else None),
               "rt_multi_render")
        return out, st

    def render_path(self, cameras, W, H, depth, out=None):
        """rt_multi_render_path: one frame per camera row (px py pz lx ly lz fov), rank k % n renders frame k, as a torch
        uint8 [K, H, W, 3] tensor on rank 0's device (cuda:0), row 0 = bottom, ordered on torch's current stream there
        (no host synchronisation).  The frames equal Renderer.render_path's; every rank keeps the last camera set."""
        cams, out, stream = _path_args(cameras, W, H, 0, out)
        _check(self._lib.rt_multi_render_path(self._h, cams.ctypes.data, cams.shape[0], W, H, depth, C.c_void_p(out.data_ptr()),
                                              C.c_void_p(stream)), "rt_multi_render_path")
        return out

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rt_multi_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
