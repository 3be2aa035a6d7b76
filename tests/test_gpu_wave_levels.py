"""Reflection levels >= 1 of table scenes (fewer than 1024 spheres) run as WAVEFRONT kernels -- k_closest1 (bundle-culled
when the general table is in shared memory), the level-k k_shadow and k_shade -- instead of the tail kernel k_bounce.
Automatically that happens only for large frames (>= 750 k pixels, or >= 60 000 rays entering a level), so the small
adversarial scenes of test_gpu_parity.py never reach these kernels.  Here every level count is forced with
rt_set_option wave_levels (1, 2, 3 and 32 = every level a wavefront), and each test asserts from the launch count and the
ray counters that it ran the kernels it is about.

The culled k_closest1 walk promises more than correct pixels: a pair is dropped only when the general filter rejects both
its spheres for every ray of the 64-ray bundle, so the culled and the full walk make the same FP64 evaluations.  The A/B
tests below compare the library with a build of the same sources with -DRT_NO_GEN_CULL (k_closest1 walks the full table):
same frames, hit maps, shadow masks and every counter but the bundle counters.  Needs a B200: run with -m gpu."""
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest

TESTS = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(TESTS)
for _p in (TESTS, ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "scripts")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from test_gpu_parity import _random_scene, _scene, check  # noqa: E402

pytestmark = pytest.mark.gpu

ALL = 32                       # wave_levels = RT_MAX_LEVELS: every level a wavefront, the tail never runs
WAVE = [1, 2, 3, ALL]
BUNDLE = ("bundle_walks", "bundle_candidates")


def launches(D, wl, L):
    """Kernels of one table-scene render (rtk_launch_fast): per wavefront level closest + shadow (at level 0 also without
    lights: it turns the per-tile ray counts into the level-1 queue offsets) + shade, then one tail launch if levels remain."""
    n = sum(3 if (L > 0 or k == 0) else 2 for k in range(min(D, wl)))
    return n + (1 if D > wl else 0)


def renderer(rt, wl, **kw):
    """A fresh context per forced level count (rt_set_option accepts 1..32 only: a context cannot go back to automatic)."""
    r = rt.Renderer(0, mode="fast", **kw)
    r.set_option("wave_levels", wl)
    return r


def transformed(rt, sc, k=1.0, off=(0.0, 0.0, 0.0)):
    """A similarity transform of a scene: x -> k x + off (radii scaled by k), as scripts/fuzz_parity.py does."""
    off = np.asarray(off, dtype=np.float64)
    sp = sc.spheres.copy(); sp[:, :3] = sp[:, :3] * k + off; sp[:, 3] *= k
    li = sc.lights.copy(); li[:, :3] = li[:, :3] * k + off
    cm = sc.camera.copy(); cm[:3] = cm[:3] * k + off; cm[3:6] = cm[3:6] * k + off
    return rt.Scene(sp, li, sc.ambient, cm)


def many_lights(rt, base, nl):
    g = np.random.default_rng(nl)
    lights = np.column_stack([g.uniform(-15, 15, nl), g.uniform(2, 14, nl), g.uniform(-25, 8, nl), g.uniform(0.05, 0.2, (nl, 3)),
                              np.ones(nl)])
    return rt.Scene(base.spheres, lights, base.ambient, base.camera)


# ---------------------------------------------------------------------------------------------
# scenes built around chosen reflected rays

def _unit(v):
    return v / np.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])


def _camera_ray(cam, W, H, i, j):
    """oracle/rt_oracle.c camera_get_ray for pixel (i, j), j = 0 the bottom row, in the oracle's FP64 operation order."""
    pos, look, fov = cam[:3], cam[3:6], cam[6]
    fwd = _unit(look - pos)
    right = _unit(np.cross(fwd, np.array([0.0, 1.0, 0.0])))
    up = _unit(np.cross(right, fwd))
    s = np.tan(fov * 0.5 * np.pi / 180.0)
    return pos, _unit(fwd + right * ((i / (W - 1) - 0.5) * s) + up * ((j / (H - 1) - 0.5) * s))


def _reflect(o, d, c, r):
    """The reflected ray of (o, d) at sphere (c, r) as the oracle's trace_ray forms it (None if the ray misses)."""
    oc = o - c
    a, b, cc = d @ d, 2.0 * (oc @ d), oc @ oc - r * r
    disc = b * b - 4 * a * cc
    if disc < 0:
        return None
    t = (-b - np.sqrt(disc)) / (2 * a)
    p = o + d * t
    n = _unit(p - c)
    return p + n * 1e-3, _unit(d - n * 2.0 * (d @ n))


GRAZE_EPS = (-1e-3, -1e-6, 0.0, 1e-7, 1e-6, 1e-4, 1e-2)
GRAZE_W, GRAZE_H = 160, 100


def grazing_scene(rt, k=1.0, off=(0.0, 0.0, 0.0)):
    """Small spheres that the reflected rays of chosen pixels graze.  One big mirror (M1) in front of the camera; for each
    chosen pixel its reflected ray (o, d) is formed in FP64 and a small sphere (r from 1e-3 to 0.5) is put at distance t
    along it, offset perpendicular to d by r (1 + eps): with eps < 0 the ray cuts the sphere's rim, with eps > 0 it misses
    it by a hair (eps = 1e-7 is below FP32 resolution) -- and the rays of its bundle neighbours pass it on both sides.
    Distances up to 1000 r bring the far-field terms of the cull (dtmax, 2e-5 (dist + R2)) into play.  A second mirror
    encloses the scene, so the grazing rays and the rays the small (reflective) spheres send on reach level 2 and beyond.
    Built directly in the transformed frame x -> k x + off, so that the rays graze at every scale."""
    off = np.asarray(off, dtype=np.float64)
    cam = np.array([0.0, 0.0, 5.0, 0.0, 0.0, -1.0, 60.0])
    cam[:3] = cam[:3] * k + off; cam[3:6] = cam[3:6] * k + off
    m1c, m1r = np.array([0.0, 0.0, -4.0]) * k + off, 2.5 * k
    spheres = [list(m1c) + [m1r, 0.8, 0.8, 0.9, 0.9, 0.1, 60],
               list(off) + [4000.0 * k, 0.3, 0.3, 0.3, 0.5, 0.5, 10]]        # the enclosing mirror (camera inside it)
    combos = [(r, t, e) for r in (1e-3, 1e-2, 0.1, 0.5) for t in (2.0 * k, 1000.0 * r * k) for e in GRAZE_EPS]
    # pixels on M1's image, spread over it (columns 40..119, rows 20..79 of the 160 x 100 frame)
    pix = [(44 + 9 * (q % 9), 22 + 7 * (q // 9)) for q in range(len(combos))]
    for q, ((r, t, e), (i, j)) in enumerate(zip(combos, pix)):
        o, d = _camera_ray(cam, GRAZE_W, GRAZE_H, i, j)
        ro, rd = _reflect(o, d, m1c, m1r)
        axis = np.array([0.0, 1.0, 0.0]) if q % 2 else np.array([1.0, 0.0, 0.0])
        perp = _unit(np.cross(rd, axis)) * (1.0 if q % 3 else -1.0)
        c = ro + rd * t + perp * (r * k * (1.0 + e))
        spheres.append(list(c) + [r * k, 0.9, 0.4 + 0.5 * (q % 2), 0.2, 0.6 if q % 4 else 0.0, 0.4, 5 + q])
    lights = [list(np.array([5.0, 8.0, 2.0]) * k + off) + [1, 1, 1, 1], list(np.array([-6.0, 3.0, 1.0]) * k + off) + [0.6, 0.5, 0.4, 1]]
    return rt.Scene(np.array(spheres), np.array(lights), (0.1, 0.1, 0.1), cam)


GRAZE_FRAMES = {"unit": (1.0, (0, 0, 0)), "small": (1e-2, (0, 0, 0)), "large": (1e3, (0, 0, 0)), "offset": (1.0, (1e4, -1e4, 1e4))}


def cluster_scene(rt, n=800, lights=False):
    """Multi-batch culled walks: a mirror floor (a sphere of radius 1000) reflects the camera's view into a cluster of
    n - 1 big, overlapping spheres.  The reflected rays of a bundle are coherent (a nearly flat mirror), and the line of
    every one of them crosses most of the cluster, so hundreds of pairs survive the cull of each level-1 walk: it is
    flushed in several kGenIds batches, an odd batch padded with a culled pair."""
    g = np.random.default_rng(n)
    m = n - 1
    c = np.column_stack([g.uniform(-4, 4, m), g.uniform(7, 13, m), g.uniform(-24, -16, m)])
    r = g.uniform(3.0, 5.0, m)
    col = g.uniform(0.1, 1.0, (m, 3))
    refl = np.where(g.random(m) < 0.5, 0.0, g.uniform(0.1, 0.9, m))
    sph = np.column_stack([c, r, col, refl, 1 - refl, g.integers(5, 121, m).astype(np.float64)])
    sph = np.vstack([sph, [0, -1000.5, -20, 1000, 0.7, 0.7, 0.75, 0.9, 0.1, 50]])
    sph = np.array([[float("%.6f" % v) for v in row] for row in sph.tolist()])
    li = np.array([[0, 20, 5, 1, 1, 1, 1], [-12, 6, -8, 0.5, 0.6, 0.7, 1]]) if lights else np.zeros((0, 7))
    return rt.Scene(sph, li, (0.1, 0.1, 0.12), np.array([0.0, 2.0, 10.0, 0.0, 1.0, -20.0, 70.0]))


def mirror_hall(rt):
    """Mirror-heavy scene: a mirror floor and a ring of mirror spheres; most pixels reflect at level 0."""
    sph = [(0, -1001, -10, 1000, 0.8, 0.8, 0.8, 0.85, 0.15, 40)]
    for q in range(10):
        a = 2 * np.pi * q / 10
        sph.append((4.5 * np.cos(a), 0.6 + 0.4 * (q % 3), -10 + 4.5 * np.sin(a), 1.3 + 0.1 * (q % 4), 0.2 + 0.08 * q, 0.5, 0.9 - 0.07 * q,
                    0.6 + 0.04 * (q % 5), 0.4, 20 + 10 * q))
    sph.append((0, 1.5, -10, 2.2, 1, 1, 1, 0.95, 0.05, 100))
    return _scene(rt, sph, lights=[(5, 8, 2, 1, 1, 1, 1), (-6, 6, -3, 0.6, 0.5, 0.4, 1)], camera=(0, 2.5, 2, 0, -0.5, -10, 60))


# ---------------------------------------------------------------------------------------------
# a. the adversarial catalogue at every split between wavefront levels and tail, against the oracle

def _catalogue():
    import gen_scene
    from conftest import scene_path
    cases = {}
    for seed in range(24):                                     # test_fuzz_random_scenes
        cases["fuzz%d" % seed] = (lambda rt, s=seed: _random_scene(rt, s), [(96, 54, 4), (61, 47, 6), (130, 40, 3)][seed % 3], None)
    s = (0.3, 0.2, -4, 1.25, 0.8, 0.3, 0.2, 0.4, 0.5, 30)
    ties = [s, s, (0.3, 0.2, -4, 1.25, 0.1, 0.9, 0.2, 0.0, 1, 5), (2.55, 0.2, -4, 1.0, 0.2, 0.3, 0.9, 0.6, 0.4, 50),
            (0.3, 0.2, -4, 0.5, 1, 1, 1, 0.9, 0.1, 90), (0, -101.05, -4, 100, 0.5, 0.5, 0.5, 0.2, 1, 5)]
    cases["ties"] = (lambda rt: _scene(rt, ties, lights=[(5, 8, 2, 1, 1, 1, 1), (-6, 3, 1, 1, 0.5, 0.5, 1)]), (320, 200, 6), None)
    cases["inside"] = (lambda rt: _scene(rt, [(0, 0, 0, 50, 1, 1, 1, 0.3, 0.5, 20)]), (64, 48, 4), None)
    cases["mirror_shin0"] = (lambda rt: _scene(rt, [(0, 0, -3, 1, 1, 0, 0, 1.0, 0.5, 0), (0, -101, -3, 100, 1, 1, 1, 0.5, 0.5, 4)]),
                             (64, 48, 4), None)
    cases["neg_refl"] = (lambda rt: _scene(rt, [(0, 0, -3, 1, 1, 0, 0, -0.2, 0.5, 8), (1.5, 0, -3, 0.5, 0, 1, 0, 0.7, 0.5, 8)]),
                         (64, 48, 4), None)
    medium = lambda rt: rt.load_scene(scene_path("medium"))
    complex_ = lambda rt: rt.load_scene(scene_path("complex"))
    cases["far_medium"] = (lambda rt: transformed(rt, medium(rt), 1.0, (1000.0, -2000.0, 500.0)), (320, 180, 5), None)
    for tag, k, off in (("s1e-2", 1e-2, (0, 0, 0)), ("s1e3", 1e3, (0, 0, 0)), ("o1e4", 1.0, (1e4, -3e3, 7e3))):
        cases["fuzz5_" + tag] = (lambda rt, k=k, off=off: transformed(rt, _random_scene(rt, 5), k, off), (96, 54, 4), None)
        cases["complex_" + tag] = (lambda rt, k=k, off=off: transformed(rt, complex_(rt), k, off), (160, 90, 5), None)
    for nl in (32, 33, 40):
        cases["lights%d" % nl] = (lambda rt, nl=nl: many_lights(rt, medium(rt), nl), (96, 54, 3), None)
    cases["dark_complex"] = (lambda rt: rt.Scene(complex_(rt).spheres, np.zeros((0, 7)), (0.1, 0.1, 0.1), complex_(rt).camera),
                             (160, 90, 5), None)
    # 1000 spheres: the light tables exceed the shared-memory budget, the level-k shadow kernel streams them (kTabStream)
    cases["gen300"] = (lambda rt: rt.Scene(*gen_scene.generate(300, 7, 0.3, 1.5)), (320, 180, 5), 1)
    cases["gen1000"] = (lambda rt: rt.Scene(*gen_scene.generate(1000, 420, 0.3, 1.5)), (240, 136, 5), 1)
    return cases


CATALOGUE = _catalogue()
_gold = {}


def oracle_gold(oracle, key, scene, W, H, D):
    if key not in _gold:
        o = oracle.render(scene, W, H, D, want_idx=True)
        _gold[key] = {"hit_idx": o["hit_idx"], "shadow_mask": o["shadow_mask"], "rgb": o["rgb"], "counters": o["counters"]}
    return _gold[key]


def check_wave(rt, oracle, r, scene, key, W, H, D, wl):
    """check() of test_gpu_parity (hit indices, shadow masks, counters, RGB gate, no filter violation) plus the ray count of
    every level, and the launch count that proves which split of wavefront levels and tail ran."""
    gold = oracle_gold(oracle, key, scene, W, H, D)
    rgb, st = check(rt, oracle, r, scene, W, H, D, gold)
    assert [int(x) for x in st.alive[:D]] == gold["counters"]["alive"][:D]
    assert st.kernel_launches == launches(D, wl, scene.nlights), (st.kernel_launches, D, wl)
    return rgb, st


@pytest.fixture(scope="module")
def wave_renderers(rt):
    rs = {}
    yield lambda wl, accel=None: rs.setdefault((wl, accel), renderer(rt, wl, **({} if accel is None else {"accel": accel})))
    for r in rs.values():
        r.close()


@pytest.mark.parametrize("wl", WAVE)
@pytest.mark.parametrize("name", list(CATALOGUE))
def test_catalogue_at_every_wavefront_split(rt, oracle, wave_renderers, name, wl):
    build, (W, H, D), accel = CATALOGUE[name]
    sc = build(rt)
    assert sc.nspheres < 1024                       # a table scene
    check_wave(rt, oracle, wave_renderers(wl, accel), sc, name, W, H, D, wl)


def test_catalogue_reaches_the_wavefront_levels(rt, oracle):
    """The catalogue is not vacuous at wave_levels >= 2: most of its scenes send rays into level 1, and several into the
    levels beyond it (the oracle's ray counts, which the tests above pin the device's to)."""
    l1 = l2 = 0
    for name, (build, (W, H, D), _) in CATALOGUE.items():
        alive = oracle_gold(oracle, name, build(rt), W, H, D)["counters"]["alive"]
        l1 += alive[1] > 0
        l2 += D > 2 and alive[2] > 0
    assert l1 >= 0.75 * len(CATALOGUE) and l2 >= 0.5 * len(CATALOGUE), (l1, l2, len(CATALOGUE))


# ---------------------------------------------------------------------------------------------
# b. grazing reflected rays: the adversary of the k_closest1 cull and of the general filter

@pytest.mark.parametrize("wl", [1, 2, 3])
@pytest.mark.parametrize("frame", list(GRAZE_FRAMES))
def test_grazing_reflected_rays(rt, oracle, frame, wl):
    sc = grazing_scene(rt, *GRAZE_FRAMES[frame])
    with renderer(rt, wl) as r:
        rgb, st = check_wave(rt, oracle, r, sc, "graze_" + frame, GRAZE_W, GRAZE_H, 3, wl)
    hit = _gold["graze_" + frame]["hit_idx"]
    # the small spheres are hit at level 1 and (through the enclosing mirror) at level 2
    assert len(np.unique(hit[..., 1][hit[..., 1] >= 2])) >= 20 and (hit[..., 2] >= 2).sum() > 0
    assert st.alive[2] > 10000


# ---------------------------------------------------------------------------------------------
# c. two rays per lane in k_closest1; culled walks flushed in several batches

def test_two_rays_per_lane(rt, oracle):
    """k_closest1 takes two rays per lane when a level has >= grid x 8 warps x 64 rays (151 552 on a 148-SM B200 at 2 CTAs
    per SM); only full-size frames get there."""
    sc = mirror_hall(rt)
    W, H, D = 1024, 576, 3
    with renderer(rt, 2) as r:
        rgb, st = check_wave(rt, oracle, r, sc, "hall", W, H, D, 2)
    assert st.alive[1] >= 160_000


def level1_counters(r, W, H):
    """Level-1 counters of a lightless scene at wave_levels 2: depth 2 minus depth 1 (k_closest1's alone)."""
    keys = BUNDLE + ("fp64_intersections", "closest_queries")
    _, s1 = r.render(W, H, 1)
    _, s2 = r.render(W, H, 2)
    return {k: int(getattr(s2, k)) - int(getattr(s1, k)) for k in keys}


def test_culled_walks_in_several_batches(rt, oracle):
    sc = cluster_scene(rt)
    W, H, D = 160, 90, 3
    assert 600 <= sc.nspheres < 1024 and sc.nlights == 0
    with renderer(rt, 2, accel=1) as r:
        check_wave(rt, oracle, r, sc, "cluster", W, H, D, 2)
        l1 = level1_counters(r, W, H)
    # more than 126 spheres (63 pairs) kept per walk on average: some walk overflowed one kGenIds batch
    assert l1["bundle_walks"] > 0 and l1["bundle_candidates"] > 126 * l1["bundle_walks"], l1


# ---------------------------------------------------------------------------------------------
# d. a general table too large for shared memory: k_closest1<false, false>

@pytest.mark.parametrize("wl", [2, 3])
def test_general_table_beyond_shared_memory(rt, wl):
    import gen_scene
    sc = rt.Scene(*gen_scene.generate(6000, 77, 0.3, 1.5))
    assert sc.nspheres > 5760                         # 3000 pairs x 32 bytes > 90 KB: the general table is not staged
    W, H, D = 160, 90, 4
    with rt.Renderer(0, mode="exact") as r:
        r.upload(sc)
        ref = r.render_debug(W, H, D)
    with renderer(rt, wl, accel=1) as r:
        r.upload(sc)
        rgb, hit, mask, st = r.render_debug(W, H, D)
    assert np.array_equal(ref[1], hit) and np.array_equal(ref[2], mask)
    ok, pct, mx = rt.compare_rgb(ref[0], rgb, 0.5)
    assert ok and mx <= 2, (pct, mx)
    assert st.filter_violations == 0
    for k in ("closest_queries", "hits", "shadow_queries", "occluded"):
        assert getattr(st, k) == getattr(ref[3], k), k
    assert [int(x) for x in st.alive] == [int(x) for x in ref[3].alive] and st.alive[1] > 0
    assert st.kernel_launches == launches(D, wl, sc.nlights)


# ---------------------------------------------------------------------------------------------
# e. the other output modes feeding a wavefront level 1

def _output_scenes(rt):
    from conftest import scene_path
    return {"complex": rt.load_scene(scene_path("complex")), "fuzz7": _random_scene(rt, 7)}


@pytest.mark.parametrize("name", ["complex", "fuzz7"])
def test_bands_and_tiles_feed_a_wavefront_level(rt, name):
    import torch
    sc = _output_scenes(rt)[name]
    W, H, D = 200, 120, 5
    with renderer(rt, 2) as r:
        r.upload(sc)
        full, st = r.render(W, H, D)
        assert st.kernel_launches == launches(D, 2, sc.nlights) and st.alive[1] > 0
        out = np.zeros_like(full)
        for rank in range(3):
            rows = rt.band_row_list(H, 8, rank, 3)
            buf = torch.zeros(len(rows) * W * 3 + 16, dtype=torch.uint8, device="cuda:0")
            torch.cuda.synchronize()
            sb = r.render_bands_device(W, H, D, 8, rank, 3, buf.data_ptr(), None, want_stats=True)
            assert sb.rows_rendered == len(rows) and sb.kernel_launches == launches(D, 2, sc.nlights)
            out[rows] = buf[:len(rows) * W * 3].cpu().numpy().reshape(len(rows), W, 3)
        assert np.array_equal(out, full)
        whole = torch.full((H, W, 3), -1.0, dtype=torch.float32, device="cuda:0")
        tiled = torch.full((H, W, 3), -1.0, dtype=torch.float32, device="cuda:0")
        torch.cuda.synchronize()
        r.render_tile_device(W, H, D, (0, 0, W, H), whole.data_ptr())
        for (x, y, w, h) in [(0, 0, 48, 40), (48, 0, 152, 40), (0, 40, 77, 80), (77, 40, 123, 33), (77, 73, 123, 47)]:
            r.render_tile_device(W, H, D, (x, y, w, h), tiled.data_ptr())
        torch.cuda.synchronize()
        assert torch.equal(whole, tiled)
        q = (255.99 * torch.clamp(whole, max=1.0)).to(torch.int32).to(torch.uint8).cpu().numpy()
        assert np.array_equal(q, full)


@pytest.mark.parametrize("name", ["complex", "fuzz7"])
def test_supersampling_feeds_a_wavefront_level(rt, oracle, name):
    sc = _output_scenes(rt)[name]
    W, H, D = 128, 72, 5
    o = oracle.render_supersampled(sc, W, H, D)
    with renderer(rt, 2) as r:
        r.set_option("antialias", 1)
        r.upload(sc)
        rgb, hit, mask, st = r.render_debug(W, H, D)
    assert st.kernel_launches == launches(D, 2, sc.nlights) + 1          # + the 2x2 resolve
    assert st.alive[1] > 0
    for s, (a, b) in enumerate(((0, 0), (1, 0), (0, 1), (1, 1))):
        assert np.array_equal(hit[b::2, a::2], o["samples"][s]["hit_idx"]), s
        assert np.array_equal(mask[b::2, a::2], o["samples"][s]["shadow_mask"]), s
    ok, pct, mx = rt.compare_rgb(o["rgb"], rgb, 0.5)
    assert ok and mx <= 2, (pct, mx)
    assert st.closest_queries == sum(p["counters"]["closest_queries"] for p in o["samples"])
    assert st.filter_violations == 0


# ---------------------------------------------------------------------------------------------
# A/B: the culled k_closest1 walk against a build whose k_closest1 walks the full table (-DRT_NO_GEN_CULL)

AB_SPEC = [(name, wl) for wl in (2, 3) for name in ["graze_" + f for f in GRAZE_FRAMES] +
           ["cluster", "cluster_lit", "complex_640", "complex_1080p", "lights40"]] + [("hall", 2)]


def _ab_case(rt, name, wl):
    """(scene, W, H, D, accel) of one case of the culled-versus-full comparison."""
    from conftest import scene_path
    if name.startswith("graze_"):
        return grazing_scene(rt, *GRAZE_FRAMES[name[6:]]), GRAZE_W, GRAZE_H, 3, None
    if name.startswith("cluster"):
        return cluster_scene(rt, lights=name == "cluster_lit"), 160, 90, 3, 1
    if name.startswith("complex"):
        return (rt.load_scene(scene_path("complex")),) + ((640, 360, 5) if name == "complex_640" else (1920, 1080, 2)) + (None,)
    if name == "lights40":
        return many_lights(rt, rt.load_scene(scene_path("medium")), 40), 320, 180, 3, None
    assert name == "hall"
    return mirror_hall(rt), 1024, 576, 3, None


COUNTERS = ("closest_queries", "hits", "shadow_queries", "occluded", "fp64_intersections", "sphere_tests", "filter_violations",
            "kernel_launches", "rows_rendered", "bundle_fallbacks")


def _ab_render(rt, name, wl):
    sc, W, H, D, accel = _ab_case(rt, name, wl)
    with renderer(rt, wl, **({} if accel is None else {"accel": accel})) as r:
        r.upload(sc)
        rgb, hit, mask, st = r.render_debug(W, H, D)
        frame, st2 = r.render(W, H, D)
        r.upload(rt.Scene(sc.spheres, np.zeros((0, 7)), sc.ambient, sc.camera))
        _, st3 = r.render(W, H, D)                      # the same closest hits and reflected rays, no shadow walks
    out = {"rgb": rgb, "hit": hit, "mask": mask, "frame": frame, "alive": np.array([int(x) for x in st.alive], dtype=np.int64),
           "nlights": np.int64(sc.nlights)}
    for k in COUNTERS + BUNDLE:
        out[k] = np.int64(getattr(st, k))
        out["render_" + k] = np.int64(getattr(st2, k))
        out["dark_" + k] = np.int64(getattr(st3, k))
    return out


def _ab_child(path):
    """Runs in a child process whose RTB200_LIB is the -DRT_NO_GEN_CULL build (the library is a process-wide ctypes
    singleton): renders every A/B case, writes the results to path (.npz)."""
    import rtb200
    res = {}
    for name, wl in AB_SPEC:
        for k, v in _ab_render(rtb200, name, wl).items():
            res["%s-wl%d/%s" % (name, wl, k)] = v
    np.savez(path, **res)


def _nvcc():
    p = shutil.which("nvcc")
    if p is None:
        home = os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda"
        p = os.path.join(home, "bin", "nvcc")
    return p if os.path.exists(p) else None


@pytest.fixture(scope="session")
def full_walk_results():
    """Builds the library with -DRT_NO_GEN_CULL (the Makefile's nvcc flags; objects and library in a temporary
    directory, nothing in the tree), renders every A/B case with it in a child process and returns the results."""
    nvcc = _nvcc()
    if nvcc is None:
        pytest.skip("nvcc not found: the -DRT_NO_GEN_CULL build cannot be made")
    tmp = tempfile.mkdtemp(prefix="rt_no_gen_cull_")
    try:
        lib = os.path.join(tmp, "librt_b200.so")
        env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
        p = subprocess.run(["make", "-C", os.path.join(ROOT, "cs420-ray-tracer_b200"), "-j3", "NVCC=" + nvcc, "BUILD=" + tmp,
                            "LIB=" + lib, "EXTRA_NVFLAGS=-DRT_NO_GEN_CULL", lib], env=env, capture_output=True, text=True)
        assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
        out = os.path.join(tmp, "full_walk.npz")
        env["RTB200_LIB"] = lib
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "--ab-child", out], env=env, capture_output=True, text=True,
                           timeout=1200)
        assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
        with np.load(out) as z:
            res = {k: z[k] for k in z.files}
        yield res
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


@pytest.mark.parametrize("name,wl", AB_SPEC, ids=["%s-wl%d" % c for c in AB_SPEC])
def test_culled_walk_equals_the_full_walk(rt, full_walk_results, name, wl):
    """Byte-identical frames, hit maps and shadow masks, and the same counters -- fp64_intersections, hits, occluded, every
    level's ray count, filter violations -- as the build whose k_closest1 walks the whole general table.  Only the bundle
    counters differ.  This holds with lights too: the hit blocks k_closest1 hands to the level-k k_shadow depend on the
    queue, not on which pairs the walk visited (but see fp64_intersections below)."""
    got = _ab_render(rt, name, wl)
    ref = {k.split("/", 1)[1]: v for k, v in full_walk_results.items() if k.startswith("%s-wl%d/" % (name, wl))}
    assert ref, "no result of the full-walk build for this case"
    for k in ("rgb", "hit", "mask", "frame"):
        assert got[k].shape == ref[k].shape and np.array_equal(got[k], ref[k]), k
    assert np.array_equal(got["alive"], ref["alive"]) and got["alive"][1] > 0
    # fp64_intersections of a lit scene traced to level 2 or deeper is not comparable between two renders, of EITHER
    # build: the queues of levels >= 2 fill in arrival order, and shadow walks grouped differently per run (wavefront
    # k_shadow or the tail) make a few FP64 evaluations more or fewer -- measured on a B200 in both builds: medium.txt with
    # 40 lights, 320x180 d3 at wave_levels 3: 47 652..47 654; the mirror hall, 1024x576 d3 at wave_levels 2: 1 439 147 or
    # 1 439 148.  At depth 2 (tile-ordered level-1 queue) and without lights the count is the same in every render.  For
    # those cases the lightless render of the same scene -- the same closest hits and reflected rays, no shadow walks --
    # carries k_closest1's FP64 count, and it must be equal.
    D = _ab_case(rt, name, wl)[3]
    lit_deep = got["nlights"] > 0 and D >= 3
    for k in COUNTERS:
        if k == "fp64_intersections" and lit_deep:
            continue
        assert got[k] == ref[k], (k, int(got[k]), int(ref[k]))
        assert got["render_" + k] == ref["render_" + k], ("render", k)
    for k in COUNTERS:
        assert got["dark_" + k] == ref["dark_" + k], ("without lights", k, int(got["dark_" + k]), int(ref["dark_" + k]))
    assert got["filter_violations"] == 0 and got["dark_filter_violations"] == 0
    # the culled walk ran: k_closest1 added bundle walks that the full-walk build does not count
    assert got["dark_bundle_walks"] > ref["dark_bundle_walks"], (int(got["dark_bundle_walks"]), int(ref["dark_bundle_walks"]))


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "--ab-child":
        _ab_child(sys.argv[2])
    else:
        raise SystemExit("usage: test_gpu_wave_levels.py --ab-child OUT.npz")
