"""The FP32 colour of every shading path against the oracle's FP64 colour, within a bound derived from the code
(tests/colour_bound.py).

Hit indices and shadow booleans are bit-exact against the oracle (test_gpu_parity.py), so every difference between the
float framebuffer of rt_render_tile and oracle.render(..., want_fb=True) comes from FP32 arithmetic, and
colour_bound() bounds it per pixel and channel -- a median of about 1/8 000 of an 8-bit LSB on the fixtures.  The 8-bit
gate of the other tests (1 LSB on 99.9 % of samples) cannot see an error in a clamped channel (>= 1.0), in a deep
reflection level with a small weight, or in a few pixels of one path; this one can.  Each case forces wave_levels and asserts the split between
wavefront levels and the tail kernel (k_bounce) from rt_render's launch count, and that quantising the float frame gives
exactly rt_render's 8-bit frame.

Paths: the wavefront k_closest0 / k_shade (level 0), k_closest1 / level-k k_shadow / k_shade (levels >= 1, tables and
LBVH: k_closest1_dyn / k_shadow_dyn), and every k_bounce instantiation that rtk_launch_fast can launch: tables in shared
memory (<true, false>; lane-cooperative and per-lane regimes), tables beyond shared memory (<false, false>), and the LBVH
tail (<false, true>: an LBVH scene with wave_levels forced below the depth)."""
import os
import sys

import numpy as np
import pytest

TESTS = os.path.dirname(os.path.abspath(__file__))
if TESTS not in sys.path:
    sys.path.insert(0, TESTS)

from colour_bound import colour_bound  # noqa: E402
from conftest import scene_path  # noqa: E402

gpu = pytest.mark.gpu
FIXTURES = ("simple", "medium", "complex")
ALL = 32


def launches(D, wl, L, bvh):
    """Kernels of one render (rtk_launch_fast): per wavefront level closest (LBVH levels >= 1: k_closest1_dyn +
    k_closest1) + shadow (at level 0 also without lights) + shade, then one tail launch if levels remain."""
    n = 0
    for k in range(min(D, wl)):
        n += (2 if bvh and k > 0 else 1) + (1 if L > 0 or k == 0 else 0) + 1
    return n + (1 if D > wl else 0)


_oracle = {}


def oracle_fb(oracle, key, scene, W, H, D):
    if key is None or key not in _oracle:
        o = oracle.render(scene, W, H, D, want_fb=True, want_idx=True)
        o["bound"] = colour_bound(scene, o["hit_idx"], W, H, D, o["shadow_mask"])
        if key is None:
            return o
        _oracle[key] = o
    return _oracle[key]


def render_colour(rt, scene, W, H, D, mode, wl, accel=None):
    """(float frame [H, W, 3] of rt_render_tile over the whole frame, that frame quantised, rt_render's 8-bit frame,
    its stats)."""
    import torch
    with rt.Renderer(0, mode=mode, accel=accel) as r:
        r.set_option("wave_levels", wl)
        r.upload(scene)
        fb = torch.full((H, W, 3), -7.0, dtype=torch.float32, device="cuda:0")
        torch.cuda.synchronize()
        r.render_tile_device(W, H, D, (0, 0, W, H), fb.data_ptr())
        torch.cuda.synchronize()
        q = (255.99 * torch.clamp(fb, max=1.0)).to(torch.int32).to(torch.uint8).cpu().numpy()
        frame, st = r.render(W, H, D)
    return fb.cpu().numpy(), q, frame, st


def check_colour(rt, oracle, scene, W, H, D, mode="fast", wl=1, key=None, accel=None):
    """Renders one case and asserts: every finite sample within the bound, non-finite samples where the oracle has them,
    the quantised float frame = rt_render's frame, and the launch count of the forced wavefront / tail split.
    Returns (stats, worst error / bound, largest error)."""
    o = oracle_fb(oracle, key, scene, W, H, D)
    fb, q, frame, st = render_colour(rt, scene, W, H, D, mode, wl, accel)
    bvh = mode == "bvh"
    assert st.kernel_launches == launches(D, wl, scene.nlights, bvh), (st.kernel_launches, D, wl, bvh)
    assert [int(x) for x in st.alive[:D]] == o["counters"]["alive"][:D]
    ref, bound = o["fb"], o["bound"]
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(fb), fin), "non-finite samples differ"
    err = np.abs(fb.astype(np.float64) - ref)
    ratio = np.where(fin, err / bound, 0.0)
    bad = np.argwhere(ratio > 1.0)
    assert bad.size == 0, "%d samples beyond the bound, first (row, col, ch) %s: gpu %r oracle %r bound %.3g hit %s" % (
        len(bad), bad[0].tolist(), float(fb[tuple(bad[0])]), float(ref[tuple(bad[0])]), bound[tuple(bad[0])],
        o["hit_idx"][bad[0][0], bad[0][1]].tolist())
    assert np.array_equal(q, frame), "the quantised float frame is not rt_render's frame"
    worst, emax = float(ratio.max()), float(err[fin].max()) if fin.any() else 0.0
    print("colour %s %dx%d d%d %s wl%d: max |err| %.3g, max err/bound %.3g" % (key, W, H, D, mode, wl, emax, worst))
    return st, worst, emax


# ---------------------------------------------------------------------------------------------
# the bound is not vacuous (no GPU needed)

@pytest.mark.parametrize("name", FIXTURES)
def test_colour_bound_is_tight_on_the_fixtures(rt, oracle, name):
    """On the fixtures at 160x90 depth 5 the bound's median is at most 2^-16 (1/256 of an 8-bit LSB), its maximum below
    1/8 LSB; it covers the FP32 rounding of the oracle's own colour (the least any FP32 renderer can be off by); and the
    bound's own FP64 trace of the oracle's paths reproduces the oracle's colour."""
    sc = rt.load_scene(scene_path(name))
    W, H, D = 160, 90, 5
    o = oracle.render(sc, W, H, D, want_fb=True, want_idx=True)
    bound, col = colour_bound(sc, o["hit_idx"], W, H, D, o["shadow_mask"], colour=True)
    assert np.abs(col - o["fb"]).max() < 1e-12
    assert np.median(bound) <= 2.0 ** -16, np.median(bound)
    assert bound.max() < 0.125 / 255, bound.max()
    assert (np.abs(o["fb"].astype(np.float32) - o["fb"]) <= bound).all()


# ---------------------------------------------------------------------------------------------
# 1. the fixtures at every split between wavefront levels and tail, tables and LBVH

@gpu
@pytest.mark.parametrize("wl", [1, 2, 3, ALL])
@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("W,H,D", [(160, 90, 5), (97, 61, 10)])
@pytest.mark.parametrize("name", FIXTURES)
def test_fixture_colour(rt, oracle, name, W, H, D, mode, wl):
    sc = rt.load_scene(scene_path(name))
    st, _, _ = check_colour(rt, oracle, sc, W, H, D, mode, wl, key=(name, W, H, D))
    assert st.alive[1] > 0 and (name == "simple" or st.alive[2] > 0)     # (simple.txt has one mirror)


# ---------------------------------------------------------------------------------------------
# 2. reflectivity edges and depth exhaustion, on a pair of facing mirrors that carries rays to deep levels

def mirror_pair(rt, refl, shin=50.0):
    """Two facing mirror spheres (reflectivity `refl`) with a 0.4 gap; the camera looks into the gap, so rays bounce
    between them for many levels.  A ground sphere and a diffuse back sphere catch the rays that leave."""
    from test_gpu_parity import _scene
    sph = [(-2.2, 0, -5, 2, 0.9, 0.6, 0.3, refl, 0.1, shin), (2.2, 0, -5, 2, 0.3, 0.6, 0.9, refl, 0.1, shin),
           (0, -102.5, -5, 100, 0.5, 0.5, 0.5, 0.2, 0.8, 10), (0, 0, -14, 4, 0.8, 0.8, 0.2, 0.0, 1, 20)]
    return _scene(rt, sph, lights=[(4, 6, 0, 1, 1, 1, 1), (-5, 3, -2, 0.7, 0.5, 0.9, 1)], camera=(0, 0.3, 1.5, 0, 0, -5, 50))


@gpu
@pytest.mark.parametrize("wl", [1, ALL])
@pytest.mark.parametrize("refl", [1.0, 0.999999, 1.5, -0.5, -2.0, 1e-300, -0.0])
def test_reflectivity_edges(rt, oracle, refl, wl):
    """1.0 (no own colour), 0.999999, 1.5 (weights grow, 1 - r < 0), -0.5 and -2 (no blend: the reference blends only
    when r > 0), 1e-300 (> 0 in FP64, 0 in FP32: the flag is decided in double, the weight is 0) and -0.0."""
    W, H, D = 96, 64, 10
    st, _, _ = check_colour(rt, oracle, mirror_pair(rt, refl), W, H, D, "fast", wl, key=("refl", refl))
    if refl > 0:
        assert st.alive[5] > 0                     # deep levels carry weight
    else:
        assert st.alive[1] > 0                     # (the ground still reflects)


def parallel_mirrors(rt):
    """Two spheres of radius 1000 (reflectivity 0.5) whose near sides are nearly flat mirrors 0.4 apart; the camera looks
    between them, so most rays bounce from one to the other until the depth runs out (1816 of the 96 x 64 pixels still
    reflect at level 31)."""
    from test_gpu_parity import _scene
    sph = [(-1000.2, 0, -20, 1000, 0.7, 0.6, 0.5, 0.5, 0.5, 30), (1000.2, 0, -20, 1000, 0.5, 0.6, 0.7, 0.5, 0.5, 30)]
    return _scene(rt, sph, lights=[(0, 30, -20, 1, 1, 1, 1), (0, -3, 10, 0.5, 0.6, 0.8, 1)], camera=(0, 0, 5, 0, 0, -20, 50))


@gpu
@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("wl", [1, ALL])
@pytest.mark.parametrize("D", [1, 2, 32])
def test_depth_exhaustion_at_a_reflective_hit(rt, oracle, D, wl, mode):
    """A reflective hit at the last level adds its own colour times (1 - r) and a black child: at depth 1 in k_shade,
    at depth 2 and 32 in k_bounce (wl 1) or in the last wavefront k_shade (wl 32)."""
    W, H = 96, 64
    st, _, _ = check_colour(rt, oracle, parallel_mirrors(rt), W, H, D, mode, wl, key=("exhaust", D))
    assert st.alive[D - 1] > 0


# ---------------------------------------------------------------------------------------------
# 3. shininess: __powf's error grows with it; for 0 < s < 1, x^s is not Lipschitz at 0

@gpu
@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("shin", [0.0, 0.5, 1.0, 200.0, 1000.0])
def test_shininess(rt, oracle, shin, mode):
    from test_gpu_parity import _scene
    sph = [(0, 0, -4, 1.2, 0.8, 0.3, 0.3, 0.3, 0.7, shin), (-1.8, -0.5, -5, 0.8, 0.3, 0.8, 0.3, 0.0, 1, shin),
           (0, -101.2, -4, 100, 0.6, 0.6, 0.6, 0.4, 0.6, shin)]
    sc = _scene(rt, sph, lights=[(2, 3, 0, 1, 1, 1, 1), (-3, 2, -1, 0.6, 0.6, 0.9, 1), (0, 5, -2, 0.5, 0.4, 0.3, 1)])
    check_colour(rt, oracle, sc, 128, 96, 4, mode, 2, key=("shin", shin))


# ---------------------------------------------------------------------------------------------
# 4. many lights (occlusion bits up to 32, per-light bytes above), transformed scenes

@gpu
@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("nl", [32, 33, 40])
def test_many_lights_colour(rt, oracle, nl, mode):
    from test_gpu_wave_levels import many_lights
    sc = many_lights(rt, rt.load_scene(scene_path("medium")), nl)
    check_colour(rt, oracle, sc, 96, 54, 3, mode, 2, key=("lights", nl))


@gpu
@pytest.mark.parametrize("wl", [1, ALL])
@pytest.mark.parametrize("tag,k,off", [("o1e4", 1.0, (1e4, 1e4, 1e4)), ("s1e-2", 1e-2, (0, 0, 0)), ("s1e3", 1e3, (0, 0, 0))])
def test_transformed_scene_colour(rt, oracle, tag, k, off, wl):
    from test_gpu_wave_levels import transformed
    sc = transformed(rt, rt.load_scene(scene_path("complex")), k, off)
    check_colour(rt, oracle, sc, 160, 90, 5, "fast", wl, key=("complex", tag))


# ---------------------------------------------------------------------------------------------
# 5. the tail kernel's two regimes and its instantiations

def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@gpu
def test_tail_lane_cooperative_regime(rt, oracle):
    """k_bounce spreads the nq rays entering it over all resident warps, per = min(32, max(4, ceil(nq / nwarps))) rays
    per warp fetch, and a warp with at most kCoopMaxLive = 12 live rays tests lane-cooperatively.  nwarps is the
    occupancy (>= 1 CTA of 4 warps per SM) times the SM count, so with nq <= 16 SMs every fetch takes 4 rays: every
    warp starts lane-cooperative at the tail's first level."""
    sc = rt.load_scene(scene_path("complex"))
    W, H, D = 64, 36, 5
    st, _, _ = check_colour(rt, oracle, sc, W, H, D, "fast", 1, key=("complex", W, H, D))
    assert 0 < st.alive[1] <= 16 * _sm_count(), st.alive[1]


@gpu
def test_tail_per_lane_regime(rt, oracle):
    """The other side: with nq > 12 x 64 warps per SM (the most a B200 SM holds) x SMs, per >= 13 and every full fetch
    starts with more than kCoopMaxLive live rays -- the per-lane tests and the culled shadow walks."""
    from test_gpu_wave_levels import mirror_hall
    W, H, D = 1024, 576, 3
    st, _, _ = check_colour(rt, oracle, mirror_hall(rt), W, H, D, "fast", 1, key=("hall", W, H, D))
    assert st.alive[1] > 12 * 64 * _sm_count(), st.alive[1]


@gpu
@pytest.mark.parametrize("wl", [1, 2])
def test_tail_tables_beyond_shared_memory(rt, oracle, wl):
    """1000 spheres and 4 lights: the tail's tables (4 light tables + the general table) exceed the 90 KB it stages, so
    k_bounce<false, false> reads them through L1/L2."""
    import gen_scene
    sc = rt.Scene(*gen_scene.generate(1000, 420, 0.3, 1.5))
    st, _, _ = check_colour(rt, oracle, sc, 240, 136, 5, "fast", wl, key=("gen1000",), accel=1)
    assert st.alive[wl] > 0


# ---------------------------------------------------------------------------------------------
# 6. fuzz scenes

@gpu
@pytest.mark.parametrize("mode,wl", [("fast", 1), ("fast", 2), ("bvh", 1), ("bvh", ALL)])
@pytest.mark.parametrize("seed", [0, 1, 2, 5, 7, 11])
def test_fuzz_scene_colour(rt, oracle, seed, mode, wl):
    from test_gpu_parity import _random_scene
    W, H, D = [(96, 54, 4), (61, 47, 6), (130, 40, 3)][seed % 3]
    check_colour(rt, oracle, _random_scene(rt, seed), W, H, D, mode, wl, key=("fuzz", seed))
