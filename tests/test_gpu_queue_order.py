"""The level-0 -> level-1 ray queue is filled in tile order: a reflected ray's position depends on its pixel tile, not on
which warp finished first.  So the level-1 bundles -- and the bundle counters that count their culled walks -- are the same
in every render.  Needs a B200: run with -m gpu."""
import numpy as np
import pytest

from test_gpu_parity import MODES, _scene, check

pytestmark = pytest.mark.gpu

BUNDLE = ("bundle_walks", "bundle_candidates", "bundle_fallbacks")


def test_level1_bundles_are_deterministic(rt, scenes):
    # depth 2 with two wavefront levels: every level runs as its own kernels, nothing reaches the tail (whose queue from
    # level 2 on keeps arrival order).  Table scenes: the level-1 k_closest1 and k_shadow walks are bundle-culled, so
    # their counters depend on which rays share a warp.
    with rt.Renderer(0, mode="fast") as r:
        r.set_option("wave_levels", 2)
        r.upload(scenes["complex"])
        runs = [r.render(1920, 1080, 2) for _ in range(3)]
    rgb0, st0 = runs[0]
    assert st0.bundle_walks > 0
    for rgb, st in runs[1:]:
        assert np.array_equal(rgb, rgb0)
        for k in BUNDLE + ("closest_queries", "hits", "shadow_queries", "occluded", "fp64_intersections"):
            assert getattr(st, k) == getattr(st0, k), k


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("wave_levels", [2, 3])
def test_reflections_without_lights_in_wavefront_levels(rt, oracle, mode, wave_levels):
    # no lights: the level-0 shadow kernel runs only to turn the per-tile ray counts into queue offsets
    spheres = [(0, 0, -3, 1, 1, 0, 0, 0.5, 0.5, 20), (1.5, 0.3, -4, 0.8, 0, 1, 0, 0.9, 0.5, 8),
               (-1.4, -0.2, -3.5, 0.7, 0, 0, 1, 0.7, 0.5, 8), (0, -101, -3, 100, 1, 1, 1, 0.3, 0.5, 4)]
    with rt.Renderer(0, mode=mode) as r:
        r.set_option("wave_levels", wave_levels)
        for W, H, D in ((64, 48, 3), (97, 61, 4), (320, 200, 6)):
            check(rt, oracle, r, _scene(rt, spheres, lights=[]), W, H, D)
