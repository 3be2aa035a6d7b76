"""Parity of the CUDA path (through the C ABI) against the oracle and the committed goldens.

Bars (BASELINE.json north_star): hit / sphere index per reflection level and shadow booleans
BIT-EXACT; 8-bit RGB within 1 LSB on >= 99.9 % of channel samples (scripts/compare_ppm.py rule
with tolerance 0.5).  Needs a B200: run with -m gpu."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu
MODES = ["exact", "fast", "bvh"]     # "bvh" = fast path with the LBVH forced for every scene size


@pytest.fixture(scope="module")
def renderers(rt):
    rs = {m: rt.Renderer(0, mode=m) for m in MODES}
    yield rs
    for r in rs.values():
        r.close()


def check(rt, oracle, renderer, scene, W, H, D, gold=None, rgb_exact_frac=None):
    renderer.upload(scene)
    rgb, hit, mask, st = renderer.render_debug(W, H, D)
    if gold is None:
        o = oracle.render(scene, W, H, D, want_idx=True)
        gold = {"hit_idx": o["hit_idx"], "shadow_mask": o["shadow_mask"], "rgb": o["rgb"], "counters": o["counters"]}
    if D > 0:
        bad = np.argwhere(hit != gold["hit_idx"])
        assert bad.size == 0, "hit index mismatch at (j,i,level) %s: got %s want %s" % (
            bad[:5].tolist(), hit[tuple(bad[0])], gold["hit_idx"][tuple(bad[0])])
        bad = np.argwhere(mask != gold["shadow_mask"])
        assert bad.size == 0, "shadow mask mismatch at %s" % bad[:5].tolist()
    ok, pct, mx = rt.compare_rgb(gold["rgb"], rgb, 0.5)
    assert ok and mx <= 2, "rgb: %.4f %% of samples beyond 1 LSB, max diff %d" % (pct, mx)
    for k in ("closest_queries", "hits", "shadow_queries", "occluded"):
        assert getattr(st, k) == gold["counters"][k], k
    assert st.filter_violations == 0           # the FP32 filter never contradicted the FP64 decider
    assert st.sphere_tests == (st.closest_queries + st.shadow_queries) * scene.nspheres
    return rgb, st


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", ["simple", "medium", "complex"])
def test_small_goldens(rt, oracle, renderers, scenes, name, mode):
    z = np.load(os.path.join(GOLDEN, "small_%s.npz" % name))
    gold = {"hit_idx": z["hit_idx"], "shadow_mask": z["shadow_mask"], "rgb": z["rgb_top_first"][::-1],
            "counters": json.loads(str(z["counters"]))}
    check(rt, oracle, renderers[mode], scenes[name], 160, 90, 5, gold)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name,W,H,D", [("simple", 1280, 720, 10), ("medium", 1920, 1080, 5), ("complex", 1920, 1080, 5),
                                        ("complex", 1280, 720, 10)])
def test_baseline_configs_full_size(rt, oracle, renderers, scenes, golden, name, W, H, D, mode):
    rgb, st = check(rt, oracle, renderers[mode], scenes[name], W, H, D)
    g = [c for c in golden["counters"] if (c["scene"], c["W"], c["H"], c["depth"]) == (name, W, H, D)]
    if g:
        assert st.closest_queries == g[0]["closest_queries"] and st.shadow_queries == g[0]["shadow_queries"]
        assert [int(x) for x in st.alive[:D]] == g[0]["alive"]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("W,H,D", [(97, 61, 3), (2, 2, 1), (33, 7, 2), (640, 1, 2), (3, 500, 4), (130, 70, 0), (64, 64, 1), (200, 120, 32)])
def test_ragged_sizes_and_depths(rt, oracle, renderers, scenes, W, H, D, mode):
    check(rt, oracle, renderers[mode], scenes["medium"], W, H, D)


def _scene(rt, spheres, lights=((5, 8, 2, 1, 1, 1, 1),), ambient=(0.1, 0.1, 0.1), camera=(0, 0, 5, 0, 0, -1, 60)):
    return rt.Scene(np.array(spheres, dtype=np.float64).reshape(-1, 10), np.array(lights, dtype=np.float64).reshape(-1, 7),
                    ambient, camera)


@pytest.mark.parametrize("mode", MODES)
def test_empty_and_degenerate_scenes(rt, oracle, renderers, mode):
    r = renderers[mode]
    check(rt, oracle, r, _scene(rt, []), 64, 48, 3)                                    # no spheres: all sky
    check(rt, oracle, r, _scene(rt, [(0, 0, -3, 1, 1, 0, 0, 0.5, 0.5, 20)], lights=[]), 64, 48, 3)   # no lights
    check(rt, oracle, r, _scene(rt, [(0, 0, 0, 50, 1, 1, 1, 0.3, 0.5, 20)]), 64, 48, 4)   # camera inside a sphere
    check(rt, oracle, r, _scene(rt, [(0, 0, -3, 1, 1, 0, 0, 1.0, 0.5, 0)]), 64, 48, 4)    # mirror, shininess 0
    check(rt, oracle, r, _scene(rt, [(0, 0, -3, 1, 1, 0, 0, -0.2, 0.5, 8)]), 64, 48, 4)   # negative reflectivity


@pytest.mark.parametrize("mode", MODES)
def test_ties_go_to_lowest_index(rt, oracle, renderers, mode):
    """include/scene.h:52 strict '<' (SURVEY F8): coincident / touching / nested spheres."""
    s = (0.3, 0.2, -4, 1.25, 0.8, 0.3, 0.2, 0.4, 0.5, 30)
    spheres = [s, s, (0.3, 0.2, -4, 1.25, 0.1, 0.9, 0.2, 0.0, 1, 5),        # three coincident spheres
               (2.55, 0.2, -4, 1.0, 0.2, 0.3, 0.9, 0.6, 0.4, 50),           # touches the first (1.25 + 1.0 = 2.25 apart)
               (0.3, 0.2, -4, 0.5, 1, 1, 1, 0.9, 0.1, 90),                  # nested inside
               (0, -101.05, -4, 100, 0.5, 0.5, 0.5, 0.2, 1, 5)]             # ground touching
    check(rt, oracle, renderers[mode], _scene(rt, spheres, lights=[(5, 8, 2, 1, 1, 1, 1), (-6, 3, 1, 1, 0.5, 0.5, 1)]), 320, 200, 6)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("n,seed,W,H,D", [(300, 7, 320, 180, 5), (1000, 420, 240, 136, 5), (2001, 9, 160, 90, 4)])
def test_synthetic_overlapping_spheres(rt, oracle, renderers, n, seed, W, H, D, mode):
    import gen_scene
    sph, lights, amb, cam = gen_scene.generate(n, seed, 0.3, 1.5)      # big radii: many overlaps
    check(rt, oracle, renderers[mode], rt.Scene(sph, lights, amb, cam), W, H, D)


@pytest.mark.parametrize("mode", MODES)
def test_far_from_origin_scene(rt, oracle, renderers, scenes, mode):
    """Input rounding must be covered by the FP32 filter margins (SURVEY 7.3-H1 'M term')."""
    sc = scenes["medium"]
    off = np.array([1000.0, -2000.0, 500.0])
    sph = sc.spheres.copy(); sph[:, :3] += off
    lig = sc.lights.copy(); lig[:, :3] += off
    cam = sc.camera.copy(); cam[:3] += off; cam[3:6] += off
    check(rt, oracle, renderers[mode], rt.Scene(sph, lig, sc.ambient, cam), 320, 180, 5)


@pytest.mark.parametrize("mode", MODES)
def test_deterministic_and_rerenderable(rt, renderers, scenes, mode):
    r = renderers[mode]
    r.upload(scenes["complex"])
    a, _ = r.render(640, 360, 5)
    b, _ = r.render(640, 360, 5)
    r.upload(scenes["simple"])
    c, _ = r.render(640, 360, 5)
    r.upload(scenes["complex"])
    d, _ = r.render(640, 360, 5)
    assert np.array_equal(a, b) and np.array_equal(a, d) and not np.array_equal(a, c)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("band_h,n", [(16, 2), (16, 8), (4, 3), (64, 5)])
def test_row_bands_reassemble_to_the_full_frame(rt, renderers, scenes, band_h, n, mode):
    import torch
    r = renderers[mode]
    r.upload(scenes["complex"])
    W, H, D = 480, 270, 5
    full, _ = r.render(W, H, D)
    out = np.zeros_like(full)
    for rank in range(n):
        rows = rt.band_row_list(H, band_h, rank, n)
        buf = torch.zeros(len(rows) * W * 3 + 16, dtype=torch.uint8, device="cuda:0")
        st = r.render_bands_device(W, H, D, band_h, rank, n, buf.data_ptr(), None, want_stats=True)
        assert st.rows_rendered == len(rows)
        out[rows] = buf[:len(rows) * W * 3].cpu().numpy().reshape(len(rows), W, 3)
    assert np.array_equal(out, full)


def test_row_bands_with_supersampling(rt, scenes):
    """rt_render_bands with antialias on: the bands of the 2x2-supersampled frame reassemble to rt_render's."""
    import torch
    W, H, D, band_h, n = 200, 114, 4, 16, 3
    with rt.Renderer(0) as r:
        r.set_option("antialias", 1)
        r.upload(scenes["complex"])
        full, _ = r.render(W, H, D)
        out = np.zeros_like(full)
        for rank in range(n):
            rows = rt.band_row_list(H, band_h, rank, n)
            buf = torch.zeros(len(rows) * W * 3 + 16, dtype=torch.uint8, device="cuda:0")
            torch.cuda.synchronize()
            r.render_bands_device(W, H, D, band_h, rank, n, buf.data_ptr(), None, want_stats=True)
            out[rows] = buf[:len(rows) * W * 3].cpu().numpy().reshape(len(rows), W, 3)
    assert np.array_equal(out, full)


@pytest.mark.parametrize("n,seed,W,H,D,modes", [(10000, 420, 480, 270, 5, ("tables", "bvh")), (100000, 421, 384, 216, 8, ("bvh",))])
def test_large_synthetic_against_fp64_brute_force(rt, renderers, n, seed, W, H, D, modes):
    """BASELINE configs 4 (10k spheres, streamed tables and LBVH) and 5 (100k spheres, device-built LBVH)
    at reduced resolution: the CPU oracle would need minutes to hours, so the FP64 brute-force kernel is
    the checker here (itself pinned to the oracle by the tests above)."""
    import gen_scene
    sc = rt.Scene(*gen_scene.generate(n, seed))
    renderers["exact"].upload(sc)
    ref = renderers["exact"].render_debug(W, H, D)
    for m in modes:
        with rt.Renderer(0, mode="fast", accel={"tables": 1, "bvh": 2}[m]) as r:
            r.upload(sc)
            out = r.render_debug(W, H, D)
        assert np.array_equal(ref[1], out[1]), m
        assert np.array_equal(ref[2], out[2]), m
        ok, pct, mx = rt.compare_rgb(ref[0], out[0], 0.5)
        assert ok and mx <= 2, m
        assert out[3].filter_violations == 0
        for k in ("closest_queries", "hits", "shadow_queries", "occluded"):
            assert getattr(out[3], k) == getattr(ref[3], k), (m, k)


@pytest.mark.parametrize("n,seed,W,H,D", [(10000, 420, 3840, 2160, 5), (100000, 421, 7680, 4320, 8)])
def test_full_size_large_configs_two_algorithms_agree(rt, n, seed, W, H, D):
    """BASELINE configs 4 and 5 at FULL size: far too large for the CPU oracle, so the check is that two independent
    candidate-selection algorithms -- streamed brute-force table walks and the device-built LBVH -- produce the
    bit-identical frame and identical ray counters (every level's alive count, hits, occluded shadow rays), with
    no filter violation.  Both decide through the same exact FP64 routines pinned by the tests above."""
    import gen_scene
    sc = rt.Scene(*gen_scene.generate(n, seed))
    out = {}
    for m, acc in (("tables", 1), ("bvh", 2)):
        with rt.Renderer(0, mode="fast", accel=acc) as r:
            r.upload(sc)
            out[m] = r.render(W, H, D)
    (fa, sa), (fb, sb) = out["tables"], out["bvh"]
    assert np.array_equal(fa, fb)
    for k in ("closest_queries", "hits", "shadow_queries", "occluded", "filter_violations"):
        assert getattr(sa, k) == getattr(sb, k), k
    assert [int(x) for x in sa.alive] == [int(x) for x in sb.alive] and sa.filter_violations == 0
    assert sa.alive[0] == W * H and sa.shadow_queries == sa.hits * sc.nlights


@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("name,W,H,D", [("simple", 160, 90, 5), ("complex", 192, 108, 5), ("medium", 97, 61, 3)])
def test_supersampling_matches_the_four_sample_oracle(rt, oracle, scenes, name, W, H, D, mode):
    """rt_set_option antialias = the reference's ray_cuda -a (src/main_gpu.cu:249-258,327-333): per-sample hit
    indices / shadow masks bit-exact against four offset renders of the oracle, averaged RGB within 1 LSB."""
    o = oracle.render_supersampled(scenes[name], W, H, D)
    with rt.Renderer(0, mode=mode) as r:
        r.set_option("antialias", 1)
        r.upload(scenes[name])
        rgb, hit, mask, st = r.render_debug(W, H, D)
        plain, _ = r.render(W, H, D)
        r.set_option("antialias", 0)
        off, _ = r.render(W, H, D)
    assert hit.shape == (2 * H, 2 * W, D)
    for s, (a, b) in enumerate(((0, 0), (1, 0), (0, 1), (1, 1))):
        assert np.array_equal(hit[b::2, a::2], o["samples"][s]["hit_idx"]), s
        assert np.array_equal(mask[b::2, a::2], o["samples"][s]["shadow_mask"]), s
    ok, pct, mx = rt.compare_rgb(o["rgb"], rgb, 0.5)
    assert ok and mx <= 2, (pct, mx)
    assert np.array_equal(rgb, plain) and not np.array_equal(rgb, off)
    assert st.closest_queries == sum(p["counters"]["closest_queries"] for p in o["samples"])
    assert st.filter_violations == 0


@pytest.mark.parametrize("mode", ["fast", "bvh"])
def test_tile_renders_assemble_to_the_frame(rt, oracle, scenes, mode):
    """rt_render_tile (the reference's launch_gpu_kernel convention: tile offsets, caller-owned float3 framebuffer,
    stream): ragged tiles assemble to exactly the whole-frame tile render; quantised, that is rt_render's frame."""
    import torch
    W, H, D = 200, 120, 5
    with rt.Renderer(0, mode=mode) as r:
        r.upload(scenes["complex"])
        whole = torch.full((H, W, 3), -1.0, dtype=torch.float32, device="cuda:0")
        torch.cuda.synchronize()
        r.render_tile_device(W, H, D, (0, 0, W, H), whole.data_ptr())
        tiled = torch.full((H, W, 3), -1.0, dtype=torch.float32, device="cuda:0")
        stream = torch.cuda.Stream()
        torch.cuda.synchronize()                     # the fills above ran on torch's default stream
        for (x, y, w, h) in [(0, 0, 64, 64), (64, 0, 136, 64), (0, 64, 33, 56), (33, 64, 167, 17), (33, 81, 167, 39)]:
            r.render_tile_device(W, H, D, (x, y, w, h), tiled.data_ptr(), stream.cuda_stream)
        stream.synchronize()
        torch.cuda.synchronize()
        assert torch.equal(whole, tiled)
        partial = torch.full((H, W, 3), -1.0, dtype=torch.float32, device="cuda:0")
        torch.cuda.synchronize()
        r.render_tile_device(W, H, D, (10, 20, 50, 30), partial.data_ptr())
        torch.cuda.synchronize()
        inside = torch.zeros((H, W), dtype=torch.bool, device="cuda:0"); inside[20:50, 10:60] = True
        assert torch.equal(partial[inside], whole[inside]) and bool((partial[~inside] == -1.0).all())
        frame, _ = r.render(W, H, D)
        q = (255.99 * torch.clamp(whole, max=1.0)).to(torch.int32).to(torch.uint8).cpu().numpy()
        assert np.array_equal(q, frame)
        with pytest.raises(rt.RtError):
            r.render_tile_device(W, H, D, (150, 0, 64, 64), whole.data_ptr())
    o = oracle.render(scenes["complex"], W, H, D, want_fb=True)
    assert np.abs(whole.cpu().numpy() - o["fb"]).max() < 2e-3


def _random_scene(rt, seed):
    """Adversarial little scenes: overlapping / nested / coincident spheres of very different sizes, lights and camera
    anywhere (inside spheres too), odd fields of view, shininess 0, zero and negative reflectivity."""
    g = np.random.default_rng(1000 + seed)
    n = int(g.integers(1, 60))
    c = g.uniform(-6, 6, (n, 3)); c[:, 2] -= 8
    r = np.exp(g.uniform(np.log(0.05), np.log(4.0), n))
    if n > 3:
        c[1] = c[0]                                       # concentric
        c[2] = c[0] + np.array([r[0] + r[2], 0, 0])        # externally tangent
    if n > 6 and seed % 3 == 0:
        c[5], r[5] = c[4], r[4]                            # coincident twins (lowest index wins, SURVEY F8)
    col = g.uniform(0, 1, (n, 3))
    refl = np.where(g.random(n) < 0.4, 0.0, g.uniform(-0.2, 1.0, n))
    shin = np.where(g.random(n) < 0.15, 0.0, g.integers(1, 200, n).astype(np.float64))
    sph = np.column_stack([c, r, col, refl, 1 - refl, shin])
    if seed % 4 == 1:
        sph = np.vstack([sph, [0, -1003, -8, 1000, 0.4, 0.4, 0.4, 0.3, 1, 10]])   # a huge ground sphere
    L = int(g.integers(0, 6))
    lights = np.column_stack([g.uniform(-8, 8, (L, 3)) - np.array([0, -4, 6]), g.uniform(0.2, 1, (L, 3)), np.ones(L)]) if L else np.zeros((0, 7))
    cam_pos = g.uniform(-3, 3, 3) + np.array([0, 0, 4.0])
    if seed % 5 == 2:
        cam_pos = sph[0, :3] + 0.3 * sph[0, 3]             # camera inside a sphere
    cam = np.concatenate([cam_pos, sph[int(g.integers(0, n)), :3] + g.uniform(-0.5, 0.5, 3), [float(g.uniform(20, 110))]])
    sph = np.array([[float("%.6f" % v) for v in row] for row in sph.tolist()])
    return rt.Scene(sph, np.asarray(lights, dtype=np.float64), g.uniform(0, 0.3, 3), cam)


@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("seed", range(24))
def test_fuzz_random_scenes(rt, oracle, renderers, seed, mode):
    W, H, D = [(96, 54, 4), (61, 47, 6), (130, 40, 3)][seed % 3]
    check(rt, oracle, renderers[mode], _random_scene(rt, seed), W, H, D)


@pytest.mark.parametrize("mode", ["fast", "bvh"])
def test_buffers_sized_by_an_earlier_frame(rt, oracle, scenes, mode):
    """Regression: work buffers only grow.  A context that rendered a large frame of a one-light scene and then renders a
    small frame of a five-light scene must stride its per-light occlusion rows by THIS frame's slot count (found by
    scripts/fuzz_parity.py: the allocated capacity as stride indexed past the buffer)."""
    one = scenes["complex"]
    one_light = rt.Scene(one.spheres, one.lights[:1], one.ambient, one.camera)
    with rt.Renderer(0, mode=mode) as r:
        r.upload(one_light)
        r.render(640, 360, 3)
        for name, W, H, D in (("complex", 96, 54, 4), ("medium", 61, 47, 6)):
            check(rt, oracle, r, scenes[name], W, H, D)


def test_errors(rt, renderers, scenes):
    r = rt.Renderer(0)
    with pytest.raises(rt.RtError, match="no scene uploaded"):
        r.render(16, 16, 2)
    r.upload(scenes["simple"])
    with pytest.raises(rt.RtError):
        r.render(0, 16, 2)
    with pytest.raises(rt.RtError):
        r.render(16, 16, 33)
    with pytest.raises(rt.RtError, match="unknown key"):
        r.set_option("frame_kernel", 1)
    r.close()


# ---------------------------------------------------------------------------------------------
# round 2: the parity holes the round-1 review named

@pytest.mark.parametrize("n,seed,W,H,D,pix_step", [(10000, 420, 3840, 2160, 5, 251), (100000, 421, 7680, 4320, 8, 2039)])
def test_full_size_large_configs_against_the_cpu_oracle_on_a_pixel_subsample(rt, oracle, n, seed, W, H, D, pix_step):
    """BASELINE configs 4 and 5 at their FULL sizes against the CPU oracle ("hit parity to brute-force serial"): the
    oracle renders every pix_step-th pixel (a prime stride, so the samples sweep all columns and rows;
    oracle/rt_oracle.c rto_render, the loop of src/main.cpp:146-157) by FP64 brute force over all spheres; on those
    pixels the production path (LBVH from 1024 spheres on) must give the same sphere index at every reflection level,
    the same per-light shadow booleans, and RGB within the compare_ppm.py gate."""
    import gen_scene
    sc = rt.Scene(*gen_scene.generate(n, seed))
    o = oracle.render(sc, W, H, D, want_idx=True, pix_step=pix_step)
    with rt.Renderer(0, mode="fast") as r:
        r.upload(sc)
        rgb, hit, mask, st = r.render_debug(W, H, D)
    sel = slice(0, W * H, pix_step)
    g_hit, o_hit = hit.reshape(-1, D)[sel], o["hit_idx"].reshape(-1, D)[sel]
    g_mask, o_mask = mask.reshape(-1, D)[sel], o["shadow_mask"].reshape(-1, D)[sel]
    assert g_hit.shape[0] == (W * H + pix_step - 1) // pix_step
    assert (o_hit[:, 0] != -2).all()                      # the oracle did trace every sampled pixel
    bad = np.argwhere(g_hit != o_hit)
    assert bad.size == 0, "hit index mismatch at sample/level %s: got %s want %s" % (bad[:5].tolist(), g_hit[tuple(bad[0])], o_hit[tuple(bad[0])])
    assert np.array_equal(g_mask, o_mask)
    ok, pct, mx = rt.compare_rgb(o["rgb"].reshape(-1, 3)[sel], rgb.reshape(-1, 3)[sel], 0.5)
    assert ok and mx <= 2, (pct, mx)
    assert st.filter_violations == 0
    # ray counters of the sampled pixels: every level's alive count follows from the index maps
    assert o["counters"]["closest_queries"] == int((o_hit != -2).sum()) == int((g_hit != -2).sum())
    assert o["counters"]["hits"] == int((g_hit >= 0).sum())


@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("name,W,H,D", [("complex", 320, 180, 5), ("medium", 97, 61, 3)])
def test_index_parity_of_the_production_launch_sequence(rt, oracle, scenes, name, W, H, D, mode):
    """Hit indices / shadow masks of (a) a render WITHOUT stats -- the bench's launch sequence, every kernel after the
    first with programmatic dependent launch -- and (b) a render with level_timing on (event records between the
    level-0 kernels, no PDL) are both bit-exact against the oracle."""
    o = oracle.render(scenes[name], W, H, D, want_idx=True)
    with rt.Renderer(0, mode=mode) as r:
        r.upload(scenes[name])
        for timing in (0, 1):
            r.set_option("level_timing", timing)
            for want_stats in (False, True):
                for _ in range(3):                       # repeated frames: the wave-level feedback switches sequences
                    rgb, hit, mask, _ = r.render_debug(W, H, D, want_stats=want_stats)
                    assert np.array_equal(hit, o["hit_idx"]) and np.array_equal(mask, o["shadow_mask"])
                    assert rt.compare_rgb(o["rgb"], rgb, 0.5)[0]


@pytest.mark.parametrize("mode", ["fast", "bvh"])
def test_tiles_round_robin_over_streams(rt, scenes, mode):
    """The reference's ray_hybrid launches ALL its tiles without a sync on streams[i++ % NUM_STREAMS]
    (src/main_hybrid.cpp:611-622).  Renders of one ctx share its work buffers, so the library serialises them on the
    device; the assembled frame must equal the single-stream one, repeatedly."""
    import torch
    W, H, D, T = 256, 192, 5, 64
    with rt.Renderer(0, mode=mode) as r:
        r.upload(scenes["complex"])
        whole = torch.full((H, W, 3), -1.0, dtype=torch.float32, device="cuda:0")
        torch.cuda.synchronize()
        r.render_tile_device(W, H, D, (0, 0, W, H), whole.data_ptr())
        torch.cuda.synchronize()
        streams = [torch.cuda.Stream() for _ in range(3)]
        for rep in range(4):
            tiled = torch.full((H, W, 3), -1.0, dtype=torch.float32, device="cuda:0")
            torch.cuda.synchronize()
            k = 0
            for y in range(0, H, T):
                for x in range(0, W, T):
                    r.render_tile_device(W, H, D, (x, y, T, T), tiled.data_ptr(), streams[k % 3].cuda_stream)
                    k += 1
            for s in streams:
                s.synchronize()
            torch.cuda.synchronize()
            assert torch.equal(whole, tiled), rep


def test_two_contexts_interleave_on_one_device(rt, oracle, scenes):
    """Two contexts with DIFFERENT scenes on the same device, each rendering on its own stream without host syncs in
    between: the per-device __constant__ bank (camera, lights, ambient) changes hands in stream order."""
    import torch
    W, H, D = 200, 120, 4
    names = ("complex", "simple")
    gold = [oracle.render(scenes[n], W, H, D)["rgb"] for n in names]
    rs = [rt.Renderer(0), rt.Renderer(0)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    try:
        for r, n in zip(rs, names):
            r.upload(scenes[n])
        bufs = [[torch.zeros(H * W * 3 + 16, dtype=torch.uint8, device="cuda:0") for _ in range(6)] for _ in rs]
        torch.cuda.synchronize()
        for k in range(6):
            for i, r in enumerate(rs):
                r.render_bands_device(W, H, D, H, 0, 1, bufs[i][k].data_ptr(), streams[i].cuda_stream)
        torch.cuda.synchronize()
        for i in range(2):
            for k in range(6):
                got = bufs[i][k][:H * W * 3].cpu().numpy().reshape(H, W, 3)
                ok, pct, mx = rt.compare_rgb(gold[i], got, 0.5)
                assert ok and mx <= 2, (names[i], k, pct, mx)
                assert np.array_equal(got, bufs[i][0][:H * W * 3].cpu().numpy().reshape(H, W, 3))
    finally:
        for r in rs:
            r.close()


def test_upload_waits_for_renders_on_caller_streams(rt, oracle, scenes):
    """rt_upload_scene rebuilds the tables in place: it must wait for renders still running on a caller's stream."""
    import torch
    W, H, D = 640, 360, 5
    gold = {n: oracle.render(scenes[n], W, H, D)["rgb"] for n in ("complex", "medium")}
    with rt.Renderer(0) as r:
        s = torch.cuda.Stream()
        bufs = {n: torch.zeros(H * W * 3 + 16, dtype=torch.uint8, device="cuda:0") for n in gold}
        torch.cuda.synchronize()
        for _ in range(3):
            for n in ("complex", "medium"):
                r.upload(scenes[n])                    # no host sync between the async render and the next upload
                r.render_bands_device(W, H, D, H, 0, 1, bufs[n].data_ptr(), s.cuda_stream)
        torch.cuda.synchronize()
        for n in gold:
            ok, pct, mx = rt.compare_rgb(gold[n], bufs[n][:H * W * 3].cpu().numpy().reshape(H, W, 3), 0.5)
            assert ok and mx <= 2, (n, pct, mx)


@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("name,W,H,D", [("complex", 320, 180, 5), ("complex", 1920, 1080, 5), ("medium", 336, 61, 3), ("simple", 1280, 720, 10),
                                        ("complex", 200, 120, 4), ("medium", 97, 61, 3), ("complex", 64, 6, 2)])
def test_tile_store_path_equals_the_pixel_store_path(rt, oracle, scenes, name, W, H, D, mode):
    """Frames without debug buffers take the production store path: level-0 tiles that contain hits are written once,
    as whole 16-byte row segments, by the shading pass (W % 16 == 0; k_closest0 stores only hit-free tiles), everything
    else pixel by pixel.  rt_render_debug keeps the pixel-by-pixel path, so the two must agree byte for byte -- at
    widths that are and are not multiples of 16, heights that are not multiples of 4, for whole frames and row bands."""
    import torch
    with rt.Renderer(0, mode=mode) as r:
        r.upload(scenes[name])
        dbg = r.render_debug(W, H, D)[0]
        for _ in range(2):
            fast, _ = r.render(W, H, D, want_stats=False)
            assert np.array_equal(dbg, fast)
        with_stats, _ = r.render(W, H, D)
        assert np.array_equal(dbg, with_stats)
        out = np.zeros_like(dbg)
        for rank in range(3):
            rows = rt.band_row_list(H, 8, rank, 3)
            buf = torch.zeros(len(rows) * W * 3 + 16, dtype=torch.uint8, device="cuda:0")
            r.render_bands_device(W, H, D, 8, rank, 3, buf.data_ptr(), None, want_stats=True)
            out[rows] = buf[:len(rows) * W * 3].cpu().numpy().reshape(len(rows), W, 3)
        assert np.array_equal(dbg, out)
        frame = torch.zeros((H, W, 3), dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        for rank in range(2):
            r.render_bands_frame(W, H, D, 16, rank, 2, frame.data_ptr(), None, want_stats=True)
        assert np.array_equal(dbg, frame.cpu().numpy())
    ok, pct, mx = rt.compare_rgb(oracle.render(scenes[name], W, H, D)["rgb"], dbg, 0.5)
    assert ok and mx <= 2


@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("nl", [32, 33, 40])
def test_many_lights(rt, oracle, renderers, scenes, nl, mode):
    """Up to 32 lights the occlusion bits of a hit travel in its record; above that in per-light byte arrays: both sides
    of the switch, hit indices / shadow masks (first 32 lights) / counters against the oracle."""
    g = np.random.default_rng(nl)
    sc = scenes["medium"]
    lights = np.column_stack([g.uniform(-15, 15, nl), g.uniform(2, 14, nl), g.uniform(-25, 8, nl), g.uniform(0.05, 0.2, (nl, 3)), np.ones(nl)])
    check(rt, oracle, renderers[mode], rt.Scene(sc.spheres, lights, sc.ambient, sc.camera), 96, 54, 3)


def test_candidates_pending_at_the_cutoff_are_walked(rt, oracle):
    """Regression (scripts/fuzz_parity.py, large scenes): the bundle-culled camera walk fills its per-warp table, walks it,
    collects a further round with <= 32 survivors and THEN reaches the distance cut-off -- the survivors of that last
    round must still be walked (one of them was the closest sphere of a pixel; the walk used to leave the loop first).
    1705 spheres with wide pixel cones (45 x 57 pixels) through the table path."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import gen_scene
    sc = rt.Scene(*gen_scene.generate(1705, 92992, 0.05, 1.4764311835476813))
    with rt.Renderer(0, accel=1) as r:
        check(rt, oracle, r, sc, 45, 57, 6)


@pytest.mark.parametrize("mode", ["fast", "bvh"])
@pytest.mark.parametrize("seed,W,H,D", [(83424, 224, 176, 1), (5, 96, 54, 4), (11, 130, 40, 3)])
def test_every_store_path_gives_the_same_pixels(rt, renderers, seed, W, H, D, mode):
    """rt_render (whole tiles stored by the shading pass) and rt_render_debug (pixel by pixel) run different inlined copies
    of the same colour code; the arithmetic is written with explicit intrinsics (phong_light, add_scaled, sky_colour) so that
    no copy is contracted into FMAs differently from another (seed 83424 once differed by one LSB in one pixel)."""
    r = renderers[mode]
    r.upload(_random_scene(rt, seed))
    plain = r.render(W, H, D)[0]
    dbg = r.render_debug(W, H, D)[0]
    assert np.array_equal(plain, dbg)
