"""Long-running parity fuzz (not part of the test suite): random adversarial scenes vs the oracle, all kernel families.
usage: fuzz_parity.py [first_seed] [count] [big|mid] [--wave-levels]

--wave-levels: the table-mode renders of each seed force rt_set_option wave_levels to one of 1, 2, 3 or 32 (every level a
wavefront), drawn per seed, each value with a context of its own.  Without it the small frames of this fuzz run their
reflection levels >= 1 in the tail kernel only."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts")):
    sys.path.insert(0, p)
import numpy as np
import rtb200, oracle_py
from test_gpu_parity import _random_scene
WAVE = "--wave-levels" in sys.argv
if WAVE:
    sys.argv.remove("--wave-levels")
first, count = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (100, 200)
MID = len(sys.argv) > 3 and sys.argv[3] == "mid"          # 60..300 spheres: tables in shared memory, several fills of a culled walk
BIG = len(sys.argv) > 3 and sys.argv[3] in ("big", "mid") # 300..4000 spheres: streamed tables (accel=1) and the LBVH
if BIG:
    import gen_scene
first0 = first
rs = {"fast": rtb200.Renderer(0, accel=1 if BIG else None), "bvh": rtb200.Renderer(0, mode="bvh")}
WAVE_LEVELS = (1, 2, 3, 32)
rs_wave = {}
for wl in WAVE_LEVELS if WAVE else ():
    rs_wave[wl] = rtb200.Renderer(0, accel=1 if BIG else None)
    rs_wave[wl].set_option("wave_levels", wl)
bad = 0
for seed in range(first, first + count):
    g = np.random.default_rng(seed)
    if BIG:
        sc = rtb200.Scene(*gen_scene.generate(int(g.integers(60, 300) if MID else g.integers(300, 4000)), seed, 0.05, float(g.uniform(0.3, 1.5))))
    else:
        sc = _random_scene(rtb200, seed)
    if BIG:
        W, H, D = int(g.integers(16, 120)), int(g.integers(16, 70)), int(g.integers(1, 7))
    elif seed % 2:
        W, H, D = [(96, 54, 4), (61, 47, 6), (130, 40, 3), (40, 90, 8)][seed % 4]
    else:                                                  # any size (buffers grow and are reused), any depth
        W, H, D = int(g.integers(2, 260)), int(g.integers(2, 200)), int(g.integers(0, 9))
    if not BIG and seed % 3 == 0:                          # similarity transform: scale 1e-2 .. 1e3, offset up to 1e4 scene units
        k = float(10.0 ** g.uniform(-2, 3)); off = g.uniform(-1, 1, 3) * float(10.0 ** g.uniform(0, 4)) * k
        sp = sc.spheres.copy(); sp[:, :3] = sp[:, :3] * k + off; sp[:, 3] *= k
        li = sc.lights.copy(); li[:, :3] = li[:, :3] * k + off
        cm = sc.camera.copy(); cm[:3] = cm[:3] * k + off; cm[3:6] = cm[3:6] * k + off
        sc = rtb200.Scene(sp, li, sc.ambient, cm)
    if not BIG and seed % 7 == 3:                          # many lights: both sides of the 32-light switch of the occlusion bits, several
        nl = int(g.integers(6, 41))                        # rounds of packed shadow queries in the tail kernel
        li = np.column_stack([g.uniform(-8, 8, (nl, 3)) - np.array([0, -4, 6]), g.uniform(0.05, 0.3, (nl, 3)), np.ones(nl)])
        sc = rtb200.Scene(sc.spheres, li, sc.ambient, sc.camera)
    if seed % 37 == 0:
        sc = rtb200.Scene(sc.spheres, sc.lights[:0], sc.ambient, sc.camera)      # no lights
    if seed % 41 == 0:
        sc = rtb200.Scene(sc.spheres[:0], sc.lights, sc.ambient, sc.camera)      # no spheres
    o = oracle_py.render(sc, W, H, D, want_idx=True)
    wl = WAVE_LEVELS[int(np.random.default_rng((seed, 1)).integers(len(WAVE_LEVELS)))] if WAVE else 0   # (own stream: the scene's draws stay as they were)
    for m, r in rs.items():
        if wl and m == "fast":
            r = rs_wave[wl]
        r.upload(sc)
        first = r.render(W, H, D)[0]                       # (the next frame may pick another wavefront / tail split)
        rgb, hit, mask, st = r.render_debug(W, H, D)
        if not np.array_equal(first, rgb):
            bad += 1; print("MISMATCH seed %d mode %s: two renders of one scene differ" % (seed, m))
        if D == 0:
            hit, mask = o["hit_idx"], o["shadow_mask"]     # (no levels: nothing to compare)
        ok_rgb, pct, mx = rtb200.compare_rgb(o["rgb"], rgb, 0.5)
        good = np.array_equal(hit, o["hit_idx"]) and np.array_equal(mask, o["shadow_mask"]) and ok_rgb and mx <= 2 and st.filter_violations == 0 \
            and st.closest_queries == o["counters"]["closest_queries"] and st.occluded == o["counters"]["occluded"]
        if not good:
            bad += 1
            print("MISMATCH seed %d mode %s wave_levels %s: hit %s mask %s rgb %s (%.4f%%, max %d) viol %d" % (
                seed, m, wl or "auto", np.array_equal(hit, o["hit_idx"]), np.array_equal(mask, o["shadow_mask"]), ok_rgb, pct, mx, st.filter_violations))
            badh = np.argwhere(hit != o["hit_idx"]); badm = np.argwhere(mask != o["shadow_mask"])
            print("   N %d L %d %dx%d d%d; hit mismatches by level %s, mask by level %s, counters gpu (%d %d %d %d) oracle %s" % (
                sc.nspheres, sc.nlights, W, H, D, np.bincount(badh[:, 2], minlength=D).tolist() if len(badh) else [],
                np.bincount(badm[:, 2], minlength=D).tolist() if len(badm) else [], st.closest_queries, st.hits, st.shadow_queries, st.occluded,
                {k: o["counters"][k] for k in ("closest_queries", "hits", "shadow_queries", "occluded")}))
            if len(badh):
                j, i, k = badh[0]
                print("   first hit mismatch (row %d col %d level %d): got %d want %d; rows %s" % (j, i, k, hit[j, i, k], o["hit_idx"][j, i, k], sorted(set(badh[:, 0].tolist()))[:16]))
            # is it the scene on the device or the render?  upload again and re-render
            r.upload(sc)
            _, hit2, mask2, _ = r.render_debug(W, H, D)
            print("   after a second upload of the same scene: hit %s mask %s" % (np.array_equal(hit2, o["hit_idx"]), np.array_equal(mask2, o["shadow_mask"])))
    if seed % 10 == 0:                                   # supersampling and the assembled-frame output mode on the same scene
        import torch
        r = (rs_wave[wl] if wl else rs["fast"]) if (seed // 10) % 2 == 0 else rs["bvh"]
        r.upload(sc)
        plain, _ = r.render(W, H, D)
        fr = torch.zeros((H, W, 3), dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        for rank in range(3):
            r.render_bands_frame(W, H, D, 8, rank, 3, fr.data_ptr())
        torch.cuda.synchronize()
        if not np.array_equal(fr.cpu().numpy(), plain):
            bad += 1; print("MISMATCH seed %d: assembled frame != rt_render" % seed)
        if W > 8 and H > 8:                              # a random tile against the whole-frame tile render
            whole = torch.full((H, W, 3), -1.0, dtype=torch.float32, device="cuda:0")
            part = torch.full((H, W, 3), -1.0, dtype=torch.float32, device="cuda:0")
            torch.cuda.synchronize()
            tx, ty = int(g.integers(0, W - 4)), int(g.integers(0, H - 4))
            tw, th = int(g.integers(1, W - tx + 1)), int(g.integers(1, H - ty + 1))
            r.render_tile_device(W, H, D, (0, 0, W, H), whole.data_ptr())
            r.render_tile_device(W, H, D, (tx, ty, tw, th), part.data_ptr())
            torch.cuda.synchronize()
            inside = torch.zeros((H, W), dtype=torch.bool, device="cuda:0"); inside[ty:ty + th, tx:tx + tw] = True
            if not torch.equal(part[inside], whole[inside]) or not bool((part[~inside] == -1.0).all()) or bool((whole == -1.0).any()):
                bad += 1; print("MISMATCH seed %d: tile render (%d,%d,%d,%d) of %dx%d d%d" % (seed, tx, ty, tw, th, W, H, D))
        osamp = oracle_py.render_supersampled(sc, W, H, D)
        r.set_option("antialias", 1)
        rgb, hit, mask, st = r.render_debug(W, H, D)
        r.set_option("antialias", 0)
        okk = D == 0 or all(np.array_equal(hit[b::2, a::2], osamp["samples"][k]["hit_idx"]) for k, (a, b) in enumerate(((0, 0), (1, 0), (0, 1), (1, 1))))
        ok_rgb, pct, mx = rtb200.compare_rgb(osamp["rgb"], rgb, 0.5)
        if not (okk and ok_rgb and mx <= 2):
            bad += 1; print("MISMATCH seed %d: supersampling hit %s rgb %s max %d" % (seed, okk, ok_rgb, mx))
    if (seed - first0 + 1) % 100 == 0:
        print("... %d scenes so far, %d mismatches" % (seed - first0 + 1, bad), flush=True)
print("fuzz: %d scenes x %d modes%s, %d mismatches" % (count, len(rs), " (tables at wave_levels 1/2/3/32)" if WAVE else "", bad))
sys.exit(1 if bad else 0)
