"""A per-pixel, per-channel bound on |fb_gpu - fb_oracle|: how far the FP32 colour of the fast path may lie from the FP64
colour of the serial renderer (oracle/rt_oracle.c) when both trace the same rays.

The device decides every hit and every shadow boolean exactly as the oracle does (tests/test_gpu_parity.py pins them bit
for bit), and forms the hit point, the reflected rays and every ray direction in FP64 in the oracle's operation order.
What it evaluates in FP32 is the colour: the sky (sky_colour), the Phong terms of each un-occluded light (phong_light),
the ambient term, and the blend of the reflection levels (add_scaled and the weight products of k_shade / k_bounce /
k_closest1), all in kernels_fast.cuh / kernels_wave.cuh.  So the only difference is FP32 arithmetic, and it is bounded
here term by term, in the form

    |fb_gpu - fb_oracle|  <=  sum over levels k of |w_k| eps_k  (+ the rounding of the running sum and of the weights)

where w_k = r_0 r_1 ... r_{k-1} is the FP64 weight product reaching level k (the oracle blends only where the
reflectivity is > 0, rt_oracle.c:169, and so does the device, with the flag decided in double) and eps_k bounds the FP32
error of level k's own term: the sky, or ambient + the sum over lights of diffuse + specular.

The geometry the bound needs (hit points, normals, light and view directions, r.v, the sky direction) is recomputed here
in numpy FP64 from the oracle's own per-level hit_idx and shadow_mask: the sphere of each level is given, so no search is
needed.  It only feeds the bound's sensitivities, each evaluated over the whole error interval, so its own FP64 rounding
does not matter.

Constants (u = 2^-24, the unit roundoff of round-to-nearest FP32; "ulp" of a value in [1, 2) is 2u):
* FP32 inputs: every material value (colour, reflectivity, shininess), light colour and the ambient is rounded once to
  FP32 on the host (rt_api.cu upload_scene, k_build_lookup): relative error u (plus 2^-150 absolute below the normal range).
* Unit vectors normalised in FP32 -- the normal (hit_geometry: FP64 p - c, then FP32), the light direction of
  phong_light (FP64 light - p, then FP32) and the level-0 camera direction of the sky (camera_dir: FP64, then FP32):
  component rounding u, sum of squares (one multiply, two FMAs, positive terms) 3u -> 1.5u after the square root,
  rsqrtf 2 ulp = 4u, the product w * inv u, and the norm of the rounded vector u: 8.5u relative per component.  DESIGN
  section 4 quotes the normal as 2-3 ulp; 8.5u is the worst case of every rounding above added up.  The oracle's own
  FP64 normalisation adds 2^-50 absolute.
* The view direction is -(float)d of the exact FP64 ray direction (u per component); the oracle normalises o - p instead,
  which differs from -d by the FP64 rounding of o - p relative to its length t: 2^-51 (1 + (|o| + |p|) / t).
* Dot products (n.l, r.v: one multiply, two FMAs): first-order error propagation of the inputs plus 3u sum |a_i b_i|.
  reflect(-l, n) = fma(2 n.l, n_i, -l_i): the propagated errors plus u |r_i|.
* __powf(x, s) = ex2.approx(s * lg2.approx(x)).  lg2.approx has an absolute error of 2^-22 for x in [0.5, 2] and 2 ulp
  (4u relative) elsewhere, the product s * log2 x rounds (u), ex2.approx is 2 ulp (4u relative).  So relative to x^s the
  intrinsic error is exp(ln2 s 2^-22) (1 + 4u) - 1 near x = 1 -- it grows with the shininess -- plus the terms
  proportional to s |log2 x| x^s <= 1 / (e ln 2) elsewhere: 5u / e absolute.  The input error delta of x = max(0, r.v)
  propagates as s max(x)^(s-1) delta for s >= 1; for 0 < s < 1, x^s is not Lipschitz at 0, and |a^s - b^s| <= |a - b|^s
  gives delta^s (or s min(x)^(s-1) delta where smaller).  Shininess rounded to FP32 adds u s |ln x| x^s <= u / e.
  Shininess 0 is 1 exactly on both sides.
* (1 - r) with r rounded to FP32 (m.w), the weights fl(wt * r) and fl(wt * (1 - r)): every product of two inexact
  factors is bounded by (|x| + dx)(|y| + dy)(1 + u) - |x||y| (mul_err).
* Every FP32 add or FMA that accumulates (the light sum of phong_light, add_scaled) rounds by u times the magnitude of
  its result, bounded by the running sum of the magnitudes of the terms plus their errors.
* The sky (sky_colour): dy = the FP32 direction's y (level 0: 8.5u |dy|; levels >= 1: (float)dy, u |dy|),
  ts = 0.5 (dy + 1) (u ts), w = 1 - ts (u w), r = fma(0.5, ts, w), g = fma(0.7f, ts, w) with |0.7f - 0.7| = 1.2e-8,
  b = w + ts (u each).
The sum is multiplied by (1 + 2^-20) for the second-order terms the first-order propagation leaves out.

Lights from the 33rd on have no bit in the oracle's shadow mask; they are bounded as if lit (an occluded light adds no
error on either side).  Negative shininess, and a nonzero shininess that rounds to FP32 zero, are outside the bound.
"""
import math

import numpy as np

U = 2.0 ** -24
SUB = 2.0 ** -150               # absolute rounding error below the FP32 normal range (half the smallest subnormal)
E_UNIT = 8.5 * U                # FP32-normalised unit vector, relative per component
E_FP64 = 2.0 ** -50             # the oracle's own FP64 normalisation, absolute per component
SECOND_ORDER = 1.0 + 2.0 ** -20


def mul_err(x, dx, y, dy):
    """Bound on |fl32(x' y') - x y| for |x' - x| <= dx, |y' - y| <= dy."""
    ax, ay = np.abs(x), np.abs(y)
    return (ax + dx) * (ay + dy) * (1.0 + U) - ax * ay + SUB


def _unit(v):
    return v / np.sqrt((v * v).sum(axis=-1, keepdims=True))


def camera_rays(cam, W, H):
    """oracle camera_get_ray for every pixel, row 0 = bottom: (origin [H*W, 3], unit direction [H*W, 3])."""
    pos, look, fov = cam[:3], cam[3:6], cam[6]
    fwd = _unit(look - pos)
    right = _unit(np.cross(fwd, np.array([0.0, 1.0, 0.0])))
    up = _unit(np.cross(right, fwd))
    s = math.tan(fov * 0.5 * math.pi / 180.0)
    uu = (np.arange(W) / (W - 1) - 0.5) * s
    vv = (np.arange(H) / (H - 1) - 0.5) * s
    d = fwd + right * uu[None, :, None] + up * vv[:, None, None]
    d = _unit(_unit(d)).reshape(-1, 3)
    return np.broadcast_to(pos, d.shape).copy(), d


def sky(dy, e_dy):
    """The sky colour (src/main.cpp:26-30) of direction y component dy, and the bound on sky_colour's FP32 error."""
    ts = 0.5 * (dy + 1.0)
    w = 1.0 - ts
    col = np.stack([w + 0.5 * ts, w + 0.7 * ts, w + ts], axis=-1)
    e_ts = 0.5 * e_dy + U * np.abs(ts)
    e_w = e_ts + U * np.abs(w)
    err = np.stack([0.5 * e_ts + e_w + U * np.abs(col[:, 0]),
                    0.7 * e_ts + 1.2e-8 * np.abs(ts) + e_w + U * np.abs(col[:, 1]),
                    e_ts + e_w + U * np.abs(col[:, 2])], axis=-1)
    return col, err


def _dot_err(a, ea, b, eb):
    """Bound on the FP32 dot product (multiply, two FMAs) of inputs within ea / eb (componentwise) of a / b."""
    return (ea * np.abs(b)).sum(-1) + (eb * np.abs(a)).sum(-1) + (ea * eb).sum(-1) + 3 * U * (np.abs(a * b) + ea * eb).sum(-1)


def pow_err(x, ex, s):
    """Bound on |__powf(x', fl32(s)) - x^s| for |x' - x| <= ex, x >= 0, s >= 0 (scalar)."""
    if s == 0.0:
        return np.zeros_like(x)
    if np.float32(s) == 0.0 or s < 0:
        raise ValueError("shininess %r is outside the colour bound" % s)
    xh, xl = x + ex, np.maximum(0.0, x - ex)
    ph = xh ** s
    if s >= 1.0:
        e_in = s * xh ** (s - 1.0) * ex
    else:
        with np.errstate(divide="ignore"):
            lip = np.where(xl > 0, s * np.where(xl > 0, xl, 1.0) ** (s - 1.0) * ex, np.inf)
        e_in = np.minimum(ex ** s, lip)
    e_exp = U * (1.0 / math.e + s * ex * ph)                       # shininess rounded to FP32
    e_intr = ph * (math.exp(math.log(2.0) * s * 2.0 ** -22) * (1.0 + 4 * U) - 1.0) + 5 * U / math.e + 2.0 ** -126
    return e_in + e_exp + e_intr


def shade(sc, idx, o, d, t, mask):
    """Level term of the hits idx (rays o + t d): the FP64 colour S [m, 3], the bound on its FP32 error, per-sphere
    1 - r and its error.  mask: the oracle's shadow bits (light l < 32 occluded)."""
    sp = sc.spheres[idx]
    c, C, r, s = sp[:, 0:3], sp[:, 4:7], sp[:, 7], sp[:, 9]
    p = o + d * t[:, None]
    n = _unit(p - c)
    e_n = E_UNIT * np.abs(n) + E_FP64
    v = -d
    on = np.abs(o).sum(-1) + np.abs(p).sum(-1)
    e_v = U * np.abs(d) + 2.0 ** -51 * (1.0 + on / np.maximum(t, 1e-300))[:, None]
    e_r = np.where(np.abs(r) >= 2.0 ** -126, U * np.abs(r), SUB)
    a = 1.0 - r
    e_a = e_r + U * (np.abs(a) + e_r) + 2.0 ** -52 * np.abs(a)
    A = sc.ambient[None, :]
    S = A * C
    eS = mul_err(A, U * np.abs(A), C, U * np.abs(C) + SUB)
    mag = np.abs(S) + eS                                              # bound on the running |sum| of phong_light
    for l in range(sc.nlights):
        lit = ((mask >> np.uint32(l)) & 1) == 0 if l < 32 else np.ones(len(idx), bool)
        if not lit.any():
            continue
        lp, Lc = sc.lights[l, 0:3], sc.lights[l, 3:6]
        ld = _unit(lp - p)
        e_l = E_UNIT * np.abs(ld) + E_FP64
        nl = (n * ld).sum(-1)
        e_nl = _dot_err(n, e_n, ld, e_l)
        nd = np.maximum(0.0, nl)
        e_kd = mul_err(a, e_a, nd, e_nl)
        diff = C * (a * nd)[:, None]
        e_diff = mul_err(C, U * np.abs(C) + SUB, (a * nd)[:, None], e_kd[:, None])
        rf = 2.0 * nl[:, None] * n - ld
        e_rf = 2 * (np.abs(n) + e_n) * e_nl[:, None] + 2 * np.abs(nl)[:, None] * e_n + e_l
        e_rf = e_rf + U * (np.abs(rf) + e_rf)
        x = np.maximum(0.0, (rf * v).sum(-1))
        e_x = _dot_err(rf, e_rf, v, e_v)
        P = np.empty_like(x)
        eP = np.empty_like(x)
        for sv in np.unique(s[lit]):
            sel = lit & (s == sv)
            P[sel] = 1.0 if sv == 0 else x[sel] ** sv
            eP[sel] = pow_err(x[sel], e_x[sel], float(sv))
        spec = (0.5 * P)[:, None] * Lc[None, :]
        e_spec = 0.5 * (np.abs(Lc) * (1 + U))[None, :] * eP[:, None] + 0.5 * U * np.abs(Lc)[None, :] * P[:, None] + SUB
        T = spec + diff
        eT = e_spec + e_diff
        eT = eT + U * (np.abs(T) + eT)                                # the FMA
        mag = mag + np.abs(T) + eT
        S = S + np.where(lit[:, None], T, 0.0)
        eS = eS + np.where(lit[:, None], eT + U * mag, 0.0)         # the add into (sr, sg, sb)
    return S, eS, r, a, e_r, e_a


def _intersect(sp, o, d):
    """include/sphere.h:26-59 for the given sphere of each ray: t (the hit is known to exist)."""
    oc = o - sp[:, 0:3]
    a = (d * d).sum(-1)
    b = 2.0 * (oc * d).sum(-1)
    cc = (oc * oc).sum(-1) - sp[:, 3] ** 2
    disc = np.maximum(b * b - 4 * a * cc, 0.0)
    t1 = (-b - np.sqrt(disc)) / (2 * a)
    t2 = (-b + np.sqrt(disc)) / (2 * a)
    t = np.minimum(t1, t2)
    return np.where(t < 0, np.maximum(t1, t2), t)


def colour_bound(scene, hit_idx, W, H, D, shadow_mask=None, colour=False):
    """Bound [H, W, 3] on |fb_gpu - fb_oracle| of a render of `scene` at W x H, depth D, from the oracle's hit_idx
    [H, W, D] (and shadow_mask; None = every light lit).  colour=True also returns this module's own FP64 colour (a
    check that it traced the same paths as the oracle)."""
    P = W * H
    hit = np.asarray(hit_idx).reshape(P, -1)
    msk = np.zeros_like(hit, dtype=np.uint32) if shadow_mask is None else np.asarray(shadow_mask).reshape(P, -1)
    o, d = camera_rays(scene.camera, W, H)
    wt, ewt = np.ones(P), np.zeros(P)
    bound, mag, col = np.zeros((P, 3)), np.zeros((P, 3)), np.zeros((P, 3))
    active = np.ones(P, bool) if D > 0 else np.zeros(P, bool)
    for k in range(D):
        if not active.any():
            break
        idx = hit[:, k]
        miss = active & (idx == -1)
        if miss.any():
            dy = d[miss, 1]
            e_dy = (E_UNIT if k == 0 else U) * np.abs(dy) + E_FP64
            skc, e_sky = sky(dy, e_dy)
            w, ew = wt[miss, None], ewt[miss, None]
            term, e_term = w * skc, (np.abs(w) + ew) * (np.abs(skc) + e_sky) - np.abs(w) * np.abs(skc)
            mag[miss] += np.abs(term) + e_term
            bound[miss] += e_term + U * mag[miss]
            col[miss] += term
        hs = active & (idx >= 0)
        active = hs.copy()
        if not hs.any():
            break
        ii = idx[hs]
        t = _intersect(scene.spheres[ii], o[hs], d[hs])
        S, eS, r, a, e_r, e_a = shade(scene, ii, o[hs], d[hs], t, msk[hs, k])
        w, ew = wt[hs], ewt[hs]
        refl = r > 0
        f = np.where(refl, a, 1.0)
        kk = w * f
        ek = np.where(refl, mul_err(w, ew, a, e_a), ew)
        term = kk[:, None] * S
        e_term = (np.abs(kk) + ek)[:, None] * (np.abs(S) + eS) - np.abs(kk)[:, None] * np.abs(S)
        mag[hs] += np.abs(term) + e_term
        bound[hs] += e_term + U * mag[hs]
        col[hs] += term
        # the path continues where the reflectivity is > 0 and depth is left (a reflective hit at the last level: black)
        cont = refl & (k + 1 < D)
        wt[hs], ewt[hs] = np.where(refl, w * r, w), np.where(refl, mul_err(w, ew, r, e_r), ew)
        p = o[hs] + d[hs] * t[:, None]
        n = _unit(p - scene.spheres[ii, 0:3])
        no = p + n * 1e-3
        nd = _unit(d[hs] - n * 2.0 * (d[hs] * n).sum(-1, keepdims=True))
        oh, dh = o[hs], d[hs]
        oh[cont], dh[cont] = no[cont], nd[cont]
        o[hs], d[hs] = oh, dh
        act = active[hs]
        act &= cont
        active[hs] = act
    out = (bound * SECOND_ORDER).reshape(H, W, 3)
    return (out, col.reshape(H, W, 3)) if colour else out
