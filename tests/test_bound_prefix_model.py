"""The constant T of the bound-only prefix scorer (make_hyp32, csrc/f_kernels.cuh; DESIGN.md section 4.2) against a
float32 model of the scorer: whenever the guarded scorer's q^ lies at or below its band G — which every reference inlier
does — the bound scorer's r^ (the same FP32 operations) has r^2 < T, and so does every reference inlier directly.  Points
are drawn at the corners of the frame and on both sides of the threshold, in frames over many decades."""
import os
import sys

import numpy as np
from hypothesis import given, settings, strategies as st

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from bounded_sweep_model import bounded_rule, prefix_points  # noqa: E402

EPS = 2.0 ** -24


def _fma32(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def _up32(x):
    """round a float64 up to float32 (__double2float_ru)"""
    f = np.float32(x)
    return f if float(f) >= x else np.nextafter(f, np.float32(np.inf))


def _hyp32(F, c1, c2, thr, B, mode):
    """numpy transcription of make_hyp32: FP32 coefficients f, g, band G and bound constant T"""
    M1 = np.array([[thr, 0, c1[0]], [0, thr, c1[1]], [0, 0, 1.0]])
    M2 = np.array([[thr, 0, c2[0]], [0, thr, c2[1]], [0, 0, 1.0]])
    Ft = M1.T @ F @ M2
    w = np.array([B, B, 1.0])
    Ft = Ft / np.sum(np.abs(Ft) * np.outer(w, w))
    f = Ft.ravel()
    hh = np.hypot(f[0], f[1])
    g = np.array([hh, (f[0] * f[3] + f[1] * f[4]) / hh, (f[0] * f[6] + f[1] * f[7]) / hh,
                  (f[0] * f[4] - f[1] * f[3]) / hh, (f[0] * f[7] - f[1] * f[6]) / hh])
    a = np.abs(f)
    rho0, rho1 = a[0] * B + a[1] * B + a[2], a[3] * B + a[4] * B + a[5]
    kap0, kap1 = abs(g[0]) * B + abs(g[1]) * B + abs(g[2]), abs(g[3]) * B + abs(g[4])
    S1, S2 = rho0 ** 2 + rho1 ** 2, kap0 ** 2 + kap1 ** 2
    if mode == 1:
        Mb, Smax = S1 + S2, 1.1 * (S1 + S2)
    else:
        Mb, Smax = min(S1, S2), max(S1, S2)
    G = _up32(1.25 * 16.0 * EPS * np.sqrt(Mb) + 2.0 * (100.0 * EPS * EPS + 10.0 * EPS * Smax + 2.0 * EPS * Mb))
    T = _up32((1.0 + 2.0 ** -16) * Mb + (1.0 + 2.0 ** -20) * float(G) + 2.0 ** -126)
    return f.astype(np.float32), g.astype(np.float32), float(G), float(T)


def _scorer32(f, g, x0, x1, y0, y1, mode):
    """the FP32 op sequence of EpiPolicy::evalN / epi_q32 (r is also EpiBoundPolicy's)"""
    bc = lambda v: np.full_like(x0, v)
    l1x = _fma32(bc(f[0]), y0, _fma32(bc(f[1]), y1, bc(f[2])))
    l1y = _fma32(bc(f[3]), y0, _fma32(bc(f[4]), y1, bc(f[5])))
    l1z = _fma32(bc(f[6]), y0, _fma32(bc(f[7]), y1, bc(f[8])))
    r = _fma32(l1x, x0, _fma32(l1y, x1, l1z))
    l2x = _fma32(bc(g[0]), x0, _fma32(bc(g[1]), x1, bc(g[2])))
    l2y = _fma32(bc(g[3]), x1, bc(g[4]))
    s1 = _fma32(l1x, l1x, (l1y * l1y).astype(np.float32))
    s2 = _fma32(l2x, l2x, (l2y * l2y).astype(np.float32))
    m = (s1 + s2).astype(np.float32) if mode == 1 else np.minimum(s1, s2)
    return r, _fma32(r, r, -m)


def _reference_inlier(F, p, thr, mode):
    x = np.column_stack([p[:, :2], np.ones(len(p))])
    y = np.column_stack([p[:, 2:], np.ones(len(p))])
    l1, l2 = y @ F.T, x @ F
    r1, r2 = np.sum(l1 * x, axis=1), np.sum(l2 * y, axis=1)
    s1, s2 = l1[:, 0] ** 2 + l1[:, 1] ** 2, l2[:, 0] ** 2 + l2[:, 1] ** 2
    with np.errstate(invalid="ignore", divide="ignore"):
        d = np.sqrt(r1 * r1 / (s1 + s2)) if mode == 1 else np.maximum(np.abs(r1 / np.sqrt(s1)), np.abs(r2 / np.sqrt(s2)))
    return d < thr


@st.composite
def frames(draw):
    seed = draw(st.integers(0, 2 ** 31 - 1))
    rng = np.random.default_rng(seed)
    scale = 10.0 ** draw(st.floats(-4, 5))
    shift = 10.0 ** draw(st.floats(-2, 7)) * draw(st.sampled_from([-1.0, 1.0]))
    thr = scale * 10.0 ** draw(st.floats(-4, 1))
    mode = draw(st.sampled_from([0, 1]))
    return rng, scale, shift, thr, mode


@settings(max_examples=150, deadline=None)
@given(frames())
def test_bound_constant_covers_every_reference_inlier(frame):
    rng, scale, shift, thr, mode = frame
    # a rank-2 F and points near its epipolar lines (on, inside and just outside the threshold) plus random ones
    U, _, Vt = np.linalg.svd(rng.normal(size=(3, 3)))
    F = U @ np.diag([1.0, rng.uniform(0.1, 1.0), 0.0]) @ Vt
    n = 2000
    y = rng.uniform(-1, 1, size=(n, 2)) * scale + shift
    x = rng.uniform(-1, 1, size=(n, 2)) * scale + shift
    l1 = np.column_stack([y, np.ones(n)]) @ F.T                    # line of image 1 through which x should pass
    nrm = np.hypot(l1[:, 0], l1[:, 1])
    foot = x - ((np.sum(l1[:, :2] * x, axis=1) + l1[:, 2]) / nrm ** 2)[:, None] * l1[:, :2]
    off = thr * rng.choice([0.0, 0.5, 0.999999, 1.0, 1.000001, 2.0], size=n) * rng.choice([-1, 1], size=n)
    x[: n // 2] = foot[: n // 2] + (off / nrm)[: n // 2, None] * l1[: n // 2, :2]
    pts = np.column_stack([x, y])
    pts[:4] = [[pts[:, k].min() if (j >> k) & 1 else pts[:, k].max() for k in range(4)] for j in (0, 5, 10, 15)]
    # frame of f_bbox / frame_from_bbox
    lo = np.array([np.nextafter(np.float32(v), np.float32(-np.inf)) if np.float32(v) > v else np.float32(v)
                   for v in pts.min(axis=0)], np.float64)
    hi = np.array([np.nextafter(np.float32(v), np.float32(np.inf)) if np.float32(v) < v else np.float32(v)
                   for v in pts.max(axis=0)], np.float64)
    c = 0.5 * (lo + hi)
    B = np.max(np.maximum(hi - c, c - lo)) / thr * (1 + 1e-6) + 1e-30
    f, g, G, T = _hyp32(F, c[:2], c[2:], thr, B, mode)
    if not (B < 1e12):
        return                                                     # G = T = inf in make_hyp32: nothing to check
    t = ((pts - c) / thr).astype(np.float32)
    r, q = _scorer32(f, g, t[:, 0], t[:, 1], t[:, 2], t[:, 3], mode)
    r2 = r.astype(np.float64) ** 2                                 # exact square of the FP32 r^
    in_band = q.astype(np.float64) <= G
    assert np.all(r2[in_band] < T), "q^ <= G but r^2 >= T"
    inl = _reference_inlier(F, pts, thr, mode)
    assert np.all(in_band[inl]), "guard-band premise"
    assert np.all(r2[inl] < T), "a reference inlier fails the bound"
    # the bound keeps the fma sign test of EpiBoundPolicy: sign(fl(r^2 - T)) is negative exactly when r^2 < T
    qb = _fma32(r, r, np.full_like(r, -np.float32(T)))
    assert np.array_equal(np.signbit(qb) & ~np.isnan(qb), r2 < T)


# ---- the pruning rule with upper-bound prefix counts (tools/bounded_sweep_model.py restates bnd_select / bnd_check) ------
@st.composite
def bound_pairs(draw):
    n = draw(st.integers(8, 400))
    k = prefix_points(n, draw(st.integers(1, 1000)) / 1000.0)
    H = draw(st.integers(1, 80))
    K = draw(st.integers(1, 40))
    rest = n - k
    pre = np.array(draw(st.lists(st.integers(0, k), min_size=H, max_size=H)), np.int64)
    add = np.array(draw(st.lists(st.integers(0, rest), min_size=H, max_size=H)), np.int64)
    if draw(st.booleans()):                       # exact ties with the maximum
        dup = draw(st.lists(st.integers(0, H - 1), max_size=H))
        src = int(np.argmax(pre + add))
        pre[dup], add[dup] = pre[src], add[src]
    bound = pre + np.array([draw(st.integers(0, k - p)) for p in pre], np.int64)      # pre <= bound <= k
    return bound, pre + add, rest, K


@settings(max_examples=400, deadline=None)
@given(bound_pairs())
def test_rule_on_upper_bounds_keeps_winner_and_ties(case):
    bound, full, rest, K = case
    r = bounded_rule(bound, full, rest, K)
    seen = r["counts"]
    top = full.max()
    assert seen.max() == top
    assert np.array_equal(np.flatnonzero(seen == top), np.flatnonzero(full == top))
    assert int(np.argmax(seen)) == int(np.argmax(full))
    if not r["fallback"]:
        assert np.all(seen[~r["cand"]] < top) and np.all(full[~r["cand"]] < top)
