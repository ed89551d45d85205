"""The corner refinement's CPU oracle (oracle/a3ref_refine.c, the specification kernel K5 is held to bit for bit):
accuracy against the synthetic renderer's ground truth, agreement with an f64 restatement of the algorithm, and the
fallback rules.  CPU only."""
import numpy as np
import pytest

SETS = [("C1", 8), ("C3", 3), ("C3n", 2), ("C5", 1)]
CLEAN_BARS = dict(mean=0.25, p95=0.5, max=1.5)
NOISY_BARS = dict(mean=0.35, p95=0.75, max=None)

# k5_refine_spec.h
PASSES, SAMPLES, T0, TSPAN, RANGE, STEP, FLOOR = 2, 16, 0.12, 0.76, 3.0, 0.25, 0.3
REJECT_MIN, REJECT_MEDIANS, MIN_KEPT, MIN_CROSS, MAX_MOVE = 1.0, 2.5, 4, 1e-3, 0.25


@pytest.fixture(scope="module")
def rr():
    from oracle import a3ref_refine_py
    a3ref_refine_py.lib()
    return a3ref_refine_py


def oracle_markers(oracle, name, n):
    """-> [(grey, oracle markers, truth markers)] for the first n frames of workload `name`"""
    from aruco3_b200 import synth
    spec = synth.CONFIGS[name]
    cfg = oracle.default_config(min_corner_separation_factor=spec.min_corner_separation_factor)
    out = []
    for f in range(n):
        img, truth = synth.render_frame(spec, f)
        res = oracle.detect(img, spec.dictionary, cfg)
        out.append((res.grey, res.markers, truth))
    return out


def errors_against_truth(pairs):
    """pairs of (integer corners [4,2], refined corners [4,2], truth markers of the frame) -> per-corner distances to the
    truth in the pixel-centre convention (synth's corners - 0.5), markers matched to the truth by nearest centre"""
    e_int, e_ref = [], []
    for ci, cr, truth in pairs:
        t = min(truth, key=lambda t: np.linalg.norm(t.corners.mean(0) - 0.5 - ci.mean(0)))
        tr = t.corners - 0.5
        assert np.linalg.norm(tr.mean(0) - ci.mean(0)) < 5
        e_int.append(np.linalg.norm(ci - tr, axis=1))
        e_ref.append(np.linalg.norm(cr - tr, axis=1))
    return np.concatenate(e_int), np.concatenate(e_ref)


# ---- f64 restatement of the algorithm (DESIGN.md §4, K5), for the cross-check ----------------------------------------
def _bilinear64(g, x, y):
    h, w = g.shape
    x0, y0 = np.floor(x), np.floor(y)
    inside = bool(np.all((x0 >= 0) & (x0 + 1 < w) & (y0 >= 0) & (y0 + 1 < h)))
    if not inside:
        return None, False
    ix, iy = x0.astype(int), y0.astype(int)
    fx, fy = x - x0, y - y0
    a, b, c, d = g[iy, ix], g[iy, ix + 1], g[iy + 1, ix], g[iy + 1, ix + 1]
    return (a * (1 - fx) + b * fx) * (1 - fy) + (c * (1 - fx) + d * fx) * fy, True


def _fit64(q, wt):
    S = wt.sum()
    if not S > 0:
        return None
    m = (wt[:, None] * q).sum(0) / S
    t = q - m
    a, b, c = (wt * t[:, 0] ** 2).sum(), (wt * t[:, 0] * t[:, 1]).sum(), (wt * t[:, 1] ** 2).sum()
    lam = (a + c) / 2 + np.sqrt(((a - c) / 2) ** 2 + b * b)
    v1, v2 = np.array([b, lam - a]), np.array([lam - c, b])
    v = v1 if v1 @ v1 >= v2 @ v2 else v2
    if not v @ v > 0:
        return None
    return m, v / np.sqrt(v @ v)


def _edge64(g, c, k, near):
    p, q = c[k], c[(k + 1) % 4]
    e = q - p
    d = e / np.linalg.norm(e)
    n = np.array([d[1], -d[0]])
    s = -RANGE + STEP * np.arange(25)
    pts, wts = np.zeros((SAMPLES, 2)), np.zeros(SAMPLES)
    for i in range(SAMPLES):
        base = p + (T0 + TSPAN * (i + 0.5) / SAMPLES) * e
        v, inside = _bilinear64(g, base[0] + s * n[0], base[1] + s * n[1])
        if not inside:
            continue
        gr = v[2:] - v[:-2]
        w = np.maximum(gr - FLOOR * gr.max(), 0)
        if w.sum() > 0:
            pts[i], wts[i] = base + (w @ s[1:-1] / w.sum()) * n, w.sum()
    L1 = _fit64(pts, wts)
    if L1 is None:
        return None
    m, dv = L1
    dist = np.abs((pts[:, 0] - m[0]) * dv[1] - (pts[:, 1] - m[1]) * dv[0])
    valid = wts > 0
    lim = max(REJECT_MIN, REJECT_MEDIANS * np.sort(dist[valid])[(valid.sum() - 1) // 2])
    near[0] |= bool(np.any(np.abs(dist[valid] - lim) < 1e-3))  # a sample f32 may keep or drop the other way
    keep = valid & (dist <= lim)
    if keep.sum() < MIN_KEPT:
        return None
    return _fit64(pts, np.where(keep, wts, 0))


def refine64(grey, corners):
    """-> (refined [4,2] f64, ok, near a rejection threshold)"""
    g = grey.astype(np.float64)
    c0 = np.asarray(corners, np.float64).reshape(4, 2)
    lens = np.linalg.norm(np.roll(c0, -1, 0) - c0, axis=1)
    cur, near = c0.copy(), [False]
    if not lens.min() > 0:
        return c0, False, False
    for _ in range(PASSES):
        lines = [_edge64(g, cur, k, near) for k in range(4)]
        if any(L is None for L in lines):
            return c0, False, near[0]
        nxt = np.zeros((4, 2))
        for k in range(4):
            (m1, d1), (m2, d2) = lines[(k - 1) % 4], lines[k]
            cr = d1[0] * d2[1] - d1[1] * d2[0]
            if not abs(cr) >= MIN_CROSS:
                return c0, False, near[0]
            u = m2 - m1
            nxt[k] = m1 + (u[0] * d2[1] - u[1] * d2[0]) / cr * d1
        e = np.roll(nxt, -1, 0) - nxt
        turns = e[:, 0] * np.roll(e, -1, 0)[:, 1] - e[:, 1] * np.roll(e, -1, 0)[:, 0]
        if not (np.all(np.isfinite(nxt)) and np.all(turns > 0) and np.all(np.linalg.norm(nxt - c0, axis=1) <= MAX_MOVE * lens.min())):
            return c0, False, near[0]
        cur = nxt
    return cur, True, near[0]


# ---- tests ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,n", SETS)
def test_accuracy_against_ground_truth(oracle, rr, name, n):
    pairs, fallbacks = [], 0
    for grey, markers, truth in oracle_markers(oracle, name, n):
        for m in markers:
            r, ok = rr.refine_corners(grey, m["corners"])
            fallbacks += not ok
            pairs.append((np.array(m["corners"], np.float64).reshape(4, 2), r.astype(np.float64), truth))
    e_int, e_ref = errors_against_truth(pairs)
    bars = NOISY_BARS if name.endswith("n") else CLEAN_BARS
    stats = dict(markers=len(pairs), fallbacks=fallbacks, mean=e_ref.mean(), p95=np.percentile(e_ref, 95), max=e_ref.max(), int_mean=e_int.mean())
    print(name, stats)
    assert stats["mean"] <= bars["mean"] and stats["p95"] <= bars["p95"], stats
    if bars["max"] is not None:
        assert stats["max"] <= bars["max"], stats
    assert stats["mean"] < stats["int_mean"] / 4, stats


def test_f32_oracle_agrees_with_f64(oracle, rr):
    compared, excluded, worst = 0, 0, 0.0
    for name, n in SETS:
        for grey, markers, _ in oracle_markers(oracle, name, n):
            for m in markers:
                r32, ok32 = rr.refine_corners(grey, m["corners"])
                r64, ok64, near = refine64(grey, m["corners"])
                if not (ok32 and ok64) or near:
                    excluded += 4
                    continue
                compared += 4
                worst = max(worst, float(np.abs(r32.astype(np.float64) - r64).max()))
    print(f"f32 vs f64: {compared} corners compared, {excluded} excluded (a fallback, or a sample at a rejection threshold), "
          f"largest difference {worst:.2e} px")
    assert compared > 1000 and worst <= 0.05


def _square_scene(w=120, h=100, x0=30.0, y0=25.0, side=50.0):
    """white background, black axis-aligned square covering [x0, x0+side) x [y0, y0+side) in pixel-edge coordinates"""
    g = np.full((h, w), 220, np.uint8)
    g[int(y0):int(y0 + side), int(x0):int(x0 + side)] = 20
    return g


def test_clean_square_is_refined_to_its_edges(rr):
    g = _square_scene()
    # integer corners one pixel outside the black square (the white pixels a contour follows)
    r, ok = rr.refine_corners(g, [(29, 24), (80, 24), (80, 75), (29, 75)])
    assert ok
    # the edges lie between pixels 29|30 and 79|80: pixel-centre coordinates 29.5 and 79.5
    np.testing.assert_allclose(r, [(29.5, 24.5), (79.5, 24.5), (79.5, 74.5), (29.5, 74.5)], atol=0.02)


def test_fallback_degenerate_quad(rr):
    g = _square_scene()
    for quad in ([(40, 40)] * 4, [(10, 10), (50, 10), (90, 10), (50, 10)], [(29, 24), (29, 75), (80, 75), (80, 24)]):
        r, ok = rr.refine_corners(g, quad)
        assert not ok and np.array_equal(r, np.asarray(quad, np.float32)), quad  # collinear, and counter-clockwise


def test_fallback_marker_cut_by_the_border(rr):
    g = np.full((100, 120), 220, np.uint8)
    g[25:75, 0:50] = 20  # the square's left edge is the image border: no profile across it fits inside
    quad = [(0, 24), (50, 24), (50, 75), (0, 75)]
    r, ok = rr.refine_corners(g, quad)
    assert not ok and np.array_equal(r, np.asarray(quad, np.float32))


def test_fallback_blank_patch(rr):
    g = np.full((100, 120), 128, np.uint8)
    quad = [(29, 24), (80, 24), (80, 75), (29, 75)]
    r, ok = rr.refine_corners(g, quad)
    assert not ok and np.array_equal(r, np.asarray(quad, np.float32))


def test_pose_entries_on_integer_corners_match_the_u32_entries(oracle, rr):
    corners = [(90, 89), (95, 150), (80, 170), (75, 90)]
    for got, want in ((rr.solve_with_undistorted_points_f32(np.array(corners, np.float32), 17.0, (1000, 1000)),
                       oracle.solve_with_undistorted_points(corners, 17.0, (1000, 1000))),
                      (rr.solve_with_intrinsics_f32(np.array(corners, np.float32), 17.0, oracle.intrinsics_new(1000, 1000, 800.0, 800.0)),
                       oracle.solve_with_intrinsics(corners, 17.0, oracle.intrinsics_new(1000, 1000, 800.0, 800.0)))):
        for p, q in zip(got, want):
            assert bytes(p) == bytes(q)
