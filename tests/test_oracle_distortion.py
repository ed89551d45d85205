"""CPU oracle of the corner undistortion (kernel K7, oracle/a3ref_distort.c): agreement with OpenCV's undistortPointsIter
and projectPoints, the fold and non-finite failure rules, exact board recovery through a lens, and the pose accuracy on
rendered frames seen through a distorting lens (with the model, without it, and through a pinhole).
"""
import functools

import numpy as np
import pytest

from aruco3_b200 import synth
from aruco3_b200.board import Board

W, H = 1280, 720
KP = (900.0, 900.0, 640.0, 360.0)  # the webcam-class example: fx = 900 on 1280 x 720
BARREL = (-0.28, 0.09, 0.0, 0.0, 0.0)
CAMERAS = {  # (fx, fy, cx, cy), (k1, k2, p1, p2, k3)
    "barrel": (KP, BARREL),
    "pincushion": ((1000.0, 1005.0, 650.0, 355.0), (0.18, 0.03, 0.0, 0.0, 0.0)),
    "tangential": ((880.0, 880.0, 630.0, 370.0), (0.0, 0.0, 0.004, -0.003, 0.0)),
    "k3_heavy": ((950.0, 950.0, 640.0, 360.0), (-0.12, 0.05, 0.001, 0.0005, -0.06)),
}


@pytest.fixture(scope="module")
def od():
    from oracle import a3ref_distort_py
    a3ref_distort_py.lib()
    return a3ref_distort_py


def _k(oracle, kp, w=W, h=H):
    return oracle.intrinsics_new(w, h, kp[0], kp[1], kp[2], kp[3])


def _points(rng, w=W, h=H):
    gx, gy = np.meshgrid(np.linspace(-0.5, w - 0.5, 41), np.linspace(-0.5, h - 0.5, 23))
    grid = np.c_[gx.ravel(), gy.ravel()]
    return np.concatenate([grid, rng.uniform([-0.5, -0.5], [w - 0.5, h - 0.5], (2000, 2))]).astype(np.float32)


@pytest.mark.parametrize("camera", list(CAMERAS))
def test_agrees_with_opencv(od, oracle, camera):
    import cv2
    kp, dc = CAMERAS[camera]
    pts = _points(np.random.default_rng(1))
    got, ok = od.undistort_points(pts, _k(oracle, kp), od.distortion(*dc))
    assert ok.all()
    km = np.array([[kp[0], 0, kp[2]], [0, kp[1], kp[3]], [0, 0, 1]], np.float64)
    d = np.array(dc, np.float64)
    crit = (cv2.TERM_CRITERIA_COUNT | cv2.TERM_CRITERIA_EPS, 100, 1e-15)
    want = cv2.undistortPointsIter(pts.astype(np.float64).reshape(-1, 1, 2), km, d, None, None, crit).reshape(-1, 2)
    assert np.abs(got.astype(np.float64) - want).max() < 1e-6
    obj = np.c_[got.astype(np.float64), np.ones(len(got))]
    back = cv2.projectPoints(obj, np.zeros(3), np.zeros(3), km, d)[0].reshape(-1, 2)
    assert np.abs(back - pts).max() < 1e-3


def test_fold_fails(od, oracle):
    """k1 = -0.5: the forward model peaks at r = sqrt(2/3), r_d = 0.544.  Beyond it there is no solution; well inside, Newton
    converges."""
    kp = (1000.0, 1000.0, 0.0, 0.0)
    k = _k(oracle, kp)
    d = od.distortion(-0.5)
    ang = np.random.default_rng(2).uniform(0, 2 * np.pi, 400)
    for rd, want in ((0.45, True), (0.52, True), (0.56, False), (0.7, False), (2.0, False)):
        pts = np.c_[np.cos(ang), np.sin(ang)] * rd * kp[0]
        out, ok = od.undistort_points(pts, k, d)
        assert ok.all() if want else not ok.any(), rd
        if want:
            r = np.hypot(out[:, 0].astype(np.float64), out[:, 1].astype(np.float64))
            assert np.abs(r * (1 - 0.5 * r * r) - rd).max() < 1e-6


def test_non_finite_inputs_fail(od, oracle):
    k = _k(oracle, KP)
    pts = np.array([[np.nan, 100], [100, np.nan], [np.inf, 0], [-np.inf, 5], [3e38, 3e38], [640, 360]], np.float32)
    out, ok = od.undistort_points(pts, k, od.distortion(*BARREL))
    assert ok.tolist() == [False] * 5 + [True] and (out[:5] == 0).all()
    assert out[5].tolist() == [0.0, 0.0]


def _rot(rng, tilt=0.5):
    from scipy.spatial.transform import Rotation
    return Rotation.from_euler("xyz", rng.uniform(-tilt, tilt, 3)).as_matrix() @ np.diag([1.0, -1.0, -1.0])


def _angle(ra, rb):
    m = ra.T @ rb
    s = np.linalg.norm([m[2, 1] - m[1, 2], m[0, 2] - m[2, 0], m[1, 0] - m[0, 1]]) / 2
    return float(np.degrees(np.arctan2(s, (np.trace(m) - 1) / 2)))


def _pose(p):
    e, r, t = p.as_tuple()
    return float(e), r.astype(np.float64), t.astype(np.float64)


def test_exact_board_recovery(od, oracle):
    """Exact distorted projections of random boards: the board solve on undistorted corners recovers the pose to f32
    precision, and agrees with OpenCV's solvePnP with the same distortion where OpenCV finds the same minimum."""
    import cv2
    rng = np.random.default_rng(4)
    kp, dc = CAMERAS["barrel"]
    k, d = _k(oracle, kp), od.distortion(*dc)
    km = np.array([[kp[0], 0, kp[2]], [0, kp[1], kp[3]], [0, 0, 1]], np.float64)
    n_cv = 0
    for _ in range(60):
        board = Board.grid(int(rng.integers(2, 7)), int(rng.integers(2, 5)), 40.0, 10.0)
        R = _rot(rng)
        t = np.array([rng.uniform(-150, 150), rng.uniform(-80, 80), rng.uniform(450, 700)])
        img = np.array([synth.project_points(c, R, t, kp, dc) for c in board.corners], np.float32)
        b, _, n, ok = od.solve_frame(board.ids, board.corners, board.ids, img, k, d)
        assert ok and n == len(board)
        e, r, tt = _pose(b)
        assert e < 1e-6 and _angle(r, R) < 0.01 and np.abs(tt - t).max() < 1e-4 * t[2], (e, _angle(r, R), tt, t)
        obj = np.c_[board.corners.reshape(-1, 2).astype(np.float64), np.zeros(4 * len(board))]
        okc, rv, tv = cv2.solvePnP(obj, img.reshape(-1, 1, 2).astype(np.float64), km, np.array(dc, np.float64), flags=cv2.SOLVEPNP_ITERATIVE)
        rc, tc = cv2.Rodrigues(rv)[0], tv.ravel()
        if okc and _angle(rc, R) < 1.0:  # the same minimum (OpenCV may stop in the other branch)
            n_cv += 1
            assert _angle(r, rc) < 0.01 and np.abs(tt - tc).max() < 1e-4 * tc[2], (_angle(r, rc), tt, tc)
    assert n_cv >= 40


# ---- accuracy on rendered frames -------------------------------------------------------------------------------------

BOARD = Board.grid(6, 4, 40.0, 10.0)  # 24 markers, 290 x 190 mm
# the default min_corner_separation_factor (0.1 of 720 px) drops quads with corners under 72 px apart, which a 65 px
# marker squeezed by the lens near the frame's corners has
CFG = dict(min_corner_separation_factor=0.05)


def board_poses(n=12, seed=8):
    """n seeded poses of BOARD at 1280 x 720 whose image reaches toward the frame's corners: the board's centre is pushed
    toward a corner (each quadrant in turn) at 430-560 mm, so its markers are 65-85 px wide."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        R = _rot(rng, 0.35)
        z = rng.uniform(430, 560)
        sx, sy = (1 if i & 1 else -1), (1 if i & 2 else -1)
        px = KP[2] + sx * rng.uniform(0.15, 0.25) * W
        py = KP[3] + sy * rng.uniform(0.08, 0.16) * H
        c = np.array([(px - KP[2]) / KP[0] * z, (py - KP[3]) / KP[1] * z, z])
        centre = BOARD.corners.reshape(-1, 2).astype(np.float64).mean(0)
        out.append((R, c - R[:, :2] @ centre))
    return out


@functools.lru_cache(maxsize=None)
def _rendered(distorted: bool):
    frames = []
    for j, (R, t) in enumerate(board_poses()):
        img, _ = synth.render_board_frame(BOARD.ids, BOARD.corners, R, t, KP, W, H, noise=3, seed=j,
                                          distortion=BARREL if distorted else None)
        frames.append(img)
    return frames


def accuracy(od, oracle, refined: bool):
    """Per frame: (rotation error in degrees, translation error in mm) of the board pose for the distorted frames with
    the model, the distorted frames without it and the pinhole frames of the same poses, then the best single marker of
    the distorted frames with the model (undistorted corners -> solve_with_normalized_points)."""
    from oracle import a3ref_board_py as ob
    from oracle import a3ref_refine_py as rr
    k, d = _k(oracle, KP), od.distortion(*BARREL)
    rows = []
    for (R, t), dimg, pimg in zip(board_poses(), _rendered(True), _rendered(False)):
        row = []
        for img, model in ((dimg, True), (dimg, False), (pimg, False)):
            res = oracle.detect(img, "ARUCO", oracle.default_config(**CFG))
            grey = oracle.to_luma8(img)
            ids = [m["id"] for m in res.markers]
            cs = np.array([rr.refine_corners(grey, m["corners"])[0] if refined else np.array(m["corners"], np.float32).reshape(4, 2)
                           for m in res.markers], np.float32).reshape(-1, 4, 2)
            if model:
                b, _, n, ok = od.solve_frame(BOARD.ids, BOARD.corners, ids, cs, k, d)
            else:
                b, _, n, ok = ob.solve_frame(BOARD.ids, BOARD.corners, ids, cs, k=k)
            assert ok and n >= 3, (n, ok)
            _, rb, tb = _pose(b)
            row += [_angle(rb, R), float(np.linalg.norm(tb - t))]
            if model:
                single = []
                for i, c in zip(ids, cs):
                    if i >= len(BOARD):
                        continue
                    u, good = od.undistort_points(c, k, d)
                    if not good.all():
                        continue
                    mb, _ = oracle.solve_with_normalized_points(u.reshape(-1).tolist(), 40.0)
                    _, rm, tm = _pose(mb)
                    tm = tm - rm[:, :2] @ BOARD.corners[i].astype(np.float64).mean(0)
                    single.append((_angle(rm, R), float(np.linalg.norm(tm - t))))
                srow = min(single)
        rows.append(row + list(srow))
    return np.array(rows)  # [frame, (model rot, tr, no-model rot, tr, pinhole rot, tr, single rot, tr)]


@pytest.mark.parametrize("refined", [False, True], ids=["integer", "refined"])
def test_rendered_accuracy(od, oracle, refined):
    """Bars (DESIGN.md §4, K7).  Integer corners: with the model, the medians on distorted frames are within 2x those of
    the pinhole frames of the same poses, and far better than without the model.  Refined corners (K5's straight-line fit
    on a curved image) must still beat integer corners with the model."""
    a = accuracy(od, oracle, refined)
    med = np.median(a, axis=0)
    m_rot, m_tr, n_rot, n_tr, p_rot, p_tr = med[:6]
    if not refined:
        assert m_rot <= 2 * p_rot and m_tr <= 2 * p_tr, med
        assert n_rot > 3 * m_rot and n_tr > 3 * m_tr, med
        assert m_rot < 1.0 and m_tr < 1.5 and n_tr > 5.0, med
    else:
        ai = accuracy(od, oracle, False)
        mi = np.median(ai, axis=0)
        assert m_rot < mi[0] and m_tr < mi[1], (med, mi)
        assert m_rot < 0.2 and m_tr < 0.8, med
