"""CPU oracle of the board pose (kernel K6, oracle/a3ref_board.c): exact recovery, agreement with independent f64
solvers (scipy, OpenCV) on noisy corners, agreement with the single-marker solve on a one-marker board, the skip and
fallback rules, and accuracy on rendered board frames taken through the oracle's detect and refinement.
"""
import numpy as np
import pytest

from aruco3_b200 import synth
from aruco3_b200.board import Board

K = (800.0, 800.0, 320.0, 240.0)  # the rendered frames' pinhole, 640 x 480


@pytest.fixture(scope="module")
def ob():
    from oracle import a3ref_board_py
    a3ref_board_py.lib()
    return a3ref_board_py


def _rot(rng, tilt=0.6):
    from scipy.spatial.transform import Rotation
    return Rotation.from_euler("xyz", rng.uniform(-tilt, tilt, 3)).as_matrix() @ np.diag([1.0, -1.0, -1.0])


def _random_case(rng, noise=0.0):
    """A board of 2..12 markers scattered on the plane, a pose in front of the camera, normalised image points."""
    m = int(rng.integers(2, 13))
    centres = rng.uniform(-0.5, 0.5, size=(m, 2))
    side = rng.uniform(0.05, 0.15)
    sq = np.array([[-1, 1], [1, 1], [1, -1], [-1, -1]]) * side / 2
    xy = (centres[:, None, :] + sq[None]).reshape(-1, 2)
    R = _rot(rng)
    t = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3), rng.uniform(2.0, 5.0)])
    X = xy @ R[:, :2].T + t
    uv = X[:, :2] / X[:, 2:] + rng.normal(0, noise, size=(len(xy), 2))
    return uv.astype(np.float32), xy.astype(np.float32), R, t


def _pose(p):
    e, r, t = p.as_tuple()
    return float(e), r.astype(np.float64), t.astype(np.float64)


def _angle(ra, rb):
    m = ra.T @ rb
    s = np.linalg.norm([m[2, 1] - m[1, 2], m[0, 2] - m[2, 0], m[1, 0] - m[0, 1]]) / 2
    return float(np.degrees(np.arctan2(s, (np.trace(m) - 1) / 2)))


def _rms(uv, xy, R, t):
    X = xy.astype(np.float64) @ R[:, :2].T + t
    d = X[:, :2] / X[:, 2:] - uv.astype(np.float64)
    return float(np.sqrt((d ** 2).sum(1).mean()))


def test_exact_projections_are_recovered(ob):
    rng = np.random.default_rng(7)
    for _ in range(200):
        uv, xy, R, t = _random_case(rng)
        best, alt, ok = ob.solve(uv, xy)
        assert ok
        e, r, tt = _pose(best)
        assert e < 2e-6 and _angle(r, R) < 2e-3 and np.abs(tt - t).max() < 1e-4 * t[2], (e, _angle(r, R), tt, t)
        assert _pose(alt)[0] >= e
        assert abs(np.linalg.det(r) - 1) < 1e-5


def test_noisy_corners_agree_with_scipy_and_opencv(ob):
    """The same objective minimised in f64 by scipy (started at the truth) and, where OpenCV is installed, OpenCV's
    iterative PnP: the oracle's best branch reaches the same minimum."""
    from scipy.optimize import least_squares
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(11)
    for _ in range(60):
        uv, xy, R, t = _random_case(rng, noise=4e-4)
        best, _, ok = ob.solve(uv, xy)
        assert ok
        e, r, tt = _pose(best)
        obj = np.c_[xy.astype(np.float64), np.zeros(len(xy))]

        def res(p):
            X = obj @ Rotation.from_rotvec(p[:3]).as_matrix().T + p[3:]
            return (X[:, :2] / X[:, 2:] - uv.astype(np.float64)).ravel()
        sol = least_squares(res, np.r_[Rotation.from_matrix(R).as_rotvec(), t], xtol=1e-15, ftol=1e-15, gtol=1e-15)
        rs, ts = Rotation.from_rotvec(sol.x[:3]).as_matrix(), sol.x[3:]
        rms = float(np.sqrt((sol.fun ** 2).sum() / len(xy)))
        assert abs(e - rms) <= 1e-6 + 1e-4 * rms, (e, rms)
        assert _angle(r, rs) < 0.01 and np.abs(tt - ts).max() < 1e-4 * ts[2], (_angle(r, rs), tt, ts)
        try:
            import cv2
        except ImportError:  # the scipy comparison above stands on its own
            continue
        okc, rv, tv = cv2.solvePnP(obj, uv.astype(np.float64).reshape(-1, 1, 2), np.eye(3), None, flags=cv2.SOLVEPNP_ITERATIVE)
        assert okc
        rc, tc = cv2.Rodrigues(rv)[0], tv.ravel()
        if _rms(uv, xy, rc, tc) <= rms * (1 + 1e-6):  # OpenCV found the same minimum (it may stop in the other branch)
            assert _angle(r, rc) < 0.01 and np.abs(tt - tc).max() < 1e-4 * tc[2], (_angle(r, rc), tt, tc)


def test_one_marker_board_matches_the_single_marker_solve(ob, oracle):
    rng = np.random.default_rng(5)
    L = 40.0
    board = Board([0], [[(-L / 2, L / 2), (L / 2, L / 2), (L / 2, -L / 2), (-L / 2, -L / 2)]])
    for _ in range(50):
        R = _rot(rng, 0.5)
        t = np.array([rng.uniform(-20, 20), rng.uniform(-20, 20), rng.uniform(200, 400)])
        X = board.corners[0].astype(np.float64) @ R[:, :2].T + t
        uv = (X[:, :2] / X[:, 2:]).astype(np.float32)
        best, _, ok = ob.solve(uv, board.corners[0])
        kb, _ = oracle.solve_with_normalized_points(uv.reshape(-1).tolist(), L)
        _, r4, t4 = _pose(kb)
        _, r, tt = _pose(best)
        assert ok and _angle(r, r4) < 0.05 and np.abs(tt - t4).max() < 1e-3 * t4[2], (_angle(r, r4), tt, t4)


def _frame(ob, board, ids, corners, **kw):
    return ob.solve_frame(board.ids, board.corners, np.asarray(ids, np.uint64), np.asarray(corners, np.float32), **kw)


def test_skips_and_fallbacks(ob, oracle):
    board = Board.grid(3, 2, 40.0, 10.0)
    rng = np.random.default_rng(3)
    R, t = _rot(rng, 0.3), np.array([5.0, -3.0, 400.0])
    img = [synth.project_points(c, R, t, K) for c in board.corners]
    k = oracle.intrinsics_new(640, 480, K[0], K[1], K[2], K[3])
    full = _frame(ob, board, board.ids, img, k=k)
    assert full[2] == 6 and full[3] and _angle(_pose(full[0])[1], R) < 0.01
    # a non-board id is skipped; the result is that of the board markers alone
    extra = _frame(ob, board, list(board.ids) + [40], img + [img[0] + 50], k=k)
    assert extra[2] == 6 and bytes(extra[0]) == bytes(full[0])
    # an id seen twice in the frame: both detections are skipped
    dup = _frame(ob, board, [0, 1, 2, 0, 3], [img[0], img[1], img[2], img[0] + 3, img[3]], k=k)
    ref = _frame(ob, board, [1, 2, 3], [img[1], img[2], img[3]], k=k)
    assert dup[2] == 3 and bytes(dup[0]) == bytes(ref[0]) and bytes(dup[1]) == bytes(ref[1])
    # no board marker: n_markers 0, not ok, both poses the default
    for ids, cs in (([], np.zeros((0, 4, 2))), ([50, 51], img[:2]), ([0, 0], img[:2])):
        b, a, n, ok = _frame(ob, board, ids, cs, k=k)
        assert n == 0 and not ok and b.error == np.float32(1e31) and a.error == np.float32(1e31)
    # degenerate: every corner at one image point (no spread), and a non-finite corner
    for cs in ([np.full((4, 2), 100.0)] * 2, [img[0], np.full((4, 2), np.nan)]):
        b, a, n, ok = _frame(ob, board, [0, 1], cs, k=k)
        assert n == 2 and not ok and b.error == np.float32(1e31) and a.error == np.float32(1e31)
    # undistorted mode normalises by the frame size, as the single-marker solve does
    und = _frame(ob, board, board.ids, [c * [640 / K[0], 480 / K[1]] for c in img], image_size=(640, 480))
    assert und[3] and und[2] == 6


def board_frames(n=12, seed=21):
    """Rendered 640 x 480 frames of a 4 x 3 grid board (40 mm markers, 10 mm apart) plus two markers that are not on it."""
    board = Board.grid(4, 3, 40.0, 10.0)
    out = []
    for R, t in synth.board_views(n, seed=seed):
        img, truth = synth.render_board_frame(board.ids, board.corners, R, t, K, 640, 480, extra_ids=(100, 101), noise=3, seed=seed)
        out.append((img, truth, R, t))
    return board, out


def accuracy(ob, oracle, refined: bool):
    """Per frame: rotation error (deg) and translation error (mm) of the board pose and of the best single-marker K4 pose."""
    from oracle import a3ref_refine_py as rr
    board, frames = board_frames()
    k = oracle.intrinsics_new(640, 480, K[0], K[1], K[2], K[3])
    rows = []
    for img, _, R, t in frames:
        res = oracle.detect(img, "ARUCO")
        grey = oracle.to_luma8(img)
        ids, cs = [], []
        for m in res.markers:
            c = np.array(m["corners"], np.float32).reshape(4, 2)
            if refined:
                c = rr.refine_corners(grey, m["corners"])[0]
            ids.append(m["id"])
            cs.append(c)
        b, _, n, ok = _frame(ob, board, ids, cs, k=k)
        assert ok and n >= 3
        _, rb, tb = _pose(b)
        single = []
        for i, c in zip(ids, cs):
            if i >= len(board):
                continue
            mb, _ = rr.solve_with_intrinsics_f32(c, 40.0, k)
            _, rm, tm = _pose(mb)
            centre = board.corners[i].astype(np.float64).mean(0)
            tm = tm - rm[:, :2] @ centre  # the board origin under the marker's pose (the marker frame is the board frame shifted)
            single.append((_angle(rm, R), float(np.linalg.norm(tm - t))))
        best_single = min(single)
        rows.append((_angle(rb, R), float(np.linalg.norm(tb - t)), best_single[0], best_single[1]))
    return np.array(rows)


@pytest.mark.parametrize("refined", [False, True], ids=["integer", "refined"])
def test_rendered_board_accuracy(ob, oracle, refined):
    """Bars (DESIGN.md §4, K6): the board's rotation and translation errors against the rendered ground truth, and the
    board against the best single marker of the same frame."""
    a = accuracy(ob, oracle, refined)
    rot, tr, srot, str_ = a.T
    if refined:
        assert np.median(rot) < 0.1 and rot.max() < 0.5 and np.median(tr) < 0.2 and tr.max() < 1.0, a
    else:
        assert np.median(rot) < 1.0 and rot.max() < 4.0 and np.median(tr) < 1.0 and tr.max() < 2.5, a
    assert np.median(rot) < np.median(srot) and np.median(tr) < np.median(str_), a
