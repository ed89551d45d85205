"""Lens distortion on the device (kernel K7) through the C ABI and the Python mirror.

Bar: BIT-EXACT against the CPU oracle (oracle/a3ref_distort.c: same operation order, no contraction) through the probe,
for the marker pose (undistort -> solve_with_normalized_points) and for the board pose, on every route of
a3_detect_batch; with the distortion off every output is what it was and K7 never runs.
"""
import ctypes as C

import numpy as np
import pytest

from tests.test_gpu_board import _detect_all
from tests.test_oracle_distortion import BARREL, BOARD, CFG, KP, H, W, board_poses

gpu = pytest.mark.gpu
SIZE = 40.0


@pytest.fixture(scope="module")
def a3():
    import aruco3_b200
    from aruco3_b200 import _ffi
    if _ffi.lib().a3_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tests have no fallback")
    return aruco3_b200


@pytest.fixture(scope="module")
def od():
    from oracle import a3ref_distort_py
    a3ref_distort_py.lib()
    return a3ref_distort_py


@pytest.fixture(scope="module")
def board_frames():
    """Four distorted 1280 x 720 frames of the 24-marker board, plus a blank one."""
    from aruco3_b200 import synth
    imgs = [synth.render_board_frame(BOARD.ids, BOARD.corners, R, t, KP, W, H, noise=3, seed=j, distortion=BARREL)[0]
            for j, (R, t) in enumerate(board_poses(4))]
    blank = np.empty_like(imgs[0])
    blank[:] = (204, 200, 192)
    return np.stack(imgs[:2] + [blank] + imgs[2:])


def _run(d, frames, mem="host", full=False):
    """a3_detect_batch -> (markers, poses [m, 2] A3Pose, corners f32 [m, 4, 2], board poses bytes per frame, status, stats)"""
    from aruco3_b200 import _ffi
    L = _ffi.lib()
    n, h, w = frames.shape[:3]
    cap = 64 * n
    ms, nm, outs, st = (_ffi.A3Marker * cap)(), C.c_uint32(), _ffi.A3Outputs(), _ffi.A3Stats()
    poses, corners, boards = (_ffi.A3Pose * (2 * cap))(), np.zeros((cap, 4, 2), np.float32), (_ffi.A3BoardPose * n)()
    outs.marker_poses = C.cast(poses, C.c_void_p).value
    outs.marker_corners = corners.ctypes.data
    outs.board_poses = C.cast(boards, C.c_void_p).value
    keep = []
    if full:
        cands, decs = np.zeros((8192, 8), np.uint32), (_ffi.A3Decode * 8192)()
        outs.candidates, outs.decodes, outs.cand_capacity = cands.ctypes.data, C.cast(decs, C.c_void_p).value, 8192
        keep = [cands, decs]
    if mem == "device":
        import torch
        src = torch.from_numpy(frames).cuda().contiguous()
        ptr, kind = src.data_ptr(), _ffi.MEM_DEVICE
    else:
        src = np.ascontiguousarray(frames)
        ptr, kind = src.ctypes.data, _ffi.MEM_HOST
    status = L.a3_detect_batch(d._h, ptr, _ffi.FMT_RGB8, kind, n, w, h, w * 3, w * h * 3, C.cast(ms, C.c_void_p), cap, C.byref(nm),
                               C.byref(outs), C.byref(st))
    del keep
    m = nm.value
    return [ms[i] for i in range(m)], [(bytes(poses[2 * i]), bytes(poses[2 * i + 1])) for i in range(m)], corners[:m].copy(), \
        [bytes(boards[i])[:2 * 52 + 5] for i in range(n)], status, st


def _oracle_k(oracle, w, h, kp):
    return oracle.intrinsics_new(w, h, kp[0], kp[1], kp[2], kp[3])


def expected_poses(oracle, od, markers, corners, refined, k, d):
    """The oracle chain per marker: undistort its four corners, then solve_with_normalized_points; a failed corner gives
    two default poses."""
    default = oracle.Pose()
    oracle._pose_lib().a3ref_pose_default(C.byref(default))
    out = []
    for i, m in enumerate(markers):
        c = corners[i] if refined else np.array(list(m.corners), np.float32).reshape(4, 2)
        u, ok = od.undistort_points(c, k, d)
        if ok.all():
            b, a = oracle.solve_with_normalized_points(u.reshape(-1).tolist(), SIZE)
            out.append((bytes(b), bytes(a)))
        else:
            out.append((bytes(default), bytes(default)))
    return out


def expected_boards(od, markers, corners, refined, n, k, d):
    out = []
    for f in range(n):
        sel = [i for i, m in enumerate(markers) if m.frame == f]
        ids = [markers[i].id for i in sel]
        cs = np.array([corners[i] if refined else np.array(list(markers[i].corners), np.float32).reshape(4, 2) for i in sel],
                      np.float32).reshape(-1, 4, 2)
        b, a, nm, ok = od.solve_frame(BOARD.ids, BOARD.corners, ids, cs, k, d)
        out.append(bytes(b) + bytes(a) + int(nm).to_bytes(4, "little") + bytes([int(ok)]))
    return out


@gpu
def test_probe_is_bit_exact(a3, od, oracle):
    rng = np.random.default_rng(5)
    cams = [(KP, BARREL), ((1000.0, 1000.0, 0.0, 0.0), (-0.5, 0.0, 0.0, 0.0, 0.0)),
            ((950.0, 940.0, 640.0, 360.0), (0.1, -0.05, 0.003, -0.002, 0.02))]
    with a3.Detector() as d:
        n_fail = 0
        for kp, dc in cams:
            pts = np.concatenate([rng.uniform(-200, 1500, (30000, 2)),                          # in and outside the frame
                                  rng.normal(0, 1, (3000, 2)) * 1e4,                           # far outside
                                  np.c_[np.cos(a := rng.uniform(0, 6.3, 2000)), np.sin(a)] * rng.uniform(0.5, 0.6, (2000, 1)) * 1000,
                                  [[np.nan, 1], [1, np.nan], [np.inf, 0], [0, -np.inf], [np.nan, np.inf], [3e38, -3e38]]]).astype(np.float32)
            k = a3.CameraIntrinsics(W, H, kp[0], kp[1], kp[2], kp[3])
            got, gok = d.undistort_points(pts, k, a3.CameraDistortion(*dc))
            want, wok = od.undistort_points(pts, _oracle_k(oracle, W, H, kp), od.distortion(*dc))
            assert np.array_equal(gok, wok) and got.tobytes() == want.tobytes()
            assert not wok[-6:].any()
            n_fail += int((~wok).sum())
        assert n_fail > 1000  # the fold and the far points fail, on the device as in the oracle


@gpu
@pytest.mark.parametrize("refined", [False, True], ids=["integer", "refined"])
def test_fused_marker_pose_is_bit_exact(a3, od, oracle, refined):
    """K4 with distortion equals undistort -> solve_with_normalized_points on distorted board frames and on C1 / C3 / C5."""
    from aruco3_b200 import synth
    sets = [("board", None)] + [(c, synth.render_batch(c, 2)[0]) for c in ("C1", "C3", "C5")]
    for name, frames in sets:
        if frames is None:
            from aruco3_b200 import synth as s
            frames = np.stack([s.render_board_frame(BOARD.ids, BOARD.corners, R, t, KP, W, H, noise=3, seed=j, distortion=BARREL)[0]
                               for j, (R, t) in enumerate(board_poses(2))])
        n, h, w = frames.shape[:3]
        kp = (900.0, 900.0, w / 2.0, h / 2.0)
        with a3.Detector(a3.DetectorConfig(**CFG), corners="refined" if refined else "integer",
                         distortion=a3.CameraDistortion(*BARREL)) as d:
            d.set_pose(SIZE, a3.CameraIntrinsics(w, h, *kp))
            for call in range(2):
                ms, poses, cs, _, status, st = _run(d, frames)
                assert status == 0 and len(ms) > 0 and st.undistort_kernel_launches == 1, (name, call)
                want = expected_poses(oracle, od, ms, cs, refined, _oracle_k(oracle, w, h, kp), od.distortion(*BARREL))
                assert poses == want, (name, call)


@gpu
@pytest.mark.parametrize("refined", [False, True], ids=["integer", "refined"])
def test_routes_are_bit_exact(a3, od, oracle, board_frames, refined):
    """Marker and board poses with distortion on the one-shot route, the ordinary route over several chunks, resident frames
    and the host contour stage; pose and board intrinsics equal (one K7 set) and different (two)."""
    from aruco3_b200 import _ffi
    frames = board_frames
    n, h, w = frames.shape[:3]
    dc = od.distortion(*BARREL)
    kp_pose, kp_board = KP, (905.0, 898.0, 641.0, 359.5)
    for kpb in (kp_pose, kp_board):
        kw = dict(config=a3.DetectorConfig(**CFG), corners="refined" if refined else "integer", board=BOARD,
                  board_intrinsics=a3.CameraIntrinsics(w, h, *kpb), distortion=a3.CameraDistortion(*BARREL))
        sets = 1 if kpb == kp_pose else 2

        def check(d, mem="host", full=False, one_shot=None):
            ms, poses, cs, boards, status, st = _run(d, frames, mem, full)
            assert status == 0 and st.undistort_kernel_launches >= sets and st.ms_undistort_kernel > 0
            if one_shot is not None:
                assert st.one_shot == one_shot
            assert poses == expected_poses(oracle, od, ms, cs, refined, _oracle_k(oracle, w, h, kp_pose), dc)
            want_b = expected_boards(od, ms, cs, refined, n, _oracle_k(oracle, w, h, kpb), dc)
            assert boards == want_b and sum(b[-1] for b in want_b) >= 3
        with a3.Detector(**kw) as d:
            d.set_pose(SIZE, a3.CameraIntrinsics(w, h, *kp_pose))
            for call in range(3):  # first call, one-shot lean, one-shot full
                check(d, full=call == 2, one_shot=1 if call else 0)
            check(d, mem="device")
        with a3.Detector(**kw) as d:  # ordinary route over several chunks and decode groups
            d.set_pose(SIZE, a3.CameraIntrinsics(w, h, *kp_pose))
            t = _ffi.A3K1Tuning()
            t.chunk_frames = 1
            _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(d._h, C.byref(t)))
            for mem in ("host", "device"):
                check(d, mem=mem, full=mem == "device")
        with a3.Detector(contours="host", **kw) as d:
            d.set_pose(SIZE, a3.CameraIntrinsics(w, h, *kp_pose))
            for mem in ("host", "device"):
                check(d, mem=mem, one_shot=0)


@gpu
def test_board_probe_uses_the_distortion(a3, od, oracle, board_frames):
    from oracle import a3ref_py
    n, h, w = board_frames.shape[:3]
    res = [a3ref_py.detect(f, "ARUCO", a3ref_py.default_config(**CFG)) for f in board_frames]
    ids = [m["id"] for r in res for m in r.markers]
    cs = np.array([m["corners"] for r in res for m in r.markers], np.float32).reshape(-1, 4, 2)
    fr = [f for f, r in enumerate(res) for _ in r.markers]
    with a3.Detector(board=BOARD, board_intrinsics=a3.CameraIntrinsics(w, h, *KP), distortion=a3.CameraDistortion(*BARREL)) as d:
        got = d.solve_board(ids, cs, fr, n)
    fr = np.array(fr)
    for f in range(n):
        sel = fr == f
        b, a, nm, ok = od.solve_frame(BOARD.ids, BOARD.corners, np.array(ids, np.uint64)[sel], cs[sel], _oracle_k(oracle, w, h, KP),
                                      od.distortion(*BARREL))
        assert (got[f].ok, got[f].n_markers) == (ok, nm) and got[f].best.rotation.tobytes() == np.array(b.rotation, np.float32).tobytes()


@gpu
def test_distortion_off_leaves_everything_alone(a3, board_frames):
    """Never set, set to NULL or all zeros, or set and switched off again: every output buffer and every counter is what a
    detector that never had a distortion returns, and K7 is never launched."""
    from aruco3_b200 import _ffi, synth
    c1, _ = synth.render_batch("C1", 3)
    n, h, w = board_frames.shape[:3]

    def run(d, fr):
        out = [_detect_all(a3, d, fr, full=f) for f in (False, False, True)] + [_detect_all(a3, d, fr, mem="device", full=True)]
        t = _ffi.A3K1Tuning()
        t.chunk_frames = 1
        _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(d._h, C.byref(t)))
        out.append(_detect_all(a3, d, fr, full=True))
        _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(d._h, None))
        return out

    def make(fr, dist):
        hh, ww = fr.shape[1:3]
        d = a3.Detector(a3.DetectorConfig(**CFG), corners="refined", board=BOARD, board_intrinsics=a3.CameraIntrinsics(ww, hh, *KP))
        d.set_pose(SIZE, a3.CameraIntrinsics(ww, hh, *KP))
        if dist == "zeros":
            d.set_distortion(a3.CameraDistortion())
        elif dist == "toggled":
            d.set_distortion(a3.CameraDistortion(*BARREL))
            d.set_distortion(None)
        return d

    for fr in (board_frames[:3], c1):
        with make(fr, None) as plain:
            base = run(plain, fr)
        assert any(r[4]["one_shot"] for r in base)
        for dist in ("zeros", "toggled"):
            with make(fr, dist) as d:
                got = run(d, fr)
            for b, o in zip(base, got):
                assert o[4]["undistort_kernel_launches"] == 0 and o == b, dist


@gpu
def test_setter_rules_and_release(a3):
    from aruco3_b200 import _ffi
    L = _ffi.lib()
    k = a3.CameraIntrinsics(W, H, *KP)
    dist = a3.CameraDistortion(*BARREL)
    with a3.Detector() as d:
        def set_d(*c):
            return L.a3_detector_set_distortion(d._h, C.byref(_ffi.A3CameraDistortion(*c)))
        for bad in ((np.nan, 0, 0, 0, 0), (0, np.inf, 0, 0, 0), (0, 0, 0, 0, -np.inf)):
            assert set_d(*bad) == _ffi.A3_ERR_INVALID_ARGUMENT
        # distortion first, then an UNDISTORTED pose or board mode
        assert set_d(*BARREL) == 0
        assert L.a3_detector_set_pose(d._h, _ffi.POSE_UNDISTORTED, C.c_float(SIZE), None) == _ffi.A3_ERR_INVALID_ARGUMENT
        cb = BOARD.to_c()
        assert L.a3_detector_set_board(d._h, C.byref(cb), _ffi.POSE_UNDISTORTED, None) == _ffi.A3_ERR_INVALID_ARGUMENT
        assert L.a3_detector_set_pose(d._h, _ffi.POSE_INTRINSICS, C.c_float(SIZE), C.byref(k._c)) == 0
        assert L.a3_detector_set_board(d._h, C.byref(cb), _ffi.POSE_INTRINSICS, C.byref(k._c)) == 0
        assert L.a3_detector_set_pose(d._h, _ffi.POSE_OFF, C.c_float(0), None) == 0
        # the other order: UNDISTORTED modes first, then the distortion
        assert set_d(0, 0, 0, 0, 0) == 0
        assert L.a3_detector_set_pose(d._h, _ffi.POSE_UNDISTORTED, C.c_float(SIZE), None) == 0
        assert set_d(*BARREL) == _ffi.A3_ERR_INVALID_ARGUMENT
        assert L.a3_detector_set_pose(d._h, _ffi.POSE_OFF, C.c_float(0), None) == 0
        assert L.a3_detector_set_board(d._h, C.byref(cb), _ffi.POSE_UNDISTORTED, None) == 0
        assert set_d(*BARREL) == _ffi.A3_ERR_INVALID_ARGUMENT
        assert L.a3_detector_set_board(d._h, None, _ffi.POSE_OFF, None) == 0
        assert set_d(*BARREL) == 0 and L.a3_detector_set_distortion(d._h, None) == 0
        with pytest.raises(a3.A3Error):
            a3.Detector(board=BOARD, distortion=dist)  # a board in undistorted mode
    # a3_detector_release resets it: the handle comes back without distortion
    cfg = a3.DetectorConfig().to_c()
    dic = a3.ARDictionary.new_from_named_dict("ARUCO")
    h = C.c_void_p()
    _ffi.check(L.a3_detector_acquire(C.byref(cfg), C.byref(dic._c), 0, C.byref(h)))
    _ffi.check(L.a3_detector_set_distortion(h, C.byref(dist._c)))
    L.a3_detector_release(h)
    h2 = C.c_void_p()
    _ffi.check(L.a3_detector_acquire(C.byref(cfg), C.byref(dic._c), 0, C.byref(h2)))
    assert h2.value == h.value
    assert L.a3_detector_set_pose(h2, _ffi.POSE_UNDISTORTED, C.c_float(SIZE), None) == 0  # legal again: no distortion held
    L.a3_detector_release(h2)


@gpu
def test_sharded_detector_passes_it_on(a3, board_frames):
    from aruco3_b200.sharding import ShardedDetector
    n, h, w = board_frames.shape[:3]
    kw = dict(board=BOARD, board_intrinsics=a3.CameraIntrinsics(w, h, *KP), distortion=a3.CameraDistortion(*BARREL))
    with a3.Detector(a3.DetectorConfig(**CFG), **kw) as d:
        want = [x.board_pose.best.rotation.tobytes() for x in d.detect_batch(board_frames)]
    with ShardedDetector(a3.DetectorConfig(**CFG), devices=[0, 0], **kw) as sd:
        assert [x.board_pose.best.rotation.tobytes() for x in sd.detect_batch(board_frames)] == want
