"""Board pose on the device (kernel K6) through the C ABI and the Python mirror.

Bar: BIT-EXACT against the CPU oracle (oracle/a3ref_board.c: same operation order, same summation trees, no contraction)
through the probe and on every route of a3_detect_batch; with the board off every output is what it was.
"""
import ctypes as C
import subprocess

import numpy as np
import pytest

from tests.test_oracle_board import K, board_frames

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def a3():
    import aruco3_b200
    from aruco3_b200 import _ffi
    if _ffi.lib().a3_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tests have no fallback")
    return aruco3_b200


@pytest.fixture(scope="module")
def ob():
    from oracle import a3ref_board_py
    a3ref_board_py.lib()
    return a3ref_board_py


def _key_c(bp):
    """bytes of an A3BoardPose (or the oracle's (best, alt, n, ok)) for exact comparison"""
    if isinstance(bp, tuple):
        b, a, n, ok = bp
        return bytes(b) + bytes(a) + int(n).to_bytes(4, "little") + bytes([int(ok)])
    return bytes(bp)[:2 * 52 + 5]


def _key_py(bp):
    return b"".join(np.float32(p.error).tobytes() + p.rotation.tobytes() + p.translation.tobytes() for p in (bp.best, bp.alt)) + \
        int(bp.n_markers).to_bytes(4, "little") + bytes([int(bp.ok)])


def _frames():
    """Board frames, a frame with no marker at all, and one with only markers that are not on the board."""
    board, fr = board_frames(n=5, seed=33)
    imgs = [f[0] for f in fr]
    blank = np.empty_like(imgs[0])
    blank[:] = (204, 200, 192)
    from aruco3_b200 import synth
    other, _ = synth.render_board_frame([200, 201], board.corners[:2], fr[0][2], fr[0][3], K, 640, 480)
    return board, np.stack(imgs[:2] + [blank, other] + imgs[2:])


def expected(oracle, ob, board, frames, refined, intrinsics):
    from oracle import a3ref_refine_py as rr
    h, w = frames.shape[1:3]
    k = oracle.intrinsics_new(w, h, K[0], K[1], K[2], K[3]) if intrinsics else None
    out = []
    for img in frames:
        res = oracle.detect(img, "ARUCO")
        grey = oracle.to_luma8(img)
        ids = [m["id"] for m in res.markers]
        cs = [rr.refine_corners(grey, m["corners"])[0] if refined else np.array(m["corners"], np.float32).reshape(4, 2) for m in res.markers]
        out.append(_key_c(ob.solve_frame(board.ids, board.corners, ids, np.array(cs, np.float32).reshape(-1, 4, 2),
                                         image_size=None if intrinsics else (w, h), k=k)))
    return out


def _intr(a3, w, h):
    return a3.CameraIntrinsics(w, h, K[0], K[1], K[2], K[3])


@gpu
def test_probe_is_bit_exact_on_random_inputs(a3, ob, oracle):
    from aruco3_b200.board import Board
    rng = np.random.default_rng(99)
    board = Board(rng.permutation(1000)[:40], rng.uniform(-100, 100, size=(40, 4, 2)))
    w, h = 640, 480
    k = oracle.intrinsics_new(w, h, 700.0, 710.0, 300.0, 250.0)
    for intr in (False, True):
        ids, cs, fr, nf = [], [], [], 600
        for f in range(nf):
            n = int(rng.integers(0, 12))
            kind = rng.random()
            for _ in range(n):
                ids.append(int(board.ids[rng.integers(0, 40)]) if rng.random() < 0.8 else int(rng.integers(0, 1100)))
                if kind < 0.6:    # plausible quads
                    c = rng.uniform(0, 600, 2) + np.array([[0, 0], [40, 0], [40, 40], [0, 40]]) + rng.normal(0, 3, (4, 2))
                elif kind < 0.8:  # wild
                    c = rng.uniform(-1e4, 1e4, (4, 2))
                elif kind < 0.9:  # degenerate: one point
                    c = np.full((4, 2), rng.uniform(0, 600))
                else:             # collinear
                    c = np.c_[np.linspace(0, 300, 4), np.linspace(0, 100, 4)]
                cs.append(c)
                fr.append(f)
        cs = np.array(cs, np.float32).reshape(-1, 4, 2)
        with a3.Detector() as d:
            d.set_board(board, a3.CameraIntrinsics(w, h, 700.0, 710.0, 300.0, 250.0) if intr else None)
            got = d.solve_board(ids, cs, fr, nf, image_size=(w, h))
        fr = np.array(fr)
        n_ok = 0
        for f in range(nf):
            sel = fr == f
            want = ob.solve_frame(board.ids, board.corners, np.array(ids, np.uint64)[sel], cs[sel], image_size=None if intr else (w, h),
                                  k=k if intr else None)
            assert _key_py(got[f]) == _key_c(want), f
            n_ok += want[3]
        assert 0.2 * nf < n_ok < 0.9 * nf  # both outcomes are exercised


def _detect_all(a3, d, frames, mem="host", full=False):
    """a3_detect_batch with every output buffer (grey, mask, candidates, homographies, decodes, offsets, marker poses and
    corners, board poses) -> (the bytes of all of them and of the markers, the status and the counters of a3_stats)"""
    from aruco3_b200 import _ffi
    L = _ffi.lib()
    n, h, w = frames.shape[:3]
    cap, cc, hs = 64 * n, 4096, 49
    ms, nm, outs, st = (_ffi.A3Marker * cap)(), C.c_uint32(), _ffi.A3Outputs(), _ffi.A3Stats()
    bufs = dict(offsets=np.zeros(n + 1, np.uint32), poses=(_ffi.A3Pose * (2 * cap))(), corners=np.zeros((cap, 8), np.float32),
                boards=(_ffi.A3BoardPose * n)())
    outs.frame_marker_offsets = bufs["offsets"].ctypes.data
    outs.marker_poses = C.cast(bufs["poses"], C.c_void_p).value
    outs.marker_corners = bufs["corners"].ctypes.data
    outs.board_poses = C.cast(bufs["boards"], C.c_void_p).value
    if full:
        bufs.update(grey=np.zeros((n, h, w), np.uint8), mask=np.zeros((n, h, w), np.uint8), cands=np.zeros((cc, 8), np.uint32),
                    cframe=np.zeros(cc, np.uint32), patches=np.zeros((cc, hs, hs), np.uint8), decs=(_ffi.A3Decode * cc)())
        outs.grey, outs.mask, outs.candidates = bufs["grey"].ctypes.data, bufs["mask"].ctypes.data, bufs["cands"].ctypes.data
        outs.candidate_frame, outs.homographies = bufs["cframe"].ctypes.data, bufs["patches"].ctypes.data
        outs.decodes, outs.cand_capacity = C.cast(bufs["decs"], C.c_void_p).value, cc
    if mem == "device":
        import torch
        src = torch.from_numpy(frames).cuda().contiguous()
        ptr, kind = src.data_ptr(), _ffi.MEM_DEVICE
    else:
        src = np.ascontiguousarray(frames)
        ptr, kind = src.ctypes.data, _ffi.MEM_HOST
    status = L.a3_detect_batch(d._h, ptr, _ffi.FMT_RGB8, kind, n, w, h, w * 3, w * h * 3, C.cast(ms, C.c_void_p), cap, C.byref(nm),
                               C.byref(outs), C.byref(st))
    counters = {f: getattr(st, f) for f, _ in _ffi.A3Stats._fields_ if not f.startswith("ms_")}
    data = {k: bytes(v) for k, v in bufs.items()}
    data["markers"] = bytes(ms)
    return data, status, outs.n_candidates, nm.value, counters


def _detect_c(a3, d, frames, mem="host", markers=True, full=False, cap=None):
    """a3_detect_batch at the C level -> (board pose keys, markers bytes, status, stats)."""
    from aruco3_b200 import _ffi
    L = _ffi.lib()
    n, h, w = frames.shape[:3]
    cap = 64 * n if cap is None else cap
    ms = (_ffi.A3Marker * max(cap, 1))()
    nm = C.c_uint32()
    outs = _ffi.A3Outputs()
    bp = (_ffi.A3BoardPose * n)()
    outs.board_poses = C.cast(bp, C.c_void_p).value
    keep = []
    if full:
        cands, decs = np.zeros((4096, 8), np.uint32), (_ffi.A3Decode * 4096)()
        outs.candidates, outs.decodes, outs.cand_capacity = cands.ctypes.data, C.cast(decs, C.c_void_p).value, 4096
        keep = [cands, decs]
    st = _ffi.A3Stats()
    if mem == "device":
        import torch
        src = torch.from_numpy(frames).cuda().contiguous()
        ptr, kind = src.data_ptr(), _ffi.MEM_DEVICE
    else:
        src = np.ascontiguousarray(frames)
        ptr, kind = src.ctypes.data, _ffi.MEM_HOST
    status = L.a3_detect_batch(d._h, ptr, _ffi.FMT_RGB8, kind, n, w, h, w * 3, w * h * 3, C.cast(ms, C.c_void_p) if markers else None, cap,
                               C.byref(nm), C.byref(outs), C.byref(st))
    del keep
    return [_key_c(bp[i]) for i in range(n)], [bytes(ms[i]) for i in range(min(nm.value, cap))], status, st


@gpu
@pytest.mark.parametrize("refined", [False, True], ids=["integer", "refined"])
@pytest.mark.parametrize("intrinsics", [False, True], ids=["undistorted", "intrinsics"])
def test_detect_batch_routes_are_bit_exact(a3, ob, oracle, refined, intrinsics):
    from aruco3_b200 import _ffi
    board, frames = _frames()
    n, h, w = frames.shape[:3]
    want = expected(oracle, ob, board, frames, refined, intrinsics)
    assert sum(k[-1] for k in want) >= 5  # boards were seen
    corners = "refined" if refined else "integer"
    kw = dict(board=board, board_intrinsics=_intr(a3, w, h) if intrinsics else None, corners=corners)
    with a3.Detector(**kw) as d:  # one-shot: lean (markers only), then full
        for call in range(3):
            keys, _, status, st = _detect_c(a3, d, frames, full=call == 2)
            assert status == 0 and keys == want, call
            assert st.one_shot == (1 if call else 0) and st.board_kernel_launches == 1 and st.ms_board_kernel > 0
        for call in range(2):  # resident frames
            keys, _, status, st = _detect_c(a3, d, frames, mem="device")
            assert status == 0 and keys == want and st.board_kernel_launches == 1
        dets = d.detect_batch(frames)  # the Python mirror
        assert [_key_py(x.board_pose) for x in dets] == want
    with a3.Detector(**kw) as d:  # ordinary route over several chunks and decode groups
        t = _ffi.A3K1Tuning()
        t.chunk_frames = 1
        _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(d._h, C.byref(t)))
        for mem in ("host", "device"):
            for call in range(2):
                keys, _, status, st = _detect_c(a3, d, frames, mem=mem, full=call == 1)
                assert status == 0 and keys == want and st.board_kernel_launches >= 1, (mem, call)
                assert st.one_shot == 0 or mem == "device"  # resident frames may take the one-shot route
        # resident frames of a new geometry take the ordinary route: one decode group whose quads are gathered on the
        # device, with the per-frame offsets of pack_offsets_kernel
        many = np.concatenate([frames] * 10)
        keys, _, status, st = _detect_c(a3, d, many, mem="device", full=True)
        assert status == 0 and keys == want * 10 and st.one_shot == 0 and st.board_kernel_launches >= 1
    with a3.Detector(contours="host", **kw) as d:  # host contour stage
        for mem in ("host", "device"):
            for call in range(2):
                keys, _, status, st = _detect_c(a3, d, frames, mem=mem, full=call == 1)
                assert status == 0 and keys == want and st.one_shot == 0 and st.board_kernel_launches >= 1, (mem, call)


@gpu
@pytest.mark.parametrize("refined", [False, True], ids=["integer", "refined"])
def test_board_poses_do_not_depend_on_other_outputs(a3, ob, oracle, refined):
    board, frames = _frames()
    want = expected(oracle, ob, board, frames, refined, False)
    for contours in ("device", "host"):
        with a3.Detector(board=board, corners="refined" if refined else "integer", contours=contours) as d:
            for _ in range(2):
                assert _detect_c(a3, d, frames, markers=False)[0] == want                # markers == NULL
                assert _detect_c(a3, d, frames)[0] == want                               # markers only (lean)
                assert _detect_c(a3, d, frames, full=True)[0] == want                    # full outputs
                keys, ms, status, _ = _detect_c(a3, d, frames, cap=3)                    # markers over capacity
                assert status == 4 and keys == want and len(ms) == 3


@gpu
def test_board_off_leaves_everything_alone(a3):
    """Never set, or set and switched off again: every output buffer and every counter is what a detector that never had a
    board returns, and K6 is never launched."""
    from aruco3_b200 import synth
    board, frames = _frames()
    c1, _ = synth.render_batch("C1", 3)

    def run(d, fr):  # first call, one-shot lean, one-shot full, resident, ordinary route over chunks
        from aruco3_b200 import _ffi
        out = [_detect_all(a3, d, fr, full=f) for f in (False, False, True)] + [_detect_all(a3, d, fr, mem="device", full=True)]
        t = _ffi.A3K1Tuning()
        t.chunk_frames = 1
        _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(d._h, C.byref(t)))
        out.append(_detect_all(a3, d, fr, full=True))
        _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(d._h, None))
        return out

    for fr in (frames, c1):
        with a3.Detector(corners="refined") as plain:
            plain.set_pose(40.0)
            base = run(plain, fr)
        with a3.Detector(corners="refined") as d:
            d.set_pose(40.0)
            d.set_board(board)
            on = run(d, fr)
            d.set_board(None)
            off = run(d, fr)
        assert [r[1] for r in base] == [0] * 5 and any(r[4]["one_shot"] for r in base)
        for b, o in zip(base, off):
            assert o[4]["board_kernel_launches"] == 0
            assert o == b  # every buffer byte for byte (board poses untouched), status, counts and counters
        for b, o in zip(base, on):  # with the board on, everything but the board poses and K6's counter is unchanged
            assert {k: v for k, v in o[0].items() if k != "boards"} == {k: v for k, v in b[0].items() if k != "boards"}
            assert {k: v for k, v in o[4].items() if k != "board_kernel_launches"} == {k: v for k, v in b[4].items() if k != "board_kernel_launches"}
        with a3.Detector() as d:
            assert all(x.board_pose is None for x in d.detect_batch(fr))


@gpu
def test_release_resets_the_board(a3):
    from aruco3_b200 import _ffi
    L = _ffi.lib()
    board, frames = _frames()
    cfg = a3.DetectorConfig().to_c()
    dic = a3.ARDictionary.new_from_named_dict("ARUCO")
    h = C.c_void_p()
    _ffi.check(L.a3_detector_acquire(C.byref(cfg), C.byref(dic._c), 0, C.byref(h)))
    cb = board.to_c()
    _ffi.check(L.a3_detector_set_board(h, C.byref(cb), _ffi.POSE_UNDISTORTED, None))
    L.a3_detector_release(h)
    h2 = C.c_void_p()
    _ffi.check(L.a3_detector_acquire(C.byref(cfg), C.byref(dic._c), 0, C.byref(h2)))
    assert h2.value == h.value

    class D:
        _h = h2
    keys, _, status, st = _detect_c(a3, D, frames)
    L.a3_detector_release(h2)
    assert status == 0 and st.board_kernel_launches == 0 and all(k == bytes(len(k)) for k in keys)  # board_poses untouched


@gpu
def test_sharded_detector_equals_one_detector(a3):
    from aruco3_b200.sharding import ShardedDetector
    board, frames = _frames()
    with a3.Detector(board=board, corners="refined") as d:
        want = [_key_py(x.board_pose) for x in d.detect_batch(frames)]
    with ShardedDetector(devices=[0, 0], board=board, corners="refined") as sd:
        assert [_key_py(x.board_pose) for x in sd.detect_batch(frames)] == want


@gpu
def test_invalid_arguments(a3):
    from aruco3_b200 import _ffi
    from aruco3_b200.board import Board
    L = _ffi.lib()
    sq = [[(-1, 1), (1, 1), (1, -1), (-1, -1)]]
    with a3.Detector(dictionary="ARTAG") as d:  # 1 024 codes: a board of 1 024 markers fits
        n_codes = len(d.dictionary.code_list)

        def status(board, mode=_ffi.POSE_UNDISTORTED, k=None):
            c = board.to_c() if board is not None else None
            return L.a3_detector_set_board(d._h, C.byref(c) if c is not None else None, mode, k)
        assert status(Board([1, 1], sq * 2)) == 1                       # duplicate ids
        assert status(Board([n_codes], sq)) == 1                        # id >= n_codes
        assert status(Board(np.zeros(0), np.zeros((0, 4, 2)))) == 1    # no markers
        assert status(Board(np.arange(1025), sq * 1025)) == 1           # too many
        assert status(Board([0], [[(np.nan, 1), (1, 1), (1, -1), (-1, -1)]])) == 1
        assert status(Board([0], [[(np.inf, 1), (1, 1), (1, -1), (-1, -1)]])) == 1
        assert status(Board([0], sq), _ffi.POSE_OFF) == 1
        assert status(Board([0], sq), _ffi.POSE_NORMALIZED) == 1
        assert status(Board([0], sq), _ffi.POSE_INTRINSICS, None) == 1  # intrinsics missing
        assert status(Board(np.arange(1024), sq * 1024)) == 0
        assert status(None) == 0


def test_struct_layouts_match_the_header(tmp_path):
    """sizeof / offsetof of the new structs and fields: the C compiler against the ctypes mirror."""
    from pathlib import Path

    from aruco3_b200 import _ffi
    root = Path(__file__).resolve().parent.parent
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "aruco3_b200.h"\nint main(void) {\n'
                   'printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(a3_board), offsetof(a3_board, ids), offsetof(a3_board, corners),'
                   ' sizeof(a3_board_pose), offsetof(a3_board_pose, alt), offsetof(a3_board_pose, n_markers), offsetof(a3_board_pose, ok),'
                   ' sizeof(a3_outputs), offsetof(a3_outputs, board_poses), sizeof(a3_stats));\n'
                   'printf("%zu %zu\\n", offsetof(a3_stats, board_kernel_launches), offsetof(a3_stats, ms_board_kernel));\nreturn 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", str(root / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    B, P, O, S = _ffi.A3Board, _ffi.A3BoardPose, _ffi.A3Outputs, _ffi.A3Stats
    assert got == [C.sizeof(B), B.ids.offset, B.corners.offset, C.sizeof(P), P.alt.offset, P.n_markers.offset, P.ok.offset, C.sizeof(O),
                   O.board_poses.offset, C.sizeof(S), S.board_kernel_launches.offset, S.ms_board_kernel.offset]
