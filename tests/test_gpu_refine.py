"""Sub-pixel marker corners on the device (kernel K5) through the C ABI and the Python mirror.

Bar: BIT-EXACT against the CPU oracle (oracle/a3ref_refine.c: same f32 operation order, same summation trees, no
contraction) through the probe and on every route of a3_detect_batch; refinement off leaves every output as it was.
"""
import ctypes as C

import numpy as np
import pytest

from tests.test_oracle_refine import SETS, errors_against_truth, oracle_markers

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def a3():
    import aruco3_b200
    from aruco3_b200 import _ffi
    if _ffi.lib().a3_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tests have no fallback")
    return aruco3_b200


@pytest.fixture(scope="module")
def rr():
    from oracle import a3ref_refine_py
    a3ref_refine_py.lib()
    return a3ref_refine_py


def _oracle_refine(rr, greys, corners, frames):
    out = np.zeros((len(corners), 4, 2), np.float32)
    ok = np.zeros(len(corners), bool)
    for i, (c, f) in enumerate(zip(corners, frames)):
        out[i], ok[i] = rr.refine_corners(greys[f], c)
    return out, ok


def _random_scene(rng, w, h, n_quads):
    """Light noisy background with dark convex quads; corners = the quads' integer corners, jittered, plus some wild ones."""
    g = rng.normal(190, 6, size=(h, w)).clip(0, 255)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64) + 0.5
    corners = []
    for _ in range(n_quads):
        cx, cy = rng.uniform(20, w - 20), rng.uniform(20, h - 20)
        r = rng.uniform(8, 40)
        a0 = rng.uniform(0, np.pi / 2)
        ang = a0 + np.array([0, 0.5, 1.0, 1.5]) * np.pi + rng.normal(0, 0.08, 4)
        q = np.stack([cx + r * np.cos(ang), cy + r * np.sin(ang)], 1)  # clockwise on screen (y down)
        inside = np.ones_like(xx, bool)
        for k in range(4):
            p, s = q[k], q[(k + 1) % 4]
            inside &= (s[0] - p[0]) * (yy - p[1]) - (s[1] - p[1]) * (xx - p[0]) >= 0
        g[inside] = rng.uniform(10, 60)
        jit = rng.integers(-3, 4, size=(4, 2)) if rng.random() < 0.7 else rng.integers(-40, 41, size=(4, 2))
        corners.append(np.clip(np.round(q) + jit, 0, [w - 1, h - 1]).astype(np.uint32))
    return g.astype(np.uint8), corners


def test_probe_is_bit_exact_on_random_quads(a3, rr):
    rng = np.random.default_rng(2024)
    w, h = 320, 240
    greys, corners, frames = [], [], []
    for f in range(96):
        g, cs = _random_scene(rng, w, h, 24)
        greys.append(g)
        corners += cs
        frames += [f] * len(cs)
    corners += [rng.integers(0, 400, size=(4, 2)).astype(np.uint32) for _ in range(200)]  # anything at all, off the image too
    frames += list(rng.integers(0, 96, size=200))
    greys, corners, frames = np.stack(greys), np.stack(corners), np.array(frames, np.uint32)
    with a3.Detector() as d:
        got, ok = d.refine_corners(greys, corners, frames)
    want, wok = _oracle_refine(rr, greys, corners, frames)
    assert np.array_equal(ok, wok)
    assert got.tobytes() == want.tobytes()
    assert 0.2 < ok.mean() < 0.95, ok.mean()  # both outcomes are exercised


@pytest.mark.parametrize("name,n", SETS)
def test_probe_is_bit_exact_on_detected_markers(a3, rr, oracle, name, n):
    with a3.Detector() as d:
        for grey, markers, _ in oracle_markers(oracle, name, n):
            corners = np.array([m["corners"] for m in markers], np.uint32)
            got, ok = d.refine_corners(grey, corners)
            want, wok = _oracle_refine(rr, grey[None], corners, [0] * len(corners))
            assert np.array_equal(ok, wok) and got.tobytes() == want.tobytes()


def _got_markers(dets):
    return [[(m.id, m.rotation, m.corners, np.array(m.corners_refined, np.float32).tobytes(), m.refined) for m in x.markers] for x in dets]


def _greys(oracle, frames):
    return [oracle.to_luma8(f) for f in frames]


def test_detect_batch_routes_are_bit_exact(a3, rr, oracle):
    from aruco3_b200 import _ffi, synth
    frames, _ = synth.render_batch("C1", 4)
    greys = _greys(oracle, frames)
    want = [[(m["id"], m["rotation"], [tuple(m["corners"][2 * k:2 * k + 2]) for k in range(4)]) + (lambda r: (r[0].tobytes(), r[1]))(
        rr.refine_corners(greys[f], m["corners"])) for m in oracle.detect(frames[f], "ARUCO").markers] for f in range(len(frames))]
    assert sum(len(x) for x in want) > 10 and all(r[4] for x in want for r in x)

    def check(dets):
        assert _got_markers(dets) == want

    # one-shot route, host input in one chunk: markers only (assembled on the device), then with every candidate output
    with a3.Detector(corners="refined") as d:
        for call in range(3):
            check(d.detect_batch(frames, full=call == 2))
            assert d.last_stats["one_shot"] == (1 if call else 0)
            assert d.last_stats["refine_kernel_launches"] == 1 and d.last_stats["ms_refine_kernel"] > 0
    # ordinary route: host input over several front-end chunks
    with a3.Detector(corners="refined") as d:
        t = _ffi.A3K1Tuning()
        t.chunk_frames = 1
        _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(d._h, C.byref(t)))
        for call in range(2):
            check(d.detect_batch(frames, full=call == 1))
            assert d.last_stats["one_shot"] == 0 and d.last_stats["refine_kernel_launches"] >= 1
    # host contour stage
    with a3.Detector(corners="refined", contours="host") as d:
        for call in range(2):
            check(d.detect_batch(frames, full=call == 1))
            assert d.last_stats["one_shot"] == 0 and d.last_stats["refine_kernel_launches"] >= 1


def _detect_resident(a3, d, frames_dev, n, w, h, poses=False):
    from aruco3_b200 import _ffi
    L = _ffi.lib()
    cap = 64 * n
    markers = (_ffi.A3Marker * cap)()
    nm = C.c_uint32()
    outs = _ffi.A3Outputs()
    corners = np.zeros((cap, 8), np.float32)
    outs.marker_corners = corners.ctypes.data
    pz = (_ffi.A3Pose * (2 * cap))()
    if poses:
        outs.marker_poses = C.cast(pz, C.c_void_p).value
    st = _ffi.A3Stats()
    _ffi.check(L.a3_detect_batch(d._h, frames_dev.data_ptr(), _ffi.FMT_RGB8, _ffi.MEM_DEVICE, n, w, h, w * 3, w * h * 3,
                                 C.cast(markers, C.c_void_p), cap, C.byref(nm), C.byref(outs), C.byref(st)))
    ms = [markers[i] for i in range(nm.value)]
    return ms, corners[:nm.value].copy(), [pz[i] for i in range(2 * nm.value)], st


def test_one_shot_resident_frames_are_bit_exact(a3, rr, oracle):
    torch = pytest.importorskip("torch")  # plumbing only: frames resident on the device
    from aruco3_b200 import synth
    frames, _ = synth.render_batch("C1", 4)
    n, h, w = frames.shape[:3]
    greys = _greys(oracle, frames)
    dev = torch.from_numpy(frames).cuda().contiguous()
    with a3.Detector(corners="refined") as d:
        for call in range(2):
            ms, corners, _, st = _detect_resident(a3, d, dev, n, w, h)
            assert st.one_shot == (1 if call else 0) and st.refine_kernel_launches == 1
            assert len(ms) > 10
            for m, c in zip(ms, corners):
                r, ok = rr.refine_corners(greys[m.frame], list(m.corners))
                assert c.tobytes() == r.tobytes() and m.corners_refined == ok


def test_refinement_leaves_everything_else_alone(a3):
    from aruco3_b200 import synth
    frames, _ = synth.render_batch("C3", 2)

    def summary(dets):
        return [([list(sum(c, ())) for c in x.candidates], [x_.tobytes() for x_ in x.homographies], x.decodes,
                 [(m.candidate, m.id, m.rotation, m.hamming_distance, m.code, m.corners) for m in x.markers]) for x in dets]

    def poses(dets):
        return [(p.error, p.rotation.tobytes(), p.translation.tobytes()) for x in dets for m in x.markers for p in m.poses]

    with a3.Detector() as plain:
        plain.set_pose(40.0)
        base = [plain.detect_batch(frames, full=True) for _ in range(2)]
    with a3.Detector() as d:  # switched on and off again: the same bytes as a detector that never had it
        d.set_pose(40.0)
        d.set_corner_refinement("refined")
        on = [d.detect_batch(frames, full=True) for _ in range(2)]
        d.set_corner_refinement("integer")
        off = [d.detect_batch(frames, full=True) for _ in range(2)]
        assert d.last_stats["refine_kernel_launches"] == 0 and d.last_stats["ms_refine_kernel"] == 0
    for b, o, r in zip(base, off, on):
        assert summary(o) == summary(b) and poses(o) == poses(b)
        assert all(m.corners_refined is None and not m.refined for x in o for m in x.markers)
        assert summary(r) == summary(b)  # refinement changes no integer output
        assert any(m.refined for x in r for m in x.markers)


def test_refinement_off_marker_bytes(a3):
    """At the C level the marker records are byte for byte those of a detector that never had the setter called."""
    torch = pytest.importorskip("torch")
    from aruco3_b200 import _ffi, synth
    frames, _ = synth.render_batch("C1", 3)
    n, h, w = frames.shape[:3]
    dev = torch.from_numpy(frames).cuda().contiguous()
    with a3.Detector() as d:
        d.set_pose(40.0)
        base = [_detect_resident(a3, d, dev, n, w, h, poses=True) for _ in range(2)]
    with a3.Detector() as d:
        d.set_pose(40.0)
        _ffi.check(_ffi.lib().a3_detector_set_corner_refinement(d._h, _ffi.CORNERS_INTEGER))
        got = [_detect_resident(a3, d, dev, n, w, h, poses=True) for _ in range(2)]
    for (bm, bc, bp, _), (gm, gc, gp, gs) in zip(base, got):
        assert [bytes(m) for m in gm] == [bytes(m) for m in bm] and all(m.corners_refined == 0 for m in gm)
        assert [bytes(p) for p in gp] == [bytes(p) for p in bp]
        assert not gc.any() and gs.refine_kernel_launches == 0


@pytest.mark.parametrize("mode", ["undistorted", "intrinsics"])
def test_poses_come_from_the_refined_corners(a3, rr, oracle, mode):
    from aruco3_b200 import synth
    from aruco3_b200.pose import CameraIntrinsics
    frames, _ = synth.render_batch("C1", 3)
    n, h, w = frames.shape[:3]
    k = CameraIntrinsics(w, h, 800.0, 810.0) if mode == "intrinsics" else None
    ok_ = oracle.intrinsics_new(w, h, 800.0, 810.0) if k is not None else None
    for full in (False, True):
        with a3.Detector(corners="refined") as d:
            d.set_pose(40.0, k)
            for _ in range(2):
                dets = d.detect_batch(frames, full=full)
                count = 0
                for x in dets:
                    for m in x.markers:
                        c = np.array(m.corners_refined, np.float32)
                        if k is None:
                            ob, oa = rr.solve_with_undistorted_points_f32(c, 40.0, (w, h))
                        else:
                            ob, oa = rr.solve_with_intrinsics_f32(c, 40.0, ok_)
                        for p, q in zip(m.poses, (ob, oa)):
                            e, r, t = q.as_tuple()
                            assert np.float32(p.error) == e and p.rotation.tobytes() == r.tobytes() and p.translation.tobytes() == t.tobytes()
                        count += 1
                assert count > 10


def test_release_resets_refinement(a3):
    from aruco3_b200 import _ffi, synth
    L = _ffi.lib()
    frames, _ = synth.render_batch("C1", 1)
    cfg = a3.DetectorConfig().to_c()
    dic = a3.ARDictionary.new_from_named_dict("ARUCO")
    h = C.c_void_p()
    _ffi.check(L.a3_detector_acquire(C.byref(cfg), C.byref(dic._c), 0, C.byref(h)))
    _ffi.check(L.a3_detector_set_corner_refinement(h, _ffi.CORNERS_REFINED))
    L.a3_detector_release(h)
    h2 = C.c_void_p()
    _ffi.check(L.a3_detector_acquire(C.byref(cfg), C.byref(dic._c), 0, C.byref(h2)))
    assert h2.value == h.value  # the same cached handle
    img = np.ascontiguousarray(frames[0])
    markers = (_ffi.A3Marker * 64)()
    nm = C.c_uint32()
    outs = _ffi.A3Outputs()
    corners = np.zeros((64, 8), np.float32)
    outs.marker_corners = corners.ctypes.data
    st = _ffi.A3Stats()
    _ffi.check(L.a3_detect_batch(h2, img.ctypes.data, _ffi.FMT_RGB8, _ffi.MEM_HOST, 1, img.shape[1], img.shape[0], img.shape[1] * 3,
                                 img.shape[1] * img.shape[0] * 3, C.cast(markers, C.c_void_p), 64, C.byref(nm), C.byref(outs), C.byref(st)))
    L.a3_detector_release(h2)
    assert nm.value > 0 and st.refine_kernel_launches == 0
    assert all(markers[i].corners_refined == 0 for i in range(nm.value)) and not corners.any()


@pytest.mark.parametrize("name,n", [s for s in SETS if s[0] in ("C3", "C5")])
def test_pipeline_accuracy(a3, name, n):
    from aruco3_b200 import synth
    spec = synth.CONFIGS[name]
    cfg = a3.DetectorConfig(min_corner_separation_factor=spec.min_corner_separation_factor)
    pairs = []
    with a3.Detector(cfg, dictionary=spec.dictionary, corners="refined") as d:
        for f in range(n):
            img, truth = synth.render_frame(spec, f)
            for m in d.detect_batch(img[None])[0].markers:
                pairs.append((np.array(m.corners, np.float64), np.array(m.corners_refined, np.float64), truth))
    e_int, e_ref = errors_against_truth(pairs)
    assert e_ref.mean() <= 0.25 and np.percentile(e_ref, 95) <= 0.5 and e_ref.max() <= 1.5, (e_ref.mean(), e_ref.max())
    assert e_ref.mean() < e_int.mean() / 4


def test_sharded_detector_equals_one_detector(a3):
    from aruco3_b200 import synth
    from aruco3_b200.sharding import ShardedDetector
    frames, _ = synth.render_batch("C1", 6)
    with a3.Detector(corners="refined") as d:
        want = _got_markers(d.detect_batch(frames))
    with ShardedDetector(devices=[0, 0], corners="refined") as sd:
        assert _got_markers(sd.detect_batch(frames)) == want
