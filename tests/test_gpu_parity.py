"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle, bit for bit.

Bar (BASELINE.json north_star): threshold masks, grey, candidates, patches, codes, ids, rotations bit-exact;
corners "within 1e-3 px" — they are integers (contour pixels, SURVEY Q10), so the test demands equality.
"""
import ctypes as C
from collections import Counter

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def a3():
    import aruco3_b200
    from aruco3_b200 import _ffi
    if _ffi.lib().a3_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tests have no fallback")
    return aruco3_b200


@pytest.fixture(scope="module")
def det(a3):
    d = a3.Detector(dictionary="ARUCO", device=0)
    yield d
    d.close()


def _noise(seed, shape):
    return np.random.default_rng(seed).integers(0, 256, size=shape, dtype=np.uint8)


def _smooth(seed, n, h, w, c):
    """Low-contrast smooth content + a little noise: exercises the `pix >= mean` tie region heavily."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    out = np.empty((n, h, w, c), np.uint8)
    for i in range(n):
        base = 120 + 60 * np.sin(xx / (7.0 + i)) * np.cos(yy / 11.0)
        for k in range(c):
            out[i, :, :, k] = np.clip(base + rng.integers(-2, 3, size=(h, w)) + 5 * k, 0, 255)
    return out


def _check_k1(det, oracle, frames, radius=7):
    grey, mask, bits = det.gray_threshold(frames, want_bits=True)
    n, h, w = grey.shape
    for i in range(n):
        g = oracle.to_luma8(frames[i])
        m = oracle.adaptive_threshold(g, radius)
        assert np.array_equal(grey[i], g), f"grey differs (frame {i}, {w}x{h})"
        bad = np.argwhere(mask[i] != m)
        assert bad.size == 0, f"mask differs at {bad[:5].tolist()} (frame {i}, {w}x{h}, r={radius})"
        # 1-bit mask: bit (x & 31) of word x >> 5; bits beyond w are zero
        unpacked = np.unpackbits(bits[i].view(np.uint8).reshape(h, -1), axis=1, bitorder="little")
        assert np.array_equal(unpacked[:, :w], (m > 0).astype(np.uint8)), f"mask bits differ (frame {i}, {w}x{h})"
        assert not unpacked[:, w:].any(), "mask bits beyond the row end must be zero"


@pytest.mark.parametrize("w,h", [(640, 480), (1920, 1080), (1, 1), (3, 2), (13, 9), (15, 15), (16, 8), (17, 33), (31, 64),
                                 (100, 50), (257, 19), (1921, 37), (2049, 16), (4100, 9)])
def test_k1_sizes_rgb(det, oracle, w, h):
    """into_luma8 + adaptive_threshold (src/aruco.rs:60-61): every clipped-window case, widths off every alignment."""
    _check_k1(det, oracle, _noise(w * 131 + h, (2, h, w, 3)))


@pytest.mark.parametrize("c", [1, 3, 4])
def test_k1_formats(det, oracle, c):
    """Luma8 passes through, Rgba8 ignores alpha (SURVEY A.1)."""
    for (w, h) in [(640, 480), (333, 77)]:
        f = _noise(7 + c, (3, h, w, c))
        _check_k1(det, oracle, f[..., 0] if c == 1 else f)
        s = _smooth(11 + c, 2, h, w, c)
        _check_k1(det, oracle, s[..., 0] if c == 1 else s)


@pytest.mark.parametrize("c", [3, 4])
@pytest.mark.parametrize("w,h", [(640, 480), (1920, 1080), (33, 17), (250, 31)])
def test_k1_bgr_formats(a3, det, oracle, c, w, h):
    """A3_FMT_BGR8 / A3_FMT_BGRA8 (SURVEY §8 f-4): camera byte order read directly == the host swizzle of
    examples/webcam_kamera.rs:38-52 followed by into_luma8, on the fast (TMA strips) and the generic kernel."""
    frames = _noise(100 + c + w, (3, h, w, c))
    grey, mask = det.gray_threshold(frames, order="bgr")
    swz = frames.copy()
    swz[..., 0], swz[..., 2] = frames[..., 2], frames[..., 0]
    grey2, mask2 = det.gray_threshold(swz)
    assert np.array_equal(grey, grey2) and np.array_equal(mask, mask2)
    for i in range(frames.shape[0]):
        assert np.array_equal(grey[i], oracle.to_luma8(frames[i], order="bgr"))
        assert np.array_equal(grey[i], oracle.to_luma8(swz[i]))


def test_detect_bgra_equals_swizzled_rgba(a3):
    from aruco3_b200 import synth
    rgb, _ = synth.render_batch("C1", 3)
    bgra = np.concatenate([rgb[..., ::-1], np.full(rgb.shape[:3] + (1,), 255, np.uint8)], axis=3)
    with a3.Detector(dictionary="ARUCO") as d:
        want = d.detect_batch(rgb)
        got = d.detect_batch(bgra, order="bgr")
    assert [[(m.id, m.corners, m.rotation) for m in x.markers] for x in got] == [[(m.id, m.corners, m.rotation) for m in x.markers] for x in want]
    assert sum(len(x.markers) for x in got) > 5


@pytest.mark.parametrize("radius", [1, 2, 3, 5, 7, 8, 12, 16, 17, 33, 64, 127])
def test_k1_radius(a3, oracle, radius):
    """threshold_window is a public config field (src/aruco.rs:24); the reference accepts any block radius, the CUDA path 1..127
    (its column sums of 2 r + 1 rows travel as 16-bit values), windows wider or taller than the frame included."""
    with a3.Detector(a3.DetectorConfig(threshold_window=radius)) as d:
        _check_k1(d, oracle, _noise(radius, (2, 120, 212, 3)), radius)
        _check_k1(d, oracle, _smooth(radius, 1, 61, 1000, 3), radius)
        if radius > 16:
            _check_k1(d, oracle, _noise(radius + 1, (1, 300, 2300, 3)), radius)  # several strips, a halo wider than a 32-column word


def test_k1_radius_beyond_the_cuda_path(a3):
    """threshold_window > 127: A3_ERR_UNSUPPORTED, stated, not a wrong answer (the reference itself has no limit)."""
    with pytest.raises(a3.A3Error) as e:
        a3.Detector(a3.DetectorConfig(threshold_window=128))
    assert e.value.status == a3._ffi.A3_ERR_UNSUPPORTED


def test_k1_extremes(det, oracle):
    """all-black / all-white / (255,255,255)->255, (0,255,0)->182, (255,0,0)->54, (0,0,255)->18 (SURVEY A.1)."""
    f = np.zeros((4, 40, 48, 3), np.uint8)
    f[1] = 255
    f[2, :, :, 1] = 255
    f[3, :20, :, 0] = 255
    f[3, 20:, :, 2] = 255
    grey, mask = det.gray_threshold(f)
    assert grey[0].max() == 0 and grey[1].min() == 255 and (grey[2] == 182).all()
    assert (grey[3, :20] == 54).all() and (grey[3, 20:] == 18).all()
    _check_k1(det, oracle, f)


def test_k1_batch_equals_single(det, oracle):
    """Frames are independent: a batch gives the same bytes as one frame at a time (sharding invariant)."""
    from aruco3_b200 import synth
    frames, _ = synth.render_batch("C1n", 5)
    g, m = det.gray_threshold(frames)
    for i in range(5):
        g1, m1 = det.gray_threshold(frames[i:i + 1])
        assert np.array_equal(g[i], g1[0]) and np.array_equal(m[i], m1[0])


def test_k1_device_pointers_and_tilings(a3, det, oracle):
    """The zero-copy flavour (A3_MEM_DEVICE) on a caller's stream, device buffers owned by torch (plumbing only)."""
    torch = pytest.importorskip("torch")
    from aruco3_b200 import _ffi
    f = _noise(5, (3, 270, 480, 3))
    d_src = torch.from_numpy(f).cuda()
    d_grey = torch.zeros((3, 270, 480), dtype=torch.uint8, device="cuda")
    d_mask = torch.zeros_like(d_grey)
    d_bits = torch.zeros((3, 270, 15), dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    _ffi.check(_ffi.lib().a3_gray_threshold_batch(det._h, d_src.data_ptr(), _ffi.FMT_RGB8, _ffi.MEM_DEVICE, 3, 480, 270,
                                                  480 * 3, 480 * 270 * 3, d_grey.data_ptr(), d_mask.data_ptr(),
                                                  d_bits.data_ptr(), C.c_void_p(stream)))
    torch.cuda.synchronize()
    for i in range(3):
        g = oracle.to_luma8(f[i])
        assert np.array_equal(d_grey[i].cpu().numpy(), g)
        assert np.array_equal(d_mask[i].cpu().numpy(), oracle.adaptive_threshold(g, 7))


def _decode_tuple(d):
    return (d["homography_ok"], d["otsu"], d["has_codes"], d["codes"] if d["has_codes"] else None)


def _check_detection(got, ref, label=""):
    assert np.array_equal(got.grey, ref.grey), f"{label}: grey"
    if got.mask is not None:
        assert np.array_equal(got.mask, ref.mask), f"{label}: mask"
    assert [list(sum(c, ())) for c in got.candidates] == ref.candidates.tolist(), f"{label}: candidates"
    for k, dc in enumerate(got.decodes):
        assert dc["homography_ok"] == bool(ref.homography_ok[k]), f"{label}: homography_ok[{k}]"
        if dc["homography_ok"]:
            assert np.array_equal(got.homographies[k], ref.homographies[k]), f"{label}: patch {k}"
        else:
            assert got.homographies[k].shape == (1, 1)
        assert dc["otsu"] == int(ref.otsu[k]), f"{label}: otsu[{k}]"
        assert dc["has_codes"] == bool(ref.has_codes[k]), f"{label}: has_codes[{k}]"
        if dc["has_codes"]:
            assert dc["codes"] == [int(c) for c in ref.codes[k]], f"{label}: codes[{k}]"
    gm = [(m.candidate, m.id, m.rotation, m.hamming_distance, m.code, [v for c in m.corners for v in c]) for m in got.markers]
    rm = [(m["candidate"], m["id"], m["rotation"], m["hamming_distance"], m["code"], m["corners"]) for m in ref.markers]
    assert gm == rm, f"{label}: markers"


@pytest.mark.parametrize("name,frames", [("C1", 6), ("C1n", 4), ("C3", 2), ("C3n", 1), ("C2a", 1), ("C5", 1)])
def test_detect_matches_oracle(a3, oracle, name, frames):
    """Detector::detect (src/aruco.rs:52-121) on BASELINE.json's configs: every intermediate equals the oracle's."""
    from aruco3_b200 import synth
    spec = synth.CONFIGS[name]
    imgs, truth = synth.render_batch(spec, frames)
    cfg = a3.DetectorConfig(min_corner_separation_factor=spec.min_corner_separation_factor)
    ocfg = oracle.default_config(min_corner_separation_factor=spec.min_corner_separation_factor)
    with a3.Detector(cfg, spec.dictionary) as d:
        got = d.detect_batch(imgs, full=True, want_mask=True)
        single = d.detect(imgs[0])
    for f in range(frames):
        ref = oracle.detect(imgs[f], spec.dictionary, ocfg)
        _check_detection(got[f], ref, f"{name}[{f}]")
        if not spec.pure_noise and spec.noise == 0 and name != "C5":
            # ground truth: no false ids on clean frames (recall itself is a property of the reference algorithm,
            # ~92 % on these scenes for the oracle too; the full-size test below bounds it)
            assert not (Counter(m.id for m in got[f].markers) - Counter(t.id for t in truth[f])), f"{name}[{f}]: false ids"
    assert [(m.id, m.corners) for m in single.markers] == [(m.id, m.corners) for m in got[0].markers]


def test_detect_all_dictionaries(a3, oracle):
    """Every table of src/dictionaries.rs:30-113 through K2 (mark sizes 6, 7, 8, 10; 64-bit CHILITAGS codes)."""
    from aruco3_b200 import synth
    for name in a3.ARDictionary.get_dictionary_names():
        spec = synth.FrameSpec("dict-" + name, 9, 640, 480, dictionary=name, markers=(4, 6), side=(70, 120))
        imgs, truth = synth.render_batch(spec, 2)
        with a3.Detector(dictionary=name) as d:
            got = d.detect_batch(imgs, full=True)
        for f in range(2):
            _check_detection(got[f], oracle.detect(imgs[f], name), f"{name}[{f}]")


def test_decode_stage_probe(det, oracle):
    """a3_decode_candidates on hand-made quads incl. degenerate ones (projection failure -> 1x1 zero patch, Q5)."""
    from aruco3_b200 import synth
    imgs, _ = synth.render_batch("C1", 2)
    grey = np.stack([oracle.to_luma8(i) for i in imgs])
    rng = np.random.default_rng(3)
    quads, qf = [], []
    for f in range(2):
        for q in oracle.detect(imgs[f]).candidates:
            quads.append(q); qf.append(f)
    for _ in range(40):  # random convex-ish and degenerate quads, some partly outside the image
        cx, cy, s = rng.integers(0, 640), rng.integers(0, 480), rng.integers(1, 200)
        q = np.array([cx, cy, cx + s, cy + rng.integers(0, 9), cx + s, cy + s, cx + rng.integers(0, 9), cy + s])
        quads.append(np.clip(q, 0, [639, 479] * 4)); qf.append(int(rng.integers(0, 2)))
    quads.append(np.array([5, 5, 5, 5, 5, 5, 5, 5])); qf.append(0)            # all corners equal
    quads.append(np.array([10, 10, 20, 20, 30, 30, 40, 40])); qf.append(1)    # collinear
    quads = np.array(quads, np.uint32)
    decs, patches = det.decode_candidates(grey, quads, np.array(qf, np.uint32))
    L = oracle.lib()
    for k in range(len(quads)):
        patch = np.zeros((49, 49), np.uint8)
        g = np.ascontiguousarray(grey[qf[k]])
        qk = np.ascontiguousarray(quads[k])
        ok = L.a3ref_extract_homography(g.ctypes.data, 640, 480, qk.ctypes.data, 49, patch.ctypes.data)
        assert bool(ok) == decs[k]["homography_ok"], f"quad {k}: homography_ok"
        assert np.array_equal(patches[k], patch), f"quad {k}: patch"
        codes = (C.c_uint64 * 4)()
        otsu = C.c_uint8()
        src = patch if ok else np.zeros((1, 1), np.uint8)
        some = L.a3ref_homography_to_code_permutations(src.ctypes.data, src.shape[1], src.shape[0], 7, codes, C.byref(otsu), None)
        assert decs[k]["otsu"] == otsu.value and decs[k]["has_codes"] == bool(some), f"quad {k}: otsu / has_codes"
        if some:
            assert decs[k]["codes"] == list(codes), f"quad {k}: codes"


def test_filter_high_bit_errors_off(a3, oracle):
    """filter_high_bit_errors = false accepts every border-passing candidate (src/aruco.rs:96)."""
    from aruco3_b200 import synth
    imgs, _ = synth.render_batch("C1n", 2)
    with a3.Detector(a3.DetectorConfig(filter_high_bit_errors=False)) as d:
        got = d.detect_batch(imgs, full=True)
    for f in range(2):
        _check_detection(got[f], oracle.detect(imgs[f], "ARUCO", oracle.default_config(filter_high_bit_errors=0)), f"nofilter[{f}]")


def test_edges_and_errors(a3, det):
    """Empty batch, tiny frames, capacity error with valid counts, and the reference's panics as status codes."""
    from aruco3_b200 import _ffi, synth
    assert det.detect_batch(np.zeros((0, 480, 640, 3), np.uint8)) == []
    assert det.detect(np.zeros((1, 1, 3), np.uint8)).markers == []
    assert det.detect(np.full((8, 8), 200, np.uint8)).markers == []
    with pytest.raises(a3.A3Error) as e:
        a3.Detector(dictionary="NOT_A_DICTIONARY")
    assert e.value.status == _ffi.A3_ERR_UNKNOWN_DICTIONARY
    with pytest.raises(a3.A3Error) as e:
        a3.Detector(a3.DetectorConfig(threshold_window=0))
    assert e.value.status == _ffi.A3_ERR_INVALID_ARGUMENT
    with pytest.raises(a3.A3Error):
        a3.Detector(a3.DetectorConfig(contour_simplification_epsilon=0.0))
    for shape in ((0, 480, 640), (1, 480, 0), (1, 0, 640)):  # a candidate but no grey to decode it on
        with pytest.raises(a3.A3Error) as e:
            det.decode_candidates(np.zeros(shape, np.uint8), np.zeros((1, 8), np.uint32))
        assert e.value.status == _ffi.A3_ERR_INVALID_ARGUMENT
    imgs, _ = synth.render_batch("C1", 1)
    markers = (_ffi.A3Marker * 1)()
    n = C.c_uint32()
    st = _ffi.lib().a3_detect_batch(det._h, imgs.ctypes.data, _ffi.FMT_RGB8, _ffi.MEM_HOST, 1, 640, 480, 1920, 1920 * 480,
                                    C.cast(markers, C.c_void_p), 1, C.byref(n), None, None)
    assert st == _ffi.A3_ERR_CAPACITY and n.value > 1


def test_probes_leave_the_pipeline_alone(a3):
    """Every stage probe between two a3_detect_batch calls of one handle with every post-decode stage on: the probes keep
    their inputs and outputs apart from the pipeline's buffers, so the second call returns every byte the first did."""
    from aruco3_b200 import synth
    from tests.test_gpu_board import _detect_all
    frames, _ = synth.render_batch("C3", 3)
    n, h, w = frames.shape[:3]
    k = a3.CameraIntrinsics(w, h, 1400.0, 1400.0, w / 2, h / 2)
    board = a3.Board.grid(6, 4, 40.0, 10.0)
    rng = np.random.default_rng(8)
    grey = rng.integers(0, 256, (2, 240, 320), np.uint8)
    cx, cy, s = rng.integers(0, 270, 30), rng.integers(0, 190, 30), rng.integers(8, 48, 30)
    quads = np.stack([cx, cy, cx + s, cy, cx + s, cy + s, cx, cy + s], 1).astype(np.uint32)
    qf = np.sort(rng.integers(0, 2, 30)).astype(np.uint32)
    with a3.Detector(corners="refined") as d:
        d.set_pose(40.0, k)
        d.set_board(board, k)
        d.set_distortion(a3.CameraDistortion(-0.1, 0.02, 0.0, 0.0, 0.0))
        first = _detect_all(a3, d, frames, full=True)
        d.decode_candidates(grey, quads, qf)
        d.refine_corners(grey, quads, qf)
        d.quads_from_masks_device(rng.integers(0, 2, (2, 150, 200), np.uint8) * 255)
        d.undistort_points(rng.uniform(0, 320, (50, 2)), k, a3.CameraDistortion(0.05, 0.0, 0.001, 0.0, 0.0))
        d.solve_board(board.ids[rng.integers(0, len(board), 30)], quads.astype(np.float32), qf, 2, image_size=(320, 240))
        a3.pose.solve_with_intrinsics(d, quads, 40.0, k)
        a3.pose.solve_with_undistorted_points(d, quads, 40.0, (320, 240))
        a3.pose.solve_with_normalized_points(d, quads.astype(np.float32) / 1000, 40.0)
        second = _detect_all(a3, d, frames, full=True)
    data, status, n_cands, n_markers, _ = first
    assert status == 0 and n_markers > 0
    # the counters are left out: they name the route, and the K3 probe replaces the size history the one-shot route reads
    assert second[:4] == (data, status, n_cands, n_markers)


def test_full_size_batch_properties(a3):
    """BASELINE.json configs[2] at full size (256 x 1080p, 20 markers each): size-independent properties against the
    rendered ground truth — the statistics the oracle itself shows on these scenes (recall 94 %, 0.25 % misread ids,
    median corner error 2.7 px: RDP epsilon is 5 % of the contour length) — and the chunking / sharding invariant:
    any sub-batch gives the same per-frame results."""
    from aruco3_b200 import synth
    n = 256
    frames, truth = synth.render_batch("C3", n)
    with a3.Detector(dictionary="ARUCO") as d:
        got = d.detect_batch(frames)
        assert d.last_stats["n_frames"] == n
        part = d.detect_batch(frames[37:41])
    found = wanted = false = 0
    errs = []
    for f in range(n):
        have, want = Counter(m.id for m in got[f].markers), Counter(t.id for t in truth[f])
        false += sum((have - want).values())
        found += sum((have & want).values())
        wanted += sum(want.values())
        for m in got[f].markers:  # corners[0] is the marker's own top-left (Q9); ids may repeat within a frame
            cand = [np.abs(np.array(m.corners, float) - t.corners).max() for t in truth[f] if t.id == m.id]
            if cand:
                errs.append(min(cand))
    assert found >= 0.88 * wanted, f"recall {found}/{wanted}"
    assert false <= 0.01 * found, f"{false} misread ids of {found}"
    assert np.median(errs) <= 5.0 and np.percentile(errs, 99) <= 30.0, f"corner error {np.percentile(errs, [50, 99, 100])}"
    assert [[(m.id, m.corners) for m in x.markers] for x in part] == [[(m.id, m.corners) for m in x.markers] for x in got[37:41]]


@pytest.mark.parametrize("contours,nframes", [("device", 7), ("host", 7), ("device", 64), ("device", 131)])
def test_resident_input_equals_host_input(a3, contours, nframes):
    """a3_detect_batch with A3_MEM_DEVICE (frames already in HBM, the flavour bench.py's `value` times) returns the same
    markers and counters as the host-pointer flavour (which runs K1 / K3 / K2 per chunk of frames, while resident input
    runs each once over the batch); the 131-frame case also carries pose output."""
    torch = pytest.importorskip("torch")
    from aruco3_b200 import _ffi, synth
    frames, _ = synth.render_batch("C1" if nframes != 64 else "C1n", nframes)
    n, h, w = frames.shape[:3]
    cap = 64 * n + 4096
    with a3.Detector(contours=contours) as d:
        if nframes == 131:
            d.set_pose(40.0)
        want = d.detect_batch(frames)
        want_stats = dict(d.last_stats)
        dev = torch.from_numpy(frames).cuda()
        markers = (_ffi.A3Marker * cap)()
        nm = C.c_uint32()
        st = _ffi.A3Stats()
        outs = _ffi.A3Outputs()
        poses = (_ffi.A3Pose * (2 * cap))()
        outs.marker_poses = C.cast(poses, C.c_void_p).value
        for _ in range(2):  # twice: the second call reuses every buffer of the first
            _ffi.check(_ffi.lib().a3_detect_batch(d._h, dev.data_ptr(), _ffi.FMT_RGB8, _ffi.MEM_DEVICE, n, w, h, w * 3, w * h * 3,
                                                  C.cast(markers, C.c_void_p), cap, C.byref(nm), C.byref(outs), C.byref(st)))
    if nframes == 131:
        k = 0
        for x in want:
            for m in x.markers:
                assert bytes(poses[2 * k]) == bytes(m.poses[0].to_c()) and bytes(poses[2 * k + 1]) == bytes(m.poses[1].to_c())
                k += 1
        assert k == nm.value
    got = [[] for _ in range(n)]
    for i in range(nm.value):
        m = markers[i]
        got[m.frame].append((int(m.id), int(m.rotation), int(m.hamming_distance), [int(v) for v in m.corners]))
    assert got == [[(m.id, m.rotation, m.hamming_distance, [v for c in m.corners for v in c]) for m in x.markers] for x in want]
    for k in ("n_contours", "n_contour_points", "n_candidates", "n_markers"):
        assert getattr(st, k) == want_stats[k], k


@pytest.mark.parametrize("channels", [1, 4])
def test_detect_other_pixel_formats(a3, oracle, channels):
    """Luma8 passes through into_luma8 unchanged and Rgba8 ignores alpha (SURVEY A.1) — through the whole path."""
    from aruco3_b200 import synth
    rgb, _ = synth.render_batch("C1", 2)
    if channels == 1:
        imgs = np.stack([oracle.to_luma8(f) for f in rgb])
    else:
        imgs = np.concatenate([rgb, np.full(rgb.shape[:3] + (1,), 77, np.uint8)], axis=3)
    with a3.Detector() as d:
        got = d.detect_batch(imgs, full=True, want_mask=True)
    for f in range(2):
        _check_detection(got[f], oracle.detect(imgs[f], "ARUCO"), f"{channels}ch[{f}]")


def _widen(rgb8, kind, seed):
    """An Rgb8 batch as one of the other integer DynamicImage variants; 16-bit subpixels = v * 257 + noise in the low byte
    region, so the 16 -> 8 bit rounding is exercised on both sides of every step."""
    rng = np.random.default_rng(seed)
    n, h, w, _ = rgb8.shape
    wide = rgb8.astype(np.int32) * 257 + rng.integers(-128, 129, size=rgb8.shape)
    rgb16 = np.clip(wide, 0, 65535).astype(np.uint16)
    if kind == "rgb16":
        return rgb16
    if kind == "rgba16":
        return np.concatenate([rgb16, rng.integers(0, 65536, size=(n, h, w, 1), dtype=np.uint16)], axis=3)
    if kind == "luma16":
        return np.ascontiguousarray(rgb16[..., 1])
    if kind == "lumaa16":
        return np.stack([rgb16[..., 1], rng.integers(0, 65536, size=(n, h, w), dtype=np.uint16)], axis=3)
    if kind == "lumaa8":
        return np.stack([rgb8[..., 1], rng.integers(0, 256, size=(n, h, w), dtype=np.uint8)], axis=3)
    raise KeyError(kind)


@pytest.mark.parametrize("kind", ["lumaa8", "luma16", "lumaa16", "rgb16", "rgba16"])
def test_detect_wide_pixel_formats(a3, oracle, kind):
    """SURVEY §8 f-4: the other integer DynamicImage variants (kernel K0 = image 0.25's into_luma8 for them, recalled
    semantics — upstream parity unpinned — then the usual path): grey, mask, candidates, patches and markers equal the
    oracle's, for a 640x480 batch (warp-strip K1 behind K0) and an odd-sized one (generic K1 behind K0)."""
    from aruco3_b200 import synth
    rgb, _ = synth.render_batch("C1", 3)
    for imgs in (_widen(rgb, kind, 11), _widen(np.ascontiguousarray(rgb[:2, :277, :401]), kind, 12)):
        with a3.Detector() as d:
            got = d.detect_batch(imgs, full=True, want_mask=True)
            g, m = d.gray_threshold(imgs)
        for f in range(len(imgs)):
            ref = oracle.detect(imgs[f], "ARUCO")
            _check_detection(got[f], ref, f"{kind}[{f}] {imgs.shape}")
            assert np.array_equal(g[f], ref.grey) and np.array_equal(m[f], ref.mask)
        if imgs.shape[2] == 640:
            assert sum(len(x.markers) for x in got) >= 10


def test_detect_4k_frame(a3, oracle):
    """BASELINE.json configs[3] frame size (3840 x 2160), one frame, every intermediate against the oracle."""
    from aruco3_b200 import synth
    img, _ = synth.render_frame(synth.CONFIGS["C4"], 0)
    with a3.Detector() as d:
        got = d.detect_batch(img[None], full=True, want_mask=True)[0]
    _check_detection(got, oracle.detect(img, "ARUCO"), "C4[0]")
    assert len(got.markers) >= 18


def test_detect_4k_batch_in_chunks(a3, oracle):
    """BASELINE.json configs[3] frames (3840 x 2160) as a batch: host input is staged 3 frames (~96 MB) per front-end
    chunk, so 5 frames cross chunk boundaries; markers of every frame equal the oracle's and do not depend on the batch."""
    from aruco3_b200 import synth
    frames, _ = synth.render_batch("C4", 5)
    with a3.Detector() as d:
        got = d.detect_batch(frames)
        assert d.last_stats["pixel_kernel_launches"] >= 2
        alone = d.detect_batch(frames[3:4])
    for f in (0, 2, 4):
        ref = oracle.detect(frames[f], "ARUCO")
        gm = [(m.candidate, m.id, m.rotation, m.hamming_distance, m.code, [v for c in m.corners for v in c]) for m in got[f].markers]
        rm = [(m["candidate"], m["id"], m["rotation"], m["hamming_distance"], m["code"], m["corners"]) for m in ref.markers]
        assert gm == rm, f"C4[{f}]"
    assert [(m.id, m.corners) for m in alone[0].markers] == [(m.id, m.corners) for m in got[3].markers]


def test_decode_stress_batch(a3, oracle):
    """BASELINE.json configs[4]: AprilTag 36h11 frames with 200+ small markers each (more than the 64 quads per frame the
    pipeline copies back unconditionally), several frames per batch."""
    from aruco3_b200 import synth
    spec = synth.CONFIGS["C5"]
    frames, _ = synth.render_batch(spec, 3)
    cfg = a3.DetectorConfig(min_corner_separation_factor=spec.min_corner_separation_factor)
    ocfg = oracle.default_config(min_corner_separation_factor=spec.min_corner_separation_factor)
    with a3.Detector(cfg, spec.dictionary) as d:
        got = d.detect_batch(frames)
    for f in range(3):
        ref = oracle.detect(frames[f], spec.dictionary, ocfg)
        gm = [(m.candidate, m.id, m.rotation, m.hamming_distance, m.code, [v for c in m.corners for v in c]) for m in got[f].markers]
        rm = [(m["candidate"], m["id"], m["rotation"], m["hamming_distance"], m["code"], m["corners"]) for m in ref.markers]
        assert gm == rm and len(gm) >= 150, f"C5[{f}]: {len(gm)} markers"


@pytest.mark.parametrize("dict_name,hs", [("ARUCO", 49), ("APRILTAG_16H5", 49), ("CHILITAGS", 49), ("APRILTAG_36H11", 32), ("ARUCO_MIP_36H12", 77),
                                          ("ARUCO", 200), ("APRILTAG_36H9", 300)])
def test_decode_fuzz(a3, oracle, dict_name, hs):
    """K2 against the oracle on 1500 arbitrary quads (any four points: rotated, concave, tiny, huge, partly outside) over a
    smooth and a noisy frame, for mark sizes 6 / 7 / 8 / 10 and other homography_sample_size values: projection class and
    failure, every patch byte, Otsu level, the four codes, the match (id, rotation, distance) and acceptance."""
    rng = np.random.default_rng(hash((dict_name, hs)) & 0xffff)
    w, h = 352, 288
    grey = np.stack([_smooth(5, 1, h, w, 1)[0, :, :, 0], _noise(6, (h, w))])
    n = 1500 if hs <= 100 else 160  # large homography_sample_size: fewer warps per CTA share the shared memory (k2_decode.cu)
    kind = rng.integers(0, 4, n)
    quads = np.zeros((n, 8), np.int64)
    for k in range(n):
        if kind[k] == 0:    # any four points
            q = np.stack([rng.integers(0, w, 4), rng.integers(0, h, 4)], 1)
        elif kind[k] == 1:  # rotated square with jitter
            c, sd, a = rng.uniform([20, 20], [w - 20, h - 20]), rng.uniform(3, 120), rng.uniform(0, 2 * np.pi)
            base = np.array([[-1, -1], [1, -1], [1, 1], [-1, 1]]) * sd
            rot = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
            q = c + base @ rot.T + rng.uniform(-0.2, 0.2, (4, 2)) * sd
        elif kind[k] == 2:  # thin sliver
            x0, y0 = rng.integers(0, w - 2), rng.integers(0, h - 2)
            q = np.array([[x0, y0], [x0 + rng.integers(1, w), y0 + 1], [x0 + rng.integers(1, w), y0 + 2], [x0, y0 + 1]])
        else:               # axis-aligned rectangle touching the frame edges
            x1, y1 = rng.integers(1, w), rng.integers(1, h)
            q = np.array([[0, 0], [x1, 0], [x1, y1], [0, y1]]) + rng.integers(0, 2, 2) * [w - 1 - x1, h - 1 - y1]
        quads[k] = np.clip(np.rint(q), 0, [w - 1, h - 1]).astype(np.int64).ravel()
    quads = quads.astype(np.uint32)
    qf = rng.integers(0, 2, n).astype(np.uint32)
    dic = oracle.dictionary(dict_name)
    ms = oracle.lib().a3ref_mark_size(C.byref(dic))
    with a3.Detector(a3.DetectorConfig(homography_sample_size=hs), dict_name) as d:
        decs, patches = d.decode_candidates(grey, quads, qf)
    L = oracle.lib()
    accepted = 0
    for k in range(n):
        patch = np.zeros((hs, hs), np.uint8)
        g = np.ascontiguousarray(grey[qf[k]])
        qk = np.ascontiguousarray(quads[k])
        ok = L.a3ref_extract_homography(g.ctypes.data, w, h, qk.ctypes.data, hs, patch.ctypes.data)
        assert bool(ok) == decs[k]["homography_ok"], f"quad {k} {quads[k].tolist()}: homography_ok"
        assert np.array_equal(patches[k], patch), f"quad {k} {quads[k].tolist()}: patch"
        codes, otsu = (C.c_uint64 * 4)(), C.c_uint8()
        src = patch if ok else np.zeros((1, 1), np.uint8)
        some = L.a3ref_homography_to_code_permutations(src.ctypes.data, src.shape[1], src.shape[0], ms, codes, C.byref(otsu), None)
        assert decs[k]["otsu"] == otsu.value and decs[k]["has_codes"] == bool(some), f"quad {k}: otsu / has_codes"
        if not some:
            assert not decs[k]["accepted"]
            continue
        assert decs[k]["codes"] == list(codes), f"quad {k}: codes"
        best, best_r, best_i = 255, 0, 0  # the match loop of src/aruco.rs:75-96
        for r in range(4):
            i, dist = oracle.find_nearest(dic, codes[r])
            if dist < best:
                best, best_r, best_i = dist, r, i
        assert (decs[k]["hamming_distance"], decs[k]["rotation"], decs[k]["id"]) == (best, best_r, best_i), f"quad {k}: match"
        assert decs[k]["accepted"] == (best < dic.tau)
        accepted += decs[k]["accepted"]
    assert sum(d_["homography_ok"] for d_ in decs) > n // 2


@pytest.mark.parametrize("w,h,side,noise,dict_name", [(333, 251, (24, 60), 0, "ARUCO"), (97, 131, (20, 40), 3, "ARUCO"),
                                                      (1282, 722, (40, 150), 6, "APRILTAG_25H9"), (1000, 37, (16, 30), 0, "ARUCO"),
                                                      (501, 499, (30, 90), 12, "ARUCO_MIP_25H7"), (2049, 65, (20, 50), 2, "ARTOOLKITPLUS")])
def test_detect_fuzz_sizes(a3, oracle, w, h, side, noise, dict_name):
    """Whole path on frame sizes that take the generic pixel kernel (widths that are not multiples of 4, strips narrower
    than a warp, one-strip-high frames), several noise levels and dictionaries, RGB and RGBA: every intermediate equals
    the oracle's."""
    from aruco3_b200 import synth
    spec = synth.FrameSpec(f"fuzz{w}x{h}", 7, w, h, dictionary=dict_name, markers=(1, 6), side=side, noise=noise)
    frames, _ = synth.render_batch(spec, 4)
    with a3.Detector(dictionary=dict_name) as d:
        got = d.detect_batch(frames, full=True, want_mask=True)
        rgba = np.concatenate([frames, np.full(frames.shape[:3] + (1,), 7, np.uint8)], axis=3)
        got4 = d.detect_batch(rgba)
    total = 0
    for f in range(frames.shape[0]):
        ref = oracle.detect(frames[f], dict_name)
        _check_detection(got[f], ref, f"{w}x{h}[{f}]")
        assert [(m.id, m.corners, m.rotation) for m in got4[f].markers] == [(m.id, m.corners, m.rotation) for m in got[f].markers]
        total += len(ref.candidates)
    assert total > 0
