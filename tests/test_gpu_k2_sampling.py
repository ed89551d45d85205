"""K2's bilinear sampling against the oracle at the places where its arithmetic is easiest to get wrong: samples exactly on
the last column / row of the frame and just inside it, quads partly or wholly outside the frame, projections that give
+-inf or NaN sample coordinates, patch sizes around the warp width (the column / row stepping), frame widths that are and
are not multiples of 4, random and flat grey.  Every patch byte, the Otsu level, the four codes, the match and acceptance
are compared with oracle/a3ref.c, in both forms of the kernel (a CTA per candidate for small calls, a warp per candidate
for large ones)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# a3_decode_candidates calls of at most 3 x (number of SMs) quads take the CTA-per-candidate form, larger ones the warp form
# (k2_decode.cu); the two sizes below are on either side of that for any B200 part
SMALL, LARGE = 256, 1200


@pytest.fixture(scope="module")
def a3():
    import aruco3_b200
    from aruco3_b200 import _ffi
    if _ffi.lib().a3_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tests have no fallback")
    return aruco3_b200


def _sample_coords(oracle, quad, hs):
    """The sample coordinates (px, py) of warp_into in f32, in the oracle's operation order, or None when the projection fails."""
    fr = np.asarray(quad, np.float64).astype(np.float32)
    to = np.array([0, 0, hs, 0, hs, hs, 0, hs], np.float32)
    fwd, inv, cls = np.zeros(9, np.float32), np.zeros(9, np.float32), C.c_int()
    if not oracle.lib().a3ref_projection_from_control_points(fr.ctypes.data, to.ctypes.data, fwd.ctypes.data, inv.ctypes.data,
                                                            C.byref(cls)):
        return None
    oy, ox = np.mgrid[0:hs, 0:hs].astype(np.float32)
    t = inv
    with np.errstate(all="ignore"):
        if cls.value == 2:
            d = t[6] * ox + t[7] * oy + t[8]
            return (t[0] * ox + t[1] * oy + t[2]) / d, (t[3] * ox + t[4] * oy + t[5]) / d
        if cls.value == 1:
            return t[0] * ox + t[1] * oy + t[2], t[3] * ox + t[4] * oy + t[5]
        return ox + t[2], oy + t[5]


def _quads(oracle, rng, w, h, hs):
    qs = []
    # squares of side hs (translations) and 2 hs / hs / 2 (affine, integer and half-integer steps) whose last column or row
    # lands on x = w - 1 / y = h - 1 (outside: right = w) or one step before it (inside)
    for side in (hs, 2 * hs, max(hs // 2, 1)):
        span = side * (hs - 1) / hs
        for dx in (-1, 0, 1):
            for dy in (-1, 0, 1):
                x0 = int(np.floor(w - 1 - span)) + dx
                y0 = int(np.floor(h - 1 - span)) + dy
                if x0 >= 0 and y0 >= 0:
                    qs.append([x0, y0, x0 + side, y0, x0 + side, y0 + side, x0, y0 + side])
    for _ in range(40):  # rotated squares across the right or bottom edge
        c = rng.uniform([w - 30, h / 2], [w + 10, h / 2 + 1]) if rng.integers(2) else rng.uniform([w / 2, h - 30], [w / 2 + 1, h + 10])
        sd, a = rng.uniform(4, 40), rng.uniform(0, 2 * np.pi)
        rot = np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
        qs.append(np.rint(c + np.array([[-1, -1], [1, -1], [1, 1], [-1, 1]]) * sd @ rot.T).clip(0).ravel().tolist())
    for _ in range(40):  # partly outside
        qs.append(rng.integers(0, [2 * w, 2 * h] * 4).tolist())
    for _ in range(20):  # wholly outside
        qs.append(rng.integers([w, h] * 4, [3 * w, 3 * h] * 4).tolist())
    for _ in range(60):  # inside, any four points
        qs.append(rng.integers(0, [w, h] * 4).tolist())
    # extreme corners: many of these solve and then project samples to +-inf or NaN; take up to 8 of each kind first
    special = np.array([0, 1, 2, 3, 5, 8, 13, 2**24, 2**24 + 1, 2**31, 2**32 - 1], np.uint64)
    n_inf = n_nan = 0
    for _ in range(20000):
        if n_inf >= 8 and n_nan >= 8:
            break
        q = rng.choice(special, 8)
        r = _sample_coords(oracle, q, hs)
        if r is None:
            continue
        has_inf, has_nan = (np.isinf(r[0]) | np.isinf(r[1])).any(), (np.isnan(r[0]) | np.isnan(r[1])).any()
        if (has_inf and n_inf < 8) or (has_nan and n_nan < 8):
            qs.append(q.tolist())
            n_inf += int(has_inf)
            n_nan += int(has_nan)
    while len(qs) < SMALL:
        qs.append(rng.choice(special, 8).tolist())
    return np.array(qs, np.uint64).astype(np.uint32)


@pytest.mark.parametrize("content", ["random", "flat"])
@pytest.mark.parametrize("w,h", [(160, 120), (157, 117)])
@pytest.mark.parametrize("hs", [7, 31, 32, 33, 49, 100])
def test_k2_sampling_edges(a3, oracle, hs, w, h, content):
    rng = np.random.default_rng(hs * 1000 + w)
    if content == "random":
        grey = rng.integers(0, 256, (2, h, w), dtype=np.uint8)
    else:  # one bin of the histogram (plus 0 for samples outside the frame)
        grey = np.stack([np.full((h, w), 200, np.uint8), np.full((h, w), 17, np.uint8)])
    quads = _quads(oracle, rng, w, h, hs)
    qf = rng.integers(0, 2, len(quads)).astype(np.uint32)

    # what the quads exercise, from the oracle's own f32 sample coordinates
    seen = dict(on_edge=0, below_edge=0, inf=0, nan=0)
    for q in quads:
        r = _sample_coords(oracle, q, hs)
        if r is None:
            continue
        px, py = r
        seen["on_edge"] += int(((px == w - 1) & (py >= 0) & (py < h - 1)).sum() + ((py == h - 1) & (px >= 0) & (px < w - 1)).sum())
        seen["below_edge"] += int(((px >= w - 2) & (px < w - 1) & (py >= 0) & (py < h - 1)).sum()
                                  + ((py >= h - 2) & (py < h - 1) & (px >= 0) & (px < w - 1)).sum())
        seen["inf"] += int((np.isinf(px) | np.isinf(py)).sum())
        seen["nan"] += int((np.isnan(px) | np.isnan(py)).sum())
    assert all(seen.values()), seen

    dict_name = "ARUCO"
    dic = oracle.dictionary(dict_name)
    ms = oracle.lib().a3ref_mark_size(C.byref(dic))
    L = oracle.lib()
    want = []
    for k in range(len(quads)):
        patch = np.zeros((hs, hs), np.uint8)
        g = np.ascontiguousarray(grey[qf[k]])
        qk = np.ascontiguousarray(quads[k])
        ok = L.a3ref_extract_homography(g.ctypes.data, w, h, qk.ctypes.data, hs, patch.ctypes.data)
        codes, otsu = (C.c_uint64 * 4)(), C.c_uint8()
        src = patch if ok else np.zeros((1, 1), np.uint8)
        some = L.a3ref_homography_to_code_permutations(src.ctypes.data, src.shape[1], src.shape[0], ms, codes, C.byref(otsu), None)
        match = None
        if some:
            best, best_r, best_i = 255, 0, 0  # the match loop of src/aruco.rs:75-96
            for r in range(4):
                i, dist = oracle.find_nearest(dic, codes[r])
                if dist < best:
                    best, best_r, best_i = dist, r, i
            match = (best, best_r, best_i, best < dic.tau)
        want.append((bool(ok), patch, otsu.value, bool(some), list(codes), match))

    reps = LARGE // len(quads) + 1
    with a3.Detector(a3.DetectorConfig(homography_sample_size=hs), dict_name) as d:
        for form, n in (("cta", 1), ("warp", reps)):
            decs, patches = d.decode_candidates(grey, np.tile(quads, (n, 1)), np.tile(qf, n))
            for j in range(len(decs)):
                k = j % len(quads)
                ok, patch, otsu, some, codes, match = want[k]
                tag = f"{form} form, quad {k} {quads[k].tolist()}"
                assert decs[j]["homography_ok"] == ok, f"{tag}: homography_ok"
                assert np.array_equal(patches[j], patch), f"{tag}: patch"
                assert decs[j]["otsu"] == otsu and decs[j]["has_codes"] == some, f"{tag}: otsu / has_codes"
                if not some:
                    assert not decs[j]["accepted"], tag
                    continue
                assert decs[j]["codes"] == codes, f"{tag}: codes"
                got = (decs[j]["hamming_distance"], decs[j]["rotation"], decs[j]["id"], decs[j]["accepted"])
                assert got == match, f"{tag}: match"
