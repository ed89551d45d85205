"""Input frames laid out as callers have them: rows wider than their pixels, gaps between frames, crops of a larger image,
base pointers at any byte offset.  a3_gray_threshold_batch and a3_detect_batch take `pitch` (bytes per row) and
`frame_stride` (bytes between frames) and must honour both; the layout only chooses the pixel stage's code path:

  strips      warp-strip K1 (k1_strips.cu), a 3-D tensor map over [n][h][pitch / 4]: radius 7, w % 4 == 0, pitch,
              frame_stride and the base 16-byte multiples, frame_stride a multiple of pitch, grey and mask 4-byte aligned
  bulk rows   generic K1 (k1_threshold.cu) staging rows with 1-D bulk copies: pitch, frame_stride, base and every strip's
              loaded span 16-byte multiples
  byte loads  generic K1 reading pixels byte by byte: anything else
  K0          LumaA8 and the 16-bit formats: converted into a padded Luma8 scratch first, reading u16 values byte by byte

Every byte of an input buffer that is not a pixel is poison: random bytes, different per seed, and the buffer ends with the
last pixel byte.  Each case runs with two poisons; both results must equal the CPU oracle on the tightly packed frames (so
they are byte-identical to each other), which catches a read of padding even where it happens not to change the mask.
Host input is copied to an aligned device slot first, so a host base offset exercises the copy only."""
import ctypes as C
import mmap
import signal
import subprocess
import sys
from functools import lru_cache
from pathlib import Path

import numpy as np
import pytest

from aruco3_b200 import _ffi

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent

# name: (a3_format, channels (0: frames are [n, h, w]), subpixel type, byte order the oracle reads)
FORMATS = {
    "rgb8": (_ffi.FMT_RGB8, 3, np.uint8, "rgb"),
    "rgba8": (_ffi.FMT_RGBA8, 4, np.uint8, "rgb"),
    "luma8": (_ffi.FMT_LUMA8, 0, np.uint8, "rgb"),
    "bgr8": (_ffi.FMT_BGR8, 3, np.uint8, "bgr"),
    "bgra8": (_ffi.FMT_BGRA8, 4, np.uint8, "bgr"),
    "lumaa8": (_ffi.FMT_LUMAA8, 2, np.uint8, "rgb"),
    "luma16": (_ffi.FMT_LUMA16, 0, np.uint16, "rgb"),
    "lumaa16": (_ffi.FMT_LUMAA16, 2, np.uint16, "rgb"),
    "rgb16": (_ffi.FMT_RGB16, 3, np.uint16, "rgb"),
    "rgba16": (_ffi.FMT_RGBA16, 4, np.uint16, "rgb"),
}
WIDE = ("lumaa8", "luma16", "lumaa16", "rgb16", "rgba16")
# frames of the pixel-stage cases: W * bpp is a 16-byte multiple for every 8-bit format, and W < 225 keeps the generic
# kernel to one strip, so that the layout alone decides between bulk rows and byte loads
N, H, W = 3, 72, 160
LAYOUTS = ("tight", "pitch16", "pitch_odd", "gap_rows", "gap16", "crop16", "crop_odd", "base+1", "base+4", "base+8", "base+16")
TUNINGS = {"auto": {}, "generic": {"force_generic": 1}, "no_tma": {"force_no_tma": 1}}
SENTINEL = 0x5A  # fills the bytes around every output buffer; they must survive the call

MARKER = np.dtype([("id", "<u8"), ("code", "<u8"), ("corners", "<u4", 8), ("frame", "<u4"), ("candidate", "<u4"),
                   ("hamming_distance", "u1"), ("rotation", "u1"), ("corners_refined", "u1"), ("reserved", "u1", 5)])
assert MARKER.itemsize == C.sizeof(_ffi.A3Marker)


@pytest.fixture(scope="module")
def a3():
    import aruco3_b200
    if _ffi.lib().a3_device_count() < 1:
        pytest.fail("no CUDA device visible: the gpu tests have no fallback")
    return aruco3_b200


@pytest.fixture(scope="module")
def torch(a3):
    return pytest.importorskip("torch")  # plumbing only: device and page-locked buffers


@pytest.fixture(scope="module")
def det(a3):
    with a3.Detector() as d:
        yield d


def _up(v, m):
    return (v + m - 1) // m * m


def _bpp(fmt):
    _, ch, dt, _ = FORMATS[fmt]
    return max(ch, 1) * np.dtype(dt).itemsize


def embed(frames, pitch, frame_stride, offset, poison_seed, out=None):
    """Tight frames [n, h, w(, c)] -> a byte buffer holding them at `offset`, rows `pitch` and frames `frame_stride` bytes
    apart.  The buffer ends with the last pixel byte; every byte that is not a pixel is random poison.  `out`: fill this
    buffer (of exactly that size) instead of a new one."""
    n, h = frames.shape[:2]
    raw = np.ascontiguousarray(frames).view(np.uint8).reshape(n, h, -1)
    row = raw.shape[2]
    size = offset + (n - 1) * frame_stride + (h - 1) * pitch + row
    buf = np.empty(size, np.uint8) if out is None else out
    assert buf.size == size
    buf[...] = np.random.default_rng(poison_seed).integers(0, 256, size, dtype=np.uint8)
    np.lib.stride_tricks.as_strided(buf[offset:], (n, h, row), (frame_stride, pitch, 1))[...] = raw
    return buf


def _layout(name, bpp, w=W, h=H):
    """-> (pitch, frame_stride, base offset) of a named layout."""
    row = w * bpp
    if name == "tight":
        return row, row * h, 0
    if name in ("pitch16", "pitch_odd"):  # padded rows: a 16-byte multiple, or not even that
        p = _up(row, 16) + 64 if name == "pitch16" else row + 5
        return p, p * h, 0
    if name == "gap_rows":  # three spare rows after each frame: frame_stride still a multiple of pitch
        return row, row * (h + 3), 0
    if name == "gap16":  # 16 spare bytes after each frame: a 16-byte multiple, not a multiple of pitch
        return row, row * h + 16, 0
    if name in ("crop16", "crop_odd"):  # the bottom-right w x h of a larger frame: pitch and stride are the parent's
        pw, ph = (w + 96, h + 5) if name == "crop16" else (w + 37, h + 11)
        p = pw * bpp
        return p, p * ph, (ph - h) * p + (pw - w) * bpp
    if name.startswith("base+"):
        return row, row * h, int(name[5:])
    raise KeyError(name)


def _pixel_path(fmt, layout, mem, radius=7, tuning="auto", out_off=0, grey=True):
    """The code path a3_gray_threshold_batch takes for a case (k1_strips_eligible in k1_strips.cu, the bulk-copy rule of
    k1_gray_threshold in k1_threshold.cu) — for the failure messages and the coverage check of the layout table."""
    if fmt in WIDE:
        return "K0"
    bpp = _bpp(fmt)
    pitch, fs, off = _layout(layout, bpp)
    src = off if mem == "device" else 0
    a16 = pitch % 16 == 0 and fs % 16 == 0 and src % 16 == 0
    if tuning != "generic" and radius == 7 and grey and W % 4 == 0 and a16 and fs % pitch == 0 and out_off % 4 == 0:
        return "strips"
    if tuning != "no_tma" and a16 and W * bpp % 16 == 0:
        return "bulk rows"
    return "byte loads"


def _frames(fmt, seed=1, n=N, h=H, w=W):
    _, ch, dt, _ = FORMATS[fmt]
    shape = (n, h, w) + ((ch,) if ch else ())
    return np.random.default_rng(seed).integers(0, np.iinfo(dt).max + 1, size=shape, dtype=dt)


def _words(w):
    return (w + 31) // 32


def _bits_of(mask):
    """Mask [h, w] (0 / 255) -> mask bits [h, ceil(w / 32)] u32: bit (x & 31) of word x >> 5."""
    h, w = mask.shape
    padded = np.zeros((h, 32 * _words(w)), np.uint8)
    padded[:, :w] = mask > 0
    return np.packbits(padded, axis=1, bitorder="little").view("<u4")


@lru_cache(maxsize=None)
def _reference(fmt, radius=7):
    """The CPU oracle on the tight frames: grey, mask and mask bits [N, ...]."""
    from oracle import a3ref_py as oracle
    frames = _frames(fmt)
    order = FORMATS[fmt][3]
    grey = np.stack([oracle.to_luma8(f, order=order) for f in frames])
    mask = np.stack([oracle.adaptive_threshold(g, radius) for g in grey])
    return grey, mask, np.stack([_bits_of(m) for m in mask])


class _Tuning:
    """a3_detector_set_k1_tuning for the duration of a `with` block."""

    def __init__(self, det, **kw):
        self.det, self.t = det, _ffi.A3K1Tuning(**kw)

    def __enter__(self):
        _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(self.det._h, C.byref(self.t)))

    def __exit__(self, *exc):
        _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(self.det._h, None))


def _input(torch, buf, mem):
    """The poisoned buffer where the call reads it: `(pointer to buf[0], keep-alive)`.  Pinned and device copies have
    exactly the buffer's size."""
    if mem == "pageable":
        return buf.ctypes.data, buf
    if mem == "pinned":
        t = torch.empty(buf.size, dtype=torch.uint8, pin_memory=True)
        t.numpy()[...] = buf
        return t.data_ptr(), t
    assert mem == "device"
    t = torch.from_numpy(buf).cuda()
    return t.data_ptr(), t


def _gray_threshold(det, torch, buf, off, fmt, mem, pitch, fs, n=N, h=H, w=W, want=("grey", "mask", "bits"), out_off=0):
    """One a3_gray_threshold_batch call over `buf` (frames at byte `off`) -> {output: array}.  mem "host" (pageable input
    and outputs) or "device" (device input and outputs, on torch's stream).  Output i starts `out_off` bytes (the mask
    bits: the nearest 4-byte multiple below) into a sentinel-filled buffer; the sentinel bytes must survive."""
    sizes = {"grey": n * h * w, "mask": n * h * w, "bits": n * h * _words(w) * 4}
    offs = {"grey": out_off, "mask": out_off, "bits": out_off & ~3}
    pad = 64
    dev = mem == "device"
    outs, ptrs = {}, {}
    for k in ("grey", "mask", "bits"):
        if k in want:
            total = pad + offs[k] + sizes[k] + pad
            outs[k] = torch.full((total,), SENTINEL, dtype=torch.uint8, device="cuda") if dev else np.full(total, SENTINEL, np.uint8)
            ptrs[k] = (outs[k].data_ptr() if dev else outs[k].ctypes.data) + pad + offs[k]
        else:
            ptrs[k] = None
    src, keep = _input(torch, buf, "device" if dev else "pageable")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream) if dev else None
    _ffi.check(_ffi.lib().a3_gray_threshold_batch(det._h, src + off, FORMATS[fmt][0], _ffi.MEM_DEVICE if dev else _ffi.MEM_HOST,
                                                  n, w, h, pitch, fs, ptrs["grey"], ptrs["mask"], ptrs["bits"], stream))
    if dev:
        torch.cuda.synchronize()
    del keep
    res = {}
    for k, o in outs.items():
        a = o.cpu().numpy() if dev else o
        lo, hi = pad + offs[k], pad + offs[k] + sizes[k]
        assert (a[:lo] == SENTINEL).all() and (a[hi:] == SENTINEL).all(), f"{k}: bytes written outside the output buffer"
        body = a[lo:hi]
        res[k] = body.view("<u4").reshape(n, h, _words(w)) if k == "bits" else body.reshape(n, h, w)
    return res


def _check_pixels(res, want, label):
    for k, ref in zip(("grey", "mask", "bits"), want):
        if k in res:
            bad = np.argwhere(res[k] != ref)
            assert bad.size == 0, f"{label}: {k} differs at (frame, y, x) {bad[:5].tolist()}"


# ---- the pixel stage: a3_gray_threshold_batch ------------------------------------------------------------------------


def test_layout_table_reaches_every_pixel_path():
    """The layout table lands on each generic and warp-strip path for every 8-bit format, host and device input."""
    for fmt in FORMATS:
        if fmt not in WIDE:
            paths = {_pixel_path(fmt, lay, mem) for lay in LAYOUTS for mem in ("host", "device")}
            assert paths == {"strips", "bulk rows", "byte loads"}, (fmt, paths)
    assert _pixel_path("rgb8", "gap16", "host") == "bulk rows" and _pixel_path("rgb8", "crop16", "device") == "strips"


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("fmt", list(FORMATS))
def test_gray_threshold_layouts(det, torch, fmt, layout):
    """grey, mask and mask bits of every format and layout, host and device input, with the automatic kernel choice,
    the generic kernel forced and its bulk copies switched off: all equal the oracle on the tight frames.  Which path each
    case takes is in the failure message (`_pixel_path`); the 16-bit formats at an odd pitch (pitch_odd) and an odd base
    (base+1) hold K0 to reading u16 values at any alignment."""
    frames, want = _frames(fmt), _reference(fmt)
    pitch, fs, off = _layout(layout, _bpp(fmt))
    for seed in (1, 2):
        buf = embed(frames, pitch, fs, off, poison_seed=seed)
        for mem in ("host", "device"):
            for tuning, kw in TUNINGS.items():
                with _Tuning(det, **kw):
                    res = _gray_threshold(det, torch, buf, off, fmt, mem, pitch, fs)
                path = _pixel_path(fmt, layout, mem, tuning=tuning)
                _check_pixels(res, want, f"{fmt} {layout} ({path}) {mem} input, tuning {tuning}, poison {seed}")


@pytest.mark.parametrize("radius", [3, 17])
@pytest.mark.parametrize("fmt", ["rgb8", "luma8", "rgb16"])
def test_gray_threshold_layouts_other_radius(a3, torch, fmt, radius):
    """threshold_window != 7 always takes the generic kernel: bulk rows or byte loads by layout."""
    frames, want = _frames(fmt), _reference(fmt, radius)
    with a3.Detector(a3.DetectorConfig(threshold_window=radius)) as d:
        for layout in ("tight", "pitch_odd", "gap16", "crop_odd", "base+1", "base+16"):
            pitch, fs, off = _layout(layout, _bpp(fmt))
            buf = embed(frames, pitch, fs, off, poison_seed=3)
            for mem in ("host", "device"):
                for tuning in ("auto", "no_tma"):
                    with _Tuning(d, **TUNINGS[tuning]):
                        res = _gray_threshold(d, torch, buf, off, fmt, mem, pitch, fs)
                    path = _pixel_path(fmt, layout, mem, radius, tuning)
                    _check_pixels(res, want, f"r={radius} {fmt} {layout} ({path}) {mem} input, tuning {tuning}")


@pytest.mark.parametrize("out_off", [1, 2, 4])
@pytest.mark.parametrize("layout", ["tight", "crop16", "crop_odd"])
def test_gray_threshold_unaligned_device_outputs(det, torch, layout, out_off):
    """grey and mask at device addresses that are not 8-byte aligned: +4 keeps the warp-strip kernel (grey and mask 4-byte
    aligned) without its 8-byte stores; +1 and +2 make it ineligible, and the generic kernel then stores byte by byte
    (out_aligned false).  No byte outside the outputs may change."""
    fmt = "rgb8"
    frames, want = _frames(fmt), _reference(fmt)
    pitch, fs, off = _layout(layout, 3)
    buf = embed(frames, pitch, fs, off, poison_seed=4)
    for tuning, kw in TUNINGS.items():
        with _Tuning(det, **kw):
            res = _gray_threshold(det, torch, buf, off, fmt, "device", pitch, fs, out_off=out_off)
        path = _pixel_path(fmt, layout, "device", tuning=tuning, out_off=out_off)
        _check_pixels(res, want, f"outputs at +{out_off}, {layout} ({path}), tuning {tuning}")


@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("subset", [("grey",), ("mask",), ("bits",), ("mask", "bits"), ("grey", "bits")], ids="+".join)
def test_gray_threshold_output_subsets(det, torch, subset, mem):
    """"Any of the three outputs may be NULL" (include/aruco3_b200.h): each subset alone, on tight and strided input.
    Without grey the warp-strip kernel is ineligible and the generic kernel runs."""
    fmt = "rgb8"
    frames, want = _frames(fmt), _reference(fmt)
    for layout in ("tight", "crop16", "gap16"):
        pitch, fs, off = _layout(layout, 3)
        buf = embed(frames, pitch, fs, off, poison_seed=5)
        res = _gray_threshold(det, torch, buf, off, fmt, mem, pitch, fs, want=subset)
        assert sorted(res) == sorted(subset)
        path = _pixel_path(fmt, layout, mem, grey="grey" in subset)
        _check_pixels(res, want, f"outputs {subset}, {layout} ({path}), {mem}")


# ---- the whole path: a3_detect_batch ----------------------------------------------------------------------------------


@lru_cache(maxsize=None)
def _frameset(name):
    """Rendered marker frames [n, h, w, 3]: "c1" is BASELINE.json's 640 x 480 config (2 frames, 1.8 MB: pageable input is
    staged), "odd" an odd-sized one (3 frames of 301 x 211, < 1 MB: pageable input goes straight to the DMA)."""
    from aruco3_b200 import synth
    if name == "c1":
        frames, _ = synth.render_batch("C1", 2)
    else:
        frames, _ = synth.render_batch(synth.FrameSpec("odd301x211", 7, 301, 211, markers=(2, 4), side=(50, 80)), 3)
    frames.setflags(write=False)
    return frames


@lru_cache(maxsize=None)
def _oracle_detect(name):
    from oracle import a3ref_py as oracle
    refs = [oracle.detect(f, "ARUCO") for f in _frameset(name)]
    assert sum(len(r.markers) for r in refs) > 0
    return refs


def _detect_layout(name, w, h, bpp=3):
    row = w * bpp
    if name == "tight":
        return row, row * h, 0
    if name == "crop":  # bottom-right crop of a frame 37 columns and 11 rows larger
        p = (w + 37) * bpp
        return p, p * (h + 11), 11 * p + 37 * bpp
    if name == "gap":  # padded rows, and 48 bytes after each frame: not a multiple of the pitch
        p = _up(row, 16) + 16
        return p, p * h + 48, 0
    raise KeyError(name)


def _detect(det, ptr, mem, n, w, h, pitch, fs, full=True, pose=False, refine=False):
    """One a3_detect_batch call on RGB8 frames at `ptr` -> dict of its outputs (markers as MARKER records)."""
    cap, cap_c = 64 * n + 64, 256 * n
    markers = (_ffi.A3Marker * cap)()
    nm = C.c_uint32()
    st = _ffi.A3Stats()
    outs = _ffi.A3Outputs()
    res = {}
    if full:
        res["grey"] = np.full((n, h, w), SENTINEL, np.uint8)
        res["mask"] = np.full((n, h, w), SENTINEL, np.uint8)
        res["cands"] = np.zeros((cap_c, 8), np.uint32)
        res["cframe"] = np.zeros(cap_c, np.uint32)
        outs.grey, outs.mask = res["grey"].ctypes.data, res["mask"].ctypes.data
        outs.candidates, outs.candidate_frame = res["cands"].ctypes.data, res["cframe"].ctypes.data
        outs.cand_capacity = cap_c
    if pose:
        poses = (_ffi.A3Pose * (2 * cap))()
        outs.marker_poses = C.cast(poses, C.c_void_p).value
    if refine:
        corners = np.zeros((cap, 8), np.float32)
        outs.marker_corners = corners.ctypes.data
    _ffi.check(_ffi.lib().a3_detect_batch(det._h, ptr, _ffi.FMT_RGB8, _ffi.MEM_DEVICE if mem == "device" else _ffi.MEM_HOST, n, w, h,
                                          pitch, fs, C.cast(markers, C.c_void_p), cap, C.byref(nm), C.byref(outs), C.byref(st)))
    k = nm.value
    res["markers"] = np.frombuffer(bytes(markers)[:k * MARKER.itemsize], MARKER)
    res["stats"] = st.as_dict()
    if full:
        res["cands"], res["cframe"] = res["cands"][:outs.n_candidates], res["cframe"][:outs.n_candidates]
    if pose:
        res["poses"] = bytes(poses)[:2 * k * C.sizeof(_ffi.A3Pose)]
    if refine:
        res["corners"] = corners[:k].tobytes()
    return res


def _check_against_oracle(res, refs, label):
    for f, ref in enumerate(refs):
        assert np.array_equal(res["grey"][f], ref.grey), f"{label}: grey of frame {f}"
        assert np.array_equal(res["mask"][f], ref.mask), f"{label}: mask of frame {f}"
        assert res["cands"][res["cframe"] == f].tolist() == ref.candidates.tolist(), f"{label}: candidates of frame {f}"
        got = [(int(m["candidate"]), int(m["id"]), int(m["rotation"]), int(m["hamming_distance"]), int(m["code"]), m["corners"].tolist())
               for m in res["markers"][res["markers"]["frame"] == f]]
        want = [(m["candidate"], m["id"], m["rotation"], m["hamming_distance"], m["code"], m["corners"]) for m in ref.markers]
        assert got == want, f"{label}: markers of frame {f}"


@lru_cache(maxsize=None)
def _tight_records(name, variant):
    """Marker records (and poses / refined corners) of a fresh detector's call on the tight frames."""
    import aruco3_b200 as a3
    frames = _frameset(name)
    n, h, w = frames.shape[:3]
    with a3.Detector(**_VARIANTS[variant]["detector"]) as d:
        if _VARIANTS[variant].get("pose"):
            d.set_pose(40.0)
        tight = np.ascontiguousarray(frames)
        res = _detect(d, tight.ctypes.data, "pageable", n, w, h, w * 3, w * 3 * h, **_call_kw(variant))
    return res


_VARIANTS = {
    "default": {"detector": {}},
    "chunk1": {"detector": {}, "tuning": {"chunk_frames": 1}},
    "host_contours": {"detector": {"contours": "host"}},
    "refined_pose": {"detector": {"corners": "refined"}, "pose": True},
}


def _call_kw(variant):
    v = _VARIANTS[variant]
    return {"pose": bool(v.get("pose")), "refine": v["detector"].get("corners") == "refined"}


def _run_detect_case(a3, torch, name, layout, mem, variant):
    frames = _frameset(name)
    n, h, w = frames.shape[:3]
    pitch, fs, off = _detect_layout(layout, w, h)
    v = _VARIANTS[variant]
    want = _tight_records(name, variant)
    staged = int(mem == "pageable" and n * fs >= 1 << 20)
    # the one-shot route needs the device contour stage and one front-end chunk per call (resident input always has one)
    one_shot_second = int(variant != "host_contours" and (variant != "chunk1" or mem == "device"))
    label = f"{name} {layout} {mem} {variant}"
    with a3.Detector(**v["detector"]) as d:
        if v.get("pose"):
            d.set_pose(40.0)
        if v.get("tuning"):
            _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(d._h, C.byref(_ffi.A3K1Tuning(**v["tuning"]))))
        for call, seed in enumerate((11, 12)):  # the first call takes the ordinary route, the second the one-shot route
            ptr, keep = _input(torch, embed(frames, pitch, fs, off, poison_seed=seed), mem)
            res = _detect(d, ptr + off, mem, n, w, h, pitch, fs, **_call_kw(variant))
            del keep
            st = res["stats"]
            assert st["input_staged"] == staged, f"{label}: input_staged"
            assert st["one_shot"] == (one_shot_second if call else 0), f"{label} call {call}: one_shot"
            if v.get("tuning") and mem != "device":
                assert st["pixel_kernel_launches"] == n, f"{label}: one front-end chunk per frame"
            _check_against_oracle(res, _oracle_detect(name), f"{label} call {call}")
            assert res["markers"].tobytes() == want["markers"].tobytes(), f"{label} call {call}: marker records"
            for k in ("poses", "corners"):
                assert res.get(k) == want.get(k), f"{label} call {call}: {k}"
        if one_shot_second:  # markers only: the one-shot route also assembles the records on the device
            ptr, keep = _input(torch, embed(frames, pitch, fs, off, poison_seed=13), mem)
            res = _detect(d, ptr + off, mem, n, w, h, pitch, fs, full=False, **_call_kw(variant))
            assert res["stats"]["one_shot"] == 1
            assert res["markers"].tobytes() == want["markers"].tobytes(), f"{label}: device-assembled marker records"


@pytest.mark.parametrize("mem", ["pageable", "pinned", "device"])
@pytest.mark.parametrize("layout", ["tight", "crop", "gap"])
@pytest.mark.parametrize("name", ["odd", "c1"])
def test_detect_layouts(a3, torch, name, layout, mem):
    """a3_detect_batch on cropped and gapped frames in pageable (staged from 1 MB on), page-locked and device memory, first
    call and one-shot repeat: grey, mask, candidates and markers equal the oracle's on the tight frames, and the marker
    records equal the tight call's byte for byte."""
    _run_detect_case(a3, torch, name, layout, mem, "default")


@pytest.mark.parametrize("variant", ["chunk1", "host_contours", "refined_pose"])
@pytest.mark.parametrize("layout", ["crop", "gap"])
@pytest.mark.parametrize("name", ["odd", "c1"])
def test_detect_layouts_variants(a3, torch, name, layout, variant):
    """The same with one front-end chunk (its own host copy) per frame, with the host contour stage, and with refined
    corners (K5) feeding the pose kernel (K4): those read only the device grey, so poses and refined corners must equal
    the tight call's byte for byte."""
    for mem in ("pageable", "pinned", "device"):
        _run_detect_case(a3, torch, name, layout, mem, variant)


@pytest.mark.parametrize("fmt", ["rgb8", "luma8", "rgb16"])
def test_pitch_and_stride_too_small(det, fmt):
    """pitch < w * bpp or frame_stride < pitch * h: A3_ERR_INVALID_ARGUMENT from both entry points, nothing read."""
    L = _ffi.lib()
    code, bpp = FORMATS[fmt][0], _bpp(fmt)
    row = W * bpp
    buf = np.zeros(N * (row + 64) * (H + 1), np.uint8)
    grey = np.empty((N, H, W), np.uint8)
    mask = np.empty_like(grey)
    markers = (_ffi.A3Marker * 16)()
    nm = C.c_uint32()
    for pitch, fs in ((row - 1, row * H), (row, row * H - 1), (0, 0)):
        st = L.a3_gray_threshold_batch(det._h, buf.ctypes.data, code, _ffi.MEM_HOST, N, W, H, pitch, fs, grey.ctypes.data,
                                       mask.ctypes.data, None, None)
        assert st == _ffi.A3_ERR_INVALID_ARGUMENT, (pitch, fs)
        st = L.a3_detect_batch(det._h, buf.ctypes.data, code, _ffi.MEM_HOST, N, W, H, pitch, fs, C.cast(markers, C.c_void_p), 16,
                               C.byref(nm), None, None)
        assert st == _ffi.A3_ERR_INVALID_ARGUMENT, (pitch, fs)


# ---- host input copies stop at the last pixel ------------------------------------------------------------------------


def _guard_child(name, layout):
    """Runs in a child process.  Puts the frames into pageable memory whose next page is inaccessible, the last pixel byte
    being the last byte before it, and runs both entry points on them (a3_detect_batch also with one front-end chunk per
    frame): a copy that reads past the last pixel ends the process with SIGSEGV.  Results must equal the tight call's."""
    import aruco3_b200 as a3
    libc = C.CDLL(None, use_errno=True)
    libc.mprotect.argtypes = [C.c_void_p, C.c_size_t, C.c_int]
    frames = _frameset(name)
    n, h, w = frames.shape[:3]
    pitch, fs, off = _detect_layout(layout, w, h)
    span = (n - 1) * fs + (h - 1) * pitch + w * 3
    page = mmap.PAGESIZE
    npages = -(-(off + span) // page) + 1
    mm = mmap.mmap(-1, npages * page)
    base = C.addressof(C.c_char.from_buffer(mm))
    guard = base + (npages - 1) * page
    assert libc.mprotect(guard, page, 0) == 0, "mprotect(PROT_NONE) failed"  # pageable memory only, never pinned or device
    buf = np.frombuffer(mm, np.uint8, count=off + span, offset=guard - (off + span) - base)
    embed(frames, pitch, fs, off, poison_seed=21, out=buf)
    assert buf.ctypes.data + off + span == guard
    tight = np.ascontiguousarray(frames)
    with a3.Detector() as d:  # host memory only: no torch in this process
        want = _gray_threshold(d, None, tight, 0, "rgb8", "host", w * 3, w * 3 * h, n, h, w)
        got = _gray_threshold(d, None, buf, off, "rgb8", "host", pitch, fs, n, h, w)
        for k in want:
            assert np.array_equal(got[k], want[k]), f"a3_gray_threshold_batch: {k}"
        ref = _detect(d, tight.ctypes.data, "pageable", n, w, h, w * 3, w * 3 * h)
        for chunk in (0, 1):
            _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(d._h, C.byref(_ffi.A3K1Tuning(chunk_frames=chunk))))
            res = _detect(d, buf.ctypes.data + off, "pageable", n, w, h, pitch, fs)
            assert res["stats"]["input_staged"] == int(n * fs >= 1 << 20)
            assert res["markers"].tobytes() == ref["markers"].tobytes(), f"a3_detect_batch (chunk_frames {chunk}): markers"
            assert np.array_equal(res["grey"], ref["grey"]) and np.array_equal(res["mask"], ref["mask"])
    print("guarded copies ok")


@pytest.mark.parametrize("layout", ["crop", "gap"])
@pytest.mark.parametrize("name", ["odd", "c1"])
def test_host_copies_stop_at_the_last_pixel(a3, name, layout):
    """Host input is copied up to the last pixel of the last frame and no further: not the rest of the parent row after a
    crop, nor the gap after the last frame.  Unstaged ("odd", < 1 MB) and staged ("c1") pageable input, both entry points;
    in a child process, so that an over-read fails this test with the child's signal instead of ending the test run."""
    code = (f"import sys; sys.path.insert(0, {str(ROOT)!r}); from tests.test_gpu_layouts import _guard_child; "
            f"_guard_child({name!r}, {layout!r})")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    how = f"signal {signal.Signals(-r.returncode).name}" if r.returncode < 0 else f"exit code {r.returncode}"
    assert r.returncode == 0 and "guarded copies ok" in r.stdout, f"child ended with {how}:\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}"
