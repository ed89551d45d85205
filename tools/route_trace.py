#!/usr/bin/env python3
"""The device work a3_detect_batch enqueues on each of its routes, so that two builds of the library can be held to the same
work.  For every call of a route matrix it records, with torch.profiler (CUDA activities), the kernels in launch order on
each stream and the memory copies and sets (direction and bytes); beside them the call's a3_stats route flags and launch
counters and a digest of every output buffer.

The matrix: host and device input; first and repeat call of a detector (the repeat takes the one-shot route where it can);
markers only (lean) and full outputs; device and host contours; post-decode stages off, each alone, all together, and all with
a lens distortion whose pose and board intrinsics are equal (one K7 set) or not (two); the ordinary route over several chunks
and decode groups, on host input also with host contours and both pinned rings; a call whose one-shot speculation fails and
retries the ordinary way; and a call of pure-noise frames after flat ones, whose K3 lists outgrow the speculation, so that
K3's exact finish behind the failed speculative one is traced too.

usage: python tools/route_trace.py --out FILE                    trace the library that A3_LIB_PATH (or the package) loads
       python tools/route_trace.py --compare OLD NEW [--out FILE]  compare two traces: kernel sequences, copies, counters, outputs"""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import tempfile
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

W, H = 640, 480
K = (500.0, 500.0, 320.0, 240.0)
K_BOARD = (505.0, 498.0, 321.0, 239.5)  # different board intrinsics: K7 writes two sets
DIST = (-0.28, 0.09, 0.0, 0.0, 0.0)
STAGES = {  # name -> (pose, refine, board, distortion: None / "shared" / "separate")
    "none": (False, False, False, None),
    "pose": (True, False, False, None),
    "refine": (False, True, False, None),
    "board": (False, False, True, None),
    "all": (True, True, True, None),
    "all+dist1": (True, True, True, "shared"),
    "all+dist2": (True, True, True, "separate"),
    "pose+dist": (True, False, False, "shared"),
}


def frames(n):
    import numpy as np

    from aruco3_b200 import Board, synth
    board = Board.grid(6, 4, 40.0, 10.0)
    out = np.empty((n, H, W, 3), np.uint8)
    for i, (R, t) in enumerate(synth.board_views(n, seed=4, distance=(450.0, 650.0))):
        out[i] = synth.render_board_frame(board.ids, board.corners, R, t, K, W, H, extra_ids=(500, 501), noise=3, seed=i)[0]
    return board, out


def make_detector(board, stages, contours, chunk):
    from aruco3_b200 import CameraDistortion, CameraIntrinsics, Detector, DetectorConfig, _ffi
    pose, refine, with_board, dist = STAGES[stages]
    d = Detector(DetectorConfig(min_corner_separation_factor=0.03), contours=contours, corners="refined" if refine else "integer")
    if pose:
        d.set_pose(40.0, CameraIntrinsics(W, H, *K))
    if with_board:
        d.set_board(board, CameraIntrinsics(W, H, *(K_BOARD if dist == "separate" else K)))
    if dist:
        d.set_distortion(CameraDistortion(*DIST))
    if chunk:
        t = _ffi.A3K1Tuning()
        t.chunk_frames = chunk
        _ffi.check(_ffi.lib().a3_detector_set_k1_tuning(d._h, C.byref(t)))
    return d


def detect(d, src, mem, n, full):
    """One a3_detect_batch call with every output of the case -> (status, stats, digest of the outputs)"""
    import numpy as np

    from aruco3_b200 import _ffi
    cap, cap_c, hs = 64 * n, 256 * n, d.config.homography_sample_size
    ms, nm, outs, st = (_ffi.A3Marker * cap)(), C.c_uint32(), _ffi.A3Outputs(), _ffi.A3Stats()
    poses, corners, boards = (_ffi.A3Pose * (2 * cap))(), np.zeros((cap, 8), np.float32), (_ffi.A3BoardPose * n)()
    offsets = np.zeros(n + 1, np.uint32)
    outs.marker_poses, outs.marker_corners = C.cast(poses, C.c_void_p).value, corners.ctypes.data
    outs.board_poses, outs.frame_marker_offsets = C.cast(boards, C.c_void_p).value, offsets.ctypes.data
    bufs = [ms, poses, corners, boards, offsets]
    if full:
        grey, cands, cframe = np.zeros((n, H, W), np.uint8), np.zeros((cap_c, 8), np.uint32), np.zeros(cap_c, np.uint32)
        patches, decs = np.zeros((cap_c, hs, hs), np.uint8), (_ffi.A3Decode * cap_c)()
        outs.grey, outs.candidates, outs.candidate_frame = grey.ctypes.data, cands.ctypes.data, cframe.ctypes.data
        outs.homographies, outs.decodes, outs.cand_capacity = patches.ctypes.data, C.cast(decs, C.c_void_p).value, cap_c
        bufs += [grey, cands, cframe, patches, decs]
    status = _ffi.lib().a3_detect_batch(d._h, src, _ffi.FMT_RGB8, mem, n, W, H, W * 3, W * H * 3, C.cast(ms, C.c_void_p), cap,
                                        C.byref(nm), C.byref(outs), C.byref(st))
    h = hashlib.sha256()
    for b in bufs:
        h.update(memoryview(b).cast("B"))
    return status, st, h.hexdigest()[:16]


def traced(fn):
    """fn() under torch.profiler -> (fn's result, {"kernels": {stream: [names]}, "copies": [...], "sets": [...]})"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    events = sorted((e for e in events if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")),
                    key=lambda e: (e["ts"], e["name"]))
    streams = sorted({e["args"].get("stream", -1) for e in events})
    label = {s: f"s{i}" for i, s in enumerate(streams)}  # streams in creation order
    kernels = {}
    copies, sets = [], []
    for e in events:
        s = label[e["args"].get("stream", -1)]
        if e["cat"] == "kernel":
            kernels.setdefault(s, []).append(e["name"])
        else:
            (copies if e["cat"] == "gpu_memcpy" else sets).append([s, e["name"], e["args"].get("bytes", -1)])
    return res, {"kernels": kernels, "copies": copies, "sets": sets}


def run_case(name, board, imgs, mem, contours, full, stages, chunk=0, retry=False):
    import numpy as np
    import torch

    from aruco3_b200 import _ffi
    n = len(imgs)
    kinds = {"host": _ffi.MEM_HOST, "device": _ffi.MEM_DEVICE}
    keep = []

    def src_of(a):
        a = np.ascontiguousarray(a)
        t = torch.from_numpy(a).cuda() if mem == "device" else a
        keep.append(t)
        return t.data_ptr() if mem == "device" else t.ctypes.data

    src = src_of(imgs)
    out = []
    with make_detector(board, stages, contours, chunk) as d:
        if retry:  # blank frames set a small history (256 quads of headroom); the traced frames then outgrow the speculated lists
            blank = src_of(np.full_like(imgs, 200))
            for _ in range(2):
                detect(d, blank, kinds[mem], n, full)
            calls = ["retry"]
        else:
            calls = ["first", "repeat"]
        for call in calls:
            (status, st, digest), tr = traced(lambda: detect(d, src, kinds[mem], n, full))
            counters = {k: getattr(st, k) for k in ("one_shot", "one_shot_retry", "pixel_kernel_launches", "contour_kernel_launches",
                                                    "decode_kernel_launches", "refine_kernel_launches", "undistort_kernel_launches",
                                                    "pose_kernel_launches", "board_kernel_launches", "n_candidates", "n_markers")}
            out.append({"case": name, "call": call, "status": status, "stats": counters, "outputs": digest, **tr})
    return out


def trace(path):
    import numpy as np
    import torch

    from aruco3_b200 import _ffi
    from board_timing import card
    board, imgs = frames(5)
    imgs[2] = 200  # a frame without markers
    many = imgs[[i % 5 for i in range(40)]]  # 40 frames: two decode groups on the ordinary route
    noise = np.random.default_rng(9).integers(0, 256, size=imgs.shape, dtype=np.uint8)  # far more long borders than flat frames
    traced(lambda: torch.zeros(1, device="cuda"))  # profiler start-up outside the cases
    cases = []
    for mem in ("host", "device"):
        for contours in ("device", "host"):
            for full in (False, True):
                for stages in STAGES:
                    name = f"{mem} input, {contours} contours, {'full' if full else 'lean'}, {stages}"
                    cases += run_case(name, board, imgs, mem, contours, full, stages)
        for stages in ("none", "all+dist2"):
            cases += run_case(f"{mem} input, device contours, full, {stages}, 40 frames in chunks of 8", board, many, mem, "device", True,
                              stages, chunk=8)
            for full in (False, True):
                cases += run_case(f"{mem} input, device contours, {'full' if full else 'lean'}, {stages}, 40 frames, one-shot retry", board,
                                  many, mem, "device", full, stages, retry=True)
        cases += run_case(f"{mem} input, device contours, full, none, 5 noise frames after flat ones, K3 speculation fails", board, noise,
                          mem, "device", True, "none", retry=True)
    # the host stage over several chunks and decode groups, from pageable frames into a pageable grey buffer
    cases += run_case("host input, host contours, full, none, 40 frames in chunks of 8", board, many, "host", "host", True, "none", chunk=8)
    res = {"library": _ffi.LIB_PATH.name, "card": card(), "calls": cases}
    Path(path).parent.mkdir(parents=True, exist_ok=True)
    Path(path).write_text(json.dumps(res, indent=1))
    print(f"{len(cases)} calls traced -> {path}")


def compare(old_path, new_path):
    """-> (summary lines, ok): kernels and memsets identical per stream, copies not more, counters and outputs equal"""
    old, new = (json.loads(Path(p).read_text()) for p in (old_path, new_path))
    lines = [f"old: {old['library']}", f"new: {new['library']}", f"card: {old.get('card')}", ""]
    ok = len(old["calls"]) == len(new["calls"])
    fewer = 0
    for a, b in zip(old["calls"], new["calls"]):
        key = f"{a['case']} [{a['call']}]"
        same_k = a["kernels"] == b["kernels"]
        same_s = sorted(a["sets"]) == sorted(b["sets"])
        same_o = a["status"] == b["status"] and a["stats"] == b["stats"] and a["outputs"] == b["outputs"]
        nk = sum(len(v) for v in a["kernels"].values())
        co, cn = len(a["copies"]), len(b["copies"])
        bo, bn = sum(c[2] for c in a["copies"]), sum(c[2] for c in b["copies"])
        route = "one-shot" if a["stats"]["one_shot"] else ("retry" if a["stats"]["one_shot_retry"] else "ordinary")
        # copies may only be merged on the ordinary route (the one-shot route already copies once)
        good = (a["case"], a["call"]) == (b["case"], b["call"]) and same_k and same_s and same_o and (cn == co or (cn < co and route != "one-shot"))
        ok &= good
        fewer += cn < co
        lines.append(f"{'ok  ' if good else 'FAIL'} {key}: {route}, {nk} kernels {'identical' if same_k else 'DIFFER'}, memsets "
                     f"{'identical' if same_s else 'DIFFER'}, copies {co} -> {cn} ({bo} -> {bn} bytes), counters and outputs "
                     f"{'equal' if same_o else 'DIFFER'}")
    lines += ["", f"{len(old['calls'])} calls; {fewer} with fewer copies; {'all checks hold' if ok else 'CHECKS FAIL'}"]
    return lines, ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--compare", nargs=2, metavar=("OLD", "NEW"))
    a = ap.parse_args()
    if a.compare:
        lines, ok = compare(*a.compare)
        text = "\n".join(lines) + "\n"
        print(text, end="")
        if a.out:
            Path(a.out).write_text(text)
        sys.exit(0 if ok else 1)
    if not a.out:
        ap.error("--out is required when tracing")
    trace(a.out)


if __name__ == "__main__":
    main()
