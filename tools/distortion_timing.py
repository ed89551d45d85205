#!/usr/bin/env python3
"""Cost of the lens distortion (kernel K7), distortion off vs on in the same process, alternating:
  - 256 x C3 frames resident on the device, marker poses in intrinsics mode;
  - 256 x 1920x1080 board frames resident on the device, board pose and marker poses in intrinsics mode;
  - one of those board frames from pinned host memory per call.
For each: K7's device time (a3_stats.ms_undistort_kernel, CUDA events around its launches) and the step / call time (host
clock around a3_detect_batch, which ends in a stream synchronisation).  Integer corners (no K5).  The card's name and
power limit are read in the same run.  Prints one JSON object and writes it to --out.
usage: python tools/distortion_timing.py [--out FILE] [--calls N] [--rounds N]"""
import argparse
import ctypes as C
import json
import statistics
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
import torch  # noqa: E402

from aruco3_b200 import CameraDistortion, CameraIntrinsics, Detector, DetectorConfig, _ffi, synth  # noqa: E402
from board_timing import BOARD, K, board_frames, card  # noqa: E402

DIST = CameraDistortion(-0.28, 0.09, 0.0, 0.0, 0.0)


def run_calls(det, ptr, mem, n, w, h, calls, on):
    """`calls` timed calls after 3 warm-up calls -> (median step ms, median K7 ms, K7 launches, markers, one_shot)"""
    L = _ffi.lib()
    det.set_distortion(DIST if on else None)
    cap = 64 * n + 1024
    markers = (_ffi.A3Marker * cap)()
    poses = (_ffi.A3Pose * (2 * cap))()
    bp = (_ffi.A3BoardPose * n)()
    outs = _ffi.A3Outputs()
    outs.marker_poses = C.cast(poses, C.c_void_p).value
    outs.board_poses = C.cast(bp, C.c_void_p).value
    nm, st = C.c_uint32(), _ffi.A3Stats()
    step, k7 = [], []
    for it in range(3 + calls):
        t0 = time.perf_counter()
        _ffi.check(L.a3_detect_batch(det._h, ptr, _ffi.FMT_RGB8, mem, n, w, h, w * 3, w * h * 3, C.cast(markers, C.c_void_p), cap,
                                     C.byref(nm), C.byref(outs), C.byref(st)))
        dt = 1e3 * (time.perf_counter() - t0)
        if it >= 3:
            step.append(dt)
            k7.append(st.ms_undistort_kernel)
    return statistics.median(step), statistics.median(k7), st.undistort_kernel_launches, nm.value, st.one_shot


def measure(name, ptr, mem, n, w, h, calls, rounds, board):
    res = {"off": [], "on": []}
    k = CameraIntrinsics(w, h, *K) if board else CameraIntrinsics(w, h, 0.75 * w, 0.75 * w)
    kw = dict(board=BOARD, board_intrinsics=k) if board else {}
    with Detector(DetectorConfig(min_corner_separation_factor=0.03) if board else None, **kw) as det:
        det.set_pose(40.0, k)
        for _ in range(rounds):
            for mode in ("off", "on"):
                res[mode].append(run_calls(det, ptr, mem, n, w, h, calls, mode == "on"))
    on, off = res["on"], res["off"]
    return {"workload": name, "markers": on[-1][3], "one_shot": on[-1][4], "k7_launches": on[-1][2],
            "k7_ms": round(statistics.median(r[1] for r in on), 4),
            "step_ms_off": round(statistics.median(r[0] for r in off), 4), "step_ms_on": round(statistics.median(r[0] for r in on), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r06_distortion_timing.json"))
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("distortion_timing: no CUDA device")
    results = []
    c3, _ = synth.render_batch("C3", 16)
    n3, h3, w3 = c3.shape[:3]
    dev = torch.from_numpy(c3).repeat(16, 1, 1, 1).contiguous().cuda()
    results.append(measure("256 x C3 resident, marker poses (intrinsics)", dev.data_ptr(), _ffi.MEM_DEVICE, 256, w3, h3, a.calls, a.rounds,
                           False))
    del dev
    base = board_frames(16)
    dev = torch.from_numpy(base).repeat(16, 1, 1, 1).contiguous().cuda()
    _, bh, bw = base.shape[:3]
    results.append(measure("256 x 1920x1080 board frames resident, board and marker poses (intrinsics)", dev.data_ptr(), _ffi.MEM_DEVICE,
                           256, bw, bh, a.calls, a.rounds, True))
    frame = torch.empty((1, bh, bw, 3), dtype=torch.uint8, pin_memory=True)
    frame.numpy()[:] = base[:1]
    results.append(measure("1 x 1920x1080 board frame, pinned host input, board and marker poses", frame.data_ptr(), _ffi.MEM_HOST, 1, bw,
                           bh, 20 * a.calls, a.rounds, True))
    out = {"card": card(), "distortion": "k1 = -0.28, k2 = 0.09", "corners": "integer",
           "method": f"median over {a.rounds} alternating off / on rounds of the median of {a.calls} calls ({20 * a.calls} for the single frame) after 3 warm-up calls each",
           "results": results}
    text = json.dumps(out, indent=1)
    print(text)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
