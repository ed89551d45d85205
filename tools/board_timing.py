#!/usr/bin/env python3
"""Cost of the board pose (kernel K6), board off vs on in the same process, alternating:
  - 256 x 1920x1080 board frames resident on the device (a 6 x 4 grid board seen from 16 seeded poses, two markers
    off the board in each frame): K6's device time (a3_stats.ms_board_kernel, CUDA events around the launch) and the step
    time (host clock around a3_detect_batch, which ends in a stream synchronisation);
  - one of those frames from pinned host memory per call: wall time per call.
Integer corners in both arms (no K5).  The card's name and power limit are read in the same run.  Prints one JSON object
and writes it to --out.
usage: python tools/board_timing.py [--out FILE] [--calls N] [--rounds N]"""
import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from aruco3_b200 import Board, CameraIntrinsics, Detector, DetectorConfig, _ffi, synth  # noqa: E402

W, H = 1920, 1080
K = (1400.0, 1400.0, 960.0, 540.0)
BOARD = Board.grid(6, 4, 40.0, 10.0)


def card():
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return {"gpu": torch.cuda.get_device_name(0), "power_limit": limit}


def board_frames(n):
    out = np.empty((n, H, W, 3), np.uint8)
    for i, (R, t) in enumerate(synth.board_views(n, seed=4, distance=(450.0, 650.0))):
        out[i] = synth.render_board_frame(BOARD.ids, BOARD.corners, R, t, K, W, H, extra_ids=(500, 501), noise=3, seed=i)[0]
    return out


def run_calls(det, frames_ptr, mem, n, calls, board):
    """`calls` timed calls after 3 warm-up calls -> (median step ms, median K6 ms, K6 launches, markers, one_shot, boards ok)"""
    L = _ffi.lib()
    if board:
        det.set_board(BOARD, CameraIntrinsics(W, H, *K))
    else:
        det.set_board(None)
    cap = 64 * n + 1024
    markers = (_ffi.A3Marker * cap)()
    bp = (_ffi.A3BoardPose * n)()
    outs = _ffi.A3Outputs()
    outs.board_poses = C.cast(bp, C.c_void_p).value
    nm, st = C.c_uint32(), _ffi.A3Stats()
    step, k6 = [], []
    for it in range(3 + calls):
        t0 = time.perf_counter()
        _ffi.check(L.a3_detect_batch(det._h, frames_ptr, _ffi.FMT_RGB8, mem, n, W, H, W * 3, W * H * 3, C.cast(markers, C.c_void_p), cap,
                                     C.byref(nm), C.byref(outs), C.byref(st)))
        dt = 1e3 * (time.perf_counter() - t0)
        if it >= 3:
            step.append(dt)
            k6.append(st.ms_board_kernel)
    return statistics.median(step), statistics.median(k6), st.board_kernel_launches, nm.value, st.one_shot, sum(bp[i].ok for i in range(n))


def measure(frames_ptr, mem, n, calls, rounds):
    res = {"off": [], "on": []}
    with Detector(DetectorConfig(min_corner_separation_factor=0.03)) as det:
        for _ in range(rounds):
            for mode in ("off", "on"):
                res[mode].append(run_calls(det, frames_ptr, mem, n, calls, mode == "on"))
    return res["on"], res["off"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r04_board_timing.json"))
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("board_timing: no CUDA device")
    base = board_frames(16)
    dev = torch.from_numpy(base).repeat(16, 1, 1, 1).contiguous().cuda()
    on, off = measure(dev.data_ptr(), _ffi.MEM_DEVICE, 256, a.calls, a.rounds)
    batch = {"workload": "256 x 1920x1080 board frames resident", "markers": on[-1][3], "boards_ok": on[-1][5], "one_shot": on[-1][4],
             "k6_ms": round(statistics.median(r[1] for r in on), 4), "k6_launches": on[-1][2],
             "step_ms_off": round(statistics.median(r[0] for r in off), 3), "step_ms_on": round(statistics.median(r[0] for r in on), 3)}
    frame = torch.empty((1, H, W, 3), dtype=torch.uint8, pin_memory=True)
    frame.numpy()[:] = base[:1]
    on, off = measure(frame.data_ptr(), _ffi.MEM_HOST, 1, 20 * a.calls, a.rounds)
    single = {"workload": "1 x 1920x1080 board frame, pinned host input", "markers": on[-1][3], "boards_ok": on[-1][5], "one_shot": on[-1][4],
              "k6_ms": round(statistics.median(r[1] for r in on), 4),
              "call_ms_off": round(statistics.median(r[0] for r in off), 4), "call_ms_on": round(statistics.median(r[0] for r in on), 4)}
    out = {"card": card(), "board": "6 x 4 grid, 40 mm markers 10 mm apart, intrinsics mode, integer corners",
           "method": f"median over {a.rounds} alternating off / on rounds of the median of {a.calls} calls ({20 * a.calls} for the single frame) after 3 warm-up calls each",
           "results": [batch, single]}
    text = json.dumps(out, indent=1)
    print(text)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
