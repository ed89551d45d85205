#!/usr/bin/env python3
"""Cost of the sub-pixel corner refinement (kernel K5), refinement on vs off in the same process, alternating:
  - 256 x C3 and 256 x C5 frames resident on the device: K5's device time (a3_stats.ms_refine_kernel, CUDA events around
    the launch) and the step time (host clock around a3_detect_batch, which ends in a stream synchronisation);
  - one 1920x1080 marker frame from pinned host memory per call (BASELINE.json configs[1]): wall time per call.
The card's name and power limit are read in the same run.  Prints one JSON object (and writes it to --out if given).
usage: python tools/refine_timing.py [--out FILE] [--calls N]"""
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

from aruco3_b200 import Detector, DetectorConfig, _ffi, synth  # noqa: E402


def card():
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                               text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return {"gpu": torch.cuda.get_device_name(0), "power_limit": limit}


def run_calls(det, frames_ptr, mem, n, w, h, calls, refine):
    """`calls` timed calls after 3 warm-up calls -> (median step ms, median K5 ms, K5 launches, markers)"""
    L = _ffi.lib()
    _ffi.check(L.a3_detector_set_corner_refinement(det._h, _ffi.CORNERS_REFINED if refine else _ffi.CORNERS_INTEGER))
    cap = 256 * n + 1024  # C5 frames carry 220 markers each
    markers = (_ffi.A3Marker * cap)()
    corners = np.zeros((cap, 8), np.float32)
    outs = _ffi.A3Outputs()
    outs.marker_corners = corners.ctypes.data if refine else None
    nm, st = C.c_uint32(), _ffi.A3Stats()
    step, k5 = [], []
    for it in range(3 + calls):
        t0 = time.perf_counter()
        _ffi.check(L.a3_detect_batch(det._h, frames_ptr, _ffi.FMT_RGB8, mem, n, w, h, w * 3, w * h * 3, C.cast(markers, C.c_void_p), cap,
                                     C.byref(nm), C.byref(outs), C.byref(st)))
        dt = 1e3 * (time.perf_counter() - t0)
        if it >= 3:
            step.append(dt)
            k5.append(st.ms_refine_kernel)
    return statistics.median(step), statistics.median(k5), st.refine_kernel_launches, nm.value, st.one_shot


def batch(name, n, calls, rounds):
    spec = synth.CONFIGS[name]
    base, _ = synth.render_batch(name, 16)
    frames = torch.from_numpy(base).repeat((n + 15) // 16, 1, 1, 1)[:n].contiguous().cuda()
    h, w = frames.shape[1:3]
    cfg = DetectorConfig(min_corner_separation_factor=spec.min_corner_separation_factor)
    res = {"off": [], "on": []}
    with Detector(cfg, dictionary=spec.dictionary) as det:
        for _ in range(rounds):
            for mode in ("off", "on"):
                res[mode].append(run_calls(det, frames.data_ptr(), _ffi.MEM_DEVICE, n, w, h, calls, mode == "on"))
    on, off = res["on"], res["off"]
    return {"workload": f"{n} x {name} resident", "markers": on[-1][3], "one_shot": on[-1][4],
            "k5_ms": round(statistics.median(r[1] for r in on), 4), "k5_launches": on[-1][2],
            "step_ms_off": round(statistics.median(r[0] for r in off), 3), "step_ms_on": round(statistics.median(r[0] for r in on), 3)}


def single_frame(calls, rounds):
    h, w = 1080, 1920
    frame = torch.empty((1, h, w, 3), dtype=torch.uint8, pin_memory=True)
    frame.numpy()[:] = synth.render_batch("C3", 1)[0]
    res = {"off": [], "on": []}
    with Detector(dictionary="ARUCO") as det:
        for _ in range(rounds):
            for mode in ("off", "on"):
                res[mode].append(run_calls(det, frame.data_ptr(), _ffi.MEM_HOST, 1, w, h, calls, mode == "on"))
    on, off = res["on"], res["off"]
    return {"workload": "1 x 1920x1080 marker frame, pinned host input", "markers": on[-1][3], "one_shot": on[-1][4],
            "k5_ms": round(statistics.median(r[1] for r in on), 4),
            "call_ms_off": round(statistics.median(r[0] for r in off), 4), "call_ms_on": round(statistics.median(r[0] for r in on), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("refine_timing: no CUDA device")
    out = {"card": card(), "method": f"median over {a.rounds} alternating off / on rounds of the median of {a.calls} calls ({20 * a.calls} for the single frame) after 3 warm-up calls each",
           "results": [batch("C3", 256, a.calls, a.rounds), batch("C5", 256, a.calls, a.rounds), single_frame(20 * a.calls, a.rounds)]}
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
