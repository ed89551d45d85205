#!/usr/bin/env python3
"""Decode-kernel (K2) time on a resident batch of one of the synthetic workloads (default: 256 x C3, the headline), from
a3_stats (CUDA events around the launch).  Prints one JSON line: the library loaded (A3_LIB_PATH for A/B builds), the
per-call K2 / contour / pixel / total ms of the timed calls and their medians.
usage: python tools/k2_timing.py [batch] [workload] [calls]"""
import ctypes as C
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import torch  # noqa: E402

from aruco3_b200 import DetectorConfig, Detector, _ffi, synth  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
wl = sys.argv[2] if len(sys.argv) > 2 else "C3"
calls = int(sys.argv[3]) if len(sys.argv) > 3 else 8
spec = synth.CONFIGS[wl]
base, _ = synth.render_batch(wl, min(n, 32))
frames = torch.from_numpy(base).repeat((n + base.shape[0] - 1) // base.shape[0], 1, 1, 1)[:n].contiguous().cuda()
h, w = frames.shape[1:3]
cfg = DetectorConfig(min_corner_separation_factor=spec.min_corner_separation_factor)
cap = 256 * n  # C5 has about 220 markers per frame
with Detector(cfg, spec.dictionary) as det:
    markers = (_ffi.A3Marker * cap)()
    nm, st = C.c_uint32(), _ffi.A3Stats()
    t = []
    for it in range(3 + calls):  # three warm-up calls
        _ffi.check(_ffi.lib().a3_detect_batch(det._h, frames.data_ptr(), _ffi.FMT_RGB8, _ffi.MEM_DEVICE, n, w, h, w * 3, w * h * 3,
                                              C.cast(markers, C.c_void_p), cap, C.byref(nm), None, C.byref(st)))
        if it >= 3:
            t.append((st.ms_decode_kernel, st.ms_contour_kernels, st.ms_pixel_kernel, st.ms_total))
    med = [statistics.median(x[k] for x in t) for k in range(4)]
    print(json.dumps({"lib": str(_ffi.LIB_PATH.relative_to(ROOT)) if _ffi.LIB_PATH.is_relative_to(ROOT) else str(_ffi.LIB_PATH),
                      "workload": f"{n} x {wl} resident", "candidates": st.n_candidates, "markers": nm.value,
                      "k2_ms": [round(x[0], 4) for x in t], "k2_ms_median": round(med[0], 4), "contour_ms_median": round(med[1], 4),
                      "pixel_ms_median": round(med[2], 4), "total_ms_median": round(med[3], 4)}))
