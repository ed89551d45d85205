#!/usr/bin/env python3
"""Benchmark of the detection hot path (BASELINE.json: frames/sec at 1080p, batch 256, on 1/2/4/8 B200;
threshold-kernel HBM GB/s vs peak).

    python bench.py --gpus N --steps K --warmup W                    # this repo's CUDA path, headline workload C3
    python bench.py --workload C4|C5|all ...                         # the other BASELINE.json configs (one JSON line each)
    python bench.py --impl reference --gpus N --steps K ...          # CPU arm: the C restatement of the reference (oracle/)
    python bench.py --dump-outputs DIR ...                           # also write the last timed call's counters and markers (.npy)

One step = one pass of `Detector::detect` (src/aruco.rs:52-121) over one batch of synthetic frames (aruco3_b200/synth.py):
  C3  BASELINE.json configs[2] (HEADLINE): 256 x 1920x1080 RGB8 per GPU, 20 ARUCO markers each; weak scaling
  C4  configs[3]: 1024 x 3840x2160 RGB8 in total, cut into contiguous frame blocks over the N ranks (sharding.shard_range);
      strong scaling; at N = 1 it exercises the super-batch loop of a3_detect_batch
  C5  configs[4]: 256 x 1080p per GPU, APRILTAG_36H11, 220 small markers each (decode-stage stress; the public field
      min_corner_separation_factor = 0.03 keeps neighbours from deleting each other); weak scaling
Frames are independent, so N GPUs run N shards with no collective (torch.distributed only carries the barrier and the
max-over-ranks of the timing).
  value         frames/s with the RGB frames already resident in HBM (a3_detect_batch, A3_MEM_DEVICE).  The steps rotate
                over `rotate` differently seeded batches of the same geometry, so the sizes the one-shot route speculates
                from the previous call are those of DIFFERENT frames; `one_shot.retries_per_step` says how often they missed
  e2e           frames/s through the same call with PINNED host frames: H2D of the frames and D2H of the markers inside
  e2e_pageable  the same with the frames in ordinary (pageable) host memory, as a `DynamicImage`'s Vec<u8> is
  e2e_full      pinned frames in, everything the reference's `Detection` holds out (grey, candidates, 49x49 patches,
                decode records, markers) into pageable host buffers
  roofline      K1 (fused gray + adaptive threshold), 5 algorithmic bytes per pixel, timed with CUDA events on the
                library's own stream inside the timed region (a3_stats.ms_pixel_kernel)
  parity_checked   frames of this rank whose markers (id, rotation, distance, code, corners) from the timed calls' own
                results were compared with oracle/a3ref.c outside the timed region (any difference aborts the run)
The reference (Rust) cannot be built in this image; `--impl reference` and `cpu_baseline` time oracle/a3ref.c
("port"), frame-parallel over the host cores.
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

ALGO_BYTES_PER_PIXEL = 5   # 3 B RGB read + 1 B grey written + 1 B mask written (SURVEY.md §8d)
DUMP_LIMIT_BYTES = 64 << 20  # --dump-outputs: larger outputs are written as a seeded sample of their marker rows

WORKLOADS = {
    "C3": dict(spec="C3", metric="frames_per_sec_1080p_batch256", per_gpu=256, total=None, scaling="weak", rotate=3, distinct=None,
               desc="C3: 1920x1080 RGB8 x 256 frames per GPU, 20 ARUCO markers/frame, noise 0 (BASELINE.json configs[2])"),
    "C4": dict(spec="C4", metric="frames_per_sec_4k_batch1024_sharded", per_gpu=None, total=1024, scaling="strong", rotate=3, distinct=16,
               desc="C4: 3840x2160 RGB8 x 1024 frames in total, contiguous frame blocks over the ranks, 20 ARUCO markers/frame "
                    "(BASELINE.json configs[3])"),
    "C5": dict(spec="C5", metric="frames_per_sec_1080p_apriltag36h11_220markers_batch256", per_gpu=256, total=None, scaling="weak", rotate=3,
               distinct=None,
               desc="C5: 1920x1080 RGB8 x 256 frames per GPU, APRILTAG_36H11, 220 markers of 40-56 px per frame, "
                    "min_corner_separation_factor 0.03 (BASELINE.json configs[4], decode-stage stress)"),
}


def bind_near_gpu(index):
    """One process per GPU: run this rank (and so first-touch its pinned frames) on the cores NVML reports as local to the
    GPU, so that the H2D stream of every rank reads host memory of its own socket.  Returns the number of cores, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index), (ncpu + 63) // 64)
        cpus = {i * 64 + b for i, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1} & os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def rank_info():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (NVML)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.sm_max = index, threading.Event(), [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
                 "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80)}
        while not self.stop_flag.is_set():
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self.stop_flag.wait(0.01)  # 100 Hz: NVML calls take a driver-wide lock, and at N = 8 eight processes poll at once

    def result(self):
        self.stop_flag.set()
        if self.is_alive():
            self.join(timeout=2)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def render_into(spec_name, indices, out, threads=8):
    """Frames `indices` of workload `spec_name` into out[0:len(indices)] (numpy releases the GIL in the big array ops)."""
    from aruco3_b200 import synth
    spec = synth.CONFIGS[spec_name]

    def one(k):
        out[k] = synth.render_frame(spec, int(indices[k]))[0]

    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(one, range(len(indices))))


def frame_indices(wl, batch, lo, hi):
    """Global synthetic-frame indices of this rank's frames [lo, hi) in rotation batch `batch`.  A workload with a `distinct`
    count (C4) tiles that many rendered frames over the shard; batches use disjoint index ranges, so they differ."""
    n_global = 1 << 20  # batches are far apart in index space
    idx = np.arange(lo, hi, dtype=np.int64)
    if wl["distinct"]:
        idx = lo + (idx - lo) % wl["distinct"]
    return idx + batch * n_global


def workload_config(wl, frames_per_gpu, frame_bytes):
    """The `config` object of the JSON line, the same in the CUDA arm and in `--impl reference`."""
    return {"workload": wl["desc"], "frames_per_gpu_per_step": frames_per_gpu,
            "l2": f"inputs larger than L2 ({frames_per_gpu * frame_bytes / 1e6:.0f} MB of RGB per step per GPU, never re-read within a step)"}


def oracle_config(spec):
    from oracle import a3ref_py
    cfg = a3ref_py.default_config()
    cfg.min_corner_separation_factor = spec.min_corner_separation_factor
    return cfg


def cpu_reference_run(frames: np.ndarray, spec, threads: int, steps: int, warmup: int, passes: int = 1):
    """oracle/a3ref.c, frame-parallel: the CPU arm (never on the product path).  One step = `passes` passes over `frames`
    (a shard that tiles its rendered frames is detected tile by tile: the same work as the tiled array)."""
    from oracle import a3ref_py
    cfg = oracle_config(spec)
    for _ in range(warmup):
        a3ref_py.detect_many(frames, spec.dictionary, cfg, threads=threads)
    t0 = time.perf_counter()
    markers = 0
    st = {}
    for _ in range(steps):
        for _ in range(passes):
            m, st = a3ref_py.detect_many(frames, spec.dictionary, cfg, threads=threads)
            markers += m
    dt = time.perf_counter() - t0
    return len(frames) * passes * steps / dt, dt / steps, markers // max(steps, 1), st


def run_reference(args, wl_name):
    """`--impl reference`: the CPU implementation of the path (the oracle port: the Rust crate cannot be built here) on the box's
    host cores, all of them, over the SAME frames rank 0 of the CUDA arm gets in its first batch: one step = that batch."""
    from aruco3_b200 import synth
    from aruco3_b200.sharding import shard_range
    rank, _, world = rank_info()
    if rank != 0:
        return 0
    wl = WORKLOADS[wl_name]
    spec = synth.CONFIGS[wl["spec"]]
    cores = os.cpu_count() or 1
    n_total = wl["total"] if wl["total"] else (args.batch or wl["per_gpu"]) * world
    lo, hi = shard_range(n_total, 0, world)
    n = hi - lo
    h, w = spec.height, spec.width
    idx = frame_indices(wl, 0, lo, hi)
    tiled = bool(wl["distinct"]) and n > wl["distinct"]
    uniq = idx[: wl["distinct"]] if tiled else idx
    passes = n // len(uniq)  # a tiled shard repeats its rendered frames (n is a multiple of `distinct` for the shipped workloads)
    frames = np.empty((len(uniq), h, w, 3), np.uint8)
    render_into(wl["spec"], uniq, frames)
    fps, s_per_step, markers, st = cpu_reference_run(frames, spec, cores, max(1, args.steps), args.warmup, passes)
    frames_per_step = len(uniq) * passes
    line = {"impl": "reference", "workload": wl_name, "metric": wl["metric"], "value": fps, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_step * 1e3,
            "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "u8/u32 integer pixels, f32/f64 decode",
            "data": "synthetic",
            "config": workload_config(wl, frames_per_step, h * w * 3),
            "run_details": {"host_threads": cores},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                             "sample": f"the {frames_per_step} frames of rank 0's first batch per step"
                                       + (f" ({len(uniq)} rendered frames x {passes} passes: the shard tiles them)" if tiled else "")
                                       + f", frame-parallel over {cores} threads (oracle/a3ref.c; the Rust reference cannot be built in this image)"},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "markers_per_step": markers, "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def k1_traffic(frames_per_launch, w, h):
    """DRAM bytes per K1 launch from the committed ncu --set full capture (profiles/k1_traffic.json), scaled to this launch's
    pixels; None when the file is absent or was captured from a different k1_strips.cu (the file records the source hash)."""
    tf = ROOT / "profiles" / "k1_traffic.json"
    if not tf.exists():
        return None, None
    t = json.loads(tf.read_text())
    src_hash = hashlib.sha256((ROOT / "aruco3_b200" / "csrc" / "k1_strips.cu").read_bytes()).hexdigest()[:16]
    if t.get("k1_strips_sha256_16") not in (None, src_hash):
        return None, f"stale: {tf.name} was captured from another k1_strips.cu ({t.get('k1_strips_sha256_16')} != {src_hash})"
    px_ratio = (w * h * frames_per_launch) / (t.get("width", 1920) * t.get("height", 1080) * t["frames_per_launch"])
    return (t["dram_bytes_read"] + t["dram_bytes_write"]) * px_ratio, t["source"]


def dump_outputs(out_dir, prefix, rec, stats):
    """--dump-outputs: what one a3_detect_batch call hands its caller, as float64 arrays that two builds can be compared by.
    `<prefix>_counts.npy` holds the call's a3_stats counters (n_frames, n_contours, n_contour_points, n_candidates_before_discard,
    n_candidates, n_markers); `<prefix>_marker_<field>.npy` one field of every marker record, rows in (frame, candidate) order.
    Marker rows beyond DUMP_LIMIT_BYTES are cut to a fixed seeded sample, still in that order."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    counts = [stats[k] for k in ("n_frames", "n_contours", "n_contour_points", "n_candidates_before_discard", "n_candidates", "n_markers")]
    np.save(out / f"{prefix}_counts.npy", np.array(counts, np.float64))
    rec = rec[np.lexsort((rec["candidate"], rec["frame"]))]
    cols = {"frame": rec["frame"], "candidate": rec["candidate"], "id": rec["id"], "code": rec["code"], "rotation": rec["rot"],
            "hamming_distance": rec["hd"], "corners": rec["corners"]}
    max_rows = (DUMP_LIMIT_BYTES - 4096) // (8 * (6 + 8))  # six scalar fields + eight corner coordinates per row
    rows = np.arange(len(rec))
    if len(rec) > max_rows:
        rows = np.sort(np.random.default_rng(0xA3D0).choice(len(rec), max_rows, replace=False))
    for name, v in cols.items():
        np.save(out / f"{prefix}_marker_{name}.npy", v[rows].astype(np.float64))  # ids and codes < 2^53: exact in float64


def run_b200(args, wl_name, ctx):
    import torch
    import torch.distributed as dist
    from aruco3_b200 import Detector, DetectorConfig, _ffi, synth
    from aruco3_b200.sharding import shard_range

    rank, local_rank, world = rank_info()
    wl = WORKLOADS[wl_name]
    spec = synth.CONFIGS[wl["spec"]]
    h, w = spec.height, spec.width
    cores = os.cpu_count() or 1
    host_threads = args.host_threads or max(1, cores // max(world, 1))
    n_total = wl["total"] if wl["total"] else (args.batch or wl["per_gpu"]) * world
    lo, hi = shard_range(n_total, rank, world)  # this rank's contiguous block of the global batch
    n = hi - lo
    rotate = max(1, args.rotate if args.rotate else wl["rotate"])
    frame_bytes = h * w * 3

    # ---- synthetic frames: `rotate` differently seeded batches resident in HBM; pinned host copies of as many of them as fit
    # 8 GB (all three for the 1080p workloads, one for a big 4K shard) ----
    rotate_host = max(1, min(rotate, int((8 << 30) // max(1, n * frame_bytes))))
    pinned = [torch.empty((n, h, w, 3), dtype=torch.uint8, pin_memory=True) for _ in range(rotate_host)]
    resident = [None] * rotate
    t_render = time.perf_counter()
    for b in reversed(range(rotate)):  # descending: pinned[j] ends up holding batch j
        idx = frame_indices(wl, b, lo, hi)
        hbuf = pinned[min(b, rotate_host - 1)]
        hn = hbuf.numpy()
        if wl["distinct"] and n > wl["distinct"]:
            d = wl["distinct"]
            render_into(wl["spec"], idx[:d], hn[:d])
            for k in range(d, n, d):
                m = min(d, n - k)
                hn[k:k + m] = hn[:m]
        else:
            render_into(wl["spec"], idx, hn)
        resident[b] = hbuf.cuda(non_blocking=False)
    torch.cuda.synchronize()
    t_render = time.perf_counter() - t_render

    cfg = DetectorConfig(min_corner_separation_factor=spec.min_corner_separation_factor)
    det = Detector(cfg, dictionary=spec.dictionary, device=local_rank, host_threads=host_threads, contours=args.contours)
    L = _ffi.lib()
    if args.chunk:
        tune = _ffi.A3K1Tuning(chunk_frames=args.chunk)
        _ffi.check(L.a3_detector_set_k1_tuning(det._h, C.byref(tune)))
    per_frame_cap = 64 if wl_name != "C5" else 320
    cap = per_frame_cap * n
    markers = (_ffi.A3Marker * cap)()
    n_markers = C.c_uint32()
    stats = _ffi.A3Stats()

    def step(ptr, mem, want_stats=True, outs=None):
        _ffi.check(L.a3_detect_batch(det._h, ptr, _ffi.FMT_RGB8, mem, n, w, h, w * 3, frame_bytes, C.cast(markers, C.c_void_p),
                                     cap, C.byref(n_markers), outs, C.byref(stats) if want_stats else None))
        return stats.as_dict() if want_stats else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(ptrs, mem, steps, warmup, stats_in_loop=True, outs=None):
        """steps rotate over `ptrs`.  stats_in_loop=False: the timed calls pass no a3_stats (the library then skips its ~100
        CUDA-event queries per chunked call); the stage statistics come from `steps` instrumented calls after the timed region."""
        k = 0
        for _ in range(warmup):
            step(ptrs[k % len(ptrs)], mem, True, outs)
            k += 1
        acc = {}
        sampler = ClockSampler(local_rank)  # NVML set up and polling before the barrier, not inside the timed region
        sampler.start()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        per_step = []
        e0.record()
        for _ in range(steps):
            t0 = time.perf_counter()
            s = step(ptrs[k % len(ptrs)], mem, stats_in_loop, outs)
            per_step.append((time.perf_counter() - t0) * 1e3)
            k += 1
            for key, v in (s or {}).items():
                acc[key] = acc.get(key, 0) + v
        e1.record()
        barrier()
        clocks = sampler.result()
        clocks["samples"] = len(sampler.sm)
        # per-rank view of the same timed region (diagnostic: which rank, which step): host wall time of every call
        mine = {"rank": rank, "ms": e0.elapsed_time(e1), "step_ms_median": float(np.median(per_step)), "step_ms_max": float(max(per_step)),
                "slowest_step": int(np.argmax(per_step)), "sm_mhz": clocks.get("sm_mhz"), "reasons": clocks.get("reasons")}
        if world > 1:
            allr = [None] * world
            dist.all_gather_object(allr, mine)
        else:
            allr = [mine]
        clocks["per_rank"] = allr
        if not stats_in_loop:
            for _ in range(steps):
                for key, v in step(ptrs[k % len(ptrs)], mem, True, outs).items():
                    acc[key] = acc.get(key, 0) + v
                k += 1
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, acc, clocks

    # ---- parity: the markers the timed calls produce, against the oracle, outside the timed region ----
    def marker_rows():
        rec = np.frombuffer(markers, dtype=np.dtype([("id", "<u8"), ("code", "<u8"), ("corners", "<u4", 8), ("frame", "<u4"),
                                                      ("candidate", "<u4"), ("hd", "u1"), ("rot", "u1"), ("pad", "u1", 6)]),
                            count=n_markers.value)
        return rec

    def check_parity(batch, frames_to_check, label):
        from oracle import a3ref_py
        rec = marker_rows()
        ocfg = oracle_config(spec)
        idx = frame_indices(wl, batch, lo, hi)
        for f in frames_to_check:
            ref = a3ref_py.detect(synth.render_frame(spec, int(idx[f]))[0], spec.dictionary, ocfg)  # the frame is a pure function of its index
            mine = rec[rec["frame"] == f]
            got = [(int(m["id"]), int(m["rot"]), int(m["hd"]), int(m["code"]), [int(v) for v in m["corners"]]) for m in mine]
            want = [(m["id"], m["rotation"], m["hamming_distance"], m["code"], m["corners"]) for m in ref.markers]
            if got != want:
                raise SystemExit(f"bench.py: PARITY FAILURE ({label}, rank {rank}, batch {batch}, frame {f}): {len(got)} markers vs oracle {len(want)}")
        return len(frames_to_check)

    check_frames = sorted({0, n // 3, (2 * n) // 3, n - 1})
    parity = 0

    dev_ptrs = [r.data_ptr() for r in resident]
    host_ptrs = [p.data_ptr() for p in pinned]
    ms_dev, acc_dev, clocks = timed(dev_ptrs, _ffi.MEM_DEVICE, args.steps, args.warmup)
    # the timed region ended on batch (warmup + steps - 1) % rotate: its markers are still in `markers`, its counters in `stats`
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, wl_name if world == 1 else f"{wl_name}_rank{rank}", marker_rows(), stats.as_dict())
    parity += check_parity((args.warmup + args.steps - 1) % rotate, check_frames, "resident")
    ms_e2e, acc_e2e, clocks_e2e = timed(host_ptrs, _ffi.MEM_HOST, args.steps, 3, stats_in_loop=False)
    parity += check_parity((3 + 2 * args.steps - 1) % rotate_host, check_frames, "e2e")

    # ---- e2e with pageable frames (a DynamicImage's Vec<u8>): batch 0 in ordinary numpy memory ----
    e2e_extra = {}
    if not args.fast:
        pageable = np.empty((n, h, w, 3), np.uint8)
        np.copyto(pageable, pinned[0].numpy())
        ms_pg, acc_pg, _ = timed([pageable.ctypes.data], _ffi.MEM_HOST, args.steps, 3, stats_in_loop=False)
        parity += check_parity(0, check_frames, "e2e_pageable")
        e2e_extra["e2e_pageable"] = {"value": n * world * args.steps / (ms_pg * 1e-3), "unit": "frames/s", "ms_per_step": ms_pg / args.steps,
                                     "input_staged_through_pinned_ring": bool(acc_pg["input_staged"]),
                                     "note": "frames in pageable host memory: the library's copy threads stage them through a pinned ring"}
        del pageable
        # ---- e2e returning the whole `Detection` (src/aruco.rs:115-120) into pageable buffers ----
        hs = 49
        cand_cap = per_frame_cap * n
        o_grey = np.empty((n, h, w), np.uint8)
        o_cands = np.empty((cand_cap, 8), np.uint32)
        o_cframe = np.empty(cand_cap, np.uint32)
        o_patches = np.empty((cand_cap, hs, hs), np.uint8)
        o_decs = (_ffi.A3Decode * cand_cap)()
        outs = _ffi.A3Outputs()
        outs.grey, outs.candidates, outs.candidate_frame = o_grey.ctypes.data, o_cands.ctypes.data, o_cframe.ctypes.data
        outs.homographies, outs.decodes, outs.cand_capacity = o_patches.ctypes.data, C.cast(o_decs, C.c_void_p).value, cand_cap
        ms_full, acc_full, _ = timed(host_ptrs, _ffi.MEM_HOST, args.steps, 3, stats_in_loop=False, outs=C.byref(outs))
        nc = int(outs.n_candidates)
        d2h_full = n * h * w + nc * (32 + 4 + hs * hs + C.sizeof(_ffi.A3Decode)) + n_markers.value * C.sizeof(_ffi.A3Marker)
        parity += check_parity((3 + 2 * args.steps - 1) % rotate_host, check_frames, "e2e_full")
        e2e_extra["e2e_full"] = {"value": n * world * args.steps / (ms_full * 1e-3), "unit": "frames/s", "ms_per_step": ms_full / args.steps,
                                 "d2h_bytes_per_step": int(d2h_full), "output_staged_through_pinned_ring": bool(acc_full["output_staged"]),
                                 "note": "pinned frames in; grey + candidates + 49x49 patches + decode records + markers out, into pageable host buffers"}
        del o_grey, o_patches

    # ---- H2D ceiling of this box with all ranks copying at once: what bounds e2e ----
    h2d = None
    if not args.fast:
        scratch = resident[0]
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        scratch.copy_(pinned[0], non_blocking=True)
        barrier()
        e0.record()
        for _ in range(3):
            scratch.copy_(pinned[0], non_blocking=True)
        e1.record()
        barrier()
        gbs = 3 * n * frame_bytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
        agg = gbs
        mn = gbs
        if world > 1:
            t = torch.tensor([gbs], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            agg = float(t.item())
            t = torch.tensor([gbs], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            mn = float(t.item())
        h2d = {"this_rank_gbs": gbs, "aggregate_gbs": agg, "slowest_rank_gbs": mn,
               "how": f"{world} rank(s) each copying their pinned batch to their GPU at the same time (torch copy_, CUDA events, 3 passes)"}

    # ---- BASELINE.json configs[1] beside the headline: one 1080p frame from host memory per call, wall-clock latency ----
    def single_frame_latency(frame_ptr, fw, fh, reps=40):
        one = (_ffi.A3Marker * 4096)()
        lat = []
        for it in range(reps + 5):
            t0 = time.perf_counter()
            _ffi.check(L.a3_detect_batch(det._h, frame_ptr, _ffi.FMT_RGB8, _ffi.MEM_HOST, 1, fw, fh, fw * 3, fw * fh * 3,
                                         C.cast(one, C.c_void_p), 4096, C.byref(n_markers), None, None))
            if it >= 5:
                lat.append((time.perf_counter() - t0) * 1e3)
        return float(np.median(lat))

    latency = None
    if rank == 0 and wl_name == "C3" and not args.fast:
        from oracle import a3ref_py
        noise = torch.empty((1, 1080, 1920, 3), dtype=torch.uint8, pin_memory=True)
        noise.numpy()[:] = np.random.default_rng(0xA3C0DE00 + 2000).integers(0, 256, size=(1, 1080, 1920, 3), dtype=np.uint8)

        def cpu_ms(img, reps=3):
            ts = []
            for _ in range(reps):
                t0 = time.perf_counter()
                a3ref_py.detect(img, "ARUCO")
                ts.append((time.perf_counter() - t0) * 1e3)
            return float(np.median(ts))

        latency = {"unit": "ms per detect() call, host frame in, markers out (median of 40)",
                   "marker_frame_1080p": single_frame_latency(pinned[0][:1].data_ptr(), w, h),
                   "noise_frame_1080p_reference_bench_workload": single_frame_latency(noise.data_ptr(), 1920, 1080),
                   "cpu_port_marker_frame_1080p_ms": cpu_ms(pinned[0].numpy()[0]),
                   "cpu_port_noise_frame_1080p_ms": cpu_ms(noise.numpy()[0]),
                   "cpu_port_note": "oracle/a3ref.c detect(), one thread, the same two frames (benches/detect_markers.rs:38-45 is the noise frame)"}

    # ---- K1 alone on the resident frames (isolated figure; the roofline entry uses the in-pipeline time) ----
    k1_iso = None
    if not args.fast:
        wpr = (w + 31) // 32
        nk = min(n, 256)
        d_grey = torch.empty((nk, h, w), dtype=torch.uint8, device="cuda")
        d_bits = torch.empty((nk, h, wpr), dtype=torch.int32, device="cuda")
        stream = torch.cuda.current_stream().cuda_stream

        def k1_alone():
            _ffi.check(L.a3_gray_threshold_batch(det._h, resident[0].data_ptr(), _ffi.FMT_RGB8, _ffi.MEM_DEVICE, nk, w, h, w * 3, frame_bytes,
                                                 d_grey.data_ptr(), None, d_bits.data_ptr(), C.c_void_p(stream)))
        for _ in range(3):
            k1_alone()
        torch.cuda.synchronize()
        reps = 10
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
        ev[0].record()
        for i in range(reps):
            k1_alone()
            ev[i + 1].record()
        torch.cuda.synchronize()
        k1_ms = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(reps))[reps // 2]
        iso_bytes = (3 + 1 + 0.125) * w * h * nk
        k1_iso = {"gbs": iso_bytes / (k1_ms * 1e-3) / 1e9, "ms": k1_ms, "bytes": iso_bytes, "frames": nk,
                  "fps": nk / (k1_ms * 1e-3), "note": "K1 alone over resident frames, grey + 1-bit mask outputs (3 + 1 + 1/8 B/px moved)"}
        del d_grey, d_bits

    peak, peak_src = measured_peaks()
    launches = int(acc_dev["pixel_kernel_launches"])
    k1_avg_ms = acc_dev["ms_pixel_kernel"] / max(launches, 1)
    frames_per_launch = n * args.steps / max(launches, 1)
    bytes_per_launch = ALGO_BYTES_PER_PIXEL * w * h * frames_per_launch
    achieved = bytes_per_launch / (k1_avg_ms * 1e-3) / 1e9 if k1_avg_ms > 0 else 0.0
    # what the in-pipeline launch really moves: RGB in, grey + 1-bit mask out (the byte mask is only written on request)
    moved = (3 + 1 + 0.125) * w * h * frames_per_launch / (k1_avg_ms * 1e-3) / 1e9 if k1_avg_ms > 0 else 0.0
    traffic, traffic_src = k1_traffic(frames_per_launch, w, h)
    if k1_iso:
        k1_iso["frac"] = k1_iso["gbs"] / peak

    total_frames = n_total * args.steps if wl["total"] else n * world * args.steps
    value = total_frames / (ms_dev * 1e-3)
    e2e_value = total_frames / (ms_e2e * 1e-3)
    # device -> host per step on the markers-only route: the finished marker records + the per-frame counters
    d2h = int(acc_e2e["n_markers"] / args.steps * C.sizeof(_ffi.A3Marker) + n * (64 * 32 + 4 * 4 + 8)
              + acc_e2e["n_candidates"] / args.steps * C.sizeof(_ffi.A3Decode))
    e2e = {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": n * frame_bytes, "d2h_bytes_per_step": d2h,
           "ms_per_step": ms_e2e / args.steps, "input": "pinned host memory"}
    if h2d:
        e2e["h2d_ceiling"] = h2d
        e2e["frac_of_h2d_ceiling"] = (n * frame_bytes / (ms_e2e / args.steps * 1e-3) / 1e9) / h2d["slowest_rank_gbs"]
    for key, v in e2e_extra.items():
        v["frac_of_pinned_e2e"] = v["value"] / e2e_value
    line = {
        "workload": wl_name, "metric": wl["metric"], "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": wl["scaling"],
        "vs_baseline": None, "dtype": "u8/u32 integer pixels, f32/f64 decode", "data": "synthetic",
        # identical in both arms (`--impl reference` prints the same dict): what the workload is
        "config": workload_config(wl, n, frame_bytes),
        "run_details": {"frames_per_step_all_gpus": n_total, "rotating_batches": rotate, "rotating_batches_host": rotate_host,
                        "distinct_rendered_frames_per_batch": wl["distinct"] if wl["distinct"] and n > wl["distinct"] else n,
                        "host_threads_per_rank": host_threads, "host_cores": cores, "rank_cpu_affinity_cores": ctx.get("numa"),
                        "parallelism": f"frame-batch sharding x{world}, no collective", "render_s": round(t_render, 1)},
        "e2e": e2e,
        **e2e_extra,
        "parity_checked": parity,
        "parity_note": f"frames {check_frames} of this rank's batch, markers of the timed calls' own results vs oracle/a3ref.c, in each of the arms",
        # ours per step: K1, K2, K3's eight kernels (candidates, walk_short, walkers, flag_all, order, emit, rdp, finalize) and, on
        # the one-shot route, the size check of the speculative K3 finish, the two kernels that gather its quads for K2 and the
        # marker assembly
        "gpu_launches": int(acc_dev["pixel_kernel_launches"] + acc_dev["decode_kernel_launches"] + acc_dev["pose_kernel_launches"]
                            + 8 * acc_dev["contour_kernel_launches"] + 4 * acc_dev["one_shot"]),
        "one_shot": {"steps_on_route": int(acc_dev["one_shot"]), "retries": int(acc_dev["one_shot_retry"]),
                     "retries_per_step": acc_dev["one_shot_retry"] / args.steps,
                     "note": f"value arm, {rotate} differently seeded batches in rotation: a retry = the sizes speculated from the previous "
                             "(different) batch did not hold and K3's second half was redone after a synchronisation"},
        "contour_stage": args.contours, "host_fallback_frames_per_step": acc_dev["host_fallback_frames"] / args.steps,
        "roofline": {"bound": "hbm", "kernel": "k1_strips_kernel<RGB8> (fused into_luma8 + adaptive_threshold, TMA tensor tiles)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                     "frac_of_nominal_8TBps": achieved / 8000.0, "traffic": traffic, "traffic_source": traffic_src,
                     "achieved_moved": moved, "frac_moved": moved / peak,
                     "note": "achieved = SURVEY 8d algorithmic 5 B/px (3 RGB + 1 grey + 1 mask) / K1 time; the pipeline writes the mask "
                             "1 bit/px, so it moves 4.125 B/px: achieved_moved",
                     "bytes_per_launch": bytes_per_launch, "avg_launch_ms": k1_avg_ms, "launches": launches, "isolated": k1_iso},
        "stages_ms_per_step": {k: acc_dev[k] / args.steps for k in ("ms_h2d", "ms_pixel_kernel", "ms_contour_kernels", "ms_mask_d2h", "ms_host_quads",
                                                                     "ms_host_cpu", "ms_decode_kernel", "ms_total")},
        # from instrumented calls after the timed region (the timed e2e calls pass no a3_stats)
        "stages_ms_per_step_e2e": {k: acc_e2e[k] / args.steps for k in ("ms_h2d", "ms_pixel_kernel", "ms_contour_kernels", "ms_mask_d2h", "ms_host_quads",
                                                                         "ms_host_cpu", "ms_decode_kernel", "ms_total")},
        "counts_per_step": {k: acc_dev[k] / args.steps for k in ("n_contours", "n_contour_points", "n_candidates", "n_markers")},
        "clocks": clocks, "clocks_e2e": clocks_e2e,
        "single_frame_latency": latency,
    }
    # SURVEY 8d (ii)/(iii): the latency-bound stages are reported as units per second of their own kernel time, not as roofline fractions
    if acc_dev["ms_decode_kernel"] > 0:
        line["k2_decode"] = {"candidates_per_s": acc_dev["n_candidates"] / (acc_dev["ms_decode_kernel"] * 1e-3), "unit": "candidates/s",
                             "ms_per_step": acc_dev["ms_decode_kernel"] / args.steps, "candidates_per_step": acc_dev["n_candidates"] / args.steps}
    if acc_dev["ms_contour_kernels"] > 0:
        line["k3_contours"] = {"border_points_per_s": acc_dev["n_contour_points"] / (acc_dev["ms_contour_kernels"] * 1e-3), "unit": "border points/s",
                               "ms_per_step": acc_dev["ms_contour_kernels"] / args.steps}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        uniq = wl["distinct"] if wl["distinct"] and n > wl["distinct"] else n
        sample = min(uniq, max(32, 2 * cores))
        fps, s_per_step, mk, st = cpu_reference_run(pinned[0].numpy()[:sample], spec, cores, 1, 1)
        fps1, _, _, st1 = cpu_reference_run(pinned[0].numpy()[:4], spec, 1, 1, 0)
        line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                                "sample": f"{sample} of the {n} frames, frame-parallel over {cores} threads (oracle/a3ref.c)",
                                "single_thread_fps": fps1,
                                "single_thread_stage_ms_per_frame": {k: st1[k] / 4 for k in ("ms_gray", "ms_threshold", "ms_contours",
                                                                                              "ms_quads", "ms_warp", "ms_decode")}}
    if rank == 0:
        print(json.dumps(line), flush=True)
    det.close()
    del pinned, resident
    torch.cuda.empty_cache()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C3", choices=["C3", "C4", "C5", "all"], help="BASELINE.json config; the headline metric is C3")
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step for the weak-scaling workloads (the metric is quoted at 256)")
    ap.add_argument("--rotate", type=int, default=0, help="differently seeded batches the steps rotate over (0 = the workload's default, 3)")
    ap.add_argument("--host-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--fast", action="store_true", help="value + pinned e2e only (skips pageable / full e2e, H2D ceiling, latency, isolated K1)")
    ap.add_argument("--chunk", type=int, default=0, help="frames per pipeline chunk (0 = library default)")
    ap.add_argument("--contours", default="device", choices=["device", "host"], help="where find_contours + quad filters run")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the counters and markers of the last timed call as DIR/<workload>_*.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    names = ["C3", "C4", "C5"] if args.workload == "all" else [args.workload]
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs the CUDA arm: the reference arm counts markers but keeps none")
        for name in names:
            run_reference(args, name)
        return 0
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist

    rank, local_rank, world = rank_info()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    ctx = {"numa": bind_near_gpu(local_rank) if world > 1 else None}  # before the pinned buffers are allocated and touched
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    for name in names:
        run_b200(args, name, ctx)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
