"""`bench.py --dump-outputs DIR`: the counters and markers of the last timed call as float64 .npy files, equal to what the
oracle finds on the frames of that call."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def test_dump_outputs_hold_the_last_timed_call(oracle, tmp_path):
    import bench
    from aruco3_b200 import synth
    steps, warmup, n = 2, 3, 4
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--batch", str(n), "--steps", str(steps), "--warmup", str(warmup), "--fast",
                        "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, check=True)
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    fields = ("frame", "candidate", "id", "code", "rotation", "hamming_distance")
    got = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert sorted(got) == sorted(["C3_counts", "C3_marker_corners"] + [f"C3_marker_{k}" for k in fields])
    assert all(v.dtype == np.float64 for v in got.values())
    wl, spec = bench.WORKLOADS["C3"], synth.CONFIGS["C3"]
    idx = bench.frame_indices(wl, (warmup + steps - 1) % wl["rotate"], 0, n)
    cfg = bench.oracle_config(spec)
    want = []
    for f in range(n):
        ref = oracle.detect(synth.render_frame(spec, int(idx[f]))[0], spec.dictionary, cfg)
        want += [[f, m["candidate"], m["id"], m["code"], m["rotation"], m["hamming_distance"]] + m["corners"] for m in ref.markers]
    rows = np.hstack([got[f"C3_marker_{k}"][:, None] for k in fields] + [got["C3_marker_corners"]])
    assert rows.tolist() == want
    assert got["C3_counts"][0] == n and got["C3_counts"][-1] == len(want) >= 4 * 15
