"""The lens distortion (kernel K7) through the C++ mirror (include/aruco3_b200.hpp): aruco3::CameraDistortion,
Detector::set_distortion (kept across rebuild()), the PlainDetector field and ShardedDetector::set_distortion, compiled with
g++, run on the GPU and compared bit for bit with the CPU oracle; the new symbols and struct layouts on the CPU."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

from tests.test_oracle_distortion import BARREL, BOARD, CFG, KP, H, W, board_poses

ROOT = Path(__file__).resolve().parent.parent

PROGRAM = r'''
#include <cstdio>
#include <cstring>
#include <vector>
#include "aruco3_b200.hpp"
static void put(const char *tag, const std::vector<aruco3::Detection> &dets) {
    for (const auto &d : dets) {
        if (!d.board_pose) { printf("%s none\n", tag); continue; }
        const aruco3::BoardPose &b = *d.board_pose;
        printf("%s", tag);
        for (const aruco3::MarkerPose *p : {&b.best, &b.alt}) {
            std::vector<float> v{p->error};
            v.insert(v.end(), p->rotation.begin(), p->rotation.end());
            v.insert(v.end(), p->translation.begin(), p->translation.end());
            for (float x : v) { uint32_t u; memcpy(&u, &x, 4); printf(" %08x", u); }
        }
        printf(" %u %d\n", b.n_markers, b.ok ? 1 : 0);
    }
}
int main(int argc, char **argv) {
    const uint32_t w = 1280, h = 720, n = (uint32_t)atoi(argv[2]);
    std::vector<uint8_t> rgb((size_t)n * w * h * 3);
    FILE *f = fopen(argv[1], "rb");
    if (!f || fread(rgb.data(), 1, rgb.size(), f) != rgb.size()) return 2;
    fclose(f);
    const aruco3::Board board = aruco3::Board::grid(6, 4, 40.0f, 10.0f);
    const float px = 640.0f, py = 360.0f;
    const aruco3::CameraIntrinsics k(w, h, 900.0f, 900.0f, &px, &py);
    const aruco3::CameraDistortion dist{-0.28f, 0.09f, 0.0f, 0.0f, 0.0f};
    aruco3::DetectorConfig cfg;
    cfg.min_corner_separation_factor = 0.05f;
    const auto dict = aruco3::ARDictionary::new_from_named_dict("ARUCO");
    aruco3::Detector det(cfg, dict, 0);
    det.set_board(&board, &k);
    det.set_distortion(&dist);
    put("det", det.detect_batch(rgb.data(), n, w, h));
    det.rebuild();  // the distortion survives a rebuild
    put("rebuilt", det.detect_batch(rgb.data(), n, w, h, aruco3::PixelFormat::Rgb8, true));
    aruco3::PlainDetector plain{cfg, dict, 0, false, board, k, dist};
    put("plain", plain.detect_batch(rgb.data(), n, w, h));
    aruco3::ShardedDetector sharded(cfg, dict, {0, 0});
    sharded.set_board(&board, &k);
    sharded.set_distortion(&dist);
    put("sharded", sharded.detect_batch(rgb.data(), n, w, h));
    det.set_distortion(nullptr);
    put("off", det.detect_batch(rgb.data(), n, w, h));
    return 0;
}
'''


def _compile(tmp_path, link=True):
    src, exe = tmp_path / "distort.cpp", tmp_path / "distort"
    src.write_text(PROGRAM)
    lib_dir = ROOT / "aruco3_b200"
    cmd = ["g++", "-std=c++17", "-Wall", "-pthread", "-I", str(ROOT / "include"), str(src)]
    if link:
        cmd += ["-o", str(exe), f"-L{lib_dir}", "-laruco3_b200", f"-Wl,-rpath,{lib_dir}"]
    else:
        cmd += ["-c", "-o", str(tmp_path / "distort.o")]
    subprocess.run(cmd, check=True)
    return exe


def test_distortion_header_compiles_without_gpu(tmp_path):
    _compile(tmp_path, link=False)


def test_new_symbols_are_exported():
    from aruco3_b200 import _ffi
    L = C.CDLL(str(_ffi.LIB_PATH))
    for name in ("a3_detector_set_distortion", "a3_undistort_points"):
        assert hasattr(L, name), name


def test_struct_layouts_match_the_header(tmp_path):
    """sizeof / offsetof of a3_camera_distortion and the new a3_stats fields: the C compiler against the ctypes mirror."""
    from aruco3_b200 import _ffi
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "aruco3_b200.h"\nint main(void) {\n'
                   'printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(a3_camera_distortion), offsetof(a3_camera_distortion, k2),'
                   ' offsetof(a3_camera_distortion, p1), offsetof(a3_camera_distortion, p2), offsetof(a3_camera_distortion, k3),'
                   ' sizeof(a3_stats), offsetof(a3_stats, undistort_kernel_launches), offsetof(a3_stats, ms_undistort_kernel));\nreturn 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    D, S = _ffi.A3CameraDistortion, _ffi.A3Stats
    assert got == [C.sizeof(D), D.k2.offset, D.p1.offset, D.p2.offset, D.k3.offset, C.sizeof(S), S.undistort_kernel_launches.offset,
                   S.ms_undistort_kernel.offset]


def _key(words):
    b = b"".join(int(x, 16).to_bytes(4, "little") for x in words[:26])
    return b + int(words[26]).to_bytes(4, "little") + bytes([int(words[27])])


@pytest.mark.gpu
def test_cpp_distortion_matches_oracle(oracle, tmp_path):
    from aruco3_b200 import _ffi, synth
    from oracle import a3ref_distort_py as od
    _ffi.lib()
    frames = np.stack([synth.render_board_frame(BOARD.ids, BOARD.corners, R, t, KP, W, H, noise=3, seed=j, distortion=BARREL)[0]
                       for j, (R, t) in enumerate(board_poses(3))])
    k = oracle.intrinsics_new(W, H, KP[0], KP[1], KP[2], KP[3])
    want = []
    for img in frames:
        res = oracle.detect(img, "ARUCO", oracle.default_config(**CFG))
        cs = np.array([m["corners"] for m in res.markers], np.float32).reshape(-1, 4, 2)
        b, a, n, ok = od.solve_frame(BOARD.ids, BOARD.corners, [m["id"] for m in res.markers], cs, k, od.distortion(*BARREL))
        want.append(bytes(b) + bytes(a) + int(n).to_bytes(4, "little") + bytes([int(ok)]))
    assert all(w[-1] for w in want)
    (tmp_path / "frames.rgb").write_bytes(frames.tobytes())
    exe = _compile(tmp_path)
    out = subprocess.run([str(exe), str(tmp_path / "frames.rgb"), str(len(frames))], check=True, capture_output=True,
                         text=True).stdout.splitlines()
    rows = {}
    for ln in out:
        tag, *words = ln.split()
        rows.setdefault(tag, []).append(words)
    for tag in ("det", "rebuilt", "plain", "sharded"):
        assert [_key(w) for w in rows[tag]] == want, tag
    assert [_key(w) for w in rows["off"]] != want  # the pinhole solve on distorted corners differs
