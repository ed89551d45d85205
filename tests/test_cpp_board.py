"""The board pose (kernel K6) through the C++ mirror (include/aruco3_b200.hpp): aruco3::Board, Detector::set_board,
Detection::board_pose, the PlainDetector option and ShardedDetector::set_board, compiled with g++, run on the GPU and
compared bit for bit with the CPU oracle."""
import subprocess
from pathlib import Path

import pytest

from tests.test_gpu_board import _frames, expected

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
    const uint32_t w = 640, h = 480, n = (uint32_t)atoi(argv[2]);
    const bool intr = argv[3][0] == '1', refined = argv[4][0] == '1';
    std::vector<uint8_t> rgb((size_t)n * w * h * 3);
    FILE *f = fopen(argv[1], "rb");
    if (!f || fread(rgb.data(), 1, rgb.size(), f) != rgb.size()) return 2;
    fclose(f);
    const aruco3::Board board = aruco3::Board::grid(4, 3, 40.0f, 10.0f);
    const float px = 320.0f, py = 240.0f;
    const aruco3::CameraIntrinsics k(w, h, 800.0f, 800.0f, &px, &py);
    const aruco3::DetectorConfig cfg;
    const auto dict = aruco3::ARDictionary::new_from_named_dict("ARUCO");
    aruco3::Detector det(cfg, dict, 0);
    det.set_corner_refinement(refined);
    det.set_board(&board, intr ? &k : nullptr);
    put("det", det.detect_batch(rgb.data(), n, w, h));
    det.rebuild();  // the board survives a rebuild
    put("rebuilt", det.detect_batch(rgb.data(), n, w, h, aruco3::PixelFormat::Rgb8, true));
    aruco3::PlainDetector plain{cfg, dict, 0, refined, board, intr ? std::optional<aruco3::CameraIntrinsics>(k) : std::nullopt};
    put("plain", plain.detect_batch(rgb.data(), n, w, h));
    aruco3::ShardedDetector sharded(cfg, dict, {0, 0});
    sharded.set_corner_refinement(refined);
    sharded.set_board(&board, intr ? &k : nullptr);
    put("sharded", sharded.detect_batch(rgb.data(), n, w, h));
    det.set_board(nullptr);
    put("off", det.detect_batch(rgb.data(), n, w, h));
    return 0;
}
'''


def _compile(tmp_path, link=True):
    src, exe = tmp_path / "board.cpp", tmp_path / "board"
    src.write_text(PROGRAM)
    lib_dir = ROOT / "aruco3_b200"
    cmd = ["g++", "-std=c++17", "-Wall", "-pthread", "-I", str(ROOT / "include"), str(src)]
    if link:
        cmd += ["-o", str(exe), f"-L{lib_dir}", "-laruco3_b200", f"-Wl,-rpath,{lib_dir}"]
    else:
        cmd += ["-c", "-o", str(tmp_path / "board.o")]
    subprocess.run(cmd, check=True)
    return exe


def test_board_header_compiles_without_gpu(tmp_path):
    _compile(tmp_path, link=False)


def _key(words):
    b = b"".join(int(x, 16).to_bytes(4, "little") for x in words[:26])
    return b + int(words[26]).to_bytes(4, "little") + bytes([int(words[27])])


@pytest.mark.gpu
@pytest.mark.parametrize("refined", [False, True], ids=["integer", "refined"])
@pytest.mark.parametrize("intrinsics", [False, True], ids=["undistorted", "intrinsics"])
def test_cpp_board_matches_oracle(oracle, tmp_path, refined, intrinsics):
    from aruco3_b200 import _ffi
    from oracle import a3ref_board_py as ob
    _ffi.lib()
    board, frames = _frames()
    want = expected(oracle, ob, board, frames, refined, intrinsics)
    (tmp_path / "frames.rgb").write_bytes(frames.tobytes())
    exe = _compile(tmp_path)
    out = subprocess.run([str(exe), str(tmp_path / "frames.rgb"), str(len(frames)), "1" if intrinsics else "0", "1" if refined else "0"],
                         check=True, capture_output=True, text=True).stdout.splitlines()
    rows = {}
    for ln in out:
        tag, *words = ln.split()
        rows.setdefault(tag, []).append(words)
    for tag in ("det", "rebuilt", "plain", "sharded"):
        assert [_key(w) for w in rows[tag]] == want, tag
    assert rows["off"] == [["none"]] * len(frames)
