"""Planar marker boards and their per-frame pose (kernel K6, include/aruco3_b200.h `a3_board` / `a3_board_pose`).

A board is a rigid sheet of markers: ids and each marker's four corners on the board plane (z = 0), in any length unit,
in the order of `Marker.corners` (the marker's own TL, TR, BR, BL), x to the right and y up on the board's face.
`Detector.set_board(board)` makes `detect` / `detect_batch` also return the sheet's pose in every frame
(`Detection.board_pose`), solved on the device from every visible marker of the board.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from ._ffi import A3Board, A3BoardPose
from .pose import MarkerPose


class Board:
    """`ids` [m] (distinct, below the dictionary's code count) and `corners` [m, 4, 2] board-plane points."""

    def __init__(self, ids, corners):
        self.ids = np.ascontiguousarray(np.asarray(ids, np.uint64).reshape(-1))
        self.corners = np.ascontiguousarray(np.asarray(corners, np.float32).reshape(-1, 4, 2))
        if self.corners.shape[0] != self.ids.shape[0]:
            raise ValueError(f"Board: {self.ids.shape[0]} ids but {self.corners.shape[0]} corner sets")

    @staticmethod
    def grid(cols: int, rows: int, marker_size: float, separation: float, first_id: int = 0) -> "Board":
        """A cols x rows grid of square markers `separation` apart, centred on the origin; row 0 at the top, ids row-major
        from `first_id` (the layout of OpenCV's GridBoard, with y up)."""
        pitch = marker_size + separation
        w, h = cols * marker_size + (cols - 1) * separation, rows * marker_size + (rows - 1) * separation
        corners = []
        for r in range(rows):
            for c in range(cols):
                x0, y0 = -w / 2 + c * pitch, h / 2 - r * pitch
                corners.append([(x0, y0), (x0 + marker_size, y0), (x0 + marker_size, y0 - marker_size), (x0, y0 - marker_size)])
        return Board(np.arange(first_id, first_id + cols * rows), corners)

    def __len__(self):
        return int(self.ids.shape[0])

    def to_c(self) -> A3Board:
        """The C view; it points into this object's arrays, so keep the Board alive while the view is used."""
        return A3Board(len(self), self.ids.ctypes.data_as(C.POINTER(C.c_uint64)), self.corners.ctypes.data_as(C.POINTER(C.c_float)))


@dataclass
class BoardPose:
    """The board's pose in one frame: board points (x, y, 0) -> camera, as `MarkerPose`.  `best` has the smaller error (RMS
    reprojection distance over the used corners, normalised units), `alt` is the other branch of the planar ambiguity;
    `n_markers` markers were used; `ok` is False when both branches failed or no board marker was seen."""
    best: MarkerPose
    alt: MarkerPose
    n_markers: int
    ok: bool

    @staticmethod
    def from_c(p: A3BoardPose) -> "BoardPose":
        return BoardPose(MarkerPose.from_c(p.best), MarkerPose.from_c(p.alt), int(p.n_markers), bool(p.ok))
