"""Seeded synthetic frames with ground truth (SURVEY.md §8d).

The reference ships no detector fixtures (its integration test renders an untextured quad and
never calls `detect`, `/root/reference/tests/integration_test_randomized_e2e.rs:5-10`), and its
benchmark feeds unseeded uniform noise (`/root/reference/benches/detect_markers.rs:37-45`).  This
module is the workload definition for BASELINE.json's configs: deterministic numpy code, PRNG =
splitmix64 seeded with `0xA3C0DE00 + 1000*config + frame_index`.

Rendering convention: interior cell (row-major, first cell = MSB of the table value) is white when
the bit is set — the order the decoder packs bits in (`/root/reference/src/aruco.rs:296-308`), so an
upright marker decodes with rotation 0 and `corners[0]` = the marker's own top-left (Q9).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from . import dictionaries

_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(seed: int, n: int) -> np.ndarray:
    """n outputs of splitmix64 started at `seed` (uint64 array)."""
    with np.errstate(over="ignore"):
        z = np.uint64(seed & 0xFFFFFFFFFFFFFFFF) + np.arange(1, n + 1, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


class Rng:
    """Tiny sequential wrapper: values are consumed in call order, so a frame is a pure function of its seed."""

    def __init__(self, seed: int):
        self.seed = seed & 0xFFFFFFFFFFFFFFFF
        self.pos = 0

    def u64(self, n: int) -> np.ndarray:
        with np.errstate(over="ignore"):
            start = (self.seed + self.pos * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        out = splitmix64(start, n)
        self.pos += n
        return out

    def uniform(self, n: int = 1) -> np.ndarray:
        return (self.u64(n) >> np.uint64(11)).astype(np.float64) / float(1 << 53)

    def randint(self, lo: int, hi: int) -> int:
        """Integer in [lo, hi]."""
        return lo + int(self.u64(1)[0] % np.uint64(hi - lo + 1))

    def bytes(self, n: int) -> np.ndarray:
        """n bytes, each u64 consumed low byte first."""
        words = self.u64((n + 7) // 8)
        return words.view(np.uint8)[:n] if words.dtype.byteorder in ("=", "<", "|") else words.byteswap().view(np.uint8)[:n]


@dataclass
class TruthMarker:
    id: int
    corners: np.ndarray  # float64 [4,2]: the marker's own TL, TR, BR, BL (outer edge of the black border), image px


@dataclass
class FrameSpec:
    """One of BASELINE.json's configs."""
    name: str
    config_index: int
    width: int
    height: int
    dictionary: str = "ARUCO"
    grid: tuple = (0, 0)          # (cols, rows) placement lattice; (0,0) = rejection sampling
    markers: tuple = (0, 0)       # inclusive range of markers per frame
    side: tuple = (0, 0)          # inclusive range of marker side, px
    noise: int = 0                # uniform +-noise per channel
    pure_noise: bool = False      # the reference bench workload: uniform random bytes
    min_corner_separation_factor: float = 0.1
    background: tuple = (204, 200, 192)
    white: tuple = (250, 248, 240)
    black: tuple = (24, 28, 36)
    extra: dict = field(default_factory=dict)


CONFIGS = {
    # tests/integration_test_randomized_e2e.rs as BASELINE.json describes it (the file itself renders no markers)
    "C1": FrameSpec("C1", 1, 640, 480, markers=(4, 8), side=(60, 120)),
    "C1n": FrameSpec("C1n", 1, 640, 480, markers=(4, 8), side=(60, 120), noise=4),
    # benches/detect_markers.rs: one 1920x1080 frame of uniform noise (seeded here)
    "C2a": FrameSpec("C2a", 2, 1920, 1080, pure_noise=True),
    # 1080p batch, 20 markers on a jittered 5x4 lattice (headline)
    "C3": FrameSpec("C3", 3, 1920, 1080, grid=(5, 4), markers=(20, 20), side=(100, 180)),
    "C3n": FrameSpec("C3n", 3, 1920, 1080, grid=(5, 4), markers=(20, 20), side=(100, 180), noise=4),
    # 4K sharded batch
    "C4": FrameSpec("C4", 4, 3840, 2160, grid=(5, 4), markers=(20, 20), side=(200, 360)),
    # decode stress: AprilTag 36h11, 220 small markers; the default discard radius (108 px) would delete
    # neighbours, so this config uses the public field min_corner_separation_factor = 0.03 (aruco.rs:27)
    "C5": FrameSpec("C5", 5, 1920, 1080, dictionary="APRILTAG_36H11", grid=(20, 11), markers=(220, 220),
                    side=(40, 56), min_corner_separation_factor=0.03),
}


def frame_seed(spec: FrameSpec, frame_index: int) -> int:
    return 0xA3C0DE00 + 1000 * spec.config_index + frame_index


def _square_to_quad(q: np.ndarray) -> np.ndarray:
    """Heckbert's closed form: 3x3 H with H @ (u,v,1) ~ image point, unit square -> quad q[4,2]."""
    (x0, y0), (x1, y1), (x2, y2), (x3, y3) = q
    dx1, dx2, dx3 = x1 - x2, x3 - x2, x0 - x1 + x2 - x3
    dy1, dy2, dy3 = y1 - y2, y3 - y2, y0 - y1 + y2 - y3
    den = dx1 * dy2 - dx2 * dy1
    g = (dx3 * dy2 - dx2 * dy3) / den
    h = (dx1 * dy3 - dx3 * dy1) / den
    return np.array([[x1 - x0 + g * x1, x3 - x0 + h * x3, x0],
                     [y1 - y0 + g * y1, y3 - y0 + h * y3, y0],
                     [g, h, 1.0]])


def _adjugate(m: np.ndarray) -> np.ndarray:
    a, b, c, d, e, f, g, h, i = m.ravel()
    return np.array([[e * i - f * h, c * h - b * i, b * f - c * e],
                     [f * g - d * i, a * i - c * g, c * d - a * f],
                     [d * h - e * g, b * g - a * h, a * e - b * d]])


def marker_cells(table: dictionaries.DictionaryTable, marker_id: int) -> np.ndarray:
    """ms x ms uint8 grid, 1 = white. Border black; interior row-major, first cell = MSB."""
    ms = table.mark_size
    inner = ms - 2
    code = int(table.codes[marker_id])
    nb = inner * inner
    cells = np.zeros((ms, ms), dtype=np.uint8)
    for k in range(nb):
        bit = (code >> (nb - 1 - k)) & 1 if nb - 1 - k < 64 else 0
        cells[1 + k // inner, 1 + k % inner] = bit
    return cells


def draw_marker(img: np.ndarray, cells: np.ndarray, quad: np.ndarray, white, black) -> None:
    """Paint a marker whose outer square maps to `quad` (TL,TR,BR,BL image px) with pixel-centre sampling."""
    h, w = img.shape[:2]
    ms = cells.shape[0]
    x_lo = max(int(np.floor(quad[:, 0].min())) - 1, 0)
    x_hi = min(int(np.ceil(quad[:, 0].max())) + 1, w - 1)
    y_lo = max(int(np.floor(quad[:, 1].min())) - 1, 0)
    y_hi = min(int(np.ceil(quad[:, 1].max())) + 1, h - 1)
    if x_hi < x_lo or y_hi < y_lo:
        return
    inv = _adjugate(_square_to_quad(quad))
    xs = np.arange(x_lo, x_hi + 1, dtype=np.float64) + 0.5
    ys = np.arange(y_lo, y_hi + 1, dtype=np.float64) + 0.5
    gx, gy = np.meshgrid(xs, ys)
    den = inv[2, 0] * gx + inv[2, 1] * gy + inv[2, 2]
    u = (inv[0, 0] * gx + inv[0, 1] * gy + inv[0, 2]) / den * ms
    v = (inv[1, 0] * gx + inv[1, 1] * gy + inv[1, 2]) / den * ms
    inside = (u >= 0) & (u < ms) & (v >= 0) & (v < ms)
    ci = np.clip(np.floor(u).astype(np.int64), 0, ms - 1)
    cj = np.clip(np.floor(v).astype(np.int64), 0, ms - 1)
    is_white = cells[cj, ci].astype(bool)
    region = img[y_lo:y_hi + 1, x_lo:x_hi + 1]
    region[inside & is_white] = white
    region[inside & ~is_white] = black


def _place(spec: FrameSpec, rng: Rng, n: int):
    """Centres + sides. Lattice placement when spec.grid is set, else rejection sampling."""
    sides = [rng.randint(*spec.side) for _ in range(n)]
    centres = []
    if spec.grid != (0, 0):
        gc, gr = spec.grid
        cw, ch = spec.width / gc, spec.height / gr
        order = np.argsort(rng.u64(gc * gr), kind="stable")[:n]
        for k, cell in enumerate(order):
            r = sides[k] * 0.5 * np.sqrt(2.0) * 1.07 + 3.0
            jx = max(cw * 0.5 - r, 0.0)
            jy = max(ch * 0.5 - r, 0.0)
            u = rng.uniform(2)
            cx = (cell % gc + 0.5) * cw + (2 * u[0] - 1) * jx
            cy = (cell // gc + 0.5) * ch + (2 * u[1] - 1) * jy
            centres.append((cx, cy))
        return centres, sides
    kept_sides = []
    for k in range(n):
        r = sides[k] * 0.5 * np.sqrt(2.0) * 1.07 + 3.0
        for _ in range(200):
            u = rng.uniform(2)
            cx = r + u[0] * (spec.width - 2 * r)
            cy = r + u[1] * (spec.height - 2 * r)
            if all((cx - ox) ** 2 + (cy - oy) ** 2 >= (r + orr + 10.0) ** 2
                   for (ox, oy), orr in zip(centres, [s * 0.5 * np.sqrt(2.0) * 1.07 + 3.0 for s in kept_sides])):
                centres.append((cx, cy))
                kept_sides.append(sides[k])
                break
    return centres, kept_sides


def render_frame(spec: FrameSpec, frame_index: int):
    """-> (uint8 [H,W,3], [TruthMarker])."""
    rng = Rng(frame_seed(spec, frame_index))
    if spec.pure_noise:
        return rng.bytes(spec.width * spec.height * 3).reshape(spec.height, spec.width, 3).copy(), []
    table = dictionaries.table(spec.dictionary)
    img = np.empty((spec.height, spec.width, 3), dtype=np.uint8)
    img[:] = np.array(spec.background, dtype=np.uint8)
    n = rng.randint(*spec.markers)
    centres, sides = _place(spec, rng, n)
    truth = []
    for (cx, cy), side in zip(centres, sides):
        marker_id = rng.randint(0, len(table.codes) - 1)
        u = rng.uniform(9)
        ang = 2.0 * np.pi * u[0]
        ca, sa = np.cos(ang), np.sin(ang)
        half = side * 0.5
        base = np.array([[-half, -half], [half, -half], [half, half], [-half, half]])  # TL TR BR BL, y down
        jitter = (u[1:9].reshape(4, 2) * 2.0 - 1.0) * (0.06 * side * 0.5)
        pts = base + jitter
        quad = np.stack([cx + ca * pts[:, 0] - sa * pts[:, 1], cy + sa * pts[:, 0] + ca * pts[:, 1]], axis=1)
        draw_marker(img, marker_cells(table, marker_id), quad, spec.white, spec.black)
        truth.append(TruthMarker(marker_id, quad))
    if spec.noise:
        nz = rng.bytes(img.size).reshape(img.shape)
        delta = (nz % np.uint8(2 * spec.noise + 1)).astype(np.int16) - spec.noise
        img = np.clip(img.astype(np.int16) + delta, 0, 255).astype(np.uint8)
    return img, truth


def render_batch(spec, n_frames: int, first_index: int = 0, out: np.ndarray | None = None):
    """-> (uint8 [n,H,W,3], [[TruthMarker]]). `spec` may be a config name."""
    if isinstance(spec, str):
        spec = CONFIGS[spec]
    if out is None:
        out = np.empty((n_frames, spec.height, spec.width, 3), dtype=np.uint8)
    truths = []
    for i in range(n_frames):
        img, truth = render_frame(spec, first_index + i)
        out[i] = img
        truths.append(truth)
    return out, truths


# ---- planar boards seen from a known pose (kernel K6) ------------------------------------------------------------------
def _coefficients(distortion) -> np.ndarray:
    """(k1, k2, p1, p2, k3) in f64 from a pose.CameraDistortion or a sequence of five numbers"""
    c = distortion.coefficients() if hasattr(distortion, "coefficients") else distortion
    return np.asarray(c, np.float64).reshape(5)


def distort_normalized(x: np.ndarray, y: np.ndarray, distortion):
    """OpenCV's forward model (k1 k2 p1 p2 k3) on normalised points, f64."""
    k1, k2, p1, p2, k3 = _coefficients(distortion)
    r2 = x * x + y * y
    rad = 1.0 + r2 * (k1 + r2 * (k2 + r2 * k3))
    return x * rad + 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x), y * rad + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y


def undistort_normalized(xd: np.ndarray, yd: np.ndarray, distortion, iters: int = 30):
    """The inverse of distort_normalized by a vectorised f64 Newton solve from the distorted point -> (x, y, ok); ok is
    False where the model folds (Jacobian determinant <= 0) or the solve does not converge to 1e-12."""
    k1, k2, p1, p2, k3 = _coefficients(distortion)
    x, y = xd.astype(np.float64).copy(), yd.astype(np.float64).copy()
    ok = np.isfinite(x) & np.isfinite(y)
    for _ in range(iters):
        r2 = x * x + y * y
        rad = 1.0 + r2 * (k1 + r2 * (k2 + r2 * k3))
        fx = x * rad + 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x) - xd
        fy = y * rad + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y - yd
        if not (np.maximum(np.abs(fx), np.abs(fy))[ok] > 1e-12).any():
            break
        dr = k1 + r2 * (2.0 * k2 + 3.0 * k3 * r2)
        j00 = rad + 2.0 * x * x * dr + 2.0 * p1 * y + 6.0 * p2 * x
        j01 = 2.0 * x * y * dr + 2.0 * p1 * x + 2.0 * p2 * y
        j11 = rad + 2.0 * y * y * dr + 6.0 * p1 * y + 2.0 * p2 * x
        det = j00 * j11 - j01 * j01
        ok &= det > 0
        det = np.where(ok, det, 1.0)
        x = np.where(ok, x - (fx * j11 - fy * j01) / det, x)
        y = np.where(ok, y - (j00 * fy - j01 * fx) / det, y)
    r2 = x * x + y * y
    rad = 1.0 + r2 * (k1 + r2 * (k2 + r2 * k3))
    res = np.maximum(np.abs(x * rad + 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x) - xd),
                     np.abs(y * rad + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y - yd))
    return x, y, ok & (res <= 1e-12)


def project_points(points: np.ndarray, R: np.ndarray, t: np.ndarray, k: tuple, distortion=None) -> np.ndarray:
    """Board points [n, 2] (z = 0) -> image points [n, 2] under X = R p + t and the pinhole k = (fx, fy, cx, cy), in the
    pixel-centre convention (grey pixel (x, y) is the point (x, y)).  `distortion` (pose.CameraDistortion or OpenCV's
    five coefficients): the lens model applied to the normalised point before the pinhole, as cv2.projectPoints does."""
    p = np.asarray(points, np.float64).reshape(-1, 2)
    X = p @ np.asarray(R, np.float64)[:, :2].T + np.asarray(t, np.float64)
    fx, fy, cx, cy = k
    x, y = X[:, 0] / X[:, 2], X[:, 1] / X[:, 2]
    if distortion is not None:
        x, y = distort_normalized(x, y, distortion)
    return np.stack([fx * x + cx, fy * y + cy], axis=1)


def _render_distorted(board_ids, board_corners, R, t, k: tuple, width: int, height: int, table, spec, distortion, ss: int):
    """The board through pinhole k and the lens model: every output pixel is the mean of ss x ss samples, each undistorted
    (f64 Newton) onto a pinhole image of the board rendered at ss times the resolution and read bilinearly there."""
    fx, fy, cx, cy = k
    sub = (np.arange(ss, dtype=np.float64) + 0.5) / ss - 0.5  # sample offsets in the pixel-centre convention
    gx = (np.arange(width, dtype=np.float64)[:, None] + sub[None, :]).reshape(-1)
    gy = (np.arange(height, dtype=np.float64)[:, None] + sub[None, :]).reshape(-1)
    X, Y = np.meshgrid(gx, gy)  # [H ss, W ss]
    xu, yu, ok = undistort_normalized((X - cx) / fx, (Y - cy) / fy, distortion)
    qx, qy = fx * xu + cx, fy * yu + cy  # pinhole pixel of every sample (pixel-centre convention)
    lo_x, hi_x = np.floor(qx[ok].min()) - 2, np.ceil(qx[ok].max()) + 2
    lo_y, hi_y = np.floor(qy[ok].min()) - 2, np.ceil(qy[ok].max()) + 2
    cw, ch = int((hi_x - lo_x) * ss) + 1, int((hi_y - lo_y) * ss) + 1
    canvas = np.empty((ch, cw, 3), dtype=np.uint8)
    canvas[:] = np.array(spec.background, dtype=np.uint8)
    for mid, corners in zip(np.asarray(board_ids).reshape(-1), np.asarray(board_corners, np.float64).reshape(-1, 4, 2)):
        quad = (project_points(corners, R, t, k) + 0.5 - np.array([lo_x, lo_y])) * ss  # draw_marker's convention on the canvas
        draw_marker(canvas, marker_cells(table, int(mid)), quad, spec.white, spec.black)
    # canvas pixel (i, j) is sampled at pinhole pixel-centre point ((i + 0.5) / ss + lo - 0.5)
    u = np.where(ok, (qx - lo_x + 0.5) * ss - 0.5, 0.0)
    v = np.where(ok, (qy - lo_y + 0.5) * ss - 0.5, 0.0)
    i0 = np.clip(np.floor(u).astype(np.int64), 0, cw - 2)
    j0 = np.clip(np.floor(v).astype(np.int64), 0, ch - 2)
    a = np.clip(u - i0, 0.0, 1.0)[..., None]
    b = np.clip(v - j0, 0.0, 1.0)[..., None]
    c = canvas.astype(np.float32)
    a, b = a.astype(np.float32), b.astype(np.float32)
    val = (c[j0, i0] * (1 - a) + c[j0, i0 + 1] * a) * (1 - b) + (c[j0 + 1, i0] * (1 - a) + c[j0 + 1, i0 + 1] * a) * b
    val[~ok] = np.array(spec.background, np.float32)
    img = val.reshape(height, ss, width, ss, 3).mean(axis=(1, 3))
    return np.clip(np.rint(img), 0, 255).astype(np.uint8)


def render_board_frame(board_ids, board_corners, R, t, k: tuple, width: int, height: int, dictionary: str = "ARUCO",
                       extra_ids=(), noise: int = 0, seed: int = 0, distortion=None, supersample: int = 2):
    """A planar board seen from pose (R, t) with pinhole k = (fx, fy, cx, cy) -> (uint8 [H, W, 3], [TruthMarker]).

    A pinhole view of a plane is a homography, so drawing each marker on its projected quad is exact.  There is no sheet
    around the markers (its outline would become a quad of its own).  `extra_ids`: markers that are not on the board, drawn
    in the frame's corners (keep the board away from them).  Truth corners are in draw_marker's convention (+0.5 px from the
    pixel-centre convention of project_points and of refined corners).

    `distortion` (pose.CameraDistortion or OpenCV's five coefficients): the view through that lens.  It is no longer a
    homography, so the frame is rendered by inverse mapping (`supersample`^2 samples per pixel, see _render_distorted) and
    the truth corners are the distorted projections.  The extra markers are drawn undistorted on top."""
    table = dictionaries.table(dictionary)
    spec = FrameSpec("board", 0, width, height)
    img = np.empty((height, width, 3), dtype=np.uint8)
    img[:] = np.array(spec.background, dtype=np.uint8)
    truth = []
    if distortion is not None:
        img = _render_distorted(board_ids, board_corners, R, t, k, width, height, table, spec, distortion, supersample)
    for mid, corners in zip(np.asarray(board_ids).reshape(-1), np.asarray(board_corners, np.float64).reshape(-1, 4, 2)):
        quad = project_points(corners, R, t, k, distortion) + 0.5
        if distortion is None:
            draw_marker(img, marker_cells(table, int(mid)), quad, spec.white, spec.black)
        truth.append(TruthMarker(int(mid), quad))
    side = 0.12 * min(width, height)
    spots = [(0.04 * width, 0.04 * height), (width - 0.04 * width - side, 0.04 * height),
             (0.04 * width, height - 0.04 * height - side), (width - 0.04 * width - side, height - 0.04 * height - side)]
    for mid, (x0, y0) in zip(extra_ids, spots):
        quad = np.array([[x0, y0], [x0 + side, y0], [x0 + side, y0 + side], [x0, y0 + side]])
        draw_marker(img, marker_cells(table, int(mid)), quad, spec.white, spec.black)
        truth.append(TruthMarker(int(mid), quad))
    if noise:
        rng = Rng(seed)
        nz = rng.bytes(img.size).reshape(img.shape)
        delta = (nz % np.uint8(2 * noise + 1)).astype(np.int16) - noise
        img = np.clip(img.astype(np.int16) + delta, 0, 255).astype(np.uint8)
    return img, truth


def board_views(n: int, seed: int = 0, distance: tuple = (300.0, 420.0), tilt: float = 0.45):
    """n seeded poses (R, t) of a board facing the camera: board y up -> image y down, the board's face toward the camera,
    tilted by up to `tilt` radians about each in-plane axis, at `distance` along the optical axis."""
    rng = Rng(seed)
    out = []
    for _ in range(n):
        u = rng.uniform(6)
        ax, ay, az = (u[0] * 2 - 1) * tilt, (u[1] * 2 - 1) * tilt, (u[2] * 2 - 1) * 0.5
        cx_, sx_ = np.cos(ax), np.sin(ax)
        cy_, sy_ = np.cos(ay), np.sin(ay)
        cz_, sz_ = np.cos(az), np.sin(az)
        rx = np.array([[1, 0, 0], [0, cx_, -sx_], [0, sx_, cx_]])
        ry = np.array([[cy_, 0, sy_], [0, 1, 0], [-sy_, 0, cy_]])
        rz = np.array([[cz_, -sz_, 0], [sz_, cz_, 0], [0, 0, 1]])
        facing = np.diag([1.0, -1.0, -1.0])
        R = rz @ ry @ rx @ facing
        z = distance[0] + (distance[1] - distance[0]) * u[3]
        t = np.array([(u[4] * 2 - 1) * 0.05 * z, (u[5] * 2 - 1) * 0.05 * z, z])
        out.append((R, t))
    return out
