"""Deterministic synthetic AprilTag scenes (the inputs SURVEY.md section 8(d) specifies).

Pure numpy, IEEE double arithmetic with only + - * / floor, so a seed gives the
same bytes on every host.  Tags are tag36h11 bitmaps (1-cell white quiet zone,
8x8 black border, 6x6 data) rendered through a homography with SxS supersampling.

The frame formats mirror what reaches the reference detector: YUYV 4:2:2
(GpuDetector::Detect, src/apriltags_cuda/src/apriltag_gpu.cu:725-729), the
`bgr8` image the node receives (apriltags_cuda_detector.cu:399) and plain gray.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

from .tag_families import FAMILIES


@dataclass
class TagPose:
    tag_id: int
    corners: np.ndarray  # (4,2) image positions of tag-frame (-1,-1),(1,-1),(1,1),(-1,1)
    family: str = "tag36h11"


@dataclass
class Scene:
    gray: np.ndarray  # (H, W) uint8
    tags: list = field(default_factory=list)


def tag_pattern(tag_id: int, family: str = "tag36h11") -> np.ndarray:
    """total_width x total_width cell image (1 = white) of tag `tag_id` of `family`, one-cell quiet zone included
    (10 x 10 for tag36h11: black border 8 x 8, data 6 x 6)."""
    fam = FAMILIES[family]
    tw, wb, nbits = fam["total_width"], fam["width_at_border"], fam["nbits"]
    pat = np.ones((tw, tw), dtype=np.float64)
    pat[1:1 + wb, 1:1 + wb] = 0.0
    code = fam["codes"][tag_id]
    for i in range(nbits):
        bit = (code >> (nbits - 1 - i)) & 1
        # border cell (bx, by) in [0, width_at_border) sits at pattern cell (bx+1, by+1)
        pat[fam["bit_y"][i] + 1, fam["bit_x"][i] + 1] = float(bit)
    return pat


def solve_homography(src, dst) -> np.ndarray:
    """3x3 H (H[2,2]=1) with dst ~ H*src from 4 correspondences; plain Gaussian elimination."""
    A = []
    for (x, y), (u, v) in zip(src, dst):
        A.append([x, y, 1.0, 0.0, 0.0, 0.0, -x * u, -y * u, u])
        A.append([0.0, 0.0, 0.0, x, y, 1.0, -x * v, -y * v, v])
    A = [list(map(float, r)) for r in A]
    n = 8
    for col in range(n):
        piv = max(range(col, n), key=lambda r: abs(A[r][col]))
        A[col], A[piv] = A[piv], A[col]
        for r in range(col + 1, n):
            f = A[r][col] / A[col][col]
            for k in range(col, 9):
                A[r][k] -= f * A[col][k]
    h = [0.0] * 8
    for col in range(n - 1, -1, -1):
        s = A[col][8]
        for k in range(col + 1, n):
            s -= A[col][k] * h[k]
        h[col] = s / A[col][col]
    return np.array(h + [1.0], dtype=np.float64).reshape(3, 3)


def _invert3(H: np.ndarray) -> np.ndarray:
    a, b, c, d, e, f, g, h, i = [float(v) for v in H.reshape(9)]
    A = e * i - f * h
    B = -(d * i - f * g)
    C = d * h - e * g
    det = a * A + b * B + c * C
    inv = np.array(
        [[A, -(b * i - c * h), b * f - c * e], [B, a * i - c * g, -(a * f - c * d)], [C, -(a * h - b * g), a * e - b * d]],
        dtype=np.float64,
    )
    return inv / det


def render_tag(img: np.ndarray, pose: TagPose, white: float, black: float, ss: int = 4) -> None:
    """Composite one tag into float image `img` (H, W) in place."""
    Himg, Wimg = img.shape
    tag_pts = [(-1.0, -1.0), (1.0, -1.0), (1.0, 1.0), (-1.0, 1.0)]
    H = solve_homography(tag_pts, [tuple(map(float, p)) for p in pose.corners])
    Hi = _invert3(H)
    fam = FAMILIES[pose.family]
    cell = 2.0 / fam["width_at_border"]   # the black border spans [-1, 1] in tag units
    # outer extent of the quiet zone: +-1.25 in tag units for tag36h11
    q = 1.0 + cell
    outer = []
    for x, y in [(-q, -q), (q, -q), (q, q), (-q, q)]:
        X = H[0, 0] * x + H[0, 1] * y + H[0, 2]
        Y = H[1, 0] * x + H[1, 1] * y + H[1, 2]
        Z = H[2, 0] * x + H[2, 1] * y + H[2, 2]
        outer.append((X / Z, Y / Z))
    xs = [p[0] for p in outer]
    ys = [p[1] for p in outer]
    x0 = max(0, int(math.floor(min(xs))) - 1)
    x1 = min(Wimg, int(math.ceil(max(xs))) + 2)
    y0 = max(0, int(math.floor(min(ys))) - 1)
    y1 = min(Himg, int(math.ceil(max(ys))) + 2)
    if x1 <= x0 or y1 <= y0:
        return
    bw, bh = x1 - x0, y1 - y0
    # pixel (x, y) covers [x, x+1) x [y, y+1); sub-sample centres
    sub = (np.arange(ss, dtype=np.float64) + 0.5) / ss
    px = (x0 + np.arange(bw, dtype=np.float64))[:, None] + sub[None, :]
    py = (y0 + np.arange(bh, dtype=np.float64))[:, None] + sub[None, :]
    PX = px.reshape(1, bw * ss)
    PY = py.reshape(bh * ss, 1)
    Z = Hi[2, 0] * PX + Hi[2, 1] * PY + Hi[2, 2]
    TX = (Hi[0, 0] * PX + Hi[0, 1] * PY + Hi[0, 2]) / Z
    TY = (Hi[1, 0] * PX + Hi[1, 1] * PY + Hi[1, 2]) / Z
    inside = (TX >= -q) & (TX < q) & (TY >= -q) & (TY < q) & (Z > 0)
    cx = np.floor((TX + q) / cell).astype(np.int64)
    cy = np.floor((TY + q) / cell).astype(np.int64)
    np.clip(cx, 0, fam["total_width"] - 1, out=cx)
    np.clip(cy, 0, fam["total_width"] - 1, out=cy)
    pat = tag_pattern(pose.tag_id, pose.family)
    val = pat[cy, cx] * (white - black) + black
    val = np.where(inside, val, 0.0)
    cov = inside.astype(np.float64)
    val = val.reshape(bh, ss, bw, ss).sum(axis=(1, 3))
    cov = cov.reshape(bh, ss, bw, ss).sum(axis=(1, 3))
    n = float(ss * ss)
    region = img[y0:y1, x0:x1]
    img[y0:y1, x0:x1] = (val + region * (n - cov)) / n


def random_pose(rng: np.random.Generator, tag_id: int, cx: float, cy: float, side: float, max_rot_deg: float,
                max_tilt_deg: float) -> TagPose:
    """Square of side `side` px (black-border edge), rotated in-plane and tilted about a random axis."""
    rot = math.radians(float(rng.uniform(-max_rot_deg, max_rot_deg)))
    tilt = math.radians(float(rng.uniform(0.0, max_tilt_deg)))
    axis = float(rng.uniform(0.0, 2.0 * math.pi))
    f = 4.0 * side  # focal length in px for the mini pinhole model
    ax, ay = math.cos(axis), math.sin(axis)
    c, s = math.cos(tilt), math.sin(tilt)
    # Rodrigues rotation about (ax, ay, 0)
    R = np.array(
        [[c + ax * ax * (1 - c), ax * ay * (1 - c), ay * s], [ax * ay * (1 - c), c + ay * ay * (1 - c), -ax * s],
         [-ay * s, ax * s, c]], dtype=np.float64)
    cr, sr = math.cos(rot), math.sin(rot)
    corners = []
    for tx, ty in [(-1.0, -1.0), (1.0, -1.0), (1.0, 1.0), (-1.0, 1.0)]:
        x = (tx * cr - ty * sr) * side / 2.0
        y = (tx * sr + ty * cr) * side / 2.0
        X = R[0, 0] * x + R[0, 1] * y
        Y = R[1, 0] * x + R[1, 1] * y
        Zc = R[2, 0] * x + R[2, 1] * y + f
        corners.append((cx + f * X / Zc, cy + f * Y / Zc))
    return TagPose(tag_id, np.array(corners, dtype=np.float64))


def make_scene(width: int, height: int, seed: int, n_tags: int, side_range=(60.0, 300.0), ids=None,
               max_rot_deg: float = 30.0, max_tilt_deg: float = 35.0, noise_sigma: float = 4.0,
               background: float = 128.0, clutter: bool = False, salt_pepper: float = 0.0,
               white: float = 230.0, black: float = 25.0, ss: int = 4, family: str = "tag36h11") -> Scene:
    rng = np.random.default_rng(seed)
    img = np.full((height, width), float(background), dtype=np.float64)
    if clutter:
        for _ in range(200):  # random rectangles
            w = int(rng.integers(10, max(11, width // 8)))
            h = int(rng.integers(10, max(11, height // 8)))
            x = int(rng.integers(0, width - w))
            y = int(rng.integers(0, height - h))
            img[y:y + h, x:x + w] = float(rng.integers(20, 236))
        for _ in range(20):  # checker patches
            cell = int(rng.integers(4, 24))
            nx, ny = int(rng.integers(3, 9)), int(rng.integers(3, 9))
            x = int(rng.integers(0, max(1, width - cell * nx)))
            y = int(rng.integers(0, max(1, height - cell * ny)))
            yy, xx = np.mgrid[0:cell * ny, 0:cell * nx]
            chk = ((xx // cell + yy // cell) % 2).astype(np.float64) * 180.0 + 40.0
            hh = min(cell * ny, height - y)
            ww = min(cell * nx, width - x)
            img[y:y + hh, x:x + ww] = chk[:hh, :ww]
    tags = []
    placed = []
    attempts = 0
    while len(tags) < n_tags and attempts < n_tags * 200:
        attempts += 1
        side = float(rng.uniform(side_range[0], side_range[1]))
        rad = side * 0.95  # circumscribed radius incl. quiet zone ~ side*1.25*sqrt2/2
        if 2 * rad + 4 >= min(width, height):
            side = (min(width, height) - 8) / 2.0
            rad = side * 0.95
        cx = float(rng.uniform(rad + 2, width - rad - 2))
        cy = float(rng.uniform(rad + 2, height - rad - 2))
        if any((cx - px) ** 2 + (cy - py) ** 2 < (rad + pr) ** 2 for px, py, pr in placed):
            continue
        tid = int(ids[len(tags)]) if ids is not None else int(rng.integers(0, len(FAMILIES[family]["codes"])))
        pose = random_pose(rng, tid, cx, cy, side, max_rot_deg, max_tilt_deg)
        pose.family = family
        render_tag(img, pose, white, black, ss)
        placed.append((cx, cy, rad))
        tags.append(pose)
    if noise_sigma > 0:
        img = img + rng.normal(0.0, noise_sigma, size=img.shape)
    if salt_pepper > 0:
        m = rng.random(img.shape)
        img = np.where(m < salt_pepper / 2, 0.0, img)
        img = np.where(m > 1.0 - salt_pepper / 2, 255.0, img)
    gray = np.clip(np.floor(img + 0.5), 0, 255).astype(np.uint8)
    return Scene(gray, tags)


def field_scene(width: int, height: int, layout, tagsize: float, camera_R, camera_t, fx: float, fy: float, cx: float,
                cy: float, seed: int, noise_sigma: float = 2.0, family: str = "tag36h11", background: float = 128.0,
                white: float = 230.0, black: float = 25.0, ss: int = 4) -> Scene:
    """A gray frame of the tags of a field layout (detector.FIELD_TAG_DT records, X_field = R X_tag + t) seen by a
    pinhole camera placed in the field by X_field = camera_R X_cam + camera_t.  Each tag's black-border corners are
    projected; the tags lying fully in front of the camera and inside the frame are rendered, farthest first.  TagPose
    corners (-1,-1), (1,-1), (1,1), (-1,1) are the tag points (-s,-s), (s,-s), (s,s), (-s,s), s = tagsize / 2.  Returns the
    Scene: the frame and the rendered tags with their true corners."""
    rng = np.random.default_rng(seed)
    Rc = np.asarray(camera_R, dtype=np.float64).reshape(3, 3)
    tc = np.asarray(camera_t, dtype=np.float64).reshape(3)
    s = tagsize / 2.0
    P = np.array([[-s, -s, 0.0], [s, -s, 0.0], [s, s, 0.0], [-s, s, 0.0]])
    visible = []
    for rec in np.asarray(layout):
        X = P @ np.asarray(rec["R"], dtype=np.float64).reshape(3, 3).T + np.asarray(rec["t"], dtype=np.float64)
        cam = (X - tc) @ Rc  # Rc^T (X - tc), row by row
        if not (cam[:, 2] > 1e-6).all():
            continue
        px = np.stack([fx * cam[:, 0] / cam[:, 2] + cx, fy * cam[:, 1] / cam[:, 2] + cy], axis=1)
        if (px[:, 0] < 0).any() or (px[:, 0] > width).any() or (px[:, 1] < 0).any() or (px[:, 1] > height).any():
            continue
        visible.append((float(cam[:, 2].mean()), TagPose(int(rec["id"]), px, family)))
    img = np.full((height, width), float(background), dtype=np.float64)
    visible.sort(key=lambda v: -v[0])
    for _, pose in visible:
        render_tag(img, pose, white, black, ss)
    if noise_sigma > 0:
        img = img + rng.normal(0.0, noise_sigma, size=img.shape)
    gray = np.clip(np.floor(img + 0.5), 0, 255).astype(np.uint8)
    return Scene(gray, [v[1] for v in visible])


# --- frame format packers -------------------------------------------------

def gray_to_yuyv(gray: np.ndarray) -> np.ndarray:
    """YUYV 4:2:2 with neutral chroma (chroma is discarded by the detector, threshold.cu:21)."""
    h, w = gray.shape
    out = np.full((h, w, 2), 128, dtype=np.uint8)
    out[:, :, 0] = gray
    return out.reshape(h, w * 2)


def gray_to_bgr(gray: np.ndarray, rng: np.random.Generator | None = None) -> np.ndarray:
    """A bgr8 frame; with `rng`, channels get independent +-6 offsets so the luma formula is exercised."""
    h, w = gray.shape
    out = np.repeat(gray[:, :, None], 3, axis=2).astype(np.int16)
    if rng is not None:
        out = out + rng.integers(-6, 7, size=out.shape, dtype=np.int16)
    return np.clip(out, 0, 255).astype(np.uint8)


def bgr_to_luma(bgr: np.ndarray) -> np.ndarray:
    """Y of cv::COLOR_BGR2YUV_YUYV (what the node feeds the detector, apriltags_cuda_detector.cu:401)."""
    b = bgr[:, :, 0].astype(np.int32)
    g = bgr[:, :, 1].astype(np.int32)
    r = bgr[:, :, 2].astype(np.int32)
    return ((4211 * r + 8258 * g + 1606 * b + (1 << 13) + (16 << 14)) >> 14).astype(np.uint8)


# --- BASELINE.json configs --------------------------------------------------

def config_frame(cfg: int, index: int = 0):
    """Returns (frame_bytes ndarray, fmt, width, height, decimate, sigma, Scene) for BASELINE config `cfg` (1..5)."""
    if cfg == 1:
        sc = make_scene(640, 480, 1 + index, 4, side_range=(90, 140), ids=[0, 1, 2, 3], max_rot_deg=30,
                        max_tilt_deg=35, noise_sigma=3.0)
        return sc.gray, "gray", 640, 480, 2, 0.0, sc
    if cfg == 2:
        rng = np.random.default_rng(2000 + index)
        nt = int(rng.integers(1, 7))
        sc = make_scene(1280, 800, 2000 + index, nt, side_range=(60, 300), noise_sigma=4.0)
        return gray_to_yuyv(sc.gray), "yuyv", 1280, 800, 2, 0.0, sc
    if cfg == 3:
        sc = make_scene(1920, 1080, 3 + index, 30, side_range=(20, 40), max_tilt_deg=45, noise_sigma=5.0)
        return gray_to_bgr(sc.gray), "bgr", 1920, 1080, 1, 0.8, sc
    if cfg == 4:
        rng = np.random.default_rng(4000 + index)
        nt = int(rng.integers(2, 9))
        sc = make_scene(1600, 1200, 4000 + index, nt, side_range=(60, 300), noise_sigma=4.0)
        return gray_to_yuyv(sc.gray), "yuyv", 1600, 1200, 2, 0.0, sc
    if cfg == 5:
        sc = make_scene(3840, 2160, 5000 + index, 100, side_range=(40, 200), noise_sigma=6.0, clutter=True,
                        salt_pepper=0.01)
        return gray_to_yuyv(sc.gray), "yuyv", 3840, 2160, 2, 0.0, sc
    raise ValueError(cfg)
