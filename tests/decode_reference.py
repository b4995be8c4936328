"""Brute-force reference for the decode stage, and the scenes its tests run.

The reference restates libapriltag's quick_decode_codeword from its definition, independently of the engine and of the
oracle: a word is tried at rotations 0..3 (rotate90 as libapriltag writes it); the first rotation that has any code
within max_hamming bits wins, and among the codes within reach there the lowest id (the entry libapriltag's hash table
holds first).  Which word the decoder reads depends on where the quad's corner 0 lies on the tag: `read_word` turns the
tag's word by the index of the truth corner nearest that corner, so a test predicts the answer for words that are
within reach of two codes too.

Scenes are placed by hand (synth.square_corners), not drawn by make_scene: every in-plane angle, tilts, flipped cells,
inverted frames and tags cut by the frame edge.  The CPU test runs them through the oracle and the GPU test through the
engine, from the same functions.
"""
from __future__ import annotations

import math

import numpy as np

from ros_vision_b200 import synth
from ros_vision_b200.tag_families import FAMILIES

FAMILY_NAMES = ("tag36h11", "tag25h9", "tag16h5")


def rotate90(w: int, nbits: int) -> int:
    """libapriltag apriltag.c rotate90: the word of the tag turned by 90 degrees; with nbits % 4 == 1 the last bit is
    the centre cell and stays put."""
    p, l = nbits, 0
    if nbits % 4 == 1:
        p, l = nbits - 1, 1
    w = ((w >> l) << (p // 4 + l)) | (w >> (3 * p // 4 + l) << l) | (w & l)
    return w & ((1 << nbits) - 1)


def family(name_or_table):
    return FAMILIES[name_or_table] if isinstance(name_or_table, str) else name_or_table


def within_reach(word: int, fam, max_hamming: int):
    """(rotation, [(id, hamming), ...]): the first rotation with codes within max_hamming bits and all of them, by id;
    (None, []) when no rotation has one."""
    fam = family(fam)
    for r in range(4):
        hits = [(i, bin(word ^ c).count("1")) for i, c in enumerate(fam["codes"])]
        hits = [(i, d) for i, d in hits if d <= max_hamming]
        if hits:
            return r, hits
        word = rotate90(word, fam["nbits"])
    return None, []


def decode(word: int, fam, max_hamming: int):
    """(id, hamming, rotation) of quick_decode_codeword, or None."""
    r, hits = within_reach(word, fam, max_hamming)
    if not hits:
        return None
    i, d = min(hits)
    return i, d, r


def tag_word(pose: synth.TagPose, fam=None) -> int:
    """The word the tag carries (its code with the flipped bits), read in the tag's own orientation."""
    fam = family(fam if fam is not None else pose.family)
    w = fam["codes"][pose.tag_id]
    for i in pose.flips:
        w ^= 1 << (fam["nbits"] - 1 - i)
    return w


def read_orientation(truth_corners, quad_corners) -> int:
    """k = index of the truth corner nearest the quad's corner 0."""
    d = np.linalg.norm(np.asarray(truth_corners, dtype=np.float64) - np.asarray(quad_corners, dtype=np.float64)[0], axis=1)
    return int(np.argmin(d))


def read_word(pose: synth.TagPose, quad_corners, fam=None) -> int:
    """The word the decoder starts from: rotate90^k of the tag's word."""
    fam = family(fam if fam is not None else pose.family)
    w = tag_word(pose, fam)
    for _ in range(read_orientation(pose.corners, quad_corners)):
        w = rotate90(w, fam["nbits"])
    return w


def truth_centre(corners) -> np.ndarray:
    """Intersection of the diagonals of the truth quad (the image of the tag centre under the tag's homography)."""
    (x0, y0), (x1, y1), (x2, y2), (x3, y3) = np.asarray(corners, dtype=np.float64)
    d1x, d1y, d2x, d2y = x2 - x0, y2 - y0, x3 - x1, y3 - y1
    t = ((x1 - x0) * d2y - (y1 - y0) * d2x) / (d1x * d2y - d1y * d2x)
    return np.array([x0 + t * d1x, y0 + t * d1y])


def quad_of(pose: synth.TagPose, quads, tol=3.0):
    """The candidate quad (row of the oracle's `corners` or the engine's FitQuads) whose corners are the tag's own, in
    any order: its outline, not an inner quad of the tag's cells.  None when no quad is."""
    from helpers import match_corner_sets
    best = [q for q in quads if match_corner_sets(q["corners"], pose.corners) <= tol]
    return best[0] if best else None


def detections_at(pose: synth.TagPose, dets, tol=2.0):
    """Detections whose centre lies within `tol` px of the tag's truth centre and whose corners are the tag's own."""
    from helpers import match_corner_sets
    c = truth_centre(pose.corners)
    return [d for d in dets if np.abs(np.asarray(d["c"]) - c).max() <= tol and match_corner_sets(d["p"], pose.corners) <= 3.0]


def complemented(name: str, max_hamming: int = 2):
    """The built-in family with every code complemented and a reversed border: what a white-bordered print of the
    family's tags reads as (the tags of `255 - frame`)."""
    fam = FAMILIES[name]
    mask = (1 << fam["nbits"]) - 1
    return dict(fam, codes=[c ^ mask for c in fam["codes"]], reversed_border=1, max_hamming=max_hamming,
                name=f"{name}-reversed")


# --- scenes -------------------------------------------------------------------------------------------------------

W, H = 640, 480


def compose(poses, seed: int, noise_sigma: float = 2.0, invert: bool = False) -> synth.Scene:
    """Gray frame of the tags `poses` on a 128 background with Gaussian noise; `invert` gives 255 - frame."""
    img = np.full((H, W), 128.0, dtype=np.float64)
    for p in poses:
        synth.render_tag(img, p, 230.0, 25.0, 4)
    img = img + np.random.default_rng(seed).normal(0.0, noise_sigma, size=img.shape)
    gray = np.clip(np.floor(img + 0.5), 0, 255).astype(np.uint8)
    return synth.Scene(255 - gray if invert else gray, list(poses))


def pose(tag_id, fam, cx, cy, side, rot_deg, tilt_deg=0.0, axis_deg=0.0, flips=()):
    return synth.TagPose(tag_id, synth.square_corners(cx, cy, side, math.radians(rot_deg), math.radians(tilt_deg),
                                                      math.radians(axis_deg)), fam, tuple(flips))


GRID = [(110.0 + 210.0 * i, 120.0 + 240.0 * j) for j in range(2) for i in range(3)]  # six tags of ~100 px per frame


def orientation_frames(fam: str, n_frames: int = 5):
    """Six tags per frame, in-plane angles stepping 360 / 30 degrees over the frames (every tag a different angle,
    offset from the multiples of 45), tilts up to 30 degrees about varying axes, no bit errors."""
    ncodes = len(FAMILIES[fam]["codes"])
    scenes = []
    for f in range(n_frames):
        poses = []
        for t, (cx, cy) in enumerate(GRID):
            k = f * len(GRID) + t
            poses.append(pose((7 * k + 3) % ncodes, fam, cx, cy, 96.0 + 4 * (k % 3), 7.0 + 12.0 * k,
                              tilt_deg=(0.0, 15.0, 30.0)[k % 3], axis_deg=53.0 * k))
        scenes.append(compose(poses, seed=100 + f))
    return scenes


def ambiguous_tags(fam: str, max_hamming: int, limit: int):
    """(tag id, flips) whose word, read in the tag's orientation, is within max_hamming bits of two codes: the tag's
    own code with bits flipped towards a lower id's.  Found by brute force, lowest ids first."""
    fm = FAMILIES[fam]
    nb, codes = fm["nbits"], fm["codes"]
    out = []
    for b in range(len(codes)):
        for a in range(b):
            diff = [i for i in range(nb) if ((codes[a] ^ codes[b]) >> (nb - 1 - i)) & 1]
            if len(diff) > 2 * max_hamming:
                continue
            flips = tuple(diff[:max_hamming])
            w = codes[b]
            for i in flips:
                w ^= 1 << (nb - 1 - i)
            r, hits = within_reach(w, fm, max_hamming)
            if r == 0 and len(hits) >= 2:
                out.append((b, flips))
                break
        if len(out) >= limit:
            break
    return out


def bit_error_frames(fam: str, n_frames: int = 5):
    """Six tags per frame with 0..4 flipped cells (positions from a seeded generator), at every quarter turn plus an
    offset; for tag16h5 the last frame carries tags flipped towards a lower id (ambiguous at max_hamming 3)."""
    fm = FAMILIES[fam]
    ncodes, nb = len(fm["codes"]), fm["nbits"]
    rng = np.random.default_rng({"tag36h11": 11, "tag25h9": 12, "tag16h5": 13}[fam])
    specials = ambiguous_tags(fam, 3, len(GRID)) if fam == "tag16h5" else []
    scenes = []
    for f in range(n_frames):
        poses = []
        for t, (cx, cy) in enumerate(GRID):
            k = f * len(GRID) + t
            if f == n_frames - 1 and t < len(specials):
                tid, flips = specials[t]
            else:
                tid = int(rng.integers(0, ncodes))
                flips = tuple(int(i) for i in rng.choice(nb, size=k % 5, replace=False))
            poses.append(pose(tid, fam, cx, cy, 100.0, 90.0 * (k % 4) + 5.0 + 3.0 * k, tilt_deg=12.0 * (k % 2),
                              axis_deg=71.0 * k, flips=flips))
        scenes.append(compose(poses, seed=200 + f))
    return scenes


def mixed_family_frames(n_frames: int = 5):
    """tag36h11 and tag25h9 tags side by side, 0..4 flipped cells, several orientations."""
    rng = np.random.default_rng(21)
    scenes = []
    for f in range(n_frames):
        poses = []
        for t, (cx, cy) in enumerate(GRID):
            k = f * len(GRID) + t
            fam = ("tag36h11", "tag25h9")[k % 2]
            fm = FAMILIES[fam]
            flips = tuple(int(i) for i in rng.choice(fm["nbits"], size=(k // 2) % 5, replace=False))
            poses.append(pose(int(rng.integers(0, len(fm["codes"]))), fam, cx, cy, 100.0, 37.0 * k, tilt_deg=10.0,
                              axis_deg=29.0 * k, flips=flips))
        scenes.append(compose(poses, seed=300 + f))
    return scenes


def edge_frames(fam: str, cut: float = 3.0):
    """Tags of side 100 px whose quiet zone and `cut` px of the black border lie outside the frame: two per edge, at
    several rotations, some with flipped cells.  One frame per pair of edges (left/right, top/bottom)."""
    fm = FAMILIES[fam]
    ncodes, nb = len(fm["codes"]), fm["nbits"]
    rng = np.random.default_rng(31)
    side = 100.0
    half = side / 2 - cut
    scenes = []
    for axis in (0, 1):
        poses = []
        for j, rot in enumerate((0.0, 90.0, 180.0, 270.0)):
            along = (160.0, 480.0)[j % 2] if axis == 1 else (140.0, 340.0)[j % 2]
            lo = j < 2
            if axis == 0:   # left / right edges
                cx, cy = (half if lo else W - half), along
            else:           # top / bottom edges
                cx, cy = along, (half if lo else H - half)
            flips = tuple(int(i) for i in rng.choice(nb, size=j % 3, replace=False))
            poses.append(pose(int(rng.integers(0, ncodes)), fam, cx, cy, side, rot, flips=flips))
        scenes.append(compose(poses, seed=400 + axis))
    return scenes


# --- truth checks shared by the CPU (oracle) and GPU (engine) tests ------------------------------------------------

CORNER_TOL_PX = 1.0   # p[i] and c against the rendered truth: the CPU rehearsal stays below 0.4 px


class Coverage:
    """What the checked frames exercised (the tests assert that each case really occurred)."""

    def __init__(self):
        self.rotations = {}     # family name -> set of decode rotations of matched tags
        self.corrected = set()  # hamming values of tags decoded to their own id with flipped cells
        self.dropped = 0        # tags with flipped cells beyond reach: no detection
        self.ambiguous = 0      # tags whose read word was within reach of two codes, decoded to the lower id
        self.decoded = 0


def check_tags(scene, quads, dets, tables, cov: Coverage, rotation_of=None):
    """Every tag of `scene` against the brute-force reference and the truth.  `tables`: family name -> (index of the
    family in the detector's list, its table with max_hamming).  `quads`: candidate quads (the tag's read orientation
    comes from the one outlining it), `dets`: the frame's detections.  `rotation_of(det)` gives a detection's decode
    rotation when the detector reports it (the oracle does)."""
    for p in scene.tags:
        index, table = tables[p.family]
        q = quad_of(p, quads)
        assert q is not None, f"no candidate quad outlines tag {p.tag_id} ({p.family}) at {truth_centre(p.corners)}"
        word = read_word(p, q["corners"], table)
        mh = int(table.get("max_hamming", 2))
        exp = decode(word, table, mh)
        at = [d for d in detections_at(p, dets) if int(d["family"]) == index]
        where = f"tag {p.tag_id} ({p.family}, flips {p.flips}, max_hamming {mh}) at {truth_centre(p.corners)}"
        if exp is None:
            assert at == [], f"{where}: beyond reach but detected as {[(int(d['id']), int(d['hamming'])) for d in at]}"
            cov.dropped += bool(p.flips)
            continue
        assert len(at) == 1, f"{where}: expected {exp[:2]}, got {[(int(d['id']), int(d['hamming'])) for d in at]}"
        d = at[0]
        assert (int(d["id"]), int(d["hamming"])) == exp[:2], f"{where}: got {(int(d['id']), int(d['hamming']))}, reference {exp[:2]}"
        cov.decoded += 1
        if rotation_of is not None:
            assert rotation_of(d) == exp[2], f"{where}: rotation {rotation_of(d)}, reference {exp[2]}"
            cov.rotations.setdefault(p.family, set()).add(exp[2])
        hits = within_reach(word, table, mh)[1]
        if len(hits) > 1:
            assert exp[0] == min(hits)[0]
            cov.ambiguous += 1
        if exp[0] == p.tag_id:
            # the tag itself: corner i of the detection is truth corner 3 - i, in that order
            if p.flips:
                cov.corrected.add(exp[1])
            for i in range(4):
                assert np.abs(np.asarray(d["p"][i]) - p.corners[3 - i]).max() <= CORNER_TOL_PX, f"{where}: p[{i}] vs truth corner {3 - i}"
            assert np.abs(np.asarray(d["c"]) - truth_centre(p.corners)).max() <= CORNER_TOL_PX, f"{where}: centre"


EDGE_MATCH_PX = 10.0  # a border cut by the frame edge moves the fitted quad (and its centre) by several pixels


def check_edge_tags(scene, dets, index):
    """Detections of tags cut by the frame edge: those of hamming 0 carry the tag's id and its corner order (p[i]
    nearest truth corner 3 - i).  Returns (detections of the tags, those of hamming 0)."""
    n = n0 = 0
    for d in dets:
        near = [p for p in scene.tags if np.abs(np.asarray(d["c"]) - truth_centre(p.corners)).max() <= EDGE_MATCH_PX]
        if int(d["family"]) != index or not near:
            continue
        n += 1
        if int(d["hamming"]) != 0:
            continue
        p = near[0]
        assert int(d["id"]) == p.tag_id, (int(d["id"]), p.tag_id)
        for i in range(4):
            assert int(np.argmin(np.linalg.norm(p.corners - np.asarray(d["p"][i]), axis=1))) == 3 - i, f"tag {p.tag_id}: p[{i}]"
        n0 += 1
    return n, n0


def check_coverage(name, cov: Coverage, edge=None, dec=None):
    """The cases each scene set exists for really occurred (counts from the oracle run on CPU)."""
    fam = name.rsplit("-", 1)[-1] if not name.startswith("mixed") else None
    if name.startswith("edge-"):
        n, n0 = edge
        assert n >= 1 or dec == 2, f"{name}: no tag cut by the frame edge decoded at quad_decimate 1"
        return
    if not name.startswith("bits-") and not name.startswith("mixed"):
        for f, rots in cov.rotations.items():
            assert rots == {0, 1, 2, 3}, f"{name}: decode rotations {sorted(rots)}"
    if name.startswith("orientation-") or name.startswith("reversed-tag"):
        assert cov.decoded == 30 and cov.rotations[fam] == {0, 1, 2, 3}
    if name.startswith("bits-"):
        mh = int(name.split("-h")[-1][0]) if "-h" in name else None
        assert cov.corrected == set(range(1, mh + 1)), f"{name}: corrected {sorted(cov.corrected)}"
        assert cov.dropped >= 1, f"{name}: no tag beyond reach"
        if name == "bits-tag16h5-h3":
            assert cov.ambiguous >= 1, f"{name}: no word within reach of two codes"
    if name.startswith("reversed-bits-"):
        assert cov.corrected == {1, 2, 3} and cov.dropped >= 1
    if name.startswith("mixed"):
        # tag36h11 corrects 1 bit only, tag25h9 3: both limits reach the decode
        assert 3 in cov.corrected and cov.dropped >= 1, vars(cov)


# --- the cases: scenes, the detector's families, and options --------------------------------------------------------

def _with(name, **kw):
    return dict(FAMILIES[name], name=name, **kw)


def cases():
    """name -> (build, kind): build() returns (scenes, families as the detector takes them, tables for check_tags,
    detector options).  kind "tags": check_tags on every tag; "edge": check_edge_tags."""
    out = {}
    for fam in FAMILY_NAMES:
        # families are given as tables throughout, so that engine and oracle number them alike (by the caller's list)
        out[f"orientation-{fam}"] = (lambda fam=fam: (orientation_frames(fam), [_with(fam)], {fam: (0, _with(fam))}, {}), "tags")
        for mh in range(4):
            out[f"bits-{fam}-h{mh}"] = (lambda fam=fam, mh=mh: (
                bit_error_frames(fam), [_with(fam, max_hamming=mh)], {fam: (0, _with(fam, max_hamming=mh))}, {}), "tags")
        # white-bordered tags: the frame inverted, decoded by the family's complemented codes with a reversed border
        out[f"reversed-{fam}"] = (lambda fam=fam: (
            [compose(s.tags, seed=100 + i, invert=True) for i, s in enumerate(orientation_frames(fam))],
            [complemented(fam)], {fam: (0, complemented(fam))}, {}), "tags")
        out[f"reversed-bits-{fam}"] = (lambda fam=fam: (
            [compose(s.tags, seed=200 + i, invert=True) for i, s in enumerate(bit_error_frames(fam))],
            [complemented(fam, 3)], {fam: (0, complemented(fam, 3))}, {}), "tags")
        out[f"edge-{fam}"] = (lambda fam=fam: (edge_frames(fam), [_with(fam)], None, {}), "edge")
        for opt in ({"decode_sharpening": 0.0}, {"decode_sharpening": 1.0}, {"refine_edges": False}):
            key = "-".join(f"{k}{v}" for k, v in opt.items())
            out[f"{key}-{fam}"] = (lambda fam=fam, opt=opt: (
                bit_error_frames(fam), [_with(fam, max_hamming=3)], {fam: (0, _with(fam, max_hamming=3))}, dict(opt)), "tags")
    mixed = [_with("tag36h11", max_hamming=1), _with("tag25h9", max_hamming=3)]
    out["mixed-36h11h1-25h9h3"] = (lambda: (mixed_family_frames(), mixed, {"tag36h11": (0, mixed[0]), "tag25h9": (1, mixed[1])}, {}), "tags")
    return out
