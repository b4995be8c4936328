"""The decode stage's brute-force reference (tests/decode_reference.py) against the CPU oracle, and the scenes of
test_gpu_decode.py through the oracle against the reference and the rendered truth, so the GPU test's expectations
hold before it runs.  Also: the flipped-cell option of synth leaves every existing scene byte for byte as it was."""
import hashlib

import numpy as np
import pytest

import decode_reference as R
from ros_vision_b200 import synth
from ros_vision_b200.tag_families import FAMILIES


def test_rotate90_turns_the_cell_layout():
    """rotate90 moves every code bit to the cell a quarter turn away (the tag's bit layout turned by 90 degrees; for
    tag25h9 the centre cell stays) and four turns give the word back."""
    for name in R.FAMILY_NAMES:
        fam = FAMILIES[name]
        nb, wb = fam["nbits"], fam["width_at_border"]
        cell = {(fam["bit_x"][i], fam["bit_y"][i]): i for i in range(nb)}
        for i in range(nb):
            j = R.rotate90(1 << (nb - 1 - i), nb).bit_length() - 1
            x, y = fam["bit_x"][i], fam["bit_y"][i]
            assert cell[(y, wb - 1 - x)] == nb - 1 - j, (name, i)
        rng = np.random.default_rng(1)
        for w in rng.integers(0, 1 << nb, size=50):
            w = int(w)
            assert R.rotate90(R.rotate90(R.rotate90(R.rotate90(w, nb), nb), nb), nb) == w


def _words(name):
    """Every code with 0..4 flipped bits at each of the four rotations, random words, and the ambiguous tags."""
    fam = FAMILIES[name]
    nb = fam["nbits"]
    rng = np.random.default_rng(nb)
    words = []
    for i, c in enumerate(fam["codes"]):
        for b in rng.choice(nb, size=i % 5, replace=False):
            c ^= 1 << int(b)
        for _ in range(i % 4):
            c = R.rotate90(c, nb)
        words.append(c)
    words += [int(w) for w in rng.integers(0, 1 << nb, size=200)]
    for tid, flips in R.ambiguous_tags(name, 3, 6):
        words.append(R.tag_word(synth.TagPose(tid, np.zeros((4, 2)), name, flips)))
    return words


@pytest.mark.parametrize("name", R.FAMILY_NAMES)
def test_reference_matches_oracle_codeword(oracle, name):
    seen = {"rotations": set(), "ambiguous": 0, "none": 0, "hamming": set()}
    for mh in range(4):
        for w in _words(name):
            exp = R.decode(w, name, mh)
            assert oracle.decode_codeword(name, w, mh) == exp, (name, hex(w), mh)
            if exp is None:
                seen["none"] += 1
                continue
            seen["rotations"].add(exp[2])
            seen["hamming"].add(exp[1])
            seen["ambiguous"] += len(R.within_reach(w, name, mh)[1]) > 1
    assert seen["rotations"] == {0, 1, 2, 3} and seen["hamming"] == {0, 1, 2, 3} and seen["none"] > 0
    if name == "tag16h5":
        assert seen["ambiguous"] > 0  # minimum distance 5: at max_hamming 3 a word can be within reach of two codes


def test_ambiguous_words_resolve_to_the_lowest_id():
    for tid, flips in R.ambiguous_tags("tag16h5", 3, 6):
        w = R.tag_word(synth.TagPose(tid, np.zeros((4, 2)), "tag16h5", flips))
        r, hits = R.within_reach(w, "tag16h5", 3)
        assert r == 0 and len(hits) >= 2 and R.decode(w, "tag16h5", 3)[0] == min(hits)[0] < tid


CASES = R.cases()


@pytest.mark.parametrize("dec", [1, 2])
@pytest.mark.parametrize("name", list(CASES))
def test_scenes_through_oracle(oracle, name, dec):
    """Each GPU scene through the oracle: every tag's (id, hamming) and decode rotation as the reference predicts, no
    detection where it predicts none, corners in the truth's order; and the case the scene exists for occurs."""
    build, kind = CASES[name]
    scenes, families, tables, opts = build()
    cov, edge = R.Coverage(), (0, 0)
    for sc in scenes:
        orc = oracle.detect(oracle.make_config(R.W, R.H, "gray", dec, 0.0, families=families, **opts), sc.gray)
        if kind == "tags":
            R.check_tags(sc, orc.corners, orc.detections, tables, cov, rotation_of=lambda d: int(d["rotation"]))
        else:
            n, n0 = R.check_edge_tags(sc, orc.detections, 0)
            edge = (edge[0] + n, edge[1] + n0)
    R.check_coverage(name, cov, edge, dec)


# SHA-256 (first 16 hex digits) of scenes rendered before tags could carry flipped cells
SCENE_DIGESTS = {
    (1, 0): "912f83955f189518", (1, 1): "49781a768fcb8e41", (1, 2): "38ac0e6a0b4906b0", (1, 3): "729eafa722a2da6a",
    (2, 0): "49199793901e3833", (2, 1): "38667b1e1dacc7ec", (3, 0): "26ab8adb537bb6ab", (4, 0): "50f7534b41590ca0",
    (4, 1): "1871650ce213e36e", (5, 0): "13f15921ac1bf029",
    "tag36h11": "d019fe81e69b2247", "tag25h9": "2fabd601412a4ed4", "tag16h5": "4d5cd3fa815099fa",
}


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def test_scenes_without_flips_are_unchanged(golden_dir):
    import os
    from helpers import load_png_gray
    for key, want in SCENE_DIGESTS.items():
        if isinstance(key, tuple):
            got = _digest(synth.config_frame(*key)[0])
        else:
            got = _digest(synth.make_scene(640, 480, {"tag36h11": 501, "tag25h9": 502, "tag16h5": 77}[key], 3,
                                           side_range=(40, 130), noise_sigma=3.0, family=key, max_rot_deg=180).gray)
        assert got == want, key
    try:
        golden = load_png_gray(os.path.join(golden_dir, "synthetic_cfg1.png"))
    except ImportError:
        return
    assert np.array_equal(golden, synth.config_frame(1)[0])
