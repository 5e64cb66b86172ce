"""CPU: pin the oracle (oracle/jpeg_oracle.c) to the reference.

* against the reference's own golden vector (testimages/testimgint.jpg ==
  `cjpeg -revert -dct int testorig.ppm`, md5 in CMakeLists.txt:1391) and the
  md5s recorded from the unmodified reference by tools/make_golden.py;
* against what the reference's library, its forward DCT and its cjpeg binary
  made of seeded odd-shaped inputs and random switch sets, recorded by
  tools/make_golden.py --checks.
"""
import os

import numpy as np
import pytest

from common import case_id, case_image, golden_cases, md5

CASES = golden_cases()
SMALL = [c for c in CASES if c["image"] == "testorig" or c["image"][1] * c["image"][2] <= 200 * 136 or 65500 in c["image"][1:3]]


def test_reference_golden_md5_is_the_cmake_one():
    assert CASES[0]["switches"] == ["-revert", "-dct", "int"] and CASES[0]["image"] == "testorig"
    assert CASES[0]["md5"] == "9a68f56bc76e466aa7e52f415d0f4a5f"      # MD5_JPEG_420_ISLOW


@pytest.mark.parametrize("case", SMALL, ids=case_id)
def test_oracle_matches_recorded_reference(built, case):
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    img = case_image(case)
    nc = 1 if img.ndim == 2 else img.shape[2]
    p = mj.params_from_switches(case["switches"], img.shape[1], img.shape[0], nc)
    out = O.oracle_encode(p, img).jpeg
    assert len(out) == case["size"] and md5(out) == case["md5"]


@pytest.mark.parametrize("size", [(640, 480), (1920, 1080)], ids=lambda s: "%dx%d" % s)
def test_oracle_large_cases(built, size):
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    for c in CASES:
        if c["image"] != "testorig" and tuple(c["image"][1:]) == size and c["switches"][0] in ("-baseline", "-fastcrush") and "75" in c["switches"] and "2x2" in c["switches"]:
            img = case_image(c)
            p = mj.params_from_switches(c["switches"], img.shape[1], img.shape[0], 3)
            assert md5(O.oracle_encode(p, img).jpeg) == c["md5"]


def _fullsize_subset():
    """The full-size fixture's cases the restatement finishes in seconds (the 4K scan search takes it a minute)."""
    import json
    from common import GOLD
    path = os.path.join(GOLD, "fullsize_golden.json")
    cases = json.load(open(path))["cases"] if os.path.exists(path) else []
    keep = []
    for c in cases:
        sw = c["switches"]
        if c["image"][0] in (300, 17, 26) and sw[0] in ("-baseline", "-fastcrush", "-precision"):
            keep.append(c)
    return keep


@pytest.mark.parametrize("case", _fullsize_subset(), ids=case_id)
def test_oracle_full_size_recorded_reference(built, case):
    """BASELINE.json's configurations at their stated sizes (4K baseline + trellis, 4K progressive, 1080p q50/q90,
    12-bit 4:4:4 4K): the restatement reproduces the reference's md5."""
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    img = case_image(case)
    p = mj.params_from_switches(case["switches"], img.shape[1], img.shape[0], 3)
    out = O.oracle_encode(p, img).jpeg
    assert len(out) == case["size"] and md5(out) == case["md5"]


def test_oracle_live_vs_reference_random_shapes(built):
    """Odd shapes x profiles against the reference's bytes for them (tests/golden/random_shapes_golden.json)."""
    import json
    import mozjpeg_b200 as mj
    from common import GOLD
    from oracle import oracle as O
    cases = json.load(open(os.path.join(GOLD, "random_shapes_golden.json")))["cases"]
    assert len(cases) == 60
    for c in cases:
        w, h, sw = c["width"], c["height"], c["switches"]
        p = mj.params_from_switches(sw, w, h)
        out = O.oracle_encode(p, O.synth_image(c["seed"], w, h)).jpeg
        assert (len(out), md5(out)) == (c["size"], c["md5"]), (w, h, sw)


def test_stage_oracles_vs_reference_internals(built):
    """jpeg_fdct_islow of the reference library vs our restatement, on 200 random blocks (tests/golden/fdct_islow_golden.npz)."""
    import ctypes as C
    from common import GOLD
    from oracle import oracle as O
    g = np.load(os.path.join(GOLD, "fdct_islow_golden.npz"))
    assert g["input"].shape == (200, 64)
    for blk, want in zip(g["input"], g["output"]):
        a = blk.astype(np.int32)
        O.orc().orc_fdct_islow(a.ctypes.data_as(C.POINTER(C.c_int)))
        assert (a == want).all()


def test_random_switch_sets_live_against_reference_cjpeg(built):
    """tools/fuzz_vs_reference.py, a short run: random cjpeg switch sets (profiles, quality, sampling, restarts, DCT,
    smoothing, tuning presets, lambda, DC weight) on random small images - what the reference's cjpeg binary did with each
    (accepted or refused, and its bytes; tests/golden/fuzz_golden.json) vs mirror + oracle."""
    import subprocess
    import sys
    from common import GOLD, ROOT
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_vs_reference.py"), "2024", "60",
                        "--recorded", os.path.join(GOLD, "fuzz_golden.json")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-500:]
