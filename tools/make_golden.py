#!/usr/bin/env python3
"""Generate tests/golden/golden.json from the UNMODIFIED reference.

Runs only where /root/reference exists (oracle/_ref built by oracle/Makefile).
For every case it records the md5 and size of what the reference encoder
produces; the tests then hold the CPU oracle and the CUDA path to those
numbers on machines where the reference is absent.

Inputs are either the reference's own test image (testimages/testorig.ppm,
copied to tests/golden/ as a data fixture) or synthetic images generated from
a seed by oracle.synth_image (SURVEY 8d).
"""
import hashlib, json, os, shutil, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
from oracle import oracle as O
import mozjpeg_b200 as cjpeg

REF = "/root/reference"
GOLD = os.path.join(ROOT, "tests", "golden")

SWITCH_SETS = [
    ["-revert", "-dct", "int"],                       # == testimages/testimgint.jpg, CMakeLists.txt:1391 (config 1)
    ["-revert", "-optimize"],
    ["-revert", "-progressive"],
    ["-revert", "-quality", "90", "-sample", "2x2"],
    ["-revert", "-sample", "1x1"],                    # ~ 444-islow family
    ["-revert", "-sample", "2x1", "-optimize"],       # ~ 422-*-opt family
    ["-revert", "-sample", "1x2"],                    # ~ 440-islow
    ["-revert", "-grayscale"],                        # ~ gray-islow
    ["-revert", "-grayscale", "-progressive"],
    ["-baseline", "-quality", "75"],                  # config 2 semantics (4:2:0 is the default)
    ["-baseline", "-quality", "75", "-sample", "2x2"],
    ["-baseline", "-quality", "50", "-sample", "2x2"],
    ["-baseline", "-quality", "90", "-sample", "2x2"],
    ["-baseline", "-quality", "75", "-sample", "1x1"],
    ["-baseline", "-quality", "85"],
    ["-baseline", "-quality", "95"],
    ["-baseline", "-quality", "100"],
    ["-baseline", "-quality", "20"],
    ["-baseline", "-notrellis", "-quality", "75"],
    ["-baseline", "-notrellis-dc", "-quality", "75"],
    ["-baseline", "-noovershoot", "-quality", "75"],
    ["-baseline", "-grayscale", "-quality", "75"],
    ["-baseline", "-quant-table", "2", "-quality", "80"],
    ["-baseline", "-lambda1", "12.0", "-lambda2", "13.0", "-quality", "75"],
    ["-fastcrush", "-quality", "75"],                 # config 3 semantics
    ["-fastcrush", "-quality", "75", "-sample", "2x2"],
    ["-fastcrush", "-quality", "50", "-sample", "2x2"],
    ["-fastcrush", "-quality", "90", "-sample", "2x2"],
    ["-fastcrush", "-quality", "92"],
    ["-fastcrush", "-grayscale", "-quality", "75"],
    ["-fastcrush", "-notrellis", "-quality", "75"],
    ["-baseline", "-quality", "75", "-restart", "1"],
    ["-fastcrush", "-quality", "75", "-restart", "2"],
    ["-revert", "-restart", "3B"],
    # the library default: 64-scan (23 for gray) search, jcparam.c:733-852 + jcmaster.c:773-962
    ["-quality", "75"],
    ["-quality", "90"],
    ["-quality", "50", "-sample", "2x2"],
    ["-grayscale", "-quality", "75"],
    ["-quality", "75", "-restart", "1"],
    ["-quality", "85", "-notrellis"],
    # JDCT_FLOAT (jfdctflt.c; this reference build is the "no-fp-contract" flavour of CMakeLists.txt:965-1024)
    ["-dct", "float", "-baseline", "-quality", "75"],
    ["-dct", "float", "-quality", "75", "-fastcrush"],
    ["-dct", "float", "-baseline", "-notrellis", "-quality", "90", "-sample", "1x1"],
    ["-dct", "float", "-baseline", "-quality", "50", "-grayscale"],
    ["-dct", "float", "-quality", "75"],
    # JDCT_IFAST (jfdctfst.c, scaled divisors + reciprocal quantizer)
    ["-dct", "fast", "-baseline", "-quality", "75"],
    ["-dct", "fast", "-fastcrush", "-quality", "40"],
    ["-dct", "fast", "-baseline", "-notrellis", "-quality", "95", "-sample", "1x1"],
    ["-dct", "fast", "-baseline", "-quality", "100", "-grayscale"],
    ["-dct", "fast", "-quality", "75"],
]
# input smoothing (jcsample.c:298-455, context-row mode of jcprepct.c) and sampling layouts that go through
# int_downsample (jcsample.c:151-190); the refshim driver hands these to the reference's cjpeg binary
SWITCH_SETS_EXTRA = [
    ["-revert", "-smooth", "10"],
    ["-baseline", "-quality", "75", "-smooth", "30"],
    ["-quality", "75", "-smooth", "100", "-sample", "1x1"],
    ["-baseline", "-quality", "80", "-smooth", "50", "-sample", "2x1"],
    ["-revert", "-smooth", "20", "-sample", "3x2"],
    ["-baseline", "-grayscale", "-smooth", "15", "-quality", "60"],
    ["-fastcrush", "-smooth", "5", "-sample", "2x2,1x1,2x2"],
    ["-dct", "float", "-baseline", "-quality", "75", "-smooth", "40"],
    # vertical-gradient weight in the DC trellis (jcdctmgr.c:1069-1086): acts on components with v_samp_factor > 1
    ["-baseline", "-quality", "75", "-trellis-dc-ver-weight", "1.0"],
    ["-quality", "85", "-trellis-dc-ver-weight", "0.5", "-sample", "2x2"],
    ["-fastcrush", "-quality", "60", "-trellis-dc-ver-weight", "2.5", "-sample", "1x2"],
    # cjpeg's tuning presets (cjpeg.c:678-704): base table index + lambda scales; -tune-psnr has lambda_log_scale2 = 0,
    # i.e. the constant-lambda branch of quantize_trellis (jcdctmgr.c:1031-1035)
    ["-tune-psnr"], ["-tune-ssim"], ["-tune-ms-ssim"], ["-tune-hvs-psnr"],
    ["-tune-psnr", "-quality", "85", "-baseline"],
    ["-baseline", "-lambda1", "10.5", "-lambda2", "0", "-quality", "70"],
    ["-revert", "-sample", "3x2"],
    ["-baseline", "-quality", "75", "-sample", "4x2"],
    ["-quality", "75", "-sample", "3x1"],
    ["-baseline", "-quality", "80", "-sample", "2x2,1x1,2x2"],
    ["-baseline", "-sample", "4x1,1x1,2x1", "-quality", "60"],
    # fast / float DCT on sampling layouts outside the tiled kernel's (the one-thread-per-block forward kernel)
    ["-baseline", "-quality", "75", "-sample", "3x1", "-dct", "fast"],
    ["-quality", "80", "-sample", "4x2", "-dct", "float"],
    ["-fastcrush", "-quality", "75", "-sample", "2x2,1x1,2x2", "-dct", "fast"],
    ["-baseline", "-quality", "75", "-sample", "3x2", "-dct", "float", "-smooth", "20"],
    ["-baseline", "-quality", "75", "-rgb", "-dct", "float"],
]
# switches that name files (rdswitch.c read_quant_tables / set_quant_slots / read_scan_script); "@GOLD/" = tests/golden/
SWITCH_SETS_FILES = [
    ["-qtables", "@GOLD/qtables_a.txt", "-quality", "75"],
    ["-qtables", "@GOLD/qtables_a.txt", "-baseline"],
    ["-quality", "60,90", "-qtables", "@GOLD/qtables_a.txt", "-qslots", "1,0,0"],
    ["-quality", "70,80", "-qslots", "1,0,1"],
    ["-scans", "@GOLD/scans_a.txt", "-quality", "75"],                       # successive approximation, band splits
    ["-scans", "@GOLD/scans_b.txt", "-quality", "80"],                       # sequential, two scans
    ["-scans", "@GOLD/scans_c.txt"],
    ["-revert", "-scans", "@GOLD/scans_a.txt"],
    ["-revert", "-scans", "@GOLD/scans_b.txt", "-optimize"],
    ["-scans", "@GOLD/scans_c.txt", "-restart", "1", "-sample", "2x1"],
]
# through the reference's cjpeg binary only (our refshim driver does not parse these switches)
CJPEG_ONLY = [
    ["-revert", "-dct", "float"],
    ["-revert", "-dct", "float", "-optimize", "-progressive"],
    ["-revert", "-dct", "fast"],
    ["-quality", "75", "-dc-scan-opt", "2"],
    ["-quality", "60", "-dc-scan-opt", "1"],
    ["-quality", "85", "-dc-scan-opt", "0"],
]
# 12-bit precision (config 5 semantics and relatives): the reference can only run these with the trellis and the
# deringing off (SURVEY F5); optimal Huffman tables are forced (jcmaster.c:1102-1105)
SWITCH_SETS_12 = [
    ["-precision", "12", "-sample", "1x1", "-quality", "75", "-notrellis", "-noovershoot", "-baseline"],      # config 5
    ["-precision", "12", "-quality", "75", "-notrellis", "-noovershoot", "-baseline"],                           # 4:2:0
    ["-precision", "12", "-quality", "90", "-notrellis", "-noovershoot", "-baseline", "-grayscale"],
    ["-precision", "12", "-quality", "60", "-notrellis", "-noovershoot", "-fastcrush", "-sample", "2x1"],
    ["-precision", "12", "-quality", "75", "-notrellis", "-noovershoot", "-fastcrush", "-restart", "1"],
    ["-precision", "12", "-quality", "100", "-notrellis", "-noovershoot", "-baseline", "-sample", "1x2"],
    # 12-bit on sampling layouts outside the tiled kernel's
    ["-precision", "12", "-quality", "75", "-notrellis", "-noovershoot", "-baseline", "-sample", "3x2"],
    ["-precision", "12", "-quality", "80", "-notrellis", "-noovershoot", "-fastcrush", "-sample", "4x1,1x1,2x1"],
    # 12-bit with the fast / float DCT (scaled divisors divided literally, jcdctmgr.c:332-336,646-678)
    ["-precision", "12", "-quality", "75", "-notrellis", "-noovershoot", "-baseline", "-dct", "fast"],
    ["-precision", "12", "-quality", "90", "-notrellis", "-noovershoot", "-baseline", "-dct", "float", "-sample", "2x1"],
    ["-precision", "12", "-quality", "60", "-notrellis", "-noovershoot", "-fastcrush", "-dct", "fast", "-sample", "3x2"],
]
SYNTH12 = [(21, 16, 16), (22, 33, 17), (23, 200, 136), (24, 640, 480), (25, 1, 1)]
SYNTH = [(11, 16, 16), (12, 33, 17), (13, 200, 136), (14, 640, 480), (15, 1, 1), (16, 8, 8), (17, 1920, 1080)]


def _key(image, sw):
    return json.dumps([image, sw])


# BASELINE.json's configurations at their stated sizes (a separate fixture: each case costs the reference seconds to a
# minute).  Images [seed, w, h] or [seed, w, h, 12]; seeds 1000.. are bench.py's first-rank inputs.
FULLSIZE = [
    ([300, 3840, 2160], ["-baseline", "-quality", "75", "-sample", "2x2"]),          # configs[1]
    ([1000, 3840, 2160], ["-baseline", "-quality", "75", "-sample", "2x2"]),
    ([300, 3840, 2160], ["-fastcrush", "-quality", "75", "-sample", "2x2"]),         # configs[2]
    ([1000, 3840, 2160], ["-fastcrush", "-quality", "75", "-sample", "2x2"]),
    ([17, 1920, 1080], ["-baseline", "-quality", "50", "-sample", "2x2"]),           # configs[3] sweep (q75 is in golden.json)
    ([17, 1920, 1080], ["-baseline", "-quality", "90", "-sample", "2x2"]),
    ([1001, 1920, 1080], ["-baseline", "-quality", "50", "-sample", "2x2"]),
    ([1001, 1920, 1080], ["-baseline", "-quality", "75", "-sample", "2x2"]),
    ([1001, 1920, 1080], ["-baseline", "-quality", "90", "-sample", "2x2"]),
    ([26, 3840, 2160, 12], ["-precision", "12", "-sample", "1x1", "-quality", "75", "-notrellis", "-noovershoot", "-baseline"]),   # configs[4]
    ([1000, 3840, 2160, 12], ["-precision", "12", "-sample", "1x1", "-quality", "75", "-notrellis", "-noovershoot", "-baseline"]),
    ([300, 3840, 2160], ["-quality", "75", "-sample", "2x2"]),                       # the library default (scan search) at 4K
    ([301, 3840, 2160], ["-baseline", "-quality", "75", "-sample", "2x2"]),          # second image of test_full_size_4k_frame
]


def reference_checks():
    """--checks: fixtures of the checks against the reference's library and binaries: odd shapes x profiles, the forward DCT on
    random blocks, the quantization tables of the reference's DQT, a recorded run of tools/fuzz_vs_reference.py, and
    the coefficient-domain re-encode of odd source files (the sources, their coefficients and jpegtran's md5s)."""
    import subprocess
    import ctypes as C
    from mozjpeg_b200.synth import synth_image12
    # test_oracle_pinning: odd shapes x profiles
    rng = np.random.default_rng(7)
    sws = [["-baseline", "-quality", "70"], ["-fastcrush", "-quality", "80"], ["-revert", "-optimize"],
           ["-baseline", "-quality", "75", "-sample", "2x1"], ["-baseline", "-quality", "75", "-sample", "1x2"]]
    shapes = []
    for _ in range(12):
        w, h = int(rng.integers(1, 97)), int(rng.integers(1, 97))
        seed = int(rng.integers(0, 1 << 30))
        im = O.synth_image(seed, w, h)
        for sw in sws:
            a = O.ref_encode(im, sw)
            shapes.append({"seed": seed, "width": w, "height": h, "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    json.dump({"generator": "tools/make_golden.py --checks", "cases": shapes}, open(os.path.join(GOLD, "random_shapes_golden.json"), "w"), indent=0)
    # test_oracle_pinning: jpeg_fdct_islow of the reference library on random blocks
    rng = np.random.default_rng(3)
    blocks = rng.integers(-128, 160, (200, 64)).astype(np.int32)
    out = blocks.copy()
    for b in out:
        O.ref().refshim_fdct_islow(b.ctypes.data_as(C.POINTER(C.c_int)))
    np.savez_compressed(os.path.join(GOLD, "fdct_islow_golden.npz"), input=blocks, output=out)
    # test_abi_host: the quantization tables the reference writes into its DQT
    img = O.synth_image(1, 32, 32)
    dqt = []
    for sw in (["-revert"], ["-baseline", "-quality", "75"], ["-baseline", "-quality", "33"], ["-baseline", "-quality", "97"],
               ["-baseline", "-quant-table", "5", "-quality", "60"], ["-revert", "-quality", "5"]):
        dqt.append({"switches": sw, "qt": O.ref_read_coefs(O.ref_encode(img, sw))["qt"].tolist()})
    json.dump({"generator": "tools/make_golden.py --checks", "cases": dqt}, open(os.path.join(GOLD, "dqt_golden.json"), "w"), indent=0)
    # test_oracle_pinning: random cjpeg switch sets through the reference's cjpeg binary
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tools", "fuzz_vs_reference.py"), "2024", "60",
                           "--record", os.path.join(GOLD, "fuzz_golden.json")])
    # test_transcode: source files the encode fixture does not have (16-bit quantization tables, RGB colourspace,
    # restart markers, gray with 2x2 sampling, 12-bit), their coefficients as the reference's decoder reads them, and
    # what the reference's jpegtran makes of them
    im = O.synth_image(3, 120, 72)
    srcs = []
    for esw in (["-revert", "-quality", "3"], ["-quality", "12", "-sample", "2x2"], ["-revert", "-rgb"], ["-revert", "-progressive", "-restart", "1"],
                ["-revert", "-quality", "50", "-sample", "2x2", "-grayscale"]):      # a gray file with 2x2 sampling leaves jpegtran as 1x1
        try:
            srcs.append(O.ref_encode(im, esw))
        except ValueError:
            srcs.append(O._ref_cjpeg_pixels(im, esw))
    srcs.append(O.ref_encode(synth_image12(4, 120, 72), ["-precision", "12", "-quality", "75", "-notrellis", "-noovershoot", "-baseline"]))
    trans = ([], ["-revert"], ["-progressive"], ["-revert", "-optimize"])
    arrays = {}
    md5s, sizes = [], []
    for k, src in enumerate(srcs):
        arrays["src%d" % k] = np.frombuffer(src, dtype=np.uint8)
        for ci, plane in enumerate(O.ref_read_coefs(src)["coefs"]):
            arrays["coef%d_%d" % (k, ci)] = plane
        outs = [O.ref_jpegtran(src, tsw) for tsw in trans]
        md5s.append([hashlib.md5(a).hexdigest() for a in outs]); sizes.append([len(a) for a in outs])
    np.savez_compressed(os.path.join(GOLD, "transcode_odd_golden.npz"), tran=np.array([" ".join(t) for t in trans]),
                        md5=np.array(md5s), size=np.array(sizes), **arrays)
    print("wrote the reference-check fixtures")


def fullsize():
    from mozjpeg_b200.synth import synth_image12
    path = os.path.join(GOLD, "fullsize_golden.json")
    have = {}
    if "--force" not in sys.argv and os.path.exists(path):
        for c in json.load(open(path))["cases"]:
            have[_key(c["image"], c["switches"])] = c
    cases = []
    for image, sw in FULLSIZE:
        if _key(image, sw) in have:
            cases.append(have[_key(image, sw)]); continue
        im = synth_image12(*image[:3]) if len(image) > 3 else O.synth_image(*image)
        a = O.ref_encode(im, sw)
        cases.append({"image": image, "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
        print(image, sw, len(a), flush=True)
    json.dump({"generator": "tools/make_golden.py --fullsize", "reference": "mozilla/mozjpeg 5.0.0 (C path, WITH_SIMD=0), oracle/_ref", "cases": cases},
              open(path, "w"), indent=0)
    print("wrote", len(cases), "full-size cases")


def main():
    if "--fullsize" in sys.argv:
        return fullsize()
    if "--checks" in sys.argv:
        return reference_checks()
    os.makedirs(GOLD, exist_ok=True)
    # cases already recorded are kept as they are unless --force is given (a full regeneration takes a while)
    have = {}
    if "--force" not in sys.argv and os.path.exists(os.path.join(GOLD, "golden.json")):
        for c in json.load(open(os.path.join(GOLD, "golden.json")))["cases"]:
            have[_key(c["image"], c["switches"])] = c
    shutil.copyfile(os.path.join(REF, "testimages", "testorig.ppm"), os.path.join(GOLD, "testorig.ppm"))
    cases = []
    ppm = os.path.join(GOLD, "testorig.ppm")
    w, h, nc, data = cjpeg.read_ppm(open(ppm, "rb").read())
    img = np.frombuffer(data, dtype=np.uint8).reshape(h, w, nc)
    for sw in SWITCH_SETS:
        if _key("testorig", sw) in have: cases.append(have[_key("testorig", sw)]); continue
        a = O.ref_cjpeg(ppm, sw)                   # the reference's own cjpeg binary
        b = O.ref_encode(img, sw)                  # our driver around the reference library
        assert a == b, ("refshim disagrees with cjpeg", sw)
        cases.append({"image": "testorig", "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    for sw in CJPEG_ONLY:
        a = O.ref_cjpeg(ppm, sw)
        cases.append({"image": "testorig", "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    for sw in SWITCH_SETS_EXTRA:
        a = O.ref_cjpeg(ppm, sw)
        cases.append({"image": "testorig", "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    expand = lambda sw: [os.path.join(GOLD, x[6:]) if x.startswith("@GOLD/") else x for x in sw]
    for sw in SWITCH_SETS_FILES:
        a = O.ref_cjpeg(ppm, expand(sw))
        cases.append({"image": "testorig", "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    for (seed, sw_, sh_) in SYNTH[:4]:
        im = O.synth_image(seed, sw_, sh_)
        for sw in SWITCH_SETS_FILES:
            a = O.ref_encode(im, expand(sw))
            cases.append({"image": [seed, sw_, sh_], "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    # maximum dimensions (JPEG_MAX_DIMENSION 65500, jmorecfg.h): one block row / one block column
    for (seed, sw_, sh_) in [(18, 65500, 3), (19, 3, 65500)]:
        im = O.synth_image(seed, sw_, sh_)
        for sw in (["-baseline", "-quality", "75"], ["-quality", "75"], ["-fastcrush", "-quality", "75", "-sample", "2x2"], ["-revert", "-restart", "1"],
                   ["-baseline", "-quality", "85", "-sample", "1x1"], ["-baseline", "-grayscale", "-quality", "75"], ["-revert", "-sample", "2x1", "-optimize"],
                   ["-baseline", "-quality", "75", "-restart", "1"], ["-dct", "float", "-baseline", "-quality", "75"], ["-baseline", "-quality", "75", "-smooth", "30"]):
            if _key([seed, sw_, sh_], sw) in have: cases.append(have[_key([seed, sw_, sh_], sw)]); continue
            a = O.ref_encode(im, sw)
            cases.append({"image": [seed, sw_, sh_], "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    for (seed, sw_, sh_) in SYNTH:
        im = O.synth_image(seed, sw_, sh_)
        sets = SWITCH_SETS + SWITCH_SETS_EXTRA if sw_ * sh_ <= 640 * 480 else [s for s in SWITCH_SETS if s in (["-revert", "-dct", "int"], ["-baseline", "-quality", "75", "-sample", "2x2"], ["-fastcrush", "-quality", "75", "-sample", "2x2"], ["-baseline", "-quality", "90", "-sample", "2x2"], ["-quality", "75"])]
        for sw in sets:
            if _key([seed, sw_, sh_], sw) in have: cases.append(have[_key([seed, sw_, sh_], sw)]); continue
            a = O.ref_encode(im, sw)
            cases.append({"image": [seed, sw_, sh_], "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    from mozjpeg_b200.synth import synth_image12
    for (seed, sw_, sh_) in SYNTH12:
        im = synth_image12(seed, sw_, sh_)
        for sw in SWITCH_SETS_12:
            if _key([seed, sw_, sh_, 12], sw) in have: cases.append(have[_key([seed, sw_, sh_, 12], sw)]); continue
            a = O.ref_encode(im, sw)
            cases.append({"image": [seed, sw_, sh_, 12], "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    # raw-data input (jpeg_write_raw_data): separate fixture, the inputs are component planes
    from mozjpeg_b200.synth import synth_planes
    raw_cases = []
    for (seed, w_, h_) in [(31, 33, 17), (32, 200, 136), (33, 227, 149), (34, 640, 480)]:
        for sw in (["-baseline", "-quality", "75"], ["-quality", "75"], ["-baseline", "-quality", "85", "-sample", "1x1"],
                   ["-fastcrush", "-quality", "60", "-sample", "2x1"], ["-baseline", "-quality", "75", "-grayscale"],
                   ["-baseline", "-notrellis", "-quality", "90", "-sample", "1x2", "-dct", "float"],
                   ["-baseline", "-quality", "75", "-sample", "4x2"], ["-fastcrush", "-quality", "70", "-sample", "2x2,1x1,2x2"]):
            pp = cjpeg.params_from_switches(sw, w_, h_, 1 if "-grayscale" in sw else 3)
            a = O.ref_encode_raw(synth_planes(pp, seed), w_, h_, sw)
            raw_cases.append({"seed": seed, "width": w_, "height": h_, "switches": sw, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    json.dump({"generator": "tools/make_golden.py", "cases": raw_cases}, open(os.path.join(GOLD, "raw_golden.json"), "w"), indent=0)
    # coefficient-domain re-encode (jpegtran = jpeg_read_coefficients + jpeg_write_coefficients): the source file is
    # what the reference's encoder makes of (seed, size, enc switches); the md5 is what the reference's own jpegtran
    # binary writes for (tran switches), its keep-the-smaller-file rule (jpegtran.c:772-775) included
    tr_cases = []
    for (seed, w_, h_) in [(41, 33, 17), (42, 200, 136), (43, 1, 1), (44, 640, 480)]:
        im = O.synth_image(seed, w_, h_)
        for esw in (["-revert"], ["-quality", "75"], ["-baseline", "-quality", "85", "-sample", "1x1"], ["-revert", "-grayscale", "-progressive"],
                    ["-fastcrush", "-quality", "60", "-sample", "2x1"], ["-revert", "-sample", "3x2"]):
            srcfile = O.ref_encode(im, esw)
            for tsw in ([], ["-revert"], ["-optimize"], ["-progressive"], ["-fastcrush"], ["-revert", "-optimize"], ["-revert", "-progressive"],
                        ["-restart", "1"], ["-fastcrush", "-restart", "2B"], ["-progressive", "-fastcrush"], ["-copy", "none", "-progressive", "-restart", "1"]):
                a = O.ref_jpegtran(srcfile, tsw)
                tr_cases.append({"seed": seed, "width": w_, "height": h_, "enc": esw, "tran": tsw, "md5": hashlib.md5(a).hexdigest(), "size": len(a),
                                 "src_md5": hashlib.md5(srcfile).hexdigest()})
    json.dump({"generator": "tools/make_golden.py", "cases": tr_cases}, open(os.path.join(GOLD, "transcode_golden.json"), "w"), indent=0)
    # extension parameters cjpeg has no switch for (jpeg_c_set_*_param): use_scans_in_trellis / trellis_freq_split
    ext_cases = []
    for (seed, w_, h_) in [(51, 33, 17), (52, 200, 136), (53, 640, 480), (54, 1, 1)]:
        im = O.synth_image(seed, w_, h_)
        for sw in (["-baseline", "-quality", "75"], ["-fastcrush", "-quality", "75"], ["-quality", "75"], ["-baseline", "-quality", "90", "-sample", "1x1"],
                   ["-fastcrush", "-quality", "50", "-grayscale"], ["-baseline", "-quality", "80", "-restart", "1", "-sample", "2x1"],
                   ["-fastcrush", "-quality", "30", "-sample", "1x1"]):
            for ext in ({"use_scans_in_trellis": 1}, {"use_scans_in_trellis": 1, "trellis_freq_split": 3}, {"use_scans_in_trellis": 1, "trellis_freq_split": 20},
                        {"trellis_num_loops": 2}, {"trellis_num_loops": 3, "use_scans_in_trellis": 1},
                        {"trellis_q_opt": 1}, {"trellis_q_opt": 1, "trellis_num_loops": 2}, {"trellis_q_opt": 1, "trellis_num_loops": 3, "use_scans_in_trellis": 1},
                        {"trellis_eob_opt": 1}, {"trellis_eob_opt": 1, "use_scans_in_trellis": 1}, {"trellis_eob_opt": 1, "trellis_q_opt": 1, "trellis_num_loops": 2}):
                a = O.ref_encode(im, sw, ext)
                ext_cases.append({"seed": seed, "width": w_, "height": h_, "switches": sw, "ext": ext, "md5": hashlib.md5(a).hexdigest(), "size": len(a)})
    json.dump({"generator": "tools/make_golden.py", "cases": ext_cases}, open(os.path.join(GOLD, "ext_golden.json"), "w"), indent=0)
    assert cases[0]["md5"] == "9a68f56bc76e466aa7e52f415d0f4a5f", "reference build does not reproduce MD5_JPEG_420_ISLOW"
    json.dump({"generator": "tools/make_golden.py", "reference": "mozilla/mozjpeg 5.0.0 (C path, WITH_SIMD=0), oracle/_ref", "cases": cases},
              open(os.path.join(GOLD, "golden.json"), "w"), indent=0)
    print("wrote", len(cases), "cases")


if __name__ == "__main__":
    main()
