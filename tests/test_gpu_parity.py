"""GPU: the CUDA path, called through the C-ABI (libb200jpeg.so), must produce
the reference's bytes.

* every golden case recorded from the unmodified reference (tests/golden/);
* live against the CPU oracle on seeded inputs,
  including stage-level taps (coefficient planes, Huffman tables);
* at BASELINE.json's full sizes through size-independent properties
  (batch == one-by-one, device-resident == host-staged) and the recorded
  1920x1080 and 3840x2160 md5s.
"""
import ctypes as C
import os

import numpy as np
import pytest

from common import case_id, case_image, golden_cases, md5

pytestmark = pytest.mark.gpu

CASES = golden_cases()


def _encode(encoder, sw, img):
    import mozjpeg_b200 as mj
    nc = 1 if img.ndim == 2 else img.shape[2]
    p = mj.params_from_switches(sw, img.shape[1], img.shape[0], nc)
    try:
        return encoder.encode_batch(p, img[None])[0]
    except mj.B200JpegError as e:
        if e.code == -2:
            pytest.skip("not on the device path yet: " + str(e))
        raise


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_device_matches_recorded_reference(encoder, case):
    img = case_image(case)
    out = _encode(encoder, case["switches"], img)
    assert len(out) == case["size"] and md5(out) == case["md5"]


def test_config1_golden_vector(encoder):
    """BASELINE.json configs[0]: testorig.ppm -> baseline q75 4:2:0 islow == testimages/testimgint.jpg."""
    import os
    import mozjpeg_b200 as mj
    from common import GOLD
    out = mj.cjpeg(["-revert", "-dct", "int"], open(os.path.join(GOLD, "testorig.ppm"), "rb").read(), encoder)
    assert md5(out) == "9a68f56bc76e466aa7e52f415d0f4a5f"


@pytest.mark.parametrize("sw", [["-baseline", "-quality", "75"], ["-baseline", "-notrellis", "-quality", "60", "-sample", "1x1"]], ids=lambda s: "_".join(s))
def test_stage_taps_match_oracle(built, sw):
    """Coefficient planes and trellis-phase Huffman tables, not just bytes."""
    import os
    os.environ["B200JPEG_KEEP_PLAIN"] = "1"
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    enc = mj.Encoder(0)
    try:
        w, h = 227, 149
        imgs = np.stack([O.synth_image(50 + i, w, h) for i in range(3)])
        p = mj.params_from_switches(sw, w, h)
        out = enc.encode_batch(p, imgs)
        for i in range(3):
            r = O.oracle_encode(p, imgs[i], want_debug=True)
            d = r.dbg
            for ci in range(3):
                hib, wib = d["hib"][ci], d["wib"][ci]
                assert (enc.debug_coefs(i, ci, 1)[:hib, :wib] == d["raw"][ci][:hib, :wib]).all(), ("raw", i, ci)
                assert (enc.debug_coefs(i, ci, 2) == d["plain"][ci]).all(), ("plain", i, ci)
                assert (enc.debug_coefs(i, ci, 0) == d["final"][ci]).all(), ("final", i, ci)
                if p.trellis_quant:
                    assert enc.debug_huff(i, -1 - ci, False, p.comp_info[ci].dc_tbl_no) == d["trellis_dc"][ci]
                    assert enc.debug_huff(i, -1 - ci, True, p.comp_info[ci].ac_tbl_no) == d["trellis_ac"][ci]
            assert out[i] == r.jpeg
    finally:
        enc.close()
        os.environ.pop("B200JPEG_KEEP_PLAIN", None)


def test_ragged_shapes_vs_oracle(encoder):
    """Non-multiple-of-MCU sizes, 1x1, single row/column, odd sampling."""
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    rng = np.random.default_rng(5)
    shapes = [(1, 1), (1, 40), (40, 1), (7, 9), (15, 17), (16, 16), (17, 15), (31, 33), (65, 63), (129, 2)]
    sws = [["-baseline", "-quality", "75"], ["-revert"], ["-baseline", "-quality", "80", "-sample", "2x1"],
           ["-baseline", "-quality", "70", "-sample", "1x2"], ["-baseline", "-grayscale", "-quality", "75"], ["-revert", "-optimize", "-sample", "1x1"]]
    for (w, h) in shapes:
        img = O.synth_image(int(rng.integers(1 << 30)), w, h)
        for sw in sws:
            p = mj.params_from_switches(sw, w, h)
            assert encoder.encode_batch(p, img[None])[0] == O.oracle_encode(p, img).jpeg, (w, h, sw)


def test_input_smoothing_vs_oracle(encoder):
    """cjpeg -smooth N (jcsample.c:298-455 + the context-row mode of jcprepct.c): ragged sizes, every sampler family,
    the three DCTs and 12-bit samples; the 8-bit cases of the oracle are pinned to the reference in golden.json."""
    import mozjpeg_b200 as mj
    from mozjpeg_b200.synth import synth_image12
    from oracle import oracle as O
    rng = np.random.default_rng(9)
    sws = [["-baseline", "-quality", "75", "-smooth", "30"], ["-revert", "-smooth", "100", "-sample", "1x1"], ["-quality", "70", "-smooth", "12"],
           ["-baseline", "-quality", "80", "-smooth", "50", "-sample", "2x1"], ["-revert", "-smooth", "20", "-sample", "3x2"],
           ["-baseline", "-grayscale", "-smooth", "15", "-quality", "60"], ["-dct", "fast", "-baseline", "-quality", "75", "-smooth", "40"],
           ["-dct", "float", "-fastcrush", "-quality", "75", "-smooth", "8", "-sample", "1x2"], ["-fastcrush", "-smooth", "5", "-sample", "2x2,1x1,2x2"]]
    for (w, h) in [(1, 1), (1, 40), (40, 1), (7, 9), (17, 15), (31, 33), (65, 63), (200, 136), (517, 260)]:
        img = O.synth_image(int(rng.integers(1 << 30)), w, h)
        for sw in sws:
            p = mj.params_from_switches(sw, w, h)
            assert encoder.encode_batch(p, img[None])[0] == O.oracle_encode(p, img).jpeg, (w, h, sw)
    for (w, h) in [(33, 17), (200, 136)]:
        img = synth_image12(int(rng.integers(1 << 30)), w, h)
        for sw in (["-precision", "12", "-quality", "75", "-notrellis", "-noovershoot", "-baseline", "-smooth", "25"],
                   ["-precision", "12", "-quality", "85", "-notrellis", "-noovershoot", "-fastcrush", "-smooth", "60", "-sample", "1x1"]):
            p = mj.params_from_switches(sw, w, h)
            assert encoder.encode_batch(p, img[None])[0] == O.oracle_encode(p, img).jpeg, (w, h, sw)
    # a batch through the chunked pipeline
    imgs = np.stack([O.synth_image(100 + i, 200, 136) for i in range(5)])
    p = mj.params_from_switches(sws[0], 200, 136)
    encoder.set_chunk_images(2)
    try:
        got = encoder.encode_batch(p, imgs)
    finally:
        encoder.set_chunk_images(0)
    assert got == [O.oracle_encode(p, im).jpeg for im in imgs]


def test_extreme_content(encoder):
    """All-white (deringing 'completely flat' exit), all-black, random noise at q100, saturated checkerboard."""
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    rng = np.random.default_rng(9)
    w, h = 96, 80
    imgs = {"white": np.full((h, w, 3), 255, np.uint8), "black": np.zeros((h, w, 3), np.uint8),
            "noise": rng.integers(0, 256, (h, w, 3), dtype=np.uint8),
            "checker": (((np.indices((h, w)).sum(0) // 3) % 2) * 255).astype(np.uint8)[..., None].repeat(3, 2)}
    for name, img in imgs.items():
        for sw in (["-baseline", "-quality", "75"], ["-baseline", "-quality", "100"], ["-baseline", "-quality", "5"], ["-revert", "-quality", "100"]):
            p = mj.params_from_switches(sw, w, h)
            assert encoder.encode_batch(p, img[None])[0] == O.oracle_encode(p, img).jpeg, (name, sw)


def test_batch_equals_one_by_one_and_device_resident(encoder):
    """Size-independent properties at a BASELINE-sized frame (1920x1080):
    batch result == per-image result; HBM-resident input == host-staged input."""
    import torch
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    w, h, n = 1920, 1080, 6
    imgs = np.stack([O.synth_image(200 + i, w, h) for i in range(n)])
    sw = ["-baseline", "-quality", "75", "-sample", "2x2"]
    p = mj.params_from_switches(sw, w, h)
    batch = encoder.encode_batch(p, imgs)
    for i in (0, n - 1):
        assert encoder.encode_batch(p, imgs[i:i + 1])[0] == batch[i]
    t = torch.from_numpy(imgs).cuda()
    encoder.encode_batch_ptr(p, t.data_ptr(), True, w * 3, w * h * 3, n)
    assert [encoder.get_output(i) for i in range(n)] == batch
    # the recorded reference md5 for seed 17 at this size
    c = next(c for c in CASES if c["image"] == [17, 1920, 1080] and c["switches"] == sw)
    assert md5(encoder.encode_batch(p, case_image(c)[None])[0]) == c["md5"]
    # and one image checked against the oracle live
    assert batch[2] == O.oracle_encode(p, imgs[2]).jpeg


def test_full_size_4k_frame(encoder):
    """BASELINE.json configs[1] frame size (3840x2160), small batch: oracle on one
    image (seconds on CPU), the reference's recorded md5 for the other + equal results for replicated inputs."""
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    w, h = 3840, 2160
    a = O.synth_image(300, w, h); b = O.synth_image(301, w, h)
    imgs = np.stack([a, b, a, b])
    p = mj.params_from_switches(["-baseline", "-quality", "75", "-sample", "2x2"], w, h)
    out = encoder.encode_batch(p, imgs)
    assert out[0] == out[2] and out[1] == out[3] and out[0] != out[1]
    assert out[0] == O.oracle_encode(p, a).jpeg
    c = next(c for c in _fullsize_cases() if c["image"] == [301, w, h] and c["switches"] == ["-baseline", "-quality", "75", "-sample", "2x2"])
    assert len(out[1]) == c["size"] and md5(out[1]) == c["md5"]


def test_streaming_shim_matches_batch(encoder):
    """jpeg_start_compress / jpeg_write_scanlines / jpeg_finish_compress shape."""
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    w, h = 123, 77
    img = O.synth_image(77, w, h)
    p = mj.params_from_switches(["-baseline", "-quality", "75"], w, h)
    ref = encoder.encode_batch(p, img[None])[0]
    encoder.start_compress(p)
    assert encoder.write_scanlines(img[:10]) == 10
    for y in range(10, h):
        assert encoder.write_scanlines(img[y]) == 1
    assert encoder.write_scanlines(img[0]) == 0            # extra rows ignored (jcapistd.c:120-123)
    assert encoder.finish_compress() == ref
    with pytest.raises(mj.B200JpegError) as ei:            # JERR_BAD_STATE
        encoder.finish_compress()
    assert ei.value.code == -7


def test_tj3compress8_parameter_block(encoder):
    """tj3Compress8 semantics (JCP_FASTEST, turbojpeg.c:330-397) == cjpeg -revert."""
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    w, h = 200, 136
    img = O.synth_image(13, w, h)
    p = mj.tj3_params(w, h, quality=75, subsamp="420")
    q = mj.params_from_switches(["-revert", "-quality", "75", "-sample", "2x2"], w, h)
    assert encoder.encode_batch(p, img[None])[0] == encoder.encode_batch(q, img[None])[0]


@pytest.mark.parametrize("sw", [["-baseline", "-quality", "75", "-sample", "2x2"], ["-fastcrush", "-quality", "80"], ["-quality", "75"]], ids=lambda s: "_".join(s))
@pytest.mark.parametrize("chunk", [0, 1, 2, 3])
def test_chunked_pipeline_matches_oracle(built, sw, chunk):
    """A batch split into pipeline chunks (staging / kernels / read-back overlapped,
    ragged last chunk) gives the oracle's bytes for every image, host-staged and
    device-resident-independent of the chunk size.  chunk 0 = the library's own choice (the
    scan search of the default profile goes out in at least two chunks per batch)."""
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    w, h = 136, 88
    imgs = np.stack([O.synth_image(40 + s, w, h) for s in range(5)])
    p = mj.params_from_switches(sw, w, h)
    enc = mj.Encoder(0)
    try:
        enc.set_chunk_images(chunk)
        out = enc.encode_batch(p, imgs)
        for rep in range(2):                      # second call reuses the pinned arena
            out = enc.encode_batch(p, imgs)
    finally:
        enc.close()
    for i in range(len(imgs)):
        assert out[i] == O.oracle_encode(p, imgs[i]).jpeg, f"image {i}, chunk {chunk}"


def test_very_wide_image_takes_the_fallback_dc_trellis(encoder):
    """A row of 3750 blocks does not fit the warp-cooperative DC trellis's shared-memory back pointers:
    the launch falls back to the older kernels, which must give the same bytes."""
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    w, h = 30000, 16
    img = O.synth_image(77, w, h)
    sw = ["-baseline", "-quality", "75", "-sample", "1x1"]
    p = mj.params_from_switches(sw, w, h)
    assert encoder.encode_batch(p, img[None])[0] == O.oracle_encode(p, img).jpeg


def test_incompressible_input_grows_the_output_buffers(built):
    """Noise at quality 100 needs more than the initial 2 bits per coefficient: the pipeline flags the
    overflow on the device, the host grows the buffers and reruns; the result must still be exact."""
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (3, 128, 192, 3), dtype=np.uint8)
    sw = ["-baseline", "-notrellis", "-quality", "100", "-sample", "1x1"]
    p = mj.params_from_switches(sw, 192, 128)
    enc = mj.Encoder(0)
    try:
        out = enc.encode_batch(p, img)
    finally:
        enc.close()
    for i in range(3):
        assert out[i] == O.oracle_encode(p, img[i]).jpeg


@pytest.mark.gpu
def test_command_line_front_end(tmp_path):
    """python -m mozjpeg_b200.cjpeg: cjpeg's command line on the device path, one file and a batch of files."""
    import shutil
    import subprocess
    import sys
    from common import GOLD, ROOT
    sw = ["-quality", "75"]
    want = next(c for c in CASES if c["image"] == "testorig" and c["switches"] == sw)
    out = tmp_path / "o.jpg"
    r = subprocess.run([sys.executable, "-m", "mozjpeg_b200.cjpeg", *sw, "-outfile", str(out), os.path.join(GOLD, "testorig.ppm")],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert md5(out.read_bytes()) == want["md5"]
    for i in range(3):
        shutil.copyfile(os.path.join(GOLD, "testorig.ppm"), tmp_path / f"in{i}.ppm")
    r = subprocess.run([sys.executable, "-m", "mozjpeg_b200.cjpeg", *sw, *[str(tmp_path / f"in{i}.ppm") for i in range(3)]],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    assert all(md5((tmp_path / f"in{i}.jpg").read_bytes()) == want["md5"] for i in range(3))


# ---------------------------------------------------------------------------
# pixel orders of the RGB family (jccolor.c:253-291 -> jccolext.c:30-75): the same picture stored as BGR / RGBX / XBGR /
# ... must give the file the reference writes for the RGB order (its converters differ only in the sample offsets)
# ---------------------------------------------------------------------------
def _reorder(img, name):
    from mozjpeg_b200 import _abi as A
    _, size, ro, go, bo = A.CS_EXT[name]
    rng = np.random.default_rng(7)
    out = rng.integers(0, 256 if img.dtype == np.uint8 else 4096, img.shape[:2] + (size,), dtype=img.dtype)   # filler sample: noise
    out[..., ro] = img[..., 0]; out[..., go] = img[..., 1]; out[..., bo] = img[..., 2]
    return np.ascontiguousarray(out)


@pytest.mark.parametrize("order", ["EXT_RGB", "EXT_RGBX", "EXT_BGR", "EXT_BGRX", "EXT_XBGR", "EXT_XRGB", "EXT_RGBA", "EXT_BGRA", "EXT_ABGR", "EXT_ARGB"])
@pytest.mark.parametrize("sw,shape", [(["-baseline", "-quality", "75", "-sample", "2x2"], (203, 141)),
                                      (["-quality", "80", "-fastcrush"], (64, 48)),
                                      (["-baseline", "-quality", "60", "-grayscale"], (131, 77)),
                                      (["-baseline", "-quality", "75", "-rgb"], (90, 50)),
                                      (["-baseline", "-quality", "70", "-sample", "3x2"], (100, 61)),
                                      (["-baseline", "-quality", "75", "-smooth", "20"], (97, 66)),
                                      (["-precision", "12", "-quality", "75", "-notrellis", "-noovershoot", "-baseline", "-sample", "2x1"], (200, 40))],
                         ids=["420", "fastcrush", "gray", "rgb", "3x2", "smooth", "12bit"])
def test_pixel_orders(order, sw, shape):
    import mozjpeg_b200 as mj
    from mozjpeg_b200 import _abi as A
    from mozjpeg_b200.synth import synth_image12
    from oracle import oracle as O
    from common import device_supports
    w, h = shape
    twelve = "-precision" in sw
    img = synth_image12(3, w, h) if twelve else O.synth_image(3, w, h)
    p = mj.params_from_switches(sw, w, h)
    if not device_supports(p):
        pytest.skip("parameter set not on the device path")
    ref = O.oracle_encode(p, img).jpeg
    q = mj.params_from_switches(sw, w, h)
    q.in_color_space, q.input_components = A.CS_EXT[order][0], A.CS_EXT[order][1]
    enc = mj.Encoder(0)
    try:
        out = enc.encode_batch(q, _reorder(img, order)[None])[0]
    finally:
        enc.close()
    assert out == ref


# ---------------------------------------------------------------------------
# BASELINE.json's configurations at their stated sizes: md5s recorded from the unmodified reference
# (tools/make_golden.py --fullsize -> tests/golden/fullsize_golden.json)
# ---------------------------------------------------------------------------
def _fullsize_cases():
    import json
    from common import GOLD
    path = os.path.join(GOLD, "fullsize_golden.json")
    return json.load(open(path))["cases"] if os.path.exists(path) else []


@pytest.mark.parametrize("case", _fullsize_cases(), ids=case_id)
def test_full_size_recorded_reference(encoder, case):
    """4K baseline+trellis (configs[1]), 4K progressive jpgcrush script (configs[2]), 1080p q50/75/90 (configs[3]),
    12-bit 4:4:4 4K (configs[4]) and the 4K library default: byte-identical to the reference at the stated sizes."""
    img = case_image(case)
    out = _encode(encoder, case["switches"], img)
    assert len(out) == case["size"] and md5(out) == case["md5"]
