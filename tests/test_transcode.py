"""Coefficient-domain re-encode (jpeg_write_coefficients, the encode half of jpegtran): quantized coefficients in,
re-optimized file out.  The md5s in tests/golden/transcode_golden.json were recorded from the unmodified reference's
own jpegtran binary (tools/make_golden.py).  Source files and their coefficient planes come from the CPU oracle
(bit-identical to the reference's encoder on these inputs: the recorded src_md5 is checked)."""
import hashlib
import json
import os

import numpy as np
import pytest

from common import GOLD

TR = json.load(open(os.path.join(GOLD, "transcode_golden.json")))["cases"]
_src_cache = {}


def _id(c):
    return "%dx%d:%s:%s" % (c["width"], c["height"], "_".join(s.lstrip("-") for s in c["enc"]), "_".join(s.lstrip("-") for s in c["tran"]) or "default")


def _source(c):
    """(source file, [per component (hib, wib, 64) int16 natural-order planes]) of a case."""
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    key = (c["seed"], c["width"], c["height"], tuple(c["enc"]))
    if key not in _src_cache:
        im = O.synth_image(c["seed"], c["width"], c["height"])
        p = mj.params_from_switches(c["enc"], c["width"], c["height"], 3)
        r = O.oracle_encode(p, im, want_debug=True)
        assert hashlib.md5(r.jpeg).hexdigest() == c["src_md5"]
        d = r.dbg
        planes = [np.ascontiguousarray(d["final"][ci][:d["hib"][ci], :d["wib"][ci]]) for ci in range(d["ncomp"])]
        _src_cache.clear()
        _src_cache[key] = (r.jpeg, planes)
    return _src_cache[key]


def _expected_ok(out, c):
    return len(out) == c["size"] and hashlib.md5(out).hexdigest() == c["md5"]


@pytest.mark.parametrize("c", TR, ids=_id)
def test_oracle_transcode_matches_recorded_jpegtran(built, c):
    from mozjpeg_b200 import jpegtran as T, _abi as A
    from oracle import oracle as O
    src, planes = _source(c)
    p, prefer_smallest = T.params_for_transcode(T.parse_header(src), c["tran"])
    out = O.oracle_encode_coefs(p, planes)
    if prefer_smallest and p.compress_profile == A.PROFILE_MAX_COMPRESSION and len(src) < len(out):
        out = src
    assert _expected_ok(out, c)


@pytest.mark.gpu
@pytest.mark.parametrize("c", TR, ids=_id)
def test_device_transcode_matches_recorded_jpegtran(encoder, c):
    from mozjpeg_b200 import jpegtran as T
    src, planes = _source(c)
    out = T.transcode(encoder, [src], [a[None] for a in planes], c["tran"])[0]
    assert _expected_ok(out, c)


@pytest.mark.gpu
def test_device_transcode_batch_and_roundtrip(encoder):
    """A batch through the chunked pipeline, padded block pitch; and the size-independent property of the row:
    re-encoding the encoder's own output with the encoder's own parameters reproduces the file byte for byte."""
    import mozjpeg_b200 as mj
    from mozjpeg_b200 import jpegtran as T
    from oracle import oracle as O
    w, h, n = 200, 136, 5
    penc = mj.params_from_switches(["-quality", "80"], w, h, 3)
    rs = [O.oracle_encode(penc, O.synth_image(70 + i, w, h), want_debug=True) for i in range(n)]
    d = rs[0].dbg
    stacked = []
    for ci in range(d["ncomp"]):
        buf = np.zeros((n, d["hib"][ci] + 1, d["wib"][ci] + 3, 64), dtype=np.int16)
        for i in range(n):
            buf[i, :d["hib"][ci], :d["wib"][ci]] = rs[i].dbg["final"][ci][:d["hib"][ci], :d["wib"][ci]]
        stacked.append(buf[:, :d["hib"][ci], :d["wib"][ci]])
    srcs = [r.jpeg for r in rs]
    p, _ = T.params_for_transcode(T.parse_header(srcs[0]), ["-progressive"])
    encoder.set_chunk_images(2)
    try:
        got = encoder.encode_batch_coefs(p, stacked)
    finally:
        encoder.set_chunk_images(0)
    want = [O.oracle_encode_coefs(p, [np.ascontiguousarray(a[i]) for a in stacked]) for i in range(n)]
    assert got == want
    # round trip: same parameters as the encode, minus the trellis (its result is already in the coefficients)
    q = penc.copy(); q.trellis_quant = 0
    assert encoder.encode_batch_coefs(q, stacked) == srcs


def test_oracle_transcode_live_against_reference_odd_sources(built):
    """Sources the recorded cases do not have: 16-bit quantization tables, an RGB-colourspace file, restart markers in
    the source, 12-bit precision - the files the reference wrote, their coefficients as the reference's decoder reads
    them, and the md5s of what the reference's jpegtran makes of them (tests/golden/transcode_odd_golden.npz)."""
    from mozjpeg_b200 import jpegtran as T, _abi as A
    from oracle import oracle as O
    g = np.load(os.path.join(GOLD, "transcode_odd_golden.npz"))
    trans = [t.split() for t in g["tran"]]
    assert g["md5"].shape == (6, len(trans))
    for k in range(g["md5"].shape[0]):
        src = g["src%d" % k].tobytes()
        info = T.parse_header(src)
        planes = [g["coef%d_%d" % (k, ci)] for ci in range(info.num_components)]
        for j, tsw in enumerate(trans):
            p, prefer_smallest = T.params_for_transcode(info, tsw)
            out = O.oracle_encode_coefs(p, planes)
            if prefer_smallest and p.compress_profile == A.PROFILE_MAX_COMPRESSION and len(src) < len(out):
                out = src
            assert (len(out), hashlib.md5(out).hexdigest()) == (g["size"][k, j], g["md5"][k, j]), (k, info.data_precision, tsw)
