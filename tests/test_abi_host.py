"""CPU: the C-ABI library loads, exports what include/b200jpeg.h declares, and
its host-side parameter logic reproduces the reference's decisions."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from common import ROOT


def test_library_exports_every_declared_symbol(built):
    from mozjpeg_b200 import _abi as A
    lib = A.load()
    hdr = open(os.path.join(ROOT, "include", "b200jpeg.h")).read()
    declared = set(re.findall(r"\b(b200jpeg_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(A.EXPORTS), declared ^ set(A.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name


def test_params_struct_size_matches_header(built, tmp_path):
    """ctypes mirror vs the C compiler's layout."""
    import subprocess
    from mozjpeg_b200 import _abi as A
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include "b200jpeg.h"\nint main(){printf("%zu %zu %zu",sizeof(b200jpeg_params),sizeof(b200jpeg_huff_tbl),sizeof(b200jpeg_scan_info));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    a, b, c = map(int, subprocess.check_output([str(exe)]).split())
    assert (a, b, c) == (C.sizeof(A.Params), C.sizeof(A.HuffTbl), C.sizeof(A.ScanInfo))


def test_quality_scaling(built):
    from mozjpeg_b200 import _abi as A
    lib = A.load()
    # jcparam.c:334-357: q75 -> 50, q50 -> 100, q90 -> 20, q10 -> 500, clamps
    assert [lib.b200jpeg_quality_scaling(q) for q in (75, 50, 90, 10, 100, 0, 101, 1)] == [50, 100, 20, 500, 0, 5000, 0, 5000]
    assert abs(lib.b200jpeg_float_quality_scaling(75.5) - 49.0) < 1e-6


def test_switch_semantics(built):
    import mozjpeg_b200 as mj
    from mozjpeg_b200 import _abi as A
    p = mj.params_from_switches(["-baseline", "-quality", "75"], 64, 48)
    assert (p.num_scans, p.trellis_quant, p.trellis_quant_dc, p.overshoot_deringing, p.optimize_coding, p.optimize_scans) == (0, 1, 1, 1, 1, 0)
    assert p.compress_profile == A.PROFILE_MAX_COMPRESSION and p.quant_tbl_master_idx == 3
    assert [(c.h_samp_factor, c.v_samp_factor) for c in p.comp_info[:3]] == [(2, 2), (1, 1), (1, 1)]
    p = mj.params_from_switches(["-fastcrush", "-quality", "75"], 64, 48)
    assert p.num_scans == 9 and p.optimize_scans == 0                      # jpgcrush script, jcparam.c:931-958
    s = [(x.comps_in_scan, x.component_index[0], x.Ss, x.Se, x.Ah, x.Al) for x in p.scan_info[:9]]
    assert s == [(3, 0, 0, 0, 0, 0), (1, 0, 1, 8, 0, 2), (1, 1, 1, 8, 0, 0), (1, 2, 1, 8, 0, 0), (1, 0, 9, 63, 0, 2),
                 (1, 0, 1, 63, 2, 1), (1, 0, 1, 63, 1, 0), (1, 1, 9, 63, 0, 0), (1, 2, 9, 63, 0, 0)]
    p = mj.params_from_switches(["-revert"], 64, 48)
    assert (p.compress_profile, p.trellis_quant, p.optimize_coding, p.num_scans, p.quant_tbl_master_idx) == (A.PROFILE_FASTEST, 0, 0, 0, 0)
    p = mj.params_from_switches(["-quality", "75"], 64, 48)                # library default: 64-scan search script
    assert p.num_scans == 64 and p.optimize_scans == 1
    assert A.load().b200jpeg_validate(C.byref(p)) == 0                     # scan search is on the device path
    p = mj.params_from_switches(["-quality", "92"], 64, 48)                # rdswitch.c:566-570
    assert [(c.h_samp_factor, c.v_samp_factor) for c in p.comp_info[:3]] == [(1, 1)] * 3
    p = mj.params_from_switches(["-revert", "-progressive"], 64, 48)       # libjpeg-turbo 10-scan script jcparam.c:960-977
    assert p.num_scans == 10
    assert A.load().b200jpeg_total_passes(C.byref(mj.params_from_switches(["-baseline", "-quality", "75"], 64, 48))) == 8      # SURVEY 3.1
    assert A.load().b200jpeg_total_passes(C.byref(mj.params_from_switches(["-fastcrush", "-quality", "75"], 64, 48))) == 24    # SURVEY 3.2


def test_quant_tables_match_reference_dqt(built):
    """Tables we derive == tables the reference writes into its DQT (as its decoder reads them back, per component;
    tests/golden/dqt_golden.json)."""
    import json
    import mozjpeg_b200 as mj
    from common import GOLD
    cases = json.load(open(os.path.join(GOLD, "dqt_golden.json")))["cases"]
    assert len(cases) == 6
    for c in cases:
        sw, qt = c["switches"], c["qt"]
        p = mj.params_from_switches(sw, 32, 32)
        for ci in range(3):
            assert list(p.quant_tbl[p.comp_info[ci].quant_tbl_no]) == qt[ci], (sw, ci)


def test_validation_errors(built):
    import mozjpeg_b200 as mj
    from mozjpeg_b200 import _abi as A
    lib = A.load()
    p = mj.params_from_switches(["-baseline"], 16, 16)
    assert lib.b200jpeg_validate(C.byref(p)) == 0
    q = p.copy(); q.image_width = 0
    assert lib.b200jpeg_validate(C.byref(q)) == A.ERR_PARAM and b"Empty" in lib.b200jpeg_last_error()
    q = p.copy(); q.comp_info[1].h_samp_factor = 5
    assert lib.b200jpeg_validate(C.byref(q)) == A.ERR_PARAM
    q = p.copy(); q.dct_method = A.DCT_FLOAT
    assert lib.b200jpeg_validate(C.byref(q)) == 0                      # float DCT is on the device path (8-bit)
    q = p.copy(); q.dct_method = A.DCT_IFAST
    assert lib.b200jpeg_validate(C.byref(q)) == 0
    q = p.copy(); q.smoothing_factor = 10
    assert lib.b200jpeg_validate(C.byref(q)) == 0                      # input smoothing is on the device path
    q = p.copy(); q.smoothing_factor = 101
    assert lib.b200jpeg_validate(C.byref(q)) == A.ERR_PARAM
    q = p.copy(); q.trellis_q_opt = 1; q.trellis_eob_opt = 1
    assert lib.b200jpeg_validate(C.byref(q)) == 0                      # both optional trellis modes are on the device path
    q = p.copy(); q.trellis_num_loops = 17
    assert lib.b200jpeg_validate(C.byref(q)) == A.ERR_UNSUPPORTED
    q = p.copy(); q.num_scans = 1; q.scan_info[0].comps_in_scan = 1; q.scan_info[0].Ss = 0; q.scan_info[0].Se = 63
    assert lib.b200jpeg_validate(C.byref(q)) == A.ERR_PARAM and b"transmit" in lib.b200jpeg_last_error()   # JERR_MISSING_DATA


def test_no_cpu_fallback(built):
    """Without a CUDA device the encode entry points refuse to run."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import mozjpeg_b200 as mj
    with pytest.raises(mj.B200JpegError) as ei:
        mj.Encoder(0)
    assert ei.value.code == -3


def test_shim_exports_the_interposed_entry_points(built):
    """The libjpeg interposition library defines exactly the calls INTEGRATION.md says it takes over."""
    import subprocess
    shim = os.path.join(ROOT, "integration", "_build", "libjpeg_b200shim.so")
    if not os.path.exists(shim):
        pytest.skip("shim not built (needs the reference's headers at build time)")
    out = subprocess.check_output(["nm", "-D", "--defined-only", shim], text=True)
    have = {ln.split()[-1] for ln in out.splitlines() if " T " in ln}
    want = {"jpeg_start_compress", "jpeg_write_scanlines", "jpeg12_write_scanlines", "jpeg_write_raw_data", "jpeg_write_coefficients",
            "jpeg_finish_compress", "jpeg_abort_compress", "jpeg_destroy_compress", "jpeg_abort", "jpeg_destroy", "jpeg_write_marker", "jpeg_write_m_header", "jpeg_write_m_byte"}
    assert want <= have, want - have
    assert not {s for s in have if s.startswith("jpeg") and s not in want}, "an undocumented libjpeg symbol is interposed"
