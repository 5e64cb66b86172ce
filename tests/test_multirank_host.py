"""CPU, world_size 2 over gloo: the host-side logic of the multi-GPU path (SURVEY 8e: images shard by rank, no
collective on the data path, elapsed time = MAX over ranks, value = all ranks' pixels / that time), and the launch
contract of the reference arm under torchrun (rank 0 alone runs and prints)."""
import hashlib
import json
import os
import socket
import subprocess
import sys

from common import ROOT


def _port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _torchrun(script_args, timeout=600):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_port()), *script_args]
    return subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout)


def test_shards_and_max_reduction_over_gloo(built):
    import mozjpeg_b200 as mj
    from oracle import oracle as O
    r = _torchrun([os.path.join(ROOT, "tests", "_gloo_worker.py")])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout                     # rank 0 alone reports
    d = json.loads(lines[0])
    assert d["world"] == 2 and [x["rank"] for x in d["ranks"]] == [0, 1]
    s0, s1 = d["ranks"][0]["seeds"], d["ranks"][1]["seeds"]
    assert not set(s0) & set(s1)                         # disjoint shards
    assert all(x["elapsed"] == 11.0 for x in d["ranks"])  # MAX over ranks, seen by every rank
    assert d["mp_per_step"] == 2 * 2 * 48 * 40 / 1e6     # whole-job pixels: weak scaling
    # the sharded job == the same images encoded in one process
    p = mj.params_from_switches(["-baseline", "-quality", "75"], 48, 40)
    for x in d["ranks"]:
        assert x["digests"] == [hashlib.md5(O.oracle_encode(p, O.synth_image(s, 48, 40)).jpeg).hexdigest() for s in x["seeds"]]


def test_reference_arm_under_torchrun_prints_once(built):
    """Where oracle/_ref is not built the arm runs the oracle port and must say so."""
    from oracle import oracle as O
    r = _torchrun([os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--width", "64", "--height", "48"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == ("reference" if O.ref_available() else "port")


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec); spec.loader.exec_module(m)
    return m


def _no_nvidia_smi(*args, **kwargs):
    raise FileNotFoundError("nvidia-smi")


def test_clock_sampler_window_and_fallback(monkeypatch):
    """bench.py's `clocks` entry: the samples between the two marks are the ones reported (median SM clock, union of the
    throttle reasons), a timed region shorter than one sampling period falls back to warm-up + timed region and says so,
    and a box without NVML / nvidia-smi yields a null entry instead of an exception."""
    b = _bench_module()
    with monkeypatch.context() as m:                      # neither source comes up, also where a GPU is present
        m.setitem(sys.modules, "pynvml", None)
        m.setattr(b.subprocess, "Popen", _no_nvidia_smi)
        c = b.ClockSampler(0)
        c.start(); out = c.stop(0, None)
    assert out["samples"] == 0 and out["sm_mhz"] is None
    c = b.ClockSampler(0); c.source = "nvml"
    c.samples = [(1500.0, 1965.0, ()), (1600.0, 1965.0, ())]                       # warm-up
    lo = c.mark()
    c.samples += [(1965.0, 1965.0, ()), (1950.0, 1965.0, ("sw_power_cap",)), (1965.0, 1965.0, ())]
    hi = c.mark()
    c.samples += [(900.0, 1965.0, ("hw_slowdown",))]                               # after the timed region: not reported
    out = c.stop(lo, hi)
    assert out["samples"] == 3 and out["sm_mhz"] == 1965.0 and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["sw_power_cap"] and out["window"] == "timed region"
    c = b.ClockSampler(0); c.source = "nvml"; c.samples = [(1800.0, 1965.0, ())]
    out = c.stop(1, 1)                                    # nothing inside the marks
    assert out["samples"] == 1 and out["window"].startswith("warm-up")


def test_dump_outputs_sample_and_budget(tmp_path):
    """bench.py --dump-outputs: every file's size, whole files of a fixed sample within the byte budget, float32 bytes."""
    import numpy as np
    b = _bench_module()
    rng = np.random.default_rng(1)
    files = [rng.integers(0, 256, int(n), dtype=np.uint8).tobytes() for n in rng.integers(1000, 50000, 40)]
    b.dump_outputs(str(tmp_path / "all"), files)                      # everything fits
    sizes = np.load(tmp_path / "all" / "jpeg_sizes.npy"); images = np.load(tmp_path / "all" / "jpeg_images.npy")
    data = np.load(tmp_path / "all" / "jpeg_bytes.npy")
    assert sizes.dtype == np.float64 and images.dtype == np.float64 and data.dtype == np.float32
    assert sizes.tolist() == [len(f) for f in files] and images.tolist() == list(range(40))
    assert data.astype(np.uint8).tobytes() == b"".join(files)
    budget = 300000
    for run in ("a", "b"):
        b.dump_outputs(str(tmp_path / run), files, budget)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= budget
    images = np.load(tmp_path / "a" / "jpeg_images.npy").astype(int).tolist()
    assert 0 < len(images) < 40 and images == sorted(images)
    assert np.load(tmp_path / "a" / "jpeg_bytes.npy").astype(np.uint8).tobytes() == b"".join(files[i] for i in images)
    for f in ("jpeg_sizes.npy", "jpeg_images.npy", "jpeg_bytes.npy"):          # the same sample every time
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes()
