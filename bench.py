#!/usr/bin/env python3
"""bench.py -- megapixels/s of the JPEG encode hot path on N B200s.

    python bench.py --gpus N --steps K --warmup W            (ours)
    python bench.py --impl reference --gpus N --steps K --warmup W   (the reference's CPU encoder)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR    (also write the files of the last step)

A "step" is one pass of the hot path over one batch of synthetic images.
Default workload = BASELINE.json configs[1]: a batch of 256 synthetic
3840x2160 RGB images, q75, 4:2:0, trellis on, baseline (cjpeg -baseline
-quality 75 -sample 2x2).  Images shard across ranks (weak scaling: every rank
encodes its own full batch); the only collective is the final MAX/SUM reduce.

One JSON line on rank 0 (see the task contract): `value` = whole-job MP/s with
inputs resident in HBM; `e2e` = the same metric through the public C-ABI call
with HOST buffers (H2D of the pixels and D2H of the JPEG files inside the timed
region); `roofline` for the dominant kernel; `cpu_baseline` = the unmodified
reference (oracle/_ref) on the host cores, bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np


# BASELINE.json configs[1..4] (configs[0] is the reference's own CPU-runnable case, a parity test) + the library default
WORKLOADS = {
    "cfg2": dict(batch=256, width=3840, height=2160, switches="-baseline -quality 75 -sample 2x2", scaling="weak",
                 label="BASELINE.json configs[1]: batch of 256 synthetic 3840x2160 RGB, q75 4:2:0, trellis on, baseline"),
    "cfg3": dict(batch=128, width=3840, height=2160, switches="-fastcrush -quality 75 -sample 2x2", scaling="weak",
                 label="BASELINE.json configs[2]: 4K batch, progressive (jcphuff), 9-scan jpgcrush script of jpeg_simple_progression"),
    "cfg4": dict(batch=1024, width=1920, height=1080, switches="-baseline -quality 75 -sample 2x2", scaling="strong", sweep=(50, 75, 90),
                 label="BASELINE.json configs[3]: 1024-image 1920x1080 batch sharded over the GPUs, q50/75/90 sweep (value = q75)"),
    "cfg5": dict(batch=64, width=3840, height=2160, switches="-precision 12 -sample 1x1 -quality 75 -notrellis -noovershoot -baseline", scaling="weak",
                 label="BASELINE.json configs[4]: 12-bit 4:4:4 3840x2160 (jfdctint 12-bit; the reference has no trellis at 12 bits)"),
    "default": dict(batch=32, width=3840, height=2160, switches="-quality 75 -sample 2x2", scaling="weak",
                    label="library default profile (progressive + 64-candidate scan search), 4K q75 4:2:0"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS), help="BASELINE.json configuration (cfg2 = configs[1], the headline)")
    ap.add_argument("--batch", type=int, default=None, help="images per step (per GPU for weak scaling, whole job for cfg4)")
    ap.add_argument("--width", type=int, default=None)
    ap.add_argument("--height", type=int, default=None)
    ap.add_argument("--switches", default=None, help="cjpeg switch set naming the profile")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic images tiled to fill the batch")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity-gate", action="store_true", help="development only: skip the untimed byte comparison with the reference")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the JPEG files of rank 0's last step to DIR as .npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    w = WORKLOADS[a.workload]
    a.custom = any(v is not None for v in (a.batch, a.width, a.height, a.switches))
    for k in ("batch", "width", "height", "switches"):
        if getattr(a, k) is None:
            setattr(a, k, w[k])
    a.scaling = w["scaling"]; a.sweep = w.get("sweep"); a.label = w["label"]
    a.precision = 12 if "-precision 12" in a.switches else 8
    return a


def workload_name(a):
    if a.custom:
        return f"batch of {a.batch} synthetic {a.width}x{a.height} {'12-bit ' if a.precision == 12 else ''}RGB, cjpeg {a.switches} (variation of {a.workload})"
    return f"{a.label} (cjpeg {a.switches})"


def metric_name(a):
    return "megapixels/sec encode (4K RGB q75 4:2:0)" if a.workload == "cfg2" else f"megapixels/sec encode ({a.workload}: {a.width}x{a.height}, cjpeg {a.switches})"


# ---------------------------------------------------------------------------
# clocks: sample nvidia-smi during the timed region
# ---------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons of one GPU while it is under load.  NVML in-process every few ms (nvidia_ml_py), the
    `nvidia-smi -lms` loop of the profiling recipe as the fallback; the device is addressed by UUID, so a
    CUDA_VISIBLE_DEVICES remapping cannot point the sampler at another GPU.  It runs from before the warm-up; mark()
    brackets the timed region and stop() reports the samples inside it (if the region was too short to catch one --
    a few tens of ms -- the samples of warm-up + timed region, said so in "window")."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index = index; self.proc = None; self.samples = []; self.source = None; self._stop = threading.Event(); self.th = None
        self.sel = str(index)
        try:
            import torch
            u = str(torch.cuda.get_device_properties(index).uuid)
            self.sel = u if u.startswith("GPU-") else "GPU-" + u
        except Exception:
            pass

    def _nvml_loop(self, nv, h, mx):
        bits = [(getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8), "hw_slowdown"), (getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40), "hw_thermal_slowdown"),
                (getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), "sw_thermal_slowdown"), (getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4), "sw_power_cap")]
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)); r = int(get_reasons(h))
                self.samples.append((sm, mx, tuple(nm for b, nm in bits if r & b)))
            except Exception:
                pass
            time.sleep(0.004)

    def _smi_loop(self):
        for ln in self.proc.stdout:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                self.samples.append((float(f[0]), float(f[1]), tuple(nm for nm, v in zip(self.NAMES, f[2:6]) if v.lower().startswith("active"))))
            except ValueError:
                continue

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByUUID(self.sel) if self.sel.startswith("GPU-") else nv.nvmlDeviceGetHandleByIndex(self.index)
            mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
            self.source = "nvml"
            self.th = threading.Thread(target=self._nvml_loop, args=(nv, h, mx), daemon=True); self.th.start()
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.sel, f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            self.th = threading.Thread(target=self._smi_loop, daemon=True); self.th.start()
        except Exception:
            self.proc = None

    def mark(self) -> int:
        return len(self.samples)

    def stop(self, lo: int = 0, hi: int | None = None):
        try:
            return self._stop_impl(lo, hi)
        except Exception as ex:                       # the sampler must never take the bench line down
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"clock sampler failed: {ex!r}"], "samples": 0}

    def _stop_impl(self, lo: int = 0, hi: int | None = None):
        self._stop.set()
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.th:
            self.th.join(timeout=2)
        if self.source is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"], "samples": 0}
        hi = len(self.samples) if hi is None else hi
        win, window = self.samples[lo:hi], "timed region"
        if not win:
            win, window = self.samples[:max(hi, lo + 1)] or self.samples, "warm-up + timed region (the timed region was shorter than one sampling period)"
        sm = [x[0] for x in win]; mx = [x[1] for x in win]; reasons = set(r for x in win for r in x[2])
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": self.source, "window": window}


# ---------------------------------------------------------------------------
# the reference's CPU encoder on the host cores (oracle/_ref via refshim)
# ---------------------------------------------------------------------------
def cpu_reference_run(images, switches, threads, reps):
    """Each thread encodes `reps` images with the UNMODIFIED reference library
    (oracle/_ref; ctypes releases the GIL).  Returns (MP/s, kind, seconds).
    Never touches the product package: with the reference library absent the
    oracle port stands in (kind "port")."""
    from oracle import oracle as O
    use_ref = O.ref_available()
    h, w = images[0].shape[:2]
    if use_ref:
        O.ref()
        fn = lambda im: O.ref_encode(im, switches)
    else:
        import mozjpeg_b200 as mj                     # parameter parsing only (cjpeg switch semantics)
        p = mj.params_from_switches(switches, w, h)
        O.orc()
        fn = lambda im: O.oracle_encode(p, im).jpeg
    done = [0] * threads

    def work(t):
        for r in range(reps):
            fn(images[(t + r) % len(images)]); done[t] += 1
    ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    t0 = time.perf_counter()
    for t in ths: t.start()
    for t in ths: t.join()
    dt = time.perf_counter() - t0
    mp = sum(done) * w * h / 1e6
    return mp / dt, ("reference" if use_ref else "port"), dt


_PROXY_IMAGES = None


def _simd_proxy_worker(args):
    import io
    from PIL import Image
    t, reps = args
    pil = [Image.fromarray(im) for im in _PROXY_IMAGES]
    for r in range(reps):
        buf = io.BytesIO()
        pil[(t + r) % len(pil)].save(buf, format="JPEG", quality=75, subsampling=2, optimize=False)
    return reps


def simd_proxy_run(images, procs, reps):
    """SURVEY 8(d)(iii): no NASM on these boxes, so the reference's SIMD objects cannot be built; Pillow's bundled
    libjpeg-turbo (AVX2) is the labelled proxy for the SIMD CPU path.  It can only encode the `-revert` profile (no
    trellis, no scan search, fixed Huffman tables) -- the profile SIMD actually accelerates: the trellis, 62 % of the
    default profile's CPU time (SURVEY 8a), has no SIMD implementation in the reference.  One forked worker process per
    host thread (Pillow holds the GIL around its encoder loop).  Returns MP/s or None."""
    global _PROXY_IMAGES
    try:
        import multiprocessing as mp
        from PIL import Image  # noqa: F401
        _PROXY_IMAGES = images
        h, w = images[0].shape[:2]
        with mp.get_context("fork").Pool(procs) as pool:
            pool.map(_simd_proxy_worker, [(t, 1) for t in range(procs)])          # workers up, images converted once
            t0 = time.perf_counter()
            done = sum(pool.map(_simd_proxy_worker, [(t, reps) for t in range(procs)]))
            dt = time.perf_counter() - t0
        return done * w * h / 1e6 / dt
    except Exception:
        return None


def host_threads():
    """Host threads the reference arm can really use: the CPU affinity mask,
    capped by the cgroup CPU quota (the GPU boxes expose 128 logical CPUs but
    cap the container at 16 CPUs' worth of time; more threads only thrash)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(round(int(quota) / int(period)))))
    except Exception:
        pass
    return n


def run_reference_arm(a, rank, world):
    """--impl reference: the reference's own CPU implementation (oracle/_ref, C path: this image has no NASM), all the
    host threads the container may use, on the same workload.  Each step is a bounded sample (one image per host thread)
    so that K+W steps end within minutes.  The process never imports the product package."""
    if rank != 0:
        return
    os.environ["B200JPEG_ORACLE_STANDALONE"] = "1"
    from oracle import oracle as O
    sw = a.switches.split()
    threads = host_threads()
    gen = O.synth_image12 if a.precision == 12 else O.synth_image
    imgs = [gen(1000 + i, a.width, a.height) for i in range(min(a.distinct, 8))]
    per = a.width * a.height / 1e6
    reps = 1
    for _ in range(a.warmup):
        cpu_reference_run(imgs, sw, threads, reps)
    t0 = time.perf_counter(); kind = "reference"
    for _ in range(a.steps):
        _, kind, _ = cpu_reference_run(imgs, sw, threads, reps)
    dt = time.perf_counter() - t0
    val = a.steps * threads * reps * per / dt
    sample = f"{threads * reps} images {a.width}x{a.height} per step (one per host thread, {len(imgs)} distinct), a bounded sample of the batch of {a.batch}"
    line = {"impl": "reference", "metric": metric_name(a), "value": val, "unit": "MP/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3,
            "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "int32 DCT / fp32 trellis costs (CPU, C path without SIMD)", "data": "synthetic",
            "config": {"workload": workload_name(a), "sample_per_step": sample},
            "cpu_baseline": {"value": val, "unit": "MP/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def bind_to_gpu_numa_node(local: int):
    """Run this rank's host thread (and so its pinned allocations, by first touch) on the NUMA node the GPU hangs off:
    on the 8-GPU boxes GPU0-3 / GPU4-7 sit on different sockets and staging across the socket link costs ~10 % of
    the end-to-end rate.  Best effort; returns a note for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return "numa node unknown"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return f"numa node {node}: no allowed cpu"
        os.sched_setaffinity(0, allowed)
        return f"numa node {node} ({len(allowed)} cpus)"
    except Exception as e:                             # containers without sysfs access: leave the affinity alone
        return f"not bound ({type(e).__name__})"


def rank_seeds(rank: int, distinct: int):
    """Synthetic-image seeds of one rank: the batch shards by rank (SURVEY 8e), every rank encodes images of its own."""
    return [1000 * (rank + 1) + i for i in range(distinct)]


def max_over_ranks(value: float, world: int, device) -> float:
    """The contract's timing rule: a multi-rank number is the MAX over ranks (one all-reduce at the end; the data path
    itself has no collective).  `device` is where the process group lives (cuda:<local> for NCCL, cpu for gloo)."""
    import torch
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def whole_job_mp_per_step(world: int, batch: int, width: int, height: int) -> float:
    """Megapixels one step encodes over ALL ranks (weak scaling: every rank has its own full batch)."""
    return world * batch * width * height / 1e6


def parity_gate(outputs, images, switches, who):
    """Untimed: the bytes the timed call produced for a few images must be the reference's bytes for the same pixels
    and switches (oracle/_ref when it is there, else the oracle port).  A mismatch voids the run."""
    from oracle import oracle as O
    use_ref = O.ref_available()
    if not use_ref:
        import mozjpeg_b200 as mj
    res = [None] * len(images)

    def one(k):
        im = images[k]
        if use_ref:
            res[k] = O.ref_encode(im, switches)
        else:
            res[k] = O.oracle_encode(mj.params_from_switches(switches, im.shape[1], im.shape[0]), im).jpeg
    ths = [threading.Thread(target=one, args=(k,)) for k in range(len(images))]
    for t in ths: t.start()
    for t in ths: t.join()
    bad = [k for k in range(len(images)) if res[k] != outputs[k]]
    if bad:
        raise SystemExit(f"bench.py: PARITY GATE FAILED ({who}): output of image(s) {bad} differs from the reference's bytes "
                         f"({[len(outputs[k]) for k in bad]} vs {[len(res[k]) for k in bad]} bytes); no number is reported")
    return {"checked_images": len(images), "against": "oracle/_ref (unmodified reference)" if use_ref else "oracle port", "identical": True}


def dump_outputs(path, files, budget=64 * 10**6):
    """--dump-outputs: the JPEG files one step returned, as float32 byte values, so that two builds can be compared
    output for output.  jpeg_sizes.npy holds every file's length in bytes; jpeg_bytes.npy the files of a seeded sample
    of the batch, concatenated in image order; jpeg_images.npy the indices of those images.  The sample takes whole
    files in a fixed random order while the three arrays stay within `budget` bytes (all files when they fit)."""
    os.makedirs(path, exist_ok=True)
    room = (budget - 3 * 4096 - 16 * len(files)) // 4          # npy headers, sizes + indices as float64
    pick = []
    for i in np.random.default_rng(0).permutation(len(files)):
        if len(files[i]) <= room:
            pick.append(int(i)); room -= len(files[i])
    pick.sort()
    np.save(os.path.join(path, "jpeg_sizes.npy"), np.array([len(f) for f in files], dtype=np.float64))
    np.save(os.path.join(path, "jpeg_images.npy"), np.array(pick, dtype=np.float64))
    np.save(os.path.join(path, "jpeg_bytes.npy"), np.frombuffer(b"".join(files[i] for i in pick), dtype=np.uint8).astype(np.float32))


def measure(a, sw, enc, host, devbuf, base, rank, world, local, dev, stream, dist, torch):
    """One configuration (switch set) on the already staged batch: resident value, e2e, stage times, parity gate."""
    import mozjpeg_b200 as mj
    W, H = a.width, a.height
    B = host.shape[0]
    p = mj.params_from_switches(sw, W, H)
    sb = 2 if a.precision == 12 else 1
    row_pitch, image_stride = W * 3 * sb, W * H * 3 * sb

    def step_resident():
        enc.encode_batch_ptr(p, devbuf.data_ptr(), True, row_pitch, image_stride, B, device_only=True)

    def step_e2e():
        enc.encode_batch_ptr(p, host.data_ptr(), False, row_pitch, image_stride, B)
        return sum(enc.output_size(i) for i in range(B))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident (kernel pipeline only) ----
    clocks = ClockSampler(local); clocks.start()
    for _ in range(a.warmup):
        step_resident()
    barrier()
    clk_lo = clocks.mark()
    l0 = enc.kernel_launches()
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(a.steps):
        step_resident()
    ev1.record(stream)
    barrier()
    clk_hi = clocks.mark()
    ms_total = ev0.elapsed_time(ev1)
    launches = enc.kernel_launches() - l0
    # per-kernel times for the roofline: one extra, untimed pass with a single compute stream
    # (in the timed region consecutive chunks overlap on two streams, so stage intervals overlap too)
    enc.set_streams(1)
    step_resident()
    torch.cuda.synchronize()
    stages = {k: v for k, v in enc.stage_times().items() if k not in ("h2d", "h2d_wait")}
    chunk = enc.chunk_images()
    enc.set_streams(max(1, min(4, int(os.environ.get("B200JPEG_STREAMS", "2")))))
    clk = clocks.stop(clk_lo, clk_hi)
    ms_total = max_over_ranks(ms_total, world, dev)

    # ---- end to end through the public API: host pixels in, JPEG files out ----
    e2e_ms = None; jpeg_bytes = 0
    if not a.no_e2e:
        for _ in range(2):                            # warm: output buffers grow to the workload's sizes, the pinned file arena is consolidated
            jpeg_bytes = step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            jpeg_bytes = step_e2e()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3     # includes host-side file assembly, which events do not see
        e2e_ms = max_over_ranks(wall_ms, world, dev)
    else:
        step_e2e()                                     # the parity gate needs files
        jpeg_bytes = sum(enc.output_size(i) for i in range(B))
    # the files of the last step (the resident steps encode the same pixels with the same parameters but leave their
    # entropy-coded bytes in HBM; the end-to-end call is the one that returns files)
    files = [enc.get_output(i) for i in range(B)] if a.dump_outputs and rank == 0 else None

    # ---- parity gate (untimed): first and last image of this rank's batch against the reference ----
    gate = None
    if not a.no_parity_gate:
        idx = sorted({0, B - 1})
        gate = parity_gate([enc.get_output(i) for i in idx], [base[i % len(base)] for i in idx], sw, f"rank {rank}, {' '.join(sw)}")
    return {"ms_total": ms_total, "launches": launches, "stages": stages, "chunk": chunk, "clk": clk, "e2e_ms": e2e_ms,
            "jpeg_bytes": jpeg_bytes, "gate": gate, "B": B, "files": files}


def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference_arm(a, rank, world)
        return

    import torch
    import torch.distributed as dist
    import mozjpeg_b200 as mj
    from mozjpeg_b200.synth import synth_image, synth_image12

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)                # before the pinned buffers are allocated (first touch)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # keep stdout to the one JSON line: NCCL writes its version banner (and, with NCCL_DEBUG=INFO, its log) to the
        # process's stdout when the communicator comes up, so file descriptor 1 points at stderr until it has
        sys.stdout.flush()
        saved_fd = os.dup(1); os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved_fd, 1); os.close(saved_fd)
    dev = torch.device("cuda", local)
    W, H = a.width, a.height
    # weak scaling: every rank encodes its own full batch; strong (cfg4): the batch is split over the ranks
    B = a.batch if a.scaling == "weak" else (a.batch + world - 1) // world
    global_images = B * world

    # ---- synthetic inputs: `distinct` images per rank, tiled to B (inputs >> 126 MB L2)
    gen = synth_image12 if a.precision == 12 else synth_image
    cache = os.environ.get("B200JPEG_BENCH_CACHE")           # development aid: reuse the synthetic images between A/B runs
    cpath = os.path.join(cache, f"synth_{W}x{H}_{a.precision}_{a.distinct}_{rank}.npy") if cache else None
    if cpath and os.path.exists(cpath):
        base = np.load(cpath)
    else:
        base = np.stack([gen(seed, W, H) for seed in rank_seeds(rank, a.distinct)])
        if cpath:
            np.save(cpath, base)
    host = torch.empty((B, H, W, 3), dtype=torch.int16 if a.precision == 12 else torch.uint8, pin_memory=True)   # 12-bit samples: 16-bit words
    hb = torch.from_numpy(base.view(np.int16) if a.precision == 12 else base)
    for i in range(B):
        host[i].copy_(hb[i % a.distinct])
    devbuf = host.to(dev, non_blocking=False)
    in_bytes = W * H * 3 * (2 if a.precision == 12 else 1)

    enc = mj.Encoder(local)
    stream = torch.cuda.current_stream()
    enc.set_stream(stream.cuda_stream)

    runs = {}
    if a.sweep and not a.custom:
        for q in a.sweep:
            sw = a.switches.replace("-quality 75", f"-quality {q}").split()
            runs[q] = measure(a, sw, enc, host, devbuf, base, rank, world, local, dev, stream, dist, torch)
            if q != 75:
                runs[q]["files"] = None                # the reported value is q75's
        r = runs[75]
    else:
        r = measure(a, a.switches.split(), enc, host, devbuf, base, rank, world, local, dev, stream, dist, torch)

    mp_per_step = global_images * W * H / 1e6
    value = mp_per_step * a.steps / (r["ms_total"] / 1e3)
    e2e = None
    if r["e2e_ms"] is not None:
        e2e = {"value": mp_per_step * a.steps / (r["e2e_ms"] / 1e3), "unit": "MP/s", "h2d_bytes_per_step": B * in_bytes,
               "d2h_bytes_per_step": int(r["jpeg_bytes"]), "ms_per_step": r["e2e_ms"] / a.steps,
               "timer": "host wall clock around the API calls, max over ranks", "bytes_are": "per rank"}

    # ---- roofline of the dominant kernel (CUDA events inside the library; one single-stream pass over the batch) ----
    stages = r["stages"]
    dom = max(stages, key=stages.get)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    out_bytes = r["jpeg_bytes"] / B
    # the dominant stage is launched once per chunk of the batch; its stage time is the sum over the chunks, so
    # (algorithmic bytes of the whole batch) / (summed time) is the mean over launches of bytes-per-launch / duration
    chunk = r["chunk"]
    per_launch = [min(chunk, B - i) for i in range(0, B, chunk)]
    alg_per_image = in_bytes + out_bytes                               # SURVEY 8(d): input bytes + JPEG bytes per image
    achieved = B * alg_per_image / (stages[dom] / 1e3) / 1e9
    pipeline = B * alg_per_image / (sum(stages.values()) / 1e3) / 1e9
    traffic = None; traffic_src = None
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")))
        if prof.get("kernel") == dom and a.workload == "cfg2":
            traffic = prof.get("dram_bytes_per_image") * max(per_launch); traffic_src = prof.get("source")
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel_ms": stages[dom] / len(per_launch),
                "launches_per_step": len(per_launch), "images_per_launch": per_launch,
                "algorithmic_bytes_per_image": alg_per_image, "algorithmic_bytes_per_launch": max(per_launch) * alg_per_image,
                "pipeline_achieved": pipeline, "pipeline_frac": pipeline / peak, "stage_ms": stages}

    # ---- the reference's CPU encoder on this box's host cores (rank 0, N=1 only; bounded sample) ----
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        threads = host_threads()
        imgs = [base[i] for i in range(min(4, a.distinct))]
        reps = 3 if W * H > 4e6 else 8
        v, kind, secs = cpu_reference_run(imgs, a.switches.split(), threads, reps)
        simd = None
        if a.precision == 8:
            sv = simd_proxy_run(imgs, threads, reps * 4)
            cv, _, _ = cpu_reference_run(imgs, ["-revert", "-quality", "75", "-sample", "2x2"], threads, reps * 2)
            if sv:
                simd = {"encoder": "Pillow (bundled libjpeg-turbo, AVX2) -- labelled proxy, SURVEY 8(d)(iii)", "profile": "cjpeg -revert -quality 75 -sample 2x2 (no trellis, fixed tables)",
                        "value": sv, "reference_c_same_profile": cv, "unit": "MP/s",
                        "note": "SIMD speeds up colour conversion / DCT / quantization / Huffman coding; the trellis passes of this workload's profile have no SIMD version"}
        cpu = {"value": v, "unit": "MP/s", "cores": threads, "kind": kind,
               "simd": "none (C path: no NASM on the box, so the reference's x86-64 SIMD objects cannot be built)", "simd_proxy": simd,
               "sample": f"{threads * reps} images {W}x{H} ({reps} per host thread, {secs:.1f} s wall = {secs * threads:.0f} CPU-seconds), same switches"}

    # ---- one image through the streaming entry points a libjpeg application drives (jpeg_start_compress /
    #      jpeg_write_scanlines / jpeg_finish_compress shape of the C-ABI): wall-clock latency, rank 0 only ----
    latency = None
    if rank == 0 and a.precision == 8 and not a.no_e2e:
        p1 = mj.params_from_switches(a.switches.split(), W, H)
        one = np.ascontiguousarray(base[0])
        lat = []
        for rep in range(5):
            t0 = time.perf_counter()
            enc.start_compress(p1); enc.write_scanlines(one); data = enc.finish_compress()
            lat.append((time.perf_counter() - t0) * 1e3)
        latency = {"ms": statistics.median(lat[1:]), "first_call_ms": lat[0], "bytes": len(data),
                   "what": "b200jpeg_start_compress + write_scanlines (all rows, pageable host memory) + finish_compress, one image, median of 4"}

    if r["files"] is not None:
        dump_outputs(a.dump_outputs, r["files"])
    if rank == 0:
        cfg = {"workload": workload_name(a), "images_per_gpu": B, "global_images": global_images,
               "l2": "inputs (%.1f GB per GPU) exceed the 126 MB L2" % (B * in_bytes / 1e9),
               "parallelism": f"images sharded over {world} GPU(s), no data-path collective", "host_affinity": numa,
               "parity_gate": r["gate"]}
        if runs:
            cfg["sweep"] = {f"q{q}": {"value": mp_per_step * a.steps / (x["ms_total"] / 1e3),
                                      "e2e": (mp_per_step * a.steps / (x["e2e_ms"] / 1e3)) if x["e2e_ms"] else None,
                                      "ms_per_step": x["ms_total"] / a.steps, "parity_gate": x["gate"],
                                      "stage_ms": x["stages"]} for q, x in runs.items()}
        line = {"metric": metric_name(a), "value": value, "unit": "MP/s", "n_gpus": world,
                "steps": a.steps, "warmup": a.warmup, "ms_per_step": r["ms_total"] / a.steps, "higher_is_better": True,
                "scaling": a.scaling, "vs_baseline": None,
                "dtype": ("u16 (12-bit) in / int32 DCT / u8 out" if a.precision == 12 else "u8 in / int32 DCT / fp32 trellis costs / u8 out"), "data": "synthetic",
                "config": cfg, "clocks": r["clk"], "e2e": e2e, "single_image_latency": latency, "gpu_launches": int(r["launches"]), "roofline": roofline, "cpu_baseline": cpu}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    enc.close()


if __name__ == "__main__":
    main()
