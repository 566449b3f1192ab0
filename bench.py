#!/usr/bin/env python
"""bench.py — IQ Msamples/s demodulated (BASELINE.json metric) on N B200s, one process per GPU.

A *launch* is one pass of the hot path over one batch: for every one of the GPU's receivers, the next
`--buffers` reference buffers of 65536 samples (128 KiB mag_buf, `--sdr-buffer-size=128`) of its synthetic
2.4 MSPS uc8 stream.  A *step* is `--launches-per-step` such launches back to back (the ring of inputs is walked
several times), so that the timed region of the default run lasts about a second: a sustained number under the chip's
power management, not a burst on a cold chip (the burst figure is reported beside it).  Default workload =
BASELINE.json configs[2] per GPU (256 concurrent streams, DF17 injected at 100/s), which at N GPUs is configs[3]
(256 streams per GPU, independent, no collective).

  value  whole-job throughput with the IQ already resident in HBM (device ring larger than L2)
  e2e    same metric through the C-ABI with HOST buffers: pinned host -> H2D -> kernels -> frames D2H
  roofline  scan kernel: 2 B/sample x samples per launch / CUDA-event duration, vs measured HBM peak
  cpu_baseline  the reference's own convert_uc8_nodc + demodulate2400 (oracle/_ref, built from
             /root/reference) on all host cores, on a bounded sample of the same batch (rank 0, N=1)

  extra  (rank 0) BASELINE configs[1] = the drop-in's own call shape (one receiver, one 128 KiB mag_buf per blocking
         call: per-call latency beside one reference core on the same buffers), configs[4] = the dense-preamble stress,
         and a frame-for-frame comparison of the timed configuration with the CPU oracle (`parity_checked`)

`--impl reference` runs only that CPU arm and prints the same JSON line with "impl": "reference".
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

BUF = 65536                      # samples per reference buffer: 128 KiB of uint16 magnitudes
ALG_BYTES_PER_SAMPLE = 2         # uc8 I + Q, read once (SURVEY.md section 8d)
REF_PASSES = 16                  # reference arm: passes over its bounded sample per step
PIPE_DEPTH = 3                   # asynchronous steps in flight (the library allows three)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--streams", type=int, default=256, help="receivers per GPU")
    ap.add_argument("--buffers", type=int, default=8, help="reference buffers per receiver per step")
    ap.add_argument("--ring", type=int, default=4, help="distinct steps of input kept resident (ring > L2)")
    ap.add_argument("--workload", choices=["config3_256streams", "config5_dense"], default="config3_256streams")
    ap.add_argument("--depth", type=int, default=0, help="asynchronous steps in flight (default PIPE_DEPTH; 1 = step by step, the order a profiler's kernel serialisation imposes anyway)")
    ap.add_argument("--launches-per-step", type=int, default=96, help="passes of the hot path over one batch that make up a step")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[1] latency leg, the configs[4] leg and the oracle comparison")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of their final launch (frames and buffer results) to DIR/*.npy")
    return ap.parse_args()


def bind_to_gpu_numa_node(local: int) -> str:
    """Best effort: run this process (and therefore allocate the pinned input slab) on the host NUMA node the GPU hangs off,
    so that the H2D copies of the e2e leg do not cross the socket interconnect.  Returns a note for the JSON line."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return "numa: single node"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        mine = cpus & os.sched_getaffinity(0)
        if not mine:
            return f"numa: GPU on node {node}, none of its CPUs usable here"
        os.sched_setaffinity(0, mine)
        return f"numa: bound to node {node} ({len(mine)} CPUs)"
    except Exception as e:
        return f"numa: not bound ({type(e).__name__})"


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


# ---------------------------------------------------------------------------------------------------------
# synthetic input
# ---------------------------------------------------------------------------------------------------------
def generate_streams(n_streams: int, samples_per_stream: int, seed0: int, workload: str, out: np.ndarray):
    """out: uint8 [n_streams, 2*samples_per_stream] (may be pinned). One distinct seeded stream per receiver."""
    from readsb_b200 import synth
    gen = synth.config5_stream if workload == "config5_dense" else synth.config2_stream
    synth.lib()

    def one(s):
        gen(seed0 + s, samples_per_stream, out=out[s])
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        list(ex.map(one, range(n_streams)))


# ---------------------------------------------------------------------------------------------------------
# reference CPU arm (oracle/_ref: the reference's own translation units, see oracle/Makefile)
# ---------------------------------------------------------------------------------------------------------
# Worker processes (fork, started before any CUDA call): readsb keeps its demodulator state in globals, so every
# receiver shard gets its own process with its own copy of the reference library, like one readsb per receiver.
_W = {}


def _worker_init(workload, n_buf):
    sys.path.insert(0, str(ROOT / "tests"))
    import oraclelib
    _W["kind"] = "reference" if oraclelib.have_ref() else "port"
    _W["ref"] = oraclelib.Reference() if _W["kind"] == "reference" else None
    _W["oraclelib"] = oraclelib
    _W["workload"], _W["n_buf"], _W["rows"] = workload, n_buf, {}


def _worker_run(task):
    """task = (seeds, passes): demodulate each seed's stream `passes` times; returns (samples, cpu seconds)."""
    from readsb_b200 import synth
    seeds, passes = task
    gen = synth.config5_stream if _W["workload"] == "config5_dense" else synth.config2_stream
    for sd in seeds:
        if sd not in _W["rows"]:
            _W["rows"][sd] = gen(sd, _W["n_buf"] * BUF)
    n = 0
    t0 = time.perf_counter()
    for _ in range(passes):
        for sd in seeds:
            row = _W["rows"][sd]
            if _W["ref"] is not None:
                _W["ref"].time_stream(row, BUF)          # convert_uc8_nodc + demodulate2400 per buffer (ifile loop)
            else:
                _W["oraclelib"].Oracle().run_stream(row, BUF)
            n += row.size // 2
    return n, time.perf_counter() - t0


class ReferencePool:
    def __init__(self, n_workers: int, workload: str, n_buf: int):
        import multiprocessing as mp
        self.n = n_workers
        self.pool = mp.get_context("fork").Pool(n_workers, initializer=_worker_init, initargs=(workload, n_buf))
        sys.path.insert(0, str(ROOT / "tests"))
        import oraclelib
        self.kind = "reference" if oraclelib.have_ref() else "port"

    def run(self, seeds, passes):
        """All seeds' streams, `passes` times, sharded over the workers; returns (samples, wall seconds)."""
        shards = [(seeds[w::self.n], passes) for w in range(self.n) if seeds[w::self.n]]
        t0 = time.perf_counter()
        res = self.pool.map(_worker_run, shards, chunksize=1)
        return sum(r[0] for r in res), time.perf_counter() - t0

    def close(self):
        self.pool.terminate()


def reference_arm(args, rank, world):
    if rank != 0:
        return 0
    cores = usable_cores()
    # bounded sample of the b200 arm's batch: the same seeded streams (rank 0's first receivers), one step = one pass
    n_streams = min(args.streams * args.gpus, max(cores, 64))
    seeds = [1 + s for s in range(n_streams)]
    pool = ReferencePool(cores, args.workload, args.buffers)
    # one step = REF_PASSES passes over the bounded sample (a single pass is ~20 ms: too short to time host cores fairly)
    pool.run(seeds, max(1, args.warmup) * REF_PASSES)            # generates the streams in the workers and warms up
    samples, dt = pool.run(seeds, args.steps * REF_PASSES)
    pool.close()
    value = samples / dt / 1e6
    line = {
        "impl": "reference", "metric": "iq_msamples_per_s_demodulated", "value": value, "unit": "Msamples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8->u16/int32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": cores, "kind": pool.kind,
                         "sample": f"{n_streams} of the {args.streams * args.gpus} streams x {args.buffers} buffers of {BUF} samples, {REF_PASSES} passes per step, "
                                   f"one receiver per process (the reference demodulator is single-threaded per receiver), {cores} processes"},
        "e2e": {"value": value, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------------
def workload_config(args, n_gpus):
    desc = ("BASELINE configs[2]/[3]: 256 concurrent synthetic 2.4 MSPS uc8 streams per GPU, DF17 injected at 100/s"
            if args.workload == "config3_256streams" else
            "BASELINE configs[4]: dense-preamble stress, 10k DF11+DF17/s per stream with overlaps, --fix on")
    return {"workload": desc, "streams_per_gpu": args.streams, "streams_total": args.streams * n_gpus,
            "buffers_per_stream_per_step": args.buffers, "buf_samples": BUF, "sample_rate_hz": 2400000,
            "samples_per_step_per_gpu": args.streams * args.buffers * BUF,
            "parallelism": f"{n_gpus} independent GPU(s), streams sharded {args.streams}/GPU, no collective",
            "pipelining": f"value: {args.depth or PIPE_DEPTH} steps in flight per GPU (run_device_uc8_async/wait); e2e: {args.depth or PIPE_DEPTH} steps in flight (run_host_uc8_async/wait: pinned host slab -> H2D on the library's copy stream, overlapping the previous steps' kernels); all results collected on the host inside the timed region",
            "l2": f"device inputs cycle through a ring of {args.ring} distinct steps "
                  f"({args.ring * args.streams * args.buffers * BUF * 2 / 2**20:.0f} MiB per GPU, L2 is 126 MB); each step reads bytes not touched for {args.ring - 1} steps"}


def usable_cores() -> int:
    """Host threads this process may really use: affinity mask and cgroup CPU quota, not the machine's core count."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


class NvmlClockSampler:
    """SM clock, board power and throttle reasons sampled through NVML every millisecond DURING a timed region:
    begin(True) ... end() brackets one region and returns its summary."""

    def __init__(self, gpu_index: int):
        self.idx, self.stop_flag, self.thread, self.max_mhz, self.nv = gpu_index, False, None, None, None
        self.active = False
        self._reset()

    def _reset(self):
        self.samples, self.power, self.reasons = [], [], set()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def _loop(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80}
        while not self.stop_flag:
            if not self.active:
                time.sleep(0.0005)
                continue
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.001)

    def begin(self, sample: bool):
        if sample:
            self._reset()
        self.active = bool(sample) and self.nv is not None

    def end(self) -> dict:
        was = self.active
        self.active = False
        if not was or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        time.sleep(0.002)       # let the sampling thread finish the reading it is in
        return {"sm_mhz": float(np.median(self.samples)), "sm_mhz_min": float(min(self.samples)), "sm_max_mhz": self.max_mhz,
                "power_w_median": float(np.median(self.power)) if self.power else None,
                "power_w_max": float(max(self.power)) if self.power else None,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=2)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.path = tempfile.NamedTemporaryFile(prefix="clocks_", suffix=".csv", delete=False).name
        self.proc = None
        self.idx = gpu_index

    def start(self):
        if shutil.which("nvidia-smi"):
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=self.fh, stderr=subprocess.DEVNULL)

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in open(self.path):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def _worker_time_buffers(task):
    """One reference core over the given seed's first `n_buf` buffers, `passes` times: seconds per buffer (convert + demodulate)."""
    from readsb_b200 import synth
    seed, n_buf, passes = task
    row = synth.config2_stream(seed, n_buf * BUF)
    best = None
    for _ in range(passes):
        t0 = time.perf_counter()
        if _W["ref"] is not None:
            _W["ref"].time_stream(row, BUF)
        else:
            _W["oraclelib"].Oracle().run_stream(row, BUF)
        dt = (time.perf_counter() - t0) / n_buf
        best = dt if best is None else min(best, dt)
    return best


def scan_source_digest() -> str:
    """What profiles/scan_traffic.json's DRAM bytes were measured on: the scan kernel's sources."""
    import hashlib
    h = hashlib.sha256()
    for name in ("scan_kernel.cu", "device_utils.cuh", "common.h"):
        h.update((ROOT / "readsb_b200" / "csrc" / name).read_bytes())
    return h.hexdigest()[:16]


def latency_leg(local, hbm_peak, cpu_pool):
    """BASELINE configs[1]: one receiver, one 65536-sample mag_buf per blocking submit -> run -> fetch (what the shim does for every
    demodulate2400() call, readsb.c:866-878), timed in C (tools/latency_probe.c) from pinned host memory."""
    import ctypes as C
    from readsb_b200 import synth
    from readsb_b200.build import build_probe
    from readsb_b200.demod import Demodulator, PinnedBuffer, uc8_lut, lib
    P = C.CDLL(str(build_probe()))
    L = lib()
    nbuf, reps, warm = 32, 400, 60
    iq = synth.config2_stream(7, nbuf * BUF)
    lut = uc8_lut()
    mag = lut[iq.view(np.uint16)]                                  # the converter's output (convert.c:64-108)
    row = BUF + 326
    pin = PinnedBuffer(nbuf * row * 2)
    m = pin.array.view(np.uint16).reshape(nbuf, row)
    for b in range(nbuf):                                          # mag_buf.data: 326 samples of the buffer before, then the new ones
        m[b, 326:] = mag[b * BUF:(b + 1) * BUF]
        m[b, :326] = mag[b * BUF - 326:b * BUF] if b else 0
    pin_iq = PinnedBuffer(nbuf * BUF * 2)
    pin_iq.array[:] = iq
    out = {"shape": "1 receiver, 1 buffer of 65536 samples per blocking call (submit -> run -> fetch), pinned host memory, timed in C"}

    def run(is_iq, ptr, stride, no_timing=True):
        # no_timing: the configuration integration/readsb_shim.c uses (no CUDA events between the kernels); the timed variant below
        # gives the device-side timeline and costs a few microseconds per call
        d = Demodulator(n_streams=1, buf_samples=BUF, max_buffers_per_run=1, device=local, no_timing=no_timing)
        us = (C.c_double * (reps + warm))()
        frames = C.c_uint64(0)
        fn = lambda name: C.cast(getattr(L, name), C.c_void_p)
        P.probe_latency.argtypes = [C.c_void_p] * 6 + [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p]
        rc = P.probe_latency(d.h, fn("b200_demod_submit_mag_u16"), fn("b200_demod_submit_iq_uc8"), fn("b200_demod_run"), fn("b200_demod_fetch"),
                             C.c_void_p(ptr), stride, BUF, nbuf, reps + warm, 1 if is_iq else 0, us, C.byref(frames))
        t = d.timing()
        launches = t["launches"]
        d.close()
        if rc != 0:
            return {"error": rc}
        v = np.sort(np.array(us[warm:]))
        return {"median_us": float(np.median(v)), "p99_us": float(v[int(0.99 * (len(v) - 1))]), "min_us": float(v[0]), "mean_us": float(v.mean()),
                "calls": reps, "frames": int(frames.value), "kernel_launches_per_call": launches,
                "device_timeline_of_last_call_us": None if no_timing else {"scan_kernel": t["scan_ms"] * 1e3, "stage_b": t["resolve_ms"] * 1e3,
                                                                           "scan_begin_to_stage_b_end": t["run_ms"] * 1e3}}
    out["mag_handoff"] = run(False, pin.ptr, row * 2)              # demodulate2400(mag_buf) call site
    out["iq_handoff"] = run(True, pin_iq.ptr, BUF * 2)             # converter call site: uc8 IQ in, magnitudes made on the GPU
    out["mag_handoff_with_cuda_events"] = run(False, pin.ptr, row * 2, no_timing=False)
    med = out["mag_handoff"].get("median_us")
    if med:
        out["msamples_per_s"] = BUF / med
        out["roofline_frac"] = ALG_BYTES_PER_SAMPLE * BUF / (med * 1e-6) / 1e9 / hbm_peak
    if cpu_pool is not None:
        try:
            sec = cpu_pool.pool.apply(_worker_time_buffers, ((7, nbuf, 5),))
            out["reference_one_core_us_per_buffer"] = sec * 1e6
            if med:
                out["speedup_vs_one_reference_core"] = sec * 1e6 / med
        except Exception as e:
            out["reference_one_core_us_per_buffer"] = repr(e)
    pin.free(); pin_iq.free()
    return out


def dense_leg(local, args, hbm_peak):
    """BASELINE configs[4]: 10k DF11+DF17 per second per stream with overlaps, device-resident, same batch shape as the main run."""
    import torch
    from readsb_b200 import synth
    from readsb_b200.demod import Demodulator
    S, B, R = args.streams, args.buffers, 2
    per_stream = R * B * BUF
    n_distinct = min(S, 32)
    base = np.empty((n_distinct, 2 * per_stream), dtype=np.uint8)
    generate_streams(n_distinct, per_stream, 5001, "config5_dense", base)
    pad = 4096
    dev = torch.empty(pad + S * 2 * per_stream + 256, dtype=torch.uint8, device="cuda")
    dev[:pad] = 0
    for s in range(S):                                             # 32 distinct captures, shifted copies for the other receivers
        row = torch.from_numpy(np.roll(base[s % n_distinct], 2 * 1013 * (s // n_distinct))).cuda()
        dev[pad + s * 2 * per_stream: pad + (s + 1) * 2 * per_stream] = row
    torch.cuda.synchronize()
    d = Demodulator(n_streams=S, buf_samples=BUF, max_buffers_per_run=B, device=local)
    stride = 2 * per_stream
    step_samples = S * B * BUF

    def go_async(k):
        d.run_device_async(dev.data_ptr() + pad + (k % R) * B * BUF * 2, stride, B, BUF, continues=(k % R) > 0, first_sample_timestamp=k * B * BUF * 5)
    n_launch, flying, frames = 60, 0, 0
    for phase in (0, 1):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        # (warm-up: long enough for the pipelined session to have measured its SM partition, ~70 steps - demod_api.cu tune_partition)
        for k in range(phase * 1000, phase * 1000 + (96 if phase == 0 else n_launch)):
            go_async(k); flying += 1
            if flying == PIPE_DEPTH:
                d.wait(); flying -= 1; frames += d.total_frames() if phase else 0
        while flying:
            d.wait(); flying -= 1; frames += d.total_frames() if phase else 0
        ev1.record(); torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    scan = 0.0
    for k in range(2000, 2020):
        d.run_device(dev.data_ptr() + pad + (k % R) * B * BUF * 2, stride, B, BUF, continues=(k % R) > 0, first_sample_timestamp=k * B * BUF * 5)
        scan += d.timing()["scan_ms"]
    d.close()
    del dev
    scan_s = scan / 20 * 1e-3
    return {"workload": "BASELINE configs[4]: dense-preamble stress, 10k DF11+DF17/s per stream with overlaps, --fix on; 256 receivers x 8 buffers per launch",
            "value": step_samples * n_launch / (ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms_per_launch": ms / n_launch, "launches_timed": n_launch,
            "frames_per_launch": frames / n_launch, "scan_kernel_ms_per_launch": scan_s * 1e3,
            "roofline_frac": ALG_BYTES_PER_SAMPLE * step_samples / scan_s / 1e9 / hbm_peak}


def parity_leg(local, args, host, dev_ptr, stride):
    """The timed configuration's first launch (all receivers, device-resident, fresh context) against the CPU oracle, frame for frame
    (outside every timed region; the oracle is the checker here, nothing more)."""
    sys.path.insert(0, str(ROOT / "tests"))
    from oraclelib import Oracle
    from paritylib import diff_frames
    from readsb_b200.demod import Demodulator
    S, B = args.streams, args.buffers
    d = Demodulator(n_streams=S, buf_samples=BUF, max_buffers_per_run=B, device=local)
    d.run_device(dev_ptr, stride, B, BUF, continues=False, first_sample_timestamp=0)
    got = [d.frames(s) for s in range(S)]
    d.close()

    def one(s):
        o = Oracle()
        fo, _ = o.run_stream(host[s, : 2 * B * BUF], BUF)
        return len(fo), diff_frames(got[s], fo)
    with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
        res = list(ex.map(one, range(S)))
    bad = [(s, r[1][:2]) for s, r in enumerate(res) if r[1]]
    return {"parity_checked": not bad, "receivers": S, "frames_compared": int(sum(r[0] for r in res)), "mismatching_receivers": len(bad),
            "first_problems": [f"receiver {s}: {p}" for s, p in bad[:3]]}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(d, out_dir: str, prefix: str = "") -> None:
    """What a caller of the timed path holds after its last launch: every receiver's frames (b200_demod_fetch) and buffer
    results (b200_demod_buffer_results), one float64 .npy per field (all values are integers below 2^53, or doubles, so
    the conversion is exact).  Frames of all receivers are concatenated in receiver order and `frame_receiver` says whose
    each one is.  Receivers are taken in order while the files stay within DUMP_LIMIT_BYTES; `receivers` lists them."""
    from readsb_b200.abi import BUFRES_DTYPE, FRAME_DTYPE
    frame_fields = [f for f in FRAME_DTYPE.names if not f.endswith("_")]
    bufres_fields = [f for f in BUFRES_DTYPE.names if not f.endswith("_")]
    per_frame = 8 * (1 + sum(int(np.prod(FRAME_DTYPE[f].shape)) for f in frame_fields))
    per_receiver = 8 * (1 + d.max_buffers_per_run * sum(int(np.prod(BUFRES_DTYPE[f].shape)) for f in bufres_fields))
    frames, bufres, total = [], [], 0
    for s in range(d.n_streams):
        f = d.frames(s)
        if total + per_receiver + per_frame * len(f) > DUMP_LIMIT_BYTES:
            break
        total += per_receiver + per_frame * len(f)
        frames.append(f)
        bufres.append(d.buffer_results(s))
    allf = np.concatenate(frames) if frames else np.zeros(0, FRAME_DTYPE)
    arrays = {"receivers": np.arange(len(frames)),
              "frame_receiver": np.repeat(np.arange(len(frames)), [len(f) for f in frames])}
    arrays.update({f"frame_{f}": allf[f] for f in frame_fields})
    b = np.stack(bufres) if bufres else np.zeros((0, d.max_buffers_per_run), BUFRES_DTYPE)     # [receiver, buffer]
    arrays.update({f"bufres_{f}": b[f] for f in bufres_fields})
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{prefix}{name}.npy", np.asarray(a, dtype=np.float64))


def b200_arm(args, rank, world, local):
    cpu_pool = None
    if not args.no_cpu and world == 1 and rank == 0:
        try:    # fork the CPU-baseline workers before this process creates a CUDA context
            cpu_pool = ReferencePool(usable_cores(), args.workload, args.buffers)
        except Exception:
            cpu_pool = None
    import torch
    from readsb_b200.demod import Demodulator, PinnedBuffer
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the demodulator has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    S, B, R, LPS = args.streams, args.buffers, args.ring, max(1, args.launches_per_step)
    launch_samples = S * B * BUF
    step_samples = launch_samples * LPS
    per_stream = R * B * BUF                       # samples of one receiver resident in the ring
    # --- inputs: pinned host slab [S, 2*per_stream] (for e2e) and a device copy (for value) -------------------
    numa_note = bind_to_gpu_numa_node(local)
    pin = PinnedBuffer(S * 2 * per_stream)
    host = pin.array.reshape(S, 2 * per_stream)
    generate_streams(S, per_stream, 1 + rank * S, args.workload, host)
    pad = 4096                                      # room in front of receiver 0 for the 326-sample halo
    dev = torch.empty(pad + S * 2 * per_stream + 256, dtype=torch.uint8, device="cuda")
    dev[pad: pad + S * 2 * per_stream] = torch.from_numpy(host.reshape(-1)).cuda()
    dev[:pad] = 0
    torch.cuda.synchronize()
    stride = 2 * per_stream

    d = Demodulator(n_streams=S, buf_samples=BUF, max_buffers_per_run=B, device=local)
    d.set_stream(torch.cuda.current_stream().cuda_stream)

    def device_step(k):
        slot = k % R
        d.run_device(dev.data_ptr() + pad + slot * B * BUF * 2, stride, B, BUF, continues=slot > 0,
                     first_sample_timestamp=k * B * BUF * 5)

    def device_step_async(k):
        slot = k % R
        d.run_device_async(dev.data_ptr() + pad + slot * B * BUF * 2, stride, B, BUF, continues=slot > 0,
                           first_sample_timestamp=k * B * BUF * 5)

    def host_step_async(k):
        # the reference-facing call with HOST buffers: the pinned slab of launch k goes up on the library's copy stream while
        # the kernels of launch k-1 run (reader thread / decode thread overlap of the reference, readsb.c:871)
        slot = k % R
        d.run_host_async(pin.ptr + slot * B * BUF * 2, stride, B, BUF, slot > 0, k * B * BUF * 5)

    depth = args.depth if args.depth > 0 else PIPE_DEPTH

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, launches, k0, pipelined=False, sample=False):
        """Times `launches` launches with CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
        pipelined: launches go through run_*_async/wait with PIPE_DEPTH in flight (the GPU never waits for the host between
        them); every launch's results are still collected on the host inside the timed region."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        acc = {"scan_ms": 0.0, "launches": 0, "frames": 0}

        def harvest():
            t = d.timing()
            acc["scan_ms"] += t["scan_ms"]; acc["launches"] += t["launches"]; acc["frames"] += d.total_frames()
        barrier()
        sampler.begin(sample)
        ev0.record()
        flying = 0
        for k in range(k0, k0 + launches):
            fn(k)
            if pipelined:
                flying += 1
                if flying == depth:
                    d.wait(); harvest(); flying -= 1
            else:
                harvest()
        while flying:
            d.wait(); harvest(); flying -= 1
        ev1.record()
        torch.cuda.synchronize()
        clk = sampler.end()
        ms = ev0.elapsed_time(ev1)
        if dist is not None:
            tmax = torch.tensor([ms], device="cuda")
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            ms = float(tmax.item())
        barrier()
        return ms, acc["scan_ms"], acc["launches"], acc["frames"], clk

    # --- value: inputs resident in HBM -------------------------------------------------------------------------
    sampler = NvmlClockSampler(local)          # SM clock / power / throttle reasons, recorded inside the timed regions only
    if rank == 0:
        sampler.start()
    # burst: a short region on a chip that has been idle (what round 1 reported as `value`)
    timed(device_step_async, 6, 0, pipelined=True)
    ms_b, _, _, _, clk_b = timed(device_step_async, 20, 6, pipelined=True, sample=True)
    burst = {"value": world * launch_samples * 20 / (ms_b * 1e-3) / 1e6, "unit": "Msamples/s", "launches": 20, "ms_per_launch": ms_b / 20, "clocks": clk_b}
    # sustained: W warm-up steps, then exactly K steps of LPS launches each
    timed(device_step_async, args.warmup * LPS, 26, pipelined=True)
    k_first = 26 + args.warmup * LPS
    ms, scan_ms, launches, frames, clocks = timed(device_step_async, args.steps * LPS, k_first, pipelined=True, sample=True)
    value = world * step_samples * args.steps / (ms * 1e-3) / 1e6
    if args.dump_outputs:
        dump_outputs(d, args.dump_outputs, f"rank{rank}_" if world > 1 else "")

    # --- e2e: host buffers through the C ABI ----------------------------------------------------------------------
    e2e = None
    scan_ms_alone = None
    if not args.no_e2e:
        # a fresh context so that receiver state (halo, ICAO filter) starts clean for the host path
        d2 = Demodulator(n_streams=S, buf_samples=BUF, max_buffers_per_run=B, device=local)
        d2.set_stream(torch.cuda.current_stream().cuda_stream)
        d_dev, d = d, d2
        timed(host_step_async, args.warmup * LPS, 0, pipelined=True)
        ms_e, _, launches_e, frames_e, clk_e = timed(host_step_async, args.steps * LPS, args.warmup * LPS, pipelined=True, sample=True)
        e2e = {"value": world * step_samples * args.steps / (ms_e * 1e-3) / 1e6, "unit": "Msamples/s",
               "h2d_bytes_per_step": (launch_samples * 2 + S * 64 + 64) * LPS,           # IQ slab + segment table + control block, per launch
               "d2h_bytes_per_step": int(frames_e / args.steps * 64) + (S * 4 + S * B * 144 + 32 + 16 * 64) * LPS,   # frames + counts + buffer results
               "ms_per_step": ms_e / args.steps, "frames_per_step": frames_e / args.steps, "host_placement": numa_note, "clocks": clk_e}
        if dist is not None:      # where every rank pinned its slab (the H2D copies of ranks on the far socket cross the interconnect)
            notes = [None] * world
            dist.all_gather_object(notes, f"rank {rank} gpu {local}: {numa_note}")
            e2e["host_placement"] = notes
        d = d_dev
        d2.close()
    # --- roofline leg: blocking device-resident launches, so that the scan kernel runs alone on the GPU ----------------
    n_alone = max(20, LPS)
    timed(device_step, 3, 0)
    _, scan_ms_alone, _, _, clk_r = timed(device_step, n_alone, 3, sample=True)

    extra = {}
    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    if rank == 0 and not args.no_extra:
        d.close()
        for name, fn in (("config2_single_stream", lambda: latency_leg(local, hbm_peak, cpu_pool)),
                         ("config5_dense", lambda: dense_leg(local, args, hbm_peak)),
                         ("parity", lambda: parity_leg(local, args, host, dev.data_ptr() + pad, stride))):
            try:
                extra[name] = fn()
            except Exception as e:      # an extra leg must never take the headline number down with it
                extra[name] = {"error": repr(e)}
    if rank == 0:
        sampler.stop()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0
    # the kernel's own duration: taken from the blocking launches where it runs alone; in the pipelined `value` loop it
    # shares the chip with the previous launch's stage B and its per-launch time is reported separately
    scan_avg_s = scan_ms_alone / n_alone * 1e-3
    achieved = ALG_BYTES_PER_SAMPLE * launch_samples / scan_avg_s / 1e9
    traffic, traffic_note = None, "no ncu capture committed for this source"
    tf = ROOT / "profiles" / "scan_traffic.json"      # per-launch DRAM bytes from the committed ncu capture of THIS source, else null
    if tf.exists():
        try:
            tj = json.loads(tf.read_text())
            if tj.get("source_digest") == scan_source_digest():
                traffic, traffic_note = tj.get("dram_bytes_per_launch"), tj.get("capture", "profiles/scan_traffic.json")
            else:
                traffic_note = "profiles/scan_traffic.json was captured on a different scan_kernel.cu (digest mismatch): not reported"
        except Exception:
            pass
    line = {
        "metric": "iq_msamples_per_s_demodulated", "value": value, "unit": "Msamples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8->u16/int32", "data": "synthetic",
        "config": workload_config(args, world),
        "frames_per_step_per_gpu": frames / args.steps,
        "timed_region_s": ms * 1e-3,
        "burst": burst,
        "roofline": {"bound": "hbm", "kernel": "scan_kernel", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                     "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_note,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                     "kernel_ms_per_launch": scan_avg_s * 1e3, "kernel_ms_per_launch_overlapped_with_stage_b": scan_ms / (args.steps * LPS),
                     "timed_in": f"{n_alone} blocking device-resident launches after the value run (kernel alone on the GPU), CUDA events around the launch on its stream",
                     "algorithmic_bytes_per_launch": ALG_BYTES_PER_SAMPLE * launch_samples, "clocks": clk_r},
        "gpu_launches": launches,
        "clocks": clocks,
    }
    if e2e:
        line["e2e"] = e2e
    if extra:
        line["extra"] = extra
        if "parity" in extra and "parity_checked" in extra["parity"]:
            line["parity_checked"] = extra["parity"]["parity_checked"]
    if cpu_pool is not None:
        # bounded CPU sample on this box's host cores, timed beside the GPU run: the same seeded streams
        try:
            cores = cpu_pool.n
            n_cpu_streams = min(S, max(cores, 64))
            seeds = [1 + s for s in range(n_cpu_streams)]
            cpu_pool.run(seeds, 1)
            passes = 4
            n, dt = cpu_pool.run(seeds, passes)
            while dt < 3.0 and passes < 256:
                passes *= 4
                n, dt = cpu_pool.run(seeds, passes)
            line["cpu_baseline"] = {"value": n / dt / 1e6, "unit": "Msamples/s", "cores": cores, "kind": cpu_pool.kind,
                                    "sample": f"{n_cpu_streams} of the {S} streams x {B} buffers of {BUF} samples, {passes} passes, one receiver per process"}
        except Exception as e:   # the CPU arm must never take the GPU number down with it
            line["cpu_baseline"] = {"value": None, "unit": "Msamples/s", "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(e)}
        cpu_pool.close()
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    args = parse_args()
    rank, world, local = dist_env()
    if world != args.gpus and world > 1:
        args.gpus = world
    if args.impl == "reference":
        return reference_arm(args, rank, world)
    return b200_arm(args, rank, world, local)


if __name__ == "__main__":
    sys.exit(main())
