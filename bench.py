#!/usr/bin/env python
"""bench.py — Window→FFT→Amplitude→Scale spectral chain, BASELINE.json configs[1]:
4096-pt × 65536-batch CF32 per GPU (weak scaling: every rank runs that workload on its own shard).

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, libb200dsp)
    python bench.py --impl reference --steps K --warmup W    # the reference's own CPU path (oracle/_ref)

A step = one pass of the fused chain over the whole [65536, 4096] CF32 batch = ONE kernel launch
(fft4096_kernel<MODE_AMP_RANGE, WIN_REAL>). `value` is device-timed (CUDA events, inputs resident in HBM,
2 GiB input + 1 GiB output per step >> 126 MB L2 so every step streams from HBM); `e2e` times
b200_chain_exec_host: the same batch from pinned HOST memory, H2D + kernel + D2H inside the timed region.
Prints ONE JSON line on rank 0.

`--steps` sets the number of timed steps of the headline and of every workload (the e2e variants time
min(--steps, --e2e-steps) host round trips, the wideband collective variants at most 5 steps). `--dump-outputs DIR`
writes what the timed path computed in its last step as DIR/<name>.npy (float32; outputs above 32 MB as a fixed, seeded
sample of rows, whose indices are written as DIR/<name>_rows.npy); the inputs are seeded, so two builds can be compared
output for output.

Besides the headline the same line carries (each measured after the headline's timed region, each guarded: a failure
is recorded as {"error": ...} and never touches the headline):
  e2e_variants   the e2e metric through the REFERENCE's own Flowgraph with provider b200 (shim/, full D2H and with the
                 lineplot + waterfall consumers = display-sized D2H), and from CI8 host samples
  workloads.fir       BASELINE configs[2]: 127-tap FIR + decimate-by-8, 2^26 CF32 samples
  workloads.fm        BASELINE configs[3]: Filter→FM→Filter→Amplitude at 10 MS/s (× real time)
  workloads.wideband  BASELINE configs[4]: [8,131072,4096] = 2^20 rows STRONG-scaled over the N ranks, timed without
                      and with the NCCL graph-boundary collective (full-result gather and display-sized reduction)
`--workload fir|fm|wideband` runs one of them alone (same JSON contract, metric = that workload's).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_FFT = 4096
ROWS = 65536
RANGE_MIN, RANGE_MAX = -120.0, 0.0
BYTES_PER_SAMPLE = 12          # 8 B CF32 in + 4 B F32 out (SURVEY.md §8d)
METRIC = "CF32 Msamples/sec Window->FFT->Amplitude->Scale"
UNIT = "Msamples/s"
WIDEBAND_ROWS = 8 * 131072     # BASELINE configs[4]


def workload_name(rows=ROWS):
    return f"spectral_chain {N_FFT}-pt x {rows}-batch CF32 (window->fft->amplitude->range[-120,0])"


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the UNMODIFIED reference CPU path (oracle/_ref), all host cores
# ------------------------------------------------------------------------------------------------

def _ref_worker(args):
    rows, cycles, warm, seed = args
    import numpy as np
    from oracle import ref
    rng = np.random.Generator(np.random.PCG64(seed))
    x = (0.01 * (rng.standard_normal((rows, N_FFT)) + 1j * rng.standard_normal((rows, N_FFT)))).astype(np.complex64)
    with ref.Session(log_level=0) as s:
        s.add_source("src", x, sample_axis=1, batch_axis=0)
        s.add_block("spec", "spectrum_engine", {"enableScale": True, "rangeMin": RANGE_MIN, "rangeMax": RANGE_MAX},
                    {"buffer": "src.signal"})
        for _ in range(max(1, warm)):       # cycle 1 also settles window/invert (static modules)
            s.compute()
        t0 = time.perf_counter()
        for _ in range(cycles):
            s.write_source("src", x)        # a fresh buffer every cycle, like a live source
            s.compute()
        dt = time.perf_counter() - t0
    return rows * N_FFT * cycles, dt


def _ref_fir_worker(args):
    """BASELINE configs[2] on the reference: the `filter` block at the size the block itself resamples (129 taps, R = 8;
    with 127 taps the reference bypasses decimation, block_impl.cc:64-90, and does 8x the output work)."""
    frames, t, cycles, seed = args
    import numpy as np
    from oracle import ref
    rng = np.random.Generator(np.random.PCG64(seed))
    x = (rng.standard_normal((frames, t)) + 1j * rng.standard_normal((frames, t))).astype(np.complex64)
    with ref.Session(log_level=0) as s:
        s.add_source("src", x, sample_axis=1, batch_axis=0)
        s.add_block("flt", "filter", {"sampleRate": 8e6, "bandwidth": 1e6, "taps": 129, "heads": 1}, {"signal": "src.signal"})
        s.compute()
        t0 = time.perf_counter()
        for _ in range(cycles):
            s.write_source("src", x)
            s.compute()
        dt = time.perf_counter() - t0
    return frames * t * cycles, dt


FM_F1 = {"sampleRate": 10e6, "bandwidth": 250e3, "taps": 161, "heads": 1, "center": [0.0]}
FM_F2 = {"sampleRate": 250e3, "bandwidth": 125e3, "taps": 41, "heads": 1}
FM_CFG = {"mode": "narrow", "deemphasis": "75us", "sampleRate": 250e3}
FM_FRAME = 4000                # 10 MS/s in frames of 4000 samples (multiple of the decimation 40)


def _ref_fm_worker(args):
    """BASELINE configs[3] on the reference: Filter(decimate 40) -> FM -> Filter(decimate 2) -> Amplitude; the reference's
    filter refuses an input that already has a channel axis, so the head axis is dropped between the stages
    (tests/test_gpu_flowgraphs.py does the same)."""
    frames, cycles, seed = args
    import numpy as np
    from oracle import ref
    rng = np.random.Generator(np.random.PCG64(seed))
    x = (rng.standard_normal((frames, FM_FRAME)) + 1j * rng.standard_normal((frames, FM_FRAME))).astype(np.complex64)
    with ref.Session(log_level=0) as s1, ref.Session(log_level=0) as s2:
        s1.add_source("src", x, sample_axis=1, batch_axis=0)
        s1.add_block("f1", "filter", FM_F1, {"signal": "src.signal"})
        s1.add_block("fm", "fm", FM_CFG, {"signal": "f1.buffer"})
        s1.compute()
        mid = np.ascontiguousarray(s1.output("fm", "signal")[:, 0, :])
        s2.add_source("src", mid, sample_axis=1, batch_axis=0)
        s2.add_block("f2", "filter", FM_F2, {"signal": "src.signal"})
        s2.add_block("amp", "amplitude", None, {"signal": "f2.buffer"})
        s2.compute()
        t0 = time.perf_counter()
        for _ in range(cycles):
            s1.write_source("src", x)
            s1.compute()
            s2.write_source("src", np.ascontiguousarray(s1.output("fm", "signal")[:, 0, :]))
            s2.compute()
        dt = time.perf_counter() - t0
    return frames * FM_FRAME * cycles, dt


def usable_cores() -> int:
    """Host threads this process may actually use: the affinity mask capped by the cgroup CPU quota
    (the GPU box exposes 128 logical CPUs but cpu.max grants 16)."""
    cores = len(os.sched_getaffinity(0))
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            cores = max(1, min(cores, int(float(quota) / float(period))))
    except Exception:
        pass
    return cores


def _pool_run(worker, jobs, cores):
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        t0 = time.perf_counter()
        results = pool.map(worker, jobs)
        wall = time.perf_counter() - t0
    return sum(r[0] for r in results), max(r[1] for r in results), wall


def run_reference_cpu(cycles: int, warm: int, rows_per_proc: int = 512, workload: str = "chain"):
    """Times the reference's own blocks (reference Flowgraph + scheduler_synchronous + NativeCpuRuntime) on every host
    core: one independent single-threaded reference process per core, each on its own shard (the reference compute
    path is single-threaded, SURVEY.md §8d)."""
    from oracle import ref
    if not ref.available():
        return None
    cores = usable_cores()
    if workload == "fir":
        frames, t = 64, 8192
        samples, slowest, wall = _pool_run(_ref_fir_worker, [(frames, t, cycles, 300 + i) for i in range(cores)], cores)
        what = (f"{cores} procs x {cycles} cycles x [{frames},{t}] CF32 through the reference filter block "
                f"(129 taps, its own decimate-by-8 plan: pad/fft/multiply/fold/ifft/overlap_add)")
    elif workload == "fm":
        frames = 250
        samples, slowest, wall = _pool_run(_ref_fm_worker, [(frames, cycles, 500 + i) for i in range(cores)], cores)
        what = (f"{cores} procs x {cycles} cycles x [{frames},{FM_FRAME}] CF32 through the reference "
                f"filter -> fm -> filter -> amplitude flowgraphs")
    else:
        samples, slowest, wall = _pool_run(_ref_worker, [(rows_per_proc, cycles, warm, 100 + i) for i in range(cores)], cores)
        what = (f"{cores} procs x {cycles} cycles x [{rows_per_proc},{N_FFT}] CF32 through the reference "
                f"spectrum_engine block (enableScale) on scheduler_synchronous")
    return {
        "value": samples / slowest / 1e6, "unit": UNIT, "cores": cores, "kind": "reference",
        "sample": f"{what}; slowest proc {slowest:.2f}s, pool wall {wall:.1f}s",
        "ms_per_cycle_per_core": slowest / cycles * 1e3,
    }


WORKLOAD_METRICS = {
    "chain": METRIC,
    "fir": "CF32 Msamples/sec 127-tap FIR + decimate-by-8",
    "fm": "CF32 Msamples/sec Filter->FM->Filter->Amplitude (10 MS/s flowgraph)",
    "wideband": "CF32 Msamples/sec 8-channel wideband spectral chain (2^20 x 4096, strong-scaled)",
}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cycles = max(1, args.steps)
    workload = args.workload if args.workload in ("fir", "fm") else "chain"
    base = run_reference_cpu(cycles, max(1, args.warmup), workload=workload)
    if base is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libjst_ref.so not built"}))
        return 0
    name = {"chain": workload_name(), "fir": "fir 129-tap decimate-by-8 (reference block plan)",
            "fm": "fm-broadcast flowgraph filter->fm->filter->amplitude"}[workload]
    line = {
        "impl": "reference", "metric": WORKLOAD_METRICS[workload], "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_cycle_per_core"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": name, "note": "reference CPU path on a bounded sample per step",
                   "range": [RANGE_MIN, RANGE_MAX]},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# clocks sampling (NVML) during the timed region
# ------------------------------------------------------------------------------------------------

class ClockSampler(threading.Thread):
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int, period: float = 0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples = []      # (t, sm_mhz, reasons_mask, power_w)
        self.stop_flag = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as exc:   # pragma: no cover
            self.error = repr(exc)

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                power = nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                self.samples.append((time.perf_counter(), mhz, mask, power))
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self, t0: float, t1: float):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable"}
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        note = "sampled inside the timed region"
        if not inside:
            inside = self.samples
            note = "timed region shorter than the sampling period; samples from warm-up + timed + e2e"
        import statistics
        mask = 0
        for s in inside:
            mask |= s[2]
        reasons = [name for bit, name in self.REASONS.items() if mask & bit and name != "gpu_idle"]
        return {"sm_mhz": statistics.median(s[1] for s in inside) if inside else None,
                "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(inside),
                "power_w_max": max((s[3] for s in inside), default=None), "note": note}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------

def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic_per_launch(key="fft4096_kernel<MODE_AMP_RANGE,WIN_REAL>"):
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get(key)
    except Exception:
        return None


def bind_to_gpu_numa_node(local: int):
    """Pins this rank's threads (and therefore its first-touch pinned host buffers) to the NUMA node its GPU hangs off:
    the e2e path moves ~77 GB/s of host memory traffic per GPU, and 4-8 ranks sharing one socket's DRAM is what limited
    the round-1 e2e scaling (0.64 at N >= 4). Returns a description for the JSON line."""
    try:
        import torch
        props = torch.cuda.get_device_properties(local)
        bus = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return {"numa_node": None, "note": "GPU reports no NUMA affinity"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return {"numa_node": node, "note": "no allowed CPU on the GPU's node; affinity unchanged"}
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed), "pci": bus}
    except Exception as exc:
        return {"numa_node": None, "note": f"binding skipped: {exc!r}"}


class Env:
    """Device, stream, library and the small helpers every workload shares."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        from cyberether_b200 import _native
        from cyberether_b200.jetstream import Context
        self.torch, self.dist, self.native = torch, dist, _native
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback")
        torch.cuda.set_device(self.local)
        self.numa = bind_to_gpu_numa_node(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            import datetime
            # a rank that fails inside a guarded extra must cost the others two minutes, not NCCL's default ten
            dist.init_process_group("nccl", device_id=self.dev, timeout=datetime.timedelta(seconds=120))
        self.lib = _native.load()          # raises if libb200dsp.so is missing
        self.ctx = Context.get(self.dev)
        self.stream = torch.cuda.current_stream(self.dev)
        self.sp = ctypes.c_void_p(self.stream.cuda_stream)
        self.peak, self.peak_src = measured_peak_gbs()
        self.launches = 0

    def check(self, rc):
        self.native.check(rc)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, value):
        from cyberether_b200.sharding import max_over_ranks
        return max_over_ranks(value, self.dev)

    def timed(self, fn, steps, warmup):
        """W warm-up calls, barrier + synchronize, K calls between two CUDA events on the launching stream, synchronize +
        barrier; returns (this rank's ms per step, max-over-ranks ms per step, t_begin, t_end)."""
        torch = self.torch
        for _ in range(max(3, warmup)):
            fn()
        self.barrier()
        torch.cuda.synchronize(self.dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_begin = time.perf_counter()
        e0.record(self.stream)
        for _ in range(steps):
            fn()
        e1.record(self.stream)
        torch.cuda.synchronize(self.dev)
        t_end = time.perf_counter()
        self.barrier()
        ms = e0.elapsed_time(e1) / steps
        return ms, self.max_over_ranks(ms), t_begin, t_end

    def synthetic_rows(self, rows, first_row=0, seed=0):
        """CF32 [rows, 4096] resident in HBM: per row three tones + Gaussian noise (cf. SURVEY.md §8d), in slabs so the
        generator never holds more than ~1 GiB of temporaries."""
        torch = self.torch
        import numpy as np
        n = N_FFT
        x = torch.empty(rows, n, dtype=torch.complex64, device=self.dev)
        g = torch.Generator(device=self.dev)
        g.manual_seed(0x5EED0000 + seed)
        t = torch.arange(n, device=self.dev, dtype=torch.float32)
        slab = 16384
        for r0 in range(0, rows, slab):
            r1 = min(rows, r0 + slab)
            b = torch.arange(r0, r1, device=self.dev, dtype=torch.int64) + first_row
            part = torch.view_as_complex(torch.randn(r1 - r0, n, 2, device=self.dev, generator=g) * 1e-3)
            for mult, add, amp in ((97, 0, 0.5), (1013, 511, 0.05), (0, n // 2, 0.005)):
                k = ((b * mult + add) % n).to(torch.float32)[:, None]
                part += amp * torch.polar(torch.ones(1, device=self.dev), 2 * np.pi * k * t[None, :] / n)
            x[r0:r1] = part
        return x

    def chain_plan(self, rows):
        torch, lib = self.torch, self.lib
        n = N_FFT
        win = torch.empty(n, dtype=torch.complex64, device=self.dev)
        winv = torch.empty(n, dtype=torch.complex64, device=self.dev)
        self.check(lib.b200_window_blackman_cf32(self.ctx.handle, win.data_ptr(), n, self.sp))
        self.check(lib.b200_invert_cf32(self.ctx.handle, win.data_ptr(), winv.data_ptr(), 1, n, 1, self.sp))
        torch.cuda.synchronize(self.dev)
        plan = ctypes.c_void_p()
        self.check(lib.b200_chain_plan_create(self.ctx.handle, n, rows, winv.data_ptr(), ctypes.byref(plan)))
        return plan


DUMP_BYTES = 32 << 20         # per output array; larger outputs are written as a seeded sample of rows


def dump_output(env, directory, name, tensor):
    """Writes `tensor` (what a caller of the timed path receives) as float32 `directory/<name>.npy`; complex values as
    trailing (re, im) pairs. Beyond DUMP_BYTES a fixed, seeded sample of rows (axis 0) is written, with its row indices
    in `<name>_rows.npy` (float64)."""
    import numpy as np
    if not directory:
        return
    torch = env.torch
    t = torch.view_as_real(tensor) if tensor.is_complex() else tensor
    if env.world > 1:
        name = f"{name}_rank{env.rank}"
    os.makedirs(directory, exist_ok=True)
    row_bytes = max(1, t[0].numel() * 4)
    if t.numel() * 4 > DUMP_BYTES:
        keep = min(t.shape[0], max(1, DUMP_BYTES // row_bytes))
        rows = np.sort(np.random.default_rng(0).choice(t.shape[0], size=keep, replace=False))
        np.save(os.path.join(directory, f"{name}_rows.npy"), rows.astype(np.float64))
        t = t[torch.from_numpy(rows).to(t.device)]
    np.save(os.path.join(directory, f"{name}.npy"), t.float().cpu().numpy())


def guarded(fn, *a, **kw):
    try:
        return fn(*a, **kw)
    except BaseException as exc:      # noqa: BLE001 — an extra must never take the headline down
        if isinstance(exc, KeyboardInterrupt):
            raise
        return {"error": f"{type(exc).__name__}: {exc}"[:400]}


# ---- e2e variants ---------------------------------------------------------------------------------

def finish_e2e(env, result):
    """The ONE collective of an e2e variant, outside its guarded body: MAX over ranks of the local wall time, and a
    failure on any rank fails the variant for everyone (ranks never wait on each other inside the guarded part, so a
    rank that raised cannot hang the rest)."""
    failed = not isinstance(result, dict) or "local_seconds" not in result
    seconds = -1.0 if failed else float(result["local_seconds"])
    if env.world > 1:
        t = env.torch.tensor([seconds, 1.0 if failed else 0.0], dtype=env.torch.float64, device=env.dev)
        env.dist.all_reduce(t, op=env.dist.ReduceOp.MAX)
        seconds, any_failed = float(t[0]), bool(t[1] > 0)
    else:
        any_failed = failed
    if failed:
        return result if isinstance(result, dict) else {"error": "no result"}
    if any_failed:
        return {"error": "the variant failed on another rank"}
    out = {k: v for k, v in result.items() if k not in ("local_seconds", "samples_all_ranks")}
    out["value"] = result["samples_all_ranks"] / seconds / 1e6
    return out


def e2e_shim(env, rows, x_host, steps, consumers):
    """The e2e metric through the REFERENCE's own Flowgraph (scheduler_synchronous + NativeCudaRuntime) with every
    block on provider b200: host bytes -> source tensor (H2D), Flowgraph::compute(), result back to the host (D2H).
    consumers = False: spectrum_engine, the whole [rows, 4096] F32 result is read back;
    consumers = True : spectrum_engine -> lineplot + waterfall (the spectrum-analyzer flowgraph); only signalPoints
    [4096, 2] and the ring [512, 4096] are read back (the chain's fused column sums feed the lineplot)."""
    from shim import binding as sb
    if not sb.available():
        return {"unavailable": "shim/_build/libjst_b200.so not built"}
    n = N_FFT
    torch = env.torch
    sb.set_cuda_device(env.local)
    with sb.Session(log_level=0) as s:
        s.add_source("src", (rows, n), "CF32", target=sb.B200, sampleAxis=1, batchAxis=0)
        s.add_block("spec", "spectrum_engine", {"enableScale": True, "rangeMin": RANGE_MIN, "rangeMax": RANGE_MAX},
                    {"buffer": "src.signal"}, target=sb.B200)
        d2h = rows * n * 4
        if consumers:
            s.add_block("lp", "lineplot", {"averaging": 4}, {"signal": "spec.buffer"}, target=sb.B200)
            s.add_block("wf", "waterfall", {"height": 512}, {"signal": "spec.buffer"}, target=sb.B200)
            d2h = n * 2 * 4 + 512 * n * 4
        out_host = torch.empty(rows, n, dtype=torch.float32, pin_memory=True) if not consumers else None

        def step():
            s.write_source_ptr("src", x_host.data_ptr(), rows * n * 8)
            s.compute()
            if consumers:
                return float(sb.viz_read("lp-lineplot")[1::2].sum()) + float(sb.viz_read("wf-waterfall")[:n].sum())
            s.read_into("spec", "buffer", out_host.data_ptr(), rows * n * 4)
            return 0.0
        step()                    # first cycle: static modules settle, plans are created
        t0 = time.perf_counter()
        check = 0.0
        for _ in range(steps):
            check = step()
        dt = time.perf_counter() - t0          # this rank's; no collective inside a guarded extra (finish_e2e reduces)
        modules = {**s.modules("spec"), **(s.modules("lp") if consumers else {}), **(s.modules("wf") if consumers else {})}
        kernel_ms = {k.split(":", 1)[1]: round(v[1] / max(1, v[0]), 4) for k, v in modules.items() if v[0] > 1}
    return {"local_seconds": dt, "samples_all_ranks": rows * n * env.world * steps, "unit": UNIT, "steps": steps,
            "h2d_bytes_per_step": rows * n * 8, "d2h_bytes_per_step": d2h,
            "api": "reference Flowgraph::compute() with provider b200 (shim/libjst_b200.so): source write (H2D) -> "
                   + ("spectrum_engine -> lineplot + waterfall -> signalPoints + ring read (D2H)" if consumers
                      else "spectrum_engine -> full result read (D2H)"),
            "module_ms_per_cycle": kernel_ms, "checksum": check}


def e2e_ci8(env, plan, rows, coeff, scale, offset, steps):
    """e2e from an SDR's native CI8 samples: 2 B/sample over PCIe instead of 8 (b200_chain_exec_host_typed)."""
    torch = env.torch
    n = N_FFT
    x_host = torch.empty(rows, n, 2, dtype=torch.int8, pin_memory=True)
    x_host.random_(-100, 100)
    out_host = torch.empty(rows, n, dtype=torch.float32, pin_memory=True)

    def step():
        env.check(env.lib.b200_chain_exec_host_typed(plan, x_host.data_ptr(), 8, out_host.data_ptr(), rows, coeff, 1,
                                                     scale, offset, 0))
    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return {"local_seconds": dt, "samples_all_ranks": rows * n * env.world * steps, "unit": UNIT, "steps": steps,
            "h2d_bytes_per_step": rows * n * 2, "d2h_bytes_per_step": rows * n * 4,
            "api": "b200_chain_exec_host_typed(CI8): cast fused into the kernel's load",
            "checksum": float(out_host[:: max(1, rows // 64)].double().sum())}


# ---- BASELINE configs[2]: FIR ----------------------------------------------------------------------

def bench_fir(env, steps, warmup, with_cpu=False, dump=None):
    """127-tap FIR + decimate-by-8 over 2^26 CF32 samples ([8192, 8192] frames, one stream): b200_fir_exec.
    Algorithmic bytes 8 + 8/R = 9 per input sample. L2: 512 MiB in + 64 MiB out per step >> 126 MB."""
    import numpy as np
    torch, lib = env.torch, env.lib
    frames, t, taps, r = 8192, 8192, 127, 8
    g = torch.Generator(device=env.dev)
    g.manual_seed(77 + env.rank)
    x = torch.view_as_complex(torch.randn(frames, t, 2, device=env.dev, generator=g)).contiguous()
    y = torch.empty(frames, 1, t // r, dtype=torch.complex64, device=env.dev)
    host_taps = np.zeros((1, taps), np.complex64)
    center = (ctypes.c_double * 1)(0.0)
    env.check(lib.b200_filter_taps_host(8e6, 1e6, center, 1, taps, host_taps.ctypes.data_as(ctypes.c_void_p)))
    plan = ctypes.c_void_p()
    env.check(lib.b200_fir_plan_create(env.ctx.handle, host_taps.ctypes.data_as(ctypes.c_void_p), taps, 1, r,
                                       ctypes.byref(plan)))

    def step():
        env.check(lib.b200_fir_exec(plan, x.data_ptr(), y.data_ptr(), frames, t, env.sp))
    ms, ms_max, t0, t1 = env.timed(step, steps, warmup)
    dump_output(env, dump, "fir_out", y)
    samples = frames * t
    # e2e: pinned host frames -> device -> decimated result back, through the C ABI's own copies
    x_host = torch.empty(frames, t, dtype=torch.complex64, pin_memory=True)
    x_host.copy_(x)
    y_host = torch.empty(frames, 1, t // r, dtype=torch.complex64, pin_memory=True)

    def e2e_step():
        env.check(lib.b200_memcpy(env.ctx.handle, x.data_ptr(), x_host.data_ptr(), samples * 8, 0, env.sp))
        step()
        env.check(lib.b200_memcpy(env.ctx.handle, y_host.data_ptr(), y.data_ptr(), samples // r * 8, 1, env.sp))
        env.check(lib.b200_stream_synchronize(env.ctx.handle, env.sp))
    e2e_step()
    e2e_n = 3
    tw = time.perf_counter()
    for _ in range(e2e_n):
        e2e_step()
    e2e_dt = env.max_over_ranks(time.perf_counter() - tw)
    env.check(lib.b200_fir_plan_destroy(plan))
    achieved = samples * 9 / (ms * 1e-3) / 1e9
    out = {"metric": WORKLOAD_METRICS["fir"], "value": samples * env.world / (ms_max * 1e-3) / 1e6, "unit": UNIT,
           "ms_per_step": ms_max, "steps": steps, "gpu_launches": steps,
           "config": {"workload": "fir 127-tap + decimate-by-8, 2^26 CF32 samples as [8192, 8192] frames",
                      "l2": "inputs larger than L2 (512 MiB in + 64 MiB out per step)"},
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": env.peak, "unit": "GB/s", "frac": achieved / env.peak,
                        "traffic": ncu_traffic_per_launch("fir_decim_kernel<127,R=8>"), "kernel": "fir_decim_kernel",
                        "algorithmic_bytes_per_launch": samples * 9, "kernel_ms": ms, "peak_source": env.peak_src},
           "e2e": {"value": samples * env.world * e2e_n / e2e_dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": samples * 8,
                   "d2h_bytes_per_step": samples, "api": "b200_memcpy(h2d) + b200_fir_exec + b200_memcpy(d2h) + sync"}}
    if with_cpu and env.rank == 0:
        out["cpu_baseline"] = guarded(run_reference_cpu, 4, 1, workload="fir")
    return out


# ---- the reference's own fft module benchmark cases (src/domains/dsp/fft/module_benchmarks.cc:7-50) ----------------------

def bench_fft(env, steps, warmup):
    """CF32-8192, CF32-65536 (C2C) and F32-8192, F32-65536 (real input, `complexOutput`) as batches of 2^26 samples, plus the
    fused spectral chain at n = 65536: b200_fft_exec / b200_fft_exec_real / b200_chain_exec, device-resident. Algorithmic
    bytes: 16 per complex sample (C2C), 8 per real sample (R2C: 4 in + 4 out), 12 per sample (chain)."""
    torch, lib = env.torch, env.lib
    total = 1 << 26
    g = torch.Generator(device=env.dev)
    g.manual_seed(55 + env.rank)
    x = torch.view_as_complex(torch.randn(total, 2, device=env.dev, generator=g)).contiguous()
    y = torch.empty_like(x)
    xr = torch.view_as_real(x).reshape(-1)
    cases, launches = {}, 0

    def record(name, ms, samples, bytes_per_sample, kernel):
        achieved = samples * bytes_per_sample / (ms * 1e-3) / 1e9
        cases[name] = {"value": samples * env.world / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms,
                       "roofline": {"bound": "hbm", "achieved": achieved, "peak": env.peak, "unit": "GB/s",
                                    "frac": achieved / env.peak, "algorithmic_bytes_per_launch": samples * bytes_per_sample,
                                    "kernel": kernel}}
    for n, kernel in ((8192, "fft_radix_kernel<13>"), (65536, "fft_cols_kernel<8> + fft_rows256_kernel (tiled two-pass, L2-resident scratch)")):
        rows = total // n
        plan = ctypes.c_void_p()
        env.check(lib.b200_fft_plan_c2c(env.ctx.handle, n, rows, ctypes.byref(plan)))
        ms, ms_max, _, _ = env.timed(lambda: env.check(lib.b200_fft_exec(plan, x.data_ptr(), y.data_ptr(), 1, env.sp)), steps, warmup)
        record(f"CF32-{n}", ms_max, total, 16, kernel)
        env.check(lib.b200_fft_plan_destroy(plan))
        launches += steps
        rrows = xr.numel() // n
        half = ctypes.c_void_p()
        env.check(lib.b200_fft_plan_c2c(env.ctx.handle, n // 2, rrows, ctypes.byref(half)))
        out = torch.empty(rrows, n // 2 + 1, dtype=torch.complex64, device=env.dev)
        ms, ms_max, _, _ = env.timed(lambda: env.check(lib.b200_fft_exec_real(half, xr.data_ptr(), out.data_ptr(), 0, env.sp)), steps, warmup)
        record(f"F32-{n}", ms_max, xr.numel(), 8, "fft_radix_kernel<MODE_R2C> (transform + unpack in one kernel)" if n // 2 <= 8192
               else "half-length tiled c2c + rfft_unpack_kernel")
        env.check(lib.b200_fft_plan_destroy(half))
        del out
        launches += 2 * steps
    n = 65536
    rows = total // n
    win = torch.zeros(n, dtype=torch.complex64, device=env.dev)
    win.real = torch.rand(n, device=env.dev, generator=g)
    torch.cuda.synchronize()
    cplan = ctypes.c_void_p()
    env.check(lib.b200_chain_plan_create(env.ctx.handle, n, rows, win.data_ptr(), ctypes.byref(cplan)))
    f = torch.empty(rows, n, dtype=torch.float32, device=env.dev)
    coeff = float(20.0 * math.log10(1.0 / n))
    ms, ms_max, _, _ = env.timed(lambda: env.check(lib.b200_chain_exec(cplan, x.data_ptr(), f.data_ptr(), rows, ctypes.c_float(coeff), 1,
                                                                      ctypes.c_float(1.0 / 120.0), ctypes.c_float(1.0), env.sp)), steps, warmup)
    record("chain-65536", ms_max, total, 12, "fft_cols_kernel<8, window> + fft_rows256_kernel<amplitude, range>")
    env.check(lib.b200_chain_plan_destroy(cplan))
    launches += 2 * steps
    return {"metric": "CF32 / F32 Msamples/sec through the fft module (the reference's module_benchmarks cases) and the fused chain at n = 65536",
            "unit": UNIT, "steps": steps, "gpu_launches": launches, "cases": cases,
            "config": {"workload": "2^26 samples per step as [2^26 / n, n] batches", "l2": "inputs larger than L2 (512 MiB per step)"}}


# ---- BASELINE configs[3]: FM-broadcast flowgraph at 10 MS/s ---------------------------------------------

def bench_fm(env, steps, warmup, with_cpu=False, dump=None):
    """Filter(161 taps, decimate 40) -> FM(narrow, 75 us) -> Filter(41 taps, decimate 2) -> Amplitude on one second of
    10 MS/s IQ ([2500, 4000] frames), module kernels back to back on one stream through the C ABI."""
    import numpy as np
    torch, lib = env.torch, env.lib
    frames = 2500
    samples = frames * FM_FRAME
    g = torch.Generator(device=env.dev)
    g.manual_seed(99 + env.rank)
    tt = torch.arange(samples, device=env.dev, dtype=torch.float64) / 10e6
    phase = 2 * np.pi * 250e3 * tt + 75.0 * torch.sin(2 * np.pi * 1e3 * tt)
    x = (torch.polar(torch.ones_like(phase), phase).to(torch.complex64)
         + 0.05 * torch.view_as_complex(torch.randn(samples, 2, device=env.dev, generator=g))).reshape(frames, FM_FRAME).contiguous()

    def taps_for(cfg):
        host = np.zeros((1, cfg["taps"]), np.complex64)
        center = (ctypes.c_double * 1)(0.0)
        env.check(lib.b200_filter_taps_host(cfg["sampleRate"], cfg["bandwidth"], center, 1, cfg["taps"],
                                            host.ctypes.data_as(ctypes.c_void_p)))
        return host
    h1, h2 = taps_for(FM_F1), taps_for(FM_F2)
    p1, p2, pfm = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
    env.check(lib.b200_fir_plan_create(env.ctx.handle, h1.ctypes.data_as(ctypes.c_void_p), 161, 1, 40, ctypes.byref(p1)))
    env.check(lib.b200_fir_plan_create(env.ctx.handle, h2.ctypes.data_as(ctypes.c_void_p), 41, 1, 2, ctypes.byref(p2)))
    env.check(lib.b200_fm_plan_create(env.ctx.handle, 1, ctypes.c_float(250e3), 0, 75, ctypes.byref(pfm)))
    t1, t2 = FM_FRAME // 40, FM_FRAME // 80
    y1 = torch.empty(frames, 1, t1, dtype=torch.complex64, device=env.dev)
    audio = torch.empty(frames, 1, t1, dtype=torch.float32, device=env.dev)
    audio_c = torch.empty(frames, t1, dtype=torch.complex64, device=env.dev)
    y2 = torch.empty(frames, 1, t2, dtype=torch.complex64, device=env.dev)
    db = torch.empty(frames, 1, t2, dtype=torch.float32, device=env.dev)
    coeff = ctypes.c_float()
    env.check(lib.b200_amplitude_scaling_coeff(t2, ctypes.byref(coeff)))

    def step():
        env.check(lib.b200_fir_exec(p1, x.data_ptr(), y1.data_ptr(), frames, FM_FRAME, env.sp))
        env.check(lib.b200_fm_exec(pfm, y1.data_ptr(), audio.data_ptr(), frames, t1, env.sp))
        env.check(lib.b200_cast_f32_cf32(env.ctx.handle, audio.data_ptr(), audio_c.data_ptr(), frames * t1, env.sp))
        env.check(lib.b200_fir_exec(p2, audio_c.data_ptr(), y2.data_ptr(), frames, t1, env.sp))
        env.check(lib.b200_amplitude_cf32(env.ctx.handle, y2.data_ptr(), db.data_ptr(), frames * t2, coeff, env.sp))
    ms, ms_max, _, _ = env.timed(step, steps, warmup)
    dump_output(env, dump, "fm_out", db)
    for plan, destroy in ((p1, lib.b200_fir_plan_destroy), (p2, lib.b200_fir_plan_destroy), (pfm, lib.b200_fm_plan_destroy)):
        env.check(destroy(plan))
    value = samples * env.world / (ms_max * 1e-3) / 1e6
    algorithmic = samples * 8 + frames * t1 * (8 + 8 + 4 + 4 + 8 + 8) + frames * t2 * (8 + 8 + 4)
    achieved = algorithmic / (ms * 1e-3) / 1e9
    out = {"metric": WORKLOAD_METRICS["fm"], "value": value, "unit": UNIT, "ms_per_step": ms_max, "steps": steps,
           "gpu_launches": steps * 5, "times_real_time": value * 1e6 / 10e6 / env.world,
           "config": {"workload": "fm-broadcast flowgraph: filter(161 taps, /40) -> fm(narrow, 75us) -> filter(41 taps, /2) "
                                  "-> amplitude, 1 s of 10 MS/s IQ as [2500, 4000] frames",
                      "l2": "80 MB in per step: L2-resident after the first step (126 MB L2) — the flowgraph is "
                            "launch / latency bound, not bandwidth bound"},
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": env.peak, "unit": "GB/s", "frac": achieved / env.peak,
                        "traffic": None, "kernel": "fir_decim_kernel (stage 1 dominates the bytes)",
                        "algorithmic_bytes_per_launch": algorithmic, "kernel_ms": ms, "peak_source": env.peak_src}}
    if with_cpu and env.rank == 0:
        out["cpu_baseline"] = guarded(run_reference_cpu, 4, 1, workload="fm")
    return out


# ---- BASELINE configs[4]: 8-channel wideband chain, strong-scaled with the NCCL boundary collective ---------

def bench_wideband(env, steps, warmup, dump=None):
    """[8, 131072, 4096] CF32 = 2^20 rows, cut into `world` contiguous slabs (one channel per GPU at N = 8). Timed:
    (a) kernel only (every rank its slab, no collective); (b) kernel + gather of the FULL F32 result on rank 0 over NCCL
    (dist.gather, 2^20 x 4096 x 4 B = 16 GiB in total); (c) kernel with fused column sums + the DISPLAY-sized boundary:
    reduce of the [4096] column sums (lineplot) + the newest 512 rows from the last rank (waterfall)."""
    torch, dist, lib = env.torch, env.dist, env.lib
    from cyberether_b200 import amplitude_scaling_coeff, range_coefficients
    from cyberether_b200.sharding import shard_bounds
    n, world, rank = N_FFT, env.world, env.rank
    begin, end = shard_bounds(WIDEBAND_ROWS, world, rank)
    rows = end - begin
    # Local set-up first, then ONE agreement collective: a rank that cannot allocate must not leave the others waiting
    # inside the timed collectives below.
    x = out = colsum = plan = parts = None
    problem = None
    try:
        x = env.synthetic_rows(rows, first_row=begin, seed=1000 + rank)
        out = torch.empty(rows, n, dtype=torch.float32, device=env.dev)
        colsum = torch.zeros(n, dtype=torch.float32, device=env.dev)
        plan = env.chain_plan(rows)
        if world > 1 and rank == 0:
            parts = [torch.empty(rows, n, dtype=torch.float32, device=env.dev) for _ in range(world)]
        torch.cuda.synchronize(env.dev)
    except BaseException as exc:      # noqa: BLE001
        problem = f"{type(exc).__name__}: {exc}"[:300]
    if world > 1:
        flag = torch.tensor([1.0 if problem else 0.0], dtype=torch.float64, device=env.dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if float(flag[0]) > 0:
            problem = problem or "set-up failed on another rank"
    if problem:
        del x, out, parts
        torch.cuda.empty_cache()
        return {"error": problem}
    coeff = amplitude_scaling_coeff(n)
    scale, offset = range_coefficients(RANGE_MIN, RANGE_MAX)

    def kernel():
        env.check(lib.b200_chain_exec(plan, x.data_ptr(), out.data_ptr(), rows, coeff, 1, scale, offset, env.sp))
    ms_k, ms_k_max, _, _ = env.timed(kernel, steps, warmup)
    dump_output(env, dump, "wideband_out", out)

    result = {"rows_total": WIDEBAND_ROWS, "rows_per_rank": rows, "scaling": "strong",
              "kernel_only": {"ms_per_step": ms_k_max, "value": WIDEBAND_ROWS * n / (ms_k_max * 1e-3) / 1e6, "unit": UNIT}}
    gather_bytes = (WIDEBAND_ROWS - rows) * n * 4 if world > 1 else 0
    same_size = WIDEBAND_ROWS % world == 0

    def kernel_gather():
        kernel()
        if world > 1 and same_size:
            dist.gather(out, parts, dst=0)
    g_steps = max(2, min(steps, 5))
    ms_g, ms_g_max, _, _ = env.timed(kernel_gather, g_steps, 1)
    nvlink = gather_bytes / max(1e-9, (ms_g_max - ms_k_max) * 1e-3) / 1e9 if world > 1 else None
    result["with_full_gather"] = {"ms_per_step": ms_g_max, "value": WIDEBAND_ROWS * n / (ms_g_max * 1e-3) / 1e6,
                                  "unit": UNIT, "steps": g_steps}
    del parts
    tail = torch.empty(512, n, dtype=torch.float32, device=env.dev)

    def kernel_display():
        env.check(lib.b200_chain_exec_colsum(plan, x.data_ptr(), 1, out.data_ptr(), rows, coeff, 1, scale, offset,
                                             colsum.data_ptr(), env.sp))
        if world > 1:
            dist.reduce(colsum, dst=0, op=dist.ReduceOp.SUM)
            if rank == world - 1:
                dist.send(out[-512:], dst=0)
            elif rank == 0:
                dist.recv(tail, src=world - 1)
    ms_d, ms_d_max, _, _ = env.timed(kernel_display, g_steps, 1)
    result["with_display_reduction"] = {"ms_per_step": ms_d_max, "value": WIDEBAND_ROWS * n / (ms_d_max * 1e-3) / 1e6,
                                        "unit": UNIT, "steps": g_steps,
                                        "bytes": (n * 4 * (world - 1) + 512 * n * 4) if world > 1 else 0}
    result["collective"] = {"kind": "dist.gather of the F32 result to rank 0 (NCCL over NVLink / NVSwitch)",
                            "excluded_ms": ms_k_max, "included_ms": ms_g_max, "bytes": gather_bytes,
                            "nvlink_gbs_into_rank0": nvlink,
                            "display_included_ms": ms_d_max,
                            "note": "N = 1: no collective, included == excluded" if world == 1 else
                                    "rank 0's ingress link bounds the full gather; the display-sized boundary (column sums "
                                    "+ 512 newest rows) is what a lineplot / waterfall consumer needs"}
    achieved = rows * n * BYTES_PER_SAMPLE / (ms_k * 1e-3) / 1e9
    result["roofline"] = {"bound": "hbm", "achieved": achieved, "peak": env.peak, "unit": "GB/s", "frac": achieved / env.peak,
                          "kernel": "fft4096_kernel<MODE_AMP_RANGE,WIN_REAL>", "kernel_ms": ms_k,
                          "algorithmic_bytes_per_launch": rows * n * BYTES_PER_SAMPLE, "peak_source": env.peak_src}
    result["gpu_launches"] = steps + 2 * g_steps
    env.check(lib.b200_chain_plan_destroy(plan))
    del x, out
    torch.cuda.empty_cache()
    return result


# ---- BASELINE configs[1]: the headline -----------------------------------------------------------------

def main_chain(env, args):
    torch, lib = env.torch, env.lib
    from cyberether_b200 import amplitude_scaling_coeff, range_coefficients
    world, rank, dev = env.world, env.rank, env.dev
    rows, n = args.rows, N_FFT
    x = env.synthetic_rows(rows, first_row=rank * rows, seed=rank)
    out = torch.empty(rows, n, dtype=torch.float32, device=dev)
    plan = env.chain_plan(rows)
    coeff = amplitude_scaling_coeff(n)
    scale, offset = range_coefficients(RANGE_MIN, RANGE_MAX)

    def step():
        env.check(lib.b200_chain_exec(plan, x.data_ptr(), out.data_ptr(), rows, coeff, 1, scale, offset, env.sp))

    sampler = ClockSampler(env.local)
    sampler.start()
    ms_local, ms_per_step, t_begin, t_end = env.timed(step, args.steps, args.warmup)
    dump_output(env, args.dump_outputs, "chain_out", out)
    samples_per_step_all = rows * n * world
    value = samples_per_step_all / (ms_per_step * 1e-3) / 1e6
    launches = args.steps

    # -- e2e: host buffers through b200_chain_exec_host (H2D + kernel + D2H every step)
    e2e_steps = max(1, min(args.steps, args.e2e_steps))
    x_host = torch.empty(rows, n, dtype=torch.complex64, pin_memory=True)
    out_host = torch.empty(rows, n, dtype=torch.float32, pin_memory=True)
    x_host.copy_(x)
    torch.cuda.synchronize(dev)

    def e2e_step():
        env.check(lib.b200_chain_exec_host(plan, x_host.data_ptr(), out_host.data_ptr(), rows, coeff, 1, scale, offset, 0))
    e2e_step()    # warm-up (allocates the staging slots)
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()  # synchronous: returns when out_host is complete
    t_e2e = time.perf_counter() - t0
    e2e_value = samples_per_step_all * e2e_steps / env.max_over_ranks(t_e2e) / 1e6
    checksum = float(out_host[:: max(1, rows // 64)].double().sum())   # the step's result is read on the host
    launches += (e2e_steps + 1) * ((rows + 4095) // 4096)

    sampler.stop_flag.set()
    sampler.join(timeout=1.0)
    clocks = sampler.summary(t_begin, t_end)

    # -- roofline of the dominant (only) kernel in the timed region
    achieved = rows * n * BYTES_PER_SAMPLE / (ms_local * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": env.peak, "unit": "GB/s", "frac": achieved / env.peak,
                "traffic": ncu_traffic_per_launch(), "kernel": "fft4096_kernel<MODE_AMP_RANGE,WIN_REAL>",
                "algorithmic_bytes_per_launch": rows * n * BYTES_PER_SAMPLE, "kernel_ms": ms_local,
                "peak_source": env.peak_src}

    variants, workloads = None, None
    if not args.no_extras:
        variants = {"ci8_host": finish_e2e(env, guarded(e2e_ci8, env, plan, rows, coeff, scale, offset, e2e_steps))}
        del out_host
        variants["shim_flowgraph"] = finish_e2e(env, guarded(e2e_shim, env, rows, x_host, e2e_steps, False))
        variants["shim_flowgraph_analyzer"] = finish_e2e(env, guarded(e2e_shim, env, rows, x_host, e2e_steps, True))
    variant_name = lib.b200_chain_plan_variant(plan).decode()
    env.check(lib.b200_chain_plan_destroy(plan))
    del x, out, x_host
    torch.cuda.empty_cache()
    if not args.no_extras:
        workloads = {"wideband": guarded(bench_wideband, env, args.steps, 3)}
        if world == 1:
            workloads["fir"] = guarded(bench_fir, env, args.steps, 5)
            workloads["fm"] = guarded(bench_fm, env, args.steps, 5)
            workloads["fft"] = guarded(bench_fft, env, args.steps, 3)
        for w in workloads.values():
            if isinstance(w, dict):
                launches += int(w.get("gpu_launches", 0) or 0)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = guarded(run_reference_cpu, 12, 1)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(rows), "rows_per_gpu": rows, "n": n,
                       "parallelism": f"batch-sharded x{world} (no data-path collective)",
                       "range": [RANGE_MIN, RANGE_MAX],
                       "l2": "inputs larger than L2 (2 GiB in + 1 GiB out per step vs 126 MB)",
                       "numa": env.numa},
            "gpu_launches": launches,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": rows * n * 8,
                    "d2h_bytes_per_step": rows * n * 4, "steps": e2e_steps,
                    "api": "b200_chain_exec_host (pinned host buffers, 3-stream chunked pipeline)",
                    "checksum": checksum},
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "e2e_variants": variants,
            "workloads": workloads,
            "kernel_variant": variant_name,
        }
        emit(line)
    return 0


def main_single_workload(env, args):
    fn = {"fir": bench_fir, "fm": bench_fm}.get(args.workload)
    if fn is not None:
        res = fn(env, args.steps, args.warmup, with_cpu=not args.no_cpu_baseline, dump=args.dump_outputs)
    else:
        res = bench_wideband(env, args.steps, args.warmup, dump=args.dump_outputs)
        res = {"metric": WORKLOAD_METRICS["wideband"], "value": res["kernel_only"]["value"], "unit": UNIT,
               "ms_per_step": res["kernel_only"]["ms_per_step"], "steps": args.steps,
               "config": {"workload": "wideband [8,131072,4096] CF32 strong-scaled", "l2": "inputs larger than L2"},
               "roofline": res["roofline"], "collective": res["collective"], "detail": res,
               "gpu_launches": res["gpu_launches"]}
    if env.rank == 0:
        line = {"n_gpus": env.world, "warmup": max(3, args.warmup), "higher_is_better": True,
                "scaling": "strong" if args.workload == "wideband" else "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic"}
        line.update(res)
        emit(line)
    return 0


_REAL_STDOUT = None


def quiet_stdout():
    """Native libraries print banners to fd 1 (NCCL's version line, the reference backend's device table): the contract is
    ONE JSON line on stdout, so fd 1 is pointed at stderr for the duration of the run and the line goes to the saved fd."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    text = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(text.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, text)


def main_ours(args):
    quiet_stdout()
    env = Env()
    try:
        if args.workload == "chain":
            return main_chain(env, args)
        return main_single_workload(env, args)
    finally:
        if env.world > 1:
            env.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="chain", choices=["chain", "fir", "fm", "wideband"])
    ap.add_argument("--rows", type=int, default=ROWS)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline only (no variants / workloads)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed path's outputs of its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's CUDA path; --impl reference has none")
    if args.impl == "reference":
        return main_reference(args)
    return main_ours(args)


if __name__ == "__main__":
    sys.exit(main())
