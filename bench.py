#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: FIR Msamples/s (cf32, 256 taps) on 1/2/4/8 B200.

One "step" = one pass of the /comms/fir_filter hot path over one batch of synthetic
tone+noise input (per GPU: 2^28 complex-float32 samples = 2 GiB in + 2 GiB out, far larger
than the 126 MB L2, so nothing is cache-resident between steps).

  python bench.py --gpus 1 --steps 20 --warmup 5
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...      # the reference's own CPU block on the host cores
  python bench.py ... --dump-outputs DIR    # also write what the last timed step computed, DIR/<name>.npy

The ONE JSON line carries the headline workload in the contract's top-level keys and, under
"configs", one record per BASELINE.json config measured in the same run (each with its own
value / roofline / cpu_baseline / e2e):
  N = 1 : c1, c2, c3 (2^30 samples), c4 (cf32 and int16), c5_bank (1024 channels x 2^20)
  N > 1 : c3 (one 2^30-sample stream cut into N segments, strong scaling) and c5_bank (1024 channels
          sharded by channel, strong scaling) next to the weak-scaling headline.
`--workload X` measures a single workload instead (profiling runs); `--configs none` drops the extras.

Multi-GPU (N>1): ONE long stream is split into contiguous segments, one per rank; before every pass rank r
pulls the last K-1 samples of rank r-1's segment out of the neighbour's HBM (b200c_halo_exchange: CUDA IPC
peer mapping, one copy over NVLink on the compute stream) -- the only exchange the path has (SURVEY.md 8e).
B200C_BENCH_HALO=nccl selects the NCCL P2P form of round 1 instead.  After the timed region every rank
r > 0 checks the halo it received against the neighbour's tail (sent once more through NCCL) and its first
halo-dependent outputs against the CPU oracle.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _baseline_metric() -> str:
    """BASELINE.json's metric string, verbatim (the file travels with the repo)."""
    try:
        with open(os.path.join(ROOT, "BASELINE.json")) as f:
            return json.load(f)["metric"]
    except Exception:
        return "FIR Msamples/s (cf32, 256 taps) at 1/2/4/8 B200; % HBM roofline; vs host CPU"


def _workloads_module():
    """pothoscomms_b200/workloads.py (numpy-only tap and signal generators) loaded BY PATH: the reference
    arm must not import the product package, whose __init__ loads libb200comms.so."""
    name = "b200c_bench_workloads"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "pothoscomms_b200", "workloads.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


METRIC = _baseline_metric()
UNIT = "Msamples/s"

WORKLOADS = {
    # name: (dtype name, taps config, decim, interp, log2 samples per GPU, bytes/input sample (algorithmic))
    "headline": ("complex_float32", "headline", 1, 1, 28, 16.0),
    "c1": ("complex_float32", "c1", 1, 1, 28, 16.0),
    "c1_real": ("complex_float32", "c1_real", 1, 1, 28, 16.0),
    "c2": ("complex_int16", "c2", 1, 1, 28, 8.0),
    "c3": ("complex_float32", "c3", 2, 3, 28, 20.0),
    "c5": ("complex_float32", "c5", 1, 1, 26, 16.0),
    # short-tap streams: the HBM-bound side of the path (north_star's ">= 70 % of HBM roofline
    # for short-tap FIR and resampling")
    "short": ("complex_float32", "short", 1, 1, 28, 16.0),
    "short_cx": ("complex_float32", "short_cx", 1, 1, 28, 16.0),
    "resamp_short": ("complex_float32", "resamp_short", 2, 3, 28, 20.0),
    "real64": ("float32", "real64", 1, 1, 29, 8.0),
    "real64_i16": ("int16", "real64", 1, 1, 29, 4.0),
    # the C3 resampler on the bit-exact fixed-point type (4 B in + 6 B out per input sample)
    "c3_i16": ("complex_int16", "c3_i16", 2, 3, 28, 10.0),
}
DTYPE_CODES = {"float32": 0, "complex_float32": 1, "float64": 2, "complex_float64": 3, "int8": 4, "complex_int8": 5,
               "int16": 6, "complex_int16": 7, "int32": 8, "complex_int32": 9, "int64": 10, "complex_int64": 11}
# CPU sample per host thread (log2 samples), sized so one pass takes ~1-2 s on the box's cores
CPU_LOG2 = {"headline": 22, "c1": 22, "c1_real": 22, "c2": 22, "c3": 22, "c5": 20, "c3_i16": 22}
# --dump-outputs keeps at most this many rows of each output (a workload returns at most two complex outputs: at most
# 2 x (16 MiB of float64 values + 8 MiB of row numbers) = 48 MiB per run)
DUMP_ROWS = 1 << 20
DUMP_SEED = 0xD0D0


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons during the timed region (NVML)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(0.02)

    def stop(self):
        self._halt.set()
        if self.ok:
            self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def workload_config(wl_name: str, log2n: int | None = None, split: str = "weak") -> dict:
    """The `config` object of a FIR workload: the same for the GPU arm and the reference arm."""
    wl = _workloads_module()
    dt_name, taps_name, M, L, log2_default, _ = WORKLOADS[wl_name]
    log2n = log2n or log2_default
    taps, tt = wl.config_taps(taps_name)
    size = (f"2^{log2n} samples per GPU" if split == "weak" else f"one 2^{log2n}-sample stream over all GPUs")
    return {"workload": f"{wl_name}: /comms/fir_filter {dt_name} {len(taps)} {tt} taps decim={M} interp={L}, "
                        f"{size} tone+noise, one stream split in contiguous segments with K-1 halo",
            "samples_per_gpu": (1 << log2n) if split == "weak" else None,
            "l2_policy": "inputs larger than L2 (GiB-sized in and out per pass)"}


def workload_traffic(wl_name: str, samples: int):
    """DRAM bytes one launch moves (ncu dram__bytes_read + write per sample, profiles/traffic.json, x the samples of
    a launch), or None when no capture of that workload's kernel is committed."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f).get(wl_name)
        return t["bytes_per_sample"] * samples if t else None
    except Exception:
        return None


def cpu_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------ CPU arm ---
def run_cpu_sample(wl_name: str, threads: int, log2_per_thread: int = 21, repeats: int = 1, taps_override=None):
    """Times the REFERENCE's own /comms/fir_filter block (oracle/_ref/libfirref.so: filter/FIRFilter.cpp compiled
    unmodified, -O3 -DNDEBUG generic x86-64 = a CMake Release build) on a bounded sample of the workload: `threads`
    block instances (the reference runs one actor per block), each filtering its own contiguous segment in one
    work() call.  Falls back to the bit-identical restatement (kind "port") only if the library is absent.
    Returns (Msamples/s, samples consumed, seconds, kind)."""
    import numpy as np

    import oracle
    wl = _workloads_module()
    dt_name, taps_name, M, L, _, _ = WORKLOADS[wl_name]
    code = DTYPE_CODES[dt_name]
    taps, tt = taps_override if taps_override is not None else wl.config_taps(taps_name)
    seg = 1 << log2_per_thread
    base = wl.tone_noise_numpy(code, min(seg, 1 << 22), seed=0xC0FFEE01)
    x = np.tile(base, (threads * seg // base.shape[0], 1))
    use_ref = oracle.have_ref_fir()
    best, cons = None, 0
    for _ in range(repeats):
        t0 = time.perf_counter()
        if use_ref:
            _, cons, _ = oracle.ref_fir(code, tt == "COMPLEX", taps, M, L, x, threads=threads) if threads > 1 else \
                oracle.ref_fir(code, tt == "COMPLEX", taps, M, L, x)
        else:
            _, cons, _ = oracle.fir(code, tt == "COMPLEX", taps, M, L, x, threads=threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return cons / best / 1e6, cons, best, ("reference" if use_ref else "port")


def cpu_baseline_record(wl_name: str, repeats: int = 1, taps_override=None):
    threads = cpu_threads()
    lg = CPU_LOG2.get(wl_name, 21)
    v, _, secs, kind = run_cpu_sample(wl_name, threads, log2_per_thread=lg, repeats=repeats, taps_override=taps_override)
    return {"value": v, "unit": UNIT, "cores": threads, "kind": kind,
            "build": "filter/FIRFilter.cpp unmodified, g++ -O3 -DNDEBUG, generic x86-64 (no -march), scalar" if kind == "reference"
                     else "oracle restatement, gcc -O3, scalar",
            "sample": f"{threads} block instances (one per host thread) x 2^{lg} samples of the same workload, one work() "
                      f"call each ({secs:.2f} s wall, best of {repeats})"}


def reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores -- the
    /comms/fir_filter block compiled from filter/FIRFilter.cpp (oracle/_ref/libfirref.so), one block instance
    per host thread, each step a bounded sample of the workload.  Never imports the product package."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = cpu_threads()
    # W warm-up steps, then exactly K timed steps; a step is a bounded sample of the workload (2^19 samples per
    # host thread: ~0.2 s at the measured 50-90 Msamples/s) so that any K the driver picks ends within minutes
    log2_step = 19
    kind = "reference"
    for _ in range(args.warmup):
        run_cpu_sample(args.workload, threads, log2_per_thread=log2_step)
    total_s, total_n = 0.0, 0
    steps = max(1, args.steps)
    for _ in range(steps):
        _, cons, dt, kind = run_cpu_sample(args.workload, threads, log2_per_thread=log2_step)
        total_s += dt
        total_n += cons
    value = total_n / total_s / 1e6
    dt_name = WORKLOADS[args.workload][0]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": total_s / steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" if "float" in dt_name else dt_name, "data": "synthetic",
        "config": workload_config(args.workload),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                         "build": "filter/FIRFilter.cpp unmodified, g++ -O3 -DNDEBUG, generic x86-64 (no -march), scalar",
                         "sample": f"{threads} block instances x 2^{log2_step} samples per step, {steps} steps"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------ GPU arm ---
class Ctx:
    """Process-wide state of the GPU arm: ranks, device, process group."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peaks, self.peak_kind = measured_peaks()

    def pcie_peak(self):
        """Plain cudaMemcpy rates of this box with pinned memory (256 MiB, both directions at once on two streams): the
        ceiling of any host-buffer path, reported next to e2e.  Measured once per process."""
        if getattr(self, "_pcie", None) is None:
            torch = self.torch
            n = 256 << 20
            h1, h2 = torch.empty(n, dtype=torch.uint8).pin_memory(), torch.empty(n, dtype=torch.uint8).pin_memory()
            d1, d2 = torch.empty(n, dtype=torch.uint8, device=self.dev), torch.empty(n, dtype=torch.uint8, device=self.dev)
            s1, s2 = torch.cuda.Stream(self.dev), torch.cuda.Stream(self.dev)
            best = None
            for _ in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                with torch.cuda.stream(s1):
                    d1.copy_(h1, non_blocking=True)
                with torch.cuda.stream(s2):
                    h2.copy_(d2, non_blocking=True)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                best = dt if best is None else min(best, dt)
            self._pcie = n / best / 1e9
        return self._pcie

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        if self.world == 1:
            return list(vals)
        t = self.torch.tensor(list(vals), device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def timed_region(ctx: Ctx, step, steps: int, warmup: int, kernel_events: bool = True):
    """W warm-ups, barrier + sync, K timed steps bracketed by CUDA events on the launching stream, max over
    ranks.  `step(record)` launches one step and calls record(0) / record(1) around its compute launch."""
    torch = ctx.torch
    noop = lambda i: None   # noqa: E731
    for _ in range(warmup):
        step(noop)
    torch.cuda.synchronize()
    sampler = ClockSampler(physical_gpu_index(ctx.local_rank))
    ctx.barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    ev0.record()
    for i in range(steps):
        step((lambda j, i=i: kev[i][j].record()) if kernel_events else noop)
    ev1.record()
    torch.cuda.synchronize()
    ctx.barrier()
    clocks = sampler.stop()
    elapsed = ev0.elapsed_time(ev1)
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / steps if kernel_events else elapsed / steps
    elapsed, kernel_ms = ctx.max_over_ranks(elapsed, kernel_ms)
    return elapsed / steps, kernel_ms, clocks


def dump_outputs(path: str, outputs: dict) -> None:
    """--dump-outputs: each CUDA tensor of `outputs` (what the timed path returned in its last step, [..., ncomp]) as
    path/<name>.npy, rows x ncomp -- float32 for float32, int8 and int16 data (exact), float64 otherwise -- and the row
    numbers it holds as path/<name>_rows.npy (float64).  An output longer than DUMP_ROWS keeps a fixed sample: one row at a
    seeded place in each of DUMP_ROWS equal spans.  The inputs are seeded as well, so two builds run with the same
    arguments can be compared row for row."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for name, t in outputs.items():
        t = t.reshape(-1, t.shape[-1])
        n = t.shape[0]
        rows = np.arange(n, dtype=np.int64)
        if n > DUMP_ROWS:
            lo = np.arange(DUMP_ROWS + 1, dtype=np.int64) * n // DUMP_ROWS
            rows = lo[:-1] + (np.random.default_rng(DUMP_SEED).random(DUMP_ROWS) * np.diff(lo)).astype(np.int64)
        vals = t.index_select(0, torch.from_numpy(rows).to(t.device)).cpu().numpy()
        exact32 = vals.dtype == np.float32 or (vals.dtype.kind == "i" and vals.itemsize <= 2)
        np.save(os.path.join(path, f"{name}.npy"), vals.astype(np.float32 if exact32 else np.float64))
        np.save(os.path.join(path, f"{name}_rows.npy"), rows.astype(np.float64))


def kernel_note(kernel: str) -> str:
    if kernel == "fir_os32x_kernel":
        return ("spectral resampler (one 1024-point forward + one 1536-point inverse transform per block): one pass over "
                "HBM, 8 B in + 12 B out per input sample whatever the tap count")
    if kernel.startswith("fir_os"):
        return "fused overlap-save (fast convolution): one pass over HBM, 16 B per sample whatever the tap count"
    if kernel.startswith("fir_umma"):
        return ("bit-exact int16 as byte-limb Toeplitz GEMMs on the int8 tensor cores (tcgen05 kind::i8, accumulators in "
                "tensor memory); HBM-normalised here, the `tensor` entry gives the tensor-pipe view")
    if kernel.startswith("fir_imma"):
        return "bit-exact int16 as byte-limb Toeplitz GEMMs on mma.sync m16n8k32 (int8 tensor cores)"
    return "direct form: FMA/IMAD-issue bound once taps x MACs/tap exceed ~11 flop/B; see DESIGN.md"


def halo_check(ctx: Ctx, fir, buf, out, K: int, M: int, L: int, code: int, taps, tt: str):
    """N > 1, outside the timed region: (1) the halo this rank pulled equals the neighbour's tail (sent once more
    through NCCL P2P, an independent path); (2) this rank's first halo-dependent outputs equal the CPU oracle's
    (filter/FIRFilter.cpp:281,283) computed from [halo | first samples].  Returns a short status string."""
    torch, dist = ctx.torch, ctx.dist
    import numpy as np

    import oracle
    if ctx.world == 1 or K <= 1:
        return "n/a"
    n = buf.shape[0]
    tail = buf[n - (K - 1):].contiguous()
    got = torch.empty_like(tail)
    ops = []
    if ctx.rank + 1 < ctx.world:
        ops.append(dist.P2POp(dist.isend, tail.view(torch.uint8), ctx.rank + 1))
    if ctx.rank > 0:
        ops.append(dist.P2POp(dist.irecv, got.view(torch.uint8), ctx.rank - 1))
    for w in dist.batch_isend_irecv(ops):
        w.wait()
    torch.cuda.synchronize()
    ok = True
    if ctx.rank > 0:
        ok = bool(torch.equal(got, buf[: K - 1]))
        nblk = -(-(K - 1) // M) + 64                      # every block that reads the halo, and a few more
        x = buf[: K - 1 + nblk * M].cpu().numpy()
        y_ref, _, p_ref = oracle.fir(code, tt == "COMPLEX", taps, M, L, x)
        y = out[:p_ref].cpu().numpy()
        if code in (0, 1):
            err = float(np.sqrt(np.mean((y.astype(np.float64) - y_ref) ** 2)) / np.sqrt(np.mean(y_ref.astype(np.float64) ** 2)))
            ok = ok and err < 1e-5
        else:
            ok = ok and bool(np.array_equal(y, y_ref))
    flag = torch.tensor([0.0 if ok else 1.0], device=ctx.dev, dtype=torch.float64)
    dist.all_reduce(flag, op=dist.ReduceOp.SUM)
    if flag.item() != 0:
        raise SystemExit(f"halo check FAILED on {int(flag.item())} rank(s): N>1 outputs differ from the single-stream oracle")
    return "ok: pulled halo == neighbour tail (NCCL resend), first halo-dependent outputs == oracle, all ranks"


def bench_stream(ctx: Ctx, name: str, steps: int, warmup: int, e2e: bool, cpu: bool, log2n: int | None = None,
                 split: str = "weak", ntaps: int | None = None, check: bool = True, dump: str | None = None) -> dict:
    """One FIR stream workload.  split = "weak": 2^log2n samples per GPU; "strong": one 2^log2n-sample stream over
    all ranks.  Returns the record (value, roofline, cpu_baseline, e2e, ...)."""
    torch = ctx.torch
    import numpy as np

    from pothoscomms_b200 import FirFilter, sharding
    wl = _workloads_module()
    dt_name, taps_name, M, L, log2_default, bytes_per_sample = WORKLOADS[name]
    if ntaps:   # tap-count sweep: the named workload's stream type with `ntaps` complex band-pass taps
        dt_name = dt_name if dt_name in ("complex_float32", "complex_int16") else "complex_float32"
        taps_name, M, L, bytes_per_sample = f"sweep{ntaps}", 1, 1, (16.0 if dt_name == "complex_float32" else 8.0)
    log2n = log2n or log2_default
    code = DTYPE_CODES[dt_name]
    taps, tt = wl.config_taps(taps_name)
    fir = FirFilter(code, tt, device=ctx.local_rank)
    fir.set_taps(taps)
    fir.set_rates(M, L)
    K = fir.K
    world, rank = ctx.world, ctx.rank
    total = (1 << log2n) * (world if split == "weak" else 1)
    n_seg = (total // world) // M * M              # new samples per rank and step (multiple of M: SURVEY 8e)
    nc = 2 if code & 1 else 1
    sharding.check_segment(n_seg, K, rank, world)

    # [K-1 halo | n_seg samples]; rank r's segment is samples [r*n_seg, (r+1)*n_seg) of one stream
    tdt = wl.tone_noise_torch(code, 1, 0, ctx.dev).dtype
    buf = torch.empty((K - 1 + n_seg, nc), dtype=tdt, device=ctx.dev)
    buf[K - 1:] = wl.tone_noise_torch(code, n_seg, 0xC0FFEE01 + rank, ctx.dev)
    buf[: K - 1] = 0   # rank 0: the stream's first K-1 samples are history only (FIRFilter.cpp:281)
    out_cap = n_seg // M * L
    out = torch.empty((out_cap, nc), dtype=tdt, device=ctx.dev)
    torch.cuda.synchronize()

    halo_mode = os.environ.get("B200C_BENCH_HALO", "peer") if world > 1 else "none"
    link = sharding.PeerHalo(buf, K, rank, world, ctx.local_rank) if halo_mode == "peer" else None

    def step(record):
        if link is not None:
            # the neighbour's tail is final before the timed region starts (inputs are resident), so the pull needs no
            # cross-process ordering here: ONE peer copy over NVLink on the compute stream, then the launch.  (An
            # interprocess event wait captures the neighbour's LATEST record at call time; with the hosts running steps
            # ahead of their GPUs that couples rank r's step i to rank r-1's step i+k and serialises the ranks --
            # measured: +0.19 ms per 0.9 ms step.  A live pipeline orders producer and consumer on the host, as Pothos'
            # actor messages do, and uses the event only for the GPU-side edge.)
            link.pull(wait=False)
        elif halo_mode == "nccl":
            sharding.exchange_halo(buf, K, rank, world)
        record(0)
        _, c, p = fir.run(buf, out=out, out_capacity=out_cap)
        record(1)
        assert c == n_seg and p == out_cap, (c, p, n_seg, out_cap)

    ms_per_step, kernel_ms, clocks = timed_region(ctx, step, steps, warmup)
    if dump and rank == 0:
        dump_outputs(dump, {"fir_out": out})
    value = world * n_seg / (ms_per_step * 1e-3) / 1e6
    halo = halo_check(ctx, fir, buf, out, K, M, L, code, taps, tt) if check else "skipped"

    # parity spot check at full size (sampled window, against the CPU oracle): rank 0's first outputs
    parity = None
    if check and rank == 0:
        import oracle
        nblk = 4096
        xw = buf[: K - 1 + nblk * M].cpu().numpy()
        y_ref, _, p_ref = oracle.fir(code, tt == "COMPLEX", taps, M, L, xw)
        y = out[:p_ref].cpu().numpy()
        if code in (0, 1):
            err = float(np.sqrt(np.mean((y.astype(np.float64) - y_ref) ** 2)) / np.sqrt(np.mean(y_ref.astype(np.float64) ** 2)))
            assert err < 1e-5, f"{name}: GPU output differs from the oracle ({err:.2e} of RMS)"
            parity = f"rel RMS error {err:.1e} vs oracle on the first {p_ref} outputs (tolerance 1e-5)"
        else:
            assert np.array_equal(y, y_ref), f"{name}: int16 output is not bit-exact"
            parity = f"bit-exact vs oracle on the first {p_ref} outputs"

    # ---- end to end through the host-buffer C-ABI call (pinned host memory, H2D + D2H timed) ----
    e2e_rec = None
    if e2e:
        # a bounded host sample for the 2^30-sample stream (pinning 20 GiB takes longer than the measurement)
        n_host = min(n_seg, 1 << 28) // M * M
        cap_host = n_host // M * L
        h_in = torch.empty((K - 1 + n_host, nc), dtype=tdt).pin_memory()
        h_out = torch.empty((cap_host, nc), dtype=tdt).pin_memory()
        h_in.copy_(buf[: K - 1 + n_host])
        x_np, y_np = h_in.numpy(), h_out.numpy()
        e2e_steps = 3
        fir.run_host(x_np, out=y_np, out_capacity=cap_host)   # warm-up (allocates the staging slots)
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            fir.run_host(x_np, out=y_np, out_capacity=cap_host)
        e2e_s = (time.perf_counter() - t0) / e2e_steps
        (e2e_s,) = ctx.max_over_ranks(e2e_s)
        assert torch.equal(h_out[:4096], out[:4096].cpu()), "host path differs from the resident path"
        hb, db = int(h_in.numel() * h_in.element_size()), int(h_out.numel() * h_out.element_size())
        e2e_rec = {"value": world * n_host / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": hb, "d2h_bytes_per_step": db,
                   "steps": e2e_steps, "h2d_gbs": hb / e2e_s / 1e9, "d2h_gbs": db / e2e_s / 1e9,
                   "memcpy_peak_gbs_each_way": ctx.pcie_peak(),   # cudaMemcpy both directions at once, pinned: the box's ceiling
                   "sample": None if n_host == n_seg else f"first 2^{n_host.bit_length() - 1} samples of the segment"}
        del h_in, h_out

    kernel = fir.kernel
    if link is not None:
        link.close()
    del buf, out
    torch.cuda.empty_cache()
    if rank != 0:
        return {}

    achieved = bytes_per_sample * n_seg / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": ctx.peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / ctx.peaks["hbm_gbs"], "traffic": workload_traffic(name, n_seg), "peak_kind": ctx.peak_kind,
                "kernel": kernel, "kernel_ms": kernel_ms, "algorithmic_bytes_per_sample": bytes_per_sample,
                "note": kernel_note(kernel)}
    if kernel.startswith(("fir_umma", "fir_imma")):
        # tensor-pipe view of the same launch: int8 MACs the byte-limb GEMMs execute (2 data limbs x tap digits x
        # 4 (complex x complex) or 2/1 real products per tap and sample) against the dense int8 rate (2x bf16)
        ntaps_eff = len(taps)
        prods = 4 if (tt == "COMPLEX") else (2 if code & 1 else 1)
        macs = 2 * 2 * prods * ntaps_eff * n_seg
        peak_i8 = 2 * ctx.peaks.get("bf16_tflops", 1590.0)
        roofline["tensor"] = {"bound": "tensor", "achieved": 2 * macs / (kernel_ms * 1e-3) / 1e12, "peak": peak_i8, "unit": "TOP/s",
                              "frac": 2 * macs / (kernel_ms * 1e-3) / 1e12 / peak_i8,
                              "note": "useful int8 MAC x 2 of the limb GEMMs (2 data limbs x 2 tap digits; Toeplitz padding not counted), "
                                      "dense int8 peak taken as 2 x the measured bf16 rate. " +
                                      ("fir_umma32t_kernel: tap tiles in tensor memory; ncu (profiles/r02ai_prof_umma32t_c2.txt) has the "
                                       "imma sub-pipe active 75 % of cycles at 1.72 GHz: tensor-pipe bound, see DESIGN 4.6"
                                       if kernel == "fir_umma32t_kernel" else
                                       "bound by shared-memory operand fetch (ncu l1tex), see DESIGN 4.6")}
    flops = {"c1": 512, "c1_real": 256, "headline": 2048, "c3": 510, "c5": 8192}.get(name)
    if flops and not kernel.startswith("fir_os"):
        roofline["fp32_tflops"] = flops * n_seg / (kernel_ms * 1e-3) / 1e12

    cpu_rec = cpu_baseline_record(name, repeats=2 if name == "headline" else 1) if cpu else None
    cfg = workload_config(name, log2n, split) if not ntaps else \
        {"workload": f"{name} stream, {ntaps}-tap complex band-pass sweep point", "samples_per_gpu": n_seg}
    return {"workload": cfg["workload"], "config": cfg, "value": value, "unit": UNIT, "ms_per_step": ms_per_step, "steps": steps,
            "warmup": warmup, "scaling": split, "n_gpus": world, "dtype": "f32" if code in (0, 1) else dt_name,
            "roofline": roofline, "cpu_baseline": cpu_rec, "e2e": e2e_rec, "gpu_launches": steps, "clocks": clocks,
            "halo": {"mode": halo_mode, "check": halo}, "parity": parity}


def bench_fft(ctx: Ctx, name: str, steps: int, warmup: int, e2e: bool, cpu: bool, log2n: int | None = None,
              dump: str | None = None) -> dict:
    """BASELINE config 4: /comms/fft 4096-point forward then inverse over 2^28 samples (per GPU: transforms are
    independent, the batch is sharded with no exchange).  One step = two passes (2 launches); value counts samples per pass."""
    torch = ctx.torch
    import numpy as np

    from pothoscomms_b200 import Fft
    wl = _workloads_module()
    dt_name = "complex_int16" if name == "c4_i16" else "complex_float32"
    code = DTYPE_CODES[dt_name]
    n, log2n = 4096, log2n or 28
    total = 1 << log2n
    x = wl.tone_noise_torch(code, total, 0xC0FFEE04 + ctx.rank, ctx.dev)
    X = torch.empty_like(x)
    y = torch.empty_like(x)
    fwd, inv = Fft(code, n, False, device=ctx.local_rank), Fft(code, n, True, device=ctx.local_rank)

    def step(record):
        record(0)
        fwd.run(x, out=X)
        inv.run(X, out=y)
        record(1)

    ms, kernel_ms, clocks = timed_region(ctx, step, steps, warmup)
    if dump and ctx.rank == 0:
        dump_outputs(dump, {"fft_forward": X, "fft_inverse": y})
    value = ctx.world * 2 * total / (ms * 1e-3) / 1e6
    esz = x.element_size() * 2
    achieved = 2 * esz * total * 2 / (kernel_ms * 1e-3) / 1e9    # (read + write) x two passes
    # size-independent property at full size (fft/TestFFT.cpp:79-80,131-132): float ifft(fft(x)) = N x; Q15 scales 1/N each way
    parity = None
    if ctx.rank == 0:
        import oracle
        if code == 1:
            err = float((y[: 1 << 20] / n - x[: 1 << 20]).double().pow(2).mean().sqrt() / x[: 1 << 20].double().pow(2).mean().sqrt())
            assert err < 1e-5, err
            ref = oracle.ref_fft(code, n, False, x[: 8 * n].cpu().numpy()) if oracle.have_ref() else oracle.fft(code, n, False, x[: 8 * n].cpu().numpy())
            e2 = float(np.sqrt(np.mean((X[: 8 * n].cpu().numpy().astype(np.float64) - ref) ** 2)) / np.sqrt(np.mean(ref.astype(np.float64) ** 2)))
            assert e2 < 1e-5, e2
            parity = f"ifft(fft(x))/N - x: {err:.1e} of RMS over 2^20 samples; first 8 transforms vs the reference's kiss_fft: {e2:.1e}"
        else:
            ref = oracle.ref_fft(code, n, False, x[: 8 * n].cpu().numpy()) if oracle.have_ref() else oracle.fft(code, n, False, x[: 8 * n].cpu().numpy())
            assert np.array_equal(X[: 8 * n].cpu().numpy(), ref), "int16 FFT is not bit-exact"
            parity = "bit-exact vs the reference's Q15 kiss_fft on the first 8 transforms"
    e2e_rec = None
    if e2e:
        h_in, h_out = x.cpu().pin_memory(), torch.empty(x.shape, dtype=x.dtype).pin_memory()
        fwd.run_host(h_in.numpy(), out=h_out.numpy())
        t0 = time.perf_counter()
        for _ in range(3):
            fwd.run_host(h_in.numpy(), out=h_out.numpy())
        e2e_s = (time.perf_counter() - t0) / 3
        (e2e_s,) = ctx.max_over_ranks(e2e_s)
        hb = int(h_in.numel() * h_in.element_size())
        e2e_rec = {"value": ctx.world * total / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": hb, "d2h_bytes_per_step": hb,
                   "h2d_gbs": hb / e2e_s / 1e9, "d2h_gbs": hb / e2e_s / 1e9, "note": "forward pass only"}
        del h_in, h_out
    cpu_rec = None
    if cpu and ctx.rank == 0:
        import oracle
        threads = cpu_threads()
        nb = threads * 512
        xs = x[: nb * n].cpu().numpy()
        t0 = time.perf_counter()
        if oracle.have_ref():
            oracle.ref_fft(code, n, False, xs, threads=threads)
            kind = "reference"
        else:
            oracle.fft(code, n, False, xs)
            kind, threads = "port", 1
        secs = time.perf_counter() - t0
        cpu_rec = {"value": nb * n / secs / 1e6, "unit": UNIT, "cores": threads, "kind": kind,
                   "sample": f"{nb} transforms of 4096 (kiss_fft compiled from the reference sources), {secs:.2f} s"}
    del x, X, y
    torch.cuda.empty_cache()
    if ctx.rank != 0:
        return {}
    wl_text = f"{name}: /comms/fft {dt_name} 4096-point batched forward then inverse over 2^{log2n} samples per GPU"
    return {"workload": wl_text, "config": {"workload": wl_text, "l2_policy": "inputs larger than L2"},
            "metric": f"FFT Msamples/s per pass ({dt_name}, 4096-point, forward+inverse)", "value": value, "unit": UNIT,
            "ms_per_step": ms, "steps": steps, "warmup": warmup, "scaling": "weak", "n_gpus": ctx.world,
            "dtype": "f32" if code == 1 else "i16",
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": ctx.peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / ctx.peaks["hbm_gbs"], "traffic": workload_traffic(name, total), "peak_kind": ctx.peak_kind,
                         "kernel": "fft4096_kernel", "kernel_ms": kernel_ms / 2, "algorithmic_bytes_per_sample": 2 * esz,
                         "note": "one CTA per 4096-point transform, one pass over HBM per direction"},
            "cpu_baseline": cpu_rec, "e2e": e2e_rec, "gpu_launches": 2 * steps, "clocks": clocks, "parity": parity}


def bench_bank(ctx: Ctx, steps: int, warmup: int, e2e: bool, cpu: bool, channels: int | None = None, log2n: int | None = None,
               dump: str | None = None) -> dict:
    """BASELINE config 5: 1024-channel filter bank, one 1024-tap complex band-pass per channel, 2^20 samples per
    channel, channels sharded over the ranks (no exchange: SURVEY.md 8e).  Strong scaling: the bank is fixed, every
    rank takes 1024/N channels.  One step = one b200c_fir_bank_run over the rank's channels (one launch)."""
    torch = ctx.torch
    import numpy as np

    from pothoscomms_b200 import FirFilter, FirFilterBank, sharding
    wl = _workloads_module()
    code = DTYPE_CODES["complex_float32"]
    nchan_total, ntaps = channels or 1024, 1024
    log2n = log2n or 20
    c0, c1 = sharding.channel_range(nchan_total, ctx.world, ctx.rank)
    nch = c1 - c0
    n_new = 1 << log2n
    bank = FirFilterBank(code, "COMPLEX", nch, device=ctx.local_rank)
    for c in range(c0, c1):
        bank.set_taps(c - c0, wl.bank_taps(c, nchan_total, ntaps))
    K = bank.info()[1]
    x = torch.empty((nch, K - 1 + n_new, 2), dtype=torch.float32, device=ctx.dev)
    base = [wl.tone_noise_torch(code, K - 1 + n_new, 0xC0FFEE05 + i, ctx.dev) for i in range(8)]
    for c in range(nch):
        x[c] = base[(c0 + c) % 8]
    del base
    out = torch.empty((nch, n_new, 2), dtype=torch.float32, device=ctx.dev)

    def step(record):
        record(0)
        cons, prod = bank.run(x, out)
        record(1)
        assert (cons, prod) == (n_new, n_new), (cons, prod)

    ms, kernel_ms, clocks = timed_region(ctx, step, steps, warmup)
    if dump and ctx.rank == 0:
        dump_outputs(dump, {"bank_out": out})
    total = nchan_total * n_new
    value = total / (ms * 1e-3) / 1e6
    # parity: this rank's first channel against a single-stream filter and against the CPU oracle (sampled window)
    f1 = FirFilter(code, "COMPLEX", device=ctx.local_rank)
    f1.set_taps(wl.bank_taps(c0, nchan_total, ntaps))
    y1, _, _ = f1.run(x[0].contiguous())
    # (the two may run different kernels -- one launch over whole channels vs a short single stream -- whose step twiddles
    # are formed differently: equal to rounding, not bit for bit)
    d1 = float((y1[:4096] - out[0, :4096]).double().pow(2).mean().sqrt() / out[0, :4096].double().pow(2).mean().sqrt())
    assert d1 < 2e-6, f"bank channel differs from its single-stream filter ({d1:.2e} of RMS)"
    import oracle
    nb = 8192
    y_ref, _, p_ref = oracle.fir(code, True, wl.bank_taps(c0, nchan_total, ntaps), 1, 1, x[0, : K - 1 + nb].cpu().numpy())
    yg = out[0, :p_ref].cpu().numpy()
    err = float(np.sqrt(np.mean((yg.astype(np.float64) - y_ref) ** 2)) / np.sqrt(np.mean(y_ref.astype(np.float64) ** 2)))
    assert err < 1e-5, f"c5_bank: {err:.2e} of RMS vs the oracle"
    e2e_rec = None
    if e2e:
        # the host-buffer call of the block, per channel (each reference block instance is one channel), on a sample of channels
        ns = min(nch, 32)
        h_in = torch.empty((ns, K - 1 + n_new, 2), dtype=torch.float32).pin_memory()
        h_out = torch.empty((ns, n_new, 2), dtype=torch.float32).pin_memory()
        h_in.copy_(x[:ns])
        f1.run_host(h_in[0].numpy(), out=h_out[0].numpy(), out_capacity=n_new)
        ctx.barrier()
        t0 = time.perf_counter()
        for c in range(ns):
            f1.run_host(h_in[c].numpy(), out=h_out[c].numpy(), out_capacity=n_new)
        e2e_s = time.perf_counter() - t0
        (e2e_s,) = ctx.max_over_ranks(e2e_s)
        hb, db = int(h_in.numel() * 4), int(h_out.numel() * 4)
        e2e_rec = {"value": ctx.world * ns * n_new / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": hb, "d2h_bytes_per_step": db,
                   "h2d_gbs": hb / e2e_s / 1e9, "d2h_gbs": db / e2e_s / 1e9,
                   "sample": f"{ns} channels per GPU, one b200c_fir_run_host per channel"}
        del h_in, h_out
    kernel = f1.kernel
    del x, out, bank, f1
    torch.cuda.empty_cache()
    if ctx.rank != 0:
        return {}
    achieved = 16.0 * nch * n_new / (kernel_ms * 1e-3) / 1e9      # this rank's kernel: its channels' bytes over its launch time
    cpu_rec = None
    if cpu:
        cpu_rec = cpu_baseline_record("c5", taps_override=(wl.bank_taps(0, nchan_total, ntaps), "COMPLEX"))
    wl_text = (f"c5_bank: {nchan_total}-channel filter bank, {ntaps}-tap complex_float32 band-pass per channel, "
               f"2^{log2n} samples per channel, channels sharded over {ctx.world} GPU(s), no exchange")
    return {"workload": wl_text, "config": {"workload": wl_text, "channels_per_gpu": nch, "l2_policy": "inputs larger than L2"},
            "value": value, "unit": UNIT, "ms_per_step": ms, "steps": steps, "warmup": warmup, "scaling": "strong",
            "n_gpus": ctx.world, "dtype": "f32",
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": ctx.peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": achieved / ctx.peaks["hbm_gbs"], "traffic": workload_traffic("c5_bank", nch * n_new), "peak_kind": ctx.peak_kind,
                         "kernel": kernel, "kernel_ms": kernel_ms, "algorithmic_bytes_per_sample": 16.0,
                         "note": "fused overlap-save, one launch over (channel, block); 16 B per sample"},
            "cpu_baseline": cpu_rec, "e2e": e2e_rec, "gpu_launches": steps, "clocks": clocks,
            "parity": f"channel {c0}: rel RMS error {err:.1e} vs oracle on {p_ref} outputs; {d1:.1e} from its single-stream filter"}


def bench_blocks(ctx: Ctx, rounds_budget_s: float = 1.0) -> dict:
    """The streaming path the drop-in actually runs (filter/FIRFilter.cpp:207-309, :196-199): the C++ /comms/fir_filter
    block of pothoscomms_b200/blocks between two device neighbours -- work() once per buffer, input in the VMM
    double-mapped HBM ring with the K-1 history left in place, one kernel launch per work(), no host<->device copy
    in the loop -- for work() buffers of 1, 4, 8 and 32 MiB.  value = the 8 MiB row (Pothos' default buffer size)."""
    from pothoscomms_b200 import blocks
    wl = _workloads_module()
    taps, tt = wl.config_taps("headline")
    pat = wl.tone_noise_numpy(DTYPE_CODES["complex_float32"], 1 << 20, seed=0xC0FFEE01)
    rows = []
    for mib in (1, 4, 8, 32):
        chunk = (mib << 20) // 8
        f = blocks.make("/comms/fir_filter", "complex_float32", tt, in_bytes=max(4 * chunk * 8, 512 << 20), out_bytes=2 * chunk * 8)
        f.call("setTaps", taps)
        f.activate()
        rounds = max(20, min(4000, int(rounds_budget_s * 250e9 / chunk)))
        secs = f.stream_bench(pat, chunk, rounds)
        calls = f.work_calls
        rows.append({"work_buffer_mib": mib, "value": rounds * chunk / secs / 1e6, "unit": UNIT, "work_calls_per_s": rounds / secs,
                     "us_per_work": secs / rounds * 1e6, "rounds": rounds, "work_calls": calls, "seam_windows": f.seam_windows,
                     "hbm_frac": 16.0 * rounds * chunk / secs / 1e9 / ctx.peaks["hbm_gbs"]})
        f.close()
    main_row = rows[2]
    wl_text = ("headline_blocks: source -> /comms/fir_filter (C++ block layer, complex_float32 256 COMPLEX taps) -> sink between "
               "device neighbours, HBM ring + slabs, one launch per work(); work() buffers 1/4/8/32 MiB")
    return {"workload": wl_text, "config": {"workload": wl_text}, "value": main_row["value"], "unit": UNIT,
            "ms_per_step": main_row["us_per_work"] / 1e3, "steps": main_row["rounds"], "warmup": 3, "scaling": "weak", "n_gpus": 1,
            "dtype": "f32",
            "roofline": {"bound": "hbm", "achieved": main_row["hbm_frac"] * ctx.peaks["hbm_gbs"], "peak": ctx.peaks["hbm_gbs"],
                         "unit": "GB/s", "frac": main_row["hbm_frac"], "traffic": None, "peak_kind": ctx.peak_kind,
                         "kernel": "fir_os32_kernel", "algorithmic_bytes_per_sample": 16.0,
                         "note": "wall clock over `rounds` work() calls incl. the block layer's host code; 8 MiB work() buffers; input "
                                 "streams from a 512 MiB HBM ring (> L2), the two output slabs are reused and stay L2-resident as they "
                                 "would between two Pothos device blocks"},
            "per_buffer_size": rows, "cpu_baseline": None, "e2e": None, "gpu_launches": main_row["rounds"], "clocks": None,
            "parity": "tests/test_blocks_gpu.py (block output == oracle, incl. across the ring seam)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="headline", choices=sorted(WORKLOADS) + ["c4", "c4_i16", "c5_bank", "headline_blocks"])
    ap.add_argument("--configs", default=None, choices=["all", "none"],
                    help="also measure the other BASELINE configs into `configs` (default: all for the headline workload)")
    ap.add_argument("--ntaps", type=int, default=None, help="tap-count sweep: cf32 L=M=1 with this many complex taps")
    ap.add_argument("--channels", type=int, default=None, help="c5_bank: total channels (default 1024)")
    ap.add_argument("--log2-samples", type=int, default=None, help="override samples per GPU (debug)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "headline_blocks"):
        ap.error("--dump-outputs is not available for --impl reference or --workload headline_blocks")
    if args.impl == "reference":
        return reference_arm(args)
    args.warmup = max(args.warmup, 3)
    want_configs = (args.configs or ("all" if args.workload == "headline" and not args.ntaps and not args.log2_samples else "none")) == "all"
    e2e, cpu = not args.no_e2e, not args.no_cpu

    ctx = Ctx()
    dump = args.dump_outputs
    if args.workload == "headline_blocks":
        main_rec = bench_blocks(ctx)
    elif args.workload in ("c4", "c4_i16"):
        main_rec = bench_fft(ctx, args.workload, args.steps, args.warmup, e2e, cpu, args.log2_samples, dump=dump)
    elif args.workload == "c5_bank":
        main_rec = bench_bank(ctx, args.steps, args.warmup, e2e, cpu and ctx.world == 1, args.channels, args.log2_samples,
                              dump=dump)
    else:
        main_rec = bench_stream(ctx, args.workload, args.steps, args.warmup, e2e, cpu and ctx.world == 1, args.log2_samples,
                                ntaps=args.ntaps, dump=dump)
    configs = []
    if want_configs:
        sub_steps, sub_warm = args.steps, 3
        if ctx.world == 1:
            plan = [("stream", "c1", 28, "weak"), ("stream", "c2", 28, "weak"), ("stream", "c3", 30, "strong"),
                    ("fft", "c4"), ("fft", "c4_i16"), ("bank",), ("blocks",)]
        else:
            plan = [("stream", "c3", 30, "strong"), ("bank",)]
        for item in plan:
            t0 = time.perf_counter()
            if item[0] == "stream":
                rec = bench_stream(ctx, item[1], sub_steps, sub_warm, e2e, cpu and ctx.world == 1, item[2], split=item[3])
            elif item[0] == "fft":
                rec = bench_fft(ctx, item[1], sub_steps, sub_warm, e2e, cpu)
            elif item[0] == "blocks":
                rec = bench_blocks(ctx)
            else:
                rec = bench_bank(ctx, sub_steps, sub_warm, e2e, cpu and ctx.world == 1)
            if rec:
                rec["wall_s"] = round(time.perf_counter() - t0, 1)
                configs.append(rec)
    if ctx.rank != 0:
        ctx.close()
        return 0

    line = {
        "metric": main_rec.get("metric", METRIC), "value": main_rec["value"], "unit": UNIT, "n_gpus": ctx.world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": main_rec["ms_per_step"], "higher_is_better": True, "scaling": main_rec["scaling"],
        "vs_baseline": None, "dtype": main_rec["dtype"], "data": "synthetic", "config": main_rec["config"],
        "roofline": main_rec["roofline"], "cpu_baseline": main_rec["cpu_baseline"], "e2e": main_rec["e2e"],
        "gpu_launches": main_rec["gpu_launches"], "clocks": main_rec["clocks"],
        "parity": main_rec.get("parity"),
    }
    if "halo" in main_rec:
        line["halo"] = main_rec["halo"]
    if configs:
        for c in configs:
            c.pop("config", None)
        line["configs"] = configs
    print(json.dumps(line))
    ctx.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
