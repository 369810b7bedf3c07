#!/usr/bin/env python
"""Stream rate of the real-input polyphase filter-bank channelizer (b200c_rchan_run): one JSON line per config and
input type, plus one line per config A, B and D done the way it had to be done before: a torch conversion of the
real stream to complex float32, then the complex Channelizer at the same M and D, timed as one unit.

Inputs are 2^28 real samples (1 GiB float32, 512 MiB int16, far larger than L2); CUDA-event timing over --iters
launches after warm-up.  Algorithmic traffic per input sample: 4 B (float32) or 2 B (int16) read, 8 (M/2+1) / D B
written; flops per frame: 2 ntaps (real taps x real samples) + 5 (M/2) log2(M/2) (one M/2-point complex FFT) + 6 M
(the even/odd split).  Every line carries a parity check of seeded frames against the direct-sum definition
(tests/_chan_oracle.py on the real stream taken as complex) at the 1e-5 per-channel bar, so a fast but wrong kernel
cannot report a number."""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))   # the direct-sum reference lives with the tests
import numpy as np  # noqa: E402
import torch  # noqa: E402

from _chan_oracle import channelize  # noqa: E402
from pothoscomms_b200 import Channelizer, RealChannelizer  # noqa: E402

# name: (M, D, ntaps, input types)
CONFIGS = {"A": (2048, 2048, 16384, ("float32", "int16")), "B": (2048, 1024, 16384, ("float32",)),
           "C": (8192, 8192, 131072, ("float32",)), "D": (128, 128, 2048, ("float32",))}
WORKAROUND = "ABD"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"], "measured"
    except Exception:
        return 6650.0, "fallback"


def gpu_name_power():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",", 1)]
        return name, power
    except Exception:
        return torch.cuda.get_device_name(), "unknown"


def prototype(M, ntaps):
    from scipy import signal
    return signal.firwin(ntaps, 1.0 / M, window=("kaiser", 10.0))


def _rel_err(y, ref):
    err = np.sqrt(np.mean(np.abs(y - ref) ** 2, axis=1)) / np.sqrt(np.mean(np.abs(ref) ** 2, axis=1))
    assert np.all(err <= 1e-5), f"parity failed: worst channel err/rms {err.max():.3g}"
    return float(err.max())


def _seeded(M, D, dtype, n):
    rng = np.random.default_rng(M * 131 + D)
    if dtype == "int16":
        return rng.integers(-32768, 32768, size=n).astype(np.int16)
    return rng.standard_normal(n).astype(np.float32)


def parity(run, M, D, h, dtype, frames, nrows):
    """run(d_in, out, s) -> produced, on seeded input; checked against rows 0 .. M/2 of the direct sum."""
    x = _seeded(M, D, dtype, len(h) - 1 + frames * D)
    s = 2**40 + 7
    out = torch.empty((nrows, frames, 2), dtype=torch.float32, device="cuda")
    assert run(torch.from_numpy(x).cuda(), out, s) == frames
    torch.cuda.synchronize()
    y = out[: M // 2 + 1].cpu().numpy().astype(np.float64)
    y = y[..., 0] + 1j * y[..., 1]
    return _rel_err(y, channelize(x.astype(np.complex128), h, M, D, s)[: M // 2 + 1])


def time_ms(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="ABCD")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--log2n", type=int, default=28)
    args = ap.parse_args()
    peak, peak_kind = peaks()
    name, power = gpu_name_power()
    n = 1 << args.log2n
    xs = {"float32": torch.randn(n, device="cuda")}
    xs["int16"] = (xs["float32"] * 8000).clamp_(-32768, 32767).to(torch.int16)
    rates = {}
    for cfg in args.configs:
        M, D, ntaps, dtypes = CONFIGS[cfg]
        h = prototype(M, ntaps)
        pf = 16 if M * ntaps <= (1 << 24) else 4 if M * ntaps <= (1 << 28) else 2   # the dense reference costs M * ntaps per frame
        F = (n - (ntaps - 1)) // D
        consumed = F * D
        flops = (2 * ntaps + 5 * (M // 2) * math.log2(M // 2) + 6 * M) * F
        for dtype in dtypes:
            ch = RealChannelizer(dtype, M, D)
            ch.set_taps(h)
            worst = parity(lambda d, o, s: ch.run(d, o, s)[1], M, D, h, dtype, pf, M // 2 + 1)
            out = torch.empty((M // 2 + 1, F, 2), dtype=torch.float32, device="cuda")
            x = xs[dtype]
            ms = time_ms(lambda: ch.run(x, out, 0), args.iters)
            nbytes = x.element_size() * consumed + 8 * (M // 2 + 1) * F
            gbs = nbytes / ms / 1e6
            rates[(cfg, dtype)] = consumed / ms / 1e3
            print(json.dumps({"name": f"rchan_{cfg}_{dtype}", "M": M, "D": D, "ntaps": ntaps, "dtype": dtype,
                              "kernel": "pfb_rchan_kernel", "in_samples": consumed, "ms": round(ms, 4),
                              "msamples_per_s": round(consumed / ms / 1e3, 1), "bytes": nbytes, "gbs": round(gbs, 1),
                              "hbm_frac": round(gbs / peak, 4), "peak_gbs": peak, "peak_kind": peak_kind,
                              "tflops": round(flops / ms / 1e9, 2), "flop_per_byte": round(flops / nbytes, 2),
                              "parity_frames": pf, "parity_max_err_rel": worst, "device": name, "power_limit": power}),
                  flush=True)
            del out, ch
            torch.cuda.empty_cache()
        if cfg not in WORKAROUND:
            continue
        # the same channels before this handle existed: convert to complex float32, then the complex channelizer
        ch = Channelizer("complex_float32", M, D)
        ch.set_taps(h)

        def convert_and_run(x, out, s):
            xc = torch.stack((x.to(torch.float32), torch.zeros_like(x, dtype=torch.float32)), dim=-1)
            return ch.run(xc, out, s)[1]
        worst = parity(convert_and_run, M, D, h, "float32", pf, M)
        out = torch.empty((M, F, 2), dtype=torch.float32, device="cuda")
        x = xs["float32"]
        ms = time_ms(lambda: convert_and_run(x, out, 0), args.iters)
        msps = consumed / ms / 1e3
        print(json.dumps({"name": f"rchan_{cfg}_float32_as_convert_plus_channelizer", "M": M, "D": D, "ntaps": ntaps,
                          "kernel": "torch.stack + pfb_chan_kernel", "in_samples": consumed, "ms": round(ms, 4),
                          "msamples_per_s": round(msps, 1),
                          "real_channelizer_speedup": round(rates[(cfg, "float32")] / msps, 2),
                          "parity_frames": pf, "parity_max_err_rel": worst, "device": name, "power_limit": power}),
              flush=True)
        del out, ch
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
