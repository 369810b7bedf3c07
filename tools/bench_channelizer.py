#!/usr/bin/env python
"""Stream rate of the polyphase filter-bank channelizer (b200c_chan_run): one JSON line per config, plus one line
for config D done with 64 band-pass FirFilter handles (the only way before the channelizer).

Inputs are 2^28 complex float32 samples (2 GiB, far larger than L2); CUDA-event timing over --iters launches after
warm-up.  Algorithmic traffic: 8 B per input sample + 8 B per output sample (M/D outputs per input); flops:
4 ntaps (real taps x complex samples) + 5 M log2 M (one M-point FFT) per frame.  Every line carries a parity
check of seeded frames against the direct-sum definition (tests/_chan_oracle.py) at the 1e-5 per-channel bar, so a fast
but wrong kernel cannot report a number."""
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
from pothoscomms_b200 import Channelizer, FirFilter  # noqa: E402

CONFIGS = {"A": (1024, 1024, 8192), "B": (1024, 512, 8192), "C": (4096, 4096, 65536), "D": (64, 64, 1024)}


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


def parity(ch, h, M, D, frames):
    rng = np.random.default_rng(M * 131 + D)
    n = len(h) - 1 + frames * D
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    s = 2**40 + 7
    out = torch.empty((M, frames, 2), dtype=torch.float32, device="cuda")
    c, p = ch.run(torch.from_numpy(x.view(np.float32).reshape(-1, 2)).cuda(), out, s)
    torch.cuda.synchronize()
    assert p == frames
    y = out.cpu().numpy().astype(np.float64)
    y = y[..., 0] + 1j * y[..., 1]
    ref = channelize(x, h, M, D, s)
    err = np.sqrt(np.mean(np.abs(y - ref) ** 2, axis=1)) / np.sqrt(np.mean(np.abs(ref) ** 2, axis=1))
    assert np.all(err <= 1e-5), f"parity failed: worst channel err/rms {err.max():.3g}"
    return float(err.max())


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
    x = torch.randn((n, 2), device="cuda")
    rates = {}
    for cfg in args.configs:
        M, D, ntaps = CONFIGS[cfg]
        ch = Channelizer("complex_float32", M, D)
        h = prototype(M, ntaps)
        ch.set_taps(h)
        pf = 64 if M * ntaps <= (1 << 24) else 4     # the dense reference costs M * ntaps per frame
        worst = parity(ch, h, M, D, pf)
        F = (n - (ntaps - 1)) // D
        out = torch.empty((M, F, 2), dtype=torch.float32, device="cuda")
        ms = time_ms(lambda: ch.run(x, out, 0), args.iters)
        consumed = F * D
        nbytes = 8 * consumed + 8 * M * F
        flops = (4 * ntaps + 5 * M * math.log2(M)) * F
        gbs = nbytes / ms / 1e6
        rates[cfg] = consumed / ms / 1e3
        print(json.dumps({"name": f"chan_{cfg}", "M": M, "D": D, "ntaps": ntaps, "kernel": "pfb_chan_kernel",
                          "in_samples": consumed, "ms": round(ms, 4), "msamples_per_s": round(consumed / ms / 1e3, 1),
                          "bytes": nbytes, "gbs": round(gbs, 1), "hbm_frac": round(gbs / peak, 4), "peak_gbs": peak,
                          "peak_kind": peak_kind, "tflops": round(flops / ms / 1e9, 2), "flop_per_byte": round(flops / nbytes, 2),
                          "parity_frames": pf, "parity_max_err_rel": worst, "device": name, "power_limit": power}), flush=True)
        del out, ch
        torch.cuda.empty_cache()
    if "D" in args.configs:
        # config D the way it had to be done before: one FirFilter per channel, complex band-pass taps
        M, D, ntaps = CONFIGS["D"]
        h = prototype(M, ntaps)
        nf = 1 << 24
        xf = x[:nf].contiguous()
        filters = []
        for c in range(M):
            f = FirFilter("complex_float32", "COMPLEX")
            f.set_taps(h * np.exp(2j * np.pi * c * np.arange(ntaps) / M))
            f.set_rates(D, 1)
            filters.append(f)
        outs = [torch.empty(((nf - (ntaps - 1)) // D + 1, 2), dtype=torch.float32, device="cuda") for _ in range(M)]

        def run_all():
            for f, o in zip(filters, outs):
                f.run(xf, out=o)
        ms = time_ms(run_all, max(3, args.iters // 2), warmup=1)
        consumed = (nf - (ntaps - 1)) // D * D
        msps = consumed / ms / 1e3
        print(json.dumps({"name": "chan_D_as_64_fir_filters", "M": M, "D": D, "ntaps": ntaps, "kernel": filters[0].kernel,
                          "in_samples": consumed, "ms": round(ms, 4), "msamples_per_s": round(msps, 1),
                          "channelizer_speedup": round(rates["D"] / msps, 1) if "D" in rates else None,
                          "device": name, "power_limit": power}), flush=True)


if __name__ == "__main__":
    main()
