#!/usr/bin/env python
"""Stream rate of the polyphase synthesis filter bank (b200c_synth_run): one JSON line per config, a channelizer ->
synthesizer round trip (config R) with its reconstruction error, and configs A and D written with torch ops
(torch.fft.ifft over frames plus a strided polyphase sum), the way a user had to do it before the synthesizer.

Outputs are 2^28 complex float32 samples (2 GiB, far larger than L2); CUDA-event timing over --iters launches after
warm-up.  Algorithmic traffic: 8 B per output sample + 8 M/D B of channel input per output sample; flops:
4 ntaps (real taps x complex samples) + 5 M log2 M (one M-point FFT) per frame.  Every line carries a parity check
of seeded frames against the reference (tests/_synth_oracle.synthesize) at 1e-5 of RMS, so a fast but wrong kernel
cannot report a number."""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))   # the reference lives with the tests
import numpy as np  # noqa: E402
import torch  # noqa: E402

from _synth_oracle import roundtrip_taps, synthesize  # noqa: E402
from pothoscomms_b200 import Channelizer, Synthesizer  # noqa: E402

# the channelizer's configs A-D (tools/bench_channelizer.py), read as (M, interpolation D, ntaps)
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


def prototype(M, D, ntaps):
    from scipy import signal
    return D * signal.firwin(ntaps, 1.0 / M, window=("kaiser", 10.0))


def torch_synth(X, g, M, D, s, F):
    """The same computation with torch ops: an inverse FFT of every frame, then y[t D + j] = sum_k g[j + k D]
    V[(s + t D + j) mod M, K-1 + t - k], one strided multiply-add per k.  X: [M, n, 2] float32; returns [F D, 2]."""
    K = -(-len(g) // D)
    Xc = torch.view_as_complex(X)
    V = torch.fft.ifft(Xc, dim=0) * M                             # [M, n]: unnormalised inverse DFT of every frame
    gp = torch.zeros(K * D, dtype=torch.float32, device=X.device)
    gp[:len(g)] = torch.from_numpy(np.asarray(g, dtype=np.float32)).to(X.device)
    gp = gp.view(K, D, 1)
    k_ = M // D
    y = torch.empty((F, D), dtype=torch.complex64, device=X.device)
    for b in range(k_):                                           # output frames t = b (mod M / D) read the same bins
        t = torch.arange(b, F, k_, device=X.device)
        if t.numel() == 0:
            continue
        rows = (s + b * D + torch.arange(D, device=X.device)) % M
        Vb = V[rows]                                              # [D, n]
        acc = torch.zeros((D, t.numel()), dtype=torch.complex64, device=X.device)
        for k in range(K):
            acc += gp[k] * Vb[:, K - 1 + b - k: K - 1 + b - k + k_ * (t.numel() - 1) + 1: k_]
        y[t] = acc.T
    return torch.view_as_real(y.reshape(-1))


def parity(run, g, M, D, frames):
    """Run `run(X, s, F)` on seeded frames and check it against the reference; returns the worst block's err/rms."""
    K = -(-len(g) // D)
    rng = np.random.default_rng(M * 131 + D)
    X = (rng.standard_normal((M, K - 1 + frames)) + 1j * rng.standard_normal((M, K - 1 + frames))).astype(np.complex64)
    s = 2**40 + 7
    y = run(torch.from_numpy(X.view(np.float32).reshape(M, -1, 2)).cuda(), s, frames).cpu().numpy().astype(np.float64)
    y = y[:, 0] + 1j * y[:, 1]
    ref = synthesize(X, g, M, D, s)
    assert y.shape == ref.shape
    blk, worst = 64 * D, 0.0
    for b0 in range(0, ref.size, blk):
        e, r = y[b0: b0 + blk], ref[b0: b0 + blk]
        worst = max(worst, float(np.sqrt(np.mean(np.abs(e - r) ** 2)) / np.sqrt(np.mean(np.abs(r) ** 2))))
    assert worst <= 1e-5, f"parity failed: worst block err/rms {worst:.3g}"
    return worst


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


def kernel_run(sy, D):
    def run(X, s, F):
        out = torch.empty((F * D, 2), dtype=torch.float32, device="cuda")
        c, p = sy.run(X, out, s)
        torch.cuda.synchronize()
        assert (c, p) == (F, F * D)
        return out
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="ABCDR")
    ap.add_argument("--torch-configs", default="AD")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--log2n", type=int, default=28, help="log2 of the output samples per launch")
    args = ap.parse_args()
    peak, peak_kind = peaks()
    name, power = gpu_name_power()
    n_out = 1 << args.log2n
    rates = {}
    for cfg in args.configs:
        if cfg == "R":
            continue
        M, D, ntaps = CONFIGS[cfg]
        K = -(-ntaps // D)
        sy = Synthesizer("complex_float32", M, D)
        g = prototype(M, D, ntaps)
        sy.set_taps(g)
        pf = max(4, min(64, (1 << 24) // (M * D * (K + 1))))     # the reference costs M D (K + 1) per frame
        worst = parity(kernel_run(sy, D), g, M, D, pf)
        F = n_out // D
        X = torch.randn((M, F + K - 1, 2), device="cuda")
        out = torch.empty((F * D, 2), dtype=torch.float32, device="cuda")
        ms = time_ms(lambda: sy.run(X, out, 0), args.iters)
        samples = F * D
        nbytes = 8 * samples + 8 * M * (F + K - 1)
        flops = (4 * ntaps + 5 * M * math.log2(M)) * F
        gbs = nbytes / ms / 1e6
        rates[cfg] = samples / ms / 1e3
        print(json.dumps({"name": f"synth_{cfg}", "M": M, "D": D, "ntaps": ntaps, "kernel": "pfb_synth_kernel",
                          "out_samples": samples, "ms": round(ms, 4), "msamples_per_s": round(rates[cfg], 1),
                          "bytes": nbytes, "gbs": round(gbs, 1), "hbm_frac": round(gbs / peak, 4), "peak_gbs": peak,
                          "peak_kind": peak_kind, "tflops": round(flops / ms / 1e9, 2), "flop_per_byte": round(flops / nbytes, 2),
                          "parity_frames": pf, "parity_max_err_rel": worst, "device": name, "power_limit": power}), flush=True)
        del X, out, sy
        torch.cuda.empty_cache()
    if "R" in args.configs:
        # channelizer -> synthesizer on one stream, D = M/2, the reconstruction recipe of INTEGRATION §1
        M = 1024
        D = M // 2
        h, g, s_shift, off = roundtrip_taps(M)
        ch = Channelizer("complex_float32", M, D)
        ch.set_taps(h)
        sy = Synthesizer("complex_float32", M, D)
        sy.set_taps(g)
        Kg = sy.info()[3]
        Fa = n_out // D
        rng = np.random.default_rng(1)
        nx = h.size - 1 + Fa * D
        x = torch.from_numpy(rng.standard_normal((nx, 2)).astype(np.float32)).cuda()
        mid = torch.empty((M, Fa, 2), dtype=torch.float32, device="cuda")
        Fs = Fa - (Kg - 1)
        out = torch.empty((Fs * D, 2), dtype=torch.float32, device="cuda")
        s_a = 2**40 + 3

        def both():
            ch.run(x, mid, s_a)
            sy.run(mid, out, s_a + s_shift)
        ms_s = time_ms(lambda: sy.run(mid, out, s_a + s_shift), args.iters)
        ms = time_ms(both, args.iters)
        yv = torch.view_as_complex(out).to(torch.complex128)
        xv = torch.view_as_complex(x[off: off + Fs * D]).to(torch.complex128)
        db = 10 * math.log10(float((yv - xv).abs().pow(2).sum() / xv.abs().pow(2).sum()))
        assert db <= -80, f"round trip reconstruction {db:.1f} dB"
        print(json.dumps({"name": "roundtrip_R", "M": M, "D": D, "ntaps_analysis": h.size, "ntaps_synthesis": g.size,
                          "kernels": "pfb_chan_kernel + pfb_synth_kernel", "out_samples": Fs * D, "ms": round(ms, 4),
                          "msamples_per_s": round(Fs * D / ms / 1e3, 1), "synth_ms": round(ms_s, 4),
                          "synth_msamples_per_s": round(Fs * D / ms_s / 1e3, 1), "reconstruction_db": round(db, 2),
                          "device": name, "power_limit": power}), flush=True)
        del x, mid, out, ch, sy
        torch.cuda.empty_cache()
    for cfg in args.torch_configs:
        M, D, ntaps = CONFIGS[cfg]
        K = -(-ntaps // D)
        g = prototype(M, D, ntaps)
        pf = max(4, min(64, (1 << 24) // (M * D * (K + 1))))
        worst = parity(lambda X, s, F: torch_synth(X, g, M, D, s, F), g, M, D, pf)
        F = n_out // D
        X = torch.randn((M, F + K - 1, 2), device="cuda")
        ms = time_ms(lambda: torch_synth(X, g, M, D, 0, F), max(3, args.iters // 2), warmup=1)
        samples = F * D
        msps = samples / ms / 1e3
        print(json.dumps({"name": f"synth_{cfg}_torch_ops", "M": M, "D": D, "ntaps": ntaps, "kernel": "torch.fft.ifft + strided sum",
                          "out_samples": samples, "ms": round(ms, 4), "msamples_per_s": round(msps, 1),
                          "synthesizer_speedup": round(rates[cfg] / msps, 1) if cfg in rates else None,
                          "parity_frames": pf, "parity_max_err_rel": worst, "device": name, "power_limit": power}), flush=True)
        del X
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
