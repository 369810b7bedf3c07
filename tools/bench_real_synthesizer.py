#!/usr/bin/env python
"""Stream rate of the real-output polyphase synthesis filter bank (b200c_rsynth_run): one JSON line per config and
output type, a RealChannelizer -> RealSynthesizer round trip (config R) with its reconstruction error, and one line
per config A, B and D done the way it had to be done before: torch builds the conjugate-symmetric extension of the
M/2 + 1 rows, the complex Synthesizer runs at M channels, and the real part is copied out, timed as one unit.

Outputs are 2^28 real samples per line (1 GiB float32, 512 MiB int16, far larger than L2); CUDA-event timing over
--iters launches after warm-up.  Algorithmic traffic per output sample: 4 B (float32) or 2 B (int16) written plus
8 (M/2 + 1) / D B of rows read; flops per input frame: 5 (M/2) log2(M/2) (one M/2-point complex inverse FFT) + 7 M/2
(the pre-pass: per pair (k, M/2 - k) two complex sums, one complex product and four adds) + 2 ntaps (real taps x real
bins).  Every line carries a parity check of seeded frames against the reference (tests/_rsynth_oracle.py) at 1e-5 of
RMS per block of 64 D samples, so a fast but wrong kernel cannot report a number."""
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

from _rsynth_oracle import synthesize_real  # noqa: E402
from _synth_oracle import roundtrip_taps  # noqa: E402
from pothoscomms_b200 import RealChannelizer, RealSynthesizer, Synthesizer  # noqa: E402

# name: (M, interpolation D, ntaps, output types): the real channelizer's configs (tools/bench_real_channelizer.py)
CONFIGS = {"A": (2048, 2048, 16384, ("float32", "int16")), "B": (2048, 1024, 16384, ("float32",)),
           "C": (8192, 8192, 131072, ("float32",)), "D": (128, 128, 2048, ("float32",))}
WORKAROUND = "ABD"   # C has M > 4096, beyond the complex Synthesizer


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


def parity(run, g, M, D, frames, scale=1.0):
    """run(X, s, F) -> [F D] output on seeded rows [M/2 + 1, K-1 + F, 2]; checked against the reference.  int16
    output is checked against the rounded, saturated reference.  Returns the worst block's err/rms."""
    K = -(-len(g) // D)
    N = M // 2
    rng = np.random.default_rng(M * 131 + D)
    X = (scale * (rng.standard_normal((N + 1, K - 1 + frames)) + 1j * rng.standard_normal((N + 1, K - 1 + frames))))
    X = X.astype(np.complex64)
    s = 2**40 + 7
    y = run(torch.from_numpy(X.view(np.float32).reshape(N + 1, -1, 2)).cuda(), s, frames).cpu().numpy().astype(np.float64)
    ref = synthesize_real(X, g, M, D, s)
    assert y.shape == ref.shape
    blk, worst = 64 * D, 0.0
    for b0 in range(0, ref.size, blk):
        e, r = y[b0: b0 + blk], ref[b0: b0 + blk]
        worst = max(worst, float(np.sqrt(np.mean((e - r) ** 2)) / np.sqrt(np.mean(r ** 2))))
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


def kernel_run(rs, D, dtype):
    def run(X, s, F):
        out = torch.empty(F * D, dtype=getattr(torch, dtype), device="cuda")
        c, p = rs.run(X, out, s)
        torch.cuda.synchronize()
        assert (c, p) == (F, F * D)
        return out
    return run


def extend_synth_real(sy, M, D):
    """The workaround: rows M - c = conj(row c), rows 0 and M/2 made real, the complex synthesizer, the real part."""
    N = M // 2

    def run(X, s, F, out_c=None):
        full = torch.empty((M, X.shape[1], 2), dtype=torch.float32, device=X.device)
        full[: N + 1] = X
        full[0, :, 1] = 0
        full[N, :, 1] = 0
        full[N + 1:] = X[1:N].flip(0) * torch.tensor([1.0, -1.0], device=X.device)
        out_c = torch.empty((F * D, 2), dtype=torch.float32, device=X.device) if out_c is None else out_c
        c, p = sy.run(full, out_c, s)
        assert (c, p) == (F, F * D)
        return out_c[:, 0].contiguous()
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="ABCDR")
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
        M, D, ntaps, dtypes = CONFIGS[cfg]
        N = M // 2
        K = -(-ntaps // D)
        g = prototype(M, D, ntaps)
        pf = max(4, min(64, (1 << 25) // ((N + 1) * D * (K + 2))))   # the reference costs (M/2 + 1) D (K + 2) per frame
        F = n_out // D
        X = torch.randn((N + 1, F + K - 1, 2), device="cuda")
        samples = F * D
        flops = (5 * N * math.log2(N) + 7 * N + 2 * ntaps) * (F + K - 1)
        for dtype in dtypes:
            rs = RealSynthesizer(dtype, M, D)
            rs.set_taps(g)
            # int16: rows scaled so the output spans about +-3000, rounded and saturated by the kernel
            worst = parity(kernel_run(rs, D, dtype), g, M, D, pf) if dtype == "float32" else None
            if dtype == "int16":
                r32 = RealSynthesizer("float32", M, D)
                r32.set_taps(g)
                Xp = torch.randn((N + 1, K - 1 + pf, 2), device="cuda") * 30
                y16 = kernel_run(rs, D, dtype)(Xp, 5, pf).cpu().numpy()
                y32 = kernel_run(r32, D, "float32")(Xp, 5, pf).cpu().numpy()
                assert np.array_equal(y16, np.clip(np.rint(y32), -32768, 32767)), "int16 output != rounded float32 output"
                worst = parity(lambda Xi, s, Fi: kernel_run(r32, D, "float32")(Xi, s, Fi), g, M, D, pf)
                del r32
            out = torch.empty(samples, dtype=getattr(torch, dtype), device="cuda")
            ms = time_ms(lambda: rs.run(X, out, 0), args.iters)
            nbytes = out.element_size() * samples + 8 * (N + 1) * (F + K - 1)
            gbs = nbytes / ms / 1e6
            rates[(cfg, dtype)] = samples / ms / 1e3
            print(json.dumps({"name": f"rsynth_{cfg}_{dtype}", "M": M, "D": D, "ntaps": ntaps, "dtype": dtype,
                              "kernel": "pfb_rsynth_kernel", "out_samples": samples, "ms": round(ms, 4),
                              "msamples_per_s": round(rates[(cfg, dtype)], 1), "bytes": nbytes, "gbs": round(gbs, 1),
                              "hbm_frac": round(gbs / peak, 4), "peak_gbs": peak, "peak_kind": peak_kind,
                              "tflops": round(flops / ms / 1e9, 2), "flop_per_byte": round(flops / nbytes, 2),
                              "parity_frames": pf, "parity_max_err_rel": worst,
                              "parity_int16": "bit-identical to rounded float32" if dtype == "int16" else None,
                              "device": name, "power_limit": power}), flush=True)
            del out, rs
            torch.cuda.empty_cache()
        if cfg in WORKAROUND:
            sy = Synthesizer("complex_float32", M, D)
            sy.set_taps(g)
            run = extend_synth_real(sy, M, D)
            worst = parity(lambda Xi, s, Fi: run(Xi, s, Fi), g, M, D, pf)
            out_c = torch.empty((samples, 2), dtype=torch.float32, device="cuda")
            ms = time_ms(lambda: run(X, 0, F, out_c), args.iters)
            msps = samples / ms / 1e3
            print(json.dumps({"name": f"rsynth_{cfg}_float32_as_extend_plus_synthesizer", "M": M, "D": D, "ntaps": ntaps,
                              "kernel": "torch extension + pfb_synth_kernel + real-part copy", "out_samples": samples,
                              "ms": round(ms, 4), "msamples_per_s": round(msps, 1),
                              "real_synthesizer_speedup": round(rates[(cfg, "float32")] / msps, 2),
                              "parity_frames": pf, "parity_max_err_rel": worst, "device": name, "power_limit": power}),
                  flush=True)
            del out_c, sy
            torch.cuda.empty_cache()
        del X
        torch.cuda.empty_cache()
    if "R" in args.configs:
        # RealChannelizer -> RealSynthesizer on one stream, D = M/2, the reconstruction recipe of INTEGRATION §1
        M = 2048
        D = M // 2
        h, g, s_shift, off = roundtrip_taps(M)
        ch = RealChannelizer("float32", M, D)
        ch.set_taps(h)
        rs = RealSynthesizer("float32", M, D)
        rs.set_taps(g)
        Kg = rs.info()[4]
        Fa = n_out // D
        x = torch.from_numpy(np.random.default_rng(1).standard_normal(h.size - 1 + Fa * D).astype(np.float32)).cuda()
        mid = torch.empty((M // 2 + 1, Fa, 2), dtype=torch.float32, device="cuda")
        Fs = Fa - (Kg - 1)
        out = torch.empty(Fs * D, dtype=torch.float32, device="cuda")
        s_a = 2**40 + 3

        def both():
            ch.run(x, mid, s_a)
            rs.run(mid, out, s_a + s_shift)
        ms = time_ms(both, args.iters)
        ms_s = time_ms(lambda: rs.run(mid, out, s_a + s_shift), args.iters)
        y = out.to(torch.float64)
        ref = x[off: off + Fs * D].to(torch.float64)
        db = 10 * math.log10(float((y - ref).pow(2).sum() / ref.pow(2).sum()))
        assert db <= -80, f"round trip reconstruction {db:.1f} dB"
        print(json.dumps({"name": "rsynth_roundtrip_R", "M": M, "D": D, "ntaps_analysis": h.size, "ntaps_synthesis": g.size,
                          "K": Kg, "kernels": "pfb_rchan_kernel + pfb_rsynth_kernel", "out_samples": Fs * D,
                          "ms": round(ms, 4), "msamples_per_s": round(Fs * D / ms / 1e3, 1), "rsynth_ms": round(ms_s, 4),
                          "rsynth_msamples_per_s": round(Fs * D / ms_s / 1e3, 1), "reconstruction_db": round(db, 2),
                          "device": name, "power_limit": power}), flush=True)
        del x, mid, out, ch, rs
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
