"""Reference of the polyphase synthesizer (b200c_synth_run) in numpy float64, and the channelizer -> synthesizer
perfect-reconstruction recipe.

Test infrastructure only, like the oracle package: tests/test_oracle_synthesizer.py pins synthesize() to oracle.fir,
numpy mixing and a sum; tests/test_synthesizer_gpu.py and tools/bench_synthesizer.py check the kernel against it.  It
evaluates the definition as per-channel FIRs and a dense exponential mix, with no FFT, so it shares none of the
kernel's algebra."""
from __future__ import annotations

import numpy as np


def synthesize(X, g, M: int, D: int, stream_index: int = 0, samples: int | None = None) -> np.ndarray:
    """b200c_synth_run's definition in float64: each channel through the polyphase FIR (real taps g, interpolation D),
    then a dense exponential mix and the sum over channels (no FFT, none of the kernel's algebra).  ``X``: [M, n]
    complex channel frames (or raw [M, n, 2]), the first K-1 of them history, K = ceil(ntaps / D).
        y[t D + j] = sum_c exp(+2 pi i c (s + t D + j) / M) sum_{k < K} g[j + k D] X[c, K-1 + t - k],   s = stream_index.
    Returns y [F D] complex128 with F = n - (K-1) (or fewer, if ``samples`` // D is fewer; 0 when n < K)."""
    X = np.asarray(X)
    if not np.iscomplexobj(X):
        X = np.ascontiguousarray(X, dtype=np.float64).reshape(M, -1, 2)
        X = X[..., 0] + 1j * X[..., 1]
    X = X.astype(np.complex128).reshape(M, -1)
    g = np.asarray(g, dtype=np.float64).ravel()
    K = -(-g.size // D)
    gp = np.zeros(K * D)
    gp[:g.size] = g
    gp = gp.reshape(K, D)                                 # gp[k, j] = g[j + k D]
    n = X.shape[1]
    F = n - (K - 1) if n >= K else 0
    if samples is not None:
        F = min(F, int(samples) // D)
    y = np.zeros(F * D, dtype=np.complex128)
    E = np.exp(2j * np.pi * np.arange(M) / M)             # E[k] = exp(+2 pi i k / M), k < M
    c = np.arange(M, dtype=np.int64)[:, None, None]
    j = np.arange(D, dtype=np.int64)[None, None, :]
    s = int(stream_index) % M                             # only s mod M enters the exponent (exactly)
    chunk = max(1, (1 << 22) // (M * D))                  # frames per step: bounds the dense arrays to ~64 MiB
    for t0 in range(0, F, chunk):
        t1 = min(F, t0 + chunk)
        U = np.zeros((M, t1 - t0, D), dtype=np.complex128)   # U[c, t, j]: channel c's interpolating FIR output
        for k in range(K):
            U += X[:, K - 1 + t0 - k: K - 1 + t1 - k, None] * gp[k][None, None, :]
        t = np.arange(t0, t1, dtype=np.int64)[None, :, None]
        ph = (c * ((s + t * D + j) % M)) % M              # exponent index of each (c, t, j), reduced exactly
        y[t0 * D: t1 * D] = (E[ph] * U).sum(axis=0).ravel()
    return y


def roundtrip_taps(M):
    """The perfect-reconstruction recipe at D = M/2: analysis h (a Nyquist(M) filter), synthesis g flat over h's band
    and stopping before the first image at 2/M, and the lag between the channelizer's input and the output."""
    from scipy import signal
    D = M // 2
    h = signal.firwin(12 * M + 1, 1.0 / M, window=("kaiser", 10.0))
    g = D * signal.firwin(28 * D + 1, 2.0 / M, window=("kaiser", signal.kaiser_beta(90.0)))
    Kg = -(-g.size // D)
    s_shift = (h.size - 1) + (D - 1) + (Kg - 1) * D          # synthesizer stream_index = channelizer's + s_shift
    off = (h.size - 1) // 2 + (D - 1) + (Kg - 1) * D - (g.size - 1) // 2
    return h, g, s_shift, off
