"""Direct-sum reference of the polyphase channelizer (b200c_chan_run), in numpy float64.

Test infrastructure only, like the oracle package: tests/test_oracle_channelizer.py pins it to numpy
mixing followed by oracle.fir, tests/test_channelizer_gpu.py and tools/bench_channelizer.py check the kernel against
it.  It evaluates the definition with a dense exponential matrix per frame and does NOT use the polyphase identity
the kernel is built on, so it shares none of the kernel's algebra."""
from __future__ import annotations

import numpy as np


def channelize(x, h, M: int, D: int, stream_index: int = 0, frames: int | None = None) -> np.ndarray:
    """b200c_chan_run's definition as a direct sum in float64 (a dense exponential matrix per frame; it does NOT
    use the polyphase identity the kernel is built on).  ``x``: complex samples (or raw [n, 2]), the first
    ntaps-1 of them history; ``h``: real prototype taps.  Frame t's newest sample is m_t = ntaps-1 + t D + D-1 and
        y[c, t] = sum_{n < ntaps} h[n] x[m_t - n] exp(-2 pi i c (s + m_t - n) / M),   s = stream_index.
    Returns y [M, F] complex128 with F = (len(x) - (ntaps-1)) // D (or ``frames``, if fewer)."""
    x = np.asarray(x)
    if not np.iscomplexobj(x):
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, 2)
        x = x[:, 0] + 1j * x[:, 1]
    x = x.astype(np.complex128).ravel()
    h = np.asarray(h, dtype=np.float64).ravel()
    ntaps = h.size
    F = max(0, (x.size - (ntaps - 1)) // D) if x.size >= ntaps - 1 + D else 0
    if frames is not None:
        F = min(F, int(frames))
    y = np.zeros((M, F), dtype=np.complex128)
    c = np.arange(M, dtype=np.int64)
    W = np.exp(-2j * np.pi * np.arange(M) / M)          # W[k] = exp(-2 pi i k / M), k < M
    n = np.arange(ntaps, dtype=np.int64)
    s = int(stream_index) % M                             # only s mod M enters the exponent (exactly)
    chunk = max(1, (1 << 22) // M)                        # bounds the dense matrix to ~64 MiB
    for t in range(F):
        m = ntaps - 1 + t * D + D - 1
        prod = h * x[m - n]                               # h[n] x[m_t - n]
        ph = (s + m - n) % M                              # exponent index of each tap, reduced exactly
        acc = np.zeros(M, dtype=np.complex128)
        for n0 in range(0, ntaps, chunk):
            E = W[np.outer(c, ph[n0:n0 + chunk]) % M]     # E[c, n] = exp(-2 pi i c (s + m_t - n) / M)
            acc += E @ prod[n0:n0 + chunk]
        y[:, t] = acc
    return y
