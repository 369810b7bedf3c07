"""Reference of the real-output polyphase synthesizer (b200c_rsynth_run) in numpy float64.

Test infrastructure only, like tests/_synth_oracle.py: tests/test_oracle_real_synthesizer.py pins synthesize_real() to
the complex synthesizer's reference on the conjugate-symmetric extension; tests/test_real_synthesizer_gpu.py and
tools/bench_real_synthesizer.py check the kernel against it.  It evaluates the weighted-real definition as per-row
FIRs and a dense cosine/sine mix, with no FFT, so it shares none of the kernel's algebra (no packed half-size
transform, no even/odd split)."""
from __future__ import annotations

import numpy as np


def synthesize_real(X, g, M: int, D: int, stream_index: int = 0, samples: int | None = None) -> np.ndarray:
    """b200c_rsynth_run's definition in float64.  ``X``: [M/2 + 1, n] complex rows c = 0 .. M/2 (or raw
    [M/2 + 1, n, 2]), the first K-1 frames history, K = ceil(ntaps / D).  With N = M/2 and s = stream_index,
        y[t D + j] = sum_{k < K} g[j + k D] sum_{c = 0..N} w_c Re(exp(+2 pi i c (s + t D + j) / M) X[c, K-1 + t - k]),
        w_0 = w_N = 1, w_c = 2 otherwise.
    Returns y [F D] float64 with F = n - (K-1) (or fewer, if ``samples`` // D is fewer; 0 when n < K)."""
    assert M >= 2 and M & (M - 1) == 0
    N = M // 2
    X = np.asarray(X)
    if not np.iscomplexobj(X):
        X = np.ascontiguousarray(X, dtype=np.float64).reshape(N + 1, -1, 2)
        X = X[..., 0] + 1j * X[..., 1]
    X = X.astype(np.complex128).reshape(N + 1, -1).copy()
    X[0] = X[0].real                                      # exp(+2 pi i c m / M) is exactly +-1 for rows 0 and N:
    X[N] = X[N].real                                      # only their real parts enter
    g = np.asarray(g, dtype=np.float64).ravel()
    K = -(-g.size // D)
    gp = np.zeros(K * D)
    gp[:g.size] = g
    gp = gp.reshape(K, D)                                 # gp[k, j] = g[j + k D]
    n = X.shape[1]
    F = n - (K - 1) if n >= K else 0
    if samples is not None:
        F = min(F, int(samples) // D)
    y = np.zeros(F * D, dtype=np.float64)
    ang = 2 * np.pi * np.arange(M) / M
    C, S = np.cos(ang), np.sin(ang)                       # exp(+2 pi i k / M) = C[k] + i S[k], k < M
    wgt = np.full((N + 1, 1), 2.0)
    wgt[0] = wgt[N] = 1.0
    c = np.arange(N + 1, dtype=np.int64)[:, None]
    j = np.arange(D, dtype=np.int64)[None, :]
    s = int(stream_index) % M                             # only s mod M enters the exponent (exactly)
    mixes = {}                                            # the mix of frame t depends on u = (s + t D) mod M only

    def mix(u):
        if u not in mixes:
            ph = (c * ((u + j) % M)) & (M - 1)            # exponent index of each (c, j), reduced exactly (M = 2^n)
            mixes[u] = (wgt * C[ph], wgt * S[ph])
        return mixes[u]

    chunk = max(1, (1 << 22) // ((N + 1) * D))            # frames per step: bounds the dense arrays to ~64 MiB
    for t0 in range(0, F, chunk):
        t1 = min(F, t0 + chunk)
        # Xw[c, t, k] = X[c, K-1 + t - k]; U[c, t, j] = sum_k Xw[c, t, k] gp[k, j]: row c's interpolating FIR output
        Xw = np.lib.stride_tricks.sliding_window_view(X[:, t0: t1 + K - 1], K, axis=1)[:, :, ::-1]
        Ur = Xw.real @ gp
        Ui = Xw.imag @ gp
        for t in range(t0, t1):
            wc, ws = mix((s + t * D) % M)                 # y = sum_c w_c (cos * Re U - sin * Im U)
            y[t * D: (t + 1) * D] = np.einsum("cj,cj->j", wc, Ur[:, t - t0]) - np.einsum("cj,cj->j", ws, Ui[:, t - t0])
    return y


def symmetric_extension(X, M: int):
    """[M/2 + 1, n] rows -> [M, n] rows of the complex synthesizer: rows 0 and M/2 with their real parts only, and
    row M - c = conj(row c) for 0 < c < M/2."""
    assert M >= 2 and M & (M - 1) == 0
    N = M // 2
    X = np.asarray(X).astype(np.complex128)
    full = np.empty((M, X.shape[1]), dtype=np.complex128)
    full[: N + 1] = X
    full[0] = X[0].real
    full[N] = X[N].real
    if N > 1:
        full[N + 1:] = np.conj(X[1:N][::-1])
    return full
