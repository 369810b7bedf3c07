"""Float64 reference for the FIR filter bank at L = M = 1: every channel's /comms/fir_filter output by FFT
convolution in complex128 (torch.fft), on whichever device the input is on.

The convention is the reference block's (filter/FIRFilter.cpp:286-302, oracle.fir): the input holds K-1
history samples then the new ones, and

    y[n] = sum_k h[k] x[n + K-1-k],   n = 0 .. n_in - K

plus K-1 more outputs with ``zero_tail`` (the burst flush: K-1 zeros appended).  That is the full linear
convolution c = h * x from index K-1 on, so one FFT convolution gives both.  tests/test_bank_ref_cpu.py
pins this module to oracle.fir; resampling and the integer types are checked against oracle.fir itself.

The work goes in chunks of channels (about 512 MiB of transform per chunk), so a bank of 1024 channels of
2^20 samples is checked a chunk at a time without holding its whole complex128 result.
"""
from __future__ import annotations

import numpy as np
import torch

CHUNK_BYTES = 1 << 29   # complex128 transform elements per chunk: 2^25


def fir_count(n_in: int, ntaps: int, zero_tail: bool = False, n_out: int | None = None) -> int:
    """Outputs one work() call produces at L = M = 1 (filter/FIRFilter.cpp:286-292)."""
    elems = n_in + (ntaps - 1 if zero_tail else 0)
    n = elems - (ntaps - 1) if elems >= ntaps else 0
    return n if n_out is None else min(n, n_out)


def _fft_len(n: int) -> int:
    return 1 << max(0, (n - 1).bit_length())


def _as_tensor(a, device) -> torch.Tensor:
    if isinstance(a, torch.Tensor):
        return a.to(device)
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def fir_ref(x, taps, zero_tail: bool = False, n_out: int | None = None) -> torch.Tensor:
    """x: [nchan, n_in] (or [n_in]) complex tensor or array, K-1 history samples first; taps: [K] shared by every
    channel or [nchan, K], real or complex.  Returns complex128 [nchan, n] (or [n]) on x's device, n = fir_count()."""
    if not isinstance(x, torch.Tensor):
        x = _as_tensor(x, "cpu")
    one = x.dim() == 1
    if one:
        x = x.unsqueeze(0)
    h = _as_tensor(taps, x.device).to(torch.complex128)
    if h.dim() == 1:
        h = h.unsqueeze(0).expand(x.shape[0], -1)
    assert h.shape[0] == x.shape[0], "one tap row per channel"
    nch, n_in = x.shape
    K = h.shape[1]
    n = fir_count(n_in, K, zero_tail, n_out)
    y = torch.empty((nch, n), dtype=torch.complex128, device=x.device)
    if n:
        L = _fft_len(n_in + K - 1)
        step = max(1, CHUNK_BYTES // (16 * L))
        for c0 in range(0, nch, step):
            c1 = min(nch, c0 + step)
            X = torch.fft.fft(x[c0:c1].to(torch.complex128), n=L, dim=1)
            X *= torch.fft.fft(h[c0:c1], n=L, dim=1)
            y[c0:c1] = torch.fft.ifft(X, n=L, dim=1)[:, K - 1:K - 1 + n]
            del X
    return y[0] if one else y
