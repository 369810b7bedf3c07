"""Float64 reference for one /comms/fir_filter stream at any decimation M and interpolation L: FFT convolution in
complex128 (torch.fft), on whichever device the input is on, a chunk of the stream at a time.

The convention is the reference block's (filter/FIRFilter.cpp:286-302, oracle.fir): the input holds K-1 history
samples then the new ones, K = ceil(ntaps / L), and output slot p of input block q is

    y[q L + p] = sum_k taps[j_p + k L] x[q M + d_p + K-1 - k],   j_p = ((p+1) M - 1) mod L,  d_p = ((p+1) M - 1) div L

(the polyphase form of csrc/fir.hpp and fir_ummap_configure).  So slot p is the full linear convolution of x with
phase p's taps, sampled at q M + d_p + K-1: one FFT convolution per slot.  A work() call takes N/M blocks,
N = min((elems - (K-1)) div M, out_capacity div L) M, where ``elems`` counts the K-1 zeros the burst flush
(``zero_tail``) appends; it consumes N and produces N/M L.  tests/test_stream_ref_cpu.py pins this module to
oracle.fir.  At L = M = 1 each chunk goes through _bank_ref.fir_ref.
"""
from __future__ import annotations

import numpy as np
import torch

from _bank_ref import fir_ref

CHUNK_BYTES = 1 << 29   # complex128 transform elements per chunk (all L slots): 2^25


def stream_count(n_in: int, ntaps: int, M: int = 1, L: int = 1, zero_tail: bool = False,
                 out_capacity: int | None = None):
    """(consumed, produced) of one work() call; out_capacity None: the oracle's default, room for every block."""
    K = -(-ntaps // L)
    elems = n_in + (K - 1 if zero_tail else 0)
    cap = (elems // M + 1) * L if out_capacity is None else out_capacity
    nb = min(max(elems - (K - 1), 0) // M, cap // L)
    return nb * M, nb * L


def _fft_len(n: int) -> int:
    return 1 << max(0, (n - 1).bit_length())


def stream_ref(x, taps, M: int = 1, L: int = 1, zero_tail: bool = False, out_capacity: int | None = None):
    """x: [n_in] complex or real tensor (or array), K-1 history samples first; taps: [ntaps] real or complex.
    Returns (y complex128 [produced] on x's device, consumed, produced)."""
    if not isinstance(x, torch.Tensor):
        x = torch.from_numpy(np.ascontiguousarray(x))
    assert x.dim() == 1, "one stream"
    dev = x.device
    h = (taps.to(dev) if isinstance(taps, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(taps)).to(dev))
    h = h.to(torch.complex128)
    ntaps = h.shape[0]
    K = -(-ntaps // L)
    n_in = x.shape[0]
    cons, prod = stream_count(n_in, ntaps, M, L, zero_tail, out_capacity)
    nb = cons // M
    y = torch.empty((prod,), dtype=torch.complex128, device=dev)
    if nb == 0:
        return y, cons, prod
    # phase p's taps h_p[k] = taps[j_p + k L] and its sample offset d_p
    j = [((p + 1) * M - 1) % L for p in range(L)]
    d = [((p + 1) * M - 1) // L for p in range(L)]
    hp = torch.zeros((L, K), dtype=torch.complex128, device=dev)
    for p in range(L):
        ph = h[j[p]::L]
        hp[p, :ph.shape[0]] = ph
    # chunk of blocks [q0, q1): it reads x[q0 M, q1 M + K - 1) (d_p <= M - 1); a circular transform of at least that
    # length is exact at the sampled indices (each >= K - 1, so no term wraps)
    nf = _fft_len(min(nb * M + K - 1, max(CHUNK_BYTES // (16 * L), 4 * (K + M))))
    per = (nf - (K - 1)) // M
    idx = torch.arange(per, device=dev) * M
    for q0 in range(0, nb, per):
        q1 = min(nb, q0 + per)
        a, b = q0 * M, q1 * M + K - 1
        xs = torch.zeros((b - a,), dtype=torch.complex128, device=dev)
        have = max(0, min(b, n_in) - a)
        xs[:have] = x[a:a + have].to(torch.complex128)                 # past n_in: the zero tail
        if L == 1 and M == 1:
            y[q0:q1] = fir_ref(xs, hp[0])
            continue
        c = torch.fft.ifft(torch.fft.fft(xs, n=nf) * torch.fft.fft(hp, n=nf, dim=1), dim=1)
        for p in range(L):
            y[q0 * L + p:q1 * L:L] = c[p, idx[:q1 - q0] + d[p] + K - 1]
        del c
    return y, cons, prod
