"""Pins tests/_stream_ref.py (the float64 single-stream reference the long-launch GPU tests compare every output
with) to oracle.fir, the C restatement of the reference block, on the CPU.

A slip in the polyphase bookkeeping -- a phase's taps taken from the wrong residue, its sample offset d_p off by one,
K rounded the wrong way, the zero tail or the output capacity counted differently, a seam between chunks -- fails
here instead of being copied into the GPU checks.  float64 data is exact in the reference's complex128 transforms,
so it is pinned to the float64 oracle at 1e-12 of the output RMS; the counts must match exactly.
"""
import numpy as np
import pytest
import torch

import _stream_ref
from _stream_ref import stream_count, stream_ref

TOL = 1e-12   # of the output RMS

RATES = [(M, L) for M in range(1, 5) for L in range(1, 5)] + [(16, 1), (1, 8)]
DATA = [("CF64", "COMPLEX"), ("CF64", "REAL"), ("F64", "REAL")]


def _taps(rng, ntaps, complex_taps):
    h = rng.standard_normal(ntaps) / np.sqrt(ntaps)
    if complex_taps:
        h = h + 1j * rng.standard_normal(ntaps) / np.sqrt(ntaps)
    return h


def _oracle(oracle, code, complex_taps, h, M, L, x, zero_tail, cap):
    raw = oracle.to_raw(x, code)
    y, cons, prod = oracle.fir(code, complex_taps, h, M, L, raw, out_capacity=cap, zero_tail=zero_tail)
    y = y.astype(np.float64)
    return (y[:, 0] + 1j * y[:, 1] if y.shape[1] == 2 else y[:, 0].astype(np.complex128)), cons, prod


def _close(got, ref, what):
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    if ref.size == 0:
        return
    rms = np.sqrt(np.mean(np.abs(ref) ** 2))
    err = np.sqrt(np.mean(np.abs(got - ref) ** 2))
    assert err <= TOL * rms, f"{what}: rel rms err {err / rms:.3e} > {TOL}"


@pytest.mark.parametrize("M,L", RATES, ids=[f"M{m}-L{l}" for m, l in RATES])
@pytest.mark.parametrize("code_name,taps_type", DATA, ids=[f"{d}-{t}" for d, t in DATA])
def test_stream_ref_matches_oracle(oracle, code_name, taps_type, M, L):
    """Tap counts with the last phase one tap short, exactly K L taps and fewer taps than phases; ragged block
    counts; the zero tail; capacities ending inside a block (not a multiple of L) and below one block."""
    code = getattr(oracle, code_name)
    cx_taps, cx_data = taps_type == "COMPLEX", code & 1 == 1
    rng = np.random.default_rng(1000 * M + 10 * L + 3 * cx_taps + cx_data)
    for ntaps in sorted({7 * L - 1, 7 * L, 37, max(1, L - 1)} - {0}):
        h = _taps(rng, ntaps, cx_taps)
        K = -(-ntaps // L)
        for n_new in (M - 1, M, 5 * M + 1, 3001):
            n_in = K - 1 + n_new
            x = rng.standard_normal(n_in) + (1j * rng.standard_normal(n_in) if cx_data else 0)
            for zero_tail in (False, True):
                blocks = stream_count(n_in, ntaps, M, L, zero_tail)[1] // L
                for cap in (None, (blocks // 2) * L + L - 1, L - 1):
                    what = f"{code_name}/{taps_type} M={M} L={L} K={ntaps} n_new={n_new} zt={zero_tail} cap={cap}"
                    y, cons, prod = stream_ref(x, h, M, L, zero_tail, cap)
                    assert y.dtype == torch.complex128 and y.device.type == "cpu", what
                    ref, c_ref, p_ref = _oracle(oracle, code, cx_taps, h, M, L, x, zero_tail, cap)
                    assert (cons, prod) == (c_ref, p_ref), what
                    _close(y.numpy(), ref, what)


@pytest.mark.parametrize("M,L,ntaps", [(1, 1, 255), (2, 3, 255), (3, 2, 64), (1, 5, 600), (4, 4, 255), (2, 1, 33)])
def test_stream_ref_over_many_chunks(oracle, monkeypatch, M, L, ntaps):
    """Chunks of a few hundred blocks: every seam between chunks (and a zero tail split across the last one) is exact."""
    monkeypatch.setattr(_stream_ref, "CHUNK_BYTES", 16 * 4096)
    rng = np.random.default_rng(77 + M + 7 * L)
    h = _taps(rng, ntaps, True)
    K = -(-ntaps // L)
    n_in = K - 1 + 20000 * M + 3
    x = rng.standard_normal(n_in) + 1j * rng.standard_normal(n_in)
    for zero_tail in (False, True):
        y, cons, prod = stream_ref(torch.from_numpy(x), torch.from_numpy(h), M, L, zero_tail)
        ref, c_ref, p_ref = _oracle(oracle, oracle.CF64, True, h, M, L, x, zero_tail, None)
        assert (cons, prod) == (c_ref, p_ref)
        _close(y.numpy(), ref, f"M={M} L={L} K={ntaps} zt={zero_tail} in chunks")


def test_stream_ref_float32_input_and_nothing_to_produce(oracle):
    """complex64 / float32 tensors go in as they are (converted exactly); below input_require nothing comes out."""
    rng = np.random.default_rng(5)
    h = _taps(rng, 40, False)
    x = (rng.standard_normal(2000) + 1j * rng.standard_normal(2000)).astype(np.complex64)
    y, _, _ = stream_ref(torch.from_numpy(x), h, 2, 3)
    ref, _, _ = _oracle(oracle, oracle.CF64, False, h, 2, 3, x.astype(np.complex128), False, None)
    _close(y.numpy(), ref, "complex64 input")
    xr = rng.standard_normal(2000).astype(np.float32)
    y, _, _ = stream_ref(torch.from_numpy(xr), h, 1, 1)
    ref, _, _ = _oracle(oracle, oracle.F64, False, h, 1, 1, xr.astype(np.float64), False, None)
    _close(y.numpy(), ref, "float32 input")
    K = -(-40 // 3)
    for n_in, zt in ((K - 1, False), (K, False), (K + 1, False), (0, True), (1, True)):
        y, cons, prod = stream_ref(x[:n_in], h, 2, 3, zt)
        _, c_ref, p_ref = _oracle(oracle, oracle.CF64, False, h, 2, 3, x[:n_in].astype(np.complex128), zt, None)
        assert (cons, prod) == (c_ref, p_ref) and y.shape == (prod,), (n_in, zt)
