"""Pins tests/_bank_ref.py (the float64 FFT-convolution reference the filter-bank GPU tests compare every
channel with) to oracle.fir, the C restatement of the reference block, on the CPU.

A convention slip in fir_ref -- taps reversed, history offset by one, the zero tail or the output capacity
handled differently -- fails here instead of being copied into the GPU checks.  Complex float32 data is
exact in float64, so its reference is pinned to the float64 oracle at the same 1e-12; the float32 oracle
(float accumulation) agrees to float32 precision.
"""
import numpy as np
import pytest
import torch

from _bank_ref import fir_count, fir_ref

TOL = 1e-12   # of the output RMS


def _taps(rng, ntaps, complex_taps):
    h = rng.standard_normal(ntaps) / np.sqrt(ntaps)
    if complex_taps:
        h = h + 1j * rng.standard_normal(ntaps) / np.sqrt(ntaps)
    return h


def _oracle(oracle, code, complex_taps, h, x, zero_tail, n_out):
    """oracle.fir on one channel x (complex numpy), output as complex128."""
    raw = oracle.to_raw(x, code)
    y, cons, prod = oracle.fir(code, complex_taps, h, 1, 1, raw, out_capacity=n_out, zero_tail=zero_tail)
    return y[:, 0].astype(np.float64) + 1j * y[:, 1].astype(np.float64), cons, prod


def _close(got, ref, tol, what):
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    if ref.size == 0:
        return
    rms = np.sqrt(np.mean(np.abs(ref) ** 2))
    err = np.sqrt(np.mean(np.abs(got - ref) ** 2))
    assert err <= tol * rms, f"{what}: rel rms err {err / rms:.3e} > {tol}"


@pytest.mark.parametrize("ntaps", [1, 2, 7, 64, 255, 1024, 2049])
@pytest.mark.parametrize("complex_taps", [False, True], ids=["real_taps", "complex_taps"])
@pytest.mark.parametrize("data", ["CF64", "CF32"])
def test_fir_ref_matches_oracle(oracle, ntaps, complex_taps, data):
    rng = np.random.default_rng(ntaps * 4 + 2 * complex_taps + (data == "CF32"))
    nch = 3
    h = np.stack([_taps(rng, ntaps, complex_taps) for _ in range(nch)])
    # ragged lengths: one new sample, a few, and an odd long run; the channels of a batch share a length
    for n_new in (1, 3, 4097, 10007):
        n_in = ntaps - 1 + n_new
        x = rng.standard_normal((nch, n_in)) + 1j * rng.standard_normal((nch, n_in))
        if data == "CF32":
            x = x.astype(np.complex64)
        for zero_tail in (False, True):
            for n_out in (None, max(1, n_new // 2)):
                what = f"{data} K={ntaps} n_new={n_new} zt={zero_tail} cap={n_out}"
                y = fir_ref(x, h, zero_tail=zero_tail, n_out=n_out).numpy()
                assert y.dtype == np.complex128
                for c in range(nch):
                    ref64, _, prod = _oracle(oracle, oracle.CF64, complex_taps, h[c], x[c].astype(np.complex128),
                                             zero_tail, n_out)
                    assert prod == fir_count(n_in, ntaps, zero_tail, n_out), what
                    _close(y[c], ref64, TOL, what + f" chan {c}")
                    if data == "CF32":
                        ref32, _, prod32 = _oracle(oracle, oracle.CF32, complex_taps, h[c], x[c], zero_tail, n_out)
                        assert prod32 == prod
                        _close(y[c], ref32, 1e-5, what + f" chan {c} (float32 oracle)")


def test_fir_ref_shapes_and_counts(oracle):
    """Shared taps broadcast over channels; one channel given as a vector; nothing to produce."""
    rng = np.random.default_rng(5)
    h = _taps(rng, 33, True)
    x = rng.standard_normal((4, 500)) + 1j * rng.standard_normal((4, 500))
    both = fir_ref(x, h)
    assert both.shape == (4, 500 - 32)
    np.testing.assert_array_equal(fir_ref(x[2], h).numpy(), both[2].numpy())
    np.testing.assert_array_equal(fir_ref(torch.from_numpy(x), torch.from_numpy(h)).numpy(), both.numpy())
    assert fir_ref(x[:, :32], h).shape == (4, 0)                  # below input_require
    assert fir_ref(x[:, :32], h, zero_tail=True).shape == (4, 32)
    assert fir_ref(x[:, :0], h, zero_tail=True).shape == (4, 0)
    for n_in, zt, cap in ((32, False, None), (33, False, None), (0, True, None), (1, True, None), (500, True, 7)):
        _, _, prod = oracle.fir(oracle.CF64, True, h, 1, 1, np.zeros((n_in, 2)), out_capacity=cap, zero_tail=zt)
        assert prod == fir_count(n_in, 33, zt, cap), (n_in, zt, cap)
