"""Pins the FFT oracle (CPU, no GPU needed).

1. the reference's own golden vectors (fft/TestFFT.cpp:19-29,55-56,79-80 float;
   :95-105,131-132,155-156 int16) against BOTH our restatement and oracle/_ref;
2. our restatement bit-for-bit against oracle/_ref (the reference's kiss_fft sources, built
   only from a PothosComms checkout: `make -C oracle REF=<checkout>`) over power-of-two,
   mixed-radix and prime sizes;
3. the committed fixtures in tests/golden/ (generated from oracle/_ref by make_golden.py).
"""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")

IN4 = np.array([0.4 + 0.6j, -0.7 + 0.6j, -0.2 + 0.8j, 0.9 + 0.2j])
OUT4 = np.array([0.4 + 2.2j, 1.0 + 1.4j, 0.0 + 0.6j, 0.2 - 1.8j])  # numpy.fft.fft(IN4), TestFFT.cpp:13-17


def _impls(oracle):
    impls = [("restated", oracle.fft)]
    if oracle.have_ref():
        impls.append(("reference", oracle.ref_fft))
    return impls


def test_golden_float_n4(oracle):
    x = oracle.to_raw(IN4.astype(np.complex64), oracle.CF32)
    for name, f in _impls(oracle):
        y = f(oracle.CF32, 4, False, x).view(np.complex64).ravel()
        assert np.all(np.abs(y.real - OUT4.real) < 0.01) and np.all(np.abs(y.imag - OUT4.imag) < 0.01), name
        # inverse is unnormalised: N * input (TestFFT.cpp:79-80)
        back = f(oracle.CF32, 4, True, oracle.to_raw(OUT4.astype(np.complex64), oracle.CF32)).view(np.complex64).ravel()
        assert np.all(np.abs(back - 4 * IN4) < 0.01), name


def test_golden_short_n4(oracle):
    xin = oracle.to_raw(np.round(IN4 * 1000), oracle.CI16)
    res = oracle.to_raw(np.round(OUT4 * 1000), oracle.CI16)
    for name, f in _impls(oracle):
        y = f(oracle.CI16, 4, False, xin)
        # forward == golden / N exactly (TestFFT.cpp:131-132: tol 0.01 on integers)
        assert np.array_equal(y, res // 4), name
        back = f(oracle.CI16, 4, True, res)
        assert np.array_equal(back, xin), name  # TestFFT.cpp:155-156


SIZES = [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 12, 15, 16, 25, 27, 30, 32, 49, 60, 64, 97, 100, 121, 125, 128, 242, 255,
         256, 343, 512, 1000, 1001, 1024, 2048, 3072, 4095, 4096, 5005]


@pytest.mark.parametrize("inverse", [False, True])
def test_restatement_matches_reference_bit_for_bit(oracle, inverse):
    if not oracle.have_ref():
        pytest.skip("no oracle/_ref")
    rng = np.random.default_rng(7)
    for n in SIZES:
        x = (rng.standard_normal((3 * n, 2))).astype(np.float32)
        a = oracle.fft(oracle.CF32, n, inverse, x)
        b = oracle.ref_fft(oracle.CF32, n, inverse, x)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"cf32 n={n}"
        xd = x.astype(np.float64)
        a = oracle.fft(oracle.CF64, n, inverse, xd)
        b = oracle.ref_fft(oracle.CF64, n, inverse, xd)
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), f"cf64 n={n}"
        xi = rng.integers(-32768, 32768, size=(3 * n, 2), dtype=np.int16)
        a = oracle.fft(oracle.CI16, n, inverse, xi)
        b = oracle.ref_fft(oracle.CI16, n, inverse, xi)
        assert np.array_equal(a, b), f"ci16 n={n}"


def test_plan_matches_reference_factorisation(oracle):
    # fft/kissfft.hh:38-55 / fft/kiss_fft.c:308-330: 4s first, then 2s, then 3,5,7...
    assert oracle.fft_plan(4096, False)[0] == [4] * 6
    assert oracle.fft_plan(2048, False)[0] == [4] * 5 + [2]
    assert oracle.fft_plan(1024, True)[0] == [4] * 5
    assert oracle.fft_plan(512, True)[0] == [4] * 4 + [2]
    assert oracle.fft_plan(60, False)[0] == [4, 3, 5]
    assert oracle.fft_plan(97, True)[0] == [97]


def test_float_fft_close_to_numpy(oracle):
    rng = np.random.default_rng(3)
    for n in (64, 1000, 4096):
        x = rng.standard_normal((n, 2)).astype(np.float32)
        y = oracle.fft(oracle.CF32, n, False, x).view(np.complex64).ravel()
        ref = np.fft.fft(x.view(np.complex64).ravel().astype(np.complex128))
        rel = np.sqrt(np.mean(np.abs(y - ref) ** 2) / np.mean(np.abs(ref) ** 2))
        assert rel < 2e-6


def test_committed_golden_fixtures(oracle):
    """tests/golden/fft_*.npz were produced by the reference's compiled sources."""
    files = sorted(f for f in os.listdir(GOLDEN) if f.startswith("fft_") and f.endswith(".npz"))
    assert files, "golden fixtures missing (tests/golden/make_golden.py)"
    for fn in files:
        g = np.load(os.path.join(GOLDEN, fn))
        dt, n, inv = int(g["dtype"]), int(g["n"]), bool(g["inverse"])
        y = oracle.fft(dt, n, inv, g["x"])
        assert np.array_equal(y.view(np.uint8), g["y"].view(np.uint8)), fn
