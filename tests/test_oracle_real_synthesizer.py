"""The real-output synthesizer's reference (tests/_rsynth_oracle.synthesize_real) against the complex synthesizer's
(tests/_synth_oracle.synthesize) on the conjugate-symmetric extension, the real channelizer -> real synthesizer
perfect-reconstruction recipe in float64, and the create-time argument checks of b200c_rsynth_create, which need no
device."""
import ctypes

import numpy as np
import pytest

from _chan_oracle import channelize
from _rsynth_oracle import symmetric_extension, synthesize_real
from _synth_oracle import roundtrip_taps, synthesize

CASES = [
    # (M, D, ntaps, stream_index)
    (2, 1, 5, 1),
    (2, 2, 1, 2**40 + 7),
    (4, 4, 1, 0),
    (8, 4, 21, 2**40 + 7),
    (16, 16, 16, 12345),
    (32, 8, 3 * 8 + 5, 3),
    (64, 32, 32 * 32, 2**40 + 7),
]


def _rows(M, n, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((M // 2 + 1, n)) + 1j * rng.standard_normal((M // 2 + 1, n))


@pytest.mark.parametrize("M,D,ntaps,s", CASES)
def test_real_part_of_complex_synthesizer_on_symmetric_extension(M, D, ntaps, s):
    K = -(-ntaps // D)
    X = _rows(M, K - 1 + 23, seed=100 * M + D + ntaps)
    g = np.random.default_rng(ntaps).standard_normal(ntaps)
    y = synthesize_real(X, g, M, D, s)
    full = synthesize(symmetric_extension(X, M), g, M, D, s)
    assert y.shape == (23 * D,)
    scale = max(1.0, np.abs(full).max())
    np.testing.assert_allclose(y, full.real, rtol=0, atol=1e-12 * scale)
    assert np.abs(full.imag).max() <= 1e-12 * scale          # the extension synthesizes a real stream
    # samples cuts the output to whole frames; the raw [rows, n, 2] float layout reads the same
    raw = np.stack([X.real, X.imag], axis=-1).astype(np.float64)
    np.testing.assert_array_equal(synthesize_real(raw, g, M, D, s, samples=5 * D + D // 2), y[: 5 * D])


@pytest.mark.parametrize("M,D,ntaps,s", CASES)
def test_imaginary_parts_of_edge_rows_never_enter(M, D, ntaps, s):
    K = -(-ntaps // D)
    X = _rows(M, K - 1 + 9, seed=7 * M + ntaps)
    g = np.random.default_rng(5).standard_normal(ntaps)
    Y = X.copy()
    Y[0] = X[0].real + 1j * 1e6
    Y[M // 2] = X[M // 2].real - 1j * 3e5
    np.testing.assert_array_equal(synthesize_real(Y, g, M, D, s), synthesize_real(X, g, M, D, s))


@pytest.mark.parametrize("M", [2, 8, 64])
def test_row_edges_give_constants_and_alternation(M):
    N, D, s = M // 2, M // 2 if M > 2 else 1, 2**40 + 7
    n = 40
    X = np.zeros((N + 1, n), dtype=np.complex128)
    X[0] = 0.5
    g = np.ones(D)                                           # one unit tap per output phase
    y0 = synthesize_real(X, g, M, D, s)
    np.testing.assert_allclose(y0, 0.5, rtol=0, atol=1e-14)
    X[:] = 0
    X[N] = 0.25
    m = np.arange(n * D)
    np.testing.assert_allclose(synthesize_real(X, g, M, D, s), 0.25 * (-1.0) ** ((s + m) % 2), rtol=0, atol=1e-14)


@pytest.mark.parametrize("M", [64, 256])
def test_roundtrip_recipe_reconstructs_real_stream(M):
    D = M // 2
    h, g, s_shift, off = roundtrip_taps(M)
    s_a = 2**40 + 3
    Fa = 200
    rng = np.random.default_rng(M)
    x = rng.standard_normal(h.size - 1 + Fa * D)
    Y = channelize(x.astype(np.complex128), h, M, D, s_a)[: M // 2 + 1]
    y = synthesize_real(Y, g, M, D, s_a + s_shift)
    ref = x[off: off + y.size]
    db = 10 * np.log10(np.sum((y - ref) ** 2) / np.sum(ref ** 2))
    assert db <= -100, db


def test_create_argument_errors_need_no_device():
    from pothoscomms_b200 import _abi
    lib = _abi.lib()
    h = ctypes.c_void_p()
    for dt in (_abi.CF32, _abi.CF64, _abi.F64, _abi.I8, _abi.CI16, 77):
        assert lib.b200c_rsynth_create(ctypes.byref(h), dt, 8, 8, 0) == _abi.ERR_UNSUPPORTED, dt
    for dt in (_abi.F32, _abi.I16):
        for M in (0, 1, 3, 6, 16384):
            assert lib.b200c_rsynth_create(ctypes.byref(h), dt, M, 1, 0) == _abi.ERR_UNSUPPORTED, (dt, M)
        for M, D in ((8, 0), (8, 3), (8, 16), (8192, 3), (64, 128)):
            assert lib.b200c_rsynth_create(ctypes.byref(h), dt, M, D, 0) == _abi.ERR_INVALID, (dt, M, D)
    assert not h.value
    assert lib.b200c_rsynth_create(None, _abi.F32, 8, 8, 0) == _abi.ERR_INVALID
    assert lib.b200c_rsynth_destroy(None) == _abi.OK
    assert lib.b200c_rsynth_set_taps(None, None, 1) == _abi.ERR_INVALID
    assert lib.b200c_rsynth_info(None, None, None, None, None, None) == _abi.ERR_INVALID
    c, p = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.b200c_rsynth_run(None, None, 0, 0, 0, None, 0, ctypes.byref(c), ctypes.byref(p), None) == _abi.ERR_INVALID


def test_python_wrapper_maps_argument_errors():
    from pothoscomms_b200 import B200CommsError, InvalidArgumentError, RealSynthesizer, _abi
    assert issubclass(InvalidArgumentError, B200CommsError)
    with pytest.raises(InvalidArgumentError) as e:
        RealSynthesizer("complex_float32", 8, 8)
    assert e.value.code == _abi.ERR_UNSUPPORTED
    with pytest.raises(InvalidArgumentError) as e:
        RealSynthesizer("int16", 16384, 8)
    assert e.value.code == _abi.ERR_UNSUPPORTED
    with pytest.raises(InvalidArgumentError) as e:
        RealSynthesizer("float32", 8, 3)
    assert e.value.code == _abi.ERR_INVALID
    with pytest.raises(InvalidArgumentError) as e:
        RealSynthesizer("float32", 8, -1)
    assert e.value.code == _abi.ERR_INVALID
