"""The synthesizer reference (tests/_synth_oracle.synthesize) pinned to the FIR oracle: channel c must be /comms/fir_filter
with real taps and interpolation D, mixed up by c/M, and the channels summed.  Plus the channelizer -> synthesizer
round trip that sets the reconstruction bar of the GPU test, and the create-time argument checks of
b200c_synth_create, which need no device."""
import ctypes

import numpy as np
import pytest

import oracle
from _chan_oracle import channelize
from _synth_oracle import roundtrip_taps, synthesize


def _fir_mix_sum(X, g, M, D, s):
    """Channel by channel: the FIR oracle (REAL taps, interpolation D), numpy mixing by exp(+2 pi i c (s+m)/M), sum."""
    out = None
    for c in range(M):
        y, cons, prod = oracle.fir(oracle.CF64, False, g, 1, D, oracle.to_raw(X[c], oracle.CF64))
        y = y[:, 0] + 1j * y[:, 1]
        assert prod == cons * D
        m = np.arange(y.size, dtype=np.int64)
        z = y * np.exp(2j * np.pi * ((c * ((s + m) % M)) % M) / M)
        out = z if out is None else out + z
    return out


CASES = [
    # (M, D, ntaps, stream_index)
    (8, 8, 21, 3),            # ntaps not a multiple of D, critically sampled
    (8, 4, 13, 2**33 + 5),    # 2x oversampled, stream_index >= 2^32
    (4, 1, 7, 1),             # D = 1
    (16, 8, 40, 0),
    (2, 2, 1, 1),             # ntaps = 1
    (16, 16, 16, 2**40 + 9),  # ntaps = D, stream_index far beyond 2^32
    (32, 8, 255, 77),         # K = 32
]


@pytest.mark.parametrize("M,D,ntaps,s", CASES)
def test_synthesize_is_mixed_sum_of_interpolating_firs(M, D, ntaps, s):
    rng = np.random.default_rng(1000 * M + 10 * D + ntaps)
    K = -(-ntaps // D)
    n = K - 1 + 19
    X = rng.standard_normal((M, n)) + 1j * rng.standard_normal((M, n))
    g = rng.standard_normal(ntaps)
    y = synthesize(X, g, M, D, s)
    ref = _fir_mix_sum(X, g, M, D, s)
    assert y.shape == ref.shape == (19 * D,)
    np.testing.assert_allclose(y, ref, rtol=0, atol=1e-12 * np.abs(ref).max())


def test_synthesize_counts_and_phase():
    # F = n - (K-1) frames, F D samples; 0 below K frames; `samples` caps F at samples // D
    X = np.ones((4, 10), dtype=np.complex128)
    assert synthesize(X, [1.0] * 9, 4, 4).shape == (8 * 4,)          # K = 3
    assert synthesize(X[:, :2], [1.0] * 9, 4, 4).shape == (0,)
    assert synthesize(X[:, :3], [1.0] * 9, 4, 4).shape == (4,)
    assert synthesize(X, [1.0] * 9, 4, 4, samples=13).shape == (12,)
    # only s mod M matters
    rng = np.random.default_rng(7)
    X = rng.standard_normal((8, 12)) + 1j * rng.standard_normal((8, 12))
    a = synthesize(X, [0.5, -1.0, 2.0], 8, 2, 3)
    b = synthesize(X, [0.5, -1.0, 2.0], 8, 2, 3 + 8 * 2**37)
    np.testing.assert_array_equal(a, b)
    # one constant channel c0 and a D-tap boxcar: a tone at +c0/M with the channel's amplitude
    M, D, c0, s = 8, 8, 3, 11
    X = np.zeros((M, 6), dtype=np.complex128)
    X[c0] = 0.5
    y = synthesize(X, np.ones(D), M, D, s)
    m = np.arange(y.size)
    np.testing.assert_allclose(y, 0.5 * np.exp(2j * np.pi * c0 * (s + m) / M), atol=1e-12)


@pytest.mark.parametrize("s_a", [0, 12345, 2**40 + 3])
def test_roundtrip_recipe_reconstructs(s_a):
    M = 16
    D = M // 2
    h, g, s_shift, off = roundtrip_taps(M)
    rng = np.random.default_rng(s_a % 1000)
    n = h.size - 1 + 400 * D
    x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    Y = channelize(x, h, M, D, s_a)
    y = synthesize(Y, g, M, D, s_a + s_shift)
    ref = x[off: off + y.size]
    assert y.size > 2000 and ref.size == y.size
    db = 10 * np.log10(np.sum(np.abs(y - ref) ** 2) / np.sum(np.abs(ref) ** 2))
    assert db <= -90, db


def test_create_argument_errors_need_no_device():
    from pothoscomms_b200 import _abi
    lib = _abi.lib()
    h = ctypes.c_void_p()
    for dt in (_abi.F32, _abi.CF64, _abi.CI16, 77):
        assert lib.b200c_synth_create(ctypes.byref(h), dt, 8, 8, 0) == _abi.ERR_UNSUPPORTED
    for M in (0, 1, 3, 6, 8192):
        assert lib.b200c_synth_create(ctypes.byref(h), _abi.CF32, M, 1, 0) == _abi.ERR_UNSUPPORTED, M
    for M, D in ((8, 0), (8, 3), (8, 16), (64, 128), (16, 5)):
        assert lib.b200c_synth_create(ctypes.byref(h), _abi.CF32, M, D, 0) == _abi.ERR_INVALID, (M, D)
    assert not h.value
    assert lib.b200c_synth_create(None, _abi.CF32, 8, 8, 0) == _abi.ERR_INVALID
    assert lib.b200c_synth_destroy(None) == _abi.OK
    assert lib.b200c_synth_set_taps(None, None, 1) == _abi.ERR_INVALID
    assert lib.b200c_synth_info(None, None, None, None, None) == _abi.ERR_INVALID
    c, p = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.b200c_synth_run(None, None, 0, 0, 0, None, 0, ctypes.byref(c), ctypes.byref(p), None) == _abi.ERR_INVALID


def test_python_wrapper_maps_argument_errors():
    from pothoscomms_b200 import InvalidArgumentError, Synthesizer, _abi
    with pytest.raises(InvalidArgumentError) as e:
        Synthesizer("complex_int16", 8, 8)
    assert e.value.code == _abi.ERR_UNSUPPORTED
    with pytest.raises(InvalidArgumentError) as e:
        Synthesizer("complex_float32", 8, 3)
    assert e.value.code == _abi.ERR_INVALID
    with pytest.raises(InvalidArgumentError) as e:
        Synthesizer("complex_float32", 8, -1)
    assert e.value.code == _abi.ERR_INVALID
