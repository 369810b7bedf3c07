"""The channelizer reference (tests/_chan_oracle.channelize, a direct sum) pinned to the FIR oracle: channel c must be
/comms/fir_filter with real taps and decimation D applied to the stream mixed down by c/M.  Plus the
create-time argument checks of b200c_chan_create, which need no device."""
import ctypes

import numpy as np
import pytest

import oracle
from _chan_oracle import channelize


def _mix_then_fir(x, h, M, D, s):
    """Channel by channel: numpy mixing z[i] = x[i] exp(-2 pi i c (s+i)/M), then the FIR oracle (REAL taps, decim D)."""
    i = np.arange(x.size, dtype=np.int64)
    out = []
    for c in range(M):
        z = x * np.exp(-2j * np.pi * ((c * ((s + i) % M)) % M) / M)
        y, cons, prod = oracle.fir(oracle.CF64, False, h, D, 1, oracle.to_raw(z, oracle.CF64))
        out.append(y[:, 0] + 1j * y[:, 1])
        assert cons == prod * D
    return np.array(out)


CASES = [
    # (M, D, ntaps, stream_index)
    (8, 8, 21, 0),            # ntaps not a multiple of M, critically sampled
    (8, 4, 1, 5),             # ntaps = 1, 2x oversampled (D = M/2)
    (4, 1, 17, 3),            # D = 1
    (16, 8, 40, 2**32 + 7),   # stream_index >= 2^32
    (16, 16, 16, 2**40 + 9),  # ntaps = M, stream_index far beyond 2^32
    (2, 1, 5, 1),
]


@pytest.mark.parametrize("M,D,ntaps,s", CASES)
def test_channelize_is_fir_of_the_mixed_stream(M, D, ntaps, s):
    rng = np.random.default_rng(1000 * M + 10 * D + ntaps)
    n = ntaps - 1 + 23 * D + D // 2
    x = rng.standard_normal(n) + 1j * rng.standard_normal(n)
    h = rng.standard_normal(ntaps)
    y = channelize(x, h, M, D, s)
    ref = _mix_then_fir(x, h, M, D, s)
    assert y.shape == ref.shape == (M, 23)
    np.testing.assert_allclose(y, ref, rtol=0, atol=1e-12 * max(1.0, np.abs(ref).max()))


def test_channelize_counts_and_phase():
    # F = (n - (ntaps-1)) // D, 0 below ntaps-1+D; only s mod M matters
    x = np.ones(10, dtype=np.complex128)
    assert channelize(x, [1.0] * 4, 4, 4).shape == (4, 1)
    assert channelize(x[:6], [1.0] * 4, 4, 4).shape == (4, 0)
    rng = np.random.default_rng(7)
    x = rng.standard_normal(64) + 1j * rng.standard_normal(64)
    a = channelize(x, [0.5, -1.0, 2.0], 8, 2, 3)
    b = channelize(x, [0.5, -1.0, 2.0], 8, 2, 3 + 8 * 2**37)
    np.testing.assert_array_equal(a, b)
    # a tone at c0/M lands in channel c0 only: an M-tap boxcar nulls every other channel centre exactly
    M, c0, s = 8, 3, 11
    i = np.arange(80)
    tone = np.exp(2j * np.pi * c0 * (s + i) / M)
    y = channelize(tone, np.ones(M) / M, M, M, s)
    np.testing.assert_allclose(y[c0], 1.0, atol=1e-12)
    assert np.abs(np.delete(y, c0, axis=0)).max() < 1e-12


def test_create_argument_errors_need_no_device():
    from pothoscomms_b200 import _abi
    lib = _abi.lib()
    h = ctypes.c_void_p()
    for dt in (_abi.F32, _abi.CF64, _abi.CI16, 77):
        assert lib.b200c_chan_create(ctypes.byref(h), dt, 8, 8, 0) == _abi.ERR_UNSUPPORTED
    for M in (0, 1, 3, 6, 8192):
        assert lib.b200c_chan_create(ctypes.byref(h), _abi.CF32, M, 1, 0) == _abi.ERR_UNSUPPORTED, M
    for M, D in ((8, 0), (8, 3), (8, 16), (64, 128), (16, 5)):
        assert lib.b200c_chan_create(ctypes.byref(h), _abi.CF32, M, D, 0) == _abi.ERR_INVALID, (M, D)
    assert not h.value
    assert lib.b200c_chan_create(None, _abi.CF32, 8, 8, 0) == _abi.ERR_INVALID
    assert lib.b200c_chan_destroy(None) == _abi.OK


def test_python_wrapper_maps_argument_errors():
    from pothoscomms_b200 import Channelizer, InvalidArgumentError, _abi
    with pytest.raises(InvalidArgumentError) as e:
        Channelizer("complex_int16", 8, 8)
    assert e.value.code == _abi.ERR_UNSUPPORTED
    with pytest.raises(InvalidArgumentError) as e:
        Channelizer("complex_float32", 8, 3)
    assert e.value.code == _abi.ERR_INVALID
