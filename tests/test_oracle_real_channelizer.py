"""The real-input channelizer's reference: tests/_chan_oracle.channelize applied to the real stream taken as complex,
rows 0 .. M/2 kept.  Checks that the rows it drops are the conjugate mirrors of the rows kept and that rows 0 and M/2
are real, plus the create-time argument checks of b200c_rchan_create, which need no device."""
import ctypes

import numpy as np
import pytest

from _chan_oracle import channelize


def real_channelize(x, h, M, D, s=0, frames=None, channels=None):
    """Rows 0 .. M/2 (or the listed ``channels``, each <= M/2) of the complex channelizer's definition on the real
    samples x.  x is made complex first: a real array handed to channelize() would be read as interleaved (re, im)
    pairs."""
    xc = np.asarray(x, dtype=np.float64).astype(np.complex128)
    if channels is None:
        return channelize(xc, h, M, D, s, frames)[: M // 2 + 1]
    assert all(0 <= c <= M // 2 for c in channels)
    return channelize(xc, h, M, D, s, frames, channels)


CASES = [
    # (M, D, ntaps, stream_index)
    (2, 1, 5, 1),
    (4, 4, 1, 0),
    (8, 4, 21, 2**40 + 7),
    (16, 16, 16, 12345),
    (32, 8, 3 * 32 + 5, 3),
]


@pytest.mark.parametrize("M,D,ntaps,s", CASES)
def test_dropped_rows_are_conjugate_mirrors(M, D, ntaps, s):
    rng = np.random.default_rng(100 * M + D + ntaps)
    x = rng.standard_normal(ntaps - 1 + 17 * D + D // 2)
    h = rng.standard_normal(ntaps)
    full = channelize(x.astype(np.complex128), h, M, D, s)
    y = real_channelize(x, h, M, D, s)
    assert y.shape == (M // 2 + 1, 17)
    np.testing.assert_array_equal(y, full[: M // 2 + 1])
    scale = max(1.0, np.abs(full).max())
    for c in range(M // 2 + 1, M):
        np.testing.assert_allclose(full[c], np.conj(full[M - c]), rtol=0, atol=1e-12 * scale)
    assert np.abs(y[0].imag).max() <= 1e-12 * scale
    assert np.abs(y[M // 2].imag).max() <= 1e-12 * scale


def test_real_values_read_as_samples_not_pairs():
    # the same real samples as float64 or int16 give the same reference; a raw real array fed to channelize() directly
    # would be taken as (re, im) pairs and give half the frames
    x = np.array([3, -1, 4, 1, -5, 9, 2, -6, 5, 3, -5, 8], dtype=np.int16)
    a = real_channelize(x, [0.5, 0.25], 4, 2, 1)
    b = real_channelize(x.astype(np.float64), [0.5, 0.25], 4, 2, 1)
    np.testing.assert_array_equal(a, b)
    assert a.shape == (3, 5)
    assert channelize(x.astype(np.float64), [0.5, 0.25], 4, 2, 1).shape[1] < a.shape[1]


def test_create_argument_errors_need_no_device():
    from pothoscomms_b200 import _abi
    lib = _abi.lib()
    h = ctypes.c_void_p()
    for dt in (_abi.CF32, _abi.CF64, _abi.F64, _abi.I8, _abi.CI16, 77):
        assert lib.b200c_rchan_create(ctypes.byref(h), dt, 8, 8, 0) == _abi.ERR_UNSUPPORTED, dt
    for dt in (_abi.F32, _abi.I16):
        for M in (0, 1, 3, 6, 16384):
            assert lib.b200c_rchan_create(ctypes.byref(h), dt, M, 1, 0) == _abi.ERR_UNSUPPORTED, (dt, M)
        for M, D in ((8, 0), (8, 3), (8, 16), (8192, 3), (64, 128)):
            assert lib.b200c_rchan_create(ctypes.byref(h), dt, M, D, 0) == _abi.ERR_INVALID, (dt, M, D)
    assert not h.value
    assert lib.b200c_rchan_create(None, _abi.F32, 8, 8, 0) == _abi.ERR_INVALID
    assert lib.b200c_rchan_destroy(None) == _abi.OK
    assert lib.b200c_rchan_set_taps(None, None, 1) == _abi.ERR_INVALID
    assert lib.b200c_rchan_info(None, None, None, None, None, None) == _abi.ERR_INVALID
    c, p = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.b200c_rchan_run(None, None, 0, 0, None, 0, 0, ctypes.byref(c), ctypes.byref(p), None) == _abi.ERR_INVALID


def test_python_wrapper_maps_argument_errors():
    from pothoscomms_b200 import InvalidArgumentError, RealChannelizer, _abi
    with pytest.raises(InvalidArgumentError) as e:
        RealChannelizer("complex_float32", 8, 8)
    assert e.value.code == _abi.ERR_UNSUPPORTED
    with pytest.raises(InvalidArgumentError) as e:
        RealChannelizer("int16", 16384, 8)
    assert e.value.code == _abi.ERR_UNSUPPORTED
    with pytest.raises(InvalidArgumentError) as e:
        RealChannelizer("float32", 8, 3)
    assert e.value.code == _abi.ERR_INVALID
    with pytest.raises(InvalidArgumentError) as e:
        RealChannelizer("float32", 8, -1)
    assert e.value.code == _abi.ERR_INVALID
