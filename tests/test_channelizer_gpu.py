"""Polyphase filter-bank channelizer (b200c_chan_*) on the B200 against the direct-sum definition
(tests/_chan_oracle.channelize)."""
import ctypes

import numpy as np
import pytest

import oracle
from _chan_oracle import channelize

pytestmark = pytest.mark.gpu

S_VALUES = (0, 12345, 2**40 + 7)


def _torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def _cx(n, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)


def _dev(x):
    torch = _torch()
    return torch.from_numpy(np.ascontiguousarray(x.astype(np.complex64)).view(np.float32).reshape(-1, 2)).cuda()


def _host(out, produced):
    o = out[:, :produced].cpu().numpy().astype(np.float64)
    return o[..., 0] + 1j * o[..., 1]


def _run(ch, x, s, frames=None):
    """One call on a fresh output tensor sized for `frames` (default: all available). Returns (y [M, F], consumed)."""
    torch = _torch()
    M, D, ntaps, _ = ch.info()
    F = (x.size - (ntaps - 1)) // D if frames is None else frames
    out = torch.empty((M, max(F, 1), 2), dtype=torch.float32, device="cuda")
    c, p = ch.run(_dev(x), out, s, out_capacity=F)
    torch.cuda.synchronize()
    assert (c, p) == (F * D, F)
    return _host(out, p), c


def _check(y, ref, tol=1e-5):
    assert y.shape == ref.shape
    err = np.sqrt(np.mean(np.abs(y - ref) ** 2, axis=1))
    rms = np.sqrt(np.mean(np.abs(ref) ** 2, axis=1))
    bad = np.nonzero(err > tol * rms)[0]
    assert bad.size == 0, f"channels {bad[:8]}: err/rms {(err[bad] / rms[bad])[:8]}"


def _tile(M):
    return max(4, min(512, 8192 // M))


def _grid():
    cases = []
    for M in (2, 8, 64, 256, 1024, 4096):
        Ds = [M, M // 2] + ([M // 4] if M >= 4 else []) + ([1] if M <= 8 else [])
        for D in sorted(set(Ds), reverse=True):
            for i, ntaps in enumerate(sorted({1, M - 1, M, 3 * M + 5, 16 * M})):
                if M == 4096 and ntaps == 16 * M and D != M:
                    continue    # the dense reference costs M * ntaps per frame
                if M >= 1024:
                    cases.append((M, D, ntaps, S_VALUES[(i + D) % 3]))
                else:
                    cases.extend((M, D, ntaps, s) for s in S_VALUES)
    return cases


@pytest.mark.parametrize("M,D,ntaps,s", _grid())
def test_parity_with_direct_sum(M, D, ntaps, s):
    from pothoscomms_b200 import Channelizer
    # frames: enough for several CTA tiles where the dense reference stays cheap, and at least 4 so that no channel's
    # RMS rests on a single (possibly tiny) sample
    F = max(4, min(2 * _tile(M) + 5, (1 << 22) // (M * ntaps)))
    x = _cx(ntaps - 1 + F * D + D // 3, seed=M * 7919 + D * 31 + ntaps)
    h = np.random.default_rng(ntaps).standard_normal(ntaps)
    ch = Channelizer("complex_float32", M, D)
    ch.set_taps(h)
    assert ch.info() == (M, D, ntaps, ntaps - 1 + D)
    y, _ = _run(ch, x, s)
    _check(y, channelize(x, h, M, D, s))


def test_frequency_convention():
    from scipy import signal
    from pothoscomms_b200 import Channelizer
    M, D, c0, s, A = 64, 32, 5, 12345, 0.75
    nt, beta = signal.kaiserord(80.0, 2.0 / M)          # 80 dB, transition one channel spacing wide
    h = signal.firwin(nt, 1.0 / M, window=("kaiser", beta))
    assert nt <= 16 * M
    ch = Channelizer("complex_float32", M, D)
    ch.set_taps(h)
    n = nt - 1 + 200 * D
    i = np.arange(n)
    x = A * np.exp(2j * np.pi * c0 * ((s + i) % M) / M)  # tone at +c0/M cycles per sample
    y, _ = _run(ch, x, s)
    np.testing.assert_allclose(y[c0], A, rtol=1e-3)      # at baseband, with the input amplitude
    for c in range(M):
        if min((c - c0) % M, (c0 - c) % M) >= 2:
            level = 20 * np.log10(np.sqrt(np.mean(np.abs(y[c]) ** 2)) / A)
            assert level <= -60, (c, level)
    # channels c >= M/2 are the negative frequencies
    xn = A * np.exp(-2j * np.pi * 3 * ((s + i) % M) / M)
    yn, _ = _run(ch, xn, s)
    np.testing.assert_allclose(yn[M - 3], A, rtol=1e-3)


@pytest.mark.parametrize("M,D,ntaps", [(64, 32, 3 * 64 + 5), (8, 1, 29), (1024, 1024, 4 * 1024 - 3)])
def test_streaming_pieces_bit_identical(M, D, ntaps):
    torch = _torch()
    from pothoscomms_b200 import Channelizer
    ch = Channelizer("complex_float32", M, D)
    ch.set_taps(np.random.default_rng(3).standard_normal(ntaps))
    s0 = 2**33 + 11
    x = _cx(ntaps - 1 + 700 * D + 17, seed=99)
    whole, cons = _run(ch, x, s0)
    rng = np.random.default_rng(5)
    pieces, carry, pos = [], x[: ntaps - 1], ntaps - 1    # history first, then ragged pieces of new data
    base = s0
    while pos < x.size:
        step = int(rng.integers(1, 3 * D + 200))
        buf = np.concatenate([carry, x[pos: pos + step]])
        pos += step
        out = torch.zeros((M, buf.size // D + 1, 2), dtype=torch.float32, device="cuda")
        c, p = ch.run(_dev(buf), out, base)
        torch.cuda.synchronize()
        pieces.append(out[:, :p].cpu())
        carry = buf[c:]
        base += c
    got = torch.cat(pieces, dim=1)
    ref = torch.from_numpy(np.stack([whole.real, whole.imag], axis=-1).astype(np.float32))
    assert got.shape == ref.shape
    assert torch.equal(got, ref), "a stream fed in pieces must give the one-call output bit for bit"


def test_capacity_and_stride():
    torch = _torch()
    from pothoscomms_b200 import Channelizer
    M, D, ntaps, s = 64, 16, 100, 77
    ch = Channelizer("complex_float32", M, D)
    h = np.random.default_rng(1).standard_normal(ntaps)
    ch.set_taps(h)
    x = _cx(ntaps - 1 + 300 * D, seed=4)
    sentinel = 12345.5
    stride, cap = 256, 211                       # 300 frames available, room for 211, rows 256 apart
    out = torch.full((M, stride, 2), sentinel, dtype=torch.float32, device="cuda")
    c, p = ch.run(_dev(x), out, s, out_capacity=cap)
    torch.cuda.synchronize()
    assert (c, p) == (cap * D, cap)
    o = out.cpu()
    assert torch.all(o[:, cap:] == sentinel), "nothing may be written past `produced`, padding included"
    _check(_host(out, cap), channelize(x, h, M, D, s, frames=cap))
    # below input_require: (0, 0) and nothing written
    req = ch.info()[3]
    out2 = torch.full((M, 8, 2), sentinel, dtype=torch.float32, device="cuda")
    assert ch.run(_dev(x[: req - 1]), out2, s) == (0, 0)
    assert ch.run(_dev(x[:req]), out2, s, out_capacity=0) == (0, 0)
    torch.cuda.synchronize()
    assert torch.all(out2.cpu() == sentinel)
    assert ch.run(_dev(x[:req]), out2, s) == (D, 1)


def test_chain_into_filter_bank():
    torch = _torch()
    from scipy import signal
    from pothoscomms_b200 import Channelizer, FirFilterBank
    M, D, ntaps, s = 64, 64, 8 * 64, 2**35 + 1
    h = signal.firwin(ntaps, 1.0 / M, window=("kaiser", 8.0))
    ch = Channelizer("complex_float32", M, D)
    ch.set_taps(h)
    F = 400
    x = _cx(ntaps - 1 + F * D, seed=8)
    stream = torch.cuda.Stream()
    mid = torch.empty((M, F, 2), dtype=torch.float32, device="cuda")
    with torch.cuda.stream(stream):
        d_in = _dev(x)
        assert ch.run(d_in, mid, s, stream=stream) == (F * D, F)
        bank = FirFilterBank("complex_float32", "REAL", M)
        lps = [signal.firwin(33, 0.45) * (1.0 + c / M) for c in range(M)]
        for c in range(M):
            bank.set_taps(c, lps[c])
        bank.set_rates(2, 1)
        F2 = (F - 32) // 2
        out = torch.empty((M, F2, 2), dtype=torch.float32, device="cuda")
        assert bank.run(mid, out, stream=stream) == (2 * F2, F2)
    stream.synchronize()
    y = channelize(x, h, M, D, s)
    ref = []
    for c in range(M):
        r, _, p = oracle.fir(oracle.CF64, False, lps[c], 2, 1, oracle.to_raw(y[c], oracle.CF64))
        ref.append(r[:F2, 0] + 1j * r[:F2, 1])
    _check(_host(out, F2), np.array(ref))


def test_taps_and_errors():
    torch = _torch()
    from pothoscomms_b200 import Channelizer, _abi
    M, D, s = 16, 8, 3
    ch = Channelizer("complex_float32", M, D)
    assert ch.info() == (M, D, 1, D)                       # taps {1} after create
    x = _cx(2000, seed=12)
    y1, _ = _run(ch, x, s)
    _check(y1, channelize(x, [1.0], M, D, s))
    h = np.random.default_rng(2).standard_normal(5 * M + 3)
    ch.set_taps(h)
    assert ch.info() == (M, D, h.size, h.size - 1 + D)
    y2, _ = _run(ch, x, s)
    _check(y2, channelize(x, h, M, D, s))
    assert y2.shape != y1.shape
    ch.set_taps(h[:7])
    assert ch.info()[3] == 6 + D
    y3, _ = _run(ch, x, s)
    _check(y3, channelize(x, h[:7], M, D, s))

    lib, hh = _abi.lib(), ch._h
    one = np.ones(16 * M + 1)
    assert lib.b200c_chan_set_taps(hh, one.ctypes.data, 0) == _abi.ERR_INVALID
    assert lib.b200c_chan_set_taps(hh, one.ctypes.data, 16 * M + 1) == _abi.ERR_INVALID
    assert ch.info()[2] == 7                                # a refused set_taps keeps the old taps
    assert lib.b200c_chan_set_taps(hh, one.ctypes.data, 16 * M) == _abi.OK
    d_in = _dev(x)
    out = torch.empty((M, 64, 2), dtype=torch.float32, device="cuda")
    c, p = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.b200c_chan_run(hh, None, d_in.shape[0], s, ctypes.c_void_p(out.data_ptr()), 64, 64,
                              ctypes.byref(c), ctypes.byref(p), None) == _abi.ERR_INVALID
    assert lib.b200c_chan_run(hh, ctypes.c_void_p(d_in.data_ptr()), d_in.shape[0], s, None, 64, 64,
                              ctypes.byref(c), ctypes.byref(p), None) == _abi.ERR_INVALID
    assert lib.b200c_chan_run(hh, ctypes.c_void_p(d_in.data_ptr()), d_in.shape[0], s, ctypes.c_void_p(out.data_ptr()), 10, 64,
                              ctypes.byref(c), ctypes.byref(p), None) == _abi.ERR_INVALID
    assert p.value == 64
    # nothing to produce: null buffers are fine
    assert lib.b200c_chan_run(hh, None, 3, s, None, 0, 64, ctypes.byref(c), ctypes.byref(p), None) == _abi.OK
    assert (c.value, p.value) == (0, 0)
    torch.cuda.synchronize()
