"""Real-input polyphase filter-bank channelizer (b200c_rchan_*) on the B200 against the direct-sum definition:
tests/_chan_oracle.channelize of the real stream taken as complex, rows 0 .. M/2."""
import ctypes

import numpy as np
import pytest

import oracle
from test_oracle_real_channelizer import real_channelize

pytestmark = pytest.mark.gpu

S_VALUES = (0, 12345, 2**40 + 7)


def _torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def _real(n, seed):
    return np.random.default_rng(seed).standard_normal(n).astype(np.float32)


def _dev(x):
    return _torch().from_numpy(np.ascontiguousarray(x)).cuda()


def _host(out, produced):
    o = out[:, :produced].cpu().numpy().astype(np.float64)
    return o[..., 0] + 1j * o[..., 1]


def _run(ch, x, s, frames=None):
    """One call on a fresh output tensor sized for `frames` (default: all available).  Returns (raw out [M/2+1, F, 2]
    on the host, consumed)."""
    torch = _torch()
    M, nch, D, ntaps, _ = ch.info()
    F = (x.size - (ntaps - 1)) // D if frames is None else frames
    out = torch.empty((nch, max(F, 1), 2), dtype=torch.float32, device="cuda")
    c, p = ch.run(_dev(x), out, s, out_capacity=F)
    torch.cuda.synchronize()
    assert (c, p) == (F * D, F)
    return out[:, :p].cpu(), c


def _cplx(raw):
    o = raw.numpy().astype(np.float64)
    return o[..., 0] + 1j * o[..., 1]


def _check(y, ref, tol=1e-5):
    assert y.shape == ref.shape
    err = np.sqrt(np.mean(np.abs(y - ref) ** 2, axis=1))
    rms = np.sqrt(np.mean(np.abs(ref) ** 2, axis=1))
    bad = np.nonzero(err > tol * rms)[0]
    assert bad.size == 0, f"channels {bad[:8]}: err/rms {(err[bad] / rms[bad])[:8]}"


def _tile(M):
    return max(4, min(512, 16384 // M))


def _grid():
    cases = []
    for M in (2, 4, 8, 64, 256, 2048, 8192):
        Ds = [M, M // 2] + ([M // 4] if M >= 4 else []) + ([1] if M <= 8 else [])
        for D in sorted(set(Ds), reverse=True):
            for i, ntaps in enumerate(sorted({1, M - 1, M, 3 * M + 5, 16 * M})):
                # the dense reference costs M * ntaps per frame
                if M == 8192 and (ntaps == 16 * M or (ntaps == 3 * M + 5 and D != M)):
                    continue
                if M == 2048 and ntaps == 16 * M and D != M:
                    continue
                if M >= 2048:
                    cases.append((M, D, ntaps, S_VALUES[(i + D) % 3]))
                else:
                    cases.extend((M, D, ntaps, s) for s in S_VALUES)
    return cases


@pytest.mark.parametrize("M,D,ntaps,s", _grid())
def test_parity_with_direct_sum(M, D, ntaps, s):
    from pothoscomms_b200 import RealChannelizer
    # frames: several CTA tiles where the dense reference stays cheap, and at least 4 so that no channel's RMS rests
    # on a single sample
    F = max(4, min(2 * _tile(M) + 5, (1 << 22) // (M * ntaps)))
    x = _real(ntaps - 1 + F * D + D // 3, seed=M * 7919 + D * 31 + ntaps)
    h = np.random.default_rng(ntaps).standard_normal(ntaps)
    ch = RealChannelizer("float32", M, D)
    ch.set_taps(h)
    assert ch.info() == (M, M // 2 + 1, D, ntaps, ntaps - 1 + D)
    raw, _ = _run(ch, x, s)
    _check(_cplx(raw), real_channelize(x, h, M, D, s))
    # channels 0 and M/2 are real: imaginary parts exactly 0
    assert raw[0, :, 1].abs().max().item() == 0.0
    assert raw[M // 2, :, 1].abs().max().item() == 0.0


@pytest.mark.parametrize("M,D,ntaps", [(64, 32, 3 * 64 + 5), (2048, 2048, 8 * 2048), (8, 1, 29)])
def test_int16_bit_identical_to_float32(M, D, ntaps):
    from pothoscomms_b200 import RealChannelizer
    rng = np.random.default_rng(M + ntaps)
    n = ntaps - 1 + 300 * D
    xi = rng.integers(-32768, 32768, size=n, dtype=np.int64).astype(np.int16)
    xi[::97] = -32768
    xi[5::89] = 32767
    h = rng.standard_normal(ntaps)
    chi, chf = RealChannelizer("int16", M, D), RealChannelizer("float32", M, D)
    chi.set_taps(h)
    chf.set_taps(h)
    s = 2**40 + 7
    yi, _ = _run(chi, xi, s)
    yf, _ = _run(chf, xi.astype(np.float32), s)
    assert _torch().equal(yi, yf), "int16 input must give the float32 output of the same values bit for bit"
    _check(_cplx(yi)[:, :8], real_channelize(xi, h, M, D, s, frames=8))


def test_frequency_convention():
    from scipy import signal
    from pothoscomms_b200 import RealChannelizer
    M, D, s, A = 64, 32, 12345, 0.75
    nt, beta = signal.kaiserord(80.0, 2.0 / M)          # 80 dB, transition one channel spacing wide
    h = signal.firwin(nt, 1.0 / M, window=("kaiser", beta))   # unit DC gain
    assert nt <= 16 * M
    ch = RealChannelizer("float32", M, D)
    ch.set_taps(h)
    n = nt - 1 + 200 * D
    i = np.arange(n)
    for c0, level0 in ((5, A / 2), (0, A), (M // 2, A)):
        x = (A * np.cos(2 * np.pi * c0 * ((s + i) % M) / M)).astype(np.float32)   # real tone at c0/M
        y = _cplx(_run(ch, x, s)[0])
        np.testing.assert_allclose(y[c0], level0, rtol=1e-3)
        for c in range(M // 2 + 1):
            if abs(c - c0) >= 2:
                level = 20 * np.log10(np.sqrt(np.mean(np.abs(y[c]) ** 2)) / A)
                assert level <= -60, (c0, c, level)


def test_agrees_with_complex_channelizer():
    torch = _torch()
    from pothoscomms_b200 import Channelizer, RealChannelizer
    M, D, ntaps, s = 256, 128, 5 * 256 + 3, 2**33 + 5
    h = np.random.default_rng(4).standard_normal(ntaps)
    x = _real(ntaps - 1 + 150 * D, seed=6)
    rc, cc = RealChannelizer("float32", M, D), Channelizer("complex_float32", M, D)
    rc.set_taps(h)
    cc.set_taps(h)
    yr = _cplx(_run(rc, x, s)[0])
    xc = torch.from_numpy(np.stack([x, np.zeros_like(x)], axis=-1)).cuda()
    out = torch.empty((M, 150, 2), dtype=torch.float32, device="cuda")
    assert cc.run(xc, out, s) == (150 * D, 150)
    torch.cuda.synchronize()
    _check(yr, _host(out, 150)[: M // 2 + 1])


@pytest.mark.parametrize("dtype", ["float32", "int16"])
@pytest.mark.parametrize("M,D,ntaps", [(64, 32, 3 * 64 + 5), (8, 1, 29), (2048, 1024, 4 * 2048 - 3)])
def test_streaming_pieces_bit_identical(dtype, M, D, ntaps):
    torch = _torch()
    from pothoscomms_b200 import RealChannelizer
    ch = RealChannelizer(dtype, M, D)
    ch.set_taps(np.random.default_rng(3).standard_normal(ntaps))
    s0 = 2**33 + 11
    rng = np.random.default_rng(99)
    n = ntaps - 1 + 701 * D + 17
    x = rng.integers(-32768, 32768, size=n).astype(np.int16) if dtype == "int16" else _real(n, 99)
    whole, _ = _run(ch, x, s0)
    pieces, carry, pos, base = [], x[: ntaps - 1], ntaps - 1, s0   # history first, then ragged pieces of new data
    while pos < x.size:
        step = int(rng.integers(1, 3 * D + 200))
        buf = np.concatenate([carry, x[pos: pos + step]])
        pos += step
        off = 1 + 2 * int(rng.integers(0, 4))                   # odd element offset: d_in only element-aligned
        big = torch.zeros(buf.size + off + 3, dtype=torch.int16 if dtype == "int16" else torch.float32, device="cuda")
        big[off: off + buf.size] = _dev(buf)
        view = big[off: off + buf.size]
        out = torch.zeros((M // 2 + 1, buf.size // D + 1, 2), dtype=torch.float32, device="cuda")
        c, p = ch.run(view, out, base)
        torch.cuda.synchronize()
        pieces.append(out[:, :p].cpu())
        carry = buf[c:]
        base += c
    got = torch.cat(pieces, dim=1)
    assert got.shape == whole.shape
    assert torch.equal(got, whole), "a stream fed in pieces must give the one-call output bit for bit"


def test_capacity_stride_and_nothing_else_written():
    torch = _torch()
    from pothoscomms_b200 import RealChannelizer
    M, D, ntaps, s = 64, 16, 100, 77
    nch = M // 2 + 1
    ch = RealChannelizer("float32", M, D)
    h = np.random.default_rng(1).standard_normal(ntaps)
    ch.set_taps(h)
    x = _real(ntaps - 1 + 301 * D, seed=4)
    sentinel = 12345.5
    stride, cap = 256, 211                       # 301 frames available, room for 211, rows 256 apart
    buf = torch.full((nch + 2, stride, 2), sentinel, dtype=torch.float32, device="cuda")
    c, p = ch.run(_dev(x), buf[:nch], s, out_capacity=cap)
    torch.cuda.synchronize()
    assert (c, p) == (cap * D, cap)
    o = buf.cpu()
    assert torch.all(o[:nch, cap:] == sentinel), "nothing may be written past `produced`"
    assert torch.all(o[nch:] == sentinel), "nothing may be written past row M/2"
    _check(_host(buf, cap)[:nch], real_channelize(x, h, M, D, s, frames=cap))
    # below input_require, or no capacity: (0, 0) and nothing written
    req = ch.info()[4]
    out2 = torch.full((nch, 8, 2), sentinel, dtype=torch.float32, device="cuda")
    assert ch.run(_dev(x[: req - 1]), out2, s) == (0, 0)
    assert ch.run(_dev(x[:req]), out2, s, out_capacity=0) == (0, 0)
    torch.cuda.synchronize()
    assert torch.all(out2.cpu() == sentinel)
    assert ch.run(_dev(x[:req]), out2, s) == (D, 1)
    torch.cuda.synchronize()
    assert torch.all(out2.cpu()[:, 1:] == sentinel)


def test_chain_into_filter_bank():
    torch = _torch()
    from scipy import signal
    from pothoscomms_b200 import FirFilterBank, RealChannelizer
    M, D, ntaps, s = 64, 64, 8 * 64, 2**35 + 1
    nch = M // 2 + 1
    h = signal.firwin(ntaps, 1.0 / M, window=("kaiser", 8.0))
    ch = RealChannelizer("int16", M, D)
    ch.set_taps(h)
    F = 400
    x = np.random.default_rng(8).integers(-20000, 20000, size=ntaps - 1 + F * D).astype(np.int16)
    stream = torch.cuda.Stream()
    mid = torch.empty((nch, F, 2), dtype=torch.float32, device="cuda")
    with torch.cuda.stream(stream):
        d_in = _dev(x)
        assert ch.run(d_in, mid, s, stream=stream) == (F * D, F)
        bank = FirFilterBank("complex_float32", "REAL", nch)
        lps = [signal.firwin(33, 0.45) * (1.0 + c / M) for c in range(nch)]
        for c in range(nch):
            bank.set_taps(c, lps[c])
        bank.set_rates(2, 1)
        F2 = (F - 32) // 2
        out = torch.empty((nch, F2, 2), dtype=torch.float32, device="cuda")
        assert bank.run(mid, out, stream=stream) == (2 * F2, F2)
    stream.synchronize()
    y = real_channelize(x, h, M, D, s)
    ref = []
    for c in range(nch):
        r, _, p = oracle.fir(oracle.CF64, False, lps[c], 2, 1, oracle.to_raw(y[c], oracle.CF64))
        ref.append(r[:F2, 0] + 1j * r[:F2, 1])
    _check(_host(out, F2), np.array(ref))


def test_taps_errors_and_stream():
    torch = _torch()
    from pothoscomms_b200 import RealChannelizer, _abi
    M, D, s = 16, 8, 3
    ch = RealChannelizer("float32", M, D)
    assert ch.info() == (M, M // 2 + 1, D, 1, D)             # taps {1} after create
    x = _real(2000, seed=12)
    y1 = _cplx(_run(ch, x, s)[0])
    _check(y1, real_channelize(x, [1.0], M, D, s))
    h = np.random.default_rng(2).standard_normal(5 * M + 3)
    ch.set_taps(h)
    assert ch.info() == (M, M // 2 + 1, D, h.size, h.size - 1 + D)
    y2 = _cplx(_run(ch, x, s)[0])
    _check(y2, real_channelize(x, h, M, D, s))
    ch.set_taps(h[:7])
    assert ch.info()[4] == 6 + D
    y3 = _cplx(_run(ch, x, s)[0])
    _check(y3, real_channelize(x, h[:7], M, D, s))

    lib, hh = _abi.lib(), ch._h
    one = np.ones(16 * M + 1)
    assert lib.b200c_rchan_set_taps(hh, one.ctypes.data, 0) == _abi.ERR_INVALID
    assert lib.b200c_rchan_set_taps(hh, one.ctypes.data, 16 * M + 1) == _abi.ERR_INVALID
    assert ch.info()[3] == 7                                # a refused set_taps keeps the old taps
    y4 = _cplx(_run(ch, x, s)[0])
    np.testing.assert_array_equal(y4, y3)

    # a run on a non-default stream, ordered after the input's upload on that stream
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_in = _dev(x)
        out = torch.empty((M // 2 + 1, 300, 2), dtype=torch.float32, device="cuda")
        c, p = ch.run(d_in, out, s, stream=stream)
    stream.synchronize()
    np.testing.assert_array_equal(_host(out, p), y3)

    assert lib.b200c_rchan_set_taps(hh, one.ctypes.data, 16 * M) == _abi.OK
    c, p = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.b200c_rchan_run(hh, None, d_in.numel(), s, ctypes.c_void_p(out.data_ptr()), 300, 64,
                               ctypes.byref(c), ctypes.byref(p), None) == _abi.ERR_INVALID
    assert lib.b200c_rchan_run(hh, ctypes.c_void_p(d_in.data_ptr()), d_in.numel(), s, None, 300, 64,
                               ctypes.byref(c), ctypes.byref(p), None) == _abi.ERR_INVALID
    assert lib.b200c_rchan_run(hh, ctypes.c_void_p(d_in.data_ptr()), d_in.numel(), s, ctypes.c_void_p(out.data_ptr()), 10, 64,
                               ctypes.byref(c), ctypes.byref(p), None) == _abi.ERR_INVALID
    assert p.value == 64
    # nothing to produce: null buffers are fine
    assert lib.b200c_rchan_run(hh, None, 3, s, None, 0, 64, ctypes.byref(c), ctypes.byref(p), None) == _abi.OK
    assert (c.value, p.value) == (0, 0)
    torch.cuda.synchronize()
