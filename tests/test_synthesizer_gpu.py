"""Polyphase synthesis filter bank (b200c_synth_*) on the B200 against the reference (tests/_synth_oracle.synthesize),
and the channelizer -> synthesizer round trip."""
import ctypes

import numpy as np
import pytest
from scipy import signal

from _chan_oracle import channelize
from _synth_oracle import roundtrip_taps, synthesize

pytestmark = pytest.mark.gpu

S_VALUES = (0, 12345, 2**40 + 7)


def _torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def _frames(M, n, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((M, n)) + 1j * rng.standard_normal((M, n))).astype(np.complex64)


def _dev(X):
    """[M, n] complex -> CUDA [M, n, 2] float32 (the channelizer's output layout)."""
    torch = _torch()
    X = np.ascontiguousarray(np.asarray(X).astype(np.complex64))
    return torch.from_numpy(X.view(np.float32).reshape(X.shape[0], -1, 2)).cuda()


def _host(out, produced):
    o = out[:produced].cpu().numpy().astype(np.float64)
    return o[:, 0] + 1j * o[:, 1]


def _run(sy, X, s, frames=None):
    """One call on a fresh output tensor sized for `frames` output frames (default: all available).
    Returns (y [F D], consumed)."""
    torch = _torch()
    M, D, ntaps, K = sy.info()
    F = X.shape[1] - (K - 1) if frames is None else frames
    out = torch.empty((max(F * D, 1), 2), dtype=torch.float32, device="cuda")
    c, p = sy.run(_dev(X), out, s, out_capacity=F * D)
    torch.cuda.synchronize()
    assert (c, p) == (F, F * D)
    return _host(out, p), c


def _check(y, ref, D, tol=1e-5):
    """RMS error within tol of the reference's RMS, per block of 64 D output samples."""
    assert y.shape == ref.shape
    blk = 64 * D
    for b0 in range(0, ref.size, blk):
        e, r = y[b0: b0 + blk], ref[b0: b0 + blk]
        err = np.sqrt(np.mean(np.abs(e - r) ** 2))
        rms = np.sqrt(np.mean(np.abs(r) ** 2))
        assert err <= tol * rms, f"samples {b0}..: err/rms {err / rms:.3g}"


def _tile(M, K):
    """Output frames per CTA, as synth_set_taps chooses them (synth.cu)."""
    P = max(1, min(16, 8192 // M))
    return max(4 * P, 16 * (K - 1))


def _grid():
    cases = []
    for M in (2, 8, 64, 256, 1024, 4096):
        Ds = [M, M // 2] + ([M // 4] if M >= 4 else []) + ([1] if M <= 8 else [])
        for D in sorted(set(Ds), reverse=True):
            taps = sorted({n for n in (1, D - 1, D, 3 * D + 5, min(16 * M, 32 * D)) if n >= 1})
            for i, ntaps in enumerate(taps):
                if M >= 1024:
                    cases.append((M, D, ntaps, S_VALUES[(i + D) % 3]))
                else:
                    cases.extend((M, D, ntaps, s) for s in S_VALUES)
    return cases


@pytest.mark.parametrize("M,D,ntaps,s", _grid())
def test_parity_with_reference(M, D, ntaps, s):
    from pothoscomms_b200 import Synthesizer
    K = -(-ntaps // D)
    # frames: several CTA tiles where the reference stays cheap (it costs M D (K + 1) per frame), at least 4
    F = max(4, min(2 * _tile(M, K) + 5, (1 << 24) // (M * D * (K + 1))))
    X = _frames(M, K - 1 + F + 3, seed=M * 7919 + D * 31 + ntaps)
    g = np.random.default_rng(ntaps).standard_normal(ntaps)
    sy = Synthesizer("complex_float32", M, D)
    sy.set_taps(g)
    assert sy.info() == (M, D, ntaps, K)
    y, _ = _run(sy, X, s, frames=F)
    _check(y, synthesize(X, g, M, D, s, samples=F * D), D)


def test_frequency_convention():
    from pothoscomms_b200 import Synthesizer
    M, D, s, A = 64, 32, 12345, 0.75
    nt, beta = signal.kaiserord(80.0, 1.0 / D)
    g = D * signal.firwin(nt, 1.0 / D, window=("kaiser", beta))   # every polyphase branch sums to 1
    assert nt <= min(16 * M, 32 * D)
    sy = Synthesizer("complex_float32", M, D)
    sy.set_taps(g)
    K = sy.info()[3]
    for c0 in (5, M - 3):                                   # c >= M/2 is the negative frequency c0 - M
        X = np.zeros((M, K - 1 + 100), dtype=np.complex64)
        X[c0] = A
        y, _ = _run(sy, X, s)
        m = np.arange(y.size)
        tone = A * np.exp(2j * np.pi * c0 * ((s + m) % M) / M)
        np.testing.assert_allclose(y, tone, rtol=0, atol=1e-3 * A)


@pytest.mark.parametrize("M,D,ntaps", [(64, 32, 3 * 32 + 5), (8, 1, 29), (1024, 1024, 4 * 1024 - 3), (256, 64, 32 * 64)])
def test_streaming_pieces_bit_identical(M, D, ntaps):
    torch = _torch()
    from pothoscomms_b200 import Synthesizer
    sy = Synthesizer("complex_float32", M, D)
    sy.set_taps(np.random.default_rng(3).standard_normal(ntaps))
    K = sy.info()[3]
    s0 = 2**33 + 11
    X = _frames(M, K - 1 + 700, seed=99)
    whole, cons = _run(sy, X, s0)
    rng = np.random.default_rng(5)
    pieces, pos, base = [], 0, s0                 # pos: first frame of the next piece's K-1 history
    while pos + K - 1 < X.shape[1]:
        step = int(rng.integers(1, 3 * _tile(M, K) // 2 + 3))
        buf = X[:, pos: pos + K - 1 + step]
        out = torch.zeros((buf.shape[1] * D + 1, 2), dtype=torch.float32, device="cuda")
        c, p = sy.run(_dev(buf), out, base)
        torch.cuda.synchronize()
        assert p == c * D
        pieces.append(out[:p].cpu())
        pos += c
        base += p
    got = torch.cat(pieces, dim=0)
    ref = torch.from_numpy(np.stack([whole.real, whole.imag], axis=-1).astype(np.float32))
    assert got.shape == ref.shape
    assert torch.equal(got, ref), "a stream fed in pieces must give the one-call output bit for bit"


def test_capacity_strides_and_padding():
    torch = _torch()
    from pothoscomms_b200 import Synthesizer
    M, D, ntaps, s = 64, 16, 100, 77
    sy = Synthesizer("complex_float32", M, D)
    g = np.random.default_rng(1).standard_normal(ntaps)
    sy.set_taps(g)
    K = sy.info()[3]
    n, stride = K - 1 + 300, K - 1 + 317
    X = _frames(M, n, seed=4)
    d_in = torch.full((M, stride, 2), float("nan"), dtype=torch.float32, device="cuda")
    d_in[:, :n] = _dev(X)                                  # NaN in every row's padding
    sentinel = 12345.5
    cap = 211 * D + 7                                      # 300 frames available, room for 211 (and 7 samples more)
    out = torch.full((300 * D + 64, 2), sentinel, dtype=torch.float32, device="cuda")
    c, p = sy.run(d_in, out, s, in_frames=n, out_capacity=cap)
    torch.cuda.synchronize()
    assert (c, p) == (211, 211 * D)
    o = out.cpu()
    assert torch.all(o[p:] == sentinel), "nothing may be written past `produced`"
    y = _host(out, p)
    assert np.all(np.isfinite(y))
    _check(y, synthesize(X, g, M, D, s, samples=cap), D)
    # below input_require: (0, 0) and nothing written
    out2 = torch.full((8 * D, 2), sentinel, dtype=torch.float32, device="cuda")
    assert sy.run(d_in, out2, s, in_frames=K - 1) == (0, 0)
    assert sy.run(d_in, out2, s, in_frames=K, out_capacity=D - 1) == (0, 0)
    torch.cuda.synchronize()
    assert torch.all(out2.cpu() == sentinel)
    assert sy.run(d_in, out2, s, in_frames=K) == (1, D)


@pytest.mark.parametrize("M", [64, 1024])
def test_roundtrip_on_one_stream(M):
    torch = _torch()
    from pothoscomms_b200 import Channelizer, Synthesizer
    D = M // 2
    h, g, s_shift, off = roundtrip_taps(M)
    s_a = 2**40 + 3
    ch = Channelizer("complex_float32", M, D)
    ch.set_taps(h)
    sy = Synthesizer("complex_float32", M, D)
    sy.set_taps(g)
    Fa = 300
    rng = np.random.default_rng(M)
    n = h.size - 1 + Fa * D
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_x = torch.from_numpy(x.view(np.float32).reshape(-1, 2)).cuda()
        mid = torch.empty((M, Fa, 2), dtype=torch.float32, device="cuda")
        assert ch.run(d_x, mid, s_a, stream=stream) == (Fa * D, Fa)
        Fs = Fa - (sy.info()[3] - 1)
        out = torch.empty((Fs * D, 2), dtype=torch.float32, device="cuda")
        assert sy.run(mid, out, s_a + s_shift, stream=stream) == (Fs, Fs * D)
    stream.synchronize()
    y = _host(out, Fs * D)
    ref = x[off: off + y.size].astype(np.complex128)
    db = 10 * np.log10(np.sum(np.abs(y - ref) ** 2) / np.sum(np.abs(ref) ** 2))
    assert db <= -80, db


def test_chain_channelizer_bank_synthesizer():
    torch = _torch()
    from pothoscomms_b200 import Channelizer, FirFilterBank, Synthesizer
    M, D = 64, 32
    h, g, s_shift, _ = roundtrip_taps(M)
    s_a = 12345
    gains = 1.0 + np.arange(M) / M
    ch = Channelizer("complex_float32", M, D)
    ch.set_taps(h)
    bank = FirFilterBank("complex_float32", "REAL", M)
    for c in range(M):
        bank.set_taps(c, [gains[c]])
    sy = Synthesizer("complex_float32", M, D)
    sy.set_taps(g)
    Fa = 200
    rng = np.random.default_rng(21)
    n = h.size - 1 + Fa * D
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_x = torch.from_numpy(x.view(np.float32).reshape(-1, 2)).cuda()
        mid = torch.empty((M, Fa, 2), dtype=torch.float32, device="cuda")
        assert ch.run(d_x, mid, s_a, stream=stream) == (Fa * D, Fa)
        eq = torch.empty((M, Fa, 2), dtype=torch.float32, device="cuda")
        assert bank.run(mid, eq, stream=stream) == (Fa, Fa)
        Fs = Fa - (sy.info()[3] - 1)
        out = torch.empty((Fs * D, 2), dtype=torch.float32, device="cuda")
        assert sy.run(eq, out, s_a + s_shift, stream=stream) == (Fs, Fs * D)
    stream.synchronize()
    Y = channelize(x, h, M, D, s_a) * gains[:, None]
    _check(_host(out, Fs * D), synthesize(Y, g, M, D, s_a + s_shift), D)


def test_taps_and_errors():
    torch = _torch()
    from pothoscomms_b200 import Synthesizer, _abi
    M, D, s = 16, 8, 3
    sy = Synthesizer("complex_float32", M, D)
    assert sy.info() == (M, D, 1, 1)                       # taps {1} after create
    X = _frames(M, 300, seed=12)
    y1, _ = _run(sy, X, s)
    _check(y1, synthesize(X, [1.0], M, D, s), D)
    g = np.random.default_rng(2).standard_normal(5 * D + 3)
    sy.set_taps(g)
    assert sy.info() == (M, D, g.size, 6)
    y2, _ = _run(sy, X, s)
    _check(y2, synthesize(X, g, M, D, s), D)
    sy.set_taps(g[:7])
    assert sy.info()[3] == 1
    y3, _ = _run(sy, X, s)
    _check(y3, synthesize(X, g[:7], M, D, s), D)

    lib, hh = _abi.lib(), sy._h
    limit = min(16 * M, 32 * D)
    one = np.ones(limit + 1)
    assert lib.b200c_synth_set_taps(hh, one.ctypes.data, 0) == _abi.ERR_INVALID
    assert lib.b200c_synth_set_taps(hh, one.ctypes.data, limit + 1) == _abi.ERR_INVALID
    assert sy.info()[2] == 7                                # a refused set_taps keeps the old taps
    y4, _ = _run(sy, X, s)
    assert np.array_equal(y4, y3)
    assert lib.b200c_synth_set_taps(hh, one.ctypes.data, limit) == _abi.OK
    assert sy.info()[3] == limit // D
    d_in = _dev(X)
    out = torch.empty((64 * D, 2), dtype=torch.float32, device="cuda")
    c, p = ctypes.c_size_t(), ctypes.c_size_t()
    args = (ctypes.byref(c), ctypes.byref(p), None)
    assert lib.b200c_synth_run(hh, None, 300, 300, s, ctypes.c_void_p(out.data_ptr()), 64 * D, *args) == _abi.ERR_INVALID
    assert lib.b200c_synth_run(hh, ctypes.c_void_p(d_in.data_ptr()), 300, 300, s, None, 64 * D, *args) == _abi.ERR_INVALID
    assert lib.b200c_synth_run(hh, ctypes.c_void_p(d_in.data_ptr()), 299, 300, s, ctypes.c_void_p(out.data_ptr()), 64 * D,
                               *args) == _abi.ERR_INVALID      # in_stride < in_frames
    assert lib.b200c_synth_run(hh, ctypes.c_void_p(d_in.data_ptr()), 300, 300, s, ctypes.c_void_p(out.data_ptr()), 64 * D,
                               *args) == _abi.OK
    assert (c.value, p.value) == (64, 64 * D)
    # nothing to produce: null buffers are fine
    assert lib.b200c_synth_run(hh, None, 3, 3, s, None, 64 * D, *args) == _abi.OK
    assert (c.value, p.value) == (0, 0)
    torch.cuda.synchronize()
