"""Real-output polyphase synthesis filter bank (b200c_rsynth_*) on the B200 against the reference
(tests/_rsynth_oracle.synthesize_real), the complex Synthesizer, and the RealChannelizer -> RealSynthesizer round
trip."""
import ctypes

import numpy as np
import pytest
from scipy import signal

from _rsynth_oracle import symmetric_extension, synthesize_real
from _synth_oracle import roundtrip_taps
from test_oracle_real_channelizer import real_channelize

pytestmark = pytest.mark.gpu

S_VALUES = (0, 12345, 2**40 + 7)


def _torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def _rows(M, n, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((M // 2 + 1, n)) + 1j * rng.standard_normal((M // 2 + 1, n))).astype(np.complex64)


def _dev(X):
    """[rows, n] complex -> CUDA [rows, n, 2] float32 (the real channelizer's output layout)."""
    torch = _torch()
    X = np.ascontiguousarray(np.asarray(X).astype(np.complex64))
    return torch.from_numpy(X.view(np.float32).reshape(X.shape[0], -1, 2)).cuda()


def _scalar(rs):
    import torch
    return torch.float32 if rs.dtype == _f32() else torch.int16


def _f32():
    from pothoscomms_b200 import _abi
    return _abi.F32


def _run(rs, X, s, frames=None):
    """One call on a fresh output tensor sized for `frames` output frames (default: all available).
    Returns (y [F D] on the host as float64, consumed)."""
    torch = _torch()
    M, nch, D, ntaps, K = rs.info()
    F = X.shape[1] - (K - 1) if frames is None else frames
    out = torch.empty(max(F * D, 1), dtype=_scalar(rs), device="cuda")
    c, p = rs.run(_dev(X), out, s, out_capacity=F * D)
    torch.cuda.synchronize()
    assert (c, p) == (F, F * D)
    return out[:p].cpu().numpy().astype(np.float64), c


def _check(y, ref, D, tol=1e-5):
    """RMS error within tol of the reference's RMS, per block of 64 D output samples."""
    assert y.shape == ref.shape
    blk = 64 * D
    for b0 in range(0, ref.size, blk):
        e, r = y[b0: b0 + blk], ref[b0: b0 + blk]
        err = np.sqrt(np.mean((e - r) ** 2))
        rms = np.sqrt(np.mean(r ** 2))
        assert err <= tol * rms, f"samples {b0}..: err/rms {err / rms:.3g}"


def _tile(M, K):
    """Output frames per CTA, as rsynth_set_taps chooses them (rsynth.cu, synth.cu)."""
    P = max(1, min(16, 8192 // (M // 2)))
    return max(4 * P, 16 * (K - 1))


def _groups(M, K):
    """CTAs that split the M real bins of one tile (gridDim.y), as rsynth_set_taps chooses them."""
    return M // min(M, 1024 if K <= 12 else 512 if K <= 24 else 256)


def _grid():
    cases = []
    for M in (2, 8, 64, 256, 1024, 2048, 8192):
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
    from pothoscomms_b200 import RealSynthesizer
    K = -(-ntaps // D)
    T = _tile(M, K)
    F = 2 * T + 5                                           # two CTA tiles and a ragged third
    X = _rows(M, K - 1 + F + 3, seed=M * 7919 + D * 31 + ntaps)
    g = np.random.default_rng(ntaps).standard_normal(ntaps)
    rs = RealSynthesizer("float32", M, D)
    rs.set_taps(g)
    assert rs.info() == (M, M // 2 + 1, D, ntaps, K)
    y, _ = _run(rs, X, s, frames=F)
    # the dense reference costs about (M/2 + 1) D (K + 2) per frame: where the whole run is too dear, check the frames
    # on both sides of every tile boundary and at both ends
    if (M // 2 + 1) * D * (K + 2) * F <= 1 << 25:
        windows = [(0, F)]
    else:
        windows = [(0, 1), (T - 1, T + 1), (2 * T - 1, 2 * T + 1), (F - 1, F)]
    for t0, t1 in windows:
        ref = synthesize_real(X[:, t0: t0 + K - 1 + t1 - t0], g, M, D, s + t0 * D)
        _check(y[t0 * D: t1 * D], ref, D)


def test_grid_splits_bins():
    # the parity grid covers bins split over gridDim.y at M = 2048 and 8192, and unsplit tiles
    cases = {(M, _groups(M, -(-n // D))) for M, D, n, _ in _grid()}
    assert (2048, 2) in cases and (8192, 8) in cases and (8192, 32) in cases and (256, 1) in cases


@pytest.mark.parametrize("M,D,ntaps", [(8, 2, 13), (256, 128, 3 * 128 + 5), (4096, 2048, 8 * 2048 + 1)])
def test_agrees_with_complex_synthesizer(M, D, ntaps):
    torch = _torch()
    from pothoscomms_b200 import RealSynthesizer, Synthesizer
    s = 2**40 + 7
    g = np.random.default_rng(M).standard_normal(ntaps)
    rs = RealSynthesizer("float32", M, D)
    rs.set_taps(g)
    sy = Synthesizer("complex_float32", M, D)
    sy.set_taps(g)
    K = rs.info()[4]
    F = 2 * _tile(M, K) + 3
    X = _rows(M, K - 1 + F, seed=M + 1)
    y, _ = _run(rs, X, s)
    out = torch.empty((F * D, 2), dtype=torch.float32, device="cuda")
    assert sy.run(_dev(symmetric_extension(X, M)), out, s) == (F, F * D)
    torch.cuda.synchronize()
    _check(y, out[:, 0].cpu().numpy().astype(np.float64), D)


def test_frequency_convention():
    from pothoscomms_b200 import RealSynthesizer
    M, D, s, A = 64, 32, 12345, 0.75
    N = M // 2
    nt, beta = signal.kaiserord(80.0, 1.0 / D)
    g = D * signal.firwin(nt, 1.0 / D, window=("kaiser", beta))   # every polyphase branch sums to 1
    assert nt <= min(16 * M, 32 * D)
    rs = RealSynthesizer("float32", M, D)
    rs.set_taps(g)
    K = rs.info()[4]
    for c0 in (0, 5, N - 1, N):
        X = np.zeros((N + 1, K - 1 + 100), dtype=np.complex64)
        X[c0] = A * (1 - 0.5j) if 0 < c0 < N else A   # a complex constant turns the cosine; rows 0 and N are real
        y, _ = _run(rs, X, s)
        m = np.arange(y.size)
        if c0 == 0:
            tone = np.full(y.size, A)
        elif c0 == N:
            tone = A * (-1.0) ** ((s + m) % 2)
        else:
            tone = 2 * np.real(A * (1 - 0.5j) * np.exp(2j * np.pi * c0 * ((s + m) % M) / M))
        np.testing.assert_allclose(y, tone, rtol=0, atol=1e-3 * A)
    # a plain real constant in row c0 gives 2 A cos(2 pi c0 (s + m) / M)
    X = np.zeros((N + 1, K - 1 + 100), dtype=np.complex64)
    X[7] = A
    y, _ = _run(rs, X, s)
    m = np.arange(y.size)
    np.testing.assert_allclose(y, 2 * A * np.cos(2 * np.pi * 7 * ((s + m) % M) / M), rtol=0, atol=1e-3 * A)


@pytest.mark.parametrize("M,D,ntaps", [(64, 32, 3 * 32 + 5), (2048, 2048, 4 * 2048 - 3), (8, 1, 29)])
def test_int16_output_is_rounded_saturated_float32(M, D, ntaps):
    from pothoscomms_b200 import RealSynthesizer
    g = np.random.default_rng(4).standard_normal(ntaps)
    r32 = RealSynthesizer("float32", M, D)
    r16 = RealSynthesizer("int16", M, D)
    r32.set_taps(g)
    r16.set_taps(g)
    K = r32.info()[4]
    F = 2 * _tile(M, K) + 7
    X = _rows(M, K - 1 + F, seed=9)
    y32, _ = _run(r32, X, 3, frames=F)
    scale = 60000.0 / np.abs(y32).max()                      # some samples beyond both rails
    Xs = (X * scale).astype(np.complex64)
    y32, _ = _run(r32, Xs, 3, frames=F)
    y16, _ = _run(r16, Xs, 3, frames=F)
    want = np.clip(np.rint(y32), -32768, 32767)               # np.rint rounds ties to even, as __float2int_rn
    assert (want == 32767).any() and (want == -32768).any()
    assert np.array_equal(y16, want)
    # a few hand-made ties and extremes through a unit tap and row 0 alone
    r16.set_taps([1.0])
    r32.set_taps([1.0])
    vals = np.array([0.5, 1.5, 2.5, -0.5, -1.5, -2.5, 32766.5, 32767.5, -32768.5, 1e9, -1e9, 7.49], dtype=np.float32)
    Xe = np.zeros((M // 2 + 1, vals.size), dtype=np.complex64)
    Xe[0] = vals
    y16, _ = _run(r16, Xe, 0)
    y32, _ = _run(r32, Xe, 0)
    assert np.array_equal(y16, np.clip(np.rint(y32), -32768, 32767))
    assert y16[::D].tolist() == [0, 2, 2, 0, -2, -2, 32766, 32767, -32768, 32767, -32768, 7]


@pytest.mark.parametrize("dtype", ["float32", "int16"])
@pytest.mark.parametrize("M,D,ntaps", [(64, 32, 3 * 32 + 5), (8, 1, 29), (2048, 1024, 16 * 1024), (8192, 8192, 8192)])
def test_streaming_pieces_bit_identical(dtype, M, D, ntaps):
    torch = _torch()
    from pothoscomms_b200 import RealSynthesizer
    rs = RealSynthesizer(dtype, M, D)
    rs.set_taps(np.random.default_rng(3).standard_normal(ntaps) * (300.0 if dtype == "int16" else 1.0))
    K = rs.info()[4]
    s0 = 2**33 + 11
    total = 3 * _tile(M, K) + 11 if M < 8192 else 2 * _tile(M, K) + 3
    X = _rows(M, K - 1 + total, seed=99)
    whole, _ = _run(rs, X, s0)
    rng = np.random.default_rng(5)
    pieces, pos, base = [], 0, s0                 # pos: first frame of the next piece's K-1 history
    while pos + K - 1 < X.shape[1]:
        step = int(rng.integers(1, 3 * _tile(M, K) // 2 + 3))
        buf = X[:, pos: pos + K - 1 + step]
        room = torch.zeros(step * D + 2, dtype=_scalar(rs), device="cuda")
        out = room[1:]                            # starts at an odd element offset
        c, p = rs.run(_dev(buf), out, base)
        torch.cuda.synchronize()
        assert p == c * D and c == min(step, buf.shape[1] - (K - 1))
        assert room[0].item() == 0
        pieces.append(out[:p].cpu())
        pos += c
        base += p
    got = torch.cat(pieces).numpy().astype(np.float64)
    assert got.shape == whole.shape
    assert np.array_equal(got, whole), "a stream fed in pieces must give the one-call output bit for bit"


def test_capacity_strides_and_padding():
    torch = _torch()
    from pothoscomms_b200 import RealSynthesizer
    M, D, ntaps, s = 64, 16, 100, 77
    N = M // 2
    rs = RealSynthesizer("float32", M, D)
    g = np.random.default_rng(1).standard_normal(ntaps)
    rs.set_taps(g)
    K = rs.info()[4]
    n, stride = K - 1 + 300, K - 1 + 317
    X = _rows(M, n, seed=4)
    d_in = torch.full((N + 1, stride, 2), float("nan"), dtype=torch.float32, device="cuda")
    d_in[:, :n] = _dev(X)                                  # NaN in every row's padding
    d_in[0, :, 1] = float("nan")                           # and in the imaginary parts of rows 0 and N
    d_in[N, :, 1] = float("nan")
    sentinel = 12345.5
    cap = 211 * D + 7                                      # 300 frames available, room for 211 (and 7 samples more)
    out = torch.full((300 * D + 64,), sentinel, dtype=torch.float32, device="cuda")
    c, p = rs.run(d_in, out, s, in_frames=n, out_capacity=cap)
    torch.cuda.synchronize()
    assert (c, p) == (211, 211 * D)
    o = out.cpu()
    assert torch.all(o[p:] == sentinel), "nothing may be written past `produced`"
    y = o[:p].numpy().astype(np.float64)
    assert np.all(np.isfinite(y))
    _check(y, synthesize_real(X, g, M, D, s, samples=cap), D)
    # below input_require: (0, 0) and nothing written
    out2 = torch.full((8 * D,), sentinel, dtype=torch.float32, device="cuda")
    assert rs.run(d_in, out2, s, in_frames=K - 1) == (0, 0)
    assert rs.run(d_in, out2, s, in_frames=K, out_capacity=D - 1) == (0, 0)
    torch.cuda.synchronize()
    assert torch.all(out2.cpu() == sentinel)
    assert rs.run(d_in, out2, s, in_frames=K) == (1, D)
    torch.cuda.synchronize()
    assert torch.all(out2[D:].cpu() == sentinel)


@pytest.mark.parametrize("M", [64, 2048])
def test_roundtrip_on_one_stream(M):
    torch = _torch()
    from pothoscomms_b200 import RealChannelizer, RealSynthesizer
    D = M // 2
    h, g, s_shift, off = roundtrip_taps(M)
    s_a = 2**40 + 3
    ch = RealChannelizer("float32", M, D)
    ch.set_taps(h)
    rs = RealSynthesizer("float32", M, D)
    rs.set_taps(g)
    Fa = 300
    x = np.random.default_rng(M).standard_normal(h.size - 1 + Fa * D).astype(np.float32)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_x = torch.from_numpy(x).cuda()
        mid = torch.empty((M // 2 + 1, Fa, 2), dtype=torch.float32, device="cuda")
        assert ch.run(d_x, mid, s_a, stream=stream) == (Fa * D, Fa)
        Fs = Fa - (rs.info()[4] - 1)
        out = torch.empty(Fs * D, dtype=torch.float32, device="cuda")
        assert rs.run(mid, out, s_a + s_shift, stream=stream) == (Fs, Fs * D)
    stream.synchronize()
    y = out.cpu().numpy().astype(np.float64)
    ref = x[off: off + y.size].astype(np.float64)
    db = 10 * np.log10(np.sum((y - ref) ** 2) / np.sum(ref ** 2))
    assert db <= -80, db


def test_int16_roundtrip_within_one_lsb():
    torch = _torch()
    from pothoscomms_b200 import RealChannelizer, RealSynthesizer
    M = 64
    D = M // 2
    h, g, s_shift, off = roundtrip_taps(M)
    s_a = 12345
    ch = RealChannelizer("int16", M, D)
    ch.set_taps(h)
    rs = RealSynthesizer("int16", M, D)
    rs.set_taps(g)
    Fa = 400
    n = h.size - 1 + Fa * D
    rng = np.random.default_rng(17)
    m = np.arange(n)
    x = np.rint(1000 * np.sin(2 * np.pi * 0.0123 * m) + 700 * rng.standard_normal(n)).astype(np.int16)
    assert 900 < np.sqrt(np.mean(x.astype(np.float64) ** 2)) < 1400
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_x = torch.from_numpy(x).cuda()
        mid = torch.empty((M // 2 + 1, Fa, 2), dtype=torch.float32, device="cuda")
        assert ch.run(d_x, mid, s_a, stream=stream) == (Fa * D, Fa)
        Fs = Fa - (rs.info()[4] - 1)
        out = torch.empty(Fs * D, dtype=torch.int16, device="cuda")
        assert rs.run(mid, out, s_a + s_shift, stream=stream) == (Fs, Fs * D)
    stream.synchronize()
    y = out.cpu().numpy().astype(np.int32)
    ref = x[off: off + y.size].astype(np.int32)
    assert np.abs(y - ref).max() <= 1


def test_chain_real_channelizer_bank_real_synthesizer():
    torch = _torch()
    from pothoscomms_b200 import FirFilterBank, RealChannelizer, RealSynthesizer
    M, D = 64, 32
    nch = M // 2 + 1
    h, g, s_shift, _ = roundtrip_taps(M)
    s_a = 2**40 + 5
    gains = 1.0 + np.arange(nch) / nch
    ch = RealChannelizer("float32", M, D)
    ch.set_taps(h)
    bank = FirFilterBank("complex_float32", "REAL", nch)
    for c in range(nch):
        bank.set_taps(c, [gains[c]])
    rs = RealSynthesizer("float32", M, D)
    rs.set_taps(g)
    Fa = 200
    x = np.random.default_rng(21).standard_normal(h.size - 1 + Fa * D).astype(np.float32)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        d_x = torch.from_numpy(x).cuda()
        mid = torch.empty((nch, Fa, 2), dtype=torch.float32, device="cuda")
        assert ch.run(d_x, mid, s_a, stream=stream) == (Fa * D, Fa)
        eq = torch.empty((nch, Fa, 2), dtype=torch.float32, device="cuda")
        assert bank.run(mid, eq, stream=stream) == (Fa, Fa)
        Fs = Fa - (rs.info()[4] - 1)
        out = torch.empty(Fs * D, dtype=torch.float32, device="cuda")
        assert rs.run(eq, out, s_a + s_shift, stream=stream) == (Fs, Fs * D)
    stream.synchronize()
    Y = real_channelize(x, h, M, D, s_a) * gains[:, None]
    _check(out.cpu().numpy().astype(np.float64), synthesize_real(Y, g, M, D, s_a + s_shift), D)


def test_taps_and_errors():
    torch = _torch()
    from pothoscomms_b200 import RealSynthesizer, _abi
    M, D, s = 16, 8, 3
    rs = RealSynthesizer("float32", M, D)
    assert rs.info() == (M, M // 2 + 1, D, 1, 1)            # taps {1} after create
    X = _rows(M, 300, seed=12)
    y1, _ = _run(rs, X, s)
    _check(y1, synthesize_real(X, [1.0], M, D, s), D)
    g = np.random.default_rng(2).standard_normal(5 * D + 3)
    rs.set_taps(g)
    assert rs.info() == (M, M // 2 + 1, D, g.size, 6)
    y2, _ = _run(rs, X, s)
    _check(y2, synthesize_real(X, g, M, D, s), D)
    rs.set_taps(g[:7])
    assert rs.info()[4] == 1
    y3, _ = _run(rs, X, s)
    _check(y3, synthesize_real(X, g[:7], M, D, s), D)

    lib, hh = _abi.lib(), rs._h
    limit = min(16 * M, 32 * D)
    one = np.ones(limit + 1)
    assert lib.b200c_rsynth_set_taps(hh, one.ctypes.data, 0) == _abi.ERR_INVALID
    assert lib.b200c_rsynth_set_taps(hh, one.ctypes.data, limit + 1) == _abi.ERR_INVALID
    assert rs.info()[3] == 7                                # a refused set_taps keeps the old taps
    y4, _ = _run(rs, X, s)
    assert np.array_equal(y4, y3)
    assert lib.b200c_rsynth_set_taps(hh, one.ctypes.data, limit) == _abi.OK
    assert rs.info()[4] == limit // D
    d_in = _dev(X)
    out = torch.empty(64 * D, dtype=torch.float32, device="cuda")
    c, p = ctypes.c_size_t(), ctypes.c_size_t()
    args = (ctypes.byref(c), ctypes.byref(p), None)
    assert lib.b200c_rsynth_run(hh, None, 300, 300, s, ctypes.c_void_p(out.data_ptr()), 64 * D, *args) == _abi.ERR_INVALID
    assert lib.b200c_rsynth_run(hh, ctypes.c_void_p(d_in.data_ptr()), 300, 300, s, None, 64 * D, *args) == _abi.ERR_INVALID
    assert lib.b200c_rsynth_run(hh, ctypes.c_void_p(d_in.data_ptr()), 299, 300, s, ctypes.c_void_p(out.data_ptr()), 64 * D,
                                *args) == _abi.ERR_INVALID      # in_stride < in_frames
    assert lib.b200c_rsynth_run(hh, ctypes.c_void_p(d_in.data_ptr()), 300, 300, s, ctypes.c_void_p(out.data_ptr()), 64 * D,
                                *args) == _abi.OK
    assert (c.value, p.value) == (64, 64 * D)
    # nothing to produce: null buffers are fine
    assert lib.b200c_rsynth_run(hh, None, 3, 3, s, None, 64 * D, *args) == _abi.OK
    assert (c.value, p.value) == (0, 0)
    torch.cuda.synchronize()
