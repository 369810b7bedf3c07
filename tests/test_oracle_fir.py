"""Tests pinning the FIR oracle (CPU, no GPU needed).

1. Against the REFERENCE ITSELF: filter/FIRFilter.cpp compiled unmodified into oracle/_ref/libfirref.so
   (oracle/Makefile ref_fir; Pothos API subset + a recalled QFormat.hpp): bit-for-bit on all 18 factory
   rows x the rate grid x burst flush x chunked streaming, plus _inputRequire and the thrown messages.
2. Structural identities that follow from filter/FIRFilter.cpp:278-302,327-354 and an independent numpy
   restatement of the loop nest (the reference's own test, filter/TestFIRFilter.cpp:78, only asserts
   rms > 0.1*amplitude).
"""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def naive_reference(x, taps, M, L):
    """Independent numpy statement of FIRFilter.cpp:286-302 via zero-stuffing:
    upsample by L (zeros), filter with the full taps, keep samples where (i+1) % M == 0."""
    K = -(-len(taps) // L)
    xs = x[K - 1:]  # x = in + (K-1)
    N = (len(x) - (K - 1)) // M * M
    up = np.zeros((len(x)) * L, dtype=np.result_type(x, taps))
    up[::L] = x  # up[(n + K - 1)*L] = x[n]
    out = []
    for i in range(N * L):
        if (i + 1) % M:
            continue
        # y = sum_k h[j + kL] x[n-k] with i = nL + j  ==  sum_t h[t] up_x[i - t]
        acc = 0
        for t in range(len(taps)):
            idx = i - t + (K - 1) * L
            if 0 <= idx < len(up):
                acc = acc + taps[t] * up[idx]
        out.append(acc)
    return np.array(out), N, xs


def test_K_and_input_require(oracle):
    assert oracle.fir_K(1, 1) == 1
    assert oracle.fir_K(101, 1) == 101
    assert oracle.fir_K(101, 3) == 34      # ceil(101/3), FIRFilter.cpp:335
    assert oracle.fir_K(255, 3) == 85
    assert oracle.fir_K(2, 5) == 1


def test_phase_split(oracle):
    # _interpTaps[j][k] = taps[j + k*L]; later phases may be one tap shorter (FIRFilter.cpp:340-350)
    taps = np.arange(1, 8, dtype=np.float64)
    tp, nt = oracle.fir_phase_taps(oracle.F64, False, taps, 3)
    assert list(nt) == [3, 2, 2]
    assert list(tp[0, :, 0]) == [1, 4, 7]
    assert list(tp[1, :, 0]) == [2, 5, 0]
    assert list(tp[2, :, 0]) == [3, 6, 0]


def test_float_to_q_truncates_toward_zero(oracle):
    # floatToQ<int32>(x) = int32(ldexp(x, 16)); parity-unpinned assumption, see oracle/qformat.h
    tp, _ = oracle.fir_phase_taps(oracle.I16, False, np.array([0.5, -0.5, 1.0 / 3, -1.0 / 3, 1.0]), 1)
    assert list(tp[0, :, 0]) == [32768, -32768, 21845, -21845, 65536]
    tp8, _ = oracle.fir_phase_taps(oracle.I8, False, np.array([0.5, -1.0 / 3]), 1)
    assert list(tp8[0, :, 0]) == [128, -85]
    tp32, _ = oracle.fir_phase_taps(oracle.I32, False, np.array([0.5, -1.0 / 3]), 1)
    assert list(tp32[0, :, 0]) == [2 ** 31, -1431655765]


@pytest.mark.parametrize("dt", ["F32", "CF32", "F64", "CF64", "I8", "CI8", "I16", "CI16", "I32", "CI32", "I64", "CI64"])
def test_default_taps_passthrough(oracle, dt):
    # ctor taps {1} (FIRFilter.cpp:125): K = 1, output == input for every type (the
    # Scale/Rotate identity in*2^n >> n == in, math/TestScale.cpp:47-53)
    code = getattr(oracle, dt)
    rng = np.random.default_rng(1)
    nc = 2 if code & 1 else 1
    sc = oracle.scalar_np(code)
    if np.issubdtype(sc, np.integer):
        info = np.iinfo(sc)
        lim = min(info.max, 2 ** 31 - 1)  # keep int64 data inside the >>32 Q range
        x = rng.integers(-lim - 1, lim + 1, size=(257, nc)).astype(sc)
    else:
        x = rng.standard_normal((257, nc)).astype(sc)
    y, cons, prod = oracle.fir(code, False, [1.0], 1, 1, x)
    assert cons == 257 and prod == 257
    assert np.array_equal(y, x)


def test_impulse_response_is_taps(oracle):
    taps = np.array([0.25, -0.5, 0.125, 1.0, 0.75])
    K = 5
    x = np.zeros((K - 1 + 10, 1), dtype=np.float32)
    x[K - 1, 0] = 1.0  # impulse at the first non-history sample
    y, cons, prod = oracle.fir(oracle.F32, False, taps, 1, 1, x)
    assert cons == 10 and prod == 10
    assert np.array_equal(y[:5, 0], taps.astype(np.float32))
    assert np.all(y[5:] == 0)


def test_valid_convolution_no_zero_history(oracle):
    # first K-1 inputs are history only (FIRFilter.cpp:281): equals numpy 'valid' convolution
    rng = np.random.default_rng(5)
    taps = rng.standard_normal(17)
    x = rng.standard_normal((300, 1))
    y, cons, prod = oracle.fir(oracle.F64, False, taps, 1, 1, x)
    ref = np.convolve(x[:, 0], taps, mode="valid")
    assert prod == len(ref) == 300 - 16
    assert np.allclose(y[:, 0], ref, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("M,L", [(1, 1), (2, 1), (3, 1), (1, 2), (1, 3), (2, 3), (3, 2), (3, 3), (5, 4), (4, 6), (7, 3)])
def test_polyphase_matches_zero_stuffing(oracle, M, L):
    rng = np.random.default_rng(M * 10 + L)
    taps = rng.standard_normal(23)
    x = rng.standard_normal(200)
    ref, N, _ = naive_reference(x, taps, M, L)
    y, cons, prod = oracle.fir(oracle.F64, False, taps, M, L, x.reshape(-1, 1))
    assert cons == N and prod == N // M * L == len(ref)
    assert np.allclose(y[:, 0], ref, rtol=1e-11, atol=1e-11)


def test_complex_taps_complex_data(oracle):
    rng = np.random.default_rng(11)
    taps = rng.standard_normal(9) + 1j * rng.standard_normal(9)
    x = rng.standard_normal(100) + 1j * rng.standard_normal(100)
    ref, N, _ = naive_reference(x, taps, 2, 3)
    y, cons, prod = oracle.fir(oracle.CF64, True, taps, 2, 3, oracle.to_raw(x, oracle.CF64))
    assert np.allclose(y.view(np.complex128).ravel(), ref, rtol=1e-11, atol=1e-11)


def test_int16_q16_exact_small_case(oracle):
    # y = (sum_k int32(trunc(h*2^16)) * x[n-k]) >> 16, wrapping int32, then int16 cast
    taps = np.array([0.5, -0.25, 0.3])
    q = np.trunc(taps * 65536).astype(np.int64)
    x = np.array([100, -200, 300, 32767, -32768, 5, 7, -9], dtype=np.int16)
    K = 3
    exp = []
    for n in range(len(x) - (K - 1)):
        acc = sum(int(q[k]) * int(x[n + K - 1 - k]) for k in range(K))
        acc = (acc + 2 ** 31) % 2 ** 32 - 2 ** 31
        exp.append(np.int16(((acc >> 16) + 2 ** 15) % 2 ** 16 - 2 ** 15))
    y, _, _ = oracle.fir(oracle.I16, False, taps, 1, 1, x.reshape(-1, 1))
    assert list(y[:, 0]) == exp


def test_int16_accumulator_wraps(oracle):
    # |sum| exceeds int32: the reference's int32 QType wraps (FIRFilter.cpp:381)
    taps = np.full(64, 1.99)
    x = np.full((64 + 63, 1), 32767, dtype=np.int16)
    y, _, _ = oracle.fir(oracle.I16, False, taps, 1, 1, x)
    acc = 64 * int(np.trunc(1.99 * 65536)) * 32767
    acc = (acc + 2 ** 31) % 2 ** 32 - 2 ** 31
    assert y[0, 0] == np.int16(((acc >> 16) + 2 ** 15) % 2 ** 16 - 2 ** 15)


def test_complex_int16_matches_python_ints(oracle):
    rng = np.random.default_rng(2)
    taps = (rng.standard_normal(5) + 1j * rng.standard_normal(5)) * 0.3
    qr = np.trunc(taps.real * 65536).astype(np.int64)
    qi = np.trunc(taps.imag * 65536).astype(np.int64)
    x = rng.integers(-32768, 32768, size=(40, 2), dtype=np.int16)
    K = 5

    def wrap32(v):
        return (v + 2 ** 31) % 2 ** 32 - 2 ** 31

    exp = []
    for n in range(40 - (K - 1)):
        ar = ai = 0
        for k in range(K):
            xr, xi = int(x[n + K - 1 - k, 0]), int(x[n + K - 1 - k, 1])
            ar += int(qr[k]) * xr - int(qi[k]) * xi
            ai += int(qr[k]) * xi + int(qi[k]) * xr
        exp.append([np.int16((((wrap32(ar) >> 16)) + 2 ** 15) % 2 ** 16 - 2 ** 15),
                    np.int16((((wrap32(ai) >> 16)) + 2 ** 15) % 2 ** 16 - 2 ** 15)])
    y, _, _ = oracle.fir(oracle.CI16, True, taps, 1, 1, x)
    assert np.array_equal(y, np.array(exp, dtype=np.int16))


def test_N_is_limited_by_output_capacity(oracle):
    # N = min((elems-(K-1))/M, outElems/L)*M (FIRFilter.cpp:278)
    x = np.arange(100, dtype=np.float32).reshape(-1, 1)
    y, cons, prod = oracle.fir(oracle.F32, False, [1.0, 1.0, 1.0], 2, 3, x, out_capacity=10)
    assert prod == 9 and cons == 6  # outElems/L = 3 blocks
    y, cons, prod = oracle.fir(oracle.F32, False, [1.0, 1.0, 1.0], 2, 3, x, out_capacity=10 ** 6)
    assert cons == (100 - 0) // 2 * 2 and prod == 150  # K = 1 for 3 taps at L=3


def test_insufficient_input_produces_nothing(oracle):
    x = np.ones((5, 1), dtype=np.float32)
    y, cons, prod = oracle.fir(oracle.F32, False, np.ones(8), 1, 1, x)  # needs M + K - 1 = 8
    assert cons == 0 and prod == 0


def test_burst_zero_tail_preserves_length(oracle):
    # flush appends K-1 zeros so B inputs give B*L/M outputs (FIRFilter.cpp:265-272,
    # filter/TestFIRDesigner.cpp:183 expects exactly fftSize outputs)
    rng = np.random.default_rng(9)
    taps = rng.standard_normal(101)
    x = rng.standard_normal((1024, 1))
    y, cons, prod = oracle.fir(oracle.F64, False, taps, 1, 1, x, zero_tail=True)
    assert cons == 1024 and prod == 1024
    full = np.convolve(np.concatenate([x[:, 0], np.zeros(100)]), taps, mode="valid")
    assert np.allclose(y[:, 0], full, atol=1e-12)


def test_multithreaded_driver_equals_single(oracle):
    rng = np.random.default_rng(4)
    taps = rng.standard_normal(31) + 1j * rng.standard_normal(31)
    x = rng.standard_normal((5000, 2)).astype(np.float32)
    a = oracle.fir(oracle.CF32, True, taps, 2, 3, x)
    b = oracle.fir(oracle.CF32, True, taps, 2, 3, x, threads=4)
    assert a[1:] == b[1:] and np.array_equal(a[0], b[0])


def test_fir_golden_fixtures(oracle):
    """tests/golden/fir_*.npz are outputs of the REFERENCE's compiled block (make_golden.py, `source` field): one work()
    call, and the first 500 inputs as a burst flushed by a frame-end label (the oracle's zero_tail=True)."""
    files = sorted(f for f in os.listdir(GOLDEN) if f.startswith("fir_") and f.endswith(".npz"))
    assert files
    for fn in files:
        g = np.load(os.path.join(GOLDEN, fn))
        args = (int(g["dtype"]), bool(g["taps_complex"]), g["taps"], int(g["M"]), int(g["L"]))
        y, cons, prod = oracle.fir(*args, g["x"])
        assert cons == int(g["consumed"]) and prod == int(g["produced"]), fn
        assert np.array_equal(y.view(np.uint8), g["y"].view(np.uint8)), fn
        yb, cb, pb = oracle.fir(*args, g["x"][:500], zero_tail=True)
        assert cb == int(g["burst_consumed"]) and pb == int(g["burst_produced"]), fn
        assert np.array_equal(yb.view(np.uint8), g["burst_y"].view(np.uint8)), fn
        assert str(g["source"]) == "reference:filter/FIRFilter.cpp", fn


# ------------------------------------------------------------------------------------------------
# Pinned against the reference's own compiled block (oracle/_ref/libfirref.so)
# ------------------------------------------------------------------------------------------------
RATES = [(1, 1), (2, 1), (3, 1), (1, 2), (1, 3), (2, 2), (2, 3), (3, 2), (3, 3), (5, 4), (4, 6), (7, 3), (16, 1), (1, 16)]
ROWS = [(dt, tcx) for dt in ("F32", "CF32", "F64", "CF64", "I8", "CI8", "I16", "CI16", "I32", "CI32", "I64", "CI64")
        for tcx in (False, True) if not (tcx and dt[0] != "C")]


def _rand_stream(oracle, code, n, rng):
    nc = 2 if code & 1 else 1
    sc = oracle.scalar_np(code)
    if np.issubdtype(sc, np.integer):
        info = np.iinfo(sc)
        return rng.integers(info.min, info.max, size=(n, nc), endpoint=True).astype(sc)   # full scale: sums wrap
    return rng.standard_normal((n, nc)).astype(sc)


def _rand_taps(ntaps, tcx, rng, scale=0.3):
    t = rng.standard_normal(ntaps) * scale
    return t + 1j * rng.standard_normal(ntaps) * scale if tcx else t


def _same_bits(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


needs_ref = pytest.mark.skipif(not os.path.exists(os.path.join(os.path.dirname(__file__), "..", "oracle", "_ref", "libfirref.so"))
                               and not os.path.exists("/root/reference/filter/FIRFilter.cpp"),
                               reason="oracle/_ref/libfirref.so not built and no reference checkout")


@needs_ref
def test_reference_factory_has_18_rows(oracle):
    assert len(ROWS) == 18   # filter/FIRFilter.cpp:373-382
    for dt, tcx in ROWS:
        oracle.ref_fir(getattr(oracle, dt), tcx, [1.0], 1, 1, np.zeros((4, 2)))
    for dt in ("F32", "F64", "I8", "I16", "I32", "I64"):   # real data + COMPLEX taps throws (:383)
        with pytest.raises(oracle.ReferenceError_, match=r"FIRFilterFactory\(.*\).*unsupported types"):
            oracle.ref_fir(getattr(oracle, dt), True, [1.0 + 0j], 1, 1, np.zeros((4, 1)))


@needs_ref
@pytest.mark.parametrize("dt,tcx", ROWS)
def test_oracle_equals_reference_block_on_rate_grid(oracle, dt, tcx):
    """oracle.fir (the restatement every GPU parity test compares with) == one work() of the reference's own
    compiled block, bit for bit (floats too: same scalar order, no contraction), 18 rows x RATES."""
    code = getattr(oracle, dt)
    rng = np.random.default_rng(sum(map(ord, dt)) * 2 + tcx)
    x = _rand_stream(oracle, code, 1500, rng)
    for M, L in RATES:
        for ntaps in (1, 2, 33, 101):
            taps = _rand_taps(ntaps, tcx, rng)
            y, c, p = oracle.fir(code, tcx, taps, M, L, x)
            yr, cr, pr = oracle.ref_fir(code, tcx, taps, M, L, x)
            assert (c, p) == (cr, pr), (M, L, ntaps)
            assert _same_bits(y, yr), (M, L, ntaps)
            assert oracle.ref_fir_input_require(code, tcx, taps, M, L) == M + oracle.fir_K(ntaps, L) - 1   # :353


@needs_ref
@pytest.mark.parametrize("dt,tcx", ROWS)
def test_oracle_zero_tail_equals_reference_burst_flush(oracle, dt, tcx):
    """A burst ending in a frame-end label: the reference flushes it through a K-1 zero tail (:226-229,263-272)
    over as many work() calls as it takes; the oracle's zero_tail=True is the same samples in one call."""
    code = getattr(oracle, dt)
    rng = np.random.default_rng(7700 + sum(map(ord, dt)) * 2 + tcx)
    for M, L in RATES:
        for ntaps, B in ((33, 400), (101, 257), (7, 64)):
            K = oracle.fir_K(ntaps, L)
            x = _rand_stream(oracle, code, B, rng)
            taps = _rand_taps(ntaps, tcx, rng)
            y, c, p = oracle.fir(code, tcx, taps, M, L, x, zero_tail=True)
            yr, cr, pr, calls = oracle.ref_fir_stream(code, tcx, taps, M, L, x, frame_end=True)
            assert (c, p) == (cr, pr) == (B // M * M, B // M * L), (M, L, ntaps, B)
            assert _same_bits(y, yr), (M, L, ntaps, B)
            assert calls >= (2 if B >= M + K - 1 and K > 1 else 1)


@needs_ref
@pytest.mark.parametrize("dt,tcx", [("CF32", True), ("CF32", False), ("F32", False), ("CI16", True), ("I16", False), ("CI8", True),
                                    ("I64", False)])
def test_reference_streaming_in_chunks_equals_one_work_call(oracle, dt, tcx):
    """The time-domain nest has no block structure: however the scheduler chunks the stream (input arriving
    in pieces, small output buffers), the reference's outputs are the oracle's one-call outputs, bit for bit."""
    code = getattr(oracle, dt)
    rng = np.random.default_rng(5)
    x = _rand_stream(oracle, code, 5000, rng)
    for (M, L), ntaps in zip([(1, 1), (2, 3), (3, 2), (4, 1)], (64, 101, 255, 17)):
        taps = _rand_taps(ntaps, tcx, rng)
        y, c, p = oracle.fir(code, tcx, taps, M, L, x)
        for in_chunk, out_chunk in ((0, 0), (700, 0), (0, 301), (333, 97)):
            yr, cr, pr, calls = oracle.ref_fir_stream(code, tcx, taps, M, L, x, in_chunk=in_chunk, out_chunk=out_chunk)
            assert (c, p) == (cr, pr), (M, L, in_chunk, out_chunk)
            assert _same_bits(y, yr), (M, L, in_chunk, out_chunk)
            if in_chunk or out_chunk:
                assert calls > 1


@needs_ref
def test_reference_setter_errors(oracle):
    x = np.zeros((8, 2), dtype=np.float32)
    with pytest.raises(oracle.ReferenceError_, match="taps cannot be empty"):         # :140
        oracle.ref_fir(oracle.CF32, False, [], 1, 1, x)
    with pytest.raises(oracle.ReferenceError_, match="decimation cannot be 0"):       # :153
        oracle.ref_fir(oracle.CF32, False, [1.0], 0, 1, x)
    with pytest.raises(oracle.ReferenceError_, match="interpolation cannot be 0"):    # :165
        oracle.ref_fir(oracle.CF32, False, [1.0], 1, 0, x)


@needs_ref
def test_reference_latent_stall_remainder_below_M(oracle):
    """SURVEY 8a5: a flushed remainder < M is never consumed (N = 0 forever, :278)."""
    x = np.arange(10, dtype=np.float32).reshape(-1, 1)
    yr, cr, pr, _ = oracle.ref_fir_stream(oracle.F32, False, [1.0, 1.0], 3, 1, x, frame_end=True)
    assert (cr, pr) == (9, 3)
    y, c, p = oracle.fir(oracle.F32, False, [1.0, 1.0], 3, 1, x, zero_tail=True)
    assert (c, p) == (9, 3) and _same_bits(y, yr)


@needs_ref
def test_multithreaded_reference_driver_equals_port_segments(oracle):
    rng = np.random.default_rng(8)
    taps = _rand_taps(31, True, rng)
    x = _rand_stream(oracle, oracle.CF32, 4 * 1000, rng)
    out, c, p = oracle.ref_fir(oracle.CF32, True, taps, 2, 3, x, threads=4)
    for t in range(4):
        y, ct, pt = oracle.fir(oracle.CF32, True, taps, 2, 3, x[t * 1000:(t + 1) * 1000])
        assert _same_bits(out[t, :pt], y)
    assert p == 4 * pt and c == 4 * ct


@needs_ref
def test_oracle_equals_reference_block_fuzz(oracle):
    """Property-based: random row of the type table, rates, tap count, window length and output capacity -- one work() of the
    reference's compiled block against the oracle, bit for bit, counts included (filter/FIRFilter.cpp:278-309)."""
    from hypothesis import HealthCheck, given, settings
    from hypothesis import strategies as st

    @settings(max_examples=120, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
    @given(row=st.integers(0, len(ROWS) - 1), M=st.integers(1, 9), L=st.integers(1, 9), ntaps=st.integers(1, 70),
           n=st.integers(0, 700), cap_frac=st.sampled_from([None, 1.0, 0.5, 0.1]), seed=st.integers(0, 2 ** 31))
    def check(row, M, L, ntaps, n, cap_frac, seed):
        dt, tcx = ROWS[row]
        code = getattr(oracle, dt)
        rng = np.random.default_rng(seed)
        x = _rand_stream(oracle, code, n, rng)
        taps = _rand_taps(ntaps, tcx, rng)
        cap = None if cap_frac is None else int(cap_frac * (n // M + 1) * L)
        y, c, p = oracle.fir(code, tcx, taps, M, L, x, out_capacity=cap)
        yr, cr, pr = oracle.ref_fir(code, tcx, taps, M, L, x, out_capacity=cap)
        assert (c, p) == (cr, pr), (dt, tcx, M, L, ntaps, n, cap)
        assert _same_bits(y, yr), (dt, tcx, M, L, ntaps, n, cap)

    check()


@needs_ref
def test_reference_chunked_streaming_fuzz(oracle):
    """Property-based: however the stream is chunked on the way in and out, with or without a frame-end flush, the reference
    block's output is the oracle's one-call output (zero_tail for the flush), bit for bit (:209-272,304-309)."""
    from hypothesis import HealthCheck, given, settings
    from hypothesis import strategies as st

    @settings(max_examples=80, deadline=None, derandomize=True, suppress_health_check=list(HealthCheck))
    @given(row=st.integers(0, len(ROWS) - 1), M=st.integers(1, 6), L=st.integers(1, 6), ntaps=st.integers(1, 60),
           n=st.integers(1, 900), in_chunk=st.sampled_from([0, 1, 17, 64, 333]), out_chunk=st.sampled_from([0, 5, 33, 200]),
           frame_end=st.booleans(), seed=st.integers(0, 2 ** 31))
    def check(row, M, L, ntaps, n, in_chunk, out_chunk, frame_end, seed):
        dt, tcx = ROWS[row]
        code = getattr(oracle, dt)
        rng = np.random.default_rng(seed)
        x = _rand_stream(oracle, code, n, rng)
        taps = _rand_taps(ntaps, tcx, rng)
        if out_chunk and out_chunk < L:
            out_chunk = L                      # an output buffer smaller than one block never makes progress (:283)
        if frame_end:
            # the whole burst is in the port when work() runs.  (A burst tail shorter than M + K - 1 that arrives in pieces
            # stalls the reference: the starved call on the first piece sets that reserve (:248-252), the piece carrying the
            # frame-end label does not reach it, and work() is never called again -- scheduler-dependent, not modelled.)
            in_chunk = 0
        y, c, p = oracle.fir(code, tcx, taps, M, L, x, zero_tail=frame_end)
        yr, cr, pr, _ = oracle.ref_fir_stream(code, tcx, taps, M, L, x, in_chunk=in_chunk, out_chunk=out_chunk, frame_end=frame_end)
        assert (c, p) == (cr, pr), (dt, tcx, M, L, ntaps, n, in_chunk, out_chunk, frame_end)
        assert _same_bits(y, yr), (dt, tcx, M, L, ntaps, n, in_chunk, out_chunk, frame_end)

    check()
