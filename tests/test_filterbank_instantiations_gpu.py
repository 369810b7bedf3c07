"""Every template instantiation of the four polyphase filter-bank kernels (pfb_chan_kernel<R>,
pfb_rchan_kernel<R, float / int16_t>, pfb_synth_kernel<K>, pfb_rsynth_kernel<K, float / int16_t>) against the float64
references, and the layouts the parity grids of test_channelizer_gpu.py, test_real_channelizer_gpu.py,
test_synthesizer_gpu.py and test_real_synthesizer_gpu.py do not reach: every decimation that divides M (branch chains
longer than a tile, synthesizer threads that emit one sample per tile), every bin-group class of the synthesizers,
stream indices where s + m0 wraps in uint64, and streams fed in pieces across 2^64.

Each kernel unrolls its register window by R or K with slots picked by compile-time indices, so every instantiation
has its own code: each one runs here, and the kernel that ran is read out of the profiler so that a dispatch to the
wrong table entry fails.  The case lists live in tests/_pfb_cases.py; tests/test_pfb_cases_cpu.py checks what they
cover."""
import re
import zlib

import numpy as np
import pytest

import _pfb_cases as pc
from _chan_oracle import channelize
from _gpu_checks import _profiled
from _rsynth_oracle import synthesize_real
from _synth_oracle import synthesize
from test_oracle_real_channelizer import real_channelize

pytestmark = pytest.mark.gpu

TOL = 1e-5                # of each channel's output RMS, or of each 64 D-sample block's (the four parity files' _check)
KERNEL_RE = {
    "chan": re.compile(r"pfb_chan_kernel<(?:\(int\))?(\d+)>"),
    "rchan": re.compile(r"pfb_rchan_kernel<(?:\(int\))?(\d+),(float|short|shortint|int16_t)>"),
    "synth": re.compile(r"pfb_synth_kernel<(?:\(int\))?(\d+)>"),
    "rsynth": re.compile(r"pfb_rsynth_kernel<(?:\(int\))?(\d+),(float|short|shortint|int16_t)>"),
}
TYPE_ARG = {"float32": "float", "int16": "int16", "complex_float32": None}


def _torch():
    import torch
    assert torch.cuda.is_available()
    return torch


def _params(cases):
    return [pytest.param(c, id=c.id) for c in cases]


def _seed(case, salt=0):
    return zlib.crc32(f"{case.id}/{salt}".encode())


def _assert_ran(case, names, dtype=None):
    """Exactly one instantiation of case.kernel ran, and it is the one its tap count selects."""
    rx = KERNEL_RE[case.kernel]
    found = set()
    for nm in names:
        m = rx.search(nm)
        if m:
            t = None if case.kernel in ("chan", "synth") else ("float" if m.group(2) == "float" else "int16")
            found.add((int(m.group(1)), t))
    want = (case.n, TYPE_ARG[dtype or case.dtype])
    assert found == {want}, f"{case.id}: expected the instantiation {want} to run, the profiler saw {sorted(found)} in {names}"


# ---- runners: one call on fresh buffers, under the profiler; output on the host

def _run_chan(case, x, s=None):
    torch = _torch()
    from pothoscomms_b200 import Channelizer
    ch = Channelizer("complex_float32", case.M, case.D)
    ch.set_taps(case.h)
    assert ch.info() == (case.M, case.D, case.ntaps, case.ntaps - 1 + case.D)
    d_in = torch.from_numpy(np.ascontiguousarray(x.astype(np.complex64)).view(np.float32).reshape(-1, 2)).cuda()
    out = torch.empty((case.M, case.F, 2), dtype=torch.float32, device="cuda")
    (c, p), names = _profiled(lambda: ch.run(d_in, out, case.s if s is None else s), key="pfb_")
    assert (c, p) == (case.F * case.D, case.F), case.id
    _assert_ran(case, names)
    o = out.cpu().numpy().astype(np.float64)
    return o[..., 0] + 1j * o[..., 1]


def _run_rchan(case, x, dtype):
    torch = _torch()
    from pothoscomms_b200 import RealChannelizer
    ch = RealChannelizer(dtype, case.M, case.D)
    ch.set_taps(case.h)
    assert ch.info() == (case.M, case.M // 2 + 1, case.D, case.ntaps, case.ntaps - 1 + case.D)
    d_in = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    out = torch.empty((case.M // 2 + 1, case.F, 2), dtype=torch.float32, device="cuda")
    (c, p), names = _profiled(lambda: ch.run(d_in, out, case.s), key="pfb_")
    assert (c, p) == (case.F * case.D, case.F), case.id
    _assert_ran(case, names, dtype)
    return out.cpu()


def _run_synth(case, X):
    torch = _torch()
    from pothoscomms_b200 import Synthesizer
    sy = Synthesizer("complex_float32", case.M, case.D)
    sy.set_taps(case.h)
    assert sy.info() == (case.M, case.D, case.ntaps, case.n)
    d_in = torch.from_numpy(np.ascontiguousarray(X.astype(np.complex64)).view(np.float32).reshape(case.M, -1, 2)).cuda()
    out = torch.empty((case.F * case.D, 2), dtype=torch.float32, device="cuda")
    (c, p), names = _profiled(lambda: sy.run(d_in, out, case.s, out_capacity=case.F * case.D), key="pfb_")
    assert (c, p) == (case.F, case.F * case.D), case.id
    _assert_ran(case, names)
    o = out.cpu().numpy().astype(np.float64)
    return o[:, 0] + 1j * o[:, 1]


def _run_rsynth(case, X, dtype, profile=True):
    torch = _torch()
    from pothoscomms_b200 import RealSynthesizer
    rs = RealSynthesizer(dtype, case.M, case.D)
    rs.set_taps(case.h)
    assert rs.info() == (case.M, case.M // 2 + 1, case.D, case.ntaps, case.n)
    d_in = torch.from_numpy(np.ascontiguousarray(X.astype(np.complex64)).view(np.float32).reshape(case.M // 2 + 1, -1, 2)).cuda()
    out = torch.empty(case.F * case.D, dtype=torch.float32 if dtype == "float32" else torch.int16, device="cuda")
    run = lambda: rs.run(d_in, out, case.s, out_capacity=case.F * case.D)   # noqa: E731
    if profile:
        (c, p), names = _profiled(run, key="pfb_")
        _assert_ran(case, names, dtype)
    else:
        c, p = run()
        torch.cuda.synchronize()
    assert (c, p) == (case.F, case.F * case.D), case.id
    return out.cpu().numpy().astype(np.float64)


# ---- inputs and reference comparisons

class _Case:
    """A _pfb_cases.Case with its random taps."""

    def __init__(self, case):
        self.__dict__.update(case._asdict())
        self.n, self.T, self.id = case.n, case.T, case.id
        self.h = np.random.default_rng(_seed(case, 1)).standard_normal(case.ntaps)


def _chan_input(case, dtype="complex_float32"):
    rng = np.random.default_rng(_seed(case, 2))
    n = case.ntaps - 1 + case.F * case.D + case.D // 3          # a partial frame's worth more: F frames exactly
    if dtype == "complex_float32":
        return (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    if dtype == "float32":
        return rng.standard_normal(n).astype(np.float32)
    x = rng.integers(-32768, 32768, size=n).astype(np.int16)
    x[::97] = -32768
    x[5::89] = 32767
    return x


def _synth_input(case):
    rows = case.M if case.kernel == "synth" else case.M // 2 + 1
    rng = np.random.default_rng(_seed(case, 3))
    n = case.n - 1 + case.F + 3
    return (rng.standard_normal((rows, n)) + 1j * rng.standard_normal((rows, n))).astype(np.complex64)


def _chan_rows(case):
    """The channels compared: all of them while the dense reference costs at most pc.REF_BUDGET multiply-adds, else the
    edge channels and a random set, every frame of each (a channelizer's per-frame and per-branch bugs show in every
    channel)."""
    top = case.M - 1 if case.kernel == "chan" else case.M // 2
    per_row = case.ntaps * case.F
    if (top + 1) * per_row <= pc.REF_BUDGET:
        return list(range(top + 1))
    edge = {0, 1, 2, case.M // 4, case.M // 2 - 1, case.M // 2, top - 1, top}
    rest = np.random.default_rng(_seed(case, 4)).permutation(top + 1)
    rows = set(edge)
    for c in rest:
        if len(rows) >= max(16, pc.REF_BUDGET // per_row):
            break
        rows.add(int(c))
    return sorted(c for c in rows if c <= top)


def _check_rows(y, ref, rows, what):
    err = np.sqrt(np.mean(np.abs(y - ref) ** 2, axis=1))
    rms = np.sqrt(np.mean(np.abs(ref) ** 2, axis=1))
    bad = np.nonzero(~(err <= TOL * rms))[0]
    assert bad.size == 0, f"{what}: channels {[rows[i] for i in bad[:8]]}: err/rms {(err[bad] / rms[bad])[:8]}"


def _synth_windows(case):
    """Output frames compared: all while the dense reference costs at most pc.REF_BUDGET multiply-adds, else the
    frames on both sides of every tile boundary and at both ends (test_real_synthesizer_gpu.py's windows)."""
    rows = case.M if case.kernel == "synth" else case.M // 2 + 1
    if rows * case.D * (case.n + 1) * case.F <= pc.REF_BUDGET:
        return [(0, case.F)]
    T, F = case.T, case.F
    w = [(0, 1)] + [(b - 1, b + 1) for b in range(T, F, T)] + [(F - 1, F)]
    return sorted({(max(0, a), min(F, b)) for a, b in w})


def _check_blocks(y, ref, D, what):
    """RMS error within TOL of the reference's RMS, per block of 64 D output samples."""
    assert y.shape == ref.shape
    blk = 64 * D
    for b0 in range(0, ref.size, blk):
        e, r = y[b0: b0 + blk], ref[b0: b0 + blk]
        err = np.sqrt(np.mean(np.abs(e - r) ** 2))
        rms = np.sqrt(np.mean(np.abs(r) ** 2))
        assert err <= TOL * rms, f"{what}: samples {b0}..: err/rms {err / rms:.3g}"


def _parity(case):
    """One call of the float kernel of `case`, the instantiation it ran, and its output against the float64 reference."""
    case = _Case(case)
    if case.kernel in ("chan", "rchan"):
        rows = _chan_rows(case)
        if case.kernel == "chan":
            x = _chan_input(case)
            y = _run_chan(case, x)
            ref = channelize(x, case.h, case.M, case.D, case.s, channels=rows)
        else:
            x = _chan_input(case, "float32")
            raw = _run_rchan(case, x, "float32")
            y = raw.numpy().astype(np.float64)
            y = y[..., 0] + 1j * y[..., 1]
            ref = real_channelize(x, case.h, case.M, case.D, case.s, channels=rows)
            # channels 0 and M/2 are real: imaginary parts exactly 0
            assert raw[0, :, 1].abs().max().item() == 0.0 and raw[case.M // 2, :, 1].abs().max().item() == 0.0
        assert y.shape[1] == ref.shape[1] == case.F
        _check_rows(y[rows], ref, rows, case.id)
        return
    X = _synth_input(case)
    y = _run_synth(case, X) if case.kernel == "synth" else _run_rsynth(case, X, "float32")
    ref_fn = synthesize if case.kernel == "synth" else synthesize_real
    K, D = case.n, case.D
    for t0, t1 in _synth_windows(case):
        ref = ref_fn(X[:, t0: t0 + K - 1 + t1 - t0], case.h, case.M, D, case.s + t0 * D)
        _check_blocks(y[t0 * D: t1 * D], ref, D, f"{case.id} frames {t0}..{t1 - 1}")


def _int16_twin(case):
    """The int16 instantiation against the float32 one: RealChannelizer input of the same values bit for bit,
    RealSynthesizer output equal to clip(rint(float32 output)) with samples past both rails."""
    torch = _torch()
    case = _Case(case)
    if case.kernel == "rchan":
        xi = _chan_input(case, "int16")
        yi = _run_rchan(case, xi, "int16")
        yf = _run_rchan(case, xi.astype(np.float32), "float32")
        assert torch.equal(yi, yf), f"{case.id}: int16 input must give the float32 output of the same values bit for bit"
        return
    X = _synth_input(case)
    y32 = _run_rsynth(case, X, "float32", profile=False)
    Xs = (X * (60000.0 / np.abs(y32).max())).astype(np.complex64)    # some samples beyond both rails
    y32 = _run_rsynth(case, Xs, "float32", profile=False)
    y16 = _run_rsynth(case, Xs, "int16")
    want = np.clip(np.rint(y32), -32768, 32767)                      # np.rint rounds ties to even, as __float2int_rn
    assert (want == 32767).any() and (want == -32768).any()
    bad = np.nonzero(y16 != want)[0]
    assert bad.size == 0, f"{case.id}: {bad.size} samples differ from clip(rint(float32)), first at {bad[:8]}"


# ---- 1. every instantiation

@pytest.mark.parametrize("case", _params(pc.instantiation_cases("chan")))
def test_channelizer_instantiation(case):
    _parity(case)


@pytest.mark.parametrize("case", _params(pc.instantiation_cases("rchan")))
def test_real_channelizer_instantiation(case):
    _parity(case) if case.dtype == "float32" else _int16_twin(case)


@pytest.mark.parametrize("case", _params(pc.instantiation_cases("synth")))
def test_synthesizer_instantiation(case):
    _parity(case)


@pytest.mark.parametrize("case", _params(pc.instantiation_cases("rsynth")))
def test_real_synthesizer_instantiation(case):
    _parity(case) if case.dtype == "float32" else _int16_twin(case)


# ---- 2. every decimation that divides M, and frame counts around one tile

@pytest.mark.parametrize("case", _params([c for k in pc.KERNELS for c in pc.decimation_cases(k)]))
def test_every_decimation(case):
    _parity(case)


# ---- 3. the synthesizers' bin-group classes

@pytest.mark.parametrize("case", _params([c for k in ("synth", "rsynth") for c in pc.bin_class_cases(k)]))
def test_bin_group_classes(case):
    _parity(case)


# ---- 4. stream indices near 2^64, and streams fed in pieces across it

@pytest.mark.parametrize("case", _params([c for k in pc.KERNELS for c in pc.wrap_cases(k)]))
def test_stream_index_wraps(case):
    _parity(case)


@pytest.mark.parametrize("kernel,dtype", [(k, d) for k in pc.KERNELS for d in pc.DTYPES[k]])
def test_streaming_pieces_across_2_64(kernel, dtype):
    torch = _torch()
    import pothoscomms_b200 as pb
    case = _Case(pc.streaming_case(kernel)._replace(dtype=dtype))
    M, D, rng = case.M, case.D, np.random.default_rng(5)
    if kernel in ("chan", "rchan"):
        assert M // D > case.T
        F = 300
        n = case.ntaps - 1 + F * D + 1
        s0 = 2**64 - F * D // 2                        # the absolute index crosses 2^64 half-way
        if kernel == "chan":
            x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
            h = pb.Channelizer("complex_float32", M, D)
            dev = lambda v: torch.from_numpy(np.ascontiguousarray(v).view(np.float32).reshape(-1, 2)).cuda()  # noqa: E731
            rows = M
        else:
            x = rng.integers(-32768, 32768, size=n).astype(np.int16) if dtype == "int16" else \
                rng.standard_normal(n).astype(np.float32)
            h = pb.RealChannelizer(dtype, M, D)
            dev = lambda v: torch.from_numpy(np.ascontiguousarray(v)).cuda()   # noqa: E731
            rows = M // 2 + 1
        h.set_taps(case.h)
        whole = torch.empty((rows, F, 2), dtype=torch.float32, device="cuda")
        assert h.run(dev(x), whole, s0) == (F * D, F)
        pieces, carry, pos, base = [], x[: case.ntaps - 1], case.ntaps - 1, s0   # history, then ragged pieces
        while pos < x.size:
            step = int(rng.integers(1, 3 * case.T * D + 7))
            buf = np.concatenate([carry, x[pos: pos + step]])
            pos += step
            out = torch.zeros((rows, buf.size // D + 1, 2), dtype=torch.float32, device="cuda")
            c, p = h.run(dev(buf), out, base)
            pieces.append(out[:, :p])
            carry = buf[c:]
            base += c
        got = torch.cat(pieces, dim=1)
    else:
        K = case.n
        F = 3 * case.T + 11
        s0 = 2**64 - F * D // 2
        rows = M if kernel == "synth" else M // 2 + 1
        X = (rng.standard_normal((rows, K - 1 + F)) + 1j * rng.standard_normal((rows, K - 1 + F))).astype(np.complex64)
        dev = lambda v: torch.from_numpy(np.ascontiguousarray(v).view(np.float32).reshape(rows, -1, 2)).cuda()  # noqa: E731
        if kernel == "synth":
            h = pb.Synthesizer("complex_float32", M, D)
            mk = lambda m: torch.empty((m, 2), dtype=torch.float32, device="cuda")   # noqa: E731
        else:
            h = pb.RealSynthesizer(dtype, M, D)
            mk = lambda m: torch.empty(m, dtype=torch.float32 if dtype == "float32" else torch.int16, device="cuda")  # noqa: E731
        h.set_taps(case.h * (300.0 if dtype == "int16" else 1.0))
        whole = mk(F * D)
        assert h.run(dev(X), whole, s0) == (F, F * D)
        pieces, pos, base = [], 0, s0                 # pos: first frame of the next piece's K-1 history
        while pos + K - 1 < X.shape[1]:
            step = int(rng.integers(1, 3 * case.T // 2 + 3))
            buf = X[:, pos: pos + K - 1 + step]
            out = mk(step * D)
            c, p = h.run(dev(buf), out, base)
            assert p == c * D and c == min(step, buf.shape[1] - (K - 1))
            pieces.append(out[:p])
            pos += c
            base += p
        got = torch.cat(pieces)
    torch.cuda.synchronize()
    assert base > 2**64 > s0, "the stream must cross 2^64"
    assert got.shape == whole.shape
    assert torch.equal(got, whole), f"{case.id}: a stream fed in pieces must give the one-call output bit for bit"
