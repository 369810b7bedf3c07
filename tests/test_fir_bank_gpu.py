"""GPU parity of the FIR filter bank (b200c_fir_bank_run) on every channel, at the shapes its batched kernels run.

A complex float32 bank at L = M = 1 runs in ONE launch over (channel, block) with a table of every channel's tap
spectrum gathered on the device: fir_os64p_kernel (persistent, CTA-tasks = (channel, part)) once the bank has at
least 4 * 4 * SMs transform blocks, fir_os64_kernel<4> below that, the bank form of fir_os32_kernel (one warp per
task, tasks crossing channels) for tap counts up to 448.  Every other type and rate runs the channels' own kernels
one after another.  Each case here:
  * gives every channel its own random taps and its own input, so a neighbour's spectrum or samples change the result;
  * fills the output with NaN (or a sentinel) first, so an output never written fails, and so does one written
    past the produced count or into the gap between channels;
  * compares every channel with a float64 reference (tests/_bank_ref.py at L = M = 1, oracle.fir otherwise) in
    windows of 4096 outputs: RMS error <= 1e-5 and max error <= 5e-4 of the channel's output RMS for float32,
    1e-13 / 5e-12 for complex float64, bit for bit for the integer types;
  * records with torch.profiler which kernels ran and asserts the one the bank's dispatch rule names.
"""
import ctypes
import re

import numpy as np
import pytest
import torch

from _bank_ref import fir_count, fir_ref

pytestmark = pytest.mark.gpu

WIN = 4096
RMS_TOL, MAX_TOL = 1e-5, 5e-4          # float32 paths, of the channel's output RMS (north-star tolerance)
CF64_RMS_TOL, CF64_MAX_TOL = 1e-13, 5e-12
B200_SMS = 148
CHUNK = 16                             # channels per reference chunk
SENTINEL = complex(1234.5, -678.25)
NAN = complex(float("nan"), float("nan"))


# ----------------------------------------------------------------------------------------------- dispatch rule ---
def bank_path(nchan, n_out, ntaps, sm_count=B200_SMS):
    """Python copy of fir_os_launch's choice (fir_os.cu) for a complex float32 bank at L = M = 1:
    (kernel, parts) with parts the persistent kernel's split of a channel's blocks, else None."""
    N = 1024 if ntaps <= 448 else 4096                       # pick_length: kFirOs1kMaxTaps
    hop = N - (ntaps - 1)
    blocks = -(-n_out // hop)
    if N == 1024:
        return ("os32_single" if nchan == 1 else "os32_bank"), None
    if nchan * blocks < 4 * 4 * sm_count:
        return "os64", None
    if nchan == 1:
        return "os64p", sm_count
    best, parts = -1.0, 1
    for q in range(1, min(max(1, blocks // 16), 32) + 1):
        T = nchan * q
        rounds = -(-T // sm_count)
        util = T / (rounds * sm_count) - 1.5e-3 * (q - 1)
        if util > best:
            best, parts = util, q
    return "os64p", parts


# demangled kernel names, spaces removed
PATH_KERNEL = {
    "os64p": r"fir_os64p_kernel\b",
    "os64": r"fir_os64_kernel<4>",
    "os32_bank": r"fir_os32_kernel<1,12[,>]",
    "os32_single": r"fir_os32_kernel<12,1[,>]",
}


def _path_id(nchan, n_out, ntaps):
    kern, parts = bank_path(nchan, n_out, ntaps)
    return kern + (f"-parts{parts}" if parts is not None else "")


def _profiled(fn):
    """Run fn() under torch.profiler (CUDA activities); returns (fn's result, names of the fir_* kernels that ran)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    names = [e.name.replace(" ", "") for e in prof.events() if str(e.device_type).endswith("CUDA")]
    return r, [n for n in names if "fir_" in n]


def _assert_kernels(names, pattern, what):
    assert names, f"{what}: the profiler recorded no fir kernel"
    bad = [n for n in names if not re.search(pattern, n)]
    assert not bad, f"{what}: expected only {pattern}, ran {sorted(set(names))}"


def _assert_path(names, nchan, n_out, ntaps, what):
    kern, _ = bank_path(nchan, n_out, ntaps, torch.cuda.get_device_properties(0).multi_processor_count)
    _assert_kernels(names, PATH_KERNEL[kern], what)


# ------------------------------------------------------------------------------------------------- comparison ---
def _check(got, ref, what, chans=None, rms_tol=RMS_TOL, max_tol=MAX_TOL):
    """got, ref: [nch, n] tensors on one device; per channel, per window of WIN outputs, relative to the channel's
    output RMS.  A NaN anywhere fails.  chans: the channel numbers of the rows, for the report."""
    assert got.shape == ref.shape, (what, tuple(got.shape), tuple(ref.shape))
    nch, n = ref.shape
    if n == 0:
        return
    ref = ref.to(torch.complex128 if ref.is_complex() else torch.float64)
    d2 = (got.to(ref.dtype) - ref).abs() ** 2
    rms = (ref.abs() ** 2).mean(dim=1).sqrt()
    nw = -(-n // WIN)
    d2 = torch.nn.functional.pad(d2, (0, nw * WIN - n)).view(nch, nw, WIN)
    cnt = torch.full((nw,), float(WIN), dtype=torch.float64, device=d2.device)
    cnt[-1] = n - (nw - 1) * WIN
    werr = (d2.sum(-1) / cnt).sqrt() / rms[:, None]
    wmax = d2.amax(-1).sqrt() / rms[:, None]
    bad = ~(werr <= rms_tol) | ~(wmax <= max_tol)
    if bool(bad.any()):
        first = bad.nonzero()[:4].tolist()
        rows = [f"(channel {chans[c] if chans is not None else c}, window {w}): rms {float(werr[c, w]):.2e}, "
                f"max {float(wmax[c, w]):.2e}" for c, w in first]
        pytest.fail(f"{what}: {int(bad.sum())} of {nch * nw} (channel, window) pairs out of tolerance "
                    f"(rms {rms_tol}, max {max_tol}); first: " + "; ".join(rows))


def _untouched(t, value, what):
    """Every element of the complex tensor t still holds `value` (NaN: still NaN)."""
    if t.numel() == 0:
        return
    if value != value:
        ok = torch.isnan(torch.view_as_real(t)).all()      # both parts still NaN
    else:
        ok = (t == value).all()
    assert bool(ok), f"{what}: written where nothing may be"


def _check_bank_out(x, taps, out, produced, zero_tail, what, chans=None):
    """x: [nch, n_in] complex64 (device), taps: [nch, K] (device), out: [nch, >= produced] complex64 NaN-filled
    before the run.  Compares a chunk of channels at a time with fir_ref."""
    nch = x.shape[0]
    for c0 in range(0, nch, CHUNK):
        c1 = min(nch, c0 + CHUNK)
        ref = fir_ref(x[c0:c1], taps[c0:c1], zero_tail=zero_tail, n_out=produced)
        _check(out[c0:c1, :produced], ref, what, chans=list(range(c0, c1)) if chans is None else chans[c0:c1])
        del ref


def _rand_taps(rng, nch, ntaps, complex_taps):
    h = rng.standard_normal((nch, ntaps)) / np.sqrt(ntaps)
    if complex_taps:
        h = h + 1j * rng.standard_normal((nch, ntaps)) / np.sqrt(ntaps)
    return h


def _randn_cf32(shape, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.view_as_complex(torch.randn((*shape, 2), generator=g, device="cuda"))


def _make_bank(taps, complex_taps, decim=1, interp=1, code=None):
    from pothoscomms_b200 import FirFilterBank
    bank = FirFilterBank("complex_float32" if code is None else code, "COMPLEX" if complex_taps else "REAL", len(taps))
    if (decim, interp) != (1, 1):
        bank.set_rates(decim, interp)
    for c, h in enumerate(taps):
        bank.set_taps(c, h)
    return bank


def _raw_run(bank, d_in, in_stride, in_elems, d_out, out_stride, capacity, zero_tail, stream=None):
    """b200c_fir_bank_run through ctypes with explicit strides; returns (rc, consumed, produced)."""
    from pothoscomms_b200 import _abi
    c, p = ctypes.c_size_t(), ctypes.c_size_t()
    s = ctypes.c_void_p((stream or torch.cuda.current_stream()).cuda_stream)
    rc = _abi.lib().b200c_fir_bank_run(bank._h, ctypes.c_void_p(d_in), in_stride, in_elems, ctypes.c_void_p(d_out),
                                       out_stride, capacity, int(zero_tail), ctypes.byref(c), ctypes.byref(p), s)
    return rc, c.value, p.value


# ------------------------------------------------------------------------------------- batched kernels, shapes ---
# (name, channels, new samples, taps, complex taps, expected path on 148 SMs)
BATCHED = [
    ("c5", 1024, 1 << 20, 1024, True, ("os64p", 1)),
    ("one_gpu_of_8", 128, 1 << 20, 1024, True, ("os64p", 8)),
    ("ragged", 150, (1 << 19) + 777, 1024, False, ("os64p", 10)),
    ("longest_taps", 64, 1 << 20, 2049, True, ("os64p", 16)),
    ("few_blocks", 7, 300000, 1024, True, ("os64", None)),
    ("short_taps", 256, 1 << 18, 255, True, ("os32_bank", None)),
]


@pytest.mark.parametrize("name,nch,n_new,ntaps,complex_taps,path", BATCHED,
                         ids=[f"{c[0]}-{c[1]}x{c[2]}-K{c[3]}-{_path_id(c[1], c[2], c[3])}" for c in BATCHED])
def test_batched_bank_every_channel(cuda_device, name, nch, n_new, ntaps, complex_taps, path):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms == B200_SMS:
        assert bank_path(nch, n_new, ntaps, sms) == path, "the Python copy of the dispatch rule drifted"
    rng = np.random.default_rng(nch * 7 + ntaps)
    h = _rand_taps(rng, nch, ntaps, complex_taps)
    bank = _make_bank(h, complex_taps)
    assert bank.info() == (nch, ntaps, ntaps)
    taps = torch.from_numpy(h).cuda()
    in_elems = ntaps - 1 + n_new
    x = _randn_cf32((nch, in_elems), seed=nch * 1000 + ntaps)
    cap = in_elems + 5
    out = torch.empty((nch, cap), dtype=torch.complex64, device="cuda")
    for zero_tail in (False, True):
        what = f"{name} zt={zero_tail}"
        out.fill_(NAN)
        (cons, prod), names = _profiled(lambda: bank.run(torch.view_as_real(x), torch.view_as_real(out), zero_tail=zero_tail))
        assert (cons, prod) == (fir_count(in_elems, ntaps, zero_tail),) * 2, what
        _assert_path(names, nch, prod, ntaps, what)
        _check_bank_out(x, taps, out, prod, zero_tail, what)
        _untouched(out[:, prod:], NAN, what + " past the produced count")
    del x, out
    torch.cuda.empty_cache()


@pytest.mark.parametrize("ntaps", [255, 1024])
def test_one_channel_bank_is_bit_identical_to_fir_filter(cuda_device, ntaps):
    """A bank of one channel runs the single-stream kernels on the gathered spectrum table: the same bits as
    FirFilter.run on the same input."""
    from pothoscomms_b200 import FirFilter
    rng = np.random.default_rng(ntaps)
    h = _rand_taps(rng, 1, ntaps, True)
    bank = _make_bank(h, True)
    f = FirFilter("complex_float32", "COMPLEX")
    f.set_taps(h[0])
    in_elems = ntaps - 1 + (1 << 20)
    x = _randn_cf32((1, in_elems), seed=ntaps)
    out = torch.empty((1, in_elems + 5), dtype=torch.complex64, device="cuda")
    for zero_tail in (False, True):
        what = f"one channel K={ntaps} zt={zero_tail}"
        out.fill_(NAN)
        (_, prod), names = _profiled(lambda: bank.run(torch.view_as_real(x), torch.view_as_real(out), zero_tail=zero_tail))
        (y, _, prod_f), names_f = _profiled(lambda: f.run(torch.view_as_real(x[0]), zero_tail=zero_tail))
        assert prod == prod_f == fir_count(in_elems, ntaps, zero_tail), what
        _assert_path(names, 1, prod, ntaps, what)
        assert sorted(set(names)) == sorted(set(names_f)), (names, names_f)
        assert torch.equal(torch.view_as_real(out[0, :prod]), y), f"{what}: bank and FirFilter differ"
        _check_bank_out(x, torch.from_numpy(h).cuda(), out, prod, zero_tail, what)
        _untouched(out[:, prod:], NAN, what + " past the produced count")


# --------------------------------------------------------------------------------------------- channel layout ---
def _odd(n):
    return n | 1


@pytest.mark.parametrize("ntaps", [1024, 255])
def test_bank_layout_strides_streams_and_short_input(cuda_device, ntaps):
    """Odd channel strides in and out (every other channel base off 16-byte alignment, channel 0 too), NaN in every
    channel's input padding, a sentinel in the output gap between channels that must survive, a non-default stream,
    and runs below input_require that return (0, 0) and write nothing."""
    nch, n_new = 40, 200003
    rng = np.random.default_rng(ntaps + 1)
    h = _rand_taps(rng, nch, ntaps, True)
    bank = _make_bank(h, True)
    taps = torch.from_numpy(h).cuda()
    in_elems = ntaps - 1 + n_new
    in_stride = _odd(in_elems + 6)
    cap = in_elems + 3                           # room for the zero-tail run's in_elems outputs
    out_stride = _odd(cap + 10)
    xbuf = torch.full((1 + nch * in_stride + 64,), NAN, dtype=torch.complex64, device="cuda")
    xv = xbuf[1:1 + nch * in_stride].view(nch, in_stride)
    x = _randn_cf32((nch, in_elems), seed=ntaps + 2)
    xv[:, :in_elems] = x
    obuf = torch.empty((nch * out_stride + 64,), dtype=torch.complex64, device="cuda")
    ov = obuf[:nch * out_stride].view(nch, out_stride)
    d_in = xbuf.data_ptr() + 8                   # one element in: channel 0 starts off 16-byte alignment as well
    side = torch.cuda.Stream()
    for zero_tail in (False, True):
        for stream in (None, side):
            what = f"layout K={ntaps} zt={zero_tail} stream={'side' if stream else 'default'}"
            obuf.fill_(SENTINEL)
            if stream is not None:
                stream.wait_stream(torch.cuda.current_stream())
            (rc, cons, prod), names = _profiled(
                lambda: _raw_run(bank, d_in, in_stride, in_elems, obuf.data_ptr(), out_stride, cap, zero_tail, stream))
            if stream is not None:
                torch.cuda.current_stream().wait_stream(stream)
            assert rc == 0, what
            assert (cons, prod) == (fir_count(in_elems, ntaps, zero_tail),) * 2, what
            _assert_path(names, nch, prod, ntaps, what)
            _check_bank_out(x, taps, ov, prod, zero_tail, what)
            _untouched(ov[:, prod:], SENTINEL, what + " gap between channels")
            _untouched(obuf[nch * out_stride:], SENTINEL, what + " past the last channel")
    # below input_require (= K at L = M = 1): nothing to do, nothing written, no kernel
    obuf.fill_(SENTINEL)
    for n_in, zero_tail in ((ntaps - 1, False), (0, True)):
        (rc, cons, prod), names = _profiled(
            lambda: _raw_run(bank, d_in, in_stride, n_in, obuf.data_ptr(), out_stride, cap, zero_tail))
        assert (rc, cons, prod) == (0, 0, 0), (n_in, zero_tail)
        assert not names, names
    _untouched(obuf, SENTINEL, "runs below input_require")


@pytest.mark.parametrize("ntaps", [1024, 255])
def test_bank_channel_offsets_past_2_31_elements(cuda_device, ntaps):
    """1040 channels 2^21 + 1 elements apart: the last 16 channels start past element 2^31 (17 GiB each way)."""
    nch, stride, n_new = 1040, (1 << 21) + 1, 20000
    need = 2 * nch * stride * 8
    free, _ = torch.cuda.mem_get_info()
    if free < need + (5 << 30):
        pytest.skip(f"needs ~{(need >> 30) + 5} GiB of free device memory, {free >> 30} GiB free (shared device)")
    rng = np.random.default_rng(ntaps + 3)
    h = _rand_taps(rng, nch, ntaps, True)
    bank = _make_bank(h, True)
    taps = torch.from_numpy(h).cuda()
    in_elems = ntaps - 1 + n_new
    past = [c for c in range(nch) if c * stride >= 1 << 31]
    assert past == list(range(1024, nch))
    chans = sorted({0, 1, 127, 128, 255, 256, nch // 2, 1023} | set(past))
    xbuf = obuf = None
    try:
        xbuf = torch.full((nch * stride,), NAN, dtype=torch.complex64, device="cuda")
        xv = xbuf.view(nch, stride)
        x = _randn_cf32((nch, in_elems), seed=ntaps + 4)
        xv[:, :in_elems] = x
        obuf = torch.empty((nch * stride,), dtype=torch.complex64, device="cuda")
        ov = obuf.view(nch, stride)
        sel = torch.tensor(chans, device="cuda")
        for zero_tail in (False, True):
            what = f"offsets K={ntaps} zt={zero_tail}"
            obuf.fill_(SENTINEL)
            (rc, cons, prod), names = _profiled(
                lambda: _raw_run(bank, xbuf.data_ptr(), stride, in_elems, obuf.data_ptr(), stride, stride, zero_tail))
            assert rc == 0, what
            assert (cons, prod) == (fir_count(in_elems, ntaps, zero_tail),) * 2, what
            _assert_path(names, nch, prod, ntaps, what)
            got = ov[sel]
            _check_bank_out(x[sel], taps[sel], got, prod, zero_tail, what, chans=chans)
            _untouched(got[:, prod:], SENTINEL, what + " gap between channels")
    finally:
        del xbuf, obuf
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------ per-channel path ---
# (type, taps, ntaps, decim, interp, kernels the channel's own FirFilter may pick)
PER_CHANNEL = [
    ("CF32", "REAL", 255, 2, 3, ("fir_os32x_kernel",)),
    ("CF32", "COMPLEX", 100, 2, 1, ("fir_os32g_kernel",)),
    ("CF32", "COMPLEX", 255, 1, 4, ("fir_osp_kernel", "fir_ospg_kernel")),
    ("F32", "REAL", 255, 1, 1, ("fir_os32r_kernel",)),
    ("CI16", "COMPLEX", 128, 1, 1, ("fir_umma32t_kernel",)),
    ("I16", "REAL", 100, 3, 2, ("fir_ummap_kernel",)),
    ("CF64", "COMPLEX", 37, 1, 1, ("fir_tile_kernel",)),
]


def _rand_raw(oracle, code, shape, rng):
    nc = 2 if code & 1 else 1
    sc = oracle.scalar_np(code)
    if np.issubdtype(sc, np.integer):
        lim = np.iinfo(sc).max // 2
        return rng.integers(-lim - 1, lim + 1, size=(*shape, nc)).astype(sc)
    return rng.standard_normal((*shape, nc)).astype(sc)


@pytest.mark.parametrize("dt,taps_type,ntaps,decim,interp,kernels", PER_CHANNEL,
                         ids=[f"{c[0]}-{c[1]}-K{c[2]}-M{c[3]}-L{c[4]}" for c in PER_CHANNEL])
def test_per_channel_bank_matches_oracle(oracle, cuda_device, dt, taps_type, ntaps, decim, interp, kernels):
    """Types and rates the bank runs channel by channel, 5 channels at odd strides with padding that must not be
    read and a gap that must not be written, zero tail off and on, every channel against oracle.fir."""
    from pothoscomms_b200 import FirFilter
    code = getattr(oracle, dt)
    cx = taps_type == "COMPLEX"
    nc = 2 if code & 1 else 1
    is_int = np.issubdtype(oracle.scalar_np(code), np.integer)
    nch, n_new = 5, 30011
    rng = np.random.default_rng(ntaps * 13 + code * 3 + decim * 5 + interp)
    h = _rand_taps(rng, nch, ntaps, cx) * (0.3 if is_int else 1.0)
    f = FirFilter(code, taps_type)
    f.set_rates(decim, interp)
    f.set_taps(h[0])
    assert f.kernel in kernels, f.kernel
    # rates before taps: the channels' L = M = 1 tap spectra are never built
    bank = _make_bank(list(h), cx, decim, interp, code=code)
    _, K, req = bank.info()
    assert (K, req) == (f.K, f.input_require)
    in_elems = K - 1 + n_new
    in_stride = _odd(in_elems + 4)
    cap = ((in_elems + K - 1) // decim + 1) * interp
    out_stride = _odd(cap + 6)
    x = _rand_raw(oracle, code, (nch, in_elems), rng)
    tdt = x.dtype
    pad_in = 23130 if is_int else float("nan")
    sent = 12345 if is_int else 1234.5
    xbuf = torch.full((nch * in_stride + 8, nc), pad_in, dtype=torch.from_numpy(x[:0]).dtype, device="cuda")
    xbuf[:nch * in_stride].view(nch, in_stride, nc)[:, :in_elems] = torch.from_numpy(x).cuda()
    obuf = torch.empty((nch * out_stride + 8, nc), dtype=xbuf.dtype, device="cuda")
    ov = obuf[:nch * out_stride].view(nch, out_stride, nc)
    for zero_tail in (False, True):
        what = f"{dt}/{taps_type} K={ntaps} M={decim} L={interp} zt={zero_tail}"
        obuf.fill_(sent)
        (rc, cons, prod), names = _profiled(
            lambda: _raw_run(bank, xbuf.data_ptr(), in_stride, in_elems, obuf.data_ptr(), out_stride, cap, zero_tail))
        assert rc == 0, f"{what}: rc {rc}: {_last_error()}"
        _assert_kernels(names, re.escape(f.kernel) + r"(?![A-Za-z0-9_])", what)
        got = ov[:, :prod].cpu().numpy()
        for c in range(nch):
            y_ref, c_ref, p_ref = oracle.fir(code, cx, h[c], decim, interp, x[c], out_capacity=cap, zero_tail=zero_tail)
            assert (cons, prod) == (c_ref, p_ref), what
            if is_int:
                assert np.array_equal(got[c], y_ref), f"{what}: channel {c} must be bit-exact"
            else:
                g, r = torch.from_numpy(got[c][None].astype(np.float64)), torch.from_numpy(y_ref[None].astype(np.float64))
                if nc == 2:
                    g, r = torch.view_as_complex(g), torch.view_as_complex(r)
                else:
                    g, r = g[..., 0], r[..., 0]
                tol = (CF64_RMS_TOL, CF64_MAX_TOL) if tdt == np.float64 else (RMS_TOL, MAX_TOL)
                _check(g, r, what, chans=[c], rms_tol=tol[0], max_tol=tol[1])
        assert bool((ov[:, prod:] == sent).all()), f"{what}: written in the gap between channels"
        assert bool((obuf[nch * out_stride:] == sent).all()), f"{what}: written past the last channel"


def _last_error():
    from pothoscomms_b200 import _abi
    return _abi.last_error()


# ------------------------------------------------------------------------------------------- state changes ---
def test_bank_follows_tap_rate_and_length_changes(oracle, cuda_device):
    """The gathered spectrum table follows every setter: one channel's new taps, 64 -> 1024 -> 64 taps (1024- and
    4096-point rows, the table grows), rates (1, 1) -> (2, 3) -> (1, 1); a bank whose channels disagree on the tap
    count is refused and writes nothing."""
    from pothoscomms_b200 import InvalidArgumentError
    nch, n_new = 6, 50000
    rng = np.random.default_rng(77)
    x = _randn_cf32((nch, 2048 + n_new), seed=77)
    bank = _make_bank(_rand_taps(rng, nch, 64, True), True)
    taps = None

    def run(h, decim=1, interp=1, path=None):
        K = -(-h.shape[1] // interp)
        xi = x[:, :K - 1 + n_new].contiguous()
        cap = ((K - 1 + n_new) // decim + 1) * interp
        out = torch.full((nch, cap + 3), NAN, dtype=torch.complex64, device="cuda")
        what = f"K={h.shape[1]} M={decim} L={interp}"
        (cons, prod), names = _profiled(lambda: bank.run(torch.view_as_real(xi), torch.view_as_real(out)))
        if (decim, interp) == (1, 1):
            assert (cons, prod) == (n_new, n_new), what
            _assert_path(names, nch, prod, h.shape[1], what)
            _check_bank_out(xi, torch.from_numpy(h).cuda(), out, prod, False, what)
        else:
            _assert_kernels(names, path, what)
            xr = torch.view_as_real(xi).cpu().numpy()
            got = out[:, :prod].cpu()
            for c in range(nch):
                y_ref, c_ref, p_ref = oracle.fir(oracle.CF32, True, h[c], decim, interp, xr[c], out_capacity=cap + 3)
                assert (cons, prod) == (c_ref, p_ref), what
                _check(got[c:c + 1], torch.view_as_complex(torch.from_numpy(y_ref.astype(np.float64)))[None], what, chans=[c])
        _untouched(out[:, prod:], NAN, what + " past the produced count")

    for ntaps in (64, 1024, 64):
        taps = _rand_taps(rng, nch, ntaps, True)
        for c in range(nch):
            bank.set_taps(c, taps[c])
        run(taps)
        taps[nch // 2] = _rand_taps(rng, 1, ntaps, True)[0]      # one channel's taps change: the next run uses them
        bank.set_taps(nch // 2, taps[nch // 2])
        run(taps)
    bank.set_rates(2, 3)
    run(taps, 2, 3, r"fir_os32x_kernel\b")
    bank.set_rates(1, 1)
    run(taps)
    bank.set_taps(2, taps[2][:63])
    out = torch.full((nch, n_new + 3), NAN, dtype=torch.complex64, device="cuda")
    xi = x[:, :63 + n_new].contiguous()
    with pytest.raises(InvalidArgumentError):
        bank.run(torch.view_as_real(xi), torch.view_as_real(out))
    torch.cuda.synchronize()
    _untouched(out, NAN, "a refused run")
    bank.set_taps(2, taps[2])
    run(taps)
