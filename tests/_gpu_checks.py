"""Checks shared by the GPU parity tests that compare every output of a launch with a float64 reference:
which kernels ran (torch.profiler), windowed error against the reference, and output that must stay untouched."""
import pytest
import torch

WIN = 4096
RMS_TOL, MAX_TOL = 1e-5, 5e-4          # float32 paths, of the channel's output RMS (north-star tolerance)


def _profiled(fn, key="fir_"):
    """Run fn() under torch.profiler (CUDA activities); returns (fn's result, names of the kernels that ran whose
    demangled name, spaces removed, contains `key`)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    # Late in a long pytest process the profiler has been seen to drop kernel records.  So the memory torch caches
    # is handed back first (the profiler's activity buffers need room), a few small kernels go before and after, and a session
    # that recorded none of the wanted kernels is run once more (every caller's fn() can be repeated: it writes the
    # same outputs).
    torch.cuda.empty_cache()
    for _ in range(2):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            warm = torch.zeros(1, device="cuda")
            for _ in range(4):
                warm.add_(1)
            torch.cuda.synchronize()
            r = fn()
            for _ in range(4):
                warm.add_(1)
            torch.cuda.synchronize()
        names = [e.name.replace(" ", "") for e in prof.events() if str(e.device_type).endswith("CUDA")]
        names = [n for n in names if key in n]
        if names:
            break
    return r, names


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
    """Every element of the tensor t still holds `value` (NaN: still NaN; complex: both parts)."""
    if t.numel() == 0:
        return
    if value != value:
        ok = torch.isnan(torch.view_as_real(t) if t.is_complex() else t).all()
    else:
        ok = (t == value).all()
    assert bool(ok), f"{what}: written where nothing may be"
