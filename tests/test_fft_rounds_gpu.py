"""Every transform of the FFT's persistent kernels at batches that take several grid-stride rounds.

fft_staged_kernel runs grid = min(ngroups, 8 SMs) CTAs over groups of tpc transforms; fft4096_kernel runs
grid = min(batch, 12 SMs) CTAs over transforms.  In the global-memory form of the staged kernel a CTA's scratch slice
(indexed by blockIdx.x) is reused on every round.  Each case sizes the batch from a Python copy of that rule with the
device's SM count, asserts the rounds it needs and a ragged last one, fills the output with NaN (int16: a sentinel) and
compares every transform (sampled ones where the int16 oracle's generic butterfly is O(n p)): int16 bit for bit with
oracle.fft, float against a complex128 torch.fft at 1e-5 (complex float32) or 1e-13 (complex float64) of that
transform's RMS.  torch.profiler names the kernel that ran.
"""
import re

import numpy as np
import pytest
import torch

from _gpu_checks import _profiled

pytestmark = pytest.mark.gpu

SENT_I16 = 12345
TOL = {"CF32": 1e-5, "CF64": 1e-13}
TRAITS = {"CF32": r"FloatTraits<float>", "CF64": r"FloatTraits<double>", "CI16": r"Q15Traits"}
TORCH_DT = {"CF32": torch.float32, "CF64": torch.float64, "CI16": torch.int16}


@pytest.fixture(autouse=True)
def _free_memory():
    yield
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _cdiv(a, b):
    return -(-a // b)


def staged_plan(n, dt):
    """fft_plan_create + fft_launch for the staged kernel: (tpc, shared-memory form?, grid per ngroups)."""
    esz = {"CF32": 8, "CF64": 16, "CI16": 4}[dt]
    generic = any(p > 5 for p in _factors(n))
    tpc = max(1, 2048 // n)
    smem = tpc * n * esz * (2 if generic else 1) <= 200 * 1024
    return (tpc if smem else 1), smem, generic


def _factors(n):
    out, p = [], 2
    while n > 1:
        while n % p == 0:
            out.append(p)
            n //= p
        p += 1
    return out


def _input(dt, rows, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if dt == "CI16":
        return torch.randint(-32768, 32768, (rows, 2), generator=g, dtype=torch.int16, device="cuda")
    return torch.randn((rows, 2), generator=g, dtype=TORCH_DT[dt], device="cuda")


def _run(dt, n, inverse, x, key):
    """One Fft.run into a NaN- (or sentinel-) filled output with a spare half transform past the batch."""
    from pothoscomms_b200 import Fft
    f = Fft({"CF32": "complex_float32", "CF64": "complex_float64", "CI16": "complex_int16"}[dt], n, inverse)
    batch = x.shape[0] // n
    out = torch.full((batch * n + n // 2, 2), SENT_I16 if dt == "CI16" else float("nan"), dtype=x.dtype, device="cuda")
    _, names = _profiled(lambda: f.run(x, out=out), key=key)
    tail = out[batch * n:]
    assert bool((tail == SENT_I16).all() if dt == "CI16" else torch.isnan(tail).all()), "written past the batch"
    return out[:batch * n], names


def _check_float(dt, n, inverse, x, y, what):
    """Every transform against complex128 torch.fft (kiss_fft's inverse is unnormalised), relative to its own RMS."""
    batch = x.shape[0] // n
    step = max(1, (1 << 26) // n)
    for b0 in range(0, batch, step):
        b1 = min(batch, b0 + step)
        xs = torch.view_as_complex(x[b0 * n:b1 * n].double().contiguous()).view(b1 - b0, n)
        ref = torch.fft.ifft(xs, dim=1) * n if inverse else torch.fft.fft(xs, dim=1)
        got = torch.view_as_complex(y[b0 * n:b1 * n].double().contiguous()).view(b1 - b0, n)
        err = ((got - ref).abs() ** 2).mean(1).sqrt() / (ref.abs() ** 2).mean(1).sqrt()
        bad = ~(err <= TOL[dt])
        if bool(bad.any()):
            idx = (bad.nonzero()[:, 0] + b0)[:6].tolist()
            pytest.fail(f"{what}: {int(bad.sum())} transforms out of tolerance {TOL[dt]}, first {idx}, "
                        f"worst {float(err.max()):.2e}")


def _check_i16(oracle, n, inverse, x, y, what, transforms=None):
    """int16 bit for bit with oracle.fft: every transform, or the listed ones."""
    xh, yh = x.cpu().numpy(), y.cpu().numpy()
    if transforms is None:
        ref = oracle.fft(oracle.CI16, n, inverse, xh)
        if not np.array_equal(yh, ref):
            bad = np.unique(np.nonzero((yh != ref).any(axis=1))[0] // n)
            pytest.fail(f"{what}: {bad.size} transforms differ, first {bad[:6].tolist()}")
        return
    for b in transforms:
        ref = oracle.fft(oracle.CI16, n, inverse, xh[b * n:(b + 1) * n])
        assert np.array_equal(yh[b * n:(b + 1) * n], ref), f"{what}: transform {b} differs"


# ------------------------------------------------------------------------- staged kernel, shared memory ---
@pytest.mark.parametrize("inverse", [False, True], ids=["fwd", "inv"])
@pytest.mark.parametrize("dt", ["CF32", "CF64", "CI16"])
@pytest.mark.parametrize("n", [1000, 97])
def test_staged_shared_memory_kernel_every_transform_over_rounds(oracle, cuda_device, n, dt, inverse):
    """n = 1000 (two transforms per CTA) and n = 97 (the generic butterfly, 21 per CTA): 3 grid rounds and one group
    more, the last group partial."""
    sms = _sms()
    tpc, smem, generic = staged_plan(n, dt)
    assert smem and tpc == {1000: 2, 97: 21}[n] and generic == (n == 97)
    grid = 8 * sms
    batch = tpc * 3 * grid + 1                            # ngroups = 3 grid + 1, the last group one transform
    ngroups = _cdiv(batch, tpc)
    assert ngroups >= 3 * grid + 1 and batch % tpc, (batch, tpc)
    x = _input(dt, batch * n, 10 * n + len(dt) + inverse)
    y, names = _run(dt, n, inverse, x, "fft")
    what = f"staged smem {dt} n={n} {'inv' if inverse else 'fwd'} (batch {batch}, {ngroups} groups, grid {grid})"
    assert names and all(re.search(rf"fft_staged_kernel<b200c::{TRAITS[dt]},true>\(", k) for k in names), names
    if dt == "CI16":
        _check_i16(oracle, n, inverse, x, y, what)
    else:
        _check_float(dt, n, inverse, x, y, what)


# ------------------------------------------------------------------------- staged kernel, global memory ---
@pytest.mark.parametrize("dt", ["CF32", "CF64", "CI16"])
@pytest.mark.parametrize("n", [1 << 17, 2 * 13001])
def test_staged_global_memory_kernel_over_rounds(oracle, cuda_device, n, dt):
    """Transforms too large for shared memory, 2 grid rounds and 3 more: the generic n = 2 * 13001 reuses each CTA's
    scratch slice on every round.  Floats: every transform; int16: transforms b, b + grid and b + 2 grid."""
    sms = _sms()
    tpc, smem, generic = staged_plan(n, dt)
    assert not smem and tpc == 1 and generic == (n != 1 << 17)
    grid = 8 * sms
    batch = 2 * grid + 3
    x = _input(dt, batch * n, n + len(dt))
    y, names = _run(dt, n, False, x, "fft")
    what = f"staged global {dt} n={n} (batch {batch}, grid {grid})"
    assert names and all(re.search(rf"fft_staged_kernel<b200c::{TRAITS[dt]},false>\(", k) for k in names), names
    if dt == "CI16":
        _check_i16(oracle, n, False, x, y, what, transforms=[t for b in (0, 1, grid - 1) for t in (b, b + grid, b + 2 * grid)
                                                             if t < batch])
    else:
        _check_float(dt, n, False, x, y, what)


# ------------------------------------------------------------------------------------------- fft4096 ---
@pytest.mark.parametrize("inverse", [False, True], ids=["fwd", "inv"])
@pytest.mark.parametrize("dt", ["CF32", "CI16"])
def test_fft4096_kernel_every_transform_over_rounds(oracle, cuda_device, dt, inverse):
    """batch = 3 * 12 SMs + 5: three grid rounds and a ragged fourth."""
    sms = _sms()
    grid = 12 * sms
    batch = 3 * grid + 5
    x = _input(dt, batch * 4096, 4096 + len(dt) + inverse)
    y, names = _run(dt, 4096, inverse, x, "fft")
    what = f"fft4096 {dt} {'inv' if inverse else 'fwd'} (batch {batch}, grid {grid})"
    traits = r"Q15Lazy," + ("1" if inverse else "0") if dt == "CI16" else TRAITS[dt]
    assert names and all(re.search(rf"fft4096_kernel<b200c::{traits}", k) for k in names), names
    if dt == "CI16":
        _check_i16(oracle, 4096, inverse, x, y, what)
    else:
        _check_float(dt, 4096, inverse, x, y, what)


def _full_scale_patterns(n):
    """Full-scale complex int16 transforms: every sample -32768; +32767 / -32768 alternating (re and im in phase, and
    in opposite phase); a full-scale tone on one bin; a full-scale impulse (both signs).  They drive the Q15 butterflies
    to the edges of the int16 range that random inputs never reach."""
    t = np.arange(n)
    alt = np.where(t % 2 == 0, 32767, -32768)
    pats = [np.full((n, 2), -32768), np.stack([alt, alt], 1), np.stack([alt, -1 - alt], 1)]
    for k in (5, n - 3):                                          # a tone on bin 5 and one on bin -3
        ph = 2 * np.pi * k * t / n
        pats.append(np.stack([np.round(32767 * np.cos(ph)), np.round(32767 * np.sin(ph))], 1))
    imp = np.zeros((n, 2))
    imp[0] = (32767, -32768)
    pats.append(imp)
    imp2 = np.zeros((n, 2))
    imp2[n // 3] = (-32768, -32768)
    pats.append(imp2)
    return np.concatenate(pats).astype(np.int16)


@pytest.mark.parametrize("inverse", [False, True], ids=["fwd", "inv"])
@pytest.mark.parametrize("n,kernel", [(4096, r"fft4096_kernel<b200c::Q15Lazy"), (1024, r"fft_staged_kernel<b200c::Q15Traits,true>"),
                                      (1000, r"fft_staged_kernel<b200c::Q15Traits,true>")])
def test_int16_full_scale_structured_inputs(oracle, cuda_device, n, kernel, inverse):
    """The lazy-wrap 4096-point kernel (Q15Lazy: int16 values carried unwrapped in 32-bit registers) and the staged
    kernel at n = 1024 and 1000 on inputs at the ends of the int16 range, bit for bit with oracle.fft."""
    xh = _full_scale_patterns(n)
    x = torch.from_numpy(xh).cuda()
    y, names = _run("CI16", n, inverse, x, "fft")
    assert names and all(re.search(kernel, k) for k in names), names
    _check_i16(oracle, n, inverse, x, y, f"full-scale patterns n={n} {'inv' if inverse else 'fwd'}")
