"""Every output of the persistent single-stream FIR kernels, at launch sizes that cycle their loops.

The single-stream kernels are persistent: a CTA or warp takes a block or tile, prefetches the next one into a landing
buffer or bulk-copy ring, flips an mbarrier parity and steps on by gridDim.x * WARPS.  Bugs live in the second and
later trips of that loop: a reused ring slot, a wrong parity, a prefetch that crosses into the next task, the ragged
last round.  Each case here:
  * sizes the launch from a Python copy of the launch rule (fir_os_launch, fir_ummap.cu's launch_up) with the
    device's SM count, and asserts the property it exists for: at least 3 blocks per warp (or group), at least
    2 rounds of the grid, or at least 2R + 1 tiles per CTA so that every ring slot and both parities are reused,
    and a ragged last round;
  * fills the output with NaN (int16: a sentinel) first and asserts nothing is written past the produced count;
  * compares every output with the float64 reference (tests/_stream_ref.py) in windows of 4096 outputs: RMS error
    <= 1e-5 and max error <= 5e-4 of the stream's output RMS for float32; int16 bit for bit against oracle.fir;
  * records with torch.profiler the demangled kernel that ran, template arguments included (FirFilter.kernel
    cannot tell fir_os64_kernel from fir_os64p_kernel, or the spread from the persistent form).
"""
import os
import re

import numpy as np
import pytest
import torch

from _gpu_checks import _check, _profiled, _untouched
from _stream_ref import stream_ref

pytestmark = pytest.mark.gpu

B200_SMS = 148
NAN = float("nan")
SENT_I16 = 12345
F32, CF32 = 0, 1                         # b200c dtype codes
THREADS = max(1, min(16, os.cpu_count() or 1))


@pytest.fixture(autouse=True)
def _free_memory():
    yield
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _cdiv(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------------------- launch rules ---
# Python copies of fir_os_launch (csrc/fir_os.cu) and launch_up (csrc/fir_ummap.cu) for one stream.
def _span(ntaps, M, L):
    """configure_general: the spread of the window positions a = floor((d_p - k) / M) over every tap."""
    a = [(((p + 1) * M - 1) // L - k) // M for p in range(L) for k in range(_cdiv(ntaps - ((p + 1) * M - 1) % L, L))]
    return max(a) - min(a)


def os32_plan(n_out, ntaps, sms):
    hop = 1024 - (ntaps - 1)
    nblk = _cdiv(n_out, hop)
    spread = nblk < 12 * sms
    grid = min(nblk if spread else _cdiv(nblk, 12), sms)
    return dict(kernel=r"fir_os32_kernel<12,1,true,false,true>\(", nblk=nblk, grid=grid, spread=spread,
                workers=grid * 12, per=nblk // (grid * 12))


def os64_plan(n_out, ntaps, sms):
    hop = 4096 - (ntaps - 1)
    nblk = _cdiv(n_out, hop)
    if nblk >= 16 * sms:    # fir_os64p_kernel, parts = SMs: group g of CTA `part` takes blocks part*4 + g, step parts*4
        return dict(kernel=r"fir_os64p_kernel\(", nblk=nblk, grid=sms, persistent=True, workers=4 * sms,
                    per=nblk // (4 * sms))
    grid = min(nblk, 16 * sms)
    return dict(kernel=r"fir_os64_kernel<4>\(", nblk=nblk, grid=grid, persistent=False, workers=grid, per=nblk // grid)


def os32r_plan(n_out, ntaps, sms):
    hop = 1024 - (ntaps - 1)
    npair = _cdiv(n_out, 2 * hop)
    grid = min(_cdiv(npair, 12), sms)
    return dict(kernel=r"fir_os32r_kernel<12,1,true>\(", nblk=npair, grid=grid, workers=grid * 12,
                per=npair // (grid * 12), lone_a=0 < n_out - (npair - 1) * 2 * hop <= hop)


def os32x_plan(nq, ntaps, sms):
    m0 = _cdiv(_cdiv(ntaps - 2, 2), 3) * 3
    nblk = _cdiv(3 * nq, 1536 - m0)
    grid = min(_cdiv(nblk, 12), sms)
    return dict(kernel=r"fir_os32x_kernel<12,1,true,true>\(", nblk=nblk, grid=grid, workers=grid * 12,
                per=nblk // (grid * 12))


def general_plan(nq, ntaps, M, L, real, sms):
    """fir_ospg_kernel / fir_osp_kernel / fir_os32g_kernel: which form, its grid and the blocks per worker."""
    hopq = 1024 - _span(ntaps, M, L)
    osp = not real and L <= 4 and M <= 4 and max(L, M) >= 2 and not (L == 1 and M <= 2)
    if osp:
        nw = max(L, M)
        G = {2: 6, 3: 4, 4: 3}[nw]
        plane = 1056 + {2: 8, 3: 11}.get(L, 12)                                   # osp_plane_stride
        group = M * 1056 + L * plane
        nblk = _cdiv(nq, hopq)
        if 8 * (L * M * 1024 + 1024 + G * group) <= 227 * 1024:
            grid = min(_cdiv(nblk, G), sms)
            return dict(kernel=rf"fir_ospg_kernel<{nw},{G}>\(", nblk=nblk, grid=grid, workers=grid * G,
                        per=nblk // (grid * G))
        minb = {2: 7, 3: 5, 4: 3}[nw]
        per_sm = max(1, min(minb, (224 * 1024) // (8 * group + 1024)))
        grid = min(nblk, sms * per_sm * 2)
        return dict(kernel=rf"fir_osp_kernel<{nw},{minb}>\(", nblk=nblk, grid=grid, workers=grid, per=nblk // grid)
    nblk = _cdiv(nq, hopq * (2 if real else 1))
    ml, tile = L > 1, 2 <= L <= 4
    minb = (12 if not ml else 10) if M == 1 else (10 if not ml else 8)
    smem = 8 * (L * (1024 + 37) if tile else 1056)
    per_sm = min(minb, max(1, (220 * 1024) // (smem + 1024)))
    grid = min(nblk, sms * per_sm * 4)
    targs = f"{M},{'true' if ml else 'false'},{'true' if real else 'false'},{'true' if tile else 'false'},{minb}"
    return dict(kernel=rf"fir_os32g_kernel<{targs}>\(", nblk=nblk, grid=grid, workers=grid, per=nblk // grid)


def ummap_plan(nq, ntaps, M, L, complex_data, sms):
    """fir_ummap_configure + launch_up: tiles of 2048 blocks, grid min(ntiles, SMs), landing ring depth R."""
    dc = 2 if complex_data else 1
    N = 16 * L * dc * 2
    K = _cdiv(ntaps, L)
    a_max = max(((p + 1) * M - 1) // L + K - 1 for p in range(L)) // M
    NB = (15 + a_max + 1 + 31) // 32
    PL = 2048 + 32 * NB
    PLa = _cdiv(PL, 128) * 128
    tab = (2 * M * dc * NB * 16 + 127) & ~127
    bm = M * dc * NB * N * 32 + tab
    stage, one = M * dc * 2 * PLa, PL * M * dc * 2
    pstage = 2 if bm + 2 * stage + 3 * one + 1024 <= 210 * 1024 else 1
    fixed = bm + pstage * stage + 1024
    R = max(2, min(6, (216 * 1024 - fixed) // one))
    ntiles = _cdiv(nq, 2048)
    grid = min(ntiles, sms)
    return dict(kernel=rf"fir_ummap_kernel<{dc}>\(", nblk=ntiles, grid=grid, R=R, per=ntiles // grid,
                ragged=nq % 2048 != 0 and ntiles % grid != 0)


def _assert_kernels(names, pattern, what):
    assert names, f"{what}: the profiler recorded no fir kernel"
    bad = [n for n in names if not re.search(pattern, n)]
    assert not bad, f"{what}: expected only {pattern}, ran {sorted(set(names))}"


# ------------------------------------------------------------------------------------------------- runners ---
def _taps(seed, ntaps, complex_taps, scale=1.0):
    rng = np.random.default_rng(seed)
    h = rng.standard_normal(ntaps) / np.sqrt(ntaps)
    if complex_taps:
        h = h + 1j * rng.standard_normal(ntaps) / np.sqrt(ntaps)
    return h * scale


def _filter(code, taps_type, taps, M=1, L=1):
    from pothoscomms_b200 import FirFilter
    f = FirFilter(code, taps_type)
    f.set_rates(M, L)
    f.set_taps(taps)
    return f


def _float_input(nc, n, seed, offset=0):
    """[n, nc] float32 on the device starting `offset` elements into its allocation (16-byte aligned at offset 0)."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    buf = torch.randn((n + offset, nc), generator=g, device="cuda")
    return buf[offset:]


def _as_stream(x):
    return torch.view_as_complex(x) if x.shape[1] == 2 else x[:, 0]


def _run_float(code, taps_type, taps, M, L, n_new, seed, what, offset=0, zero_tail=False, cap=None):
    """One work() call on a fresh filter; every output against stream_ref; nothing past the produced count.
    Returns (profiled kernel names, produced)."""
    f = _filter(code, taps_type, taps, M, L)
    K = f.K
    nc = 2 if code & 1 else 1
    x = _float_input(nc, K - 1 + n_new, seed, offset)
    if offset:
        assert x.data_ptr() % 16 != 0
    n_in = x.shape[0]
    cap = f.default_capacity(n_in, zero_tail) if cap is None else cap
    out = torch.full((cap + 64, nc), NAN, dtype=torch.float32, device="cuda")
    (_, cons, prod), names = _profiled(lambda: f.run(x, out=out, out_capacity=cap, zero_tail=zero_tail))
    ref, c_ref, p_ref = stream_ref(_as_stream(x), taps, M, L, zero_tail, cap)
    assert (cons, prod) == (c_ref, p_ref), what
    _check(_as_stream(out[:prod])[None], ref[None], f"{what} [{f.kernel}]")
    _untouched(out[prod:], NAN, what + " past the produced count")
    return names, prod


# ------------------------------------------------------------------------ int16 resampling on tcgen05 (ummap) ---
# (dtype, taps type, M, L); 255 taps in two-digit Q16, full-scale input
UMMAP = [("CI16", "COMPLEX", 2, 3), ("CI16", "COMPLEX", 4, 4), ("CI16", "COMPLEX", 2, 1), ("I16", "REAL", 1, 2)]
UMMAP_R_B200 = {(2, 3): 6, (4, 4): 3, (2, 1): 6, (1, 2): 6}


def _ummap_setup(oracle, dt, taps_type, M, L, seed):
    code = getattr(oracle, dt)
    cx = taps_type == "COMPLEX"
    taps = _taps(seed, 255, cx, 0.3 * np.sqrt(L))
    f = _filter(code, taps_type, taps, M, L)
    assert f.kernel == "fir_ummap_kernel", f.kernel
    return code, cx, taps, f


def _i16_input(nc, n, seed, offset=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    buf = torch.randint(-32768, 32768, (n + offset, nc), generator=g, dtype=torch.int16, device="cuda")
    return buf[offset:]


def _run_ummap(oracle, code, cx, taps, f, M, L, n_blocks, seed, what, offset=0):
    nc = 2 if code & 1 else 1
    x = _i16_input(nc, f.K - 1 + n_blocks * M, seed, offset)
    cap = n_blocks * L
    obuf = torch.full((cap + offset + 16, nc), SENT_I16, dtype=torch.int16, device="cuda")
    out = obuf[offset:]
    (_, cons, prod), names = _profiled(lambda: f.run(x, out=out, out_capacity=cap))
    xh = x.cpu().numpy()
    y_ref, c_ref, p_ref = oracle.fir(code, cx, taps, M, L, xh, out_capacity=cap, threads=THREADS)
    assert (cons, prod) == (c_ref, p_ref) == (n_blocks * M, n_blocks * L), what
    got = out[:prod].cpu().numpy()
    if not np.array_equal(got, y_ref):
        bad = np.nonzero((got != y_ref).any(axis=1))[0]
        tiles = np.unique(bad // L // 2048)
        pytest.fail(f"{what}: {bad.size} outputs differ, first at {bad[:4].tolist()} (tiles {tiles[:8].tolist()})")
    _untouched(obuf[offset + prod:], SENT_I16, what + " past the produced count")
    _untouched(obuf[:offset], SENT_I16, what + " before the output")
    return names, x


@pytest.mark.parametrize("dt,taps_type,M,L", UMMAP, ids=[f"{c[0]}-{c[1]}-M{c[2]}-L{c[3]}" for c in UMMAP])
def test_ummap_every_output_over_many_tiles_per_cta(oracle, cuda_device, dt, taps_type, M, L):
    """At least 2R + 1 tiles per CTA: every slot of the raw-tile ring, both accumulator and plane stages and both
    parities of each are reused; a ragged last tile and a ragged last round."""
    sms = _sms()
    code, cx, taps, f = _ummap_setup(oracle, dt, taps_type, M, L, 31 * M + L)
    R = ummap_plan(2048, 255, M, L, code & 1 == 1, sms)["R"]
    if sms == B200_SMS:
        assert R == UMMAP_R_B200[(M, L)], "the Python copy of launch_up's ring depth drifted"
    n_blocks = ((2 * R + 1) * sms + sms // 2) * 2048 + 1001        # half the CTAs take one tile more; the last is ragged
    plan = ummap_plan(n_blocks, 255, M, L, code & 1 == 1, sms)
    assert plan["per"] >= 2 * R + 1 and plan["ragged"], plan
    what = f"ummap {dt}/{taps_type} M={M} L={L} ({plan['nblk']} tiles, grid {plan['grid']}, R {R})"
    names, _ = _run_ummap(oracle, code, cx, taps, f, M, L, n_blocks, 7 * M + L, what)
    _assert_kernels(names, plan["kernel"], what)


@pytest.mark.parametrize("dt,taps_type,M,L,offsets", [("CI16", "COMPLEX", 2, 3, (1, 2, 3)),
                                                      ("I16", "REAL", 1, 2, (1, 2, 3, 4, 5, 6, 7))],
                         ids=["CI16-COMPLEX-M2-L3", "I16-REAL-M1-L2"])
def test_ummap_unaligned_input_every_tile_without_bulk_copy(oracle, cuda_device, dt, taps_type, M, L, offsets):
    """An input that starts off 16-byte alignment: no tile may be bulk-copied, every tile's ring slot is released by
    the issuer's arrive alone and the stagers read the stream with guarded loads.  The output is shifted as well
    (the epilogue's unaligned stores).  A few tiles per CTA."""
    sms = _sms()
    code, cx, taps, f = _ummap_setup(oracle, dt, taps_type, M, L, 5 * M + L)
    n_blocks = 3 * sms * 2048 + 5 * 2048 + 333
    plan = ummap_plan(n_blocks, 255, M, L, code & 1 == 1, sms)
    assert plan["per"] >= 3, plan
    for off in offsets:
        what = f"ummap {dt} M={M} L={L} input offset {off}"
        names, x = _run_ummap(oracle, code, cx, taps, f, M, L, n_blocks, 100 + off, what, offset=off)
        assert x.data_ptr() % 16 != 0
        _assert_kernels(names, plan["kernel"], what)


# ------------------------------------------------------------------- headline: fir_os32_kernel, one stream ---
def _os32_n_new(kind, ntaps, sms):
    hop = 1024 - (ntaps - 1)
    if kind == "spread":          # just under one wave of warps: 12 SMs - 1 blocks, the last one ragged
        return (12 * sms - 2) * hop + hop // 2
    return (1 << 24) + 333


OS32 = [   # (id, ntaps, size, input offset, zero tail, capacity as a fraction of the outputs)
    ("K256-spread", 256, "spread", 0, False, None),
    ("K256-persistent", 256, "long", 0, False, None),
    ("K9-persistent", 9, "long", 0, False, None),
    ("K448-persistent", 448, "long", 0, False, None),
    ("K256-persistent-offset1", 256, "long", 1, False, None),
    ("K256-spread-offset1", 256, "spread", 1, False, None),
    ("K256-persistent-zero-tail", 256, "long", 0, True, None),
    ("K256-persistent-capacity-mid-block", 256, "long", 0, False, 0.7),
]


@pytest.mark.parametrize("name,ntaps,size,offset,zero_tail,capfrac", OS32, ids=[c[0] for c in OS32])
def test_headline_kernel_every_output(cuda_device, name, ntaps, size, offset, zero_tail, capfrac):
    """Complex float32, complex taps, L = M = 1.  Spread: one block per warp, dealt warp-major.  Persistent: about
    12 blocks per warp through the landing buffers.  An input one element in (the `mis` shift of every bulk copy,
    block 0 guarded), the burst zero tail, a capacity ending inside a block."""
    sms = _sms()
    n_new = _os32_n_new(size, ntaps, sms)
    taps = _taps(ntaps + 1, ntaps, True)
    n_out = n_new + (ntaps - 1 if zero_tail else 0)
    cap = None
    if capfrac is not None:
        hop = 1024 - (ntaps - 1)
        cap = int(n_out * capfrac) // hop * hop + hop // 3        # ends a third of the way into a block
        n_out = cap
    plan = os32_plan(n_out, ntaps, sms)
    if size == "spread":
        assert plan["spread"] and plan["nblk"] == 12 * sms - 1, plan
    else:
        assert not plan["spread"] and plan["per"] >= 3 and plan["nblk"] % plan["workers"], plan
    what = f"os32 {name} ({plan['nblk']} blocks, grid {plan['grid']}, {plan['per']}+ per warp)"
    names, prod = _run_float(CF32, "COMPLEX", taps, 1, 1, n_new, 1000 + ntaps + offset, what,
                             offset=offset, zero_tail=zero_tail, cap=cap)
    assert prod == n_out, what
    _assert_kernels(names, plan["kernel"], what)


def test_headline_kernel_chain_with_programmatic_dependent_launch(cuda_device):
    """A (64 taps) -> B (256 taps) through one device buffer, six rounds with no host synchronisation: both launches
    above 12 SMs blocks, so the persistent form's griddepcontrol.wait is what orders B's reads after A's writes.  Every
    round's every output against the float64 chain."""
    sms = _sms()
    ta, tb = _taps(64, 64, True), _taps(256, 256, True)
    fa, fb = _filter(CF32, "COMPLEX", ta), _filter(CF32, "COMPLEX", tb)
    n_a = 12 * sms * 961 + 12345                      # A's outputs
    pa_plan, pb_plan = os32_plan(n_a, 64, sms), os32_plan(n_a - 255, 256, sms)
    assert not pa_plan["spread"] and not pb_plan["spread"], (pa_plan, pb_plan)
    rounds, nx = 6, 3
    xs = [_float_input(2, 63 + n_a, 500 + k) for k in range(nx)]
    mid = torch.full((n_a, 2), NAN, device="cuda")
    outs = [torch.full((n_a, 2), NAN, device="cuda") for _ in range(rounds)]

    def chain():
        prods = []
        for r in range(rounds):
            _, _, pa = fa.run(xs[r % nx], out=mid)
            _, _, pb = fb.run(mid[:pa], out=outs[r])
            prods.append((pa, pb))
        return prods

    prods, names = _profiled(chain)
    _assert_kernels(names, pa_plan["kernel"], "chain")
    for k in range(nx):
        ya, _, _ = stream_ref(_as_stream(xs[k]), ta)
        yb, _, pb = stream_ref(ya, tb)
        del ya
        for r in range(k, rounds, nx):
            assert prods[r] == (n_a, n_a - 255) and pb == n_a - 255, prods[r]
            _check(_as_stream(outs[r][:pb])[None], yb[None], f"chain round {r}")
            _untouched(outs[r][pb:], NAN, f"chain round {r} past the produced count")


# -------------------------------------------------------------------- 4096-point: fir_os64 / fir_os64p ---
OS64 = [   # (id, ntaps, size, input offset)
    ("K1024-below-switch", 1024, "below", 0),
    ("K1024-at-switch", 1024, "at", 0),
    ("K1024-long", 1024, "long", 0),
    ("K1024-long-offset1", 1024, "long", 1),
    ("K2049-below-switch", 2049, "below", 0),
    ("K2049-at-switch", 2049, "at", 0),
    ("K2049-long", 2049, "long", 0),
    ("K2049-at-switch-offset1", 2049, "at", 1),
]


@pytest.mark.parametrize("name,ntaps,size,offset", OS64, ids=[c[0] for c in OS64])
def test_4096_point_kernels_every_output(cuda_device, name, ntaps, size, offset):
    """16 SMs - 1 blocks run fir_os64_kernel<4>, 16 SMs blocks the persistent fir_os64p_kernel (parts = SMs), and
    2^24 + 1001 outputs give each of its transform groups about 9 (1024 taps) or 13 (2049 taps) blocks."""
    sms = _sms()
    hop = 4096 - (ntaps - 1)
    n_new = {"below": (16 * sms - 2) * hop + 5, "at": (16 * sms - 1) * hop + 7, "long": (1 << 24) + 1001}[size]
    plan = os64_plan(n_new, ntaps, sms)
    if size == "below":
        assert not plan["persistent"] and plan["nblk"] == 16 * sms - 1, plan
    elif size == "at":
        assert plan["persistent"] and plan["nblk"] == 16 * sms, plan
    else:
        assert plan["persistent"] and plan["per"] >= 3 and plan["nblk"] % plan["workers"], plan
    what = f"os64 {name} ({plan['nblk']} blocks, grid {plan['grid']}, {plan['per']}+ per group)"
    names, _ = _run_float(CF32, "COMPLEX", _taps(ntaps, ntaps, True), 1, 1, n_new, 2000 + ntaps + offset, what,
                          offset=offset)
    _assert_kernels(names, plan["kernel"], what)


# ------------------------------------------------------------------------- real float32: fir_os32r_kernel ---
@pytest.mark.parametrize("ntaps,offset", [(64, 0), (448, 0), (64, 1), (448, 3)])
def test_real_float32_kernel_every_output(cuda_device, ntaps, offset):
    """Real float32 stream, real taps: two blocks per complex transform, a warp taking a pair per trip.  2^24 + 7
    samples is an odd number of blocks (64 taps: the last pair a lone block A) and several pairs per warp."""
    sms = _sms()
    n_new = (1 << 24) + 7
    hop = 1024 - (ntaps - 1)
    if ntaps == 448:
        n_new = (n_new // (2 * hop)) * 2 * hop + hop // 2          # a lone block A as well
    plan = os32r_plan(n_new, ntaps, sms)
    assert plan["per"] >= 3 and plan["lone_a"] and plan["nblk"] % plan["workers"], plan
    what = f"os32r K={ntaps} offset {offset} ({plan['nblk']} pairs, grid {plan['grid']}, {plan['per']}+ per warp)"
    names, _ = _run_float(F32, "REAL", _taps(ntaps + 7, ntaps, False), 1, 1, n_new, 3000 + ntaps + offset, what,
                          offset=offset)
    _assert_kernels(names, plan["kernel"], what)


@pytest.mark.parametrize("ntaps", [449, 600])
def test_real_float32_beyond_448_taps_runs_the_direct_kernel(oracle, cuda_device, ntaps):
    """Above 448 taps a real float32 stream at L = M = 1 leaves fir_os32r_kernel.  The polyphase kernel refuses a
    window span above 400 (at M = 1 the span is ntaps - 1), so the direct kernel keeps the job."""
    taps = _taps(ntaps + 9, ntaps, False)
    f = _filter(oracle.F32, "REAL", taps)
    assert f.kernel == "fir_tile_kernel", f.kernel
    names, _ = _run_float(oracle.F32, "REAL", taps, 1, 1, 200003, 4000 + ntaps, f"F32 K={ntaps}")
    _assert_kernels(names, r"fir_tile_kernel\b", f"F32 K={ntaps}")


# --------------------------------------------------------------------- 3/2 resampler: fir_os32x_kernel ---
OS32X = [   # (id, taps, input offset, capacity fraction)
    ("c3", "c3", 0, None),
    ("K1200", 1200, 0, None),
    ("c3-offset1", "c3", 1, None),
    ("K1200-capacity-mid-block", 1200, 0, 0.6),
]


@pytest.mark.parametrize("name,taps_kind,offset,capfrac", OS32X, ids=[c[0] for c in OS32X])
def test_resampler_3_2_kernel_every_output(cuda_device, name, taps_kind, offset, capfrac):
    """Complex float32, L = 3, M = 2: C3's 255 real taps and 1200 complex taps, 2^24 inputs (about 10 and 15 blocks
    per warp), an input one element in, a capacity that is not a multiple of L and ends inside a block."""
    from pothoscomms_b200 import workloads as wl
    sms = _sms()
    if taps_kind == "c3":
        taps, tt = wl.config_taps("c3")
    else:
        taps, tt = _taps(1200, 1200, True), "COMPLEX"
    ntaps = len(taps)
    n_new = 1 << 24
    nq = n_new // 2
    cap = None
    if capfrac is not None:
        cap = int(nq * 3 * capfrac) + 1
        nq = cap // 3
    plan = os32x_plan(nq, ntaps, sms)
    assert plan["per"] >= 3 and plan["nblk"] % plan["workers"], plan
    what = f"os32x {name} ({plan['nblk']} blocks, grid {plan['grid']}, {plan['per']}+ per warp)"
    names, prod = _run_float(CF32, tt, taps, 2, 3, n_new, 5000 + ntaps + offset, what, offset=offset, cap=cap)
    assert prod == nq * 3, what
    _assert_kernels(names, plan["kernel"], what)


# --------------------------------------------------- polyphase / real-data kernels: ospg, osp, os32g ---
GENERAL = [   # (id, dtype code, taps type, M, L, ntaps, rounds wanted: per-worker blocks)
    ("ospg-CF32-M3-L2", 1, "COMPLEX", 3, 2, 255, 3),
    ("osp-CF32-M4-L4", 1, "COMPLEX", 4, 4, 255, 2),
    ("os32g-CF32-M2-L1", 1, "COMPLEX", 2, 1, 255, 2),
    ("os32g-CF32-M1-L5", 1, "COMPLEX", 1, 5, 600, 2),
    ("os32g-F32-M2-L1", 0, "REAL", 2, 1, 255, 2),
]
GENERAL_KERNEL_B200 = {
    "ospg-CF32-M3-L2": "fir_ospg_kernel<3,4>",
    "osp-CF32-M4-L4": "fir_osp_kernel<4,3>",
    "os32g-CF32-M2-L1": "fir_os32g_kernel<2,false,false,false,10>",
    "os32g-CF32-M1-L5": "fir_os32g_kernel<1,true,false,false,10>",
    "os32g-F32-M2-L1": "fir_os32g_kernel<2,false,true,false,10>",
}


@pytest.mark.parametrize("name,code,taps_type,M,L,ntaps,want", GENERAL, ids=[c[0] for c in GENERAL])
def test_polyphase_kernels_every_output_over_grid_rounds(cuda_device, name, code, taps_type, M, L, ntaps, want):
    """The grouped resampler (3, 2) takes at least 3 blocks per group, the ungrouped one (4, 4) and the general kernel
    at least 2 rounds of their grids, each with a ragged last round.  Which form runs is decided by whether G groups and
    the tap spectra fit 227 KB of shared memory: the profiler says which one did."""
    sms = _sms()
    real = code == F32
    blk_q = (1024 - _span(ntaps, M, L)) * (2 if real else 1)        # blocks q one transform block covers
    workers = general_plan(1 << 40, ntaps, M, L, real, sms)["workers"]  # at the full grid
    nq = (want * workers + workers // 3) * blk_q + blk_q // 2           # `want` per worker, a third more, a ragged last
    plan = general_plan(nq, ntaps, M, L, real, sms)
    assert plan["per"] >= want and plan["nblk"] % plan["workers"], plan
    assert plan["kernel"].startswith(re.escape(GENERAL_KERNEL_B200[name])), plan
    what = f"{name} ({plan['nblk']} blocks, grid {plan['grid']}, {plan['per']}+ per worker)"
    names, prod = _run_float(code, taps_type, _taps(ntaps + M + L, ntaps, taps_type == "COMPLEX"), M, L, nq * M,
                             6000 + M * 10 + L, what)
    assert prod == nq * L, what
    _assert_kernels(names, plan["kernel"], what)
