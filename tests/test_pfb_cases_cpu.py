"""What tests/test_filterbank_instantiations_gpu.py covers, checked without a GPU: every template instantiation of the
four polyphase filter-bank kernels, every decimation that divides M, branch chains longer than a tile, the
synthesizers' bin-group classes and stream indices near 2^64 (case lists in tests/_pfb_cases.py)."""
import pytest

import _pfb_cases as pc

CHANS = ("chan", "rchan")
SYNTHS = ("synth", "rsynth")


def _inst(kernel):
    return pc.instantiation_cases(kernel)


@pytest.mark.parametrize("kernel", pc.KERNELS)
def test_every_instantiation_runs(kernel):
    cases = _inst(kernel)
    want = {(dt, n) for dt in pc.DTYPES[kernel] for n in range(1, pc.MAX_N[kernel] + 1)}
    assert {(c.dtype, c.n) for c in cases} == want
    assert len(want) == {"chan": 16, "rchan": 32, "synth": 32, "rsynth": 64}[kernel]
    unit = (lambda c: c.M) if kernel in CHANS else (lambda c: c.D)
    for dt, n in want:
        for M in pc.INST_M[kernel]:
            got = {c.ntaps for c in cases if (c.dtype, c.n, c.M) == (dt, n, M)}
            u = M if kernel in CHANS else M // 2
            assert got == {n * u, (n - 1) * u + 1}, (dt, n, M, got)   # every branch full, and the last one with one tap
    for c in cases:
        assert 1 <= c.ntaps <= pc.tap_limit(kernel, c.M, c.D) and c.M % c.D == 0, c
        assert -(-c.ntaps // unit(c)) == c.n
        assert c.F >= 2 * c.T + 5, c                                  # two full tiles and a ragged one


def test_instantiation_total():
    assert sum(len({(c.dtype, c.n) for c in _inst(k)}) for k in pc.KERNELS) == 144


@pytest.mark.parametrize("kernel", pc.KERNELS)
def test_every_decimation_divides_m(kernel):
    cases = pc.decimation_cases(kernel)
    for M in pc.SWEEP_M[kernel]:
        assert {c.D for c in cases if c.M == M} == {1 << j for j in range(M.bit_length())}, M
    for c in cases:
        assert c.ntaps <= pc.tap_limit(kernel, c.M, c.D)
        assert c.n == 3
    # a lone partial tile, one full tile, and a full tile plus one frame
    big = [c for c in cases if c.M == pc.SWEEP_M[kernel][-1]]
    for rel in (lambda c: c.F < c.T, lambda c: c.F == c.T, lambda c: c.F == c.T + 1):
        assert any(rel(c) for c in big)


@pytest.mark.parametrize("kernel", CHANS)
def test_channelizers_run_chains_longer_than_a_tile(kernel):
    # k = M / D > T: chains = min(k, nt), one frame per chain (chan.cu, rchan.cu)
    cases = pc.decimation_cases(kernel)
    k_gt_t = {(c.M, c.D) for c in cases if c.M // c.D > c.T}
    if kernel == "chan":
        assert {(1024, d) for d in (1, 2, 4, 8, 16, 32, 64)} <= k_gt_t
        assert pc.chan_tile(1024) == 8
    else:
        assert {(2048, d) for d in (1, 2, 4, 8, 16, 32, 64, 128)} <= k_gt_t
        assert pc.rchan_tile(2048) == 8
    # and a tile with fewer frames than chains
    assert any(c.M // c.D > c.F for c in cases)
    s = pc.streaming_case(kernel)
    assert s.M // s.D > s.T


@pytest.mark.parametrize("kernel", SYNTHS)
def test_synthesizers_run_mostly_idle_tiles(kernel):
    # small D at large M: thread l emits frames with (t0 + t) & (M/D - 1) == l >> log D, at most one per tile
    cases = pc.decimation_cases(kernel)
    assert any(c.M >= 1024 and c.M // c.D > c.T for c in cases)


def test_synthesizer_thread_classes():
    assert [pc.synth_max_threads(K) for K in (8, 9, 16, 17)] == [1024, 512, 512, 256]
    assert [pc.rsynth_max_threads(K) for K in (12, 13, 24, 25)] == [1024, 512, 512, 256]


@pytest.mark.parametrize("kernel", SYNTHS)
def test_bin_group_classes(kernel):
    """Mirror of the launch's B = bins per CTA and gridDim.y = M / B: every thread-count class runs at every M
    listed, and at each of those M the bins are split over gridDim.y in at least one class."""
    cases = pc.bin_class_cases(kernel)
    mt = pc.synth_max_threads if kernel == "synth" else pc.rsynth_max_threads
    got = {(c.M, c.n) for c in cases}
    assert got == {(M, K) for M in pc.BIN_CLASS_M[kernel] for K in pc.BIN_CLASS_K[kernel]}
    pairs = {(c.M, pc.bins_per_cta(kernel, c.M, c.n)) for c in cases}
    assert pairs == {(M, B) for M in pc.BIN_CLASS_M[kernel] for B in (1024, 512, 256)}
    for c in cases:
        assert c.ntaps <= pc.tap_limit(kernel, c.M, c.D) and c.F >= 2 * c.T + 5
        assert c.M // pc.bins_per_cta(kernel, c.M, c.n) >= 2 or mt(c.n) == 1024
    groups = {(c.M, c.M // pc.bins_per_cta(kernel, c.M, c.n)) for c in cases}
    if kernel == "synth":
        assert {(1024, 4), (2048, 8), (4096, 16), (4096, 4)} <= groups
    else:
        assert {(2048, 8), (4096, 16), (8192, 32), (8192, 8)} <= groups


@pytest.mark.parametrize("kernel", pc.KERNELS)
def test_stream_indices_near_2_64(kernel):
    cases = pc.wrap_cases(kernel)
    assert {c.s for c in cases} == {2**64 - 1, 2**64 - cases[0].M + 3}
    s = pc.streaming_case(kernel)
    assert s.s < 2**64 and s.D == 2 and s.M >= 1024


def test_mirrored_host_formulas():
    # chan_plan_create / rchan_plan_create: T M (or T M/2) about 8192, 4 .. 512
    assert [pc.chan_tile(M) for M in (2, 64, 1024, 4096)] == [512, 128, 8, 4]
    assert [pc.rchan_tile(M) for M in (2, 64, 2048, 8192)] == [512, 256, 8, 4]
    # synth_plan_create / rsynth_plan_create: P M (or P M/2) about 8192, 1 .. 16; T = max(4 P, 16 (K - 1))
    assert [pc.synth_chunk(M) for M in (64, 1024, 4096)] == [16, 8, 2]
    assert [pc.rsynth_chunk(M) for M in (64, 2048, 8192)] == [16, 8, 2]
    assert pc.tile("synth", 1024, 1) == 32 and pc.tile("synth", 1024, 32) == 496
    assert pc.tile("rsynth", 8192, 2) == 16
