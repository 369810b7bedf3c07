"""Case lists of tests/test_filterbank_instantiations_gpu.py, in plain Python so that tests/test_pfb_cases_cpu.py can
check what they cover without a GPU.

Each of the four polyphase filter-bank kernels is a template on the length of its register window, and the host picks
the instantiation from the tap count: pfb_chan_kernel<R> and pfb_rchan_kernel<R, float / int16_t> with
R = ceil(ntaps / M) (csrc/chan.cu, csrc/rchan.cu), pfb_synth_kernel<K> and pfb_rsynth_kernel<K, float / int16_t> with
K = ceil(ntaps / D) (csrc/synth.cu, csrc/rsynth.cu).  The formulas below mirror the host code that sizes a launch, so
the cases can be placed on the shapes where the kernels change layout."""
from __future__ import annotations

from typing import NamedTuple

CHAN_MAX_R = 16           # kChanMaxTapsPerBranch (csrc/chan.hpp): ntaps <= 16 M
SYNTH_MAX_K = 32          # kSynthMaxTapsPerPhase (csrc/synth.hpp): ntaps <= min(16 M, 32 D)
KERNELS = ("chan", "rchan", "synth", "rsynth")
DTYPES = {"chan": ("complex_float32",), "rchan": ("float32", "int16"), "synth": ("complex_float32",),
          "rsynth": ("float32", "int16")}
MAX_N = {"chan": CHAN_MAX_R, "rchan": CHAN_MAX_R, "synth": SYNTH_MAX_K, "rsynth": SYNTH_MAX_K}
S_VALUES = (0, 12345, 2**40 + 7)
INST_M = {"chan": (64, 1024), "rchan": (64, 2048), "synth": (64, 1024), "rsynth": (64, 2048)}
SWEEP_M = {"chan": (64, 1024), "rchan": (64, 2048), "synth": (64, 1024), "rsynth": (64, 2048)}
BIN_CLASS_M = {"synth": (1024, 2048, 4096), "rsynth": (2048, 4096, 8192)}
BIN_CLASS_K = {"synth": (8, 9, 16, 17), "rsynth": (12, 13, 24, 25)}
REF_BUDGET = 1 << 26      # multiply-adds of the float64 reference per case, above which only part of the output is compared


def _pow2_floor(v):
    return 1 << (v.bit_length() - 1)


def chan_tile(M):
    """Frames per CTA of pfb_chan_kernel: chan_plan_create (csrc/chan.cu), a power of two of about 8192 / M frames,
    4 .. 512.  (Its shared-memory loop never shrinks T at M <= 4096.)"""
    return _pow2_floor(max(4, min(512, 8192 // M)))


def rchan_tile(M):
    """Frames per CTA of pfb_rchan_kernel: rchan_plan_create (csrc/rchan.cu), about 8192 / (M/2) frames, 4 .. 512."""
    return _pow2_floor(max(4, min(512, 8192 // (M // 2))))


def synth_chunk(M):
    """Frames per shared-memory chunk P of pfb_synth_kernel: synth_plan_create (csrc/synth.cu)."""
    return max(1, min(16, 8192 // M))


def rsynth_chunk(M):
    """Frames per shared-memory chunk P of pfb_rsynth_kernel: rsynth_plan_create (csrc/rsynth.cu), on M/2 slots."""
    return max(1, min(16, 8192 // (M // 2)))


def synth_max_threads(K):
    """synth_max_threads (csrc/synth.cu): threads, and so bins, per CTA of pfb_synth_kernel<K>."""
    return 1024 if K <= 8 else 512 if K <= 16 else 256


def rsynth_max_threads(K):
    """rsynth_max_threads (csrc/rsynth.cu): threads, and so real bins, per CTA of pfb_rsynth_kernel<K>."""
    return 1024 if K <= 12 else 512 if K <= 24 else 256


def tile(kernel, M, n):
    """Frames per CTA (T) of `kernel` at M branches and window length n (R or K).  The synthesizers' T is
    synth_set_taps's max(4 P, 16 (K - 1)) (csrc/synth.cu; rsynth_set_taps calls it with its own P)."""
    if kernel == "chan":
        return chan_tile(M)
    if kernel == "rchan":
        return rchan_tile(M)
    P = synth_chunk(M) if kernel == "synth" else rsynth_chunk(M)
    return max(4 * P, 16 * (n - 1))


def bins_per_cta(kernel, M, K):
    """B = min(M, max threads): the bins of one CTA; M / B CTAs split a tile's bins over gridDim.y (synth_set_taps,
    rsynth_set_taps)."""
    return min(M, synth_max_threads(K) if kernel == "synth" else rsynth_max_threads(K))


class Case(NamedTuple):
    kernel: str
    dtype: str
    M: int
    D: int
    ntaps: int
    s: int
    F: int                # frames produced: output frames of the channelizers, output frames (F D samples) of the synthesizers

    @property
    def n(self):
        """The template argument the host picks: R = ceil(ntaps / M) or K = ceil(ntaps / D)."""
        return -(-self.ntaps // (self.M if self.kernel in ("chan", "rchan") else self.D))

    @property
    def T(self):
        return tile(self.kernel, self.M, self.n)

    @property
    def id(self):
        s = f"2^64-{2**64 - self.s}" if self.s >= 2**63 else "2^40+7" if self.s == 2**40 + 7 else str(self.s)
        return f"{self.kernel}-{self.dtype}-{'R' if self.kernel in ('chan', 'rchan') else 'K'}{self.n}-M{self.M}-D{self.D}-" \
               f"taps{self.ntaps}-F{self.F}-s{s}"


def tap_limit(kernel, M, D):
    return 16 * M if kernel in ("chan", "rchan") else min(16 * M, 32 * D)


def instantiation_cases(kernel):
    """Every instantiation of `kernel`, at a small and a large M, each with two tap counts that select it: every branch
    (phase) full, and the last one holding a single tap.  F = 2 T + 5: two full tiles and a ragged one.  The
    channelizers take D = M, M/2, M/4 in turn along R; the synthesizers take D = M/2, where K = 32 is allowed."""
    cases = []
    for dtype in DTYPES[kernel]:
        for n in range(1, MAX_N[kernel] + 1):
            for M in INST_M[kernel]:
                if kernel in ("chan", "rchan"):
                    D, unit = M >> (n % 3), M
                else:
                    D = unit = M // 2
                for i, ntaps in enumerate(sorted({n * unit, (n - 1) * unit + 1})):
                    s = S_VALUES[(n + i + (M > 64)) % 3]
                    cases.append(Case(kernel, dtype, M, D, ntaps, s, 2 * tile(kernel, M, n) + 5))
    return cases


def decimation_cases(kernel):
    """Every D = 2^j <= M at the sweep sizes, with about 3 taps per branch (R = 3) or phase (K = 3), F = 2 T + 5;
    and at the large M, D = 1 and D = 8, the frame counts F < T, F = T and F = T + 1 (a lone partial tile, and a tile
    with fewer frames than branch chains when M / D > T)."""
    cases = []
    dtype = DTYPES[kernel][0]
    for M in SWEEP_M[kernel]:
        for j in range(M.bit_length()):
            D = 1 << j
            ntaps = 3 * M - 1 if kernel in ("chan", "rchan") else 3 * D
            c = Case(kernel, dtype, M, D, ntaps, S_VALUES[j % 3], 0)
            frames = [2 * c.T + 5]
            if M == SWEEP_M[kernel][-1] and D in (1, 8):
                frames += [max(1, c.T // 2 - 1), c.T, c.T + 1]
            cases += [c._replace(F=F) for F in frames]
    return cases


def bin_class_cases(kernel):
    """The synthesizers' thread-count classes (both sides of each switch of synth_max_threads / rsynth_max_threads)
    at every M where bins are split over gridDim.y; D = 64 keeps K <= 25 under the 16 M tap limit and the
    reference cheap."""
    cases = []
    for M in BIN_CLASS_M[kernel]:
        for i, K in enumerate(BIN_CLASS_K[kernel]):
            D = 64
            c = Case(kernel, DTYPES[kernel][0], M, D, K * D - 5 * i, S_VALUES[(i + M // 1024) % 3], 0)
            cases.append(c._replace(F=2 * c.T + 5))
    return cases


def wrap_cases(kernel):
    """One shape per kernel at stream indices 2^64 - 1 and 2^64 - M + 3, where s + m0 wraps in uint64."""
    M, D = 64, 16
    ntaps = 3 * M + 5 if kernel in ("chan", "rchan") else 3 * D + 5
    base = Case(kernel, DTYPES[kernel][0], M, D, ntaps, 0, 0)
    base = base._replace(F=2 * base.T + 5)
    return [base._replace(s=2**64 - 1), base._replace(s=2**64 - M + 3)]


def streaming_case(kernel):
    """A k = M / D > T shape per kernel for the pieces-vs-one-call bit identity (M = 1024 or 2048, D = 2)."""
    M = 1024 if kernel in ("chan", "synth") else 2048
    D = 2
    ntaps = 3 * M + 5 if kernel in ("chan", "rchan") else 3 * D + 1
    return Case(kernel, DTYPES[kernel][-1], M, D, ntaps, 2**64 - 1000, 0)
