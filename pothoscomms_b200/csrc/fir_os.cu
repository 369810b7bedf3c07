// Fused overlap-save FIR for /comms/fir_filter, complex float32, L = M = 1, 2..2049 taps.
//
// The reference convolves in the time domain (filter/FIRFilter.cpp:286-302): 8K flop per
// sample for K complex taps, which on B200 is FMA-bound from K ~ 22 taps up (DESIGN.md 4.1).
// Here every CTA takes 4096 consecutive input samples (K-1 of them history), transforms them,
// multiplies by the taps' spectrum Hf (computed once per setTaps() on the host in double,
// pre-scaled by 1/4096), transforms back and stores the 4096-(K-1) alias-free outputs: ONE
// pass over HBM, 8 B in + 8 B out per sample whatever K is.
//
// Kernel shape (os64_core.cuh): 64 threads per transform, 64 points (128 registers) per
// thread, 4096 = 64 x 64.  Forward = two decimation-in-time register passes around one
// shared-memory exchange; inverse = the mirrored decimation-in-frequency passes, so the
// pointwise product sits between two passes that share registers and one overlap-save block
// costs TWO exchanges.  All arithmetic is packed f32x2 (packed.cuh).
#include <algorithm>
#include <cmath>
#include <complex>
#include <cstdlib>
#include <vector>

#include "bulk.cuh"
#include "fft.hpp"
#include "os64_core.cuh"

namespace b200c {

struct FirOs64Args {
    const void *in;     // channel 0, element 0 = first history sample
    void *out;
    const void *hf;     // [nchan][4096] spectrum of the taps / 4096, natural order
    const void *twa;    // [8][64]  W4096^(8*a*t)
    const void *twb;    // [8][64]  W4096^(b*t)
    const void *twf;    // [64][64] W4096^(j*t): the whole step-twiddle table (fir_os64p_kernel stages it in shared memory)
    long long n_in;     // valid input elements per channel (beyond: zeros -> burst zero tail)
    long long n_out;    // outputs to produce per channel
    long long in_stride, out_stride;   // elements between consecutive channels (filter bank)
    int nchan;
    int K;              // taps
    int parts;          // fir_os64p_kernel: a channel's blocks are dealt over this many CTA-tasks
};

// v[slot(j)] *= W4096^(j*t) (CONJ: conjugate), j = 8a + b, from the two 8-entry tables.
// SLOT_REV: element j lives in register rev64(j) (decimation-in-frequency output order).
template <bool CONJ, bool SLOT_REV>
__device__ __forceinline__ void step_twiddle(c2 (&v)[64], const c2 *__restrict__ twa, const c2 *__restrict__ twb, const int t)
{
    c2 A[8], B[8];
#pragma unroll
    for (int i = 1; i < 8; i++) { A[i] = twa[i * 64 + t]; B[i] = twb[i * 64 + t]; }
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int b = 0; b < 8; b++) {
            const int j = 8 * a + b, r = SLOT_REV ? rev64(j) : j;
            if (a) v[r] = cmul_p<CONJ>(v[r], A[a]);
            if (b) v[r] = cmul_p<CONJ>(v[r], B[b]);
        }
}

constexpr int kBulkElems = 4098;   // 4096 + 2: room to start one element early when the block start is not 16-byte aligned

template <int MINB>
__global__ void __launch_bounds__(64, MINB) fir_os64_kernel(const FirOs64Args a)
{
    __shared__ __align__(16) c2 F[kOs64SmemElems];
    __shared__ __align__(8) unsigned long long bar;
    const int t = threadIdx.x;
    const c2 *__restrict__ twa = static_cast<const c2 *>(a.twa);
    const c2 *__restrict__ twb = static_cast<const c2 *>(a.twb);
    const int Km1 = a.K - 1;
    const int hop = 4096 - Km1;
    const long long nblk = (a.n_out + hop - 1) / hop;
    // Tasks = (channel, block), channel-major, taken grid-stride: at any moment the resident CTAs
    // sweep one contiguous window of the stream(s) (DRAM-page friendly; a contiguous run per CTA
    // measured 18 % slower), and a block's overlap with its neighbour is an L2 hit.
    // (one 64-bit division per launch, none per task: the step is kept as (channels, blocks))
    const long long tstep = gridDim.x, dch = tstep / nblk, dblk = tstep - dch * nblk;
    long long ch = (long long)blockIdx.x / nblk, blk = (long long)blockIdx.x - ch * nblk;
    // A block whose 4096 inputs (plus alignment slack) are all inside the stream is fetched by one
    // bulk copy, issued while the previous block is still in its last register pass; the few
    // edge blocks (zero tail, unaligned stream start) use guarded loads.
    auto bulk_src = [&](long long ch, long long blk, const c2 *&src) {
        if (ch >= a.nchan) return false;
        const long long base = blk * hop;
        const c2 *in = static_cast<const c2 *>(a.in) + ch * a.in_stride;
        const int mis = (int)(((reinterpret_cast<unsigned long long>(in) >> 3) + base) & 1);
        src = in + (base - mis);
        return base - mis >= 0 && base - mis + kBulkElems <= a.n_in;
    };
    if (t == 0) mbar_init(&bar, 1);
    __syncthreads();
    const c2 *src = nullptr;
    bool pending = bulk_src(ch, blk, src);
    if (pending && t == 0) bulk_load(F, src, kBulkElems * (unsigned)sizeof(c2), &bar);
    unsigned parity = 0;

    while (ch < a.nchan) {
        const long long base = blk * hop;
        long long nch = ch + dch, nblkpos = blk + dblk;      // this CTA's next task
        if (nblkpos >= nblk) { nblkpos -= nblk; nch++; }
        const c2 *__restrict__ in = static_cast<const c2 *>(a.in) + ch * a.in_stride;
        const c2 *__restrict__ hf = static_cast<const c2 *>(a.hf) + ch * 4096;
        c2 *__restrict__ out = static_cast<c2 *>(a.out) + ch * a.out_stride;
        c2 v[64];
        // ---- forward step 1: thread n2 = t, x[64 n1 + n2] over n1
        if (pending) {
            const int mis = (int)(((reinterpret_cast<unsigned long long>(in) >> 3) + base) & 1);
            mbar_wait(&bar, parity);
            parity ^= 1;
#pragma unroll
            for (int n1 = 0; n1 < 64; n1++) v[rev64(n1)] = F[mis + 64 * n1 + t];
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 64; n1++) {
                const long long g = base + 64 * n1 + t;
                v[rev64(n1)] = g < a.n_in ? __ldcg(in + g) : 0ull;
            }
        }
        dft64_dit<false>(v);                                 // v[k1] = Y[n2 = t][k1]
        step_twiddle<false, false>(v, twa, twb, t);          // * W4096^(n2 k1)
        __syncthreads();                                     // every thread has taken its input out of F
#pragma unroll
        for (int k1 = 0; k1 < 64; k1++) F[k1 * kOs64Stride + t] = v[k1];
        __syncthreads();
        // ---- forward step 2: thread k1 = t, over n2
#pragma unroll
        for (int n2 = 0; n2 < 64; n2++) v[rev64(n2)] = F[t * kOs64Stride + n2];
        dft64_dit<false>(v);                                 // v[k2] = X[k1 + 64 k2]
        // ---- tap spectrum
#pragma unroll
        for (int k2 = 0; k2 < 64; k2++) v[k2] = cmul_p<false>(v[k2], hf[64 * k2 + t]);
        // ---- inverse step 2': same thread, same registers, over k2 -> n2 (register rev64(n2))
        dft64_dif<true>(v);
        step_twiddle<true, true>(v, twa, twb, t);            // * conj W4096^(n2 k1)
        __syncthreads();                                     // step-2 readers are done
#pragma unroll
        for (int n2 = 0; n2 < 64; n2++) F[t * kOs64Stride + n2] = v[rev64(n2)];
        __syncthreads();
        // ---- inverse step 1': thread n2 = t, over k1 -> n1 (register rev64(n1))
#pragma unroll
        for (int k1 = 0; k1 < 64; k1++) v[k1] = F[k1 * kOs64Stride + t];
        __syncthreads();                                     // F is free: fetch the next block into it
        pending = bulk_src(nch, nblkpos, src);
        if (pending && t == 0) bulk_load(F, src, kBulkElems * (unsigned)sizeof(c2), &bar);
        dft64_dif<true>(v);
        // circular result c[i], i = 64 n1 + t; the alias-free part i >= K-1 is y[base + i - (K-1)]
        c2 *o = out + (base - Km1);
        if (base + hop <= a.n_out) {
#pragma unroll
            for (int n1 = 0; n1 < 64; n1++) {
                const int i = 64 * n1 + t;
                if (i >= Km1) __stcg(o + i, v[rev64(n1)]);
            }
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 64; n1++) {
                const int i = 64 * n1 + t;
                if (i >= Km1 && base + i - Km1 < a.n_out) __stcg(o + i, v[rev64(n1)]);
            }
        }
        ch = nch; blk = nblkpos;
    }
}

// ------------------------------------------------- 4096-point variant, persistent form ---
// The same 64 x 64 algorithm as fir_os64_kernel with the four transform groups of an SM gathered in ONE persistent
// 256-thread CTA (group = 2 warps, synchronised on its own named barrier) that keeps, in shared memory, one copy of
//   * the WHOLE step-twiddle table W4096^(j t) (32 KB): a step twiddle is 63 LDS + 63 complex multiplies instead of
//     14 global loads + 112 multiplies (two factors per element), 7 % fewer FMA-pipe instructions;
//   * the tap spectrum of the channel the CTA is working on (32 KB): a CTA-task is (channel, part) -- the channel's
//     blocks part*4 + g, + parts*4, ... for the four groups g -- so the spectrum is staged once per task (once per
//     channel when parts = 1) and the 64 loads per thread and block become LDS; ncu had the global loads as the
//     long_scoreboard / lg_throttle stalls of the one-transform-per-CTA kernel (profiles/r02j_prof_os64p_c5.txt).
// The host picks `parts` so that nchan * parts tasks fill whole rounds of CTAs: 1 for a 1024-channel bank, 8 for the
// 128 channels one of 8 GPUs holds, gridDim.x for a single stream (every CTA one task, the spectrum staged once).
constexpr int kOs64Groups = 4;
__global__ void __launch_bounds__(64 * kOs64Groups, 1) fir_os64p_kernel(const FirOs64Args a)
{
    extern __shared__ __align__(16) c2 os64p_dyn[];            // [4][kOs64SmemElems] tiles | [4096] twiddles | [4096] tap spectrum
    __shared__ __align__(8) unsigned long long bars[kOs64Groups];
    const int g = threadIdx.x >> 6, t = threadIdx.x & 63;
    c2 *F = os64p_dyn + g * kOs64SmemElems;
    c2 *TW = os64p_dyn + kOs64Groups * kOs64SmemElems;
    c2 *HF = TW + 4096;
    unsigned long long *bar = &bars[g];
    auto gsync = [&] { asm volatile("bar.sync %0, 64;" ::"r"(g + 1) : "memory"); };
    const int Km1 = a.K - 1;
    const int hop = 4096 - Km1;
    const long long nblk = (a.n_out + hop - 1) / hop;
    const long long parts = a.parts, ntask = (long long)a.nchan * parts;
    const long long bstep = parts * kOs64Groups;
    auto bulk_src = [&](long long ch, long long blk, const c2 *&src) {
        if (ch >= a.nchan || blk >= nblk) return false;
        const long long base = blk * hop;
        const c2 *in = static_cast<const c2 *>(a.in) + ch * a.in_stride;
        const int mis = (int)(((reinterpret_cast<unsigned long long>(in) >> 3) + base) & 1);
        src = in + (base - mis);
        return base - mis >= 0 && base - mis + kBulkElems <= a.n_in;
    };
    long long task = blockIdx.x;
    if (t == 0) mbar_init(bar, 1);
    gsync();
    const c2 *src = nullptr;
    bool pending = task < ntask && bulk_src(task / parts, (task % parts) * kOs64Groups + g, src);
    if (pending && t == 0) bulk_load(F, src, kBulkElems * (unsigned)sizeof(c2), bar);
    unsigned parity = 0;
    {   // the twiddle table is staged while the first blocks are in flight
        const c2 *__restrict__ twf = static_cast<const c2 *>(a.twf);
        for (int i = threadIdx.x; i < 4096; i += 64 * kOs64Groups) TW[i] = twf[i];
    }
    long long staged = -1;
    for (; task < ntask; task += gridDim.x) {
        const long long ch = task / parts, first = (task - ch * parts) * kOs64Groups + g;
        if (ch != staged) {   // this channel's tap spectrum (the previous task's readers are past the barrier that ends the loop body)
            const c2 *__restrict__ hfg = static_cast<const c2 *>(a.hf) + ch * 4096;
            for (int i = threadIdx.x; i < 4096; i += 64 * kOs64Groups) HF[i] = __ldg(hfg + i);
            staged = ch;
        }
        __syncthreads();
        const c2 *__restrict__ in = static_cast<const c2 *>(a.in) + ch * a.in_stride;
        c2 *__restrict__ out = static_cast<c2 *>(a.out) + ch * a.out_stride;
        for (long long blk = first; blk < nblk; blk += bstep) {
            const long long base = blk * hop;
            c2 v[64];
            if (pending) {
                const int mis = (int)(((reinterpret_cast<unsigned long long>(in) >> 3) + base) & 1);
                mbar_wait(bar, parity);
                parity ^= 1;
#pragma unroll
                for (int n1 = 0; n1 < 64; n1++) v[rev64(n1)] = F[mis + 64 * n1 + t];
            } else {
#pragma unroll
                for (int n1 = 0; n1 < 64; n1++) {
                    const long long gi = base + 64 * n1 + t;
                    v[rev64(n1)] = gi < a.n_in ? __ldcg(in + gi) : 0ull;
                }
            }
            dft64_dit<false>(v);                             // v[k1] = Y[n2 = t][k1]
#pragma unroll
            for (int k1 = 1; k1 < 64; k1++) v[k1] = cmul_p<false>(v[k1], TW[k1 * 64 + t]);   // * W4096^(n2 k1)
            gsync();                                         // every thread of the group has taken its input out of F
#pragma unroll
            for (int k1 = 0; k1 < 64; k1++) F[k1 * kOs64Stride + t] = v[k1];
            gsync();
#pragma unroll
            for (int n2 = 0; n2 < 64; n2++) v[rev64(n2)] = F[t * kOs64Stride + n2];
            dft64_dit<false>(v);                             // v[k2] = X[k1 + 64 k2]
#pragma unroll
            for (int k2 = 0; k2 < 64; k2++) v[k2] = cmul_p<false>(v[k2], HF[64 * k2 + t]);
            dft64_dif<true>(v);
#pragma unroll
            for (int n2 = 1; n2 < 64; n2++) v[rev64(n2)] = cmul_p<true>(v[rev64(n2)], TW[n2 * 64 + t]);   // * conj W4096^(n2 k1)
            gsync();                                         // step-2 readers are done
#pragma unroll
            for (int n2 = 0; n2 < 64; n2++) F[t * kOs64Stride + n2] = v[rev64(n2)];
            gsync();
#pragma unroll
            for (int k1 = 0; k1 < 64; k1++) v[k1] = F[k1 * kOs64Stride + t];
            gsync();                                         // F is free: fetch the group's next block into it
            {
                const bool last = blk + bstep >= nblk;       // next: the same task, or the first block of the CTA's next task
                const long long nt = task + gridDim.x;
                pending = last ? (nt < ntask && bulk_src(nt / parts, (nt % parts) * kOs64Groups + g, src)) : bulk_src(ch, blk + bstep, src);
                if (pending && t == 0) bulk_load(F, src, kBulkElems * (unsigned)sizeof(c2), bar);
            }
            dft64_dif<true>(v);
            c2 *o = out + (base - Km1);
            if (base + hop <= a.n_out) {
#pragma unroll
                for (int n1 = 0; n1 < 64; n1++) {
                    const int i = 64 * n1 + t;
                    if (i >= Km1) __stcg(o + i, v[rev64(n1)]);
                }
            } else {
#pragma unroll
                for (int n1 = 0; n1 < 64; n1++) {
                    const int i = 64 * n1 + t;
                    if (i >= Km1 && base + i - Km1 < a.n_out) __stcg(o + i, v[rev64(n1)]);
                }
            }
        }
        __syncthreads();                                     // every group is done with this task's spectrum
    }
}

// (Round 2 also built this transform on 128 threads x 32 points -- half the register state, 16 warps per SM, the
// radix-4 stage of each 128-point row folded into a 4x redundant read of the exchange tile.  Correct (same tests) and
// 25 % SLOWER than fir_os64_kernel: four warps per transform branch into four different straight-line code paths after
// every barrier, so no two warps share instruction-cache lines (ncu: no_instruction 3.7 stall cycles per issue) and the
// shared-memory pipe is 2.2x as busy.  profiles/r02l_prof_os128_c5.txt; the code was removed.)

constexpr bool kOs32PartialTwiddles = false;   // fir_os32_kernel: measured no gain on B200 (headline 269 vs 272 Gsamples/s); the resampler keeps them

// v[slot(k)] *= W1024^(k t) (CONJ: conjugate) for k = 1..31 from TEN loaded twiddles instead of 31:
// k = 4a + b, W^(kt) = W^(4a t) W^(b t).  The 21 extra complex multiplies cost FMA issue slots, the 21
// saved loads were a fifth of the kernel's L1/shared data-pipe traffic, which is the busier pipe
// (profiles/r01c_prof_os32_headline.txt).  One more rounding per twiddled element (~1e-7 relative).
template <bool CONJ, bool SLOT_REV>
__device__ __forceinline__ void twiddle32(c2 (&v)[32], const c2 *__restrict__ tw, const int t)
{
    c2 A[8], B[4];
#pragma unroll
    for (int a = 1; a < 8; a++) A[a] = tw[(4 * a) * 32 + t];
#pragma unroll
    for (int b = 1; b < 4; b++) B[b] = tw[b * 32 + t];
#pragma unroll
    for (int k = 1; k < 32; k++) {
        const int a = k >> 2, b = k & 3, r = SLOT_REV ? rev32(k) : k;
        if (a) v[r] = cmul_p<CONJ>(v[r], A[a]);
        if (b) v[r] = cmul_p<CONJ>(v[r], B[b]);
    }
}

// ---------------------------------------------------------------- 1024-point variant ---
// Same algorithm on 1024 = 32 x 32: ONE WARP per transform, 32 points (64 registers) per
// thread, exchanges through a per-warp shared-memory tile with __syncwarp() only.  Less
// register state per thread => ~2.5x the resident warps of the 4096-point kernel, which is
// what keeps the FMA pipe fed; the price is a shorter hop (1024 - (K-1)), so it is used for
// the shorter tap counts (fir_os_launch).
struct FirOs32Args {
    const void *in;
    void *out;
    const void *hf;     // [nchan][1024] spectrum of the taps / 1024
    const void *tw;     // [17][32] signed step twiddles W1024^(r s(t)) (os32_signed_twiddles; row 0 unused)
    long long n_in, n_out;             // per channel
    long long in_stride, out_stride;   // elements between consecutive channels (filter bank)
    int nchan;
    int K;
    int spread;         // TABS form: warp-major task order (launches smaller than one wave of warps)
    int pdl;            // TABS form: launched with programmatic stream serialization (prologue before griddepcontrol.wait)
};

// TABS: one persistent CTA per SM whose warps share ONE copy of the tap spectrum and the twiddles in (dynamic) shared
// memory -- single-channel streams only (a filter bank has one spectrum per channel)
// EARLY (TABS form): every warp also owns a landing buffer, so the bulk copy of its NEXT block is issued as soon as the
// current block sits in registers and has the whole block's compute time to arrive (instead of the last register pass).
// Lanes and register indices are signed (os32_signed): lane t >= 16 takes the elements 32 m + t - 32 (mod 1024) of the
// block, and multiplies bin t - 32 + 32 k2 (mod 1024) of the spectrum, so a step twiddle is 16 loads from the 16-row
// table instead of 31 from the 32-row one.  Only row 0 (m = 0, k2 = 0) wraps, to the end of the block.
// (PT is not read: the partial twiddles measured no gain here; the parameter stays in the kernel's name.)
constexpr int kOs32Landing = 1032;   // c2 elements per landing buffer (1026 used)
constexpr int kOs32TabElems = 1024 + 512;   // TABS: tap spectrum, then rows 1..16 of the signed twiddles
template <int WARPS, int MINB, bool TABS = false, bool PT = kOs32PartialTwiddles, bool EARLY = false>
__global__ void __launch_bounds__(32 * WARPS, MINB) fir_os32_kernel(const FirOs32Args a)
{
    extern __shared__ __align__(16) c2 os32_dyn[];
    __shared__ __align__(16) c2 Fs[TABS ? 1 : WARPS][TABS ? 1 : kOs32SmemElems];
    __shared__ __align__(8) unsigned long long bars[WARPS];
    const int t = threadIdx.x & 31, w = threadIdx.x >> 5;
    // the lane's signed index and its element in row 0 (t, or 992 + t for the lanes that wrap)
    const int so = os32_signed(t), s0 = so & 1023;
    c2 *F = TABS ? os32_dyn + w * kOs32SmemElems : Fs[TABS ? 0 : w];
    unsigned long long *bar = &bars[w];
    const c2 *__restrict__ tw = static_cast<const c2 *>(a.tw);
    const c2 *__restrict__ hf_tab = nullptr;
    c2 *Lb = F;                                               // where the bulk copy lands
    if constexpr (TABS && EARLY) Lb = os32_dyn + WARPS * kOs32SmemElems + kOs32TabElems + w * kOs32Landing;
    const int Km1 = a.K - 1;
    const int hop = 1024 - Km1;
    const long long nblk = (a.n_out + hop - 1) / hop;
    // tasks = (channel, block), channel-major, taken grid-stride by the warps (see fir_os64_kernel).  A launch with
    // fewer tasks than resident warps (a small work() buffer) is spread warp-major, so that every SM gets a block
    // before any SM gets a second one.
    const long long tstep = (long long)gridDim.x * WARPS, dch = tstep / nblk, dblk = tstep - dch * nblk;
    const long long task0 = a.spread ? (long long)w * gridDim.x + blockIdx.x : (long long)blockIdx.x * WARPS + w;
    long long ch = task0 / nblk, blk = task0 - ch * nblk;
    // the warp's next block is fetched into its exchange tile by one bulk copy while the warp is
    // in its last register pass; edge blocks use guarded loads
    constexpr int kBulk = 1026;
    auto bulk_src = [&](long long ch, long long blk, const c2 *&src) {
        if (ch >= a.nchan) return false;
        const long long base = blk * hop;
        const c2 *in = static_cast<const c2 *>(a.in) + ch * a.in_stride;
        const int mis = (int)(((reinterpret_cast<unsigned long long>(in) >> 3) + base) & 1);
        src = in + (base - mis);
        return base - mis >= 0 && base - mis + kBulk <= a.n_in;
    };
    if (t == 0) mbar_init(bar, 1);
    __syncwarp();
    const c2 *src = nullptr;
    bool pending = bulk_src(ch, blk, src);
    unsigned parity = 0;
    if constexpr (TABS) {
        // Programmatic dependent launch (the host sets the attribute on this form, B200C_PDL=0 turns it off): the NEXT launch
        // in the stream may start its CTAs on the SMs this one has left, and this launch ran its own prologue -- barrier
        // init, 12 KB of tables -- while its predecessor was still finishing; only here, before the first access to stream
        // data, does it wait for the predecessor to complete and flush.  Back-to-back work() calls on small buffers pay the
        // launch latency and the prologue once, not per call (DESIGN 4.10).  Both instructions are no-ops in a plain launch.
        asm volatile("griddepcontrol.launch_dependents;");
        c2 *tab = os32_dyn + WARPS * kOs32SmemElems;
        const c2 *__restrict__ hf0 = static_cast<const c2 *>(a.hf);
        // every load of the 12 KB is issued before the first store: one memory latency, not one per element a thread
        // copies (a launch of one block per warp waits for this prologue)
        auto stage = [&] {
            constexpr int kStep = 32 * WARPS, kIt = (kOs32TabElems + kStep - 1) / kStep;
            c2 r[kIt];
#pragma unroll
            for (int j = 0; j < kIt; j++) {
                const int i = (int)threadIdx.x + j * kStep;
                if (i < kOs32TabElems) r[j] = i < 1024 ? hf0[i] : tw[i - 1024 + 32];
            }
#pragma unroll
            for (int j = 0; j < kIt; j++) {
                const int i = (int)threadIdx.x + j * kStep;
                if (i < kOs32TabElems) tab[i] = r[j];
            }
        };
        if (a.pdl) {
            stage();
            asm volatile("griddepcontrol.wait;" ::: "memory");
            if (pending && t == 0) bulk_load(Lb, src, kBulk * (unsigned)sizeof(c2), bar);
        } else {
            // plain launch: the tables are staged while the first block is in flight
            if (pending && t == 0) bulk_load(Lb, src, kBulk * (unsigned)sizeof(c2), bar);
            stage();
        }
        __syncthreads();
        hf_tab = tab; tw = tab + 1024 - 32;                   // tw[32 r + t], r = 1..16
    } else {
        if (pending && t == 0) bulk_load(Lb, src, kBulk * (unsigned)sizeof(c2), bar);
    }
    const c2 *__restrict__ twl = tw + t;
    while (ch < a.nchan) {
        const long long base = blk * hop;
        long long nch = ch + dch, nblkpos = blk + dblk;      // this warp's next task
        if (nblkpos >= nblk) { nblkpos -= nblk; nch++; }
        const c2 *__restrict__ in = static_cast<const c2 *>(a.in) + ch * a.in_stride;
        const c2 *__restrict__ hf = TABS ? hf_tab : static_cast<const c2 *>(a.hf) + ch * 1024;
        c2 *__restrict__ out = static_cast<c2 *>(a.out) + ch * a.out_stride;
        c2 v[32];
        // register rev32(n1) of lane t: element 32 n1 + s(t) of the block (mod 1024)
        if (pending) {
            const int mis = (int)(((reinterpret_cast<unsigned long long>(in) >> 3) + base) & 1);
            mbar_wait(bar, parity);
            parity ^= 1;
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) v[rev32(n1)] = Lb[mis + (n1 ? 32 * n1 + so : s0)];
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) {
                const long long g = n1 ? base + so + 32 * n1 : base + s0;
                v[rev32(n1)] = g < a.n_in ? __ldcg(in + g) : 0ull;
            }
        }
        if constexpr (TABS && EARLY) {
            __syncwarp();                                    // the landing buffer is in registers: fetch the next block now
            pending = bulk_src(nch, nblkpos, src);
            if (pending && t == 0) bulk_load(Lb, src, kBulk * (unsigned)sizeof(c2), bar);
        }
        dft32_dit<false>(v);
#pragma unroll
        for (int k1 = 1; k1 < 32; k1++) v[k1] = os32_step<false>(v[k1], twl, k1);   // * W1024^(s(k1) s(t))
        __syncwarp();
#pragma unroll
        for (int k1 = 0; k1 < 32; k1++) F[k1 * kOs32Stride + t] = v[k1];
        __syncwarp();
#pragma unroll
        for (int n2 = 0; n2 < 32; n2++) v[rev32(n2)] = F[t * kOs32Stride + n2];
        dft32_dit<false>(v);                                 // v[k2] = X[s(t) + 32 k2]
#pragma unroll
        for (int k2 = 0; k2 < 32; k2++) v[k2] = cmul_p<false>(v[k2], hf[k2 ? 32 * k2 + so : s0]);
        dft32_dif<true>(v);
#pragma unroll
        for (int n2 = 1; n2 < 32; n2++) v[rev32(n2)] = os32_step<true>(v[rev32(n2)], twl, n2);   // * conj W1024^(s(n2) s(t))
        __syncwarp();
#pragma unroll
        for (int n2 = 0; n2 < 32; n2++) F[t * kOs32Stride + n2] = v[rev32(n2)];
        __syncwarp();
#pragma unroll
        for (int k1 = 0; k1 < 32; k1++) v[k1] = F[k1 * kOs32Stride + t];
        if constexpr (!(TABS && EARLY)) {
            __syncwarp();                                    // the tile is free: fetch the next block into it
            pending = bulk_src(nch, nblkpos, src);
            if (pending && t == 0) bulk_load(F, src, kBulk * (unsigned)sizeof(c2), bar);
        }
        dft32_dif<true>(v);
        // register rev32(n1) of lane t: circular result c[i], i = 32 n1 + s(t) (mod 1024); i >= K-1 is y[base + i - (K-1)]
        c2 *o = out + (base - Km1), *ol = o + so;
        if (base + hop <= a.n_out) {
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) {
                const int i = n1 ? 32 * n1 + so : s0;
                if (i >= Km1) __stcg(n1 ? ol + 32 * n1 : o + s0, v[rev32(n1)]);
            }
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) {
                const int i = n1 ? 32 * n1 + so : s0;
                if (i >= Km1 && base + i - Km1 < a.n_out) __stcg(n1 ? ol + 32 * n1 : o + s0, v[rev32(n1)]);
            }
        }
        ch = nch; blk = nblkpos;
    }
}

// ------------------------------------- spectral resampler, interpolation 3 / decimation 2 ---
// The polyphase nest (filter/FIRFilter.cpp:286-302) for L = 3, M = 2 as ONE forward and ONE inverse
// transform per block instead of M + L transforms of 1024 points: with u the zero-stuffed input
// (u[3 n] = x[n]) and v = h * u at the high rate, the reference's outputs are y[m] = v[2 m + 1 + 3 (K - 1)].
// On a block of 1024 inputs, DFT_3072(u)[k] = X[k mod 1024] (X = DFT_1024 of the block), V = X . H, and
// keeping every second sample of v (phase 1) folds the spectrum:
//   W[kk] = X[kk mod 1024] H'[kk] + X[(kk + 512) mod 1024] H'[kk + 1536],  kk < 1536,
//   H'[k] = DFT_3072(h)[k] exp(2 pi i k / 3072) / 3072,            w[m'] = sum_kk W[kk] exp(2 pi i kk m' / 1536).
// Outputs m' >= m0 = ceil((ntaps - 2) / 2) (rounded up to a multiple of 3) are alias free: a block yields
// 1536 - m0 outputs from (1536 - m0) 2 / 3 new inputs (C3: 1407 from 938).
// One warp per block, as fir_os32_kernel.  After the forward transform thread t holds X[t + 32 k2]; every
// bin of W it needs is then one of ITS registers (both X indices are congruent to kk mod 32), so the fold
// is register arithmetic: thread t forms W[t + 32 c], c < 48.  1536 = 32 x 48: the thread transforms its
// 48 bins (three 16-point transforms, constant twiddles, sixteen 3-point butterflies), twiddles by
// exp(2 pi i t n2 / 1536), and after ONE exchange the 48 rows n2 are 32-point transforms over t: lane n2
// takes row n2, lanes 0..15 also row 32 + n2 (the second round runs half empty: 1.5 rows per lane).
// Row n2 gives w[48 n1 + n2]: for every n1 the warp stores 32 (16) consecutive outputs.
B200C_HD constexpr float cos48(int e)
{
    constexpr float t[48] = {
        1.0f, 0.9914448857307434f, 0.9659258127212524f, 0.9238795042037964f, 0.8660253882408142f, 0.7933533191680908f,
        0.7071067690849304f, 0.6087614297866821f, 0.5f, 0.3826834261417389f, 0.258819043636322f, 0.13052618503570557f, 0.0f,
        -0.13052618503570557f, -0.258819043636322f, -0.3826834261417389f, -0.5f, -0.6087614297866821f, -0.7071067690849304f,
        -0.7933533191680908f, -0.8660253882408142f, -0.9238795042037964f, -0.9659258127212524f, -0.9914448857307434f, -1.0f,
        -0.9914448857307434f, -0.9659258127212524f, -0.9238795042037964f, -0.8660253882408142f, -0.7933533191680908f,
        -0.7071067690849304f, -0.6087614297866821f, -0.5f, -0.3826834261417389f, -0.258819043636322f, -0.13052618503570557f, 0.0f,
        0.13052618503570557f, 0.258819043636322f, 0.3826834261417389f, 0.5f, 0.6087614297866821f, 0.7071067690849304f,
        0.7933533191680908f, 0.8660253882408142f, 0.9238795042037964f, 0.9659258127212524f, 0.9914448857307434f};
    return t[e % 48];
}
B200C_HD constexpr float sin48(int e) { return cos48(e + 36); }   // sin(x) = cos(x - pi/2)

// 16-point DFT in place, decimation in frequency: input n in x[n], output k in x[rev16(k)]
B200C_HD constexpr int rev16(int k) { return 4 * (k & 3) + (k >> 2); }
template <bool INV> B200C_HD void dft16_dif(c2 (&x)[16])
{
#pragma unroll
    for (int k = 0; k < 4; k++) {
        dft4_p<INV>(x[k], x[k + 4], x[k + 8], x[k + 12]);
        x[k + 4] = mul_w64<INV>(x[k + 4], 4 * k);      // W16^k
        x[k + 8] = mul_w64<INV>(x[k + 8], 8 * k);
        x[k + 12] = mul_w64<INV>(x[k + 12], 12 * k);
    }
#pragma unroll
    for (int g = 0; g < 4; g++) dft4_p<INV>(x[4 * g], x[4 * g + 1], x[4 * g + 2], x[4 * g + 3]);
}

// acc + f * w
B200C_HD c2 cmul_acc(c2 f, c2 w, c2 acc)
{
    float fx, fy, wx, wy;
    upk(f, fx, fy); upk(w, wx, wy);
    return fma2(f, pk(wx, wx), fma2(pk(-fy, fx), pk(wy, wy), acc));
}

struct FirOsX32Args {
    const void *in;
    void *out;
    const void *hx;     // [3072] H'
    const void *tw;     // [32][32] W1024^(j t)
    const void *tw3;    // [48][32] exp(+2 pi i n2 t / 1536)
    long long n_in, n_out;
    long long p0;       // input element at which block 0's window starts (<= 0: zeros in front)
    int m0;             // first alias-free output of a block
    int pdl;            // launched with programmatic stream serialization (see fir_os32_kernel)
};
constexpr int kX32Rows = 48, kX32SmemElems = kX32Rows * kOs32Stride;

// WARPS == 1: one warp per CTA, MINB CTAs per SM, tables read through L1.  WARPS > 1: one persistent CTA per SM
// whose warps share ONE copy of the tables (tap spectrum 24 KB, step twiddles 12 KB + 8 KB) in shared memory.
constexpr int kX32TabElems = 3072 + 1536 + 1024;
// SPLIT: the 16 rows left for the second inverse round (rows 32..47 on 32 lanes) are transformed by lane PAIRS instead
// of by lanes 0..15 alone: lane (tt, h) takes the inputs k1 = 2 j + h of row 32 + tt through a 16-point transform, the odd
// half is twiddled, one shuffle exchange (xor 16) combines them -- w[m] = S0[m] + W^m S1[m] on h = 0, w[m + 16] = S0[m] -
// W^m S1[m] on h = 1.  126 packed instructions on all lanes instead of 222 on half of them.
// (Round 2 also built 8- and 9-warp forms with a landing buffer per warp, compact twiddle tables and an interleaved tap
// spectrum read with 128-bit loads: 3 % and 17 % SLOWER than this 12-warp form -- profiles/r02_osx_variants.txt -- removed.)
template <int WARPS, int MINB, bool PT = false, bool SPLIT = false>
__global__ void __launch_bounds__(32 * WARPS, MINB) fir_os32x_kernel(const FirOsX32Args a)
{
    extern __shared__ __align__(16) c2 x32_smem[];
    __shared__ __align__(8) unsigned long long bars[WARPS];
    const int t = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const c2 *__restrict__ tw = static_cast<const c2 *>(a.tw);
    const c2 *__restrict__ tw3 = static_cast<const c2 *>(a.tw3);
    const c2 *__restrict__ hx = static_cast<const c2 *>(a.hx);
    c2 *F = x32_smem + wp * kX32SmemElems;
    c2 *const Lb = F;                                            // where the bulk copy lands: the exchange tile
    unsigned long long &bar = bars[wp];
    const c2 *__restrict__ in = static_cast<const c2 *>(a.in);
    c2 *__restrict__ out = static_cast<c2 *>(a.out);
    const int m0 = a.m0, hop_out = 1536 - m0, hop_in = hop_out / 3 * 2;
    const long long nblk = (a.n_out + hop_out - 1) / hop_out;
    constexpr int kBulk = 1026;
    auto bulk_src = [&](long long blk, const c2 *&src) {
        if (blk >= nblk) return false;
        const long long P = a.p0 + blk * hop_in;
        const int mis = (int)(((reinterpret_cast<unsigned long long>(in) >> 3) + (unsigned long long)P) & 1);
        src = in + (P - mis);
        return P - mis >= 0 && P - mis + kBulk <= a.n_in;
    };
    if (t == 0) mbar_init(&bar, 1);
    __syncwarp();
    long long blk = (long long)blockIdx.x * WARPS + wp;
    const long long bstep = (long long)gridDim.x * WARPS;
    const c2 *src = nullptr;
    bool pending = bulk_src(blk, src);
    unsigned parity = 0;
    if constexpr (WARPS > 1) {
        // dependent launch as in fir_os32_kernel: with a.pdl the 44 KB of tables are staged while the predecessor in the stream
        // is still running and stream data is touched only after griddepcontrol.wait; a plain launch stages them while its
        // first block is in flight
        asm volatile("griddepcontrol.launch_dependents;");
        c2 *tab = x32_smem + WARPS * kX32SmemElems;
        auto stage = [&] {
            for (int i = threadIdx.x; i < 3072; i += 32 * WARPS) tab[i] = hx[i];
            for (int i = threadIdx.x; i < 1536; i += 32 * WARPS) tab[3072 + i] = tw3[i];
            for (int i = threadIdx.x; i < 1024; i += 32 * WARPS) tab[3072 + 1536 + i] = tw[i];
        };
        if (a.pdl) {
            stage();
            asm volatile("griddepcontrol.wait;" ::: "memory");
            if (pending && t == 0) bulk_load(Lb, src, kBulk * (unsigned)sizeof(c2), &bar);
        } else {
            if (pending && t == 0) bulk_load(Lb, src, kBulk * (unsigned)sizeof(c2), &bar);
            stage();
        }
        __syncthreads();
        hx = tab; tw3 = tab + 3072; tw = tab + 3072 + 1536;
    } else {
        if (pending && t == 0) bulk_load(Lb, src, kBulk * (unsigned)sizeof(c2), &bar);
    }
    for (; blk < nblk; blk += bstep) {
        const long long P = a.p0 + blk * hop_in;
        c2 v[32];
        if (pending) {
            const int mis = (int)(((reinterpret_cast<unsigned long long>(in) >> 3) + (unsigned long long)P) & 1);
            mbar_wait(&bar, parity);
            parity ^= 1;
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) v[rev32(n1)] = Lb[mis + 32 * n1 + t];
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) {
                const long long g = P + 32 * n1 + t;
                v[rev32(n1)] = (g >= 0 && g < a.n_in) ? __ldcg(in + g) : 0ull;
            }
        }
        // forward 1024 = 32 x 32 (as fir_os32_kernel): thread t ends with X[t + 32 k2] in v[k2]
        dft32_dit<false>(v);
        if constexpr (PT) twiddle32<false, false>(v, tw, t);   // ten loaded + 21 computed twiddles
        else {
#pragma unroll
            for (int k1 = 1; k1 < 32; k1++) v[k1] = cmul_p<false>(v[k1], tw[k1 * 32 + t]);
        }
        __syncwarp();
#pragma unroll
        for (int k1 = 0; k1 < 32; k1++) F[k1 * kOs32Stride + t] = v[k1];
        __syncwarp();
#pragma unroll
        for (int n2 = 0; n2 < 32; n2++) v[rev32(n2)] = F[t * kOs32Stride + n2];
        dft32_dit<false>(v);
        // replicate x taps, fold: W[t + 32 c] in s[c % 3][c / 3].  Bins c, c + 16, c + 32 (c < 16) are the three
        // combinations of the SAME two inputs X[c], X[c + 16], which retire with them: at most 48 values stay
        // live, which leaves registers for the tap-spectrum loads to run ahead.
        c2 s[3][16];
#pragma unroll
        for (int c = 0; c < 16; c++) {
            const c2 xa = v[c], xb = v[c + 16];
            const c2 h0 = hx[32 * c + t], g0 = hx[1536 + 32 * c + t];
            const c2 h1 = hx[32 * (c + 16) + t], g1 = hx[1536 + 32 * (c + 16) + t];
            const c2 h2 = hx[32 * (c + 32) + t], g2 = hx[1536 + 32 * (c + 32) + t];
            s[c % 3][c / 3] = cmul_acc(xb, g0, cmul_p<false>(xa, h0));
            s[(c + 16) % 3][(c + 16) / 3] = cmul_acc(xa, g1, cmul_p<false>(xb, h1));
            s[(c + 32) % 3][(c + 32) / 3] = cmul_acc(xb, g2, cmul_p<false>(xa, h2));
        }
        // 48-point inverse transform of the thread's bins: c = 3 c2 + c1, n2 = 16 v1 + v2
#pragma unroll
        for (int c1 = 0; c1 < 3; c1++) dft16_dif<true>(s[c1]);
        __syncwarp();
        // step twiddles exp(2 pi i t n2 / 1536), n2 = 16 v1 + v2: PT loads the 15 + 2 factors and multiplies
        c2 twb1 = 0, twb2 = 0;
        if constexpr (PT) { twb1 = tw3[16 * 32 + t]; twb2 = tw3[32 * 32 + t]; }
#pragma unroll
        for (int v2 = 0; v2 < 16; v2++) {
            const int r = rev16(v2);
            const c2 a0 = s[0][r];
            const c2 a1 = v2 ? cmul_s(s[1][r], cos48(v2), sin48(v2)) : s[1][r];             // exp(+2 pi i v2 / 48)
            const c2 a2 = v2 ? cmul_s(s[2][r], cos48(2 * v2), sin48(2 * v2)) : s[2][r];
            const c2 t1 = add2(a1, a2);
            const c2 t2 = fma2(t1, pk(-0.5f, -0.5f), a0);
            const c2 t3 = rot_p<true>(mul2(sub2(a1, a2), pk(0.8660254037844386f, 0.8660254037844386f)));   // +i sin(2 pi / 3) (a1 - a2)
            const c2 y0 = add2(a0, t1), y1 = add2(t2, t3), y2 = sub2(t2, t3);
            // step twiddle exp(2 pi i t n2 / 1536), then row n2 of the exchange tile
            if constexpr (PT) {
                const c2 wa = v2 ? tw3[v2 * 32 + t] : pk(1.f, 0.f);
                F[v2 * kOs32Stride + t] = v2 ? cmul_p<false>(y0, wa) : y0;
                F[(16 + v2) * kOs32Stride + t] = cmul_p<false>(y1, v2 ? cmul_p<false>(wa, twb1) : twb1);
                F[(32 + v2) * kOs32Stride + t] = cmul_p<false>(y2, v2 ? cmul_p<false>(wa, twb2) : twb2);
            } else {
                F[v2 * kOs32Stride + t] = v2 ? cmul_p<false>(y0, tw3[v2 * 32 + t]) : y0;
                F[(16 + v2) * kOs32Stride + t] = cmul_p<false>(y1, tw3[(16 + v2) * 32 + t]);
                F[(32 + v2) * kOs32Stride + t] = cmul_p<false>(y2, tw3[(32 + v2) * 32 + t]);
            }
        }
        __syncwarp();
        const long long mbase = blk * hop_out - m0;          // global output index of w[0]
        const bool whole = (blk + 1) * (long long)hop_out <= a.n_out;
        c2 *const o = out + mbase + t;                       // w[48 n1 + t] goes to o[48 n1]
        const int d0 = t - m0;                               // w[m'] is kept when m' >= m0
        const int left = whole ? 0x7fffffff : (int)(a.n_out - mbase) - t;   // ... and inside the output: 48 n1 (+ 32) < left
        // round 1: lane t transforms row n2 = t -> w[48 n1 + t]
#pragma unroll
        for (int k1 = 0; k1 < 32; k1++) v[rev32(k1)] = F[t * kOs32Stride + k1];
        if constexpr (SPLIT) {
            // rows 0..31 are in registers and the copy lands in elements [0, 1026) only -- below row 32 (element 1056),
            // which the second round still reads: the next block can be fetched now, a round and a half ahead
            __syncwarp();
            pending = bulk_src(blk + bstep, src);
            if (pending && t == 0) bulk_load(F, src, kBulk * (unsigned)sizeof(c2), &bar);
        }
        dft32_dit<true>(v);
        if (whole) {
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++)
                if (d0 + 48 * n1 >= 0) __stcg(o + 48 * n1, v[n1]);
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++)
                if (d0 + 48 * n1 >= 0 && 48 * n1 < left) __stcg(o + 48 * n1, v[n1]);
        }
        if constexpr (SPLIT) {
            // round 2 by lane pairs: lane (tt, h) -> sub-transform over k1 = 2 j + h of row 32 + tt
            const int tt = t & 15, h = t >> 4;
            c2 x[16];
#pragma unroll
            for (int j = 0; j < 16; j++) x[j] = F[(32 + tt) * kOs32Stride + 2 * j + h];
            __syncwarp();                                    // (the next block's copy was issued after the first round's reads)
            dft16_dif<true>(x);                              // S_h[m] in x[rev16(m)]
            c2 *const o2 = out + mbase + tt + 32 + 48 * 16 * h;   // w[48 (m + 16 h) + 32 + tt]
            const int d2 = tt - m0 + 32 + 48 * 16 * h;
            const int left2 = whole ? 0x7fffffff : (int)(a.n_out - mbase) - tt - 32 - 48 * 16 * h;
#pragma unroll
            for (int m = 0; m < 16; m++) {
                const c2 mine = h ? mul_w64<true>(x[rev16(m)], 2 * m) : x[rev16(m)];     // h = 1: e^{+2 pi i m / 32} S1[m]
                const c2 other = __shfl_xor_sync(0xffffffffu, mine, 16);
                const c2 y = h ? sub2(other, mine) : add2(mine, other);
                if (d2 + 48 * m >= 0 && 48 * m < left2) __stcg(o2 + 48 * m, y);
            }
            continue;
        }
        // round 2: lanes 0..15 transform rows 32 + t -> w[48 n1 + 32 + t]
        if (t < 16) {
#pragma unroll
            for (int k1 = 0; k1 < 32; k1++) v[rev32(k1)] = F[(32 + t) * kOs32Stride + k1];
        }
        __syncwarp();                                        // the tile is free: fetch the next block into it
        pending = bulk_src(blk + bstep, src);
        if (pending && t == 0) bulk_load(F, src, kBulk * (unsigned)sizeof(c2), &bar);
        if (t < 16) {
            dft32_dit<true>(v);
            if (whole) {
#pragma unroll
                for (int n1 = 0; n1 < 32; n1++)
                    if (d0 + 48 * n1 + 32 >= 0) __stcg(o + 48 * n1 + 32, v[n1]);
            } else {
#pragma unroll
                for (int n1 = 0; n1 < 32; n1++)
                    if (d0 + 48 * n1 + 32 >= 0 && 48 * n1 + 32 < left) __stcg(o + 48 * n1 + 32, v[n1]);
            }
        }
    }
}

// ------------------------------------------------------- real float32 data, L = M = 1 ---
// float32 streams carry REAL taps only (filter/FIRFilter.cpp:373-376), so the filter is real and
// linear: two consecutive stream blocks ride in one complex transform, z = x_A + i x_B gives
// Re = y_A, Im = y_B.  Same warp-per-transform structure as fir_os32_kernel; the two blocks overlap in
// the input (hop < 1024), so ONE bulk copy of hop + 1024 floats feeds both.
struct FirOs32RArgs {
    const float *in;
    float *out;
    const void *hf;     // [1024] spectrum of the taps / 1024
    const void *tw;     // [32][32] W1024^(j*t)
    long long n_in, n_out;
    int K;
};

// WARPS == 1: one warp per CTA, MINB CTAs per SM, tables through L1.  WARPS > 1: one persistent CTA per SM whose warps
// share one copy of the tap spectrum and the twiddles in shared memory (as fir_os32_kernel's TABS form).
template <int WARPS, int MINB, bool EARLY = false>
__global__ void __launch_bounds__(32 * WARPS, MINB) fir_os32r_kernel(const FirOs32RArgs a)
{
    extern __shared__ __align__(16) c2 os32r_dyn[];
    __shared__ __align__(8) unsigned long long bars[WARPS];
    const int t = threadIdx.x & 31, wp = threadIdx.x >> 5;
    c2 *F = os32r_dyn + wp * kOs32SmemElems;
    // EARLY (WARPS > 1): a landing buffer per warp, the next pair is fetched while this one is computed
    c2 *Lb = (WARPS > 1 && EARLY) ? os32r_dyn + WARPS * kOs32SmemElems + 2048 + wp * kOs32Landing : F;
    unsigned long long &bar = bars[wp];
    const float *Ff = reinterpret_cast<const float *>(Lb);
    const c2 *__restrict__ tw = static_cast<const c2 *>(a.tw);
    const c2 *__restrict__ hf = static_cast<const c2 *>(a.hf);
    if constexpr (WARPS > 1) {
        c2 *tab = os32r_dyn + WARPS * kOs32SmemElems;
        for (int i = threadIdx.x; i < 1024; i += 32 * WARPS) { tab[i] = hf[i]; tab[1024 + i] = tw[i]; }
        __syncthreads();
        hf = tab; tw = tab + 1024;
    }
    const int Km1 = a.K - 1, hop = 1024 - Km1;
    const long long npair = (a.n_out + 2LL * hop - 1) / (2LL * hop);
    // pair bp: block A = inputs [base, base + 1024), block B = [base + hop, base + hop + 1024), base = 2 hop bp
    auto bulk_src = [&](long long bp, const float *&src, int &mis, unsigned &bytes) {
        if (bp >= npair) return false;
        const long long base = bp * 2LL * hop;
        mis = (int)(((reinterpret_cast<unsigned long long>(a.in) >> 2) + base) & 3);
        const int count = (mis + hop + 1024 + 3) & ~3;       // floats, a multiple of 16 bytes, <= 2052
        src = a.in + (base - mis);
        bytes = (unsigned)count * 4u;
        return base - mis >= 0 && base - mis + count <= a.n_in;
    };
    if (t == 0) mbar_init(&bar, 1);
    __syncwarp();
    long long bp = (long long)blockIdx.x * WARPS + wp;
    const float *src = nullptr;
    int mis = 0, mis_next = 0;
    unsigned bytes = 0;
    bool pending = bulk_src(bp, src, mis, bytes);
    if (pending && t == 0) bulk_load(Lb, src, bytes, &bar);
    unsigned parity = 0;
    while (bp < npair) {
        const long long base = bp * 2LL * hop, nbp = bp + (long long)gridDim.x * WARPS;
        c2 v[32];
        if (pending) {
            mbar_wait(&bar, parity);
            parity ^= 1;
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) v[rev32(n1)] = pk(Ff[mis + 32 * n1 + t], Ff[mis + hop + 32 * n1 + t]);
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) {
                const long long ga = base + 32 * n1 + t, gb = ga + hop;
                v[rev32(n1)] = pk(ga < a.n_in ? __ldg(a.in + ga) : 0.f, gb < a.n_in ? __ldg(a.in + gb) : 0.f);
            }
        }
        if constexpr (WARPS > 1 && EARLY) {
            __syncwarp();                                    // the landing buffer is in registers: fetch the next pair now
            pending = bulk_src(nbp, src, mis_next, bytes);
            if (pending && t == 0) bulk_load(Lb, src, bytes, &bar);
        }
        dft32_dit<false>(v);
#pragma unroll
        for (int k1 = 1; k1 < 32; k1++) v[k1] = cmul_p<false>(v[k1], tw[k1 * 32 + t]);
        __syncwarp();
#pragma unroll
        for (int k1 = 0; k1 < 32; k1++) F[k1 * kOs32Stride + t] = v[k1];
        __syncwarp();
#pragma unroll
        for (int n2 = 0; n2 < 32; n2++) v[rev32(n2)] = F[t * kOs32Stride + n2];
        dft32_dit<false>(v);
#pragma unroll
        for (int k2 = 0; k2 < 32; k2++) v[k2] = cmul_p<false>(v[k2], hf[32 * k2 + t]);
        dft32_dif<true>(v);
#pragma unroll
        for (int n2 = 1; n2 < 32; n2++) v[rev32(n2)] = cmul_p<true>(v[rev32(n2)], tw[n2 * 32 + t]);
        __syncwarp();
#pragma unroll
        for (int n2 = 0; n2 < 32; n2++) F[t * kOs32Stride + n2] = v[rev32(n2)];
        __syncwarp();
#pragma unroll
        for (int k1 = 0; k1 < 32; k1++) v[k1] = F[k1 * kOs32Stride + t];
        if constexpr (!(WARPS > 1 && EARLY)) {
            __syncwarp();                                    // the tile is free: fetch the next pair into it
            pending = bulk_src(nbp, src, mis_next, bytes);
            if (pending && t == 0) bulk_load(F, src, bytes, &bar);
        }
        dft32_dif<true>(v);
        // circular results c[i], i = 32 n1 + t >= K-1: Re -> y[base + i - (K-1)], Im -> y[base + hop + i - (K-1)]
        float *oa = a.out + (base - Km1), *ob = oa + hop;
        if (base + 2LL * hop <= a.n_out) {
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) {
                const int i = 32 * n1 + t;
                float ya, yb;
                upk(v[rev32(n1)], ya, yb);
                if (i >= Km1) { __stcg(oa + i, ya); __stcg(ob + i, yb); }
            }
        } else {
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) {
                const int i = 32 * n1 + t;
                float ya, yb;
                upk(v[rev32(n1)], ya, yb);
                if (i >= Km1 && base + i - Km1 < a.n_out) __stcg(oa + i, ya);
                if (i >= Km1 && base + hop + i - Km1 < a.n_out) __stcg(ob + i, yb);
            }
        }
        bp = nbp; mis = mis_next;
    }
}

// ------------------------------------------------- polyphase / real-data generalisation ---
// The reference's resampling nest (filter/FIRFilter.cpp:286-302) in polyphase form (fir.hpp):
//   y[q L + p] = sum_e sum_a g_{p,e}[a] * x_e[q + a],   x_e[i] = x[i M + e],  a in [a_min, a_max]
// i.e. L*M stride-1 correlations over the M de-interleaved input streams.  One overlap-save
// block: forward-transform the M residue streams (b_e[i] = x_e[Q0 + a_min + i], i < 1024), form
// C_p = sum_e H_{p,e} . B_e for each output slot p, inverse-transform and keep the first
// hop = 1024 - (a_max - a_min) results c_p[u] = y[(Q0 + u) L + p].  M forward + L inverse
// transforms per hop*M inputs instead of 2 K L flop-pairs per input.
// REAL: float32 data (always REAL taps): the filter is linear and real, so two consecutive
// blocks ride in one complex transform, z = x_A + i x_B  ->  Re = y_A, Im = y_B.
struct FirOs32GArgs {
    const void *in;      // element 0 = first history sample
    void *out;
    const void *H;       // [L*M][1024] tap-phase spectra / 1024
    const void *tw;      // [32][32] W1024^(j*t)
    long long n_in;      // valid input elements (beyond: zeros)
    long long nq;        // output blocks q to produce (outputs = nq * L)
    long long start0;    // input element index of b_0[0] for block 0: K-1 + a_min*M (may be < 0)
    int L, hop;
};

// one 1024-point transform of the warp's 32 x 32 register tile through its shared-memory tile
template <bool INV, bool PT = false>
__device__ __forceinline__ void fft1024_fwd(c2 (&v)[32], c2 *F, const c2 *__restrict__ tw, const int t)
{
    // in: v[rev32(n1)] = x[32 n1 + t]; out: v[k2] = X[t + 32 k2]   (PT: ten loaded twiddles instead of 31)
    dft32_dit<INV>(v);
    if constexpr (PT) twiddle32<INV, false>(v, tw, t);
    else {
#pragma unroll
        for (int k1 = 1; k1 < 32; k1++) v[k1] = cmul_p<INV>(v[k1], tw[k1 * 32 + t]);
    }
    __syncwarp();
#pragma unroll
    for (int k1 = 0; k1 < 32; k1++) F[k1 * kOs32Stride + t] = v[k1];
    __syncwarp();
#pragma unroll
    for (int n2 = 0; n2 < 32; n2++) v[rev32(n2)] = F[t * kOs32Stride + n2];
    dft32_dit<INV>(v);
}
template <bool PT = false>
__device__ __forceinline__ void fft1024_inv(c2 (&v)[32], c2 *F, const c2 *__restrict__ tw, const int t)
{
    // in: v[k2] = X[t + 32 k2]; out: v[rev32(n1)] = x[32 n1 + t] (unnormalised inverse)
    dft32_dif<true>(v);
    if constexpr (PT) twiddle32<true, true>(v, tw, t);
    else {
#pragma unroll
        for (int n2 = 1; n2 < 32; n2++) v[rev32(n2)] = cmul_p<true>(v[rev32(n2)], tw[n2 * 32 + t]);
    }
    __syncwarp();
#pragma unroll
    for (int n2 = 0; n2 < 32; n2++) F[t * kOs32Stride + n2] = v[rev32(n2)];
    __syncwarp();
#pragma unroll
    for (int k1 = 0; k1 < 32; k1++) v[k1] = F[k1 * kOs32Stride + t];
    dft32_dif<true>(v);
}

// Shared memory of one warp: the 32 x 33 exchange tile, or -- when the L output slots are staged
// for a coalesced store (TILE_OUT) -- L planes of `plane` elements [p][u] with the exchange tile
// aliased onto the LAST plane (slot L-1 is written into its plane only after its own exchanges).
// Without staging, stores of slot p would touch every L-th element: partial 32-byte sectors,
// which cost 3x the L2 write transactions and read-modify-write DRAM traffic (ncu, C3).
constexpr int kOsgPlane = 1024 + 37;   // >= kOs32SmemElems; odd offset between planes spreads the banks
__host__ __device__ constexpr int osg_smem_elems(int L, bool tile_out) { return tile_out ? L * kOsgPlane : kOs32SmemElems; }

template <int M, bool MULTI_L, bool REAL, bool TILE_OUT, int MINB>
__global__ void __launch_bounds__(32, MINB) fir_os32g_kernel(const FirOs32GArgs a)
{
    extern __shared__ __align__(16) c2 smem_g[];
    const int t = threadIdx.x;
    const c2 *__restrict__ tw = static_cast<const c2 *>(a.tw);
    const c2 *__restrict__ H = static_cast<const c2 *>(a.H);
    const int L = a.L, hop = a.hop;
    c2 *F = TILE_OUT ? smem_g + (L - 1) * kOsgPlane : smem_g;
    constexpr int NB = REAL ? 2 : 1;                      // stream blocks per transform
    const long long nblk = (a.nq + (long long)hop * NB - 1) / ((long long)hop * NB);
    for (long long blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const long long Q0 = blk * hop * NB;              // first output block q of stream block A
        c2 B[M][32];
#pragma unroll
        for (int e = 0; e < M; e++) {
            const long long s0 = a.start0 + Q0 * M + e;   // input element of b_e[0] (block A)
            if constexpr (REAL) {
                const float *__restrict__ in = static_cast<const float *>(a.in);
                const long long s1 = s0 + (long long)hop * M;
                const bool inner = s0 >= 0 && s1 + 1023LL * M < a.n_in;
#pragma unroll
                for (int n1 = 0; n1 < 32; n1++) {
                    const long long ia = s0 + (long long)(32 * n1 + t) * M, ib = s1 + (long long)(32 * n1 + t) * M;
                    const float xa = (inner || (ia >= 0 && ia < a.n_in)) ? __ldg(in + ia) : 0.f;
                    const float xb = (inner || (ib >= 0 && ib < a.n_in)) ? __ldg(in + ib) : 0.f;
                    B[e][rev32(n1)] = pk(xa, xb);
                }
            } else {
                const c2 *__restrict__ in = static_cast<const c2 *>(a.in);
                const bool inner = s0 >= 0 && s0 + 1023LL * M < a.n_in;
#pragma unroll
                for (int n1 = 0; n1 < 32; n1++) {
                    const long long ia = s0 + (long long)(32 * n1 + t) * M;
                    B[e][rev32(n1)] = (inner || (ia >= 0 && ia < a.n_in)) ? __ldg(in + ia) : 0ull;
                }
            }
            fft1024_fwd<false>(B[e], F, tw, t);
        }
        for (int p = 0; p < L; p++) {
            c2 wloc[MULTI_L ? 32 : 1];
            c2(&w)[32] = *reinterpret_cast<c2(*)[32]>(MULTI_L ? &wloc[0] : &B[0][0]);
            const c2 *__restrict__ Hp = H + (size_t)p * M * 1024 + t;
#pragma unroll
            for (int k2 = 0; k2 < 32; k2++) {
                c2 acc = cmul_p<false>(B[0][k2], Hp[32 * k2]);
#pragma unroll
                for (int e = 1; e < M; e++) {
                    // acc += B_e * H_{p,e}
                    float fx, fy, hx, hy;
                    upk(B[e][k2], fx, fy); upk(Hp[e * 1024 + 32 * k2], hx, hy);
                    acc = fma2(B[e][k2], pk(hx, hx), fma2(pk(-fy, fx), pk(hy, hy), acc));
                }
                w[k2] = acc;
            }
            fft1024_inv(w, F, tw, t);
            // c_p[u], u = 32 n1 + t < hop, is y[(Q0 + u) L + p]  (REAL: Im part belongs to block B)
            if constexpr (TILE_OUT) {
                __syncwarp();                             // the last plane doubles as the exchange tile
                c2 *plane = smem_g + p * kOsgPlane;
#pragma unroll
                for (int n1 = 0; n1 < 32; n1++) plane[32 * n1 + t] = w[rev32(n1)];
            } else if constexpr (REAL) {
                float *__restrict__ out = static_cast<float *>(a.out);
#pragma unroll
                for (int n1 = 0; n1 < 32; n1++) {
                    const int u = 32 * n1 + t;
                    float ya, yb;
                    upk(w[rev32(n1)], ya, yb);
                    if (u < hop) {
                        const long long qa = Q0 + u, qb = qa + hop;
                        if (qa < a.nq) __stcg(out + qa * L + p, ya);
                        if (qb < a.nq) __stcg(out + qb * L + p, yb);
                    }
                }
            } else {
                c2 *__restrict__ out = static_cast<c2 *>(a.out);
#pragma unroll
                for (int n1 = 0; n1 < 32; n1++) {
                    const int u = 32 * n1 + t;
                    if (u < hop && Q0 + u < a.nq) __stcg(out + (Q0 + u) * L + p, w[rev32(n1)]);
                }
            }
        }
        if constexpr (TILE_OUT) {
            // flush: output j = u L + p of this block, contiguous in memory, lane-contiguous here
            __syncwarp();
            const long long left = a.nq - Q0;             // output blocks q still wanted from Q0 on
            const int nu = left < hop ? (int)left : hop;  // block A
            const int total = nu * L;
            const int dq = 32 / L, dr = 32 - dq * L;      // (u, p) step for j += 32, no division in the loop
            if constexpr (REAL) {
                float *__restrict__ out = static_cast<float *>(a.out);
                const long long leftb = left - hop;
                const int totalb = (leftb <= 0 ? 0 : (leftb < hop ? (int)leftb : hop)) * L;
                float *oa = out + Q0 * L, *ob = oa + (long long)hop * L;
                int u = t / L, p = t - u * L;
                for (int j = t; j < total; j += 32) {
                    float ya, yb;
                    upk(smem_g[p * kOsgPlane + u], ya, yb);
                    __stcg(oa + j, ya);
                    if (j < totalb) __stcg(ob + j, yb);
                    u += dq; p += dr;
                    if (p >= L) { p -= L; u++; }
                }
            } else {
                c2 *__restrict__ o = static_cast<c2 *>(a.out) + Q0 * L;
                int u = t / L, p = t - u * L;
                for (int j = t; j < total; j += 32) {
                    __stcg(o + j, smem_g[p * kOsgPlane + u]);
                    u += dq; p += dr;
                    if (p >= L) { p -= L; u++; }
                }
            }
            __syncwarp();                                 // planes are free for the next block
        }
    }
}

// ------------------------------------------- polyphase resampler, one warp per transform ---
// Same algebra as fir_os32g_kernel for complex float32 streams with 2 <= max(L, M) <= 4, spread
// over a CTA of NW = max(L, M) warps so that no thread ever holds more than ONE 1024-point
// sequence (64 data registers instead of 192): warp e < M transforms residue stream e and leaves
// its spectrum in shared memory, warp p < L forms C_p = sum_e H_{p,e} . B_e from those, inverse
// transforms it and stages its output slot as a plane [u]; the CTA then stores the L planes
// interleaved, fully coalesced.  ~110 registers x 96 threads and 42 KB of shared memory per CTA
// (L = 3, M = 2) keep 15 warps per SM resident where the one-warp kernel had 8.
// Plane stride (elements) of the staged output slots: a half-warp of the interleaved flush reads
// 16 consecutive outputs j = u L + p, i.e. ~16/L consecutive u from each of the L planes; the
// stride mod 16 (8-byte banks) is chosen so that those 16 reads hit 16 different banks.
__host__ __device__ constexpr int osp_plane_stride(int L) { return kOs32SmemElems + (L == 2 ? 8 : L == 3 ? 11 : 12); }

template <int NW, int MINB>
__global__ void __launch_bounds__(32 * NW, MINB) fir_osp_kernel(const FirOs32GArgs a, const int M)
{
    extern __shared__ __align__(16) c2 smem_p[];
    const int t = threadIdx.x & 31, w = threadIdx.x >> 5;
    const c2 *__restrict__ tw = static_cast<const c2 *>(a.tw);
    const c2 *__restrict__ in = static_cast<const c2 *>(a.in);
    const int L = a.L, hop = a.hop;
    c2 *S = smem_p;                                    // [M][kOs32SmemElems]: exchange tile, then spectrum [k2][t]
    c2 *P = smem_p + M * kOs32SmemElems;               // [L][pstride]: exchange tile, then output slot [u]
    const int pstride = osp_plane_stride(L);
    const long long nblk = (a.nq + hop - 1) / hop;
    const int dq = (32 * NW) / L, dr = (32 * NW) - dq * L;   // (u, p) step of the flush, no division in the loop
    for (long long blk = blockIdx.x; blk < nblk; blk += gridDim.x) {
        const long long Q0 = blk * hop;
        if (w < M) {
            c2 *F = S + w * kOs32SmemElems;
            const long long s0 = a.start0 + Q0 * M + w;   // input element of b_e[0]
            const bool inner = s0 >= 0 && s0 + 1023LL * M < a.n_in;
            c2 v[32];
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) {
                const long long ia = s0 + (long long)(32 * n1 + t) * M;
                v[rev32(n1)] = (inner || (ia >= 0 && ia < a.n_in)) ? __ldg(in + ia) : 0ull;
            }
            fft1024_fwd<false>(v, F, tw, t);
            __syncwarp();
#pragma unroll
            for (int k2 = 0; k2 < 32; k2++) F[32 * k2 + t] = v[k2];
        }
        __syncthreads();                                // spectra complete; the previous block's flush is done
        if (w < L) {
            c2 *plane = P + w * pstride;
            const c2 *__restrict__ Hp = static_cast<const c2 *>(a.H) + (size_t)w * M * 1024 + t;
            c2 v[32];
#pragma unroll
            for (int k2 = 0; k2 < 32; k2++) v[k2] = cmul_p<false>(S[32 * k2 + t], Hp[32 * k2]);
            for (int e = 1; e < M; e++) {
                const c2 *Se = S + e * kOs32SmemElems + t;
#pragma unroll
                for (int k2 = 0; k2 < 32; k2++) {
                    float fx, fy, hx, hy;
                    const c2 b = Se[32 * k2];
                    upk(b, fx, fy); upk(Hp[e * 1024 + 32 * k2], hx, hy);
                    v[k2] = fma2(b, pk(hx, hx), fma2(pk(-fy, fx), pk(hy, hy), v[k2]));
                }
            }
            fft1024_inv(v, plane, tw, t);
            __syncwarp();
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) plane[32 * n1 + t] = v[rev32(n1)];
        }
        __syncthreads();                                // all L slots staged
        {
            const long long left = a.nq - Q0;
            const int nu = left < hop ? (int)left : hop;
            const int total = nu * L;
            c2 *__restrict__ o = static_cast<c2 *>(a.out) + Q0 * L;
            int u = (int)threadIdx.x / L, p = (int)threadIdx.x - u * L;
            for (int j = threadIdx.x; j < total; j += 32 * NW) {
                __stcg(o + j, P[p * pstride + u]);
                u += dq; p += dr;
                if (p >= L) { p -= L; u++; }
            }
        }
        // no barrier here: the planes are next written after the next block's first barrier
    }
}

// Grouped variant: G independent NW-warp groups per CTA (one CTA per SM) share ONE copy of the tap
// spectra and twiddles in shared memory.  In fir_osp_kernel those are global loads through an L1
// that 5 x 42 KB of shared memory had shrunk to 40 KB: 37 % hit rate, long-scoreboard stalls
// (profiles/r01d_prof_osp_c3.txt).  Groups synchronise on their own named barriers.
#ifndef B200C_OSPG_PARTIAL_TW
#define B200C_OSPG_PARTIAL_TW 1
#endif
constexpr bool kOspgPartialTwiddles = B200C_OSPG_PARTIAL_TW != 0;

template <int NW, int G>
__global__ void __launch_bounds__(32 * NW * G, 1) fir_ospg_kernel(const FirOs32GArgs a, const int M)
{
    extern __shared__ __align__(16) c2 smem_q[];
    const int L = a.L, hop = a.hop;
    const int pstride = osp_plane_stride(L);
    c2 *Hs = smem_q;                                   // [L*M][1024]
    c2 *tws = Hs + (size_t)L * M * 1024;               // [32][32]
    const int group_elems = M * kOs32SmemElems + L * pstride;
    const int g = (threadIdx.x >> 5) / NW, w = (threadIdx.x >> 5) % NW, t = threadIdx.x & 31, tg = threadIdx.x - g * 32 * NW;
    c2 *S = tws + 1024 + (size_t)g * group_elems;      // [M][kOs32SmemElems]
    c2 *P = S + M * kOs32SmemElems;                    // [L][pstride]
    {
        const c2 *__restrict__ Hg = static_cast<const c2 *>(a.H), *__restrict__ twg = static_cast<const c2 *>(a.tw);
        for (int i = threadIdx.x; i < L * M * 1024; i += 32 * NW * G) Hs[i] = Hg[i];
        for (int i = threadIdx.x; i < 1024; i += 32 * NW * G) tws[i] = twg[i];
    }
    __syncthreads();
    auto group_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(g + 1), "r"(32 * NW) : "memory"); };
    const c2 *__restrict__ in = static_cast<const c2 *>(a.in);
    const long long nblk = (a.nq + hop - 1) / hop;
    const int dq = (32 * NW) / L, dr = (32 * NW) - dq * L;
    for (long long blk = (long long)blockIdx.x * G + g; blk < nblk; blk += (long long)gridDim.x * G) {
        const long long Q0 = blk * hop;
        if (w < M) {
            c2 *F = S + w * kOs32SmemElems;
            const long long s0 = a.start0 + Q0 * M + w;
            const bool inner = s0 >= 0 && s0 + 1023LL * M < a.n_in;
            c2 v[32];
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) {
                const long long ia = s0 + (long long)(32 * n1 + t) * M;
                v[rev32(n1)] = (inner || (ia >= 0 && ia < a.n_in)) ? __ldg(in + ia) : 0ull;
            }
            fft1024_fwd<false, kOspgPartialTwiddles>(v, F, tws, t);
            __syncwarp();
#pragma unroll
            for (int k2 = 0; k2 < 32; k2++) F[32 * k2 + t] = v[k2];
        }
        group_sync();
        if (w < L) {
            c2 *plane = P + w * pstride;
            const c2 *Hp = Hs + (size_t)w * M * 1024 + t;
            c2 v[32];
#pragma unroll
            for (int k2 = 0; k2 < 32; k2++) v[k2] = cmul_p<false>(S[32 * k2 + t], Hp[32 * k2]);
            for (int e = 1; e < M; e++) {
                const c2 *Se = S + e * kOs32SmemElems + t;
#pragma unroll
                for (int k2 = 0; k2 < 32; k2++) {
                    float fx, fy, hx, hy;
                    const c2 b = Se[32 * k2];
                    upk(b, fx, fy); upk(Hp[e * 1024 + 32 * k2], hx, hy);
                    v[k2] = fma2(b, pk(hx, hx), fma2(pk(-fy, fx), pk(hy, hy), v[k2]));
                }
            }
            fft1024_inv<kOspgPartialTwiddles>(v, plane, tws, t);
            __syncwarp();
#pragma unroll
            for (int n1 = 0; n1 < 32; n1++) plane[32 * n1 + t] = v[rev32(n1)];
        }
        group_sync();
        {
            const long long left = a.nq - Q0;
            const int nu = left < hop ? (int)left : hop;
            const int total = nu * L;
            c2 *__restrict__ o = static_cast<c2 *>(a.out) + Q0 * L;
            int u = tg / L, p = tg - u * L;
            for (int j = tg; j < total; j += 32 * NW) {
                __stcg(o + j, P[p * pstride + u]);
                u += dq; p += dr;
                if (p >= L) { p -= L; u++; }
            }
        }
    }
}

// ------------------------------------------------------------------------------- host ---
// in-place forward DFT (e^{-2 pi i nk/N}), N a power of two, double precision (host, setTaps path)
static void host_fft(std::vector<std::complex<double>> &x)
{
    const size_t n = x.size();
    for (size_t i = 1, j = 0; i < n; i++) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) std::swap(x[i], x[j]);
    }
    const double two_pi = 2.0 * 3.14159265358979323846264338327950288;
    for (size_t len = 2; len <= n; len <<= 1) {
        std::vector<std::complex<double>> w(len / 2);
        for (size_t k = 0; k < len / 2; k++) w[k] = std::polar(1.0, -two_pi * (double)k / (double)len);
        for (size_t i = 0; i < n; i += len)
            for (size_t k = 0; k < len / 2; k++) {
                const std::complex<double> u = x[i + k], v = x[i + k + len / 2] * w[k];
                x[i + k] = u + v;
                x[i + k + len / 2] = u - v;
            }
    }
}

static void taps_spectrum(std::vector<float> &hf, int N, const double *taps, size_t ntaps, bool complex_taps)
{
    // Hf[f] = (1/N) * sum_k h[k] exp(-2*pi*i*f*k/N) in double, rounded once to float
    std::vector<std::complex<double>> x((size_t)N);
    for (size_t k = 0; k < ntaps; k++) x[k] = complex_taps ? std::complex<double>(taps[2 * k], taps[2 * k + 1]) : std::complex<double>(taps[k], 0.0);
    host_fft(x);
    hf.resize(2 * (size_t)N);
    for (int f = 0; f < N; f++) {
        hf[2 * f] = (float)(x[f].real() / N);
        hf[2 * f + 1] = (float)(x[f].imag() / N);
    }
}

static void unit_root_table(std::vector<float> &tb, int N, int rows, int cols, int row_mul)
{
    // tb[r][c] = exp(-2*pi*i*(row_mul*r*c)/N)
    const double two_pi = 2.0 * 3.14159265358979323846264338327950288;
    tb.assign(2 * (size_t)rows * cols, 0.f);
    for (int r = 0; r < rows; r++)
        for (int c = 0; c < cols; c++) {
            const int e = (row_mul * r * c) & (N - 1);
            tb[2 * ((size_t)r * cols + c)] = (float)std::cos(-two_pi * e / N);
            tb[2 * ((size_t)r * cols + c) + 1] = (float)std::sin(-two_pi * e / N);
        }
}

static int upload(void **d, const std::vector<float> &h)
{
    if (!*d) B200C_CUDA_TRY(cudaMalloc(d, h.size() * sizeof(float)));
    B200C_CUDA_TRY(cudaMemcpy(*d, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    return B200C_OK;
}

// Transform length for K taps: the 1024-point warp kernel while its hop keeps >= ~70 % of the
// block (measured crossover, DESIGN.md 4.2), the 4096-point kernel above.  B200C_OS_N overrides.
static int pick_length(size_t ntaps)
{
    static const int forced = [] { const char *e = std::getenv("B200C_OS_N"); return e ? std::atoi(e) : 0; }();
    if (forced == 1024 && ntaps <= 769) return 1024;
    if (forced == 4096) return 4096;
    return ntaps <= kFirOs1kMaxTaps ? 1024 : 4096;
}

static inline long long floordiv_ll(long long x, long long y)
{
    long long q = x / y;
    if ((x % y != 0) && ((x < 0) != (y < 0))) q--;
    return q;
}

// Polyphase / real-data plan: spectra of the L*M tap phases on the 1024-point grid.
static int configure_general(FirOsPlan &p, bool real_data, const double *taps, size_t ntaps, bool complex_taps, size_t M,
                             size_t L)
{
    const int N = 1024;
    const long long K = (long long)((ntaps + L - 1) / L);   // filter/FIRFilter.cpp:335
    struct Term { int p, e; long long a; double hr, hi; };
    std::vector<Term> terms;
    long long a_min = 0, a_max = 0;
    bool first = true;
    for (size_t ps = 0; ps < L; ps++) {
        const long long i = (long long)((ps + 1) * M - 1), j = i % (long long)L, d = i / (long long)L;
        for (long long k = 0; j + k * (long long)L < (long long)ntaps; k++) {
            const size_t ti = (size_t)(j + k * (long long)L);
            const long long a = floordiv_ll(d - k, (long long)M);
            const int e = (int)((d - k) - a * (long long)M);
            terms.push_back({(int)ps, e, a, complex_taps ? taps[2 * ti] : taps[ti], complex_taps ? taps[2 * ti + 1] : 0.0});
            if (first) { a_min = a_max = a; first = false; }
            a_min = std::min(a_min, a); a_max = std::max(a_max, a);
        }
    }
    const long long span = a_max - a_min;
    if (first || span > kFirOsGenMaxSpan) return B200C_OK;   // not applicable: the direct kernel keeps the job
    // c_p[u] = sum_e sum_a g[a] b_e[u + (a - a_min)]  ==  circular convolution with g'[(N - (a - a_min)) mod N] = g[a]
    std::vector<std::vector<std::complex<double>>> gp((size_t)L * M, std::vector<std::complex<double>>((size_t)N));
    for (const Term &t : terms) gp[(size_t)t.p * M + t.e][(size_t)((N - (t.a - a_min)) % N)] += std::complex<double>(t.hr, t.hi);
    std::vector<float> H(2 * (size_t)L * M * N);
    for (size_t sub = 0; sub < gp.size(); sub++) {
        host_fft(gp[sub]);
        for (int f = 0; f < N; f++) {
            H[2 * (sub * N + f)] = (float)(gp[sub][f].real() / N);
            H[2 * (sub * N + f) + 1] = (float)(gp[sub][f].imag() / N);
        }
    }
    if (p.d_H && p.H_floats < H.size()) { cudaFree(p.d_H); p.d_H = nullptr; }
    int rc;
    if ((rc = upload(&p.d_H, H))) return rc;
    p.H_floats = std::max(p.H_floats, H.size());
    if (!p.d_tw1k) {
        std::vector<float> tb;
        unit_root_table(tb, 1024, 32, 32, 1);
        if ((rc = upload(&p.d_tw1k, tb))) return rc;
    }
    p.general = true; p.real = real_data;
    p.N = N; p.M = (int)M; p.L = (int)L;
    p.hopq = (int)(N - span);
    p.start0 = (K - 1) + a_min * (long long)M;
    p.K = (int)K;
    p.ready = true;
    return B200C_OK;
}

// Decides whether (and how) the fused overlap-save path serves this configuration; leaves
// p.ready false when the direct kernel (fir.cu) should run instead.
int fir_os_configure(FirOsPlan &p, int dtype, const double *taps, size_t ntaps, bool complex_taps, size_t M, size_t L,
                     bool force)
{
    p.ready = false; p.general = false; p.real = false; p.osp = false; p.real32 = false; p.x32 = false;
    // complex float32, interpolation 3 / decimation 2: one forward + one inverse transform per block
    // (fir_os32x_kernel); its rate does not depend on the tap count while the hop stays above ~60 % of the block
    const bool no_x32 = [] { const char *e = std::getenv("B200C_OSX"); return e && std::atoi(e) == 0; }();   // read per configure: tests compare both
    if (dtype == B200C_CF32 && L == 3 && M == 2 && !no_x32 && ntaps >= 2 && ntaps <= 1200 &&
        (force || (ntaps + L - 1) / L >= kFirOsAutoMinTapsX32)) {
        const long long K = (long long)((ntaps + L - 1) / L);            // filter/FIRFilter.cpp:335
        int m0 = (int)((ntaps - 2 + 1) / 2);                             // ceil((ntaps - 2) / 2): v[i] is alias free from i = ntaps - 1
        m0 = (m0 + 2) / 3 * 3;                                           // whole output blocks q per transform block
        const double two_pi = 2.0 * 3.14159265358979323846264338327950288;
        std::vector<float> hx(2 * 3072), tb(2 * 48 * 32);
        for (int k = 0; k < 3072; k++) {
            // H'[k] = (1/3072) exp(2 pi i k (M - 1) / 3072) sum_t h[t] exp(-2 pi i k t / 3072), in double
            std::complex<double> acc(0.0, 0.0);
            for (size_t tt = 0; tt < ntaps; tt++) {
                const std::complex<double> h = complex_taps ? std::complex<double>(taps[2 * tt], taps[2 * tt + 1]) : std::complex<double>(taps[tt], 0.0);
                const long long e = ((long long)k * (long long)tt) % 3072;
                acc += h * std::polar(1.0, -two_pi * (double)e / 3072.0);
            }
            acc *= std::polar(1.0 / 3072.0, two_pi * (double)k / 3072.0);
            hx[2 * k] = (float)acc.real();
            hx[2 * k + 1] = (float)acc.imag();
        }
        for (int n2 = 0; n2 < 48; n2++)
            for (int t = 0; t < 32; t++) {
                tb[2 * (n2 * 32 + t)] = (float)std::cos(two_pi * (double)(n2 * t) / 1536.0);
                tb[2 * (n2 * 32 + t) + 1] = (float)std::sin(two_pi * (double)(n2 * t) / 1536.0);
            }
        int rc;
        if ((rc = upload(&p.d_hx, hx))) return rc;
        if ((rc = upload(&p.d_tw3, tb))) return rc;
        if (!p.d_tw1k) {
            unit_root_table(tb, 1024, 32, 32, 1);
            if ((rc = upload(&p.d_tw1k, tb))) return rc;
        }
        p.N = 1024; p.K = (int)K; p.M = 2; p.L = 3; p.m0 = m0; p.p0 = (K - 1) - 2 * (long long)(m0 / 3);
        p.x32 = true;
        p.ready = true;
        return B200C_OK;
    }
    if (dtype == B200C_CF32 && M == 1 && L == 1) {
        // measured (tools/sweep.sh): the fused kernel beats the direct one from 2 taps up; short filters keep the
        // time-domain kernel all the same (kFirOsAutoMinTapsFloat)
        if (ntaps < 2 || ntaps > kFirOsMaxTaps || (!force && ntaps < kFirOsAutoMinTapsFloat)) return B200C_OK;
        std::vector<float> tb, hf;
        int rc;
        p.N = pick_length(ntaps);
        if (p.N == 4096) {
            if (!p.d_twa) {
                // step twiddles W4096^(j t) = W^(8 a t) * W^(b t), j = 8a + b
                unit_root_table(tb, 4096, 8, 64, 8);
                if ((rc = upload(&p.d_twa, tb))) return rc;
                unit_root_table(tb, 4096, 8, 64, 1);
                if ((rc = upload(&p.d_twb, tb))) return rc;
                unit_root_table(tb, 4096, 64, 64, 1);          // the whole table, for the persistent form
                if ((rc = upload(&p.d_twf, tb))) return rc;
            }
            taps_spectrum(hf, 4096, taps, ntaps, complex_taps);
            if ((rc = upload(&p.d_hf, hf))) return rc;
        } else {
            if (!p.d_tw1ks) {
                tb.resize(2 * 32 * (size_t)kOs32SignedTwRows);
                os32_signed_twiddles(tb.data());
                if ((rc = upload(&p.d_tw1ks, tb))) return rc;
            }
            taps_spectrum(hf, 1024, taps, ntaps, complex_taps);
            if ((rc = upload(&p.d_hf1k, hf))) return rc;
        }
        p.K = (int)ntaps;
        p.ready = true;
        return B200C_OK;
    }
    if (dtype == B200C_F32 && M == 1 && L == 1 && !complex_taps && ntaps >= (force ? 2 : kFirOsAutoMinTapsFloat) && ntaps <= kFirOs1kMaxTaps &&
        !(std::getenv("B200C_OS32R") && std::atoi(std::getenv("B200C_OS32R")) == 0)) {
        // real float32 stream: two blocks per complex 1024-point transform (fir_os32r_kernel)
        std::vector<float> tb, hf;
        int rc;
        if (!p.d_tw1k) {
            unit_root_table(tb, 1024, 32, 32, 1);
            if ((rc = upload(&p.d_tw1k, tb))) return rc;
        }
        taps_spectrum(hf, 1024, taps, ntaps, false);
        if ((rc = upload(&p.d_hf1k, hf))) return rc;
        p.N = 1024; p.K = (int)ntaps; p.real32 = true;
        p.ready = true;
        return B200C_OK;
    }
    // multi-warp resampler kernel: complex float32, 2 <= max(L, M) <= 4 (pure M <= 2 decimators stay on the one-warp kernel)
    const bool osp = dtype == B200C_CF32 && L <= 4 && M <= 4 && std::max(L, M) >= 2 && !(L == 1 && M <= 2) &&
                     !(std::getenv("B200C_OSP") && std::atoi(std::getenv("B200C_OSP")) == 0);
    if ((dtype == B200C_CF32 || dtype == B200C_F32) && (M <= 2 || osp) && L <= (force ? kFirOsGenForcedMaxInterp : kFirOsGenMaxInterp)) {
        const size_t per_phase = (ntaps + L - 1) / L;
        // the grouped resampler runs at the same rate whatever the tap count and beats the direct kernel
        // from 16 taps per phase (measured: 48-tap RRC, L = 3, M = 2: 151 vs 137 Gsamples/s)
        static const bool no_group = [] { const char *e = std::getenv("B200C_OSPG"); return e && std::atoi(e) == 0; }();
        const int nw = (int)std::max(L, M), G = nw == 2 ? 6 : nw == 3 ? 4 : 3;
        const bool grouped = osp && !no_group &&
                             sizeof(c2) * ((size_t)L * M * 1024 + 1024 + G * ((size_t)M * kOs32SmemElems + (size_t)L * osp_plane_stride((int)L))) <= 227 * 1024;
        const size_t min_taps = (M == 1 && L == 1) ? kFirOsAutoMinTapsReal
                                : (osp && M == 4 && L == 1) ? kFirOsAutoMinTapsOspDecim4
                                : osp ? kFirOsAutoMinTapsOsp
                                : L >= 5 ? kFirOsAutoMinTapsWideInterp : kFirOsAutoMinTapsResamp;
        if (!force && per_phase < min_taps) return B200C_OK;
        if (ntaps < 2) return B200C_OK;
        p.osp = osp;
        p.ospg = 0;
        const int rc = configure_general(p, dtype == B200C_F32, taps, ntaps, complex_taps, M, L);
        // grouped form: G groups + one copy of the tap spectra and twiddles fit 227 KB
        if (rc == B200C_OK && p.ready && grouped) p.ospg = G;
        return rc;
    }
    return B200C_OK;
}

void fir_os_destroy(FirOsPlan &p)
{
    for (void **d : {&p.d_hf, &p.d_twa, &p.d_twb, &p.d_twf, &p.d_hf1k, &p.d_tw1k, &p.d_tw1ks, &p.d_H, &p.d_hx, &p.d_tw3}) {
        if (*d) cudaFree(*d);
        *d = nullptr;
    }
    p.H_floats = 0;
    p.ready = false;
}

const char *fir_os_kernel_name(const FirOsPlan &p)
{
    if (p.x32) return "fir_os32x_kernel";
    if (p.general) return p.osp ? (p.ospg ? "fir_ospg_kernel" : "fir_osp_kernel") : "fir_os32g_kernel";
    if (p.real32) return "fir_os32r_kernel";
    // (4096-point: launches too small for the persistent form -- a few hundred blocks, or a bank of fewer channels than
    // SMs -- run fir_os64_kernel, the same transform with one group per CTA)
    return p.N == 1024 ? "fir_os32_kernel" : "fir_os64p_kernel";
}

template <int M, bool MULTI_L, bool REAL, bool TILE_OUT, int MINB>
static int launch_general(const FirOs32GArgs &a, long long nblk, int sm_count, cudaStream_t stream)
{
    auto kern = fir_os32g_kernel<M, MULTI_L, REAL, TILE_OUT, MINB>;
    const size_t smem = sizeof(c2) * (size_t)osg_smem_elems(a.L, TILE_OUT);
    static thread_local bool configured[16] = {false};
    int dev = 0;
    B200C_CUDA_TRY(cudaGetDevice(&dev));
    if (dev < 16 && !configured[dev]) {
        B200C_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        configured[dev] = true;
    }
    const long long by_smem = std::max<long long>(1, (220 * 1024) / (long long)(smem + 1024));
    const int per_sm = (int)std::min<long long>(MINB, by_smem);
    const int grid = (int)std::min<long long>(nblk, (long long)sm_count * per_sm * 4);
    kern<<<grid, 32, smem, stream>>>(a);
    B200C_CUDA_TRY(cudaGetLastError());
    return B200C_OK;
}

template <int NW, int MINB>
static void launch_osp(const FirOs32GArgs &a, int M, size_t smem, long long nblk, int sm_count, cudaStream_t stream)
{
    auto kern = fir_osp_kernel<NW, MINB>;
    static thread_local bool configured[16] = {false};
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && dev < 16 && !configured[dev]) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
        if (const char *e = std::getenv("B200C_OSP_CARVE")) cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, std::atoi(e));
        configured[dev] = true;
    }
    static const int forced = [] { const char *e = std::getenv("B200C_OSP_PERSM"); return e ? std::atoi(e) : 0; }();
    const long long per_sm = std::max<long long>(1, std::min<long long>(forced > 0 ? forced : MINB, (224 * 1024) / (long long)(smem + 1024)));
    const int grid = (int)std::min<long long>(nblk, (long long)sm_count * per_sm * 2);
    kern<<<grid, 32 * NW, smem, stream>>>(a, M);
}

template <int NW, int G>
static void launch_ospg(const FirOs32GArgs &a, int M, size_t smem, long long nblk, int sm_count, cudaStream_t stream)
{
    auto kern = fir_ospg_kernel<NW, G>;
    static thread_local bool configured[16] = {false};
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && dev < 16 && !configured[dev]) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        configured[dev] = true;
    }
    const int grid = (int)std::min<long long>((nblk + G - 1) / G, (long long)sm_count);
    kern<<<grid, 32 * NW * G, smem, stream>>>(a, M);
}

// Launch with programmatic stream serialization: the kernel may start while its predecessor in the stream is still running;
// it must execute griddepcontrol.wait before touching stream data (fir_os32_kernel, fir_os32x_kernel persistent forms).
static bool pdl_enabled()
{
    static const bool on = [] { const char *e = std::getenv("B200C_PDL"); return !e || std::atoi(e) != 0; }();
    return on;
}
template <typename Kernel, typename Args>
static cudaError_t launch_dependent(Kernel kern, int grid, int block, size_t smem, cudaStream_t stream, const Args &a)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, a);
}

bool fir_os_batchable(const FirOsPlan &p) { return p.ready && !p.x32 && !p.general && !p.real32; }

int fir_os_launch(const FirOsPlan &p, const void *d_in, size_t in_elems, void *d_out, size_t nq, int sm_count,
                  cudaStream_t stream, const FirOsBatch *batch)
{
    if (nq == 0) return B200C_OK;
    if (batch && !fir_os_batchable(p)) { set_error("filter bank: the batched launch serves complex float32 L = M = 1 only"); return B200C_ERR_UNSUPPORTED; }
    const int nchan = batch ? batch->nchan : 1;
    if (p.x32) {
        FirOsX32Args a;
        a.in = d_in; a.out = d_out; a.hx = p.d_hx; a.tw = p.d_tw1k; a.tw3 = p.d_tw3;
        a.n_in = (long long)in_elems; a.n_out = (long long)nq * 3; a.p0 = p.p0; a.m0 = p.m0;
        const long long nblk = (a.n_out + (1536 - p.m0) - 1) / (1536 - p.m0);
        // One persistent 12-warp CTA per SM, tables in shared memory, partial twiddles, second inverse round by lane pairs.
        // Measured alternatives (profiles/r02_osx_variants.txt): 12 one-warp CTAs per SM with tables through L1 (-11 %),
        // all twiddles loaded (-2 %), 8 / 9 warps with landing buffers and compact tables (-3 % / -17 %: the kernel is
        // FMA-pipe bound, fewer warps lose more than the earlier prefetch gains), lanes 0..15 alone in the second round (-1.5 %),
        // 13 / 14 warps at 128 registers (-14 % / -9 %: the register cap costs more than the extra warps hide).
        const size_t tile = sizeof(c2) * kX32SmemElems;
        const size_t smem = 12 * tile + sizeof(c2) * kX32TabElems;
        static thread_local bool configured[16] = {false};
        int dev = 0;
        B200C_CUDA_TRY(cudaGetDevice(&dev));
        if (dev < 16 && !configured[dev]) {
            B200C_CUDA_TRY(cudaFuncSetAttribute(fir_os32x_kernel<12, 1, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            configured[dev] = true;
        }
        const int grid = (int)std::min<long long>((nblk + 11) / 12, (long long)sm_count);
        a.pdl = pdl_enabled() ? 1 : 0;
        if (a.pdl) B200C_CUDA_TRY(launch_dependent(fir_os32x_kernel<12, 1, true, true>, grid, 32 * 12, smem, stream, a));
        else fir_os32x_kernel<12, 1, true, true><<<grid, 32 * 12, smem, stream>>>(a);
        B200C_CUDA_TRY(cudaGetLastError());
        return B200C_OK;
    }
    if (p.general) {
        FirOs32GArgs a;
        a.in = d_in; a.out = d_out; a.H = p.d_H; a.tw = p.d_tw1k;
        a.n_in = (long long)in_elems; a.nq = (long long)nq; a.start0 = p.start0; a.L = p.L; a.hop = p.hopq;
        if (p.osp) {
            const int nw = std::max(p.L, p.M);
            const size_t smem = sizeof(c2) * ((size_t)p.M * kOs32SmemElems + (size_t)p.L * osp_plane_stride(p.L));
            const long long nblk = ((long long)nq + p.hopq - 1) / p.hopq;
            // grouped variant (tap spectra + twiddles once per SM in shared memory) when its groups fit
            const size_t shared_tab = sizeof(c2) * ((size_t)p.L * p.M * 1024 + 1024);
            if (p.ospg && nw == 3) launch_ospg<3, 4>(a, p.M, shared_tab + 4 * smem, nblk, sm_count, stream);
            else if (p.ospg && nw == 2) launch_ospg<2, 6>(a, p.M, shared_tab + 6 * smem, nblk, sm_count, stream);
            else if (p.ospg && nw == 4) launch_ospg<4, 3>(a, p.M, shared_tab + 3 * smem, nblk, sm_count, stream);
            else if (nw == 2) launch_osp<2, 7>(a, p.M, smem, nblk, sm_count, stream);
            else if (nw == 3) launch_osp<3, 5>(a, p.M, smem, nblk, sm_count, stream);
            else launch_osp<4, 3>(a, p.M, smem, nblk, sm_count, stream);
            B200C_CUDA_TRY(cudaGetLastError());
            return B200C_OK;
        }
        const long long per = (long long)p.hopq * (p.real ? 2 : 1);
        const long long nblk = ((long long)nq + per - 1) / per;
        // slot staging for a coalesced store pays from L = 2 and fits shared memory up to L = 4
        const bool ml = p.L > 1, tile = p.L >= 2 && p.L <= 4;
#define OSG(MM, RR, MB1, MBL)                                                                                      \
    (!ml ? launch_general<MM, false, RR, false, MB1>(a, nblk, sm_count, stream)                                      \
         : tile ? launch_general<MM, true, RR, true, MBL>(a, nblk, sm_count, stream)                                 \
                : launch_general<MM, true, RR, false, MBL>(a, nblk, sm_count, stream))
        if (p.M == 1) return p.real ? OSG(1, true, 12, 10) : OSG(1, false, 12, 10);
        return p.real ? OSG(2, true, 10, 8) : OSG(2, false, 10, 8);
#undef OSG
    }
    if (p.real32) {
        FirOs32RArgs a;
        a.in = static_cast<const float *>(d_in); a.out = static_cast<float *>(d_out); a.hf = p.d_hf1k; a.tw = p.d_tw1k;
        a.n_in = (long long)in_elems; a.n_out = (long long)nq; a.K = p.K;
        const long long npair = ((long long)nq + p.hop() - 1) / p.hop();
        // one persistent 12-warp CTA per SM, tables in shared memory, a landing buffer per warp (the next pair is fetched a
        // whole pair ahead).  Round 1 measured the alternatives: 12 one-warp CTAs 656, no landing buffers 690, this 707 Gsamples/s.
        const size_t tile = sizeof(c2) * kOs32SmemElems;
        const size_t smem_early = 12 * tile + sizeof(c2) * 2048 + sizeof(c2) * 12 * kOs32Landing;
        static thread_local bool configured[16] = {false};
        int dev = 0;
        B200C_CUDA_TRY(cudaGetDevice(&dev));
        if (dev < 16 && !configured[dev]) {
            B200C_CUDA_TRY(cudaFuncSetAttribute(fir_os32r_kernel<12, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_early));
            configured[dev] = true;
        }
        const int grid = (int)std::min<long long>((npair + 11) / 12, (long long)sm_count);
        fir_os32r_kernel<12, 1, true><<<grid, 32 * 12, smem_early, stream>>>(a);
        B200C_CUDA_TRY(cudaGetLastError());
        return B200C_OK;
    }
    const size_t n_out = nq;
    const long long nblk = (((long long)n_out + p.hop() - 1) / p.hop()) * nchan;
    if (p.N == 1024) {
        FirOs32Args a;
        a.in = d_in; a.out = d_out; a.hf = batch ? batch->d_hf : p.d_hf1k; a.tw = p.d_tw1ks;
        a.n_in = (long long)in_elems; a.n_out = (long long)n_out; a.K = p.K;
        a.nchan = nchan; a.in_stride = batch ? batch->in_stride : 0; a.out_stride = batch ? batch->out_stride : 0;
        a.spread = 0; a.pdl = 0;
        if (nchan == 1) {
            // single stream: one persistent 12-warp CTA per SM, tap spectrum + twiddles in shared memory, a landing buffer per
            // warp (the next block is fetched a whole block ahead).  Round-1 steps, headline Gsamples/s: 12 one-warp CTAs 272,
            // persistent + shared tables 288, + landing buffers 300; partial twiddles measured no gain and are gone.
            const size_t smem_early = sizeof(c2) * (12 * (size_t)kOs32SmemElems + kOs32TabElems + 12 * (size_t)kOs32Landing);
            static thread_local bool configured[16] = {false};
            int dev = 0;
            B200C_CUDA_TRY(cudaGetDevice(&dev));
            if (dev < 16 && !configured[dev]) {
                B200C_CUDA_TRY(cudaFuncSetAttribute(fir_os32_kernel<12, 1, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_early));
                configured[dev] = true;
            }
            // fewer blocks than one wave of warps: one CTA per SM anyway, blocks dealt warp-major
            a.spread = nblk < 12LL * sm_count ? 1 : 0;
            const int grid = (int)std::min<long long>(a.spread ? nblk : (nblk + 11) / 12, (long long)sm_count);
            a.pdl = pdl_enabled() ? 1 : 0;
            if (a.pdl) B200C_CUDA_TRY(launch_dependent(fir_os32_kernel<12, 1, true, false, true>, grid, 32 * 12, smem_early, stream, a));
            else fir_os32_kernel<12, 1, true, false, true><<<grid, 32 * 12, smem_early, stream>>>(a);
            B200C_CUDA_TRY(cudaGetLastError());
            return B200C_OK;
        }
        // filter bank (one spectrum per channel): one-warp CTAs, 12 per SM, tables through L1
        {
            const int grid = (int)std::min<long long>(nblk, (long long)sm_count * 12 * 4);
            fir_os32_kernel<1, 12><<<grid, 32, 0, stream>>>(a);
        }
        B200C_CUDA_TRY(cudaGetLastError());
        return B200C_OK;
    }
    FirOs64Args a;
    a.in = d_in; a.out = d_out; a.hf = batch ? batch->d_hf : p.d_hf; a.twa = p.d_twa; a.twb = p.d_twb; a.twf = p.d_twf;
    a.n_in = (long long)in_elems; a.n_out = (long long)n_out; a.K = p.K;
    a.nchan = nchan; a.in_stride = batch ? batch->in_stride : 0; a.out_stride = batch ? batch->out_stride : 0;
    a.parts = 1;
    // default: the persistent form wherever it applies (B200C_OS64P=0: always the one-transform-per-CTA kernel, for A/B runs)
    static const bool persistent = [] { const char *e = std::getenv("B200C_OS64P"); return !e || std::atoi(e) != 0; }();
    const long long blocks_per_chan = ((long long)n_out + p.hop() - 1) / p.hop();
    if (persistent && (long long)nchan * blocks_per_chan >= 4LL * kOs64Groups * sm_count) {
        // one persistent 256-thread CTA per SM: four transform groups sharing the step-twiddle table and the tap spectrum.
        // CTA-tasks = (channel, part); `parts` is the split (>= 16 blocks per part) whose task count fills rounds of CTAs best
        const size_t smem = sizeof(c2) * ((size_t)kOs64Groups * kOs64SmemElems + 4096 + 4096);
        if (nchan == 1) a.parts = sm_count;
        else {
            const long long maxp = std::max<long long>(1, blocks_per_chan / 16);
            double best = -1.0;
            for (long long q = 1; q <= std::min<long long>(maxp, 32); q++) {
                const long long T = (long long)nchan * q, rounds = (T + sm_count - 1) / sm_count;
                // every extra part re-stages the 32 KB spectrum once more per channel: measured ~0.15 % per part at 342 blocks per channel
                const double util = (double)T / (double)(rounds * sm_count) - 1.5e-3 * (double)(q - 1);
                if (util > best) { best = util; a.parts = (int)q; }
            }
        }
        static thread_local bool configured[16] = {false};
        int dev = 0;
        B200C_CUDA_TRY(cudaGetDevice(&dev));
        if (dev < 16 && !configured[dev]) {
            B200C_CUDA_TRY(cudaFuncSetAttribute(fir_os64p_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            configured[dev] = true;
        }
        fir_os64p_kernel<<<sm_count, 64 * kOs64Groups, smem, stream>>>(a);
        B200C_CUDA_TRY(cudaGetLastError());
        return B200C_OK;
    }
    // 4 CTAs of 64 threads per SM (252 registers); 3 / 5 / 6 per SM measured slower in round 1
    const int grid = (int)std::min<long long>(nblk, (long long)sm_count * 4 * 4);
    fir_os64_kernel<4><<<grid, 64, 0, stream>>>(a);
    B200C_CUDA_TRY(cudaGetLastError());
    return B200C_OK;
}

} // namespace b200c
