// Host-side plan of one configured /comms/fft block (libb200comms.so).
#pragma once
#include <cstddef>
#include <cstdint>
#include <vector>

#include "common.hpp"

namespace b200c {

// The radix plan and tables a reference FFTAux holds (fft/FFTAux.h:16-48):
//   float/double: kissfft<T>::_twiddles/_stageRadix/_stageRemainder (fft/kissfft.hh:28-56,306-309)
//   int16       : kiss_fft_state factors + Q15 twiddles (fft/kiss_fft.c:339-368)
struct FftPlan {
    int dtype = B200C_CF32;
    int n = 0;
    int inverse = 0;
    int nstages = 0;
    int radix[64];
    int rem[64];          // m of each stage
    bool has_generic = false;   // any radix outside {2,3,4,5}
    // device tables
    void *d_tw = nullptr;       // n twiddles in the element type
    int *d_scatter = nullptr;   // scatter[i] = output slot o of input index i (inverse of kf_work's leaf copy)
    // execution shape
    int tpc = 1;                // transforms per CTA
    int threads = 256;
    bool smem = true;           // working buffer in shared memory (else: in d_out + scratch)
    size_t smem_bytes = 0;
    void *d_scratch = nullptr;  // generic-radix scratch for the global path
    size_t scratch_bytes = 0;
    int fast = 0;               // 0 = generic staged kernel, 4096 = three-pass register kernel
    void *d_fast[3] = {nullptr, nullptr, nullptr};   // per-pass twiddle tables of the fast kernel
    void *d_fastw[3] = {nullptr, nullptr, nullptr};  // the same unpacked to (int32 re, int32 im): complex int16, lazy-wrap kernel
    bool force_staged = false;  // tests: run the generic staged kernel even when a fast path exists
};

int fft_plan_create(FftPlan &p, int dtype, size_t nbins, int inverse, size_t smem_budget);
void fft_plan_destroy(FftPlan &p);
int fft_launch(FftPlan &p, const void *d_in, void *d_out, size_t batch, int sm_count, cudaStream_t stream);

// Fused overlap-save FIR, fir_os.cu.
//  * complex float32, L = M = 1, 2..2049 taps: 1024-point (one warp per block) kernel for the
//    shorter tap counts, 4096-point (64 threads per block) above;
//  * complex float32 / float32 with M <= 2, any L <= 64 (polyphase resampler) and real data:
//    generalised 1024-point kernel over the L*M tap-phase spectra.
struct FirOsPlan {
    bool ready = false;
    bool general = false;     // polyphase / real-data kernel
    bool real = false;        // float32 data: two stream blocks per complex transform
    bool osp = false;         // general: the multi-warp resampler kernel (fir_osp_kernel) serves it
    int ospg = 0;             // > 0: its grouped form (fir_ospg_kernel) with this many groups per CTA
    bool real32 = false;      // float32 data, L = M = 1: fir_os32r_kernel (two blocks per transform)
    bool x32 = false;         // complex float32, L = 3, M = 2: fir_os32x_kernel (one 1024-point forward, one 1536-point inverse)
    int m0 = 0;               // x32: first alias-free output of a block (hop = 1536 - m0 outputs)
    long long p0 = 0;         // x32: input element at which block 0's window starts
    void *d_hx = nullptr;     // x32: [3072] float2 folded tap spectrum H'
    void *d_tw3 = nullptr;    // x32: [48][32] float2 exp(+2 pi i n2 t / 1536)
    int N = 4096;             // transform length in use
    int K = 0;                // L = M = 1 kernels: taps; general: K = ceil(ntaps / L)
    int M = 1, L = 1;
    int hopq = 0;             // general: output blocks q per transform block
    long long start0 = 0;     // general: input element of b_0[0] for block 0
    void *d_hf = nullptr;     // [4096] float2: spectrum of the taps / 4096
    void *d_twa = nullptr;    // [8][64] float2: W4096^(8*a*t)
    void *d_twb = nullptr;    // [8][64] float2: W4096^(b*t)
    void *d_twf = nullptr;    // [64][64] float2: W4096^(j*t), the whole step-twiddle table
    void *d_hf1k = nullptr;   // [1024] float2: spectrum of the taps / 1024
    void *d_tw1k = nullptr;   // [32][32] float2: W1024^(j*t)
    void *d_H = nullptr;      // general: [L*M][1024] float2 tap-phase spectra / 1024
    size_t H_floats = 0;
    // output blocks q covered by one kernel block (host-buffer chunking aligns to this)
    int hop() const { return x32 ? (1536 - m0) / 3 : general ? hopq * (real ? 2 : 1) : (N - (K - 1)) * (real32 ? 2 : 1); }
};
constexpr size_t kFirOsMaxTaps = 2049;
constexpr size_t kFirOs1kMaxTaps = 448;       // measured crossover of the 1024- and 4096-point kernels
// automatic switch from the direct kernel (taps per output phase at or above this take the fused
// path): real float32 streams, and resamplers where the direct kernel still wins for short phases
constexpr size_t kFirOsAutoMinTapsReal = 9;
// float32 / complex float32, L = M = 1: filters of up to this many taps stay on the direct time-domain kernel (HBM-bound
// there anyway: <= 64 flop per 16 B), which keeps the reference's per-output semantics for the trivially exact filters
// (delays, integer gains pass samples bit for bit) and confines a NaN/Inf input sample to K outputs instead of a
// transform block.  B200C_FIR_ALGO=fft forces the fused path from 2 taps.
constexpr size_t kFirOsAutoMinTapsFloat = 9;
constexpr size_t kFirOsAutoMinTapsResamp = 24;
// complex float32 resamplers served by fir_osp(g)_kernel: crossover against the direct kernel measured between 24 and
// 64 taps per phase for every rate pair of the sweep (profiles/r02_sweep_dispatch.jsonl); pure decimation by 4 only
// from ~192 taps; the spectral resampler (L = 3, M = 2) already wins at 16 per phase
constexpr size_t kFirOsAutoMinTapsOsp = 40;
constexpr size_t kFirOsAutoMinTapsOspDecim4 = 192;
constexpr size_t kFirOsAutoMinTapsX32 = 16;
// general kernel with L >= 5 (one inverse transform per output slot): wins only from ~128 taps per phase at L = 8 and
// never at L = 16 in the sweep
constexpr size_t kFirOsAutoMinTapsWideInterp = 112;
constexpr long long kFirOsGenMaxSpan = 400;   // general kernel: keep hop >= ~60 % of the block
constexpr size_t kFirOsGenForcedMaxInterp = 64;   // what the kernel supports (B200C_FIR_ALGO=fft)
constexpr size_t kFirOsGenMaxInterp = 8;    // measured: the direct kernel wins at L = 16 for every tap count
int fir_os_configure(FirOsPlan &p, int dtype, const double *taps, size_t ntaps, bool complex_taps, size_t M, size_t L,
                     bool force);
void fir_os_destroy(FirOsPlan &p);
const char *fir_os_kernel_name(const FirOsPlan &p);
// Filter bank: `nchan` equal-length streams `in_stride` / `out_stride` elements apart, each with its
// own tap spectrum in d_hf[chan][N] (same tap count, so same transform length and hop), one launch.
struct FirOsBatch {
    int nchan = 1;
    long long in_stride = 0, out_stride = 0;
    const void *d_hf = nullptr;
};
// Whether one batched launch can serve a bank whose channels all have this plan: complex float32, L = M = 1, a
// 1024- or 4096-point tap spectrum (d_hf1k / d_hf).  Every other plan runs channel by channel.
bool fir_os_batchable(const FirOsPlan &p);
// nq = output blocks q (= consumed / M); outputs written = nq * L
int fir_os_launch(const FirOsPlan &p, const void *d_in, size_t in_elems, void *d_out, size_t nq, int sm_count,
                  cudaStream_t stream, const FirOsBatch *batch = nullptr);

} // namespace b200c
