// Polyphase synthesis filter bank: M baseband channels back into one complex float32 stream (the transpose of chan.cu).
//
// Definition (include/b200comms.h): with K = ceil(ntaps / D) and s = stream_index, output sample m = t D + j (j < D) is
//   y[t D + j] = sum_{c < M} exp(+2 pi i c (s + t D + j) / M) sum_{k < K} g[j + k D] X_c[K-1 + t - k]
// (g zero beyond ntaps), i.e. channel c is /comms/fir_filter with real taps g and interpolation D, mixed up by c/M and
// summed over c.  The exponent depends on the output sample only, so with one inverse M-point DFT per input frame,
//   V_i[q] = sum_c X_c[i] exp(+2 pi i c q / M),
//   y[t D + j] = sum_k g[j + k D] V_{K-1+t-k}[(s + t D + j) mod M].
// Output sample m reads bin q = (s + m) mod M, so the bin fixes j = (q - s) mod D and t mod (M/D): thread l < M owns
// bin (s + l) mod M and emits the samples t D + j with j = l mod D and t = l / D (mod M/D).  Along its bin the frames
// arrive in order, so a K-frame register window slides by one frame per input frame and every frame is loaded from
// shared memory once per bin.
//
// One CTA owns T consecutive output frames (T D samples) and the bins [blockIdx.y B, blockIdx.y B + B) in ONE launch.
// It walks its T + K - 1 input frames in chunks of P:
//  1. cp.async copies chunk c + 1 (P frames of every channel; channel c's frames are one contiguous run) into the
//     other of two shared-memory buffers while chunk c is transformed and consumed.  Channel ch lands in slot
//     bitrev(ch), the input order of a decimation-in-time transform.
//  2. the P inverse DFTs in place: a radix-2 stage first when log2 M is odd, then fused radix-4 DIT stages (bfly4_p of
//     packed.cuh with conjugated twiddles and the +i rotation), natural-order output.  Natural order makes the bin
//     read of step 3 conflict-free and the output store coalesced: consecutive threads read consecutive bins and
//     write consecutive samples.
//  3. each owner thread pushes V_i[q] into its window and, when the window ends an output frame of its chain, forms
//     the K-term sum and stores the sample.  The D samples of one output frame are one contiguous run.
// The window holds 3 K registers per bin (K samples, K taps); above 1024 bins per CTA (M = 2048, 4096) or when the
// window outgrows the per-thread register share, the bins are split over gridDim.y CTAs, each of which recomputes the
// whole transform.  A sample's arithmetic does not depend on the tile or the bin group that computes it (same frames,
// same transform, same summation order), so a stream fed in pieces gives output bit-identical to one call.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "packed.cuh"
#include "synth.hpp"

namespace b200c {

// register budget of the window: 2 K + K registers per bin plus addressing must fit 65536 / threads
constexpr int synth_max_threads(int K) { return K <= 8 ? 1024 : K <= 16 ? 512 : 256; }

struct SynthArgs {
    const c2 *in;
    c2 *out;
    const float *taps;        // [K][D]
    const c2 *tw;             // [M]
    long long in_stride;
    long long frames;         // F output frames
    unsigned s;               // stream_index mod M
    int M, logM, D, logD;
    int kmask;                // M / D - 1
    int T, P, logP, rs, B;
};

__device__ __forceinline__ void cp_async8(c2 *dst, const c2 *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

template <int K>
__global__ void __launch_bounds__(synth_max_threads(K), 1) pfb_synth_kernel(const SynthArgs a)
{
    extern __shared__ __align__(16) c2 synth_smem[];
    const int M = a.M, P = a.P, rs = a.rs, tid = threadIdx.x, nthr = blockDim.x;
    c2 *W = synth_smem;                     // [M] twiddles exp(-2 pi i k / M)
    c2 *buf = synth_smem + M;               // [2][P][rs]: two chunk buffers
    for (int i = tid; i < M; i += nthr) W[i] = a.tw[i];
    const long long t0 = (long long)blockIdx.x * a.T;
    const int nt = (int)min((long long)a.T, a.frames - t0);
    const int nr = nt + K - 1;              // input frames t0 .. t0 + nr - 1
    const int nchunks = (nr + P - 1) >> a.logP;

    // this thread's bin q and the output phase it feeds
    const bool owner = tid < a.B;
    const int l = blockIdx.y * a.B + (owner ? tid : 0);
    const int q = (int)((a.s + (unsigned)l) & (unsigned)(M - 1));
    const int j = l & (a.D - 1), b = l >> a.logD;
    float g[K];
#pragma unroll
    for (int k = 0; k < K; k++) g[k] = __ldg(a.taps + k * a.D + j);

    auto load = [&](int c) {   // chunk c -> buffer c & 1; frame f of channel ch at [f][bitrev(ch)]
        c2 *S = buf + (size_t)(c & 1) * P * rs;
        const int f0 = c << a.logP, nf = min(P, nr - f0);
        for (int e = tid; e < M * P; e += nthr) {
            const int f = e & (P - 1), ch = e >> a.logP;
            if (f < nf)
                cp_async8(S + f * rs + (int)(__brev((unsigned)ch) >> (32 - a.logM)), a.in + ch * a.in_stride + t0 + f0 + f);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto transform = [&](c2 *S) {   // P inverse DFTs in place, bit-reversed in, natural order out
        int m = 1;
        if (a.logM & 1) {   // radix-2 stage, span 1, twiddle 1
            for (int bf = tid; bf < P * (M >> 1); bf += nthr) {
                const int f = bf >> (a.logM - 1), bb = bf & ((M >> 1) - 1);
                c2 *X = S + f * rs + 2 * bb;
                const c2 x0 = X[0], x1 = X[1];
                X[0] = add2(x0, x1); X[1] = sub2(x0, x1);
            }
            __syncthreads();
            m = 2;
        }
        // fused radix-4 DIT: spans m and 2m; (x[j], x[j+2m] w, x[j+m] w^2, x[j+3m] w^3) through the 4-point IDFT go
        // to j, j+m, j+2m, j+3m, with w = W_4m^-j = conj(W_M^(j M / 4m))
        for (; 4 * m <= M; m <<= 2) {
            const int logm = __ffs(m) - 1, tstep = (M >> 2) >> logm;
            for (int bf = tid; bf < P * (M >> 2); bf += nthr) {
                const int f = bf >> (a.logM - 2), bb = bf & ((M >> 2) - 1);
                const int jj = bb & (m - 1), grp = bb >> logm;
                c2 *X = S + f * rs + grp * 4 * m + jj;
                c2 f0 = X[0], f1 = X[2 * m], f2 = X[m], f3 = X[3 * m];
                if (m == 1) {
                    dft4_p<true>(f0, f1, f2, f3);
                } else {
                    const int e = jj * tstep;
                    bfly4_p<true, true>(f0, f1, f2, f3, W[e], W[2 * e], W[3 * e]);
                }
                X[0] = f0; X[m] = f1; X[2 * m] = f2; X[3 * m] = f3;
            }
            __syncthreads();
        }
    };

    c2 w[K];
#pragma unroll
    for (int k = 0; k < K; k++) w[k] = 0ull;
    load(0);
    const c2 *S = buf;
    // frame r of the tile sits in window slot r mod K: the loop is unrolled by K so every slot is a fixed register
    for (int rb = 0; rb < nr; rb += K) {
#pragma unroll
        for (int u = 0; u < K; u++) {
            const int r = rb + u;
            if (r < nr) {
                if ((r & (P - 1)) == 0) {   // a new chunk (uniform over the CTA)
                    const int c = r >> a.logP;
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                    __syncthreads();        // chunk c has landed and nobody still reads chunk c - 1's buffer
                    if (c + 1 < nchunks) load(c + 1);
                    c2 *Sc = buf + (size_t)(c & 1) * P * rs;
                    transform(Sc);
                    S = Sc;
                }
                if (owner) {
                    w[u] = S[(r & (P - 1)) * rs + q];
                    const int tr = r - (K - 1);
                    if (tr >= 0 && (int)((t0 + tr) & a.kmask) == b) {
                        c2 acc = mul2(w[u], pk(g[0], g[0]));
#pragma unroll
                        for (int k = 1; k < K; k++) acc = fma2(w[(u - k + K) % K], pk(g[k], g[k]), acc);
                        a.out[(t0 + tr) * a.D + j] = acc;
                    }
                }
            }
        }
    }
}

typedef void (*SynthKernel)(const SynthArgs);
static const SynthKernel kSynthKernels[kSynthMaxTapsPerPhase] = {
    pfb_synth_kernel<1>, pfb_synth_kernel<2>, pfb_synth_kernel<3>, pfb_synth_kernel<4>, pfb_synth_kernel<5>,
    pfb_synth_kernel<6>, pfb_synth_kernel<7>, pfb_synth_kernel<8>, pfb_synth_kernel<9>, pfb_synth_kernel<10>,
    pfb_synth_kernel<11>, pfb_synth_kernel<12>, pfb_synth_kernel<13>, pfb_synth_kernel<14>, pfb_synth_kernel<15>,
    pfb_synth_kernel<16>, pfb_synth_kernel<17>, pfb_synth_kernel<18>, pfb_synth_kernel<19>, pfb_synth_kernel<20>,
    pfb_synth_kernel<21>, pfb_synth_kernel<22>, pfb_synth_kernel<23>, pfb_synth_kernel<24>, pfb_synth_kernel<25>,
    pfb_synth_kernel<26>, pfb_synth_kernel<27>, pfb_synth_kernel<28>, pfb_synth_kernel<29>, pfb_synth_kernel<30>,
    pfb_synth_kernel<31>, pfb_synth_kernel<32>};

static int ilog2(size_t v) { int l = 0; while (((size_t)1 << l) < v) l++; return l; }

// Frames per chunk: about kSynthChunkElems elements (P M) per buffer, at most 16 frames.
constexpr size_t kSynthChunkElems = 8192;

int synth_plan_create(SynthPlan &p, size_t nchan, size_t interp, size_t smem_optin)
{
    p.M = (int)nchan; p.logM = ilog2(nchan); p.D = (int)interp; p.logD = ilog2(interp);
    size_t P = std::max<size_t>(1, std::min<size_t>(16, kSynthChunkElems / nchan));
    auto smem_for = [&](size_t f) { return (2 * f * (nchan + 1) + nchan) * sizeof(c2); };
    while (P > 1 && smem_for(P) > smem_optin) P >>= 1;
    if (smem_for(P) > smem_optin) { set_error("synthesizer: %zu channels do not fit in shared memory", nchan); return B200C_ERR_UNSUPPORTED; }
    p.P = (int)P;
    p.smem_bytes = smem_for(P);
    std::vector<float> tw(2 * nchan);
    for (size_t i = 0; i < nchan; i++) {
        const double ph = -2.0 * M_PI * (double)i / (double)nchan;
        tw[2 * i] = (float)std::cos(ph);
        tw[2 * i + 1] = (float)std::sin(ph);
    }
    B200C_CUDA_TRY(cudaMalloc(&p.d_tw, tw.size() * sizeof(float)));
    B200C_CUDA_TRY(cudaMemcpy(p.d_tw, tw.data(), tw.size() * sizeof(float), cudaMemcpyHostToDevice));
    return B200C_OK;
}

void synth_plan_destroy(SynthPlan &p)
{
    if (p.d_taps) cudaFree(p.d_taps);
    if (p.d_tw) cudaFree(p.d_tw);
    p.d_taps = nullptr; p.d_tw = nullptr; p.taps_capacity = 0;
}

int synth_set_taps(SynthPlan &p, const double *taps, size_t ntaps)
{
    const size_t D = (size_t)p.D, K = (ntaps + D - 1) / D;
    std::vector<float> tab(K * D, 0.0f);
    for (size_t n = 0; n < ntaps; n++) tab[n] = (float)taps[n];   // [k][j] = g[k D + j]
    const size_t bytes = tab.size() * sizeof(float);
    if (bytes > p.taps_capacity) {
        if (p.d_taps) cudaFree(p.d_taps);
        p.d_taps = nullptr; p.taps_capacity = 0;
        B200C_CUDA_TRY(cudaMalloc((void **)&p.d_taps, bytes));
        p.taps_capacity = bytes;
    }
    // a control-path call: the blocking copy also orders against in-flight runs on the legacy stream
    B200C_CUDA_TRY(cudaDeviceSynchronize());
    B200C_CUDA_TRY(cudaMemcpy(p.d_taps, tab.data(), bytes, cudaMemcpyHostToDevice));
    p.ntaps = ntaps;
    p.K = (int)K;
    p.B = std::min(p.M, synth_max_threads((int)K));
    // output frames per CTA: the K - 1 overlap frames each tile transforms again cost (K - 1) / T extra transforms;
    // T = 16 (K - 1) keeps that at 1/16.  B200C_SYNTH_TILE overrides T for A/B runs.
    static const long tile_env = [] { const char *e = std::getenv("B200C_SYNTH_TILE"); return e ? std::atol(e) : 0L; }();
    p.T = tile_env > 0 ? (int)tile_env : std::max(4 * p.P, 16 * ((int)K - 1));
    return B200C_OK;
}

int synth_launch(const SynthPlan &p, const void *d_in, size_t in_stride, size_t frames, uint64_t stream_index, void *d_out,
                 cudaStream_t stream)
{
    SynthArgs a;
    a.in = static_cast<const c2 *>(d_in);
    a.out = static_cast<c2 *>(d_out);
    a.taps = p.d_taps;
    a.tw = static_cast<const c2 *>(p.d_tw);
    a.in_stride = (long long)in_stride;
    a.frames = (long long)frames;
    a.s = (unsigned)(stream_index & (uint64_t)(p.M - 1));
    a.M = p.M; a.logM = p.logM; a.D = p.D; a.logD = p.logD;
    a.kmask = p.M / p.D - 1;
    a.T = p.T; a.P = p.P; a.logP = ilog2((size_t)p.P); a.rs = p.M + 1; a.B = p.B;
    const SynthKernel kern = kSynthKernels[p.K - 1];
    if (p.smem_bytes > 48 * 1024)
        B200C_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bytes));
    const size_t grid = (frames + (size_t)p.T - 1) / (size_t)p.T;
    if (grid > 0x7fffffffu) { set_error("synthesizer: %zu frames exceed one launch", frames); return B200C_ERR_INVALID; }
    const dim3 g((unsigned)grid, (unsigned)(p.M / p.B));
    kern<<<g, std::max(p.B, 32), p.smem_bytes, stream>>>(a);
    B200C_CUDA_TRY(cudaGetLastError());
    return B200C_OK;
}

} // namespace b200c
