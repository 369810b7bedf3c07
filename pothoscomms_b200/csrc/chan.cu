// Polyphase filter-bank (PFB) channelizer: one complex float32 stream into M baseband channels.
//
// Definition (include/b200comms.h): frame t's newest sample is m_t = (ntaps-1) + t D + (D-1) and
//   y_c[t] = sum_{n < ntaps} h[n] x[m_t - n] exp(-2 pi i c (s + m_t - n) / M),
// i.e. channel c is /comms/fir_filter (real taps h, decimation D) applied to the stream mixed down by c/M.
// Grouping n = r M + p turns the exponent into a function of p alone, so per frame
//   v_p = sum_r h[r M + p] x[m_t - r M - p]     (M branch sums, ceil(ntaps/M) real-tap products each)
//   u_q = v_{(s + m_t - q) mod M}               (commutator rotation, here folded into the shared-memory address)
//   y_c = sum_q u_q exp(-2 pi i c q / M)        (one forward M-point DFT)
//
// One CTA owns T consecutive frames, all M channels, in ONE launch:
//  1. branch sums.  Thread (p, b) walks the frames t = b, b + k, b + 2k, ... (k = M / D) of its branch: frame t + k
//     needs the same samples as frame t shifted by one branch, so a register window of R = ceil(ntaps/M) samples
//     slides along the chain and every frame loads ONE new sample per branch (L1/L2 hits for the CTA overlap).
//     The window's slot indices are compile-time constants (R is a template parameter, the loop is unrolled by R).
//  2. the T transforms in shared memory: in-place radix-4 decimation in frequency (each stage = two radix-2
//     stages, natural-order input, bit-reversed output), a radix-2 stage last when log2 M is odd.
//  3. the channel-major store: channel c's T frames are one contiguous run of 8 T bytes in d_out.
// A frame's arithmetic does not depend on the tile that computes it (same sample values, same summation order,
// same transform), so a stream fed in pieces gives output bit-identical to one call.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "chan.hpp"
#include "packed.cuh"

namespace b200c {

constexpr int kChanThreads = 256;

struct ChanArgs {
    const c2 *in;
    c2 *out;
    const float *taps;        // [R][M]
    const c2 *tw;             // [M]
    long long frames;         // F
    long long out_stride;
    long long first;          // m_0 - (R-1) M: input index of frame 0's oldest window sample of branch 0
    unsigned long long phase0;   // (s + m_0) mod M
    int M, logM, D, T, logT, rs;
    int k;                    // M / D
    int segs, seg_len;        // each branch chain is cut into `segs` pieces of seg_len frames (thread parallelism)
};

template <int R>
__global__ void __launch_bounds__(kChanThreads) pfb_chan_kernel(const ChanArgs a)
{
    extern __shared__ __align__(16) c2 chan_smem[];
    const int M = a.M, D = a.D, T = a.T, rs = a.rs, tid = threadIdx.x, nthr = blockDim.x;
    c2 *S = chan_smem;                      // [T][rs]: frame t's transform
    c2 *W = chan_smem + (size_t)T * rs;     // [M] twiddles
    for (int i = tid; i < M; i += nthr) W[i] = a.tw[i];
    const long long t0 = (long long)blockIdx.x * T;
    const int nt = (int)min((long long)T, a.frames - t0);

    // ---- 1. branch sums, written to their rotated position q = (s + m_t - p) mod M
    const int k = a.k, chains = min(k, nt);
    const int items = M * chains * a.segs;
    for (int item = tid; item < items; item += nthr) {
        const int p = item & (M - 1), rest = item >> a.logM;
        const int b = rest % chains, g = rest / chains;
        const int na_all = (nt - b + k - 1) / k;            // frames of chain b inside this tile
        const int a_beg = g * a.seg_len, na = min(na_all, a_beg + a.seg_len) - a_beg;
        if (na <= 0) continue;
        c2 h[R];
#pragma unroll
        for (int r = 0; r < R; r++) { const float hv = __ldg(a.taps + r * M + p); h[r] = pk(hv, hv); }
        // sample e of the chain (e = 0 is the oldest sample of the first frame's window):
        //   x[first + (t0 + b + k a_beg) D - p + e M];  frame a_beg + i uses e = i .. i + R-1, tap r at e = i + R-1-r
        const long long zb = a.first + (t0 + b + (long long)k * a_beg) * D - p;
        auto ld = [&](int e) -> c2 { const long long i = zb + (long long)e * M; return i >= 0 ? __ldg(a.in + i) : 0ull; };
        c2 w[R];
#pragma unroll
        for (int e = 0; e < R - 1; e++) w[e] = ld(e);
        for (int a0 = 0; a0 < na; a0 += R) {
#pragma unroll
            for (int i = 0; i < R; i++) {
                if (a0 + i < na) {
                    w[(i + R - 1) % R] = ld(a0 + i + R - 1);
                    c2 acc = mul2(w[(i + R - 1) % R], h[0]);
#pragma unroll
                    for (int r = 1; r < R; r++) acc = fma2(w[(i + R - 1 - r) % R], h[r], acc);
                    const int t = b + k * (a_beg + a0 + i);
                    const int q = (int)((a.phase0 + (unsigned long long)(t0 + t) * D - (unsigned long long)p) & (M - 1));
                    S[t * rs + q] = acc;
                }
            }
        }
    }
    __syncthreads();

    // ---- 2. forward M-point DFTs, radix-4 DIF in place: (a, b, c, d) at j + {0, m, 2m, 3m} of a 4m group become
    //      X0 -> j, X2 W^2j -> j+m, X1 W^j -> j+2m, X3 W^3j -> j+3m  (W = W_4m), the two radix-2 DIF stages fused
    const int quarter = M >> 2;
    for (int m = quarter; m >= 1; m >>= 2) {
        const int logm = __ffs(m) - 1, tstep = quarter >> logm;   // W_4m^j = W_M^(j M / 4m)
        for (int bf = tid; bf < T * quarter; bf += nthr) {
            const int f = bf >> (a.logM - 2), bb = bf & (quarter - 1);
            const int j = bb & (m - 1), grp = bb >> logm;
            c2 *X = S + f * rs + grp * 4 * m + j;
            const c2 x0 = X[0], x1 = X[m], x2 = X[2 * m], x3 = X[3 * m];
            const c2 s0 = add2(x0, x2), s1 = sub2(x0, x2), s2 = add2(x1, x3), s3 = rot_p<false>(sub2(x1, x3));
            const int e = j * tstep;
            X[0] = add2(s0, s2);
            if (e == 0) {
                X[m] = sub2(s0, s2); X[2 * m] = add2(s1, s3); X[3 * m] = sub2(s1, s3);
            } else {
                X[m] = cmul_p<false>(sub2(s0, s2), W[2 * e]);
                X[2 * m] = cmul_p<false>(add2(s1, s3), W[e]);
                X[3 * m] = cmul_p<false>(sub2(s1, s3), W[3 * e]);
            }
        }
        __syncthreads();
    }
    if (a.logM & 1) {   // last radix-2 stage (span 2, twiddle 1)
        for (int bf = tid; bf < T * (M >> 1); bf += nthr) {
            const int f = bf >> (a.logM - 1), bb = bf & ((M >> 1) - 1);
            c2 *X = S + f * rs + 2 * bb;
            const c2 x0 = X[0], x1 = X[1];
            X[0] = add2(x0, x1); X[1] = sub2(x0, x1);
        }
        __syncthreads();
    }

    // ---- 3. channel-major store: y_c[t0 + t] = S[t][bitrev(c)], the T frames of one channel contiguous
    for (int e = tid; e < M * T; e += nthr) {
        const int c = e >> a.logT, t = e & (T - 1);
        if (t < nt) a.out[c * a.out_stride + t0 + t] = S[t * rs + (int)(__brev((unsigned)c) >> (32 - a.logM))];
    }
}

typedef void (*ChanKernel)(const ChanArgs);
static const ChanKernel kChanKernels[kChanMaxTapsPerBranch] = {
    pfb_chan_kernel<1>, pfb_chan_kernel<2>, pfb_chan_kernel<3>, pfb_chan_kernel<4>, pfb_chan_kernel<5>, pfb_chan_kernel<6>,
    pfb_chan_kernel<7>, pfb_chan_kernel<8>, pfb_chan_kernel<9>, pfb_chan_kernel<10>, pfb_chan_kernel<11>, pfb_chan_kernel<12>,
    pfb_chan_kernel<13>, pfb_chan_kernel<14>, pfb_chan_kernel<15>, pfb_chan_kernel<16>};

static int ilog2(size_t v) { int l = 0; while (((size_t)1 << l) < v) l++; return l; }

// Frames per CTA: a tile of about kChanTileElems elements (T M), at least 4 frames (one 32-byte sector per channel
// run); B200C_CHAN_TILE overrides the element budget for A/B runs.
constexpr size_t kChanTileElems = 8192;

int chan_plan_create(ChanPlan &p, size_t nchan, size_t decim, size_t smem_optin)
{
    p.M = (int)nchan; p.logM = ilog2(nchan); p.D = (int)decim;
    static const size_t budget = [] { const char *e = std::getenv("B200C_CHAN_TILE"); const long v = e ? std::atol(e) : 0; return v > 0 ? (size_t)v : kChanTileElems; }();
    size_t T = std::max<size_t>(4, std::min<size_t>(512, budget / nchan));
    T = (size_t)1 << ilog2(T + 1) >> 1;   // round down to a power of two
    if (T < 1) T = 1;
    auto smem_for = [&](size_t t) { return (t * (nchan + 1) + nchan) * sizeof(c2); };
    while (T > 1 && smem_for(T) > smem_optin) T >>= 1;
    if (smem_for(T) > smem_optin) { set_error("channelizer: %zu channels do not fit in shared memory", nchan); return B200C_ERR_UNSUPPORTED; }
    p.T = (int)T;
    p.smem_bytes = smem_for(T);
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

void chan_plan_destroy(ChanPlan &p)
{
    if (p.d_taps) cudaFree(p.d_taps);
    if (p.d_tw) cudaFree(p.d_tw);
    p.d_taps = nullptr; p.d_tw = nullptr; p.taps_capacity = 0;
}

int chan_set_taps(ChanPlan &p, const double *taps, size_t ntaps)
{
    const size_t M = (size_t)p.M, R = (ntaps + M - 1) / M;
    std::vector<float> tab(R * M, 0.0f);
    for (size_t n = 0; n < ntaps; n++) tab[n] = (float)taps[n];   // [r][p] = h[r M + p]
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
    p.R = (int)R;
    return B200C_OK;
}

int chan_launch(const ChanPlan &p, const void *d_in, size_t frames, uint64_t stream_index, void *d_out, size_t out_stride,
                cudaStream_t stream)
{
    const size_t M = (size_t)p.M, D = (size_t)p.D, R = (size_t)p.R, T = (size_t)p.T;
    const unsigned long long m0 = (unsigned long long)(p.ntaps - 1 + D - 1);   // newest sample of frame 0
    ChanArgs a;
    a.in = static_cast<const c2 *>(d_in);
    a.out = static_cast<c2 *>(d_out);
    a.taps = p.d_taps;
    a.tw = static_cast<const c2 *>(p.d_tw);
    a.frames = (long long)frames;
    a.out_stride = (long long)out_stride;
    a.first = (long long)m0 - (long long)((R - 1) * M);
    a.phase0 = ((unsigned long long)stream_index + m0) & (M - 1);
    a.M = p.M; a.logM = p.logM; a.D = p.D; a.T = p.T; a.logT = ilog2(T); a.rs = p.M + 1;
    a.k = (int)(M / D);
    // cut the branch chains until every thread has one (a cut costs R-1 extra window loads)
    const size_t chains = std::min<size_t>(M / D, T), chain_len = (T + M / D - 1) / (M / D);
    size_t segs = std::max<size_t>(1, (size_t)kChanThreads / (M * chains));
    segs = std::min(segs, chain_len);
    a.seg_len = (int)((chain_len + segs - 1) / segs);
    a.segs = (int)((chain_len + a.seg_len - 1) / a.seg_len);
    const ChanKernel kern = kChanKernels[R - 1];
    if (p.smem_bytes > 48 * 1024)
        B200C_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bytes));
    const size_t grid = (frames + T - 1) / T;
    if (grid > 0x7fffffffu) { set_error("channelizer: %zu frames exceed one launch", frames); return B200C_ERR_INVALID; }
    kern<<<(unsigned)grid, kChanThreads, p.smem_bytes, stream>>>(a);
    B200C_CUDA_TRY(cudaGetLastError());
    return B200C_OK;
}

} // namespace b200c
