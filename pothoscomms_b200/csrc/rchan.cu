// Real-input polyphase filter-bank channelizer: one real float32 or int16 stream into M/2 + 1 baseband channels.
//
// Definition (include/b200comms.h): the complex channelizer's (chan.cu) applied to a real stream x, keeping the
// channels c = 0 .. M/2; the others are conj(y_{M-c}).  Per frame, with N = M/2:
//   v_p = sum_r h[r M + p] x[m_t - r M - p]     (M real branch sums, ceil(ntaps/M) scalar products each)
//   u_q = v_{(s + m_t - q) mod M}               (commutator rotation, folded into the shared-memory address)
//   z_r = u_{2r} + i u_{2r+1}                   (the real frame packed into N complex slots, r < N)
//   Z_k = sum_r z_r exp(-2 pi i k r / N)        (one forward N-point DFT)
//   E = (Z_c + conj Z_{N-c}) / 2,  O = (Z_c - conj Z_{N-c}) / (2i),  y_c = E + W_M^c O,  y_{N-c} = conj(E - W_M^c O)
// with Z_N = Z_0, so y_0 = Re Z_0 + Im Z_0 and y_N = Re Z_0 - Im Z_0 (both written with imaginary part exactly 0).
// A frame is packed into its own transform, never paired with a neighbour frame, so its rounding does not depend
// on where a call starts or ends: a stream fed in pieces gives output bit-identical to one call.
//
// One CTA owns T consecutive frames, all M/2 + 1 channels, in ONE launch:
//  1. branch sums, as pfb_chan_kernel: thread (p, b) slides a register window of R = ceil(ntaps/M) samples along
//     the chain of frames t = b, b + k, ... (k = M / D) of branch p, one new sample per frame; the sample loads
//     convert float32 or int16 (exactly) to float.  u_q is written as float q of the frame's slots.
//  2. the T N-point transforms in shared memory: radix-4 decimation in frequency as pfb_chan_kernel (natural-order
//     input, bit-reversed output), radix-2 last when log2 N is odd, twiddles W_N^k = W_M^2k from the M-point table.
//  3. the split and the channel-major store: thread (c, t), c <= N/2, reads Z_c and Z_{N-c} of frame t and writes
//     y_c[t] and y_{N-c}[t]; each channel's T frames are one contiguous run of 8 T bytes in d_out.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <vector>

#include "packed.cuh"
#include "rchan.hpp"

namespace b200c {

constexpr int kRChanThreads = 256;

struct RChanArgs {
    const void *in;
    c2 *out;
    const float *taps;        // [R][M]
    const c2 *tw;             // [M] W_M^k
    long long frames;         // F
    long long out_stride;
    long long first;          // m_0 - (R-1) M: input index of frame 0's oldest window sample of branch 0
    unsigned long long phase0;   // (s + m_0) mod M
    int M, logM, D, T, logT, rs;
    int k;                    // M / D
    int segs, seg_len;        // each branch chain is cut into `segs` pieces of seg_len frames (thread parallelism)
};

template <int R, typename In>
__global__ void __launch_bounds__(kRChanThreads) pfb_rchan_kernel(const RChanArgs a)
{
    extern __shared__ __align__(16) c2 rchan_smem[];
    const int M = a.M, N = M >> 1, logN = a.logM - 1, D = a.D, T = a.T, rs = a.rs, tid = threadIdx.x, nthr = blockDim.x;
    c2 *S = rchan_smem;                     // [T][rs]: frame t's packed real frame, then its N-point transform
    c2 *W = rchan_smem + (size_t)T * rs;    // [M] twiddles W_M^k
    for (int i = tid; i < M; i += nthr) W[i] = a.tw[i];
    const long long t0 = (long long)blockIdx.x * T;
    const int nt = (int)min((long long)T, a.frames - t0);
    const In *in = static_cast<const In *>(a.in);

    // ---- 1. branch sums, written to float q = (s + m_t - p) mod M of the frame: even q the real part of slot q/2,
    //      odd q its imaginary part
    float *Sf = reinterpret_cast<float *>(S);
    const int k = a.k, chains = min(k, nt);
    const int items = M * chains * a.segs;
    for (int item = tid; item < items; item += nthr) {
        const int p = item & (M - 1), rest = item >> a.logM;
        const int b = rest % chains, g = rest / chains;
        const int na_all = (nt - b + k - 1) / k;            // frames of chain b inside this tile
        const int a_beg = g * a.seg_len, na = min(na_all, a_beg + a.seg_len) - a_beg;
        if (na <= 0) continue;
        float h[R];
#pragma unroll
        for (int r = 0; r < R; r++) h[r] = __ldg(a.taps + r * M + p);
        // sample e of the chain (e = 0 is the oldest sample of the first frame's window):
        //   x[first + (t0 + b + k a_beg) D - p + e M];  frame a_beg + i uses e = i .. i + R-1, tap r at e = i + R-1-r
        const long long zb = a.first + (t0 + b + (long long)k * a_beg) * D - p;
        auto ld = [&](int e) -> float { const long long i = zb + (long long)e * M; return i >= 0 ? (float)__ldg(in + i) : 0.0f; };
        float w[R];
#pragma unroll
        for (int e = 0; e < R - 1; e++) w[e] = ld(e);
        for (int a0 = 0; a0 < na; a0 += R) {
#pragma unroll
            for (int i = 0; i < R; i++) {
                if (a0 + i < na) {
                    w[(i + R - 1) % R] = ld(a0 + i + R - 1);
                    float acc = w[(i + R - 1) % R] * h[0];
#pragma unroll
                    for (int r = 1; r < R; r++) acc = fmaf(w[(i + R - 1 - r) % R], h[r], acc);
                    const int t = b + k * (a_beg + a0 + i);
                    const int q = (int)((a.phase0 + (unsigned long long)(t0 + t) * D - (unsigned long long)p) & (M - 1));
                    Sf[2 * t * rs + q] = acc;
                }
            }
        }
    }
    __syncthreads();

    // ---- 2. forward N-point DFTs, radix-4 DIF in place: (a, b, c, d) at j + {0, m, 2m, 3m} of a 4m group become
    //      X0 -> j, X2 W^2j -> j+m, X1 W^j -> j+2m, X3 W^3j -> j+3m  (W = W_4m = W_M^(2 N / 4m)), the two radix-2
    //      DIF stages fused
    const int quarter = N >> 2;
    for (int m = quarter; m >= 1; m >>= 2) {
        const int logm = __ffs(m) - 1, tstep = quarter >> logm;   // W_4m^j = W_N^(j N / 4m) = W_M^(2 j N / 4m)
        for (int bf = tid; bf < T * quarter; bf += nthr) {
            const int f = bf >> (logN - 2), bb = bf & (quarter - 1);
            const int j = bb & (m - 1), grp = bb >> logm;
            c2 *X = S + f * rs + grp * 4 * m + j;
            const c2 x0 = X[0], x1 = X[m], x2 = X[2 * m], x3 = X[3 * m];
            const c2 s0 = add2(x0, x2), s1 = sub2(x0, x2), s2 = add2(x1, x3), s3 = rot_p<false>(sub2(x1, x3));
            const int e = 2 * j * tstep;
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
    if (logN & 1) {   // last radix-2 stage (span 2, twiddle 1)
        for (int bf = tid; bf < T * (N >> 1); bf += nthr) {
            const int f = bf >> (logN - 1), bb = bf & ((N >> 1) - 1);
            c2 *X = S + f * rs + 2 * bb;
            const c2 x0 = X[0], x1 = X[1];
            X[0] = add2(x0, x1); X[1] = sub2(x0, x1);
        }
        __syncthreads();
    }

    // ---- 3. split and channel-major store: Z_k of frame t sits at S[t][bitrev(k)]
    auto slot = [&](int kk) { return logN ? (int)(__brev((unsigned)kk) >> (32 - logN)) : 0; };
    const long long os = a.out_stride;
    for (int e = tid; e < ((N >> 1) + 1) * T; e += nthr) {
        const int c = e >> a.logT, t = e & (T - 1);
        if (t >= nt) continue;
        const c2 *Z = S + t * rs;
        float ar, ai, br, bi;
        upk(Z[slot(c)], ar, ai);
        upk(Z[slot((N - c) & (N - 1))], br, bi);
        c2 *o = a.out + t0 + t;
        if (c == 0) {   // E = Re Z_0, O = Im Z_0
            o[0] = pk(ar + ai, 0.0f);
            o[N * os] = pk(ar - ai, 0.0f);
        } else {
            const c2 E = pk(0.5f * (ar + br), 0.5f * (ai - bi));
            const c2 O = pk(0.5f * (ai + bi), 0.5f * (br - ar));
            const c2 WO = cmul_p<false>(O, W[c]);
            o[c * os] = add2(E, WO);
            if (2 * c != N) {
                float dr, di;
                upk(sub2(E, WO), dr, di);
                o[(N - c) * os] = pk(dr, -di);
            }
        }
    }
}

typedef void (*RChanKernel)(const RChanArgs);
template <typename In>
static RChanKernel rchan_kernel(size_t R)
{
    static const RChanKernel k[kChanMaxTapsPerBranch] = {
        pfb_rchan_kernel<1, In>, pfb_rchan_kernel<2, In>, pfb_rchan_kernel<3, In>, pfb_rchan_kernel<4, In>,
        pfb_rchan_kernel<5, In>, pfb_rchan_kernel<6, In>, pfb_rchan_kernel<7, In>, pfb_rchan_kernel<8, In>,
        pfb_rchan_kernel<9, In>, pfb_rchan_kernel<10, In>, pfb_rchan_kernel<11, In>, pfb_rchan_kernel<12, In>,
        pfb_rchan_kernel<13, In>, pfb_rchan_kernel<14, In>, pfb_rchan_kernel<15, In>, pfb_rchan_kernel<16, In>};
    return k[R - 1];
}

static int ilog2(size_t v) { int l = 0; while (((size_t)1 << l) < v) l++; return l; }

// Frames per CTA: a tile of about kRChanTileSlots complex slots (T M/2, the complex channelizer's 64 KiB tile), at
// least 4 frames (one 32-byte sector per channel run)
constexpr size_t kRChanTileSlots = 8192;

int rchan_plan_create(ChanPlan &p, size_t m, size_t decim, size_t smem_optin)
{
    const size_t N = m / 2;
    p.M = (int)m; p.logM = ilog2(m); p.D = (int)decim;
    size_t T = std::max<size_t>(4, std::min<size_t>(512, kRChanTileSlots / N));
    T = (size_t)1 << ilog2(T + 1) >> 1;   // round down to a power of two
    auto smem_for = [&](size_t t) { return (t * (N + 1) + m) * sizeof(c2); };
    while (T > 1 && smem_for(T) > smem_optin) T >>= 1;
    if (smem_for(T) > smem_optin) { set_error("real channelizer: %zu branches do not fit in shared memory", m); return B200C_ERR_UNSUPPORTED; }
    p.T = (int)T;
    p.smem_bytes = smem_for(T);
    std::vector<float> tw(2 * m);
    for (size_t i = 0; i < m; i++) {
        const double ph = -2.0 * M_PI * (double)i / (double)m;
        tw[2 * i] = (float)std::cos(ph);
        tw[2 * i + 1] = (float)std::sin(ph);
    }
    B200C_CUDA_TRY(cudaMalloc(&p.d_tw, tw.size() * sizeof(float)));
    B200C_CUDA_TRY(cudaMemcpy(p.d_tw, tw.data(), tw.size() * sizeof(float), cudaMemcpyHostToDevice));
    return B200C_OK;
}

int rchan_launch(const ChanPlan &p, int dtype, const void *d_in, size_t frames, uint64_t stream_index, void *d_out,
                 size_t out_stride, cudaStream_t stream)
{
    const size_t M = (size_t)p.M, D = (size_t)p.D, R = (size_t)p.R, T = (size_t)p.T;
    const unsigned long long m0 = (unsigned long long)(p.ntaps - 1 + D - 1);   // newest sample of frame 0
    RChanArgs a;
    a.in = d_in;
    a.out = static_cast<c2 *>(d_out);
    a.taps = p.d_taps;
    a.tw = static_cast<const c2 *>(p.d_tw);
    a.frames = (long long)frames;
    a.out_stride = (long long)out_stride;
    a.first = (long long)m0 - (long long)((R - 1) * M);
    a.phase0 = ((unsigned long long)stream_index + m0) & (M - 1);
    a.M = p.M; a.logM = p.logM; a.D = p.D; a.T = p.T; a.logT = ilog2(T); a.rs = p.M / 2 + 1;
    a.k = (int)(M / D);
    // cut the branch chains until every thread has one (a cut costs R-1 extra window loads)
    const size_t chains = std::min<size_t>(M / D, T), chain_len = (T + M / D - 1) / (M / D);
    size_t segs = std::max<size_t>(1, (size_t)kRChanThreads / (M * chains));
    segs = std::min(segs, chain_len);
    a.seg_len = (int)((chain_len + segs - 1) / segs);
    a.segs = (int)((chain_len + a.seg_len - 1) / a.seg_len);
    const RChanKernel kern = dtype == B200C_I16 ? rchan_kernel<int16_t>(R) : rchan_kernel<float>(R);
    if (p.smem_bytes > 48 * 1024)
        B200C_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bytes));
    const size_t grid = (frames + T - 1) / T;
    if (grid > 0x7fffffffu) { set_error("real channelizer: %zu frames exceed one launch", frames); return B200C_ERR_INVALID; }
    kern<<<(unsigned)grid, kRChanThreads, p.smem_bytes, stream>>>(a);
    B200C_CUDA_TRY(cudaGetLastError());
    return B200C_OK;
}

} // namespace b200c
