// Real-output polyphase synthesis filter bank: M/2 + 1 baseband channels back into one real float32 or int16 stream
// (the transpose of rchan.cu).
//
// Definition (include/b200comms.h): with N = M/2, K = ceil(ntaps / D) and s = stream_index, output sample m = t D + j
// (j < D) is the real part of the complex synthesizer's (synth.cu) output at M channels, where rows 0 .. N are given
// and row M - c is conj(X_c) for 0 < c < N:
//   y[t D + j] = sum_k g[j + k D] V_{K-1+t-k}[(s + t D + j) mod M],
//   V_i[q] = sum_{c = 0..N} w_c Re(exp(+2 pi i c q / M) X_c[i]),   w_0 = w_N = 1, w_c = 2 otherwise.
// V_i is the real inverse M-point DFT of the conjugate-symmetric frame, computed as ONE N-point complex inverse DFT
// (the inverse of rchan.cu's even/odd split):
//   Z_k = (X_k + conj X_{N-k}) + i exp(+2 pi i k / M) (X_k - conj X_{N-k}),   1 <= k < N
//   Z_0 = (Re X_0 + Re X_N) + i (Re X_0 - Re X_N)
//   z = unnormalised inverse N-point DFT of Z;   V[2r] = Re z_r,  V[2r+1] = Im z_r
// so the M real bins of a frame are the 2N floats of its transform in natural order.  Only the real parts of rows 0
// and N are read.  As in synth.cu, output sample m reads bin q = (s + m) mod M: thread l owns real bin (s + l) mod M
// and emits the samples t D + j with j = l mod D and t = l / D (mod M/D), sliding a K-float register window along
// its bin.
//
// One CTA owns T consecutive output frames (T D samples) and the real bins [blockIdx.y B, blockIdx.y B + B) in ONE
// launch.  It walks its T + K - 1 input frames in chunks of P:
//  1. cp.async copies chunk c + 1 (P frames of every row; row c's frames are one contiguous run) into the other of
//     two shared-memory buffers while chunk c is transformed and consumed.  Row c < N lands in slot bitrev_N(c), the
//     input order of a decimation-in-time transform; row N lands in the spare slot N.
//  2. the pre-pass: for each pair k <= N/2 one thread reads the slots of X_k and X_{N-k} (X_0 and X_N for k = 0) and
//     writes Z_k and Z_{N-k} over them, in place; threads are laid out by slot, so the accesses are conflict-free.
//  3. the P inverse N-point DFTs in place, as synth.cu's: a radix-2 stage first when log2 N is odd, then fused
//     radix-4 DIT stages with twiddles W_N^e = W_M^2e from the M-point table, natural-order output.  Consecutive
//     threads then read consecutive floats (real bins) and write consecutive samples.
//  4. each owner thread pushes V_i[q] into its window and, when the window ends an output frame of its chain, forms
//     the K-term sum and stores the sample (float32, or int16 rounded to nearest even and saturated).
// The window holds 2 K registers per bin (K samples, K taps); above 1024 bins per CTA, or when the window outgrows the
// per-thread register share, the bins are split over gridDim.y CTAs, each of which recomputes the whole transform.  A
// frame is never packed with another one, and a sample's arithmetic does not depend on the tile or the bin group
// that computes it, so a stream fed in pieces gives output bit-identical to one call.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <vector>

#include "packed.cuh"
#include "rsynth.hpp"

namespace b200c {

// register budget of the window: K + K registers per bin plus addressing must fit 65536 / threads (synth.cu's share
// per window register)
constexpr int rsynth_max_threads(int K) { return K <= 12 ? 1024 : K <= 24 ? 512 : 256; }

struct RSynthArgs {
    const c2 *in;
    void *out;
    const float *taps;        // [K][D]
    const c2 *tw;             // [M] W_M^k = exp(-2 pi i k / M)
    long long in_stride;
    long long frames;         // F output frames
    unsigned s;               // stream_index mod M
    int M, logN, D, logD;
    int kmask;                // M / D - 1
    int T, P, logP, rs, B;
};

__device__ __forceinline__ void rsynth_cp_async8(c2 *dst, const c2 *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

__device__ __forceinline__ void rsynth_store(float *o, float v) { *o = v; }
__device__ __forceinline__ void rsynth_store(int16_t *o, float v) { *o = (int16_t)min(max(__float2int_rn(v), -32768), 32767); }

template <int K, typename Out>
__global__ void __launch_bounds__(rsynth_max_threads(K), 1) pfb_rsynth_kernel(const RSynthArgs a)
{
    extern __shared__ __align__(16) c2 rsynth_smem[];
    const int M = a.M, N = M >> 1, logN = a.logN, P = a.P, rs = a.rs, tid = threadIdx.x, nthr = blockDim.x;
    c2 *W = rsynth_smem;                    // [M] twiddles W_M^k
    c2 *buf = rsynth_smem + M;              // [2][P][rs]: two chunk buffers, N slots + row N per frame
    for (int i = tid; i < M; i += nthr) W[i] = a.tw[i];
    const long long t0 = (long long)blockIdx.x * a.T;
    const int nt = (int)min((long long)a.T, a.frames - t0);
    const int nr = nt + K - 1;              // input frames t0 .. t0 + nr - 1
    const int nchunks = (nr + P - 1) >> a.logP;
    auto slot = [&](int c) { return logN ? (int)(__brev((unsigned)c) >> (32 - logN)) : 0; };

    // this thread's real bin q and the output phase it feeds
    const bool owner = tid < a.B;
    const int l = blockIdx.y * a.B + (owner ? tid : 0);
    const int q = (int)((a.s + (unsigned)l) & (unsigned)(M - 1));
    const int j = l & (a.D - 1), b = l >> a.logD;
    float g[K];
#pragma unroll
    for (int k = 0; k < K; k++) g[k] = __ldg(a.taps + k * a.D + j);

    auto load = [&](int c) {   // chunk c -> buffer c & 1; frame f of row ch at [f][bitrev(ch)], row N at [f][N]
        c2 *S = buf + (size_t)(c & 1) * P * rs;
        const int f0 = c << a.logP, nf = min(P, nr - f0);
        for (int e = tid; e < (N + 1) * P; e += nthr) {
            const int f = e & (P - 1), ch = e >> a.logP;
            if (f < nf) rsynth_cp_async8(S + f * rs + (ch < N ? slot(ch) : N), a.in + ch * a.in_stride + t0 + f0 + f);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto transform = [&](c2 *S) {   // P packed inverse DFTs in place, bit-reversed in, natural order out
        // pre-pass: (X_k, X_{N-k}) -> (Z_k, Z_{N-k}) in their own slots; with d = X_k - conj X_{N-k} and
        // r = d exp(+2 pi i k / M): Z_k = (X_k + conj X_{N-k}) + i r, Z_{N-k} = conj(X_k + conj X_{N-k}) + i conj(r).
        // Thread e takes slot p = e mod N, k = bitrev(p), and does the pair when k <= N/2: consecutive threads then
        // touch consecutive slots and partner slots bitrev(N - k) on distinct banks (consecutive k would put a
        // half-warp's bit-reversed slots on one bank)
        for (int e = tid; e < P * N; e += nthr) {
            const int f = e >> logN, p = e & (N - 1), k = slot(p);
            c2 *X = S + f * rs;
            if (k == 0) {
                float a0, b0, an, bn;
                upk(X[0], a0, b0); upk(X[N], an, bn);
                X[0] = pk(a0 + an, a0 - an);
            } else if (2 * k <= N) {
                const int sa = p, sb = slot(N - k);
                float xr, xi, yr, yi;
                upk(X[sa], xr, xi); upk(X[sb], yr, yi);
                const c2 r = cmul_p<true>(pk(xr - yr, xi + yi), W[k]);
                float rr, ri;
                upk(r, rr, ri);
                const float sr = xr + yr, si = xi - yi;
                X[sa] = pk(sr - ri, si + rr);
                if (sb != sa) X[sb] = pk(sr + ri, rr - si);
            }
        }
        __syncthreads();
        int m = 1;
        if (logN & 1) {   // radix-2 stage, span 1, twiddle 1
            for (int bf = tid; bf < P * (N >> 1); bf += nthr) {
                const int f = bf >> (logN - 1), bb = bf & ((N >> 1) - 1);
                c2 *X = S + f * rs + 2 * bb;
                const c2 x0 = X[0], x1 = X[1];
                X[0] = add2(x0, x1); X[1] = sub2(x0, x1);
            }
            __syncthreads();
            m = 2;
        }
        // fused radix-4 DIT: spans m and 2m; (x[j], x[j+2m] w, x[j+m] w^2, x[j+3m] w^3) through the 4-point IDFT go
        // to j, j+m, j+2m, j+3m, with w = W_4m^-j = conj(W_M^(j M / 4m))
        for (; 4 * m <= N; m <<= 2) {
            const int logm = __ffs(m) - 1, tstep = (M >> 2) >> logm;
            for (int bf = tid; bf < P * (N >> 2); bf += nthr) {
                const int f = bf >> (logN - 2), bb = bf & ((N >> 2) - 1);
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

    Out *out = static_cast<Out *>(a.out);
    float w[K];
#pragma unroll
    for (int k = 0; k < K; k++) w[k] = 0.0f;
    load(0);
    const float *Sf = reinterpret_cast<const float *>(buf);
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
                    Sf = reinterpret_cast<const float *>(Sc);
                }
                if (owner) {
                    w[u] = Sf[2 * (r & (P - 1)) * rs + q];   // real bin q = float q of the frame's transform
                    const int tr = r - (K - 1);
                    if (tr >= 0 && (int)((t0 + tr) & a.kmask) == b) {
                        float acc = w[u] * g[0];
#pragma unroll
                        for (int k = 1; k < K; k++) acc = fmaf(w[(u - k + K) % K], g[k], acc);
                        rsynth_store(out + (t0 + tr) * a.D + j, acc);
                    }
                }
            }
        }
    }
}

typedef void (*RSynthKernel)(const RSynthArgs);
template <typename Out>
static RSynthKernel rsynth_kernel(int K)
{
    static const RSynthKernel k[kSynthMaxTapsPerPhase] = {
        pfb_rsynth_kernel<1, Out>, pfb_rsynth_kernel<2, Out>, pfb_rsynth_kernel<3, Out>, pfb_rsynth_kernel<4, Out>,
        pfb_rsynth_kernel<5, Out>, pfb_rsynth_kernel<6, Out>, pfb_rsynth_kernel<7, Out>, pfb_rsynth_kernel<8, Out>,
        pfb_rsynth_kernel<9, Out>, pfb_rsynth_kernel<10, Out>, pfb_rsynth_kernel<11, Out>, pfb_rsynth_kernel<12, Out>,
        pfb_rsynth_kernel<13, Out>, pfb_rsynth_kernel<14, Out>, pfb_rsynth_kernel<15, Out>, pfb_rsynth_kernel<16, Out>,
        pfb_rsynth_kernel<17, Out>, pfb_rsynth_kernel<18, Out>, pfb_rsynth_kernel<19, Out>, pfb_rsynth_kernel<20, Out>,
        pfb_rsynth_kernel<21, Out>, pfb_rsynth_kernel<22, Out>, pfb_rsynth_kernel<23, Out>, pfb_rsynth_kernel<24, Out>,
        pfb_rsynth_kernel<25, Out>, pfb_rsynth_kernel<26, Out>, pfb_rsynth_kernel<27, Out>, pfb_rsynth_kernel<28, Out>,
        pfb_rsynth_kernel<29, Out>, pfb_rsynth_kernel<30, Out>, pfb_rsynth_kernel<31, Out>, pfb_rsynth_kernel<32, Out>};
    return k[K - 1];
}

static int ilog2(size_t v) { int l = 0; while (((size_t)1 << l) < v) l++; return l; }

// Frames per chunk: about kRSynthChunkSlots complex slots (P M/2) per buffer, at most 16 frames
constexpr size_t kRSynthChunkSlots = 8192;

int rsynth_plan_create(SynthPlan &p, size_t m, size_t interp, size_t smem_optin)
{
    const size_t N = m / 2;
    p.M = (int)m; p.logM = ilog2(m); p.D = (int)interp; p.logD = ilog2(interp);
    size_t P = std::max<size_t>(1, std::min<size_t>(16, kRSynthChunkSlots / N));
    auto smem_for = [&](size_t f) { return (2 * f * (N + 1) + m) * sizeof(c2); };
    while (P > 1 && smem_for(P) > smem_optin) P >>= 1;
    if (smem_for(P) > smem_optin) { set_error("real synthesizer: %zu branches do not fit in shared memory", m); return B200C_ERR_UNSUPPORTED; }
    p.P = (int)P;
    p.smem_bytes = smem_for(P);
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

int rsynth_set_taps(SynthPlan &p, const double *taps, size_t ntaps)
{
    const int rc = synth_set_taps(p, taps, ntaps);   // taps table, K and the tile T = max(4 P, 16 (K - 1))
    if (rc) return rc;
    p.B = std::min(p.M, rsynth_max_threads(p.K));
    return B200C_OK;
}

int rsynth_launch(const SynthPlan &p, int dtype, const void *d_in, size_t in_stride, size_t frames, uint64_t stream_index,
                  void *d_out, cudaStream_t stream)
{
    RSynthArgs a;
    a.in = static_cast<const c2 *>(d_in);
    a.out = d_out;
    a.taps = p.d_taps;
    a.tw = static_cast<const c2 *>(p.d_tw);
    a.in_stride = (long long)in_stride;
    a.frames = (long long)frames;
    a.s = (unsigned)(stream_index & (uint64_t)(p.M - 1));
    a.M = p.M; a.logN = p.logM - 1; a.D = p.D; a.logD = p.logD;
    a.kmask = p.M / p.D - 1;
    a.T = p.T; a.P = p.P; a.logP = ilog2((size_t)p.P); a.rs = p.M / 2 + 1; a.B = p.B;
    const RSynthKernel kern = dtype == B200C_I16 ? rsynth_kernel<int16_t>(p.K) : rsynth_kernel<float>(p.K);
    if (p.smem_bytes > 48 * 1024)
        B200C_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_bytes));
    const size_t grid = (frames + (size_t)p.T - 1) / (size_t)p.T;
    if (grid > 0x7fffffffu) { set_error("real synthesizer: %zu frames exceed one launch", frames); return B200C_ERR_INVALID; }
    const dim3 g((unsigned)grid, (unsigned)(p.M / p.B));
    kern<<<g, std::max(p.B, 32), p.smem_bytes, stream>>>(a);
    B200C_CUDA_TRY(cudaGetLastError());
    return B200C_OK;
}

} // namespace b200c
