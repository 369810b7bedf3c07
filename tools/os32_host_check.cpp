// CPU check of the 32 x 32 (1024-point) overlap-save index logic of fir_os32_kernel: signed lanes and register indices
// (os32_signed), the 16-row signed step-twiddle table and the row shifts of the landing read, the tap spectrum and the
// store, run with the same transforms and twiddle helper the kernel uses.  Every forward bin of every lane and register,
// and every alias-free output of a block, is compared with a double-precision DFT / convolution.
//   g++ -std=c++17 -O2 -I pothoscomms_b200/csrc -o /tmp/os32_check tools/os32_host_check.cpp && /tmp/os32_check [K ...]
// Exit status 0 when every K passes.  --fault conj:k (conjugate the wrong way at register k) and --fault lane:L (lane L
// without its row shift) break the model on purpose, to show that the check catches such a slip.
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

#include "os64_core.cuh"
using namespace b200c;
typedef std::complex<double> cd;
static c2 from(cd z) { return pk((float)z.real(), (float)z.imag()); }
static cd to(c2 p) { float a, b; upk(p, a, b); return cd(a, b); }

static int fault_conj = -1, fault_lane = -1;

// v * (forward) step twiddle of register k, lane t, with the injected fault if any
static c2 step(c2 v, const c2 *twl, int k, bool inv)
{
    if (k == fault_conj) inv = !inv;
    return inv ? os32_step<true>(v, twl, k) : os32_step<false>(v, twl, k);
}

static bool check(int K, unsigned seed)
{
    const int N = 1024;
    std::mt19937 rng(seed);
    std::normal_distribution<double> g;
    std::vector<cd> x(N), h(K);
    for (auto &v : x) v = cd(g(rng), g(rng));
    for (auto &v : h) v = cd(g(rng), g(rng)) / (double)K;
    const double PI = 3.14159265358979323846;
    std::vector<c2> hf(N), tw(32 * kOs32SignedTwRows);
    for (int f = 0; f < N; f++) {
        cd s = 0;
        for (int k = 0; k < K; k++) s += h[k] * std::polar(1.0, -2 * PI * ((long long)f * k % N) / N);
        hf[f] = from(s / (double)N);
    }
    {
        std::vector<float> tb(2 * tw.size());
        os32_signed_twiddles(tb.data());
        for (size_t i = 0; i < tw.size(); i++) tw[i] = pk(tb[2 * i], tb[2 * i + 1]);
    }
    // the lane's signed index and its element in row 0, as the kernel has them
    auto so_of = [](int t) { return t == fault_lane ? t : os32_signed(t); };
    auto row = [&](int t, int n) { return n ? 32 * n + so_of(t) : so_of(t) & 1023; };
    static c2 v[32][32];
    std::vector<c2> F(kOs32SmemElems);
    for (int t = 0; t < 32; t++) {
        for (int n1 = 0; n1 < 32; n1++) v[t][rev32(n1)] = from(x[row(t, n1)]);
        dft32_dit<false>(v[t]);
        for (int k1 = 1; k1 < 32; k1++) v[t][k1] = step(v[t][k1], tw.data() + t, k1, false);
        for (int k1 = 0; k1 < 32; k1++) F[k1 * kOs32Stride + t] = v[t][k1];
    }
    std::vector<cd> X(N);
    for (int k = 0; k < N; k++) {
        cd s = 0;
        for (int n = 0; n < N; n++) s += x[n] * std::polar(1.0, -2 * PI * ((long long)n * k % N) / N);
        X[k] = s;
    }
    double xrms = 0;
    for (const cd &z : X) xrms += std::norm(z);
    xrms = std::sqrt(xrms / N);
    double ferr = 0;
    for (int t = 0; t < 32; t++) {
        for (int n2 = 0; n2 < 32; n2++) v[t][rev32(n2)] = F[t * kOs32Stride + n2];
        dft32_dit<false>(v[t]);
        for (int k2 = 0; k2 < 32; k2++) ferr = std::max(ferr, std::abs(to(v[t][k2]) - X[row(t, k2)]) / xrms);   // bin s(t) + 32 k2
        for (int k2 = 0; k2 < 32; k2++) v[t][k2] = cmul_p<false>(v[t][k2], hf[row(t, k2)]);
        dft32_dif<true>(v[t]);
        for (int n2 = 1; n2 < 32; n2++) v[t][rev32(n2)] = step(v[t][rev32(n2)], tw.data() + t, n2, true);
    }
    for (int t = 0; t < 32; t++)
        for (int n2 = 0; n2 < 32; n2++) F[t * kOs32Stride + n2] = v[t][rev32(n2)];
    std::vector<cd> y(N);
    std::vector<int> seen(N, 0);
    for (int t = 0; t < 32; t++) {
        for (int k1 = 0; k1 < 32; k1++) v[t][k1] = F[k1 * kOs32Stride + t];
        dft32_dif<true>(v[t]);
        for (int n1 = 0; n1 < 32; n1++) {
            const int i = row(t, n1) & 1023;
            y[i] = to(v[t][rev32(n1)]);
            seen[i]++;
        }
    }
    double err = 0, ref = 0;
    bool cover = true;
    std::vector<cd> yref(N);
    for (int i = K - 1; i < N; i++) {
        cd s = 0;
        for (int k = 0; k < K; k++) s += h[k] * x[i - k];
        yref[i] = s;
        ref += std::norm(s);
    }
    ref = std::sqrt(ref / (N - K + 1));
    for (int i = 0; i < N; i++) {
        cover = cover && seen[i] == 1;
        if (i >= K - 1) err = std::max(err, std::abs(y[i] - yref[i]) / ref);
    }
    const bool ok = cover && ferr < 1e-5 && err < 1e-5;
    printf("K = %4d: forward max err %.3g of bin RMS, overlap-save max err %.3g of output RMS, every output once: %s -> %s\n",
           K, ferr, err, cover ? "yes" : "no", ok ? "ok" : "FAIL");
    return ok;
}

int main(int argc, char **argv)
{
    std::vector<int> Ks;
    for (int i = 1; i < argc; i++) {
        if (!std::strcmp(argv[i], "--fault") && i + 1 < argc) {
            const char *f = argv[++i];
            if (!std::strncmp(f, "conj:", 5)) fault_conj = std::atoi(f + 5);
            else if (!std::strncmp(f, "lane:", 5)) fault_lane = std::atoi(f + 5);
        } else {
            Ks.push_back(std::atoi(argv[i]));
        }
    }
    if (Ks.empty()) Ks = {9, 100, 256, 448};
    bool ok = true;
    for (int K : Ks) ok = check(K, 1u + (unsigned)K) && ok;
    return ok ? 0 : 1;
}
