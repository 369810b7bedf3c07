// CPU check of the tangent-factored 32-point transforms of os64_core.cuh (dft32_dit, dft32_dif; DESIGN.md section 4.2,
// step 9) against a double-precision DFT, with the plain form they replaced (a complex multiply per twiddle, then the
// butterfly) kept below as the yardstick.  For each transform, direction and input kind it prints the relative RMS
// error of both forms over all trials and the largest difference between them per output register.
//   g++ -std=c++17 -O2 -I pothoscomms_b200/csrc -o /tmp/dft32_check tools/dft32_tangent_check.cpp && /tmp/dft32_check
// Arguments pick cases: dit|dif, fwd|inv, random|fullscale|tone (default: all).  Exit status 0 when every case passes:
// error at most 1.5 times the plain form's, and every output register within 1e-5 of output RMS of the plain form's value.
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstring>
#include <random>
#include <string>
#include <vector>

#include "os64_core.cuh"
using namespace b200c;
typedef std::complex<double> cd;
static c2 from(cd z) { return pk((float)z.real(), (float)z.imag()); }
static cd to(c2 p) { float a, b; upk(p, a, b); return cd(a, b); }

// the plain form: every nontrivial twiddle a complex multiply (cmul_s), then the adds of the butterfly
template <bool INV> void plain_dit(c2 (&v)[32])
{
    for (int g = 0; g < 8; g++) dft4_p<INV>(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
    for (int g = 0; g < 2; g++)
        for (int k = 0; k < 4; k++) {
            const int i = 16 * g + k;
            v[i + 4] = mul_w64<INV>(v[i + 4], 4 * k);
            v[i + 8] = mul_w64<INV>(v[i + 8], 8 * k);
            v[i + 12] = mul_w64<INV>(v[i + 12], 12 * k);
            dft4_p<INV>(v[i], v[i + 4], v[i + 8], v[i + 12]);
        }
    for (int k = 0; k < 16; k++) {
        const c2 b = mul_w64<INV>(v[k + 16], 2 * k);
        v[k + 16] = sub2(v[k], b);
        v[k] = add2(v[k], b);
    }
}
template <bool INV> void plain_dif(c2 (&v)[32])
{
    for (int k = 0; k < 16; k++) {
        const c2 d = sub2(v[k], v[k + 16]);
        v[k] = add2(v[k], v[k + 16]);
        v[k + 16] = mul_w64<INV>(d, 2 * k);
    }
    for (int g = 0; g < 2; g++)
        for (int k = 0; k < 4; k++) {
            const int i = 16 * g + k;
            dft4_p<INV>(v[i], v[i + 4], v[i + 8], v[i + 12]);
            v[i + 4] = mul_w64<INV>(v[i + 4], 4 * k);
            v[i + 8] = mul_w64<INV>(v[i + 8], 8 * k);
            v[i + 12] = mul_w64<INV>(v[i + 12], 12 * k);
        }
    for (int g = 0; g < 8; g++) dft4_p<INV>(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
}

// one case: relative RMS error of the tangent and plain forms over all trials, largest register difference between them
static bool run(bool dif, bool inv, const std::string &kind)
{
    std::mt19937 rng(dif * 4 + inv * 2 + (unsigned)kind.size());
    std::normal_distribution<double> g;
    std::uniform_int_distribution<int> sign(0, 1);
    const double PI = 3.14159265358979323846;
    const int trials = kind == "tone" ? 32 : 200;
    double e_new = 0, e_old = 0, e_ref = 0, reg_diff = 0;
    for (int tr = 0; tr < trials; tr++) {
        cd x[32];
        for (int n = 0; n < 32; n++) {
            if (kind == "random") x[n] = cd(g(rng), g(rng));
            else if (kind == "fullscale") x[n] = cd(sign(rng) ? 1.0 : -1.0, sign(rng) ? 1.0 : -1.0);
            else x[n] = std::polar(1.0, 2 * PI * tr * n / 32);   // full-scale tone at bin tr
            x[n] = to(from(x[n]));   // the reference transforms the float input both forms see
        }
        // input element n sits in register rev32(n) (dit) or n (dif); output k in k (dit) or rev32(k) (dif)
        c2 vn[32], vo[32];
        for (int n = 0; n < 32; n++) vn[dif ? n : rev32(n)] = from(x[n]);
        std::memcpy(vo, vn, sizeof(vn));
        if (dif) {
            if (inv) { dft32_dif<true>(vn); plain_dif<true>(vo); }
            else { dft32_dif<false>(vn); plain_dif<false>(vo); }
        } else {
            if (inv) { dft32_dit<true>(vn); plain_dit<true>(vo); }
            else { dft32_dit<false>(vn); plain_dit<false>(vo); }
        }
        double rms = 0;
        cd X[32];
        for (int k = 0; k < 32; k++) {
            cd s = 0;
            for (int n = 0; n < 32; n++) s += x[n] * std::polar(1.0, (inv ? 2 : -2) * PI * (n * k % 32) / 32);
            X[k] = s;
            rms += std::norm(s);
        }
        rms = std::sqrt(rms / 32);
        for (int k = 0; k < 32; k++) {
            const int r = dif ? rev32(k) : k;
            e_new += std::norm(to(vn[r]) - X[k]);
            e_old += std::norm(to(vo[r]) - X[k]);
            e_ref += std::norm(X[k]);
            reg_diff = std::max(reg_diff, std::abs(to(vn[r]) - to(vo[r])) / rms);
        }
    }
    const double rn = std::sqrt(e_new / e_ref), ro = std::sqrt(e_old / e_ref);
    const bool ok = rn <= 1.5 * ro && reg_diff < 1e-5;
    printf("%s %s %-9s: tangent %.3g, plain %.3g of RMS (ratio %.2f), largest register difference %.3g of RMS -> %s\n",
           dif ? "dif" : "dit", inv ? "inv" : "fwd", kind.c_str(), rn, ro, rn / ro, reg_diff, ok ? "ok" : "FAIL");
    return ok;
}

int main(int argc, char **argv)
{
    std::vector<std::string> forms, dirs, kinds;
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        (a == "dit" || a == "dif" ? forms : a == "fwd" || a == "inv" ? dirs : kinds).push_back(a);
    }
    if (forms.empty()) forms = {"dit", "dif"};
    if (dirs.empty()) dirs = {"fwd", "inv"};
    if (kinds.empty()) kinds = {"random", "fullscale", "tone"};
    bool ok = true;
    for (const auto &f : forms)
        for (const auto &d : dirs)
            for (const auto &k : kinds) {
                if (k != "random" && k != "fullscale" && k != "tone") { fprintf(stderr, "unknown case %s\n", k.c_str()); return 2; }
                ok = run(f == "dif", d == "inv", k) && ok;
            }
    return ok ? 0 : 1;
}
