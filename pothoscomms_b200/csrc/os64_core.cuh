// Register-resident 64-point transforms and the 64 x 64 decomposition of the 4096-point
// transform used by the fused overlap-save FIR kernel (fir_os.cu).
//
// 4096 = 64 * 64 (four-step):  n = 64*n1 + n2,  k = k1 + 64*k2
//   X[k1 + 64 k2] = sum_n2 W64^(n2 k2) * { W4096^(n2 k1) * sum_n1 x[64 n1 + n2] W64^(n1 k1) }
// One thread owns 64 points (128 registers), 64 threads own one transform:
//   step 1: thread n2 transforms x[64 n1 + n2] over n1           -> Y[n2][k1]   (registers)
//           and multiplies by the step twiddle W4096^(n2 k1)
//   exchange through shared memory (the only one per transform)
//   step 2: thread k1 transforms Y[.][k1] over n2                -> X[k1 + 64 k2]
// The inverse runs the mirror image (decimation in frequency, conjugate twiddles), so the
// forward's step 2 and the inverse's first step meet in the SAME registers: per overlap-save
// block there are two shared-memory exchanges instead of the four (2 x 2) of the 16-point-
// per-thread kernel -- the L1/shared data pipe was that kernel's limiter (ncu: 75 % busy).
//
// All register indices are compile-time constants after unrolling, so the base-4 digit
// reversal the in-place transforms need is free (it only renames registers).
#pragma once
#include <cmath>

#include "packed.cuh"

namespace b200c {

// cos / sin of 2*pi*e/64, e = 0..63, rounded to float
B200C_HD constexpr float cos64(int e)
{
    constexpr float t[64] = {
        1.0f, 0.9951847195625305f, 0.9807852506637573f, 0.9569403529167175f, 0.9238795042037964f, 0.8819212913513184f,
        0.8314695954322815f, 0.7730104327201843f, 0.7071067690849304f, 0.6343932747840881f, 0.5555702447891235f,
        0.4713967442512512f, 0.3826834261417389f, 0.290284663438797f, 0.19509032368659973f, 0.0980171412229538f, 0.0f,
        -0.0980171412229538f, -0.19509032368659973f, -0.290284663438797f, -0.3826834261417389f, -0.4713967442512512f,
        -0.5555702447891235f, -0.6343932747840881f, -0.7071067690849304f, -0.7730104327201843f, -0.8314695954322815f,
        -0.8819212913513184f, -0.9238795042037964f, -0.9569403529167175f, -0.9807852506637573f, -0.9951847195625305f, -1.0f,
        -0.9951847195625305f, -0.9807852506637573f, -0.9569403529167175f, -0.9238795042037964f, -0.8819212913513184f,
        -0.8314695954322815f, -0.7730104327201843f, -0.7071067690849304f, -0.6343932747840881f, -0.5555702447891235f,
        -0.4713967442512512f, -0.3826834261417389f, -0.290284663438797f, -0.19509032368659973f, -0.0980171412229538f, 0.0f,
        0.0980171412229538f, 0.19509032368659973f, 0.290284663438797f, 0.3826834261417389f, 0.4713967442512512f,
        0.5555702447891235f, 0.6343932747840881f, 0.7071067690849304f, 0.7730104327201843f, 0.8314695954322815f,
        0.8819212913513184f, 0.9238795042037964f, 0.9569403529167175f, 0.9807852506637573f, 0.9951847195625305f};
    return t[e & 63];
}
B200C_HD constexpr float sin64(int e) { return cos64(e + 48); }   // sin(x) = cos(x - pi/2)

// f * W64^e, W64 = exp(-2 pi i / 64); INV: f * conj(W64^e).  `e` is a compile-time constant
// at every call site (fully unrolled loops), so the branches and table reads fold away.
template <bool INV> B200C_HD c2 mul_w64(c2 f, int e)
{
    e &= 63;
    if (e == 0) return f;
    if (e == 16) return rot_p<INV>(f);          // forward: * (-i)
    if (e == 48) return rot_p<!INV>(f);
    const float c = cos64(e), s = INV ? sin64(e) : -sin64(e);
    return cmul_s(f, c, s);
}

// position of element n (base-4 digits n = a + 4b + 16c) in the digit-reversed register order
B200C_HD constexpr int rev64(int n) { return 16 * (n & 3) + 4 * ((n >> 2) & 3) + ((n >> 4) & 3); }

// In-place 64-point DFT, decimation in time: input element n in v[rev64(n)], output k in v[k].
template <bool INV> B200C_HD void dft64_dit(c2 (&v)[64])
{
#pragma unroll
    for (int g = 0; g < 16; g++) dft4_p<INV>(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
#pragma unroll
    for (int g = 0; g < 4; g++)
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int i = 16 * g + k;
            v[i + 4] = mul_w64<INV>(v[i + 4], 4 * k);
            v[i + 8] = mul_w64<INV>(v[i + 8], 8 * k);
            v[i + 12] = mul_w64<INV>(v[i + 12], 12 * k);
            dft4_p<INV>(v[i], v[i + 4], v[i + 8], v[i + 12]);
        }
#pragma unroll
    for (int k = 0; k < 16; k++) {
        v[k + 16] = mul_w64<INV>(v[k + 16], k);
        v[k + 32] = mul_w64<INV>(v[k + 32], 2 * k);
        v[k + 48] = mul_w64<INV>(v[k + 48], 3 * k);
        dft4_p<INV>(v[k], v[k + 16], v[k + 32], v[k + 48]);
    }
}

// In-place 64-point DFT, decimation in frequency (the transpose of dft64_dit): input element
// n in v[n], output k in v[rev64(k)].
template <bool INV> B200C_HD void dft64_dif(c2 (&v)[64])
{
#pragma unroll
    for (int k = 0; k < 16; k++) {
        dft4_p<INV>(v[k], v[k + 16], v[k + 32], v[k + 48]);
        v[k + 16] = mul_w64<INV>(v[k + 16], k);
        v[k + 32] = mul_w64<INV>(v[k + 32], 2 * k);
        v[k + 48] = mul_w64<INV>(v[k + 48], 3 * k);
    }
#pragma unroll
    for (int g = 0; g < 4; g++)
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int i = 16 * g + k;
            dft4_p<INV>(v[i], v[i + 4], v[i + 8], v[i + 12]);
            v[i + 4] = mul_w64<INV>(v[i + 4], 4 * k);
            v[i + 8] = mul_w64<INV>(v[i + 8], 8 * k);
            v[i + 12] = mul_w64<INV>(v[i + 12], 12 * k);
        }
#pragma unroll
    for (int g = 0; g < 16; g++) dft4_p<INV>(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
}

// Shared-memory exchange buffer of one transform: element (row r, column c) at r*65 + c.
// Row stride 65 (odd) makes both the row-contiguous and the column accesses conflict free.
constexpr int kOs64Stride = 65;
constexpr int kOs64SmemElems = 64 * kOs64Stride;

// ------------------------------------------------------ tangent-factored butterflies ---
// A twiddle w = W64^e (INV: its conjugate) is written as f (1 + i t) with f = Re w, t = Im w / Re w when |Re w| >= |Im w|,
// and as f (t + i) with f = Im w, t = Re w / Im w otherwise, so that |t| <= 1.  u = b (1 + i t) or b (t + i) is then ONE
// FFMA2 (i b is an operand swap and negate), and the scale f folds into the butterfly's add and subtract, which become
// FFMA2 as well: a twiddled radix-2 butterfly a +- w b costs 3 instead of 4 packed instructions, a radix-4 one 11 instead
// of 14.  The error stays that of the plain form (tools/dft32_tangent_check.cpp).  f and t are compile-time constants
// at every call site.
struct TanW64 {
    float f, t;
    bool cot;   // f (t + i) rather than f (1 + i t)
};
template <bool INV> B200C_HD constexpr TanW64 tan_w64(int e)
{
    const float c = cos64(e), s = INV ? sin64(e) : -sin64(e);
    const bool cot = (c < 0 ? -c : c) < (s < 0 ? -s : s);
    return cot ? TanW64{s, c / s, true} : TanW64{c, s / c, false};
}
// b (1 + i t) or b (t + i)
B200C_HD c2 tan_mul(c2 b, const TanW64 w)
{
    float x, y;
    upk(b, x, y);
    return w.cot ? fma2(b, pk(w.t, w.t), pk(-y, x)) : fma2(pk(-y, x), pk(w.t, w.t), b);
}

// (a, b) <- (a + W64^e b, a - W64^e b)  (INV: conjugate twiddle)
template <bool INV> B200C_HD void bfly2_w64(c2 &a, c2 &b, int e)
{
    e &= 63;
    if (e == 0 || e == 16 || e == 48) {
        const c2 wb = mul_w64<INV>(b, e);
        b = sub2(a, wb);
        a = add2(a, wb);
        return;
    }
    const TanW64 w = tan_w64<INV>(e);
    const c2 u = tan_mul(b, w);
    b = fma2(u, pk(-w.f, -w.f), a);
    a = fma2(u, pk(w.f, w.f), a);
}

// Decimation-in-time radix-4 butterfly with twiddles W64^e, W64^2e, W64^3e on f1, f2, f3, then the 4-point DFT.
// e = 0 (no twiddles) or 1 <= e <= 15, so that the twiddles of f1 and f3 are not trivial: with w1 = f1 u1 / b and
// w3 = f3 u3 / d, w1 b +- w3 d = f1 (u1 +- (f3 / f1) u3), and f1 folds into the last four adds.
template <bool INV> B200C_HD void bfly4_w64(c2 &a, c2 &b, c2 &c, c2 &d, int e)
{
    if (e == 0) {
        dft4_p<INV>(a, b, c, d);
        return;
    }
    c2 p, m;   // a +- W64^2e c
    const int e2 = (2 * e) & 63;
    if (e2 == 16 || e2 == 48) {
        const c2 wc = mul_w64<INV>(c, e2);
        p = add2(a, wc);
        m = sub2(a, wc);
    } else {
        const TanW64 w2 = tan_w64<INV>(e2);
        const c2 u2 = tan_mul(c, w2);
        p = fma2(u2, pk(w2.f, w2.f), a);
        m = fma2(u2, pk(-w2.f, -w2.f), a);
    }
    const TanW64 w1 = tan_w64<INV>(e), w3 = tan_w64<INV>(3 * e);
    const float r = w3.f / w1.f, f = w1.f;
    const c2 u1 = tan_mul(b, w1), u3 = tan_mul(d, w3);
    const c2 s3 = fma2(u3, pk(r, r), u1), s4 = rot_p<INV>(fma2(u3, pk(-r, -r), u1));
    a = fma2(s3, pk(f, f), p);
    c = fma2(s3, pk(-f, -f), p);
    b = fma2(s4, pk(f, f), m);
    d = fma2(s4, pk(-f, -f), m);
}

// ---------------------------------------------------------------- 32-point transforms ---
// Radix 4, 4, 2.  Element n = q + 2 q' + 8 n'' (q < 2, q' < 4, n'' < 4) sits in register
// rev32(n) = 16 q + 4 q' + n'' for the decimation-in-time input / decimation-in-frequency output.
// 190 packed FMA-pipe instructions per transform (the plain form, a complex multiply per twiddle: 220).
B200C_HD constexpr int rev32(int n) { return 16 * (n & 1) + 4 * ((n >> 1) & 3) + ((n >> 3) & 3); }

template <bool INV> B200C_HD void dft32_dit(c2 (&v)[32])
{
#pragma unroll
    for (int g = 0; g < 8; g++) dft4_p<INV>(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
#pragma unroll
    for (int g = 0; g < 2; g++)
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int i = 16 * g + k;
            bfly4_w64<INV>(v[i], v[i + 4], v[i + 8], v[i + 12], 4 * k);   // W16^k
        }
#pragma unroll
    for (int k = 0; k < 16; k++) bfly2_w64<INV>(v[k], v[k + 16], 2 * k);   // W32^k
}

// The same transform with input n in v[n] and output k in v[rev32(k)]: dft32_dit on renamed registers (every index is
// a compile-time constant, so the renaming costs no instruction).
template <bool INV> B200C_HD void dft32_dif(c2 (&v)[32])
{
    c2 w[32];
#pragma unroll
    for (int n = 0; n < 32; n++) w[rev32(n)] = v[n];
    dft32_dit<INV>(w);
#pragma unroll
    for (int k = 0; k < 32; k++) v[rev32(k)] = w[k];
}

// exchange buffer of one 1024-point transform (one warp): element (r, c) at r*33 + c
constexpr int kOs32Stride = 33;
constexpr int kOs32SmemElems = 32 * kOs32Stride;

// Signed indices of the 32 x 32 decomposition (fir_os32_kernel).  Any index may be replaced by a representative modulo
// 32 if its neighbour in n = 32 n1 + n2 (k = k1 + 32 k2) shifts to match, so lanes and register indices i >= 16 stand
// for s(i) = i - 32: lane L >= 16 works on row-shifted data (element 32 m + L - 32, mod 1024), and every step twiddle
// W1024^(s(k) s(L)) is T[|s(k)|][L] = W1024^(|s(k)| s(L)) or, for s(k) < 0, its conjugate.  |s(k)| <= 16, so one
// 16-row table serves both directions: 16 loads per step twiddle instead of 31, the inverse taking the conjugates.
B200C_HD constexpr int os32_signed(int i) { return i < 16 ? i : i - 32; }

// v * W1024^(s(k) s(L)) (INV: its conjugate) for register index k = 1..31 of lane L; twl = T + L.  The conjugate is
// picked by k, a compile-time constant after unrolling, so it is the operand negate of cmul_p.
template <bool INV> B200C_HD c2 os32_step(c2 v, const c2 *twl, const int k)
{
    const int s = os32_signed(k);
    return s > 0 ? cmul_p<INV>(v, twl[32 * s]) : cmul_p<!INV>(v, twl[-32 * s]);
}

// T[r][L] = W1024^(r s(L)), r = 0..16 (row 0 unused, so that the row is |s(k)|), as float2 pairs: 2 * 17 * 32 floats.
// Computed in double and rounded once to float.
constexpr int kOs32SignedTwRows = 17;
inline void os32_signed_twiddles(float *tb)
{
    const double two_pi = 2.0 * 3.14159265358979323846264338327950288;
    for (int r = 0; r < kOs32SignedTwRows; r++)
        for (int L = 0; L < 32; L++) {
            const int e = (r * os32_signed(L)) & 1023;
            tb[2 * (r * 32 + L)] = (float)std::cos(-two_pi * e / 1024);
            tb[2 * (r * 32 + L) + 1] = (float)std::sin(-two_pi * e / 1024);
        }
}

} // namespace b200c
