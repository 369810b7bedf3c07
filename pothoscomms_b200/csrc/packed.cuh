// Packed complex-float32 arithmetic for sm_100a.
//
// Blackwell has two-lane fp32 instructions (FADD2 / FMUL2 / FFMA2; PTX add/sub/mul/fma.f32x2)
// on aligned 64-bit register pairs.  Their operands take a half swap, a per-half negate and a
// scalar broadcast for free (ptxas folds the mov.b64 pack/unpack patterns below into operand
// modifiers), so on interleaved (re, im) pairs a complex add is ONE instruction and a complex
// multiply TWO (FMUL2 + FFMA2).  A packed instruction holds the FMA pipe for two cycles but
// takes a single issue slot (measured: tools/probe_issue.cu, profiles/r01_probe_issue.jsonl).
//
// The same functions compile for the host (plain float maths) so that the index logic of the
// kernels built on them can be checked on a CPU-only box (tools/os64_host_check.cu).
#pragma once
#include <cmath>
#include <cstring>

#if defined(__CUDACC__)
#define B200C_HD __host__ __device__ __forceinline__
#else
#define B200C_HD inline
#endif

namespace b200c {

typedef unsigned long long c2;   // (re, im) in one aligned 64-bit register pair

#if defined(__CUDA_ARCH__)
B200C_HD c2 pk(float a, float b) { c2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
B200C_HD void upk(c2 p, float &a, float &b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(p)); }
B200C_HD c2 fma2(c2 a, c2 b, c2 c) { c2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
B200C_HD c2 mul2(c2 a, c2 b) { c2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
B200C_HD c2 add2(c2 a, c2 b) { c2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
B200C_HD c2 sub2(c2 a, c2 b) { c2 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
#else
B200C_HD c2 pk(float a, float b) { float f[2] = {a, b}; c2 r; std::memcpy(&r, f, 8); return r; }
B200C_HD void upk(c2 p, float &a, float &b) { float f[2]; std::memcpy(f, &p, 8); a = f[0]; b = f[1]; }
B200C_HD c2 fma2(c2 a, c2 b, c2 c)   // one rounding, as FFMA2
{
    float ax, ay, bx, by, cx, cy; upk(a, ax, ay); upk(b, bx, by); upk(c, cx, cy);
    return pk(std::fma(ax, bx, cx), std::fma(ay, by, cy));
}
B200C_HD c2 mul2(c2 a, c2 b) { float ax, ay, bx, by; upk(a, ax, ay); upk(b, bx, by); return pk(ax * bx, ay * by); }
B200C_HD c2 add2(c2 a, c2 b) { float ax, ay, bx, by; upk(a, ax, ay); upk(b, bx, by); return pk(ax + bx, ay + by); }
B200C_HD c2 sub2(c2 a, c2 b) { float ax, ay, bx, by; upk(a, ax, ay); upk(b, bx, by); return pk(ax - bx, ay - by); }
#endif

// f * w  (CONJ: f * conj(w))
template <bool CONJ> B200C_HD c2 cmul_p(c2 f, c2 w)
{
    float fx, fy, wx, wy;
    upk(f, fx, fy); upk(w, wx, wy);
    return fma2(f, pk(wx, wx), mul2(CONJ ? pk(fy, -fx) : pk(-fy, fx), pk(wy, wy)));
}
// f * (wx + i*wy) with scalar parts (compile-time constants in the unrolled transforms)
B200C_HD c2 cmul_s(c2 f, float wx, float wy)
{
    float fx, fy;
    upk(f, fx, fy);
    return fma2(f, pk(wx, wx), mul2(pk(-fy, fx), pk(wy, wy)));
}
// forward: -i*s = (s.y, -s.x); inverse: +i*s = (-s.y, s.x)
template <bool INV> B200C_HD c2 rot_p(c2 s) { float x, y; upk(s, x, y); return INV ? pk(-y, x) : pk(y, -x); }

// 4-point DFT in place (forward: e^{-2 pi i jq/4}; INV: conjugate), no twiddles
template <bool INV> B200C_HD void dft4_p(c2 &f0, c2 &f1, c2 &f2, c2 &f3)
{
    const c2 s5 = sub2(f0, f2);
    f0 = add2(f0, f2);
    const c2 s3 = add2(f1, f3), s4 = sub2(f1, f3);
    f2 = sub2(f0, s3);
    f0 = add2(f0, s3);
    const c2 r = rot_p<INV>(s4);
    f1 = add2(s5, r);
    f3 = sub2(s5, r);
}

// decimation-in-time radix-4 butterfly: twiddle the inputs, then the 4-point DFT
template <bool CONJ, bool INV>
B200C_HD void bfly4_p(c2 &f0, c2 &f1, c2 &f2, c2 &f3, const c2 t1, const c2 t2, const c2 t3)
{
    f1 = cmul_p<CONJ>(f1, t1); f2 = cmul_p<CONJ>(f2, t2); f3 = cmul_p<CONJ>(f3, t3);
    dft4_p<INV>(f0, f1, f2, f3);
}

} // namespace b200c
