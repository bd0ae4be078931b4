// fq_arith.cuh -- "float-quotient" modular arithmetic of the fused small-modulus kernels
// (ntt_fast_fq.cu).  Shared by device code and by a host model (tools/fq_model.cpp) that checks the
// arithmetic and the proven bounds bit for bit without a GPU.
//
// Why: on B200 the fma-heavy pipe issues IMAD at 16 lanes/clk/SMSP and IMAD.HI at 8; FFMA also runs on
// the fma-lite pipe (profiles/int_peaks_r02.txt).  A modular product whose quotient estimate comes from
// ONE FFMA and whose remainder comes from two low-half IMADs leaves the heavy pipe at 4 clk per
// butterfly instead of 8 (IMAD + IMAD.HI + IMAD).
//
// Representation: every coefficient x travels as the integer  xb = x + kBias,  kBias = 0x4B400000 = the bit
// pattern of 1.5 * 2^23.  For |x| < 2^22 those same 32 bits, read as a float, are exactly 1.5 * 2^23 + x
// (ulp is 1 in [2^23, 2^24)), so no int->float conversion is ever issued.
//
// Product by a constant w in [0, q):   k22 = round(w * 2^22 / q),  wq = k22 * 2^-22 (exact float),
// c = 1.5 * 2^23 - 3 * k22 (an integer below 2^24, exact float).  Then
//     fmaf(as_float(xb), wq, c)  =  RN( (1.5 * 2^23 + x) * wq + c )  =  RN( 1.5 * 2^23 + x * wq )
// because 1.5 * 2^23 * wq = 3 * k22 cancels exactly inside the FMA: one rounding, to an integer, and the
// bits of the result are kBias + qe with qe = rint(x * k22 / 2^22),  |qe - x w / q| <= 1/2 + |x| 2^-23.
//     t = xb * w + K - bits * q   (mod 2^32),   K = kBias * q - kBias * w (+ kBias for a biased result)
// is x w - qe q exactly (|t| <= q (1/2 + |x| 2^-23) < 2^31, so the wrap-around is harmless).
#pragma once
#include <cstdint>
#include <cstring>
#include <cmath>

#ifdef __CUDACC__
#define FQ_HD __host__ __device__ __forceinline__
#else
#define FQ_HD inline
#endif

namespace scgpu {
namespace fq {

constexpr int32_t kBias = 0x4B400000;
constexpr float kBiasF = 12582912.0f;
constexpr int32_t kLimit = 1 << 22;          // |x| must stay below this wherever x is read as a float

struct alignas(16) Tw {
    int32_t w;      // multiplier in [0, q)
    float wq;       // k22 * 2^-22
    int32_t k;      // additive constant of the low product (includes the output bias when wanted)
    float c;        // 1.5 * 2^23 - 3 * k22
};

FQ_HD float as_f(int32_t x)
{
#ifdef __CUDA_ARCH__
    return __int_as_float(x);
#else
    float f; memcpy(&f, &x, 4); return f;
#endif
}
FQ_HD int32_t as_i(float f)
{
#ifdef __CUDA_ARCH__
    return __float_as_int(f);
#else
    int32_t x; memcpy(&x, &f, 4); return x;
#endif
}
FQ_HD float fma_rn(float a, float b, float c)
{
#ifdef __CUDA_ARCH__
    return __fmaf_rn(a, b, c);
#else
    return fmaf(a, b, c);
#endif
}
// wrap-around 32-bit multiply-add (signed overflow is undefined in C++, the hardware IMAD is not)
FQ_HD int32_t mad(int32_t a, int32_t b, int32_t c)
{
    return (int32_t)((uint32_t)a * (uint32_t)b + (uint32_t)c);
}

// xb biased, |x| < 2^22.  Result: x * w - qe * q, plus kBias when tw.k was built with the output bias.
FQ_HD int32_t mul(int32_t xb, const Tw &tw, int32_t nq)
{
    const float f = fma_rn(as_f(xb), tw.wq, tw.c);
    const int32_t p = mad(xb, tw.w, tw.k);
    return mad(as_i(f), nq, p);
}

// product of two UNBIASED values, |a b| / q < 2^22, |a|, |b| < 2^24.  pwk = kBias * q.
FQ_HD int32_t mul_var(int32_t a, int32_t b, float invq, int32_t pwk, int32_t nq)
{
#ifdef __CUDA_ARCH__
    const float g = __fmul_rn(__int2float_rn(a), __int2float_rn(b));
#else
    const float g = (float)a * (float)b;
#endif
    const float f = fma_rn(g, invq, kBiasF);
    const int32_t p = mad(a, b, pwk);
    return mad(as_i(f), nq, p);
}

FQ_HD float mul_rn(float a, float b)
{
#ifdef __CUDA_ARCH__
    return __fmul_rn(a, b);
#else
    return a * b;                                  // compiled with -ffp-contract=off
#endif
}
FQ_HD float i2f(int32_t a)
{
#ifdef __CUDA_ARCH__
    return __int2float_rn(a);
#else
    return (float)a;
#endif
}

// x UNBIASED with its float copy xf (|x| < 2^22): x * w - qe * q, unbiased.  Only tw.w / tw.wq are read:
// the magic number is the FMA's addend, pwk = kBias * q cancels the bias of the quotient's bit pattern.
FQ_HD int32_t mul_unb(int32_t x, float xf, int32_t w, float wq, int32_t pwk, int32_t nq)
{
    const float f = fma_rn(xf, wq, kBiasF);
    const int32_t p = mad(x, w, pwk);
    return mad(as_i(f), nq, p);
}

// ---- products by a twiddle known at compile time: every per-twiddle word is an instruction immediate -----------
// An FFMA and an IMAD take one immediate each, so the two addends c and k of Tw cannot both stay per twiddle.
// The twiddle is centred, w = sigma a with 0 < a < q/2, and the float side multiplies by a:  k22 = round(a 2^22 / q),
// wq = k22 2^-22 <= 1/2.  With ONE addend 2^23 for every twiddle
//     fmaf(as_float(xb), wq, 2^23)  =  RN( 2^23 + 3 k22 + x wq )
// stays inside the binade [2^23, 2^24) for |x| < 2^22 (0 <= wq (3 2^22 -+ |x|) < 2^23), so it is again one rounding
// to an integer and its bits are 0x4B000000 + 3 k22 + qe, qe = rint(x wq), |qe - x a / q| <= 1/2 + |x| 2^-23: the
// bound of mul.  The integer side takes the per-twiddle constant in its FIRST multiply-add:
//     p2 = bits (-sigma q) + K,   r = xb w + p2  =  x w - sigma qe q + extra,   K = extra - K0,
//     K0 = kBias w - sigma q (0x4B000000 + 3 k22)   (mod 2^32)
// so a product is FFMA (wq immediate) + IMAD (K immediate) + IMAD (w immediate) and the butterfly's two adds carry no
// per-twiddle constant.  2^23 and -+q come from registers (ImmK).
struct ImmTw {
    int32_t w;      // centred multiplier sigma a
    float wq;       // k22 2^-22, for a
    bool neg;       // sigma = -1
    uint32_t k0;    // K0
};

constexpr ImmTw make_imm(int64_t w, int64_t q)
{
    w = ((w % q) + q) % q;
    if (w > q / 2) w -= q;
    const int64_t a = w < 0 ? -w : w;
    const int64_t k22 = (a * (1ll << 23) + q) / (2 * q);             // round(a * 2^22 / q) <= 2^21
    const uint32_t sq = w < 0 ? (uint32_t)(-q) : (uint32_t)q;
    return ImmTw{(int32_t)w, (float)k22 / 4194304.0f, w < 0,
                 (uint32_t)kBias * (uint32_t)w - sq * (0x4B000000u + 3u * (uint32_t)k22)};
}

struct ImmK { float two23; int32_t q, nq; };        // 2^23, q, -q

// xb biased, |x| < 2^22: x w - sigma qe q + extra.
// On the device every operation is opaque to the compiler: with 2^23 or -+q as literals it would give the FFMA's or the
// IMAD's one immediate to them and move wq / K into a register per twiddle, and seen through, the product of a value
// that an add with a constant produced, (a + C) w, becomes a w + C w, with w in a register.
FQ_HD uint32_t mul_imm(uint32_t xb, const ImmTw &t, uint32_t extra, const ImmK &kk)
{
    const uint32_t K = extra - t.k0;
    const int32_t sq = t.neg ? kk.q : kk.nq;
#ifdef __CUDA_ARCH__
    float f;
    uint32_t p2, r;
    asm("fma.rn.f32 %0, %1, %2, %3;" : "=f"(f) : "f"(__uint_as_float(xb)), "f"(t.wq), "f"(kk.two23));
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(p2) : "r"(__float_as_uint(f)), "r"(sq), "r"(K));
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(xb), "r"(t.w), "r"(p2));
    return r;
#else
    const float f = fma_rn(as_f((int32_t)xb), t.wq, kk.two23);
    return (uint32_t)mad((int32_t)xb, t.w, mad(as_i(f), sq, (int32_t)K));
#endif
}

// ---- degree-3 base multiplication: the transform stops two stages early -------------------------------------
// After stage logn - 3 the polynomial is split into n/4 residues modulo X^4 - zeta_b (four consecutive elements,
// natural order).  Their products
//     c0 = a0 b0 + zeta (a1 b3 + a2 b2 + a3 b1)      c1 = a0 b1 + a1 b0 + zeta (a2 b3 + a3 b2)
//     c2 = a0 b2 + a1 b1 + a2 b0 + zeta a3 b3        c3 = a0 b3 + a1 b2 + a2 b1 + a3 b0
// replace the last two forward stages of both operands, the n pointwise products and the first two inverse stages
// (92 instructions per four coefficients) by 3 products with zeta, 16 multiply-adds on the integer side, 16 on the
// float side and ONE quotient per output coefficient (60 instructions).  The integer sums wrap around; the float
// sums only have to estimate the quotient: |sum| < 2^22 q, four roundings of half an ulp each (fq_host.h:
// analyse32_bm bounds the error of the quotient and the size of the result).
// a, b UNBIASED (the stage before emits them so inside its 3-input adds); c is BIASED.  pwb = kBias * q + kBias.
FQ_HD void basemul4(int32_t (&c)[4], const int32_t (&a)[4], const int32_t (&b)[4], int32_t zw, float zwq,
                    float invq, int32_t pwk, int32_t pwb, int32_t nq)
{
    float af[4], bf[4];
#pragma unroll
    for (int i = 0; i < 4; i++) { af[i] = i2f(a[i]); bf[i] = i2f(b[i]); }
    int32_t z[4]; float zf[4];
    z[0] = 0; zf[0] = 0.0f;
#pragma unroll
    for (int i = 1; i < 4; i++) { z[i] = mul_unb(a[i], af[i], zw, zwq, pwk, nq); zf[i] = i2f(z[i]); }
#pragma unroll
    for (int k = 0; k < 4; k++) {
        // terms i + j = k use a_i, terms i + j = k + 4 use zeta a_i
        int32_t p = mad(a[0], b[k], pwb);
        float f = mul_rn(af[0], bf[k]);
#pragma unroll
        for (int i = 1; i < 4; i++) {
            const int j = (k - i) & 3;
            const bool wrap = i > k;
            p = mad(wrap ? z[i] : a[i], b[j], p);
            f = fma_rn(wrap ? zf[i] : af[i], bf[j], f);
        }
        const float g = fma_rn(f, invq, kBiasF);
        c[k] = mad(as_i(g), nq, p);
    }
}

// The same product against a KEY whose residues modulo X^4 - zeta were prepared once per launch (ntt_fast_fq32.cu:
// k_key_residues): b[0..3] and zb[i] = zeta b[i] (centred, |.| <= q/2) with their float copies, so the run-time side
// needs no product with zeta and converts only a:
//     c_k = sum_{i <= k} a_i b_{k-i}  +  sum_{i > k} a_i zb_{k-i+4}
// a UNBIASED, c BIASED.  4 conversions + 16 + 16 multiply-adds + 4 quotients = 44 instructions per four coefficients.
FQ_HD void basemul4_key(int32_t (&c)[4], const int32_t (&a)[4], const int32_t (&b)[4], const float (&bf)[4],
                        const int32_t (&zb)[4], const float (&zbf)[4], float invq, int32_t pwb, int32_t nq)
{
    float af[4];
#pragma unroll
    for (int i = 0; i < 4; i++) af[i] = i2f(a[i]);
#pragma unroll
    for (int k = 0; k < 4; k++) {
        int32_t p = mad(a[0], b[k], pwb);
        float f = mul_rn(af[0], bf[k]);
#pragma unroll
        for (int i = 1; i < 4; i++) {
            const int j = (k - i) & 3;
            const bool wrap = i > k;
            p = mad(a[i], wrap ? zb[j] : b[j], p);
            f = fma_rn(af[i], wrap ? zbf[j] : bf[j], f);
        }
        const float g = fma_rn(f, invq, kBiasF);
        c[k] = mad(as_i(g), nq, p);
    }
}

}  // namespace fq
}  // namespace scgpu
