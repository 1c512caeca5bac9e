// Branch-free double-precision exp / log / divide for the fp64 check rule.
//
// ncu on the fp64 kernels showed that 70 % of the issued instructions inside libdevice's exp / log / divide are not
// FP64 arithmetic but their scaffolding: 64-bit polynomial constants materialised through UMOV pairs, register moves and
// special-case branches (profiles/r01_summary.md). These versions keep every coefficient in constant memory (a direct DFMA
// operand), have no branches, and are specialised to the argument ranges the decoder produces:
//   exp_neg(x)   x in [-64, 0]           Cody-Waite reduction by ln 2 (round-to-nearest through the 1.5*2^52 shift), degree-13
//                                        Taylor polynomial in Horner form, exponent insertion by integer add.  <= 1 ulp
//   exp_neg_abs(m)  any m                e^-min(|m|, ~1024), the form the check rules use: table-driven (Tang 1989) -- reduction by
//                                        ln 2 / 32, 2^(j/32) as a (hi, lo) pair from a 512-byte table, degree-6 polynomial:
//                                        12 FP64 operations instead of 17, 0.54 ulp. +5.3 % on the fp64 resident kernel (A/B on one
//                                        B200: 4.54 -> 4.78 M frame-iterations/s), every parity test incl. the 49 152-frame campaign
//                                        unchanged. -DQLB_F64_EXP_TAYLOR13 restores the degree-13 form.
//   div_any(a,d) d normal, either sign    MUFU.RCP64H seed (rcp.approx.ftz.f64: ONE instruction on the double's high word, no
//                                        fp64<->fp32 conversions), one Newton step, one residual correction: the quotient before
//                                        its final rounding is within 2^-80 of a / d. d = 0 gives NaN for a = 0 (the reference's
//                                        0/0) and for any other a (never asked); a subnormal d counts as 0 (ftz)
//   log_pos(y)   y >= 2^-60, finite      the classical fdlibm scheme: y = 2^k m, m in [sqrt(1/2), sqrt 2), s = f/(2+f), f = m-1,
//                                        log m = f - (f^2/2 - s (f^2/2 + R(s^2))), R = the degree-14 minimax polynomial
//                                        Lg1..Lg7 of fdlibm's e_log.c (published algorithm and constants).     <= 1 ulp
// Accuracy was measured on the CPU with the same FMA arithmetic against glibc over 4e6 random arguments each
// (/tmp prototype, numbers above). Like any libm they differ from glibc at the ulp level; the decoder's contract is the
// per-frame outcome (profiles/parity_r01.md).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace qlb
{
    namespace f64m
    {
        static __constant__ double kExp[14] = {1.0, 1.0, 0.5, 1.0 / 6, 1.0 / 24, 1.0 / 120, 1.0 / 720, 1.0 / 5040, 1.0 / 40320, 1.0 / 362880,
                                               1.0 / 3628800, 1.0 / 39916800, 1.0 / 479001600, 1.0 / 6227020800.0};
        static __constant__ double kLg[7] = {6.666666666666735130e-01, 3.999999999940941908e-01, 2.857142874366239149e-01, 2.222219843214978396e-01,
                                             1.818357216161805012e-01, 1.531383769920937332e-01, 1.479819860511658591e-01};
        static __constant__ double kLn2Hi = 6.93147180369123816490e-01, kLn2Lo = 1.90821492927058770002e-10;
        // 2^(j/32), j = 0 ... 31, as (leading double, remainder) pairs: the table of the table-driven exp below (P. T. P. Tang's scheme,
        // "Table-driven implementation of the exponential function in IEEE floating-point arithmetic", ACM TOMS 15, 1989; the values
        // themselves computed here to 70 digits). Read with one 128-bit L1-cached load per call (512 B: always resident), or from
        // a copy in shared memory (the resident fp64 kernel).
        static __device__ const double2 kExpTab[32] = {
            {0x1.0000000000000p+0, 0x0.0p+0}, {0x1.059b0d3158574p+0, 0x1.d73e2a475b465p-55}, {0x1.0b5586cf9890fp+0, 0x1.8a62e4adc610bp-54},
            {0x1.11301d0125b51p+0, -0x1.6c51039449b3ap-54}, {0x1.172b83c7d517bp+0, -0x1.19041b9d78a76p-55}, {0x1.1d4873168b9aap+0, 0x1.e016e00a2643cp-54},
            {0x1.2387a6e756238p+0, 0x1.9b07eb6c70573p-54}, {0x1.29e9df51fdee1p+0, 0x1.612e8afad1255p-55}, {0x1.306fe0a31b715p+0, 0x1.6f46ad23182e4p-55},
            {0x1.371a7373aa9cbp+0, -0x1.63aeabf42eae2p-54}, {0x1.3dea64c123422p+0, 0x1.ada0911f09ebcp-55}, {0x1.44e086061892dp+0, 0x1.89b7a04ef80d0p-59},
            {0x1.4bfdad5362a27p+0, 0x1.d4397afec42e2p-56}, {0x1.5342b569d4f82p+0, -0x1.07abe1db13cadp-55}, {0x1.5ab07dd485429p+0, 0x1.6324c054647adp-54},
            {0x1.6247eb03a5585p+0, -0x1.383c17e40b497p-54}, {0x1.6a09e667f3bcdp+0, -0x1.bdd3413b26456p-54}, {0x1.71f75e8ec5f74p+0, -0x1.16e4786887a99p-55},
            {0x1.7a11473eb0187p+0, -0x1.41577ee04992fp-55}, {0x1.82589994cce13p+0, -0x1.d4c1dd41532d8p-54}, {0x1.8ace5422aa0dbp+0, 0x1.6e9f156864b27p-54},
            {0x1.93737b0cdc5e5p+0, -0x1.75fc781b57ebcp-57}, {0x1.9c49182a3f090p+0, 0x1.c7c46b071f2bep-56}, {0x1.a5503b23e255dp+0, -0x1.d2f6edb8d41e1p-54},
            {0x1.ae89f995ad3adp+0, 0x1.7a1cd345dcc81p-54}, {0x1.b7f76f2fb5e47p+0, -0x1.5584f7e54ac3bp-56}, {0x1.c199bdd85529cp+0, 0x1.11065895048ddp-55},
            {0x1.cb720dcef9069p+0, 0x1.503cbd1e949dbp-56}, {0x1.d5818dcfba487p+0, 0x1.2ed02d75b3707p-55}, {0x1.dfc97337b9b5fp+0, -0x1.1a5cd4f184b5cp-54},
            {0x1.ea4afa2a490dap+0, -0x1.e9c23179c2893p-54}, {0x1.f50765b6e4540p+0, 0x1.9d3e12dd8a18bp-54}};
        static __constant__ double kExpL32Hi = 0x1.62e42fee00000p-6, kExpL32Lo = 0x1.a39ef35793c76p-38; // ln 2 / 32, 32 + 53 bits
        static __constant__ double kExpQ[4] = {1.0 / 720, 1.0 / 120, 1.0 / 24, 1.0 / 6};

        __device__ __forceinline__ double exp_neg(double x)
        {
            const double kMagic = 6755399441055744.0; // 1.5 * 2^52: adding it rounds to the nearest integer in the low word
            const double t = fma(x, 1.4426950408889634, kMagic);
            const int k = __double2loint(t);
            const double kf = t - kMagic;
            double r = fma(kf, -kLn2Hi, x);
            r = fma(kf, -kLn2Lo, r);
            double p = kExp[13];
#pragma unroll
            for (int i = 12; i >= 0; --i)
                p = fma(p, r, kExp[i]);
            return __hiloint2double(__double2hiint(p) + (k << 20), __double2loint(p));
        }

        // e^-min(|m|, ~1024) for ANY double m, with the cap and the |.| made on the integer pipe (2 ALU instructions + one on the
        // exponent) instead of the FP64 pipe's DADD / DSETP and two selects: the high word of |m| is limited to that of 1024.0
        // (an infinity becomes 1024, a NaN some value in [1024, 1025): callers that can see a NaN track it themselves), and the
        // binary exponent k is kept above -1000 so that the integer exponent insertion cannot wrap: beyond |m| ~ 693 the result is
        // a positive number far below 2^-54 instead of e^-|m|, which is all tanh(|m| / 2) = (1 - e) / (1 + e) = 1 needs.
        // s_tab: a copy of kExpTab in shared memory (a 32-bit-addressed LDS.128 instead of a 64-bit address and an LDG), or null.
        __device__ __forceinline__ double exp_neg_abs(double m, const double2 *s_tab = nullptr)
        {
            const double kMagic = 6755399441055744.0;
            const double a = __hiloint2double(min(__double2hiint(m) & 0x7fffffff, 0x40900000), __double2loint(m));
#ifdef QLB_F64_EXP_TAYLOR13 // the first version: reduction by ln 2, degree-13 Taylor polynomial (17 FP64 operations, <= 1 ulp)
            const double t = fma(-a, 1.4426950408889634, kMagic);
            const int k = max(__double2loint(t), -1000);
            const double kf = t - kMagic;
            double r = fma(kf, -kLn2Hi, -a);
            r = fma(kf, -kLn2Lo, r);
            double p = kExp[13];
#pragma unroll
            for (int i = 12; i >= 0; --i)
                p = fma(p, r, kExp[i]);
            return __hiloint2double(__double2hiint(p) + (k << 20), __double2loint(p));
#else
            // Table-driven: -a = (32 k + j) ln2/32 + r, |r| <= ln2/64, e^-a = 2^k * 2^(j/32) * e^r with e^r - 1 = q from a degree-6 Taylor
            // polynomial (next term r^7/5040 < 4e-18) and 2^(j/32) = T_hi + T_lo: 12 FP64 operations instead of 17 and a dependent chain
            // of 9 instead of 16; 0.54 ulp against exp() to 70 digits on 3e5 arguments (the degree-13 form: <= 1 ulp).
            const double t = fma(-a, 46.16624130844683, kMagic); // 32 / ln 2
            const int n = max(__double2loint(t), -32000);        // (the cap keeps the exponent insertion below from wrapping)
            const double nf = t - kMagic;
            double r = fma(nf, -kExpL32Hi, -a);
            r = fma(nf, -kExpL32Lo, r);
            double c = fma(r, kExpQ[0], kExpQ[1]);
            c = fma(r, c, kExpQ[2]);
            c = fma(r, c, kExpQ[3]);
            c = fma(r, c, 0.5);
            const double q = fma(r * r, c, r);
            const double2 T = s_tab ? s_tab[n & 31] : __ldg(&kExpTab[n & 31]);
            const double p = T.x + fma(T.x, q, T.y);
            return __hiloint2double(__double2hiint(p) + ((n >> 5) << 20), __double2loint(p));
#endif
        }

        // MUFU.RCP64H seed (relative error ~2^-20) and ONE Newton step: y = (1/d)(1 + eps), |eps| <~ 2^-40. Either sign of d.
        __device__ __forceinline__ double rcp_any(double d)
        {
            double y0;
            asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y0) : "d"(d));
            return fma(y0, fma(-d, y0, 1.0), y0);
        }
        // q = a y is ~40 bits good; the residual a - d q is exact in an FMA and |residual * y| carries a relative error of 2^-40
        // again, so the corrected quotient is the rounding of a / d (1 + O(2^-80)): a second Newton step on y would buy nothing.
        __device__ __forceinline__ double div_any(double a, double d)
        {
            const double y = rcp_any(d);
            const double q = a * y;
            return fma(fma(-d, q, a), y, q);
        }
        __device__ __forceinline__ double div_pos(double a, double d) { return div_any(a, d); }

        __device__ __forceinline__ double log_pos(double y)
        {
            const int hi = __double2hiint(y);
            int k = (hi >> 20) - 1023;
            double m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, __double2loint(y));
            const bool big = m > 1.4142135623730951;
            m = big ? 0.5 * m : m;
            k += big ? 1 : 0;
            const double f = m - 1.0;
            const double s = div_pos(f, 2.0 + f);
            const double z = s * s, w = z * z;
            const double t1 = w * fma(w, fma(w, kLg[5], kLg[3]), kLg[1]);
            const double t2 = z * fma(w, fma(w, fma(w, kLg[6], kLg[4]), kLg[2]), kLg[0]);
            const double R = t2 + t1;
            const double hfsq = 0.5 * f * f, dk = (double)k;
            return dk * kLn2Hi - ((hfsq - (s * (hfsq + R) + dk * kLn2Lo)) - f);
        }

        // ln(num / den) for 0 < den <= num without forming the quotient: ONE division for the ratio and the logarithm together.
        // den is rescaled by the power of two 2^j that brings m = num / (den 2^j) into ~[sqrt(1/2), sqrt 2] (exponent difference,
        // corrected by one through a comparison of the leading mantissa bits; the boundary need not be exact, the
        // polynomial holds a little beyond it). Then s = (m - 1) / (m + 1) = (num - den') / (num + den') -- the numerator is exact
        // (Sterbenz) -- and ln m = 2 s + s R(s^2) with fdlibm's R (e_log.c: "log(1+f) = 2s + s*R"), result j ln 2 + ln m. <= 2 ulp.
        // (the special outcomes are selected by the caller from `num`, `den`: for operands outside 0 < den <= num the value
        // returned here is meaningless, but nothing traps)
        __device__ __forceinline__ double log_ratio(double num, double den)
        {
            const int hn = __double2hiint(num), hd = __double2hiint(den);
            // The leading 16 mantissa bits (with the hidden one) of both, u and d, as the floats U = u 2^-15 and D = d 2^-15 in [1, 2).
            // j = exponent difference + [u / d > sqrt 2] - [u / d < sqrt(1/2)], the two tests being u 46341 > d 65536 and
            // u 65536 < d 46341. Each is the sign of ONE fp32 FMA: U c - D (c = 46341 / 65536, exact) is the rounding of the exact
            // difference, rounding keeps the sign, and the difference is never zero (65536 would have to divide u 46341) -- so the
            // sign bits give both tests without predicates, for every pair of high words (checked on all 2^30 pairs (u, d)).
            const float U = __int_as_float(((hn << 3) & 0x007fff00) | 0x3f800000), D = __int_as_float(((hd << 3) & 0x007fff00) | 0x3f800000);
            const uint32_t not_above = (uint32_t)__float_as_int(fmaf(U, 46341.f / 65536.f, -D)) >> 31; // 1: u / d < sqrt 2
            const uint32_t not_below = (uint32_t)__float_as_int(fmaf(D, 46341.f / 65536.f, -U)) >> 31; // 1: u / d > sqrt(1/2)
            const int j = (hn >> 20) - (hd >> 20) + (int)not_below - (int)not_above;
            const double ds = __hiloint2double(hd + (j << 20), __double2loint(den));
            const double s = div_pos(num - ds, num + ds);
            const double z = s * s;
#ifdef QLB_F64_LOG_SPLIT_POLY // fdlibm's even / odd split (two shorter chains, two FP64 operations more)
            const double w = z * z;
            const double t1 = w * fma(w, fma(w, kLg[5], kLg[3]), kLg[1]);
            const double t2 = z * fma(w, fma(w, fma(w, kLg[6], kLg[4]), kLg[2]), kLg[0]);
            const double R = t2 + t1;
#else // Horner: the check rule is bound by the FP64 pipe's throughput, not by this chain's latency (six independent edges per check)
            double R = fma(z, kLg[6], kLg[5]);
            R = fma(z, R, kLg[4]);
            R = fma(z, R, kLg[3]);
            R = fma(z, R, kLg[2]);
            R = fma(z, R, kLg[1]);
            R = fma(z, R, kLg[0]);
            R = z * R;
#endif
            const double dj = (double)j;
            return fma(dj, kLn2Hi, fma(2., s, fma(s, R, dj * kLn2Lo)));
        }

        // tanh(m / 2) = (1 - e^-|m|) / (1 + e^-|m|); |m| capped (exp_neg_abs; the quotient is exactly +-1 far earlier).
        // m = NaN comes back as +-1, NOT NaN: callers that can see a NaN message track it themselves (MathF64::check poisons the
        // row product, TwoPass<MathF64>::t passes the NaN through) so that the hot loop pays one compare instead of a select pair.
        __device__ __forceinline__ double tanh_half(double m, const double2 *s_tab = nullptr)
        {
            const double e = exp_neg_abs(m, s_tab);
            return copysign(div_any(1. - e, 1. + e), m);
        }
        // 2 atanh(p) = ln((1 + |p|) / (1 - |p|)) with p's sign, |p| <= 1 (the caller's p is a product of tanh values divided by one
        // of its own factors, which cannot exceed 1 in magnitude: every partial product of factors <= 1 is <= each factor, and the
        // quotient of a <= d rounds to <= 1). ONE division serves the ratio and the logarithm (log_ratio). Edges: |p| = 1 gives
        // log_ratio(2, 0) = 1024 ln 2 -- finite, above any clamp the decoder can apply -- unless `want_inf`, the IEEE outcome +-inf
        // of the literal expression (needed only when the clamp is off); p = NaN gives NaN through the arithmetic itself.
        __device__ __forceinline__ double two_atanh_mag(double p, bool want_inf)
        {
            const double a = fabs(p);
            const double den = 1. - a;
            double r = log_ratio(1. + a, den);
            if (want_inf)
                r = den == 0. ? __longlong_as_double(0x7ff0000000000000LL) : r;
            return r; // >= 0 or NaN; the caller clamps the magnitude and then gives it p's sign
        }
        __device__ __forceinline__ double two_atanh(double p, bool want_inf) { return copysign(two_atanh_mag(p, want_inf), p); }
    }
}
