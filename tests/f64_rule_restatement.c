/* TEST INFRASTRUCTURE ONLY: the fp64 check rule of the resident decoder (MathF64::check_fast, csrc/qlb_kernels.cuh, with
 * exp_neg_abs and log_ratio of csrc/qlb_f64_math.cuh) restated in C as plainly as it can be written: integer mantissa
 * comparisons in log_ratio, a run-time want_inf select, the exp table read from an array. tests/test_gpu_f64_rule.py compares
 * the GPU rule with it bit for bit. Built with -ffp-contract=off: the only fused operations are the explicit fma() calls, as in the CUDA source.
 * Divisions are IEEE divisions, except that a -0 numerator over a positive divisor gives +0, as the rule's own division does
 * (its exact-residual correction adds the opposite zeros -0 and +0). */
#include <math.h>
#include <stdint.h>
#include <string.h>

static const double kTab[32][2] = {
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
static const double kL32Hi = 0x1.62e42fee00000p-6, kL32Lo = 0x1.a39ef35793c76p-38;
static const double kQ[4] = {1.0 / 720, 1.0 / 120, 1.0 / 24, 1.0 / 6};
static const double kLg[7] = {6.666666666666735130e-01, 3.999999999940941908e-01, 2.857142874366239149e-01, 2.222219843214978396e-01,
                              1.818357216161805012e-01, 1.531383769920937332e-01, 1.479819860511658591e-01};
static const double kLn2Hi = 6.93147180369123816490e-01, kLn2Lo = 1.90821492927058770002e-10;

static uint32_t hi_of(double x) { uint64_t b; memcpy(&b, &x, 8); return (uint32_t)(b >> 32); }
static uint32_t lo_of(double x) { uint64_t b; memcpy(&b, &x, 8); return (uint32_t)b; }
static double make(uint32_t hi, uint32_t lo) { uint64_t b = ((uint64_t)hi << 32) | lo; double x; memcpy(&x, &b, 8); return x; }

static double div_rule(double a, double d)
{
    if (a == 0. && signbit(a) && d > 0.)
        return 0.;
    return a / d;
}

static double exp_neg_abs(double m)
{
    const double kMagic = 6755399441055744.0;
    uint32_t h = hi_of(m) & 0x7fffffffu;
    const double a = make(h < 0x40900000u ? h : 0x40900000u, lo_of(m));
    const double t = fma(-a, 46.16624130844683, kMagic);
    int32_t n = (int32_t)lo_of(t);
    n = n > -32000 ? n : -32000;
    const double nf = t - kMagic;
    double r = fma(nf, -kL32Hi, -a);
    r = fma(nf, -kL32Lo, r);
    double c = fma(r, kQ[0], kQ[1]);
    c = fma(r, c, kQ[2]);
    c = fma(r, c, kQ[3]);
    c = fma(r, c, 0.5);
    const double q = fma(r * r, c, r);
    const double *T = kTab[n & 31];
    const double p = T[0] + fma(T[0], q, T[1]);
    return make(hi_of(p) + ((uint32_t)(n >> 5) << 20), lo_of(p));
}

static double log_ratio(double num, double den)
{
    const int32_t hn = (int32_t)hi_of(num), hd = (int32_t)hi_of(den);
    int32_t j = (hn >> 20) - (hd >> 20);
    const uint32_t u = (((uint32_t)hn & 0x000fffffu) | 0x00100000u) >> 5, d = (((uint32_t)hd & 0x000fffffu) | 0x00100000u) >> 5;
    j += (u * 46341u > d * 65536u) ? 1 : 0;
    j -= (u * 65536u < d * 46341u) ? 1 : 0;
    const double ds = make((uint32_t)hd + ((uint32_t)j << 20), lo_of(den));
    const double s = div_rule(num - ds, num + ds);
    const double z = s * s;
    double R = fma(z, kLg[6], kLg[5]);
    R = fma(z, R, kLg[4]);
    R = fma(z, R, kLg[3]);
    R = fma(z, R, kLg[2]);
    R = fma(z, R, kLg[1]);
    R = fma(z, R, kLg[0]);
    R = z * R;
    const double dj = (double)j;
    return fma(dj, kLn2Hi, fma(2., s, fma(s, R, dj * kLn2Lo)));
}

/* One check of weight w (<= 16): v in place; s = syndrome bit; thr_eff = the clamp or +inf. */
void f64_rule_check(double *v, int w, int s, double thr_eff)
{
    const int want_inf = !(thr_eff <= 700.);
    double row = s ? -1. : 1.;
    int poisoned = 0;
    for (int k = 0; k < w; ++k)
    {
        poisoned |= v[k] != v[k];
        const double e = exp_neg_abs(v[k]);
        v[k] = copysign(div_rule(1. - e, 1. + e), v[k]);
        row *= v[k];
    }
    if (poisoned)
        row = make(0x7ff80000u, 0);
    for (int k = 0; k < w; ++k)
    {
        const double q = div_rule(row, v[k]);
        const double a = fabs(q), den = 1. - a;
        double r = log_ratio(1. + a, den);
        if (want_inf && den == 0.)
            r = INFINITY;
        r = r > thr_eff ? thr_eff : r;
        v[k] = copysign(r, q);
    }
}

/* records of 8 doubles, as the qlb_test_f64_math probe's op 6 takes them */
void f64_rule_records(long n_checks, const double *a, const double *b, double *out)
{
    for (long c = 0; c < n_checks; ++c)
    {
        const int w = (int)b[8 * c];
        for (int k = 0; k < 8; ++k)
            out[8 * c + k] = k < w ? a[8 * c + k] : 0.;
        f64_rule_check(out + 8 * c, w, b[8 * c + 1] != 0., b[8 * c + 2]);
    }
}
