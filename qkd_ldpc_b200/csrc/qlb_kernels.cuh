// sm_100a kernels of libqkdldpc_b200.so: batched syndrome and the fused reconcile / sum-product decoder.
//
// Decoder design ("frame-resident"): one persistent CTA decodes one frame at a time and pulls the next frame from
// a global queue, so early termination is exact per frame and costs nothing (no compaction, no idle lanes). The
// frame's whole message state is ONE in-place array of E values addressed by "physical slot" (qlb_layout.hpp):
//   check pass : thread per check, reads/overwrites its own slots  -> consecutive threads = consecutive addresses
//   bit pass   : thread per bit, gathers/overwrites the slots of its edges through bit_slots[a][i]
//   parity     : thread per check XORs the hard decisions the bit pass left beside the messages (zedge)
// For fp32 on the N=10240 code (E=30720) messages (120 KB) + bit_slots (60 KB) + zedge (30 KB) fit in the 227 KB
// of shared memory of one SM, so a decode iteration touches no HBM/L2 at all; fp64 keeps the messages in a per-CTA
// global scratch that stays L2-resident (148 CTAs x 240 KB << 126 MB). Larger codes fall back to global scratch
// for everything. Operation order inside a node is the reference's (see MathF64).
//
// Reference functions restated here (paths relative to the reference repository):
//   sum_product_decoding_irregular   src/qkd_ldpc_algorithm.cpp:175-345
//   QKD_LDPC_irregular               src/qkd_ldpc_algorithm.cpp:398-447
//   calculate_syndrome_irregular     src/array_and_matrix_operations.cpp:476-486
//   threshold_matrix_irregular       src/array_and_matrix_operations.cpp:508-524
//   arrays_equal                     src/array_and_matrix_operations.cpp:96-106
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

#include "qlb_f64_math.cuh"

namespace qlb
{
    constexpr int kMaxCW = 128;

    // -DQLB_BOUNDS_CHECK: the kernels test the indices they are about to use (message slots, frame columns, scratch offsets) and
    // trap on the first one out of range -- the stand-in for compute-sanitizer's memcheck, which is closed on the B200 pool
    // (profiles/r02_compute_sanitizer_closed.log). Built and run by scripts/bounds_check_build.sh; off in the product build.
#ifdef QLB_BOUNDS_CHECK
#define QLB_CHECK_INDEX(i, n)                                                                                             \
    do                                                                                                                    \
    {                                                                                                                     \
        if (!((unsigned long long)(i) < (unsigned long long)(n)))                                                         \
        {                                                                                                                 \
            printf("QLB_BOUNDS_CHECK %s:%d: %s = %llu not below %s = %llu (block %d thread %d)\n", __FILE__, __LINE__, #i, \
                   (unsigned long long)(i), #n, (unsigned long long)(n), (int)blockIdx.x, (int)threadIdx.x);               \
            __trap();                                                                                                     \
        }                                                                                                                 \
    } while (0)
#else
#define QLB_CHECK_INDEX(i, n) ((void)0)
#endif

    enum Tier
    {
        kTierSmemAll = 0, // messages + bit_slots + zedge + bit arrays in shared memory (16-bit slot indices)
        kTierSmemIdx = 1, // bit_slots + zedge + bit arrays in shared memory, messages in global scratch
        kTierGlobal = 2   // everything in global scratch (32-bit slot indices)
    };

    struct CodeDev
    {
        int32_t n, m, e, words_n, words_m, max_check_w, max_bit_w;
        int32_t uniform_bit_w; // the common bit weight, or 0 when bits differ in weight
        int32_t slots;         // physical message slots (>= e; rows of slots are 32-aligned)
        uint32_t cnt[kMaxCW];  // checks with weight > k
        uint32_t base[kMaxCW]; // first slot of edge position k
        uint32_t base4[16];    // 4 * base[k] for the fp32 resident kernel (byte offsets, constant-bank operands)
        const uint16_t *bit_slots16; // [max_bit_w][n] (0xFFFF = none), valid when e < 65535
        const uint32_t *bit_slots32; // [max_bit_w][n] (0xFFFFFFFF = none)
        const uint16_t *col_of_slot16; // [slots] bit index of the edge stored at a slot, valid when n < 65536
        const uint32_t *col_of_slot32; // [slots] the same, any n (0xFFFFFFFF = padding slot)
        const uint32_t *check_order; // [m]
        const int32_t *row_ptr;      // [m+1]
        const int32_t *col_idx;      // [e]
        // tables of the fp64 SM-resident kernel (qlb_resident_f64.cuh; null when the code or the device does not take it)
        const uint32_t *r64_check_group_table; // [r64_check_groups]
        const uint16_t *r64_bit_group_table;   // [r64_bit_groups]
        int32_t r64_check_groups, r64_bit_groups;
        uint32_t r64_smem_slots; // message slots kept in shared memory
    };

    struct DecodeArgs
    {
        CodeDev code;
        long long n_frames;
        int32_t max_it;
        int32_t enable_thr;
        float cap_f32; // (float)thr, or +inf when the clamp is disabled
        double thr;
        // reconcile mode
        const uint32_t *alice;    // [F][words_n]
        const uint32_t *bob;      // [F][words_n]
        const double *log_prior;  // [F]
        // sum-product mode
        const double *llr;           // [F][n]
        const uint32_t *syndrome_in; // [F][words_m], natural check order
        // outputs
        uint32_t *iterations; // [F]
        uint8_t *result;      // [F]
        uint32_t *decoded;    // [F][words_n] or null
        uint32_t *syndrome_out; // [F][words_m] or null (reconcile mode)
        unsigned long long *queue;      // next frame to take
        unsigned long long *iter_total; // sum of executed iterations
        unsigned char *scratch;         // per-CTA global scratch (tiers 1, 2)
        size_t scratch_stride;
        // host-side launch knobs (qlb_decode_params; not read by kernels)
        int32_t stream_max_bundles, stream_no_repack, block_threads;
    };

    // ------------------------------------------------------------------------------------------------------------
    // message clamp: src/array_and_matrix_operations.cpp:508-524 (NaN passes through, +-inf -> +-thr)
    template <typename Real>
    __device__ __forceinline__ Real clamp_msg(Real x, Real thr, bool enable)
    {
        if (enable)
        {
            if (x > thr)
                x = thr;
            else if (x < -thr)
                x = -thr;
        }
        return x;
    }

    // ------------------------------------------------------------------------------------------------------------
    // Check-node rules. Each processes the W-slot register tile v[0..w) of one check in place.
    //   s: the check's syndrome bit (seed of the product is -1 when set, qkd_ldpc_algorithm.cpp:231)

    // fp64, the reference's arithmetic and order: t = tanh(m/2.) (:220-226); row_prod = (+-1.) * t0 * t1 ... left to
    // right (:231-235); out_k = 2.*atanh(row_prod / t_k) (:237-243); clamp (:246-249).
    struct MathF64
    {
        typedef double real;
#if !defined(QLB_F64_LIBM_FORMS)
        // tanh(m/2) = (1 - e^-|m|) / (1 + e^-|m|) and 2 atanh(p) = ln((1 + p) / (1 - p)): the same functions as the reference's
        // tanh(m / 2.) and 2. * atanh(p), evaluated branch-free with the constant-memory exp / log / divide of qlb_f64_math.cuh
        // (libdevice's tanh/atanh take divergent small/large-argument paths, and 70 % of what its exp/log/divide issue is
        // constant and register shuffling). They differ from glibc's results at the ulp level, as libdevice's own do; what is
        // contractual is the per-frame outcome, checked against the reference's own outcomes on the campaign fixture
        // (tests/golden/campaign_n10240.npz, 49 152 frames). -DQLB_F64_LIBM_FORMS restores the literal tanh / atanh calls.
        //
        // NaN (0/0 of an exactly-zero message, or inf - inf with the clamp off): the reference's tanh(NaN) = NaN poisons the row
        // product, so EVERY output of the check is NaN (:231-243). f64m::tanh_half does not propagate NaN by itself; the rule
        // tracks it with one compare per edge and poisons the product once per check.
        static constexpr bool kOwnForms = true;
        static __device__ __forceinline__ double tanh_half(double m) { return f64m::tanh_half(m); }
        // |out| before the clamp; want_inf: the clamp is off, a saturated product must give inf (see f64m::two_atanh)
        static __device__ __forceinline__ double two_atanh(double p, bool want_inf) { return f64m::two_atanh(p, want_inf); }
        // the clamp of :246-249 on the magnitude (NaN passes: the comparison is false), then p's sign: one FP64 compare per edge
        static __device__ __forceinline__ double out(double p, bool en, double thr)
        {
            double r = f64m::two_atanh_mag(p, !en);
            r = (en && r > thr) ? thr : r;
            return copysign(r, p);
        }
#else
        static constexpr bool kOwnForms = false;
        static __device__ __forceinline__ double tanh_half(double m) { return tanh(m / 2.); }
        static __device__ __forceinline__ double two_atanh(double p, bool) { return 2. * atanh(p); }
        static __device__ __forceinline__ double out(double p, bool en, double thr) { return clamp_msg(2. * atanh(p), thr, en); }
#endif
        static __device__ __forceinline__ double quotient(double a, double d)
        {
#if !defined(QLB_F64_LIBM_FORMS)
            return f64m::div_any(a, d);
#else
            return a / d;
#endif
        }
        template <int W>
        static __device__ __forceinline__ void check(double (&v)[W], int w, bool s, bool en, double thr)
        {
            double row = s ? -1. : 1.;
            bool poisoned = false;
#pragma unroll
            for (int k = 0; k < W; ++k)
                if (k < w)
                {
                    if (kOwnForms)
                        poisoned |= v[k] != v[k];
                    v[k] = tanh_half(v[k]);
                    row *= v[k];
                }
            if (kOwnForms)
                row = poisoned ? __longlong_as_double(0x7ff8000000000000LL) : row;
#pragma unroll
            for (int k = 0; k < W; ++k)
                if (k < w)
                    v[k] = out(quotient(row, v[k]), en, thr);
        }
        // The same rule for a check of weight exactly W with the clamp folded into its operands: thr_eff = the clamp, or +inf
        // when it is disabled (no magnitude exceeds it; a NaN fails the comparison and passes, :508-524); want_inf = the clamp is
        // disabled or above ln(2^1024), i.e. a saturated product must come out as the IEEE infinity before the clamp.
        template <int W>
        static __device__ __forceinline__ void check_fast(double (&v)[W], bool s, double thr_eff, bool want_inf)
        {
#if !defined(QLB_F64_LIBM_FORMS)
            double row = s ? -1. : 1.;
            bool poisoned = false;
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                poisoned |= v[k] != v[k];
                v[k] = tanh_half(v[k]);
                row *= v[k];
            }
            row = poisoned ? __longlong_as_double(0x7ff8000000000000LL) : row;
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                const double q = quotient(row, v[k]);
                const double a = fabs(q), den = 1. - a;
                double r = f64m::log_ratio(1. + a, den);
                if (want_inf)
                    r = den == 0. ? __longlong_as_double(0x7ff0000000000000LL) : r;
                r = r > thr_eff ? thr_eff : r;
                v[k] = copysign(r, q);
            }
#else
            check<W>(v, W, s, thr_eff < __longlong_as_double(0x7ff0000000000000LL), thr_eff);
#endif
        }
    };

    // fp64, fused-ratio form of the same rule (QLB_FLAG_F64_FUSED_RATIO): with e_j = e^-|m_j|, tanh(|m_j|/2) = (1-e_j)/(1+e_j);
    // A = prod(1-e_j), B = prod(1+e_j), S = B + A, D = B - A give for edge k
    //     (1 + row/t_k) / (1 - row/t_k) = (S - e_k D) / (D - e_k S),      2 atanh(row / t_k) = ln of that,
    // so an edge costs one exp, ONE division and one log polynomial (f64m::log_ratio) instead of exp + three divisions + log:
    // ~35 % fewer FP64 instructions. The reference's special outcomes are kept: a zero message (t_k = 0) gives NaN on its own
    // edge and 0 on the others, a saturated product gives +-inf (then the clamp), a NaN input floods the check. D carries
    // an absolute rounding error of ~2^-52 B, so -- like the reference's own tanh, which rounds to exactly 1 beyond |m| ~ 37.4
    // (:220-226) -- magnitudes above ~36 are quantised and then saturate; the two saturate at slightly different places, which
    // is why this form is opt-in and carries its own parity campaign (profiles/parity_r01.md) instead of replacing MathF64.
    struct MathF64Fused
    {
        typedef double real;
        template <int W>
        static __device__ __forceinline__ void check(double (&v)[W], int w, bool s, bool en, double thr)
        {
            double e[W];
            double A = 1., B = 1.;
            int neg = s ? 1 : 0;
            bool poisoned = false;
#pragma unroll
            for (int k = 0; k < W; ++k)
                if (k < w)
                {
                    poisoned |= v[k] != v[k];
                    neg ^= (int)((uint32_t)__double2hiint(v[k]) >> 31);
                    e[k] = f64m::exp_neg_abs(v[k]);
                    A *= 1. - e[k];
                    B *= 1. + e[k];
                }
            const double S = B + A, D = B - A;
#pragma unroll
            for (int k = 0; k < W; ++k)
                if (k < w)
                {
                    // num >= den by construction, so den > 0 is the regular case. Otherwise the IEEE outcomes of ln(num / den):
                    // den <= 0 < num (a saturated product; a denominator rounded below zero counts as zero) -> +inf, which the
                    // clamp then turns into thr (:246-249); 0 / 0 (the message on this edge was exactly 0) or a NaN -> NaN.
                    const double num = fma(-e[k], D, S), den = fma(-e[k], S, D);
                    const double r = f64m::log_ratio(num, den);
                    const bool ok = den > 0. && !poisoned, to_inf = num > 0. && den <= 0. && !poisoned;
                    int hi = ok ? __double2hiint(r) : (to_inf ? 0x7ff00000 : 0x7ff80000);
                    int lo = ok ? __double2loint(r) : 0;
                    if (en && __hiloint2double(hi, lo) > thr) // the magnitude is >= 0 or NaN (a NaN passes the clamp, :508-524)
                    {
                        hi = __double2hiint(thr);
                        lo = __double2loint(thr);
                    }
                    const int sg = neg ^ (int)((uint32_t)__double2hiint(v[k]) >> 31);
                    v[k] = __hiloint2double(hi ^ (sg << 31), lo);
                }
        }
        // Weight exactly W, clamp folded into thr_eff (see MathF64::check_fast). The regular case (den > 0) pays two FP64
        // compares; everything else -- a saturated product, a zero or NaN message -- goes through one rarely-taken branch.
        template <int W>
        static __device__ __forceinline__ void check_fast(double (&v)[W], bool s, double thr_eff, bool)
        {
            double e[W];
            double A = 1., B = 1.;
            uint32_t neg = s ? 0x80000000u : 0u;
            bool poisoned = false;
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                poisoned |= v[k] != v[k];
                neg ^= (uint32_t)__double2hiint(v[k]);
                e[k] = f64m::exp_neg_abs(v[k]);
                A *= 1. - e[k];
                B *= 1. + e[k];
            }
            const double S = B + A;
            double D = B - A;
            D = poisoned ? __longlong_as_double(0x7ff8000000000000LL) : D; // a NaN input floods the check through the denominators
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                const double num = fma(-e[k], D, S), den = fma(-e[k], S, D);
                double r = f64m::log_ratio(num, den);
                if (!(den > 0.)) // the IEEE outcomes of ln(num / den): +inf for a saturated product, NaN for 0 / 0 or a NaN
                    r = (num > 0. && den <= 0.) ? __longlong_as_double(0x7ff0000000000000LL) : __longlong_as_double(0x7ff8000000000000LL);
                r = r > thr_eff ? thr_eff : r;
                const uint32_t sg = (neg ^ (uint32_t)__double2hiint(v[k])) & 0x80000000u;
                v[k] = __hiloint2double((int)((uint32_t)__double2hiint(r) ^ sg), __double2loint(r));
            }
        }
    };

    // fp32 with libdevice tanhf/atanhf and a leave-one-out product (prefix * suffix), which cannot produce the 0/0 the
    // divide form hits in single precision (SURVEY.md 8a "fp32 note").
    struct MathF32
    {
        typedef float real;
        template <int W>
        static __device__ __forceinline__ void check(float (&v)[W], int w, bool s, bool en, float thr)
        {
            float pre[W];
            float run = s ? -1.f : 1.f;
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                pre[k] = run;
                if (k < w)
                {
                    v[k] = tanhf(0.5f * v[k]);
                    run *= v[k];
                }
            }
            float suf = 1.f;
#pragma unroll
            for (int k = W - 1; k >= 0; --k)
                if (k < w)
                {
                    const float t = v[k];
                    v[k] = clamp_msg(2.f * atanhf(pre[k] * suf), thr, en);
                    suf *= t;
                }
        }
    };

    // fp32 on the SFU: with v = exp(-|m|), tanh(|m|/2) = (1-v)/(1+v); the leave-one-out products A_k = prod(1-v),
    // B_k = prod(1+v) give 2*atanh(A_k/B_k) = ln((B_k+A_k)/(B_k-A_k)): one ex2, one rcp, one lg2 per edge, signs by XOR.
    struct MathF32Fast
    {
        typedef float real;
        template <int W>
        static __device__ __forceinline__ void check(float (&v)[W], int w, bool s, bool en, float thr)
        {
            float preA[W], preB[W];
            float a[W], b[W];
            uint32_t sign = s ? 0x80000000u : 0u;
            float runA = 1.f, runB = 1.f;
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                preA[k] = runA;
                preB[k] = runB;
                if (k < w)
                {
                    sign ^= __float_as_uint(v[k]) & 0x80000000u;
                    const float e = exp2f(-1.4426950408889634f * fabsf(v[k])); // MUFU.EX2
                    a[k] = 1.f - e;
                    b[k] = 1.f + e;
                    runA *= a[k];
                    runB *= b[k];
                }
            }
            float sufA = 1.f, sufB = 1.f;
            const float cap = en ? thr : __int_as_float(0x7f800000);
#pragma unroll
            for (int k = W - 1; k >= 0; --k)
                if (k < w)
                {
                    const float Ak = preA[k] * sufA, Bk = preB[k] * sufB;
                    const uint32_t sk = (sign ^ __float_as_uint(v[k])) & 0x80000000u;
                    float mag = 0.6931471805599453f * __log2f(__fdividef(Bk + Ak, Bk - Ak)); // MUFU.RCP + MUFU.LG2
                    mag = fminf(mag, cap);
                    v[k] = __uint_as_float(__float_as_uint(mag) | sk);
                    sufA *= a[k];
                    sufB *= b[k];
                }
        }
    };

    // two-pass helpers for the generic (any weight) path of the fp32 rules: divide form with explicit zero handling,
    // equivalent to the leave-one-out product
    template <typename Math>
    struct TwoPass;
    template <>
    struct TwoPass<MathF64>
    {
        static constexpr bool kZeroAware = false; // the reference divides, 0/0 included
        static __device__ __forceinline__ double t(double m)
        {
            const double r = MathF64::tanh_half(m);
            return (MathF64::kOwnForms && m != m) ? m : r; // tanh(NaN) = NaN (stored, then multiplied into the row product)
        }
        static __device__ __forceinline__ double quotient(double a, double d) { return MathF64::quotient(a, d); }
        static __device__ __forceinline__ double out(double p, bool en, double thr) { return MathF64::out(p, en, thr); }
    };
    template <>
    struct TwoPass<MathF64Fused> : TwoPass<MathF64> // checks wider than the unrolled shapes keep the literal order
    {
    };
    template <>
    struct TwoPass<MathF32>
    {
        static constexpr bool kZeroAware = true;
        static __device__ __forceinline__ float t(float m) { return tanhf(0.5f * m); }
        static __device__ __forceinline__ float quotient(float a, float d) { return a / d; }
        static __device__ __forceinline__ float out(float p, bool en, float thr) { return clamp_msg(2.f * atanhf(p), thr, en); }
    };
    template <>
    struct TwoPass<MathF32Fast>
    {
        static constexpr bool kZeroAware = true;
        static __device__ __forceinline__ float t(float m)
        {
            const float e = exp2f(-1.4426950408889634f * fabsf(m));
            return copysignf(__fdividef(1.f - e, 1.f + e), m);
        }
        static __device__ __forceinline__ float quotient(float a, float d) { return a / d; }
        static __device__ __forceinline__ float out(float p, bool en, float thr)
        {
            const float ap = fabsf(p);
            float mag = 0.6931471805599453f * __log2f(__fdividef(1.f + ap, 1.f - ap));
            mag = fminf(mag, en ? thr : __int_as_float(0x7f800000));
            return copysignf(mag, p);
        }
    };

    // ------------------------------------------------------------------------------------------------------------
    template <typename IdxT>
    struct IdxTraits;
    template <>
    struct IdxTraits<uint16_t>
    {
        static constexpr uint32_t kNone = 0xFFFFu;
    };
    template <>
    struct IdxTraits<uint32_t>
    {
        static constexpr uint32_t kNone = 0xFFFFFFFFu;
    };

    __host__ __device__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

    // Byte layout of the per-CTA working set; the same carve-up is applied to shared memory and to global scratch.
    struct Carve
    {
        size_t msg, bit_slots, zedge, bob, alice, z, synp, synn, misc, total_smem, total_scratch;
    };
    template <typename Real, int kTier>
    __host__ __device__ inline Carve make_carve(int n, int m, int e, int max_bit_w)
    {
        Carve c{};
        const size_t wn = (size_t)(n + 31) / 32 * 4, wm = (size_t)(m + 31) / 32 * 4;
        const size_t msg = align_up((size_t)e * sizeof(Real), 16);
        const size_t idx = align_up((size_t)max_bit_w * n * (kTier == kTierGlobal ? 4 : 2), 16);
        const size_t zed = align_up((size_t)e, 16);
        const size_t small = align_up(wn, 16) * 3 + align_up(wm, 16) * 2 + 64;
        size_t s = 0, g = 0;
        // shared memory
        if (kTier == kTierSmemAll) { c.msg = s; s += msg; }
        if (kTier != kTierGlobal)
        {
            c.bit_slots = s; s += idx;
            c.zedge = s; s += zed;
            c.bob = s; s += align_up(wn, 16);
            c.alice = s; s += align_up(wn, 16);
            c.z = s; s += align_up(wn, 16);
            c.synp = s; s += align_up(wm, 16);
            c.synn = s; s += align_up(wm, 16);
        }
        c.misc = s; s += 64;
        c.total_smem = s;
        // global scratch
        if (kTier != kTierSmemAll) { c.msg = g; g += msg; }
        if (kTier == kTierGlobal)
        {
            c.zedge = g; g += zed;
            c.bob = g; g += align_up(wn, 16);
            c.alice = g; g += align_up(wn, 16);
            c.z = g; g += align_up(wn, 16);
            c.synp = g; g += align_up(wm, 16);
            c.synn = g; g += align_up(wm, 16);
        }
        c.total_scratch = align_up(g, 256);
        (void)small;
        return c;
    }

    // ------------------------------------------------------------------------------------------------------------
    // The decoder. kShapeW: 0 = any node weights (two-pass check rule, re-gathering bit pass);
    //                       8 / 16 = register tiles for checks of weight <= 8 / 16 and bits of weight <= 4.
    template <typename Math, int kTier, bool kReconcile, int kShapeW, int kThreads>
    __global__ void __launch_bounds__(kThreads, kThreads <= 512 ? 2 : 1) decode_kernel(const DecodeArgs args)
    {
        typedef typename Math::real Real;
        typedef typename std::conditional<kTier == kTierGlobal, uint32_t, uint16_t>::type IdxT;
        constexpr uint32_t kNone = IdxTraits<IdxT>::kNone;
        constexpr int W = kShapeW == 0 ? 1 : kShapeW;
        constexpr int WV = 4;

        extern __shared__ __align__(16) unsigned char smem[];
        const CodeDev &code = args.code;
        const int n = code.n, m = code.m, tid = threadIdx.x;
        const int words_n = code.words_n, words_m = code.words_m;
        const int max_cw = code.max_check_w, max_bw = code.max_bit_w;
        const Carve cv = make_carve<Real, kTier>(n, m, code.slots, max_bw);
        unsigned char *scratch = args.scratch + (size_t)blockIdx.x * args.scratch_stride;

        Real *msg = reinterpret_cast<Real *>((kTier == kTierSmemAll ? smem : scratch) + cv.msg);
        unsigned char *small_base = (kTier == kTierGlobal) ? scratch : smem;
        unsigned char *zedge = small_base + cv.zedge;
        uint32_t *s_bob = reinterpret_cast<uint32_t *>(small_base + cv.bob);
        uint32_t *s_alice = reinterpret_cast<uint32_t *>(small_base + cv.alice);
        uint32_t *s_z = reinterpret_cast<uint32_t *>(small_base + cv.z);
        uint32_t *s_synp = reinterpret_cast<uint32_t *>(small_base + cv.synp); // syndrome, sorted-check order
        uint32_t *s_synn = reinterpret_cast<uint32_t *>(small_base + cv.synn); // syndrome, natural order
        long long *s_frame = reinterpret_cast<long long *>(smem + cv.misc);

        const IdxT *bit_slots;
        if (kTier == kTierGlobal)
            bit_slots = reinterpret_cast<const IdxT *>(code.bit_slots32);
        else
        {
            // stage the bit->slot table once per (persistent) CTA
            IdxT *dst = reinterpret_cast<IdxT *>(smem + cv.bit_slots);
            const IdxT *src = reinterpret_cast<const IdxT *>(code.bit_slots16);
            for (int i = tid; i < max_bw * n; i += kThreads)
                dst[i] = src[i];
            bit_slots = dst;
        }

        const Real thr = (Real)args.thr;
        const bool en = args.enable_thr != 0;
        const int n_round = (n + 31) & ~31, m_round = (m + 31) & ~31;

        for (;;)
        {
            __syncthreads(); // previous frame fully retired (also orders the staging above)
            if (tid == 0)
                *s_frame = (long long)atomicAdd(args.queue, 1ULL);
            __syncthreads();
            const long long f = *s_frame;
            if (f >= args.n_frames)
                break;

            // ---- frame set-up ------------------------------------------------------------------------------------
            Real lp = 0;
            const double *llr_f = nullptr;
            if (kReconcile)
            {
                lp = (Real)args.log_prior[f];
                for (int w = tid; w < words_n; w += kThreads)
                {
                    s_bob[w] = args.bob[f * words_n + w];
                    s_alice[w] = args.alice[f * words_n + w];
                }
                for (int w = tid; w < words_m; w += kThreads)
                    s_synn[w] = 0;
            }
            else
            {
                llr_f = args.llr + f * n;
                for (int w = tid; w < words_m; w += kThreads)
                    s_synn[w] = args.syndrome_in[f * words_m + w];
            }
            __syncthreads();

            // messages start as the prior of the bit on each edge (qkd_ldpc_algorithm.cpp:182-190, unclamped); in
            // reconcile mode Alice's bits ride along in zedge so that the parity step below yields her syndrome
            for (int i = tid; i < n; i += kThreads)
            {
                Real prior;
                unsigned char abit = 0;
                if (kReconcile)
                {
                    const uint32_t bb = (s_bob[i >> 5] >> (i & 31)) & 1u;
                    abit = (unsigned char)((s_alice[i >> 5] >> (i & 31)) & 1u);
                    prior = bb ? -lp : lp; // :401-405
                }
                else
                    prior = (Real)llr_f[i];
                for (int a = 0; a < max_bw; ++a)
                {
                    const uint32_t s = bit_slots[(size_t)a * n + i];
                    if (s != kNone)
                    {
                        msg[s] = prior;
                        if (kReconcile)
                            zedge[s] = abit;
                    }
                }
            }
            __syncthreads();

            // target syndrome in sorted-check order
            for (int p = tid; p < m_round; p += kThreads)
            {
                uint32_t bit = 0;
                if (p < m)
                {
                    if (kReconcile)
                    {
                        // calculate_syndrome_irregular on Alice's key (:413-414)
                        for (int k = 0; k < max_cw; ++k)
                            if ((uint32_t)p < code.cnt[k])
                                bit ^= zedge[code.base[k] + p];
                        if (bit)
                        {
                            const uint32_t j = code.check_order[p];
                            atomicOr(&s_synn[j >> 5], 1u << (j & 31));
                        }
                    }
                    else
                    {
                        const uint32_t j = code.check_order[p];
                        bit = (s_synn[j >> 5] >> (j & 31)) & 1u;
                    }
                }
                const uint32_t word = __ballot_sync(0xffffffffu, bit != 0);
                if ((tid & 31) == 0)
                    s_synp[p >> 5] = word;
            }
            __syncthreads();

            // ---- iterations ----------------------------------------------------------------------------------------
            int it = 0;
            bool success = false;
            while (it < args.max_it)
            {
                // check pass (:220-249)
                for (int p = tid; p < m; p += kThreads)
                {
                    const bool s = (s_synp[p >> 5] >> (p & 31)) & 1u;
                    if (kShapeW != 0)
                    {
                        Real v[W];
                        int w = 0;
#pragma unroll
                        for (int k = 0; k < W; ++k)
                            if (k < max_cw && (uint32_t)p < code.cnt[k])
                            {
                                v[k] = msg[code.base[k] + p];
                                w = k + 1;
                            }
                        Math::template check<W>(v, w, s, en, thr);
#pragma unroll
                        for (int k = 0; k < W; ++k)
                            if (k < w)
                                msg[code.base[k] + p] = v[k];
                    }
                    else
                    {
                        typedef TwoPass<Math> TP;
                        Real row = s ? (Real)-1 : (Real)1;
                        int zeros = 0;
                        for (int k = 0; k < max_cw; ++k)
                            if ((uint32_t)p < code.cnt[k])
                            {
                                const Real t = TP::t(msg[code.base[k] + p]);
                                msg[code.base[k] + p] = t;
                                if (TP::kZeroAware && t == (Real)0)
                                    ++zeros;
                                else
                                    row *= t;
                            }
                        for (int k = 0; k < max_cw; ++k)
                            if ((uint32_t)p < code.cnt[k])
                            {
                                const Real t = msg[code.base[k] + p];
                                Real prod;
                                if (!TP::kZeroAware)
                                    prod = TP::quotient(row, t);
                                else if (zeros == 0)
                                    prod = TP::quotient(row, t);
                                else if (zeros == 1)
                                    prod = (t == (Real)0) ? row : (Real)0;
                                else
                                    prod = (Real)0;
                                msg[code.base[k] + p] = TP::out(prod, en, thr);
                            }
                    }
                }
                __syncthreads();

                // bit pass: total (:256-258), hard decision (:259-266), extrinsic + clamp (:300-316)
                for (int i = tid; i < n_round; i += kThreads)
                {
                    bool z = false;
                    if (i < n)
                    {
                        Real prior;
                        if (kReconcile)
                            prior = ((s_bob[i >> 5] >> (i & 31)) & 1u) ? -lp : lp;
                        else
                            prior = (Real)llr_f[i];
                        Real total = prior;
                        if (kShapeW != 0)
                        {
                            Real c[WV];
                            uint32_t sl[WV];
#pragma unroll
                            for (int a = 0; a < WV; ++a)
                            {
                                sl[a] = kNone;
                                if (a < max_bw)
                                    sl[a] = bit_slots[(size_t)a * n + i];
                                c[a] = (sl[a] != kNone) ? msg[sl[a]] : (Real)0;
                            }
#pragma unroll
                            for (int a = 0; a < WV; ++a)
                                if (sl[a] != kNone)
                                    total = total + c[a];
                            z = total <= (Real)0;
#pragma unroll
                            for (int a = 0; a < WV; ++a)
                                if (sl[a] != kNone)
                                {
                                    msg[sl[a]] = clamp_msg(total - c[a], thr, en);
                                    zedge[sl[a]] = (unsigned char)z;
                                }
                        }
                        else
                        {
                            for (int a = 0; a < max_bw; ++a)
                            {
                                const uint32_t s = bit_slots[(size_t)a * n + i];
                                if (s != kNone)
                                    total = total + msg[s];
                            }
                            z = total <= (Real)0;
                            for (int a = 0; a < max_bw; ++a)
                            {
                                const uint32_t s = bit_slots[(size_t)a * n + i];
                                if (s != kNone)
                                {
                                    msg[s] = clamp_msg(total - msg[s], thr, en);
                                    zedge[s] = (unsigned char)z;
                                }
                            }
                        }
                    }
                    const uint32_t word = __ballot_sync(0xffffffffu, z);
                    if ((tid & 31) == 0)
                        s_z[i >> 5] = word;
                }
                __syncthreads();

                // parity of the hard decision against the target syndrome (:277-298)
                int bad = 0;
                for (int p = tid; p < m; p += kThreads)
                {
                    uint32_t par = (s_synp[p >> 5] >> (p & 31)) & 1u;
                    for (int k = 0; k < max_cw; ++k)
                        if ((uint32_t)p < code.cnt[k])
                            par ^= zedge[code.base[k] + p];
                    bad |= (int)par;
                }
                ++it;
                if (!__syncthreads_or(bad))
                {
                    success = true;
                    break;
                }
            }

            // ---- results -------------------------------------------------------------------------------------------
            int differs = 0;
            for (int w = tid; w < words_n; w += kThreads)
            {
                const uint32_t zw = s_z[w];
                if (args.decoded)
                    args.decoded[f * words_n + w] = zw;
                // arrays_equal(alice, decoded) (:433) over the n key bits: the padding bits of Alice's last word are not part of the key
                const uint32_t key_mask = (w == words_n - 1 && (n & 31)) ? (1u << (n & 31)) - 1u : 0xFFFFFFFFu;
                if (kReconcile)
                    differs |= ((zw ^ s_alice[w]) & key_mask) != 0;
            }
            if (kReconcile && args.syndrome_out)
                for (int w = tid; w < words_m; w += kThreads)
                    args.syndrome_out[f * words_m + w] = s_synn[w];
            const int any_diff = __syncthreads_or(differs);
            if (tid == 0)
            {
                uint8_t r = success ? 1 : 0;
                if (kReconcile && !any_diff)
                    r |= 2;
                args.iterations[f] = (uint32_t)it; // == max_it on failure (:344)
                args.result[f] = r;
                atomicAdd(args.iter_total, (unsigned long long)it);
            }
        }
    }

    // ------------------------------------------------------------------------------------------------------------
    // Batched syndrome: one CTA per group of up to kSynFrames frames; packed key words staged in shared memory when
    // they fit (stage != 0), else read in place; thread per check, __ballot_sync packs 32 checks into one output word.
    // calculate_syndrome_irregular (src/array_and_matrix_operations.cpp:476-486).
    constexpr int kSynFrames = 8;
    constexpr int kSynThreads = 256;
    template <int kThreads> // (a template so that the header can be included by several translation units)
    __global__ void __launch_bounds__(kThreads) syndrome_kernel(const CodeDev code, long long n_frames, int group, int stage,
                                                                  const uint32_t *bits, uint32_t *syndrome_out)
    {
        extern __shared__ __align__(16) unsigned char smem[];
        const int words_n = code.words_n, words_m = code.words_m, m = code.m;
        const long long f0 = (long long)blockIdx.x * group;
        const int nf = (int)min((long long)group, n_frames - f0);
        const uint32_t *src = bits + f0 * words_n;
        if (stage)
        {
            uint32_t *s_bits = reinterpret_cast<uint32_t *>(smem); // [group][words_n]
            for (int i = threadIdx.x; i < nf * words_n; i += kSynThreads)
                s_bits[i] = src[i];
            __syncthreads();
            src = s_bits;
        }
        const int m_round = (m + 31) & ~31;
        for (int j = threadIdx.x; j < m_round; j += kSynThreads)
        {
            uint32_t acc[kSynFrames];
#pragma unroll
            for (int g = 0; g < kSynFrames; ++g)
                acc[g] = 0;
            if (j < m)
                for (int p = code.row_ptr[j]; p < code.row_ptr[j + 1]; ++p)
                {
                    const int b = code.col_idx[p];
#pragma unroll
                    for (int g = 0; g < kSynFrames; ++g)
                        if (g < nf)
                            acc[g] ^= (src[g * words_n + (b >> 5)] >> (b & 31)) & 1u;
                }
#pragma unroll
            for (int g = 0; g < kSynFrames; ++g)
            {
                const uint32_t word = __ballot_sync(0xffffffffu, acc[g] != 0);
                if ((threadIdx.x & 31) == 0 && g < nf)
                    syndrome_out[(f0 + g) * words_m + (j >> 5)] = word;
            }
        }
    }
}
