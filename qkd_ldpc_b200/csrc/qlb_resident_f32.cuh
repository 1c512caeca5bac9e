// fp32 "SM-resident" decoder: the specialised hot kernel for codes whose whole message state fits in one SM's shared
// memory and whose bits all have the same weight (the CW=3 family of BASELINE.json, N=10240: 120 KB of messages +
// 60 KB of slot indices). Same schedule and node arithmetic as decode_kernel (qlb_kernels.cuh), re-organised so that
// the inner loops carry (almost) nothing but the node arithmetic:
//
//   * checks are sorted by weight, so the check pass runs weight segment by weight segment through code fully unrolled
//     for that weight -- no per-edge predicates, no local arrays, no per-check dispatch;
//   * the hard decision z of a bit travels in the least-significant mantissa bit of the bit-to-check messages that bit
//     sends (a <= 1 ulp perturbation; fp32 has no bit-exactness contract, its bar is statistical). The check pass
//     XORs the raw words it loads anyway: bit 31 of the XOR is the product's sign, bit 0 is the check's parity. The
//     separate parity phase, its barrier, and the per-edge byte array of decode_kernel disappear;
//   * convergence of iteration t is therefore seen by the check pass of iteration t+1 (one speculative check pass per
//     successful frame, < 1 % of the sweep's work, against ~20 % saved in every iteration);
//   * a thread visits the same checks and bits in every iteration, so their syndrome bits and prior signs are packed
//     once per frame into two registers;
//   * the bit->slot table is staged into shared memory by one TMA bulk copy (cp.async.bulk + mbarrier) per CTA;
//   * two block barriers per iteration.
//
// Reference semantics restated (paths relative to the reference repository): src/qkd_ldpc_algorithm.cpp:175-345, 398-447;
// iteration counts, success flags and decoded keys follow the reference's definitions exactly
// (iterations_num = index of the first bit pass whose hard decision satisfies the syndrome, else max_it).
#pragma once
#include "qlb_kernels.cuh"

namespace qlb
{
    __device__ __forceinline__ float ex2_approx(float x)
    {
        float y;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
        return y;
    }
    __device__ __forceinline__ float lg2_approx(float x)
    {
        float y;
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
        return y;
    }
    __device__ __forceinline__ float rcp_approx(float x)
    {
        float y;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
        return y;
    }

    // ---- TMA bulk copy global -> shared, completion on an mbarrier ---------------------------------------------------
    __device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
    __device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
    {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
    {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
    }
    __device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
    {
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                     "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                     : "memory");
    }
    __device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
    {
        asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                     "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(smem_u32(bar)),
                     "r"(parity)
                     : "memory");
    }

    __device__ __forceinline__ void tma_bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes)
    {
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
    }
    __device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
    template <int N>
    __device__ __forceinline__ void bulk_wait_read()
    {
        asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
    }
    __device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
    __device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

    // ---- check rules for a check of weight exactly W -------------------------------------------------------------------
    // v[] holds the raw incoming messages and receives the outgoing ones. xr = XOR of the raw message words, with the
    // check's syndrome bit folded into bit 31 (sign of the seeded product, src/qkd_ldpc_algorithm.cpp:231).
    // Arg: what apply() takes besides the messages, formed once per launch by check_arg(cap, DecodeArgs::ms_scale) -- the clamp
    // in message units for the sum-product rules, the clamp and the scale for min-sum.
    struct RuleF32Fast
    {
        typedef float Arg;
        static __device__ __forceinline__ Arg check_arg(float cap, float) { return cap; }
        // Messages are kept in base-2 units (LLR / ln 2): with e = 2^-|m|, tanh(|m| ln2 / 2) = (1-e)/(1+e). For the whole
        // check A = prod(1-e_j), B = prod(1+e_j), S = B + A, D = B - A; the leave-one-out ratio of edge k follows without
        // a division or prefix/suffix products:
        //     (B_k + A_k) / (B_k - A_k) = (S - e_k D) / (D - e_k S),     out_k = log2 of that, sign by XOR.
        // One MUFU.EX2 + MUFU.RCP + MUFU.LG2 per edge. The absolute error floor of the denominator (~6e-8) is that of
        // forming B_k - A_k directly. A denominator rounded to zero gives +inf, one rounded below zero gives NaN out of
        // lg2; fminf(NaN or +inf, cap) = cap, so both saturate to the clamp exactly like a saturated product (:246-249).
        static constexpr float kUnit = 1.4426950408889634f; // messages = LLR * kUnit
        // The parity-first look (decode_resident_f32_kernel) pays for the rules whose check pass is expensive -- fp32 accurate
        // +7 %, fp64 +36 % frames/s at QBER 0.03 -- but not for this one: +0.6 % at QBER 0.03, -1.5 % at 0.09 (B200, 14 800
        // frames; its extra live state costs the 64-register hot loops more than the skipped 108-instruction pass returns).
#ifndef QLB_F32FAST_PARITY_FIRST
#define QLB_F32FAST_PARITY_FIRST 0
#endif
        static constexpr bool kParityFirst = QLB_F32FAST_PARITY_FIRST != 0;
        template <int W>
        static __device__ __forceinline__ void apply(float (&v)[W], uint32_t xr, float cap)
        {
            float e[W];
            float A = 1.f, B = 1.f;
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                e[k] = ex2_approx(-fabsf(v[k]));
                A = fmaf(-A, e[k], A); // A (1 - e), one rounding
                B = fmaf(B, e[k], B);  // B (1 + e)
            }
            const float S = B + A, D = B - A;
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                const float num = fmaf(-e[k], D, S);
                const float den = fmaf(-e[k], S, D);
                float mag = lg2_approx(num * rcp_approx(den));
                mag = fminf(mag, cap);
                v[k] = __uint_as_float(((xr ^ __float_as_uint(v[k])) & 0x80000000u) | __float_as_uint(mag));
            }
        }
    };

    struct RuleF32Accurate
    {
        typedef float Arg;
        static __device__ __forceinline__ Arg check_arg(float cap, float) { return cap; }
        static constexpr float kUnit = 1.f; // natural-log units
        static constexpr bool kParityFirst = true;
        // libdevice tanhf / atanhf, leave-one-out product by prefix * suffix
        template <int W>
        static __device__ __forceinline__ void apply(float (&v)[W], uint32_t xr, float cap)
        {
            float t[W], pre[W];
            uint32_t sx = xr; // bit 31: syndrome ^ all message signs; strip the message signs to get the seed's sign
#pragma unroll
            for (int k = 0; k < W; ++k)
                sx ^= __float_as_uint(v[k]);
            float run = (sx & 0x80000000u) ? -1.f : 1.f;
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                t[k] = tanhf(0.5f * v[k]);
                pre[k] = run;
                run *= t[k];
            }
            float suf = 1.f;
#pragma unroll
            for (int k = W - 1; k >= 0; --k)
            {
                float o = 2.f * atanhf(pre[k] * suf);
                o = fminf(fmaxf(o, -cap), cap); // NaN cannot arise here: |pre*suf| <= 1
                v[k] = o;
                suf *= t[k];
            }
        }
    };

    // Normalized min-sum (QLB_FLAG_F32_MIN_SUM; the rule is defined to the bit in include/qkd_ldpc_b200.h, its pieces are
    // MathF32MinSum's). Per edge: a mask, two integer min/max, one compare, one select, one LOP3 for the sign; per check: two
    // multiplies and two fminf. Every operation is exact or one IEEE rounding, so the result equals the CPU restatement's
    // (tests/min_sum_restatement.c) on every frame.
    struct RuleF32MinSum
    {
        struct Arg
        {
            float cap, scale;
        };
        static __device__ __forceinline__ Arg check_arg(float cap, float scale) { return Arg{cap, scale}; }
        // natural-log units: the clamp and the priors mean what they mean for the accurate rule, and the bit pass always clamps
        static constexpr float kUnit = 1.f;
        // No parity-first look: it pays for rules whose check pass is expensive, and this check pass is cheaper than the fast
        // rule's, for which the look already measured no gain (RuleF32Fast) -- its extra live state would cost the hot loops more.
        static constexpr bool kParityFirst = false;
        template <int W>
        static __device__ __forceinline__ void apply(float (&v)[W], uint32_t xr, Arg a)
        {
            uint32_t x = 0, m1 = 0x7F800000u, m2 = 0x7F800000u; // x: unused, the caller's xr already holds the XOR
#pragma unroll
            for (int k = 0; k < W; ++k)
                MathF32MinSum::take(__float_as_uint(v[k]), x, m1, m2);
            const uint32_t w1 = MathF32MinSum::word(m1, xr, a.cap, a.scale), w2 = MathF32MinSum::word(m2, xr, a.cap, a.scale);
#pragma unroll
            for (int k = 0; k < W; ++k)
                v[k] = MathF32MinSum::out(__float_as_uint(v[k]), m1, w1, w2);
        }
    };

    // Where the byte offset of edge position k's slot row comes from: the kernel parameters (constant bank, a free operand
    // for compile-time k) on the hot path, a shared-memory copy for the out-of-line wide weights.
    struct BaseFromParams
    {
        const DecodeArgs &args;
        __device__ __forceinline__ uint32_t operator()(int k) const { return args.code.base4[k]; }
    };
#ifdef QLB_BOUNDS_CHECK
    static __device__ uint32_t g_bounds_msg_bytes = 0xFFFFFFFFu; // 4 * slots of the code being decoded (set by the launcher in bounds-check builds)
#endif
    struct BaseFromSmem
    {
        const uint32_t *base4;
        __device__ __forceinline__ uint32_t operator()(int k) const { return base4[k]; }
    };

    // All checks of weight exactly W: sorted positions [lo, hi). Round r of the thread's walk uses bit `rbit` of my_syn.
    // Returns the OR over the thread's checks of (parity of the riding hard decisions) ^ (syndrome bit), in bit 0.
    template <typename Rule, int W, typename Base>
    __device__ __forceinline__ uint32_t check_segment(const int kThreads, unsigned char *__restrict__ msg_bytes, const Base base4, uint32_t lo, uint32_t hi,
                                                      uint32_t my_syn, int &rbit, typename Rule::Arg cap)
    {
        uint32_t bad = 0;
#pragma unroll 1
        for (uint32_t p = lo + threadIdx.x; p < hi; p += kThreads, ++rbit)
        {
            const uint32_t sb = (my_syn >> rbit) & 1u;
            uint32_t xr = sb * 0x80000001u; // bit 31: sign seed, bit 0: parity seed
            unsigned char *row = msg_bytes + 4u * p; // + (uniform) row offset per edge position
            float v[W];
#pragma unroll
            for (int k = 0; k < W; ++k)
            {
                QLB_CHECK_INDEX((size_t)(row - msg_bytes) + base4(k), g_bounds_msg_bytes);
                v[k] = *reinterpret_cast<const float *>(row + base4(k));
                xr ^= __float_as_uint(v[k]);
            }
            bad |= xr;
            Rule::template apply<W>(v, xr, cap);
#pragma unroll
            for (int k = 0; k < W; ++k)
                *reinterpret_cast<float *>(row + base4(k)) = v[k];
        }
        return bad;
    }

    // weights 9..16 are kept out of line: their register appetite must not leak into the hot (narrow) instantiations
    template <typename Rule, int W>
    __device__ __noinline__ uint32_t check_segment_wide(const int kThreads, unsigned char *msg_bytes, const uint32_t *s_base4, uint32_t lo, uint32_t hi,
                                                        uint32_t my_syn, int rbit, typename Rule::Arg cap)
    {
        const uint32_t bad = check_segment<Rule, W>(kThreads, msg_bytes, BaseFromSmem{s_base4}, lo, hi, my_syn, rbit, cap);
        return (bad & 1u) | ((uint32_t)rbit << 1); // bit 0: parity failure, bits 1..: advanced round counter
    }

    constexpr int kResidentMaxCW = 16;
    constexpr int kQuietChecks = 16; // at most this many threads saw an unsatisfied check: the frame is about to converge
    constexpr int kBitUnroll = 1; // bits per thread in flight in the bit pass (2 measured no faster: the pass is bandwidth-, not latency-bound)
#ifndef QLB_RESIDENT_MAX_THREADS
#define QLB_RESIDENT_MAX_THREADS 1024
#endif
    constexpr int kResidentThreads = QLB_RESIDENT_MAX_THREADS; // launch bound (register budget: 64 at 1024, 80 at 768)
    constexpr size_t kResidentStaticSmem = 2 * kResidentThreads * 4 + 512; // static bookkeeping declared inside the kernel

    __host__ __device__ inline size_t resident_smem_bytes(int n, int m, int slots, int bw)
    {
        const size_t wn = align_up((size_t)(n + 31) / 32 * 4, 16), wm = align_up((size_t)(m + 31) / 32 * 4, 16);
        return align_up((size_t)slots * 4, 16) + align_up((size_t)bw * n * 2, 16) + 3 * wn + wm;
    }

    // One bit pass over the thread's bits: total (:256-258), hard decision (:259-266), extrinsic (+ clamp) (:300-316).
    // kClamp = false when the clamp cannot change what the check rule sees (see decode_resident_f32_kernel).
    template <bool kReconcile, bool kClamp, int kBW>
    __device__ __forceinline__ void bit_pass(const int kThreads, unsigned char *__restrict__ msg_bytes, const uint16_t *__restrict__ bslot, uint32_t *__restrict__ s_z,
                                             int n, uint32_t my_bob, float lp, const double *__restrict__ llr_f, float unit, float cap)
    {
        const int tid = threadIdx.x;
        const uint16_t *bs = bslot + tid;
        uint32_t *zw = s_z + (tid >> 5);
        const bool lane0 = (tid & 31) == 0;
#pragma unroll kBitUnroll
        for (int i = tid; i < n; i += kThreads)
        {
            float prior;
            if (kReconcile)
            {
                prior = __uint_as_float(__float_as_uint(lp) ^ (my_bob << 31));
                my_bob >>= 1;
            }
            else
                prior = __fmul_rn(unit, (float)llr_f[i]); // never contracted into the sum below: every fp32 kernel forms the same prior
            uint32_t sl[kBW];
            float c[kBW];
#pragma unroll
            for (int a = 0; a < kBW; ++a)
                sl[a] = 4u * (uint32_t)bs[a * n];
#pragma unroll
            for (int a = 0; a < kBW; ++a)
            {
                QLB_CHECK_INDEX(sl[a], g_bounds_msg_bytes);
                c[a] = *reinterpret_cast<const float *>(msg_bytes + sl[a]);
            }
            float total = prior;
#pragma unroll
            for (int a = 0; a < kBW; ++a)
                total = total + c[a];
            const bool z = total <= 0.f;
#pragma unroll
            for (int a = 0; a < kBW; ++a)
            {
                float v = total - c[a];
                if (kClamp)
                    v = fminf(fmaxf(v, -cap), cap);
                *reinterpret_cast<float *>(msg_bytes + sl[a]) = __uint_as_float((__float_as_uint(v) & ~1u) | (uint32_t)z);
            }
            const uint32_t word = __ballot_sync(0xffffffffu, z); // n % 32 == 0: whole warps only
            if (lane0)
                *zw = word;
            bs += kThreads;
            zw += kThreads >> 5;
        }
    }

    // Parity of the riding hard decisions against the target syndrome for every check this thread visits -- the convergence test
    // of :277-298 on its own, without the check rule. Bit 0 of the result: some check of this thread fails. Out of line: it runs
    // once or twice per converging frame and must not cost the hot loops a register.
    static __device__ __noinline__ uint32_t parity_walk(const int kThreads, const unsigned char *__restrict__ msg_bytes, const uint32_t *s_base4,
                                                        const uint32_t *s_seg_w, const uint32_t *s_seg_lo, const uint32_t *s_seg_hi, int nseg, uint32_t my_syn)
    {
        uint32_t bad = 0;
        int r = 0;
        for (int sg = 0; sg < nseg; ++sg)
        {
            const int w = (int)s_seg_w[sg];
            for (uint32_t p = s_seg_lo[sg] + threadIdx.x; p < s_seg_hi[sg]; p += kThreads, ++r)
            {
                uint32_t x = my_syn >> r;
                for (int k = 0; k < w; ++k)
                    x ^= *reinterpret_cast<const uint32_t *>(msg_bytes + s_base4[k] + 4u * p);
                bad |= x;
            }
        }
        return bad & 1u;
    }

    // kBW: the (uniform) bit weight. Host-checked requirements: slots < 65535, max_check_w <= 16, every bit of weight kBW,
    // n % 32 == 0, and m, n <= 32 * kThreads (one register bit per node a thread visits).
    template <typename Rule, bool kReconcile, int kBW, int kMaxThreads>
    __global__ void __launch_bounds__(kMaxThreads, 1) decode_resident_f32_kernel(const DecodeArgs args)
    {
        const int kThreads = blockDim.x; // multiple of 32 chosen by the host (balanced_block_size), <= kMaxThreads
        extern __shared__ __align__(16) unsigned char smem[];
        // small bookkeeping at fixed (static) shared addresses
        __shared__ uint32_t s_seg_w[kResidentMaxCW + 1], s_seg_lo[kResidentMaxCW + 1], s_seg_hi[kResidentMaxCW + 1];
        __shared__ uint32_t s_base4[kResidentMaxCW];
        __shared__ uint32_t s_park_bob[kMaxThreads], s_park_syn[kMaxThreads];
        __shared__ int s_nseg;
        __shared__ __align__(8) uint64_t s_bar;
        __shared__ long long s_frame;

        const CodeDev &code = args.code;
        const int n = code.n, m = code.m, tid = threadIdx.x, lane = tid & 31;
        const int words_n = code.words_n, words_m = code.words_m;
        const size_t wn = align_up((size_t)words_n * 4, 16);
        const uint32_t idx_bytes = (uint32_t)align_up((size_t)kBW * n * 2, 16);

        float *msg = reinterpret_cast<float *>(smem);
        unsigned char *msg_bytes = smem;
        uint16_t *bslot = reinterpret_cast<uint16_t *>(smem + align_up((size_t)code.slots * 4, 16));
        unsigned char *tail = reinterpret_cast<unsigned char *>(bslot) + idx_bytes;
        uint32_t *s_bob = reinterpret_cast<uint32_t *>(tail);
        uint32_t *s_alice = reinterpret_cast<uint32_t *>(tail + wn);
        uint32_t *s_z = reinterpret_cast<uint32_t *>(tail + 2 * wn);
        uint32_t *s_synn = reinterpret_cast<uint32_t *>(tail + 3 * wn); // syndrome, natural check order

        // stage the bit->slot table: one TMA bulk copy per CTA (the table is 16-byte padded on the device)
        if (tid == 0)
        {
            mbar_init(&s_bar, 1);
            // weight segments of the sorted checks: [lo, hi) holds the checks of weight exactly w; w = 0 last
            int ns = 0;
            for (int w = code.max_check_w; w >= 0; --w)
            {
                const uint32_t lo = (w < code.max_check_w) ? code.cnt[w] : 0u, hi = (w > 0) ? code.cnt[w - 1] : (uint32_t)m;
                if (lo < hi)
                {
                    s_seg_w[ns] = (uint32_t)w;
                    s_seg_lo[ns] = lo;
                    s_seg_hi[ns] = hi;
                    ++ns;
                }
            }
            s_nseg = ns;
        }
        if (tid < kResidentMaxCW)
            s_base4[tid] = code.base4[tid];
        __syncthreads();
        if (tid == 0)
        {
            mbar_expect_tx(&s_bar, idx_bytes);
            tma_bulk_g2s(bslot, code.bit_slots16, idx_bytes, &s_bar);
        }
        mbar_wait(&s_bar, 0);

        const float unit = Rule::kUnit;
        const float cap = args.cap_f32 * unit;
        // Below |m| = 2^-25-resolution the fast rule maps every message to exactly (1-e, 1+e) = (1, 1): clamping bit-to-check
        // messages at a threshold >= 25 base-2 units cannot change any later value, so that clamp is skipped.
        const bool clamp_b2c = !(Rule::kUnit != 1.f && cap >= 25.f);
        const int nseg = s_nseg;
        const typename Rule::Arg rule_arg = Rule::check_arg(cap, args.ms_scale);

        for (;;)
        {
            __syncthreads();
            if (tid == 0)
                s_frame = (long long)atomicAdd(args.queue, 1ULL);
            __syncthreads();
            const long long f = s_frame;
            if (f >= args.n_frames)
                break;

            // ---- frame set-up ------------------------------------------------------------------------------------
            float lp = 0.f;
            const double *llr_f = nullptr;
            if (kReconcile)
            {
                lp = unit * (float)args.log_prior[f];
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

            // messages <- priors (src/qkd_ldpc_algorithm.cpp:182-190); in reconcile mode Alice's bit rides in bit 0 so
            // that the parity of the first walk over the checks is her syndrome (:413-414). Bob's bit of the r-th bit this
            // thread visits is parked as bit r of s_park_bob[tid].
            {
                uint32_t my_bob = 0;
                int r = 0;
                for (int i = tid; i < n; i += kThreads, ++r)
                {
                    float prior;
                    uint32_t abit = 0;
                    if (kReconcile)
                    {
                        const uint32_t bb = (s_bob[i >> 5] >> lane) & 1u;
                        abit = (s_alice[i >> 5] >> lane) & 1u;
                        my_bob |= bb << r;
                        prior = bb ? -lp : lp;
                    }
                    else
                        prior = __fmul_rn(unit, (float)llr_f[i]);
                    const float pv = __uint_as_float((__float_as_uint(prior) & ~1u) | abit);
#pragma unroll
                    for (int a = 0; a < kBW; ++a)
                        msg[bslot[a * n + i]] = pv;
                }
                s_park_bob[tid] = my_bob;
            }
            __syncthreads();

            // target syndrome bit of the r-th check this thread visits (same walk as the check pass) -> bit r
            {
                uint32_t my_syn = 0;
                int r = 0;
                for (int sg = 0; sg < nseg; ++sg)
                {
                    const int w = (int)s_seg_w[sg];
                    for (uint32_t p = s_seg_lo[sg] + tid; p < s_seg_hi[sg]; p += kThreads, ++r)
                    {
                        const uint32_t j = code.check_order[p];
                        uint32_t bit = 0;
                        if (kReconcile)
                        {
                            for (int k = 0; k < w; ++k)
                                bit ^= __float_as_uint(msg[code.base[k] + p]);
                            bit &= 1u;
                            if (bit && args.syndrome_out)
                                atomicOr(&s_synn[j >> 5], 1u << (j & 31));
                        }
                        else
                            bit = (s_synn[j >> 5] >> (j & 31)) & 1u;
                        my_syn |= bit << r;
                    }
                }
                s_park_syn[tid] = my_syn;
            }
            // (no barrier needed: every thread only re-reads the slots of its own checks next)

            // ---- iterations ----------------------------------------------------------------------------------------
            // `it` counts completed bit passes. The check pass of round `it` also evaluates the parity of the hard
            // decisions of bit pass `it` (meaningless for it == 0: bit 0 then still holds Alice's / zero bits).
            // A converged frame would otherwise pay one more full check pass just to learn it. When the previous check pass saw only
            // a handful of unsatisfied checks -- the signature of the last rounds of a converging frame, never of a failing one,
            // which keeps hundreds of them -- the parity is looked at on its own first (~1/4 of a check pass).
            int it = 0;
            bool success = false, quiet = false;
            for (;;)
            {
                if (Rule::kParityFirst && quiet && it > 0 && !__syncthreads_or((int)parity_walk(kThreads, msg_bytes, s_base4, s_seg_w, s_seg_lo, s_seg_hi, nseg, s_park_syn[tid])))
                {
                    success = true; // :285-298
                    break;
                }
                uint32_t bad = 0;
                {
                    const uint32_t my_syn = s_park_syn[tid];
                    int rbit = 0;
#pragma unroll 1
                    for (int sg = 0; sg < nseg; ++sg)
                    {
                        const uint32_t lo = s_seg_lo[sg], hi = s_seg_hi[sg];
                        switch (s_seg_w[sg])
                        {
#define QLB_SEG(W_) case W_: bad |= check_segment<Rule, W_>(kThreads, msg_bytes, BaseFromParams{args}, lo, hi, my_syn, rbit, rule_arg); break;
#define QLB_SEGW(W_) case W_: { const uint32_t rv = check_segment_wide<Rule, W_>(kThreads, msg_bytes, s_base4, lo, hi, my_syn, rbit, rule_arg); bad |= rv & 1u; rbit = (int)(rv >> 1); } break;
                            QLB_SEG(1) QLB_SEG(2) QLB_SEG(3) QLB_SEG(4) QLB_SEG(5) QLB_SEG(6) QLB_SEG(7) QLB_SEG(8)
                            QLB_SEGW(9) QLB_SEGW(10) QLB_SEGW(11) QLB_SEGW(12) QLB_SEGW(13) QLB_SEGW(14) QLB_SEGW(15) QLB_SEGW(16)
#undef QLB_SEG
#undef QLB_SEGW
                        default: // checks without edges can only be satisfied by a zero syndrome bit
                            for (uint32_t p = lo + tid; p < hi; p += kThreads, ++rbit)
                                bad |= (my_syn >> rbit) & 1u;
                            break;
                        }
                    }
                }
                const int any_bad = __syncthreads_count((int)(bad & 1u)); // threads with an unsatisfied check
                if (it > 0 && !any_bad)
                {
                    success = true; // the decisions of bit pass `it` satisfy the syndrome (:285-298)
                    break;
                }
                quiet = Rule::kParityFirst && it > 0 && any_bad <= kQuietChecks;
                if (it == args.max_it)
                    break; // :337-344
                if (clamp_b2c)
                    bit_pass<kReconcile, true, kBW>(kThreads, msg_bytes, bslot, s_z, n, s_park_bob[tid], lp, llr_f, unit, cap);
                else
                    bit_pass<kReconcile, false, kBW>(kThreads, msg_bytes, bslot, s_z, n, s_park_bob[tid], lp, llr_f, unit, cap);
                ++it;
                __syncthreads();
            }

            // ---- results -------------------------------------------------------------------------------------------
            int differs = 0;
            for (int w = tid; w < words_n; w += kThreads)
            {
                const uint32_t zw = s_z[w];
                if (args.decoded)
                    args.decoded[f * words_n + w] = zw;
                if (kReconcile)
                    differs |= (zw != s_alice[w]);
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
                args.iterations[f] = (uint32_t)it;
                args.result[f] = r;
                atomicAdd(args.iter_total, (unsigned long long)it);
            }
        }
    }
}
