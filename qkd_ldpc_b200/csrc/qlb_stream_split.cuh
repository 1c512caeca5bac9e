// The frame-interleaved streaming decoder (layout and node helpers in qlb_stream_common.cuh): data layout (msg[slot][G], keys and
// decisions bit-transposed per group), same node arithmetic (stream_check, the resident kernel's rules), but every pass of
// the flooding schedule is its own kernel over ALL groups of the launch:
//
//     setup init | check(0) update(0) bit | check(1) update(1) bit | ... | check(max_it) update(max_it) | finalize
//
// Why: a persistent one-CTA-per-group kernel (the first version, retired) ties a group to one SM for its whole life -- it needs as many groups as SMs
// (N = 1 000 000: HBM holds 99 groups, so 49 SMs idle), the last groups of a launch run on a mostly empty chip, and one
// register budget (128) has to serve both passes, capping the bit pass at 16 warps per SM although it is pure gather/scatter.
// Here work items are (group, chunk of consecutive nodes), spread evenly over a grid sized to the SM count; the check kernel
// and the bit kernel each get the register count and occupancy that suits them, kernel boundaries are the grid barriers, and
// groups whose frames have all converged drop out of the work list (group-granular active-frame compaction; converged
// frames inside a live group are frozen as before). No host synchronisation: every kernel reads the number of live
// groups from device memory and returns at once when it is zero.
// Bundles: B groups share one message array, interleaved slot by slot (msg[slot][B][G]), and the B rows of a slot are
// handled by adjacent warps of one CTA. The bit pass is a random gather of rows; with B = 4 the unit the DRAM sees is 2 KB
// instead of 512 B (measured on B200, N = 100 000: bit kernel 3.4 TB/s at B = 1 against 5.4 TB/s for the sequential check
// kernel -- row-buffer locality, not occupancy, is what the gather lacks). Bookkeeping stays per group.
// Results are identical to the SM-resident kernels of the same precision, frame by frame (tests/test_gpu_codes.py). fp32 and fp64 share
// every kernel here through a precision policy (StreamF32<Rule> / StreamF64<Math>, qlb_stream_common.cuh).
#pragma once
#include "qlb_stream_common.cuh"

namespace qlb
{
    // tuning knobs (compile-time so that each kernel gets its own register budget); defaults = best measured on B200
#ifndef QLB_SPLIT_CHECK_THREADS
#define QLB_SPLIT_CHECK_THREADS 256
#endif
#ifndef QLB_SPLIT_CHECK_MINB
#define QLB_SPLIT_CHECK_MINB 2
#endif
#ifndef QLB_SPLIT_BIT_THREADS
#define QLB_SPLIT_BIT_THREADS 256
#endif
#ifndef QLB_SPLIT_BIT_MINB
#define QLB_SPLIT_BIT_MINB 4
#endif
#ifndef QLB_SPLIT_BIT_U
#define QLB_SPLIT_BIT_U 2 // bits per warp in flight
#endif
    // the fp64 check pass is bound by FP64 issue, not by the loads in flight: more, leaner warps (measured on B200, below)
#ifndef QLB_SPLIT64_CHECK_THREADS
#define QLB_SPLIT64_CHECK_THREADS 256
#endif
#ifndef QLB_SPLIT64_CHECK_MINB
#define QLB_SPLIT64_CHECK_MINB 2
#endif
    constexpr int kSplitBitThreads = QLB_SPLIT_BIT_THREADS, kSplitSetupThreads = 512;
    template <typename P>
    struct SplitTune
    {
        static constexpr int kCheckThreads = P::kLsbDecision ? QLB_SPLIT_CHECK_THREADS : QLB_SPLIT64_CHECK_THREADS;
        static constexpr int kCheckMinB = P::kLsbDecision ? QLB_SPLIT_CHECK_MINB : QLB_SPLIT64_CHECK_MINB;
        static constexpr int kCheckChunk = 8 * (kCheckThreads / 32); // sorted check positions per work item
#ifndef QLB_SPLIT64_BIT_U
#define QLB_SPLIT64_BIT_U QLB_SPLIT_BIT_U
#endif
#ifndef QLB_STREAM64_BUNDLE
#define QLB_STREAM64_BUNDLE 4
#endif
        static constexpr int kBitU = P::kLsbDecision ? QLB_SPLIT_BIT_U : QLB_SPLIT64_BIT_U; // bits per warp in flight
        static constexpr int kBundle = P::kLsbDecision ? 4 : QLB_STREAM64_BUNDLE;           // groups per bundle
    };
    constexpr int kSplitBitChunk = 16 * (kSplitBitThreads / 32);    // bits per work item

    struct SplitState
    {
        unsigned char *bundles; // per bundle: the interleaved message array, then the B per-group carves (split_small_carve)
        size_t bundle_stride;
        uint32_t *act;  // [n_groups][4] word j, bit l: frame VEC*l + j of the group still decoding
        uint32_t *bad;  // [n_groups][4] same indexing: some check of that frame failed in the last check pass
        uint32_t *succ; // [n_groups][4] frames whose decisions satisfied the syndrome
        uint32_t *list; // [n_bundles] bundles with a live group, [0, *n_live)
        uint32_t *n_live;
        long long group0; // index of this wave's first group in the whole batch (initially frame = (group0 + g) * G + column)
        int n_groups;
        int bundle; // B: groups per bundle (1, 2, 4 or 8; divides the warps per CTA of the pass kernels)
        // frame-granular compaction (stream_repack_* kernels)
        uint32_t *fmap;     // [n_groups][G] frame index held by each column (kNoFrame: none); column = VEC * lane + j
        uint32_t *src_of;   // [n_groups][G] repack plan: old column id (g * G + column) that moves to new column id k
        uint32_t *fmap_new; // [n_groups][G]
        uint32_t *repack;   // [0] repack decided, [1] live frames, [2] groups after the repack
        int repack_pct;     // repack when the live columns are at most this percentage of the streamed ones
    };
    constexpr uint32_t kNoFrame = 0xFFFFFFFFu;
    constexpr int kMaxRepackGroups = 256; // per wave: the bit-array move stages one word per group and frame word in shared memory

    // per-group arrays other than the messages (bytes)
    struct SplitSmall
    {
        size_t bobT, aliceT, zT, synT, total;
    };
    __host__ __device__ inline SplitSmall split_small_carve(int n, int m, int vec)
    {
        SplitSmall c{};
        size_t o = 0;
        c.bobT = o; o += align_up((size_t)n * vec * 4, 256);
        c.aliceT = o; o += align_up((size_t)n * vec * 4, 256);
        c.zT = o; o += align_up((size_t)n * vec * 4, 256);
        c.synT = o; o += align_up((size_t)m * vec * 4, 256);
        c.total = o;
        return c;
    }
    // real_bytes: 4 (fp32 messages) or 8 (fp64)
    __host__ __device__ inline size_t split_bundle_bytes(int n, int m, int slots, int vec, int bundle, int real_bytes)
    {
        return align_up((size_t)slots * bundle * 32 * vec * real_bytes, 256) + (size_t)bundle * split_small_carve(n, m, vec).total;
    }

    template <typename Real>
    struct SplitGroup
    {
        Real *msg;         // row of slot s for this group: msg + s * row_stride (+ VEC * lane)
        uint32_t row_stride; // B * G values; slot * row_stride < 2^32 (checked by the launcher), so row offsets are 32-bit products
        uint32_t *bobT, *aliceT, *zT, *synT;
    };
    template <typename Real>
    __device__ __forceinline__ SplitGroup<Real> split_group(const SplitState &st, const CodeDev &code, int vec, uint32_t g)
    {
        const int B = st.bundle, G = 32 * vec;
        const uint32_t bu = g / (uint32_t)B, gb = g % (uint32_t)B;
        const SplitSmall cv = split_small_carve(code.n, code.m, vec);
        unsigned char *p = st.bundles + (size_t)bu * st.bundle_stride;
        QLB_CHECK_INDEX(g, st.n_groups);
        QLB_CHECK_INDEX(align_up((size_t)code.slots * B * G * sizeof(Real), 256) + (size_t)(gb + 1) * cv.total - 1, st.bundle_stride);
        unsigned char *small = p + align_up((size_t)code.slots * B * G * sizeof(Real), 256) + (size_t)gb * cv.total;
        SplitGroup<Real> r;
        r.msg = reinterpret_cast<Real *>(p) + (size_t)gb * G;
        r.row_stride = (uint32_t)(B * G);
        r.bobT = reinterpret_cast<uint32_t *>(small + cv.bobT);
        r.aliceT = reinterpret_cast<uint32_t *>(small + cv.aliceT);
        r.zT = reinterpret_cast<uint32_t *>(small + cv.zT);
        r.synT = reinterpret_cast<uint32_t *>(small + cv.synT);
        return r;
    }

    // weight segments of the sorted checks into shared memory (thread 0), as in the other kernels
    __device__ __forceinline__ int split_segments(const CodeDev &code, uint32_t *s_seg_w, uint32_t *s_seg_lo, uint32_t *s_seg_hi)
    {
        int ns = 0;
        for (int w = code.max_check_w; w >= 0; --w)
        {
            const uint32_t lo = (w < code.max_check_w) ? code.cnt[w] : 0u, hi = (w > 0) ? code.cnt[w - 1] : (uint32_t)code.m;
            if (lo < hi)
            {
                s_seg_w[ns] = (uint32_t)w;
                s_seg_lo[ns] = lo;
                s_seg_hi[ns] = hi;
                ++ns;
            }
        }
        return ns;
    }

    // ---- set-up, part 1: transposed keys / syndromes and frame bookkeeping; one CTA per group at a time --------------------------
    template <typename Real, bool kReconcile, int VEC>
    __global__ void __launch_bounds__(kSplitSetupThreads) stream_setup_kernel(const DecodeArgs args, const SplitState st)
    {
        constexpr int G = 32 * VEC;
        const CodeDev &code = args.code;
        const int n = code.n, m = code.m, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
        for (uint32_t g = blockIdx.x; g < (uint32_t)st.n_groups; g += gridDim.x)
        {
            const SplitGroup<Real> sg = split_group<Real>(st, code, VEC, g);
            const long long f0 = (st.group0 + g) * G;
            if (kReconcile)
            {
                transpose_in<VEC>(args.bob, f0, args.n_frames, code.words_n, n, sg.bobT);
                transpose_in<VEC>(args.alice, f0, args.n_frames, code.words_n, n, sg.aliceT);
            }
            else
            {
                transpose_in<VEC>(args.syndrome_in, f0, args.n_frames, code.words_m, m, sg.aliceT);
                __syncthreads();
                for (int p = tid; p < m; p += kSplitSetupThreads)
#pragma unroll
                    for (int j = 0; j < VEC; ++j)
                        sg.synT[(size_t)p * VEC + j] = sg.aliceT[(size_t)code.check_order[p] * VEC + j];
            }
            if (warp == 0)
            {
#pragma unroll
                for (int j = 0; j < VEC; ++j)
                {
                    const long long f = f0 + (long long)VEC * lane + j;
                    const bool live = f < args.n_frames;
                    if (live)
                        args.iterations[f] = (uint32_t)args.max_it;
                    st.fmap[(size_t)g * G + VEC * lane + j] = live ? (uint32_t)f : kNoFrame;
                    const uint32_t word = __ballot_sync(0xffffffffu, live);
                    if (lane == 0)
                    {
                        st.act[g * 4 + j] = word;
                        st.bad[g * 4 + j] = 0;
                        st.succ[g * 4 + j] = 0;
                    }
                }
                if (lane == 0 && g % (uint32_t)st.bundle == 0)
                    st.list[g / (uint32_t)st.bundle] = g / (uint32_t)st.bundle;
            }
            __syncthreads();
        }
        if (blockIdx.x == 0 && tid == 0)
            *st.n_live = (uint32_t)((st.n_groups + st.bundle - 1) / st.bundle);
    }

    // ---- set-up, part 2: messages <- priors (src/qkd_ldpc_algorithm.cpp:182-190), Alice's bit riding in bit 0 (reconcile mode) so
    // that the first check pass yields her syndrome; decisions <- 0. Same work split as the bit pass: (bundle, chunk of bits),
    // adjacent warps on the B groups of the bundle, so the scattered rows are written in 2 KB units.
    template <typename P, typename Real>
    __device__ __forceinline__ Real stream_unit()
    {
        if constexpr (P::kLsbDecision)
            return P::Rule::kUnit;
        else
            return Real(1);
    }
    // the prior of a bit whose received value is `bb` (src/qkd_ldpc_algorithm.cpp:401-405): +-lp
    __device__ __forceinline__ float stream_signed(float lp, uint32_t bb) { return __uint_as_float(__float_as_uint(lp) ^ (bb << 31)); }
    __device__ __forceinline__ double stream_signed(double lp, uint32_t bb) { return __hiloint2double(__double2hiint(lp) ^ (int)(bb << 31), __double2loint(lp)); }

    template <typename P, bool kReconcile, int kBW, int VEC>
    __global__ void __launch_bounds__(kSplitBitThreads) stream_init_kernel(const DecodeArgs args, const SplitState st)
    {
        typedef typename P::real Real;
        constexpr int G = 32 * VEC;
        constexpr int kWarps = kSplitBitThreads / 32;
        const CodeDev &code = args.code;
        const int n = code.n, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const Real unit = stream_unit<P, Real>();
        const int B = st.bundle, step = kWarps / B;
        const uint32_t n_bundles = (uint32_t)((st.n_groups + B - 1) / B);
        const uint32_t chunks = ((uint32_t)n + kSplitBitChunk - 1) / kSplitBitChunk;
        const unsigned long long items = (unsigned long long)n_bundles * chunks;
        for (unsigned long long item = blockIdx.x; item < items; item += gridDim.x)
        {
            const uint32_t g = (uint32_t)(item / chunks) * (uint32_t)B + (uint32_t)(warp % B);
            const int i0 = (int)(item % chunks) * kSplitBitChunk, i1 = min(n, i0 + kSplitBitChunk);
            if (g >= (uint32_t)st.n_groups)
                continue;
            const SplitGroup<Real> sg = split_group<Real>(st, code, VEC, g);
            const long long f0 = (st.group0 + g) * G;
            Real lp[VEC];
#pragma unroll
            for (int j = 0; j < VEC; ++j)
            {
                const long long f = f0 + (long long)VEC * lane + j;
                lp[j] = (kReconcile && f < args.n_frames) ? unit * (Real)args.log_prior[f] : Real(0);
            }
            for (int i = i0 + warp / B; i < i1; i += step)
            {
                Real pv[VEC];
#pragma unroll
                for (int j = 0; j < VEC; ++j)
                {
                    Real prior;
                    uint32_t abit = 0;
                    if (kReconcile)
                    {
                        const uint32_t bb = (sg.bobT[(size_t)i * VEC + j] >> lane) & 1u;
                        abit = (sg.aliceT[(size_t)i * VEC + j] >> lane) & 1u;
                        prior = stream_signed(lp[j], bb);
                    }
                    else
                    {
                        const long long f = f0 + (long long)VEC * lane + j;
                        if constexpr (P::kLsbDecision)
                            prior = f < args.n_frames ? __fmul_rn(unit, (float)args.llr[f * n + i]) : 0.f;
                        else
                            prior = f < args.n_frames ? args.llr[f * n + i] : 0.;
                    }
                    if constexpr (P::kLsbDecision)
                        pv[j] = __uint_as_float((__float_as_uint(prior) & ~1u) | abit); // Alice's bit rides in bit 0 through the first check pass
                    else
                        pv[j] = prior; // unclamped (:182-190)
                }
                if constexpr (kBW > 0)
                {
#pragma unroll
                    for (int a = 0; a < kBW; ++a)
                    {
                        QLB_CHECK_INDEX(code.bit_slots32[(size_t)a * n + i], code.slots);
                        VecIO<Real, VEC>::store(sg.msg + VEC * lane + (size_t)(code.bit_slots32[(size_t)a * n + i] * sg.row_stride), pv);
                    }
                }
                else // any bit weights: the bit's list ends at the first empty entry
                    for (int a = 0; a < code.max_bit_w; ++a)
                    {
                        const uint32_t slot = code.bit_slots32[(size_t)a * n + i];
                        if (slot == 0xFFFFFFFFu)
                            break;
                        QLB_CHECK_INDEX(slot, code.slots);
                        VecIO<Real, VEC>::store(sg.msg + VEC * lane + (size_t)(slot * sg.row_stride), pv);
                    }
                if (lane == 0)
#pragma unroll
                    for (int j = 0; j < VEC; ++j)
                        sg.zT[(size_t)i * VEC + j] = 0;
            }
        }
    }

    // ---- check pass over the live bundles: work item = (bundle, kSplitCheckChunk consecutive sorted checks) -------------------
    template <typename P, bool kReconcile, int VEC>
    __global__ void __launch_bounds__(SplitTune<P>::kCheckThreads, SplitTune<P>::kCheckMinB) stream_check_kernel(const DecodeArgs args, const SplitState st, int it)
    {
        typedef typename P::real Real;
        constexpr int kSplitCheckThreads = SplitTune<P>::kCheckThreads, kSplitCheckChunk = SplitTune<P>::kCheckChunk;
        constexpr int kWarps = kSplitCheckThreads / 32;
        __shared__ uint32_t s_seg_w[kResidentMaxCW + 1], s_seg_lo[kResidentMaxCW + 1], s_seg_hi[kResidentMaxCW + 1];
        const uint32_t n_live = *st.n_live;
        if (n_live == 0)
            return;
        const CodeDev &code = args.code;
        const int m = code.m, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        if (threadIdx.x == 0)
            split_segments(code, s_seg_w, s_seg_lo, s_seg_hi);
        __syncthreads();
        const float cap = args.cap_f32 * (float)stream_unit<P, Real>();
        const double thr_eff = args.enable_thr ? args.thr : __longlong_as_double(0x7ff0000000000000LL); // fp64: the clamp as an operand
        const bool want_inf = !(thr_eff <= 700.);
        (void)cap; (void)thr_eff; (void)want_inf;
        const bool first = kReconcile && it == 0;
        const uint32_t chunks = ((uint32_t)m + kSplitCheckChunk - 1) / kSplitCheckChunk;
        const unsigned long long items = (unsigned long long)n_live * chunks;
        const int B = st.bundle, step = kWarps / B; // adjacent warps: the B groups of the bundle on the same check
        for (unsigned long long item = blockIdx.x; item < items; item += gridDim.x)
        {
            const uint32_t g = st.list[item / chunks] * (uint32_t)B + (uint32_t)(warp % B);
            const uint32_t p0 = (uint32_t)(item % chunks) * kSplitCheckChunk, p1 = min((uint32_t)m, p0 + kSplitCheckChunk);
            if (g >= (uint32_t)st.n_groups)
                continue;
            uint32_t alive = 0;
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                alive |= st.act[g * 4 + j];
            if (!alive)
                continue; // every frame of this group has converged: its rows are left alone
            const SplitGroup<Real> sg = split_group<Real>(st, code, VEC, g);
            Real *__restrict__ msg = sg.msg;
            const uint32_t *bitsT = first ? sg.aliceT : sg.zT; // fp64: what a check's parity is formed from
            (void)bitsT;
            const uint32_t rs = sg.row_stride;
            uint32_t bad[VEC];
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                bad[j] = 0;
            int s = 0;
#pragma unroll 1
            for (uint32_t p = p0 + warp / B; p < p1; p += step)
            {
                while (p >= s_seg_hi[s])
                    ++s;
                if (p + step < p1) // the rows of this warp's next check -> L2 while this one is computed (cnt[k]: checks with an edge position k)
                    for (int k = 0; k < (int)s_seg_w[s]; ++k)
                        if (p + step < code.cnt[k])
                            prefetch_l2(msg + VEC * lane + (size_t)((code.base[k] + p + step) * rs));
                switch (s_seg_w[s])
                {
#define QLB_PSEG(W_)                                                                                                          \
    case W_:                                                                                                                  \
        if constexpr (P::kLsbDecision)                                                                                        \
            stream_check<typename P::Rule, W_, VEC>(msg, code, p, lane, sg.synT, P::Rule::check_arg(cap, args.ms_scale), first, bad, rs); \
        else                                                                                                                  \
            stream_check64<typename P::Math, W_, VEC>(msg, code, p, lane, sg.synT, bitsT, thr_eff, want_inf, first, bad, rs); \
        break;
                    QLB_PSEG(1) QLB_PSEG(2) QLB_PSEG(3) QLB_PSEG(4) QLB_PSEG(5) QLB_PSEG(6) QLB_PSEG(7) QLB_PSEG(8)
                    QLB_PSEG(9) QLB_PSEG(10) QLB_PSEG(11) QLB_PSEG(12) QLB_PSEG(13) QLB_PSEG(14) QLB_PSEG(15) QLB_PSEG(16)
#undef QLB_PSEG
                default: // a check without edges is satisfied only by a zero syndrome bit
#pragma unroll
                    for (int j = 0; j < VEC; ++j)
                    {
                        if (first)
                        {
                            if (lane == 0)
                                sg.synT[(size_t)p * VEC + j] = 0;
                        }
                        else
                            bad[j] |= (sg.synT[(size_t)p * VEC + j] >> lane) & 1u;
                    }
                    break;
                }
            }
            if (!first)
#pragma unroll
                for (int j = 0; j < VEC; ++j)
                {
                    const uint32_t word = __ballot_sync(0xffffffffu, bad[j] & 1u);
                    if (lane == 0 && word)
                        atomicOr(&st.bad[g * 4 + j], word);
                }
        }
    }

    // ---- frame bookkeeping between the check pass and the bit pass of round `it` (one small CTA) ----------------------------------
    // Frames whose last decisions satisfied every check are done (src/qkd_ldpc_algorithm.cpp:285-298): iterations = it. Groups
    // without a live frame leave the work list.
    template <int VEC>
    __global__ void __launch_bounds__(1024) stream_update_kernel(const DecodeArgs args, const SplitState st, int it)
    {
        constexpr int G = 32 * VEC;
        __shared__ uint32_t s_count;
        if (*st.n_live == 0)
            return;
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
        if (threadIdx.x == 0)
            s_count = 0;
        __syncthreads();
        const int B = st.bundle;
        const uint32_t n_bundles = (uint32_t)((st.n_groups + B - 1) / B);
        for (uint32_t bu = warp; bu < n_bundles; bu += nwarps)
        {
            // lane = 4 * (group within the bundle) + word j
            const uint32_t g = bu * (uint32_t)B + (uint32_t)(lane >> 2);
            const int j = lane & 3;
            uint32_t a = 0;
            if ((lane >> 2) < B && j < VEC && g < (uint32_t)st.n_groups)
            {
                a = st.act[g * 4 + j];
                const uint32_t b = st.bad[g * 4 + j];
                if (it > 0 && a)
                {
                    uint32_t done = a & ~b;
                    if (done)
                    {
                        st.succ[g * 4 + j] |= done;
                        a &= ~done;
                        st.act[g * 4 + j] = a;
                        while (done)
                        {
                            const int l = __ffs(done) - 1;
                            done &= done - 1;
                            QLB_CHECK_INDEX(st.fmap[(size_t)g * G + VEC * l + j], args.n_frames);
                            args.iterations[st.fmap[(size_t)g * G + VEC * l + j]] = (uint32_t)it;
                        }
                    }
                }
                st.bad[g * 4 + j] = 0;
            }
            const uint32_t any = __ballot_sync(0xffffffffu, a != 0);
            if (lane == 0 && any)
                st.list[atomicAdd(&s_count, 1u)] = bu;
        }
        __syncthreads();
        if (threadIdx.x == 0)
            *st.n_live = s_count;
    }

    // ---- bit pass over the live bundles: work item = (bundle, kSplitBitChunk consecutive bits), U bits per warp in flight -----------
    // fr[j]: frame index held by this lane's column j (kNoFrame: none)
    template <typename P, bool kReconcile, int kBW, int VEC, int U>
    __device__ __forceinline__ void split_bits(const DecodeArgs &args, const SplitGroup<typename P::real> &sg, const int (&bit)[U], int lane,
                                               const typename P::real (&lp)[VEC], const uint32_t (&act_word)[VEC], const uint32_t (&fr)[VEC],
                                               typename P::real unit, typename P::real cap, bool clamp_b2c)
    {
        typedef typename P::real Real;
        const CodeDev &code = args.code;
        const int n = code.n;
        Real *row[U][kBW];
        Real c[U][kBW][VEC];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int a = 0; a < kBW; ++a)
            {
                QLB_CHECK_INDEX(bit[u], n);
                QLB_CHECK_INDEX(code.bit_slots32[(size_t)a * n + bit[u]], code.slots);
                row[u][a] = sg.msg + VEC * lane + (size_t)(code.bit_slots32[(size_t)a * n + bit[u]] * sg.row_stride);
            }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int a = 0; a < kBW; ++a)
                VecIO<Real, VEC>::load(row[u][a], c[u][a]);
#pragma unroll
        for (int u = 0; u < U; ++u)
        {
            const int i = bit[u];
            Real total[VEC];
            uint32_t zbits = 0;
#pragma unroll
            for (int j = 0; j < VEC; ++j)
            {
                Real prior;
                if (kReconcile)
                    prior = stream_signed(lp[j], (sg.bobT[(size_t)i * VEC + j] >> lane) & 1u);
                else if constexpr (P::kLsbDecision)
                    prior = fr[j] != kNoFrame ? __fmul_rn(unit, (float)args.llr[(size_t)fr[j] * n + i]) : 0.f;
                else
                    prior = fr[j] != kNoFrame ? args.llr[(size_t)fr[j] * n + i] : 0.;
                Real t = prior; // left to right from the prior, in the bit's arrival order (:256-258)
#pragma unroll
                for (int a = 0; a < kBW; ++a)
                    t = t + c[u][a][j];
                total[j] = t;
                zbits |= (uint32_t)(t <= Real(0)) << j; // :259-266 (a NaN total decides 0)
            }
#pragma unroll
            for (int a = 0; a < kBW; ++a)
            {
                Real o[VEC];
#pragma unroll
                for (int j = 0; j < VEC; ++j)
                {
                    Real v = total[j] - c[u][a][j]; // :300-311
                    if constexpr (P::kLsbDecision)
                    {
                        if (clamp_b2c)
                            v = fminf(fmaxf(v, -cap), cap);
                        o[j] = __uint_as_float((__float_as_uint(v) & ~1u) | ((zbits >> j) & 1u));
                    }
                    else
                        o[j] = clamp_f64(v, cap); // :313-316; cap = +inf when the clamp is disabled, NaN passes
                }
                VecIO<Real, VEC>::store(row[u][a], o);
            }
#pragma unroll
            for (int j = 0; j < VEC; ++j)
            {
                const uint32_t word = __ballot_sync(0xffffffffu, (zbits >> j) & 1u);
                if (lane == 0)
                {
                    const size_t at = (size_t)i * VEC + j;
                    sg.zT[at] = (sg.zT[at] & ~act_word[j]) | (word & act_word[j]); // converged frames keep their decision
                }
            }
        }
    }

    // The same for a bit of ANY weight (irregular codes): nothing is held in registers between the sum and the extrinsic values --
    // the rows are read twice, the second time from L2 (they were fetched a moment ago), so the HBM traffic is unchanged.
    template <typename P, bool kReconcile, int VEC>
    __device__ __forceinline__ void split_bit_any_weight(const DecodeArgs &args, const SplitGroup<typename P::real> &sg, int i, int lane,
                                                         const typename P::real (&lp)[VEC], const uint32_t (&act_word)[VEC], const uint32_t (&fr)[VEC],
                                                         typename P::real unit, typename P::real cap, bool clamp_b2c)
    {
        typedef typename P::real Real;
        const CodeDev &code = args.code;
        const int n = code.n;
        QLB_CHECK_INDEX(i, n);
        Real total[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j)
        {
            if (kReconcile)
                total[j] = stream_signed(lp[j], (sg.bobT[(size_t)i * VEC + j] >> lane) & 1u);
            else if constexpr (P::kLsbDecision)
                total[j] = fr[j] != kNoFrame ? __fmul_rn(unit, (float)args.llr[(size_t)fr[j] * n + i]) : 0.f;
            else
                total[j] = fr[j] != kNoFrame ? args.llr[(size_t)fr[j] * n + i] : 0.;
        }
        for (int a = 0; a < code.max_bit_w; ++a) // left to right from the prior, in the bit's arrival order (:256-258)
        {
            const uint32_t slot = code.bit_slots32[(size_t)a * n + i];
            if (slot == 0xFFFFFFFFu)
                break;
            QLB_CHECK_INDEX(slot, code.slots);
            Real c[VEC];
            VecIO<Real, VEC>::load(sg.msg + VEC * lane + (size_t)(slot * sg.row_stride), c);
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                total[j] = total[j] + c[j];
        }
        uint32_t zbits = 0;
#pragma unroll
        for (int j = 0; j < VEC; ++j)
            zbits |= (uint32_t)(total[j] <= Real(0)) << j; // :259-266
        for (int a = 0; a < code.max_bit_w; ++a)
        {
            const uint32_t slot = code.bit_slots32[(size_t)a * n + i];
            if (slot == 0xFFFFFFFFu)
                break;
            Real *row = sg.msg + VEC * lane + (size_t)(slot * sg.row_stride);
            Real c[VEC], o[VEC];
            VecIO<Real, VEC>::load(row, c);
#pragma unroll
            for (int j = 0; j < VEC; ++j)
            {
                Real v = total[j] - c[j]; // :300-311
                if constexpr (P::kLsbDecision)
                {
                    if (clamp_b2c)
                        v = fminf(fmaxf(v, -cap), cap);
                    o[j] = __uint_as_float((__float_as_uint(v) & ~1u) | ((zbits >> j) & 1u));
                }
                else
                    o[j] = clamp_f64(v, cap);
            }
            VecIO<Real, VEC>::store(row, o);
        }
#pragma unroll
        for (int j = 0; j < VEC; ++j)
        {
            const uint32_t word = __ballot_sync(0xffffffffu, (zbits >> j) & 1u);
            if (lane == 0)
            {
                const size_t at = (size_t)i * VEC + j;
                sg.zT[at] = (sg.zT[at] & ~act_word[j]) | (word & act_word[j]);
            }
        }
    }

    template <typename P, bool kReconcile, int kBW, int VEC>
    __global__ void __launch_bounds__(kSplitBitThreads, QLB_SPLIT_BIT_MINB) stream_bit_kernel(const DecodeArgs args, const SplitState st)
    {
        typedef typename P::real Real;
        constexpr int G = 32 * VEC;
        constexpr int kWarps = kSplitBitThreads / 32;
        const uint32_t n_live = *st.n_live;
        if (n_live == 0)
            return;
        const CodeDev &code = args.code;
        const int n = code.n, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const Real unit = stream_unit<P, Real>();
        Real cap;
        bool clamp_b2c = true;
        if constexpr (P::kLsbDecision)
        {
            cap = args.cap_f32 * unit;
            clamp_b2c = !(unit != 1.f && cap >= 25.f);
        }
        else
            cap = args.enable_thr ? args.thr : __longlong_as_double(0x7ff0000000000000LL);
        const uint32_t chunks = ((uint32_t)n + kSplitBitChunk - 1) / kSplitBitChunk;
        const unsigned long long items = (unsigned long long)n_live * chunks;
        const int B = st.bundle, step = kWarps / B; // adjacent warps: the B groups of the bundle on the same bit
        for (unsigned long long item = blockIdx.x; item < items; item += gridDim.x)
        {
            const uint32_t g = st.list[item / chunks] * (uint32_t)B + (uint32_t)(warp % B);
            const int i0 = (int)(item % chunks) * kSplitBitChunk, i1 = min(n, i0 + kSplitBitChunk);
            if (g >= (uint32_t)st.n_groups)
                continue;
            const SplitGroup<Real> sg = split_group<Real>(st, code, VEC, g);
            Real lp[VEC];
            uint32_t act_word[VEC], fr[VEC], alive = 0;
#pragma unroll
            for (int j = 0; j < VEC; ++j)
            {
                fr[j] = st.fmap[(size_t)g * G + VEC * lane + j];
                lp[j] = (kReconcile && fr[j] != kNoFrame) ? unit * (Real)args.log_prior[fr[j]] : Real(0);
                act_word[j] = st.act[g * 4 + j];
                alive |= act_word[j];
            }
            if (!alive)
                continue;
            if constexpr (kBW == 0)
            {
#pragma unroll 1
                for (int i = i0 + warp / B; i < i1; i += step)
                    split_bit_any_weight<P, kReconcile, VEC>(args, sg, i, lane, lp, act_word, fr, unit, cap, clamp_b2c);
            }
            else
            {
                constexpr int U = SplitTune<P>::kBitU;
                int i = i0 + warp / B;
#pragma unroll 1
                for (; i + (U - 1) * step < i1; i += U * step)
                {
                    int many[U];
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        many[u] = i + u * step;
                    split_bits<P, kReconcile, kBW, VEC, U>(args, sg, many, lane, lp, act_word, fr, unit, cap, clamp_b2c);
                }
#pragma unroll 1
                for (; i < i1; i += step)
                {
                    const int one[1] = {i};
                    split_bits<P, kReconcile, kBW, VEC, 1>(args, sg, one, lane, lp, act_word, fr, unit, cap, clamp_b2c);
                }
            }
        }
    }

    // ---- results: flags, key comparison, decoded keys and syndromes back in frame-major order; one CTA per group at a time ----
    // only_done: called from a repack (and only when one was decided): the frames that have finished -- about to lose their
    // columns -- get their results now; the final call handles whatever the map still holds.
    template <typename Real, bool kReconcile, int VEC>
    __global__ void __launch_bounds__(kSplitSetupThreads) stream_finalize_kernel(const DecodeArgs args, const SplitState st, int only_done)
    {
        constexpr int G = 32 * VEC;
        constexpr int kWarps = kSplitSetupThreads / 32;
        __shared__ uint32_t s_flags[kWarps][4];
        if (only_done && !st.repack[0])
            return;
        const CodeDev &code = args.code;
        const int n = code.n, m = code.m, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
        for (uint32_t g = blockIdx.x; g < (uint32_t)st.n_groups; g += gridDim.x)
        {
            const SplitGroup<Real> sg = split_group<Real>(st, code, VEC, g);
            const uint32_t *fmap_g = st.fmap + (size_t)g * G;
            uint32_t keep[VEC], fr[VEC], any = 0; // keep[j] bit l: column (l, j) holds a frame this call reports
#pragma unroll
            for (int j = 0; j < VEC; ++j)
            {
                fr[j] = fmap_g[VEC * lane + j];
                keep[j] = __ballot_sync(0xffffffffu, fr[j] != kNoFrame) & (only_done ? ~st.act[g * 4 + j] : 0xFFFFFFFFu);
                any |= keep[j];
            }
            if (!any)
                continue;
            uint32_t differs = 0;
            if (kReconcile)
            {
                uint32_t d[VEC];
#pragma unroll
                for (int j = 0; j < VEC; ++j)
                    d[j] = 0;
                for (int i = tid; i < n; i += kSplitSetupThreads)
#pragma unroll
                    for (int j = 0; j < VEC; ++j)
                        d[j] |= sg.zT[(size_t)i * VEC + j] ^ sg.aliceT[(size_t)i * VEC + j];
#pragma unroll
                for (int j = 0; j < VEC; ++j)
                {
                    uint32_t x = d[j];
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1)
                        x |= __shfl_xor_sync(0xffffffffu, x, o);
                    if (lane == 0)
                        s_flags[warp][j] = x;
                }
                __syncthreads();
#pragma unroll
                for (int j = 0; j < VEC; ++j)
                {
                    uint32_t x = 0;
                    for (int w = 0; w < kWarps; ++w)
                        x |= s_flags[w][j];
                    differs |= ((x >> lane) & 1u) << j;
                }
            }
            if (warp == 0)
            {
                unsigned long long it_sum = 0;
#pragma unroll
                for (int j = 0; j < VEC; ++j)
                    if ((keep[j] >> lane) & 1u)
                    {
                        uint8_t r = (st.succ[g * 4 + j] >> lane) & 1u ? 1 : 0;
                        if (kReconcile && !((differs >> j) & 1u))
                            r |= 2;
                        QLB_CHECK_INDEX(fr[j], args.n_frames);
                        args.result[fr[j]] = r;
                        it_sum += args.iterations[fr[j]];
                    }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)
                    it_sum += __shfl_xor_sync(0xffffffffu, it_sum, o);
                if (lane == 0)
                    atomicAdd(args.iter_total, it_sum);
            }
            if (args.decoded)
                transpose_out<VEC>(sg.zT, 0, args.n_frames, code.words_n, n, args.decoded, fmap_g, keep);
            if (kReconcile && args.syndrome_out)
                for (int p = warp; p < m; p += kWarps)
                {
                    const uint32_t jn = code.check_order[p];
#pragma unroll
                    for (int j = 0; j < VEC; ++j)
                        if (((keep[j] >> lane) & 1u) && ((sg.synT[(size_t)p * VEC + j] >> lane) & 1u))
                            atomicOr(&args.syndrome_out[(size_t)fr[j] * code.words_m + (jn >> 5)], 1u << (jn & 31));
                }
            __syncthreads();
        }
    }

    // =============================================================================================================================
    // Frame-granular compaction. At a waterfall QBER most frames of a group converge early while a few run to max_it; their
    // columns would keep streaming. A repack (attempted at a few fixed rounds, decided on the device) moves the columns of the
    // live frames of ALL groups to the front -- new column k = rank of the frame among the live ones in (group, column)
    // order -- so that the passes touch ceil(live / G) groups from then on. Per-frame inputs and outputs are reached through
    // `fmap`. All moves are in place: a live column never moves to a later position, so for one message row set (one slot)
    // or one node's bit words, reading every source before writing any destination is enough.
    //   plan -> finalize(only_done) -> move_msg -> move_bits -> commit      (each returns at once when no repack was decided)
    // =============================================================================================================================
    template <int VEC>
    __global__ void __launch_bounds__(1024) stream_repack_plan_kernel(const SplitState st)
    {
        constexpr int G = 32 * VEC;
        __shared__ uint32_t s_cnt[kMaxRepackGroups + 1];
        __shared__ uint32_t s_live_groups;
        const int tid = threadIdx.x, ng = st.n_groups;
        if (tid == 0)
        {
            st.repack[0] = 0;
            s_live_groups = 0;
        }
        if (*st.n_live == 0 || ng > kMaxRepackGroups || ng < 2)
            return;
        __syncthreads();
        uint32_t cnt = 0;
        if (tid < ng)
        {
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                cnt += __popc(st.act[tid * 4 + j]);
            s_cnt[tid] = cnt;
            if (cnt)
                atomicAdd(&s_live_groups, 1u);
        }
        __syncthreads();
        if (tid == 0) // exclusive scan over <= 256 groups
        {
            uint32_t run = 0;
            for (int g = 0; g < ng; ++g)
            {
                const uint32_t c = s_cnt[g];
                s_cnt[g] = run;
                run += c;
            }
            s_cnt[ng] = run;
        }
        __syncthreads();
        const uint32_t live = s_cnt[ng], new_groups = (live + G - 1) / G;
        // worth it when enough of the streamed columns are dead (repack_pct) and at least one group disappears
        const bool go = live > 0 && 100ull * live <= (unsigned long long)st.repack_pct * s_live_groups * G && new_groups < s_live_groups;
        if (!go)
            return;
        if (tid < ng)
        {
            uint32_t k = s_cnt[tid];
            for (int c = 0; c < G; ++c)
                if ((st.act[tid * 4 + c % VEC] >> (c / VEC)) & 1u)
                {
                    st.src_of[k] = (uint32_t)tid * G + c;
                    st.fmap_new[k] = st.fmap[(size_t)tid * G + c];
                    ++k;
                }
        }
        for (uint32_t k = live + tid; k < (uint32_t)ng * G; k += blockDim.x)
        {
            st.src_of[k] = kNoFrame;
            st.fmap_new[k] = kNoFrame;
        }
        if (tid == 0)
        {
            st.repack[1] = live;
            st.repack[2] = new_groups;
            __threadfence();
            st.repack[0] = 1;
        }
    }

    // message columns: one CTA owns a slot at a time (all groups of the wave), staging <= kRepackStage values between the reads
    // and the writes
    constexpr int kRepackStage = 4096, kRepackThreads = 256;
    template <typename Real, int VEC>
    __global__ void __launch_bounds__(kRepackThreads) stream_repack_msg_kernel(const DecodeArgs args, const SplitState st)
    {
        constexpr int G = 32 * VEC;
        __shared__ Real s_val[kRepackStage];
        if (!st.repack[0])
            return;
        const uint32_t live = st.repack[1];
        const int B = st.bundle;
        const size_t rs = (size_t)B * G;
        const int slots = args.code.slots;
        auto at = [&](uint32_t slot, uint32_t col_id) -> Real *
        {
            const uint32_t g = col_id / G, c = col_id % G;
            return reinterpret_cast<Real *>(st.bundles + (size_t)(g / B) * st.bundle_stride) + ((size_t)slot * rs + (size_t)(g % B) * G + c);
        };
        for (uint32_t slot = blockIdx.x; slot < (uint32_t)slots; slot += gridDim.x)
            for (uint32_t k0 = 0; k0 < live; k0 += kRepackStage)
            {
                const uint32_t k1 = min(live, k0 + kRepackStage);
                for (uint32_t k = k0 + threadIdx.x; k < k1; k += kRepackThreads)
                {
                    QLB_CHECK_INDEX(st.src_of[k], (unsigned)st.n_groups * G);
                    QLB_CHECK_INDEX(k, st.src_of[k] + 1u); // in place: a live column never moves to a later position
                    s_val[k - k0] = *at(slot, st.src_of[k]);
                }
                __syncthreads();
                for (uint32_t k = k0 + threadIdx.x; k < k1; k += kRepackThreads)
                    *at(slot, k) = s_val[k - k0];
                __syncthreads();
            }
    }

    // bit-transposed words (Bob, Alice, decisions: per bit; syndromes: per check): one warp owns a node of one array at a time
    template <typename Real, int VEC>
    __global__ void __launch_bounds__(kRepackThreads) stream_repack_bits_kernel(const DecodeArgs args, const SplitState st)
    {
        constexpr int G = 32 * VEC;
        constexpr int kWarps = kRepackThreads / 32;
        __shared__ uint32_t s_old[kWarps][kMaxRepackGroups * VEC];
        if (!st.repack[0])
            return;
        const CodeDev &code = args.code;
        const int n = code.n, m = code.m, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, ng = st.n_groups;
        const uint32_t new_groups = st.repack[2];
        const SplitSmall cv = split_small_carve(n, m, VEC);
        const int B = st.bundle;
        const size_t small0 = align_up((size_t)code.slots * B * G * sizeof(Real), 256);
        const unsigned long long nodes = 3ull * n + m;
        for (unsigned long long q = (unsigned long long)blockIdx.x * kWarps + warp; q < nodes; q += (unsigned long long)gridDim.x * kWarps)
        {
            const int which = q < 3ull * n ? (int)(q / n) : 3;
            const size_t node = which < 3 ? (size_t)(q % n) : (size_t)(q - 3ull * n);
            const size_t off = (which == 0 ? cv.bobT : which == 1 ? cv.aliceT : which == 2 ? cv.zT : cv.synT) + node * VEC * 4;
            auto words_of = [&](uint32_t g) -> uint32_t *
            { return reinterpret_cast<uint32_t *>(st.bundles + (size_t)(g / B) * st.bundle_stride + small0 + (size_t)(g % B) * cv.total + off); };
            for (int x = lane; x < ng * VEC; x += 32)
                s_old[warp][x] = words_of((uint32_t)(x / VEC))[x % VEC];
            __syncwarp();
            for (uint32_t gn = 0; gn < new_groups; ++gn)
#pragma unroll
                for (int j = 0; j < VEC; ++j)
                {
                    const uint32_t old = st.src_of[(size_t)gn * G + VEC * lane + j];
                    uint32_t bit = 0;
                    if (old != kNoFrame)
                    {
                        const uint32_t c = old % G;
                        bit = (s_old[warp][(old / G) * VEC + c % VEC] >> (c / VEC)) & 1u;
                    }
                    const uint32_t word = __ballot_sync(0xffffffffu, bit);
                    if (lane == 0)
                        words_of(gn)[j] = word;
                }
            __syncwarp();
        }
    }

    template <int VEC>
    __global__ void __launch_bounds__(1024) stream_repack_commit_kernel(const SplitState st)
    {
        constexpr int G = 32 * VEC;
        if (!st.repack[0])
            return;
        const uint32_t live = st.repack[1], new_groups = st.repack[2];
        const int tid = threadIdx.x, ng = st.n_groups, B = st.bundle;
        for (uint32_t k = tid; k < (uint32_t)ng * G; k += blockDim.x)
            st.fmap[k] = st.fmap_new[k];
        for (int x = tid; x < ng * 4; x += blockDim.x)
        {
            const uint32_t g = x / 4, j = x % 4;
            uint32_t word = 0;
            if ((int)j < VEC)
                for (int l = 0; l < 32; ++l)
                    if (g * G + (uint32_t)(VEC * l) + j < live)
                        word |= 1u << l;
            st.act[x] = word;
            st.bad[x] = 0;
            st.succ[x] = 0;
        }
        const uint32_t new_bundles = (new_groups + B - 1) / B;
        for (uint32_t b = tid; b < new_bundles; b += blockDim.x)
            st.list[b] = b;
        if (tid == 0)
            *st.n_live = new_bundles;
    }
}
