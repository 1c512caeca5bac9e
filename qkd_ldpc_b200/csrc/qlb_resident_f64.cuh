// fp64 SM-resident decoder: the reference's arithmetic and operation order (MathF64, qlb_kernels.cuh) with the frame's
// messages kept on the SM instead of in an L2-resident scratch.
//
// Storage. 30 720 doubles (240 KB) do not fit in the 227 KB of shared memory of one SM, so the message array is SPLIT: the
// first `smem_slots` physical slots (~92 % on the N=10240 code: all of edge positions 0..4 and the head of position 5) live
// in shared memory, the tail in a small per-CTA global scratch (L2-resident). Two properties of the code layout
// (qlb_layout.hpp) keep the split out of the hot loops:
//   * a run of sorted checks of one weight sees the split the same way for every check -- all rows in shared memory, or
//     exactly the last row in the tail -- so the check pass addresses its messages without a per-access test;
//   * inside a weight class the checks are ordered by the bit index of their last edge, so the tail slots belong to bits of
//     high index only: ~85 % of the 32-bit groups of the bit pass never leave shared memory and run a loop without any
//     shared / global predicate (`fast` groups); the others take the generic path.
//
// Schedule. Work is dealt to WARPS in groups of 32 consecutive nodes, round-robin over tables that list the slow groups (those
// that reach into the global tail) first, so that every warp gets the same mix and whole groups only: the two block barriers
// of an iteration wait for one group at most (the thread-strided walk of the first version left 16 % of the time in them,
// ncu). Drawing the groups from a shared-memory counter was tried and dropped: the atomic's latency and the shorter prefetch
// distance for the slot indices cost more than the balance returns. The tables (built once per code and device by
// resident64_build_tables) sit in shared memory.
//
// Convergence (calculate_syndrome + arrays_equal after every bit pass, src/qkd_ldpc_algorithm.cpp:277-298) is tracked
// INCREMENTALLY, in integers, exactly: s_unsat holds one bit per check, syndrome(z) ^ target. It is initialised once per
// frame from the bit side -- every bit with Alice's bit != the prior's hard decision toggles the bits of its checks, as it
// writes its prior into its message slots -- and from then on a bit whose decision flips in a bit pass does the same. The frame has converged when the words are all zero -- known right
// after the bit pass, so a converged frame pays no speculative check pass, and the check pass itself carries nothing but
// the check rule (bit-exact fp64 messages leave no spare mantissa bit to carry the decision as the fp32 kernel does).
// Iteration counts, flags and keys follow the reference's definitions exactly (src/qkd_ldpc_algorithm.cpp:175-345,
// 398-447); the generic decode_kernel<MathF64> stays as the fallback for codes this kernel does not take.
#pragma once
#include "qlb_resident_f32.cuh"

namespace qlb
{
#ifndef QLB_R64_THREADS
#define QLB_R64_THREADS 768
#endif
    constexpr int kResident64Threads = QLB_R64_THREADS; // launch bound (768: 80 registers)
    constexpr int kResident64FastW = 8;     // weights up to this get the split-specialised loops
    constexpr size_t kResident64StaticSmem = 768; // s_base, s_frame, the exp table s_exp_tab (512 B), and the system's reserve

    // A group of the check walk: sorted positions p0 + l0 .. p0 + l1 (p0 a multiple of 32), all of weight w, the split falling
    // the same way for each: `tail` rows (edge positions w - tail .. w - 1) in the global tail (0 or 1), or 3: decide per access.
    //   bits 0..10  p0 / 32     bits 11..15  l0     bits 16..20  l1     bits 21..27  type = w * 4 + tail
    __host__ __device__ inline uint32_t r64_pack_group(uint32_t p0, int l0, int l1, int w, int tail)
    {
        return (p0 >> 5) | ((uint32_t)l0 << 11) | ((uint32_t)l1 << 16) | ((uint32_t)(w * 4 + tail) << 21);
    }
    // A group of the bit walk: bits 32 g .. 32 g + 31; bit 15 set: every slot of the group lies in shared memory.
    constexpr uint16_t kR64BitGroupFast = 0x8000;

    struct Split64
    {
        double *smem;
        double *gmem; // slot s >= smem_slots is gmem[s - smem_slots]
        uint32_t smem_slots;
        uint32_t slots; // read by bounds-check builds only
        __device__ __forceinline__ double ld(uint32_t slot) const
        {
            QLB_CHECK_INDEX(slot, slots);
            return slot < smem_slots ? smem[slot] : gmem[slot - smem_slots];
        }
        __device__ __forceinline__ void st(uint32_t slot, double v) const
        {
            QLB_CHECK_INDEX(slot, slots);
            if (slot < smem_slots)
                smem[slot] = v;
            else
                gmem[slot - smem_slots] = v;
        }
    };

    // shared memory beside the messages: Bob, decisions | target syndrome, unsatisfied checks (both in sorted check order) | tables
    __host__ __device__ inline size_t resident64_small_bytes(int n, int m, int check_groups, int bit_groups)
    {
        const size_t wn = align_up((size_t)(n + 31) / 32 * 4, 16), wm = align_up((size_t)(m + 31) / 32 * 4, 16);
        return 2 * wn + 2 * wm + align_up((size_t)check_groups * 4, 16) + align_up((size_t)bit_groups * 2, 16);
    }

    // The clamp of :313-316 (threshold_matrix: x > thr -> thr, x < -thr -> -thr, NaN untouched) with ONE FP64 compare; thr_eff is
    // +inf when the clamp is disabled.
    __device__ __forceinline__ double clamp_f64(double x, double thr_eff)
    {
        return fabs(x) > thr_eff ? copysign(thr_eff, x) : x;
    }

    struct Base64FromParams // constant-bank operands
    {
        const DecodeArgs &args;
        __device__ __forceinline__ uint32_t operator()(int k) const { return args.code.base[k]; }
    };
    struct Base64FromSmem
    {
        const uint32_t *base;
        __device__ __forceinline__ uint32_t operator()(int k) const { return base[k]; }
    };

    // The check rule (:220-249) on the checks p0 + lane of one group.
    template <typename Math, bool kWantInf, int W, int kTail, typename Base>
    __device__ __forceinline__ void check_group64(const Split64 &msg, const Base s_base, uint32_t p, bool active, bool syn, double thr_eff,
                                                  const double2 *s_exp_tab)
    {
        if (!active)
            return;
        double *gm = msg.gmem - msg.smem_slots;
        double v[W];
#pragma unroll
        for (int k = 0; k < W; ++k)
        {
            const uint32_t slot = s_base(k) + p;
            QLB_CHECK_INDEX(slot, msg.slots);
            if (kTail != 3 && k < W - kTail)
                QLB_CHECK_INDEX(slot, msg.smem_slots); // a row the group table promises to shared memory ...
            if (kTail != 3 && k >= W - kTail)
                QLB_CHECK_INDEX(msg.smem_slots, slot + 1u); // ... and one it promises to the global tail
            v[k] = kTail == 3 ? msg.ld(slot) : (k < W - kTail ? msg.smem[slot] : gm[slot]);
        }
        Math::template check_fast<W, kWantInf>(v, syn, thr_eff, s_exp_tab);
#pragma unroll
        for (int k = 0; k < W; ++k)
        {
            const uint32_t slot = s_base(k) + p;
            if (kTail == 3)
                msg.st(slot, v[k]);
            else if (k < W - kTail)
                msg.smem[slot] = v[k];
            else
                gm[slot] = v[k];
        }
    }
    // Weights 9..16 (the R >= 0.7 codes of the CW = 3 family) are kept out of line: their register appetite (2 x W doubles live) must
    // not leak into the hot instantiations; some spilling inside them is still far cheaper than the generic kernel's L2 round trips.
    template <typename Math, bool kWantInf, int W>
    __device__ __noinline__ void check_group64_wide(const Split64 msg, const uint32_t *s_base, uint32_t p, bool active, bool syn, double thr_eff,
                                                    const double2 *s_exp_tab)
    {
        check_group64<Math, kWantInf, W, 3>(msg, Base64FromSmem{s_base}, p, active, syn, thr_eff, s_exp_tab);
    }

    // Sorted position of the check that owns `slot` (rows are laid out one edge position after the other, qlb_layout.hpp).
    __device__ __forceinline__ uint32_t check_of_slot64(uint32_t slot, const uint32_t *s_base, int max_cw)
    {
        uint32_t b = 0;
        for (int k = 1; k < max_cw; ++k)
            b = slot >= s_base[k] ? s_base[k] : b;
        return slot - b;
    }

    __device__ __forceinline__ void toggle_bit(uint32_t *words, uint32_t p)
    {
        asm volatile("red.shared.xor.b32 [%0], %1;" ::"r"(smem_u32(words + (p >> 5))), "r"(1u << (p & 31)) : "memory");
    }

    // kBW: uniform bit weight. Host-checked: slots < 65535, n < 65536, m < 65536, max_check_w <= 16, n % 32 == 0.
    // kWantInf: the clamp is off or above 700, so a saturated check product must give the IEEE infinity (MathF64::check_fast).
    template <typename Math, bool kReconcile, int kBW, int kMaxThreads, bool kWantInf>
    __global__ void __launch_bounds__(kMaxThreads, 1) decode_resident_f64_kernel(const DecodeArgs args)
    {
        const int kThreads = blockDim.x; // multiple of 32, <= kMaxThreads
        extern __shared__ __align__(16) unsigned char smem[];
        __shared__ uint32_t s_base[kResidentMaxCW];
        __shared__ long long s_frame;
        __shared__ double2 s_exp_tab[32];

        const CodeDev &code = args.code;
        const int n = code.n, m = code.m, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, warps = kThreads >> 5;
        const int words_n = code.words_n, words_m = code.words_m;
        const size_t wn = align_up((size_t)words_n * 4, 16), wm = align_up((size_t)words_m * 4, 16);
        const int n_cg = code.r64_check_groups, n_bg = code.r64_bit_groups;
        const uint32_t smem_slots = code.r64_smem_slots;
        (void)m;

        Split64 msg;
        msg.smem = reinterpret_cast<double *>(smem);
        msg.smem_slots = smem_slots;
        msg.slots = (uint32_t)code.slots;
        msg.gmem = reinterpret_cast<double *>(args.scratch + (size_t)blockIdx.x * args.scratch_stride);
        unsigned char *tail = smem + (size_t)smem_slots * 8;
        uint32_t *s_bob = reinterpret_cast<uint32_t *>(tail);
        uint32_t *s_z = reinterpret_cast<uint32_t *>(tail + wn);
        uint32_t *s_syn = reinterpret_cast<uint32_t *>(tail + 2 * wn);         // target syndrome, sorted check order
        uint32_t *s_unsat = reinterpret_cast<uint32_t *>(tail + 2 * wn + wm);  // syndrome(z) ^ target, sorted check order
        uint32_t *s_cg = reinterpret_cast<uint32_t *>(tail + 2 * wn + 2 * wm);
        uint16_t *s_bg = reinterpret_cast<uint16_t *>(tail + 2 * wn + 2 * wm + align_up((size_t)n_cg * 4, 16));

        if (tid < kResidentMaxCW)
            s_base[tid] = code.base[tid];
        if (tid < 32)
            s_exp_tab[tid] = f64m::kExpTab[tid];
        for (int g = tid; g < n_cg; g += kThreads)
            s_cg[g] = code.r64_check_group_table[g];
        for (int g = tid; g < n_bg; g += kThreads)
            s_bg[g] = code.r64_bit_group_table[g];
        const uint16_t *bslot = code.bit_slots16;
        const double kInf = __longlong_as_double(0x7ff0000000000000LL);
        const double thr_eff = args.enable_thr ? args.thr : kInf; // the clamp as an operand: nothing exceeds +inf

        for (;;)
        {
            __syncthreads();
            if (tid == 0)
                s_frame = (long long)atomicAdd(args.queue, 1ULL);
            __syncthreads();
            const long long f = s_frame;
            if (f >= args.n_frames)
                break;

            // ---- A: Bob's key / the target syndrome into shared memory -----------------------------------------------------
            double lp = 0.;
            const double *llr_f = nullptr;
            if (kReconcile)
            {
                lp = args.log_prior[f];
                for (int w = tid; w < words_n; w += kThreads)
                    s_bob[w] = args.bob[f * words_n + w];
                for (int w = tid; w < words_m; w += kThreads)
                    s_syn[w] = s_unsat[w] = 0;
            }
            else
            {
                llr_f = args.llr + f * n;
                // target syndrome (natural check order in the API) -> sorted order; s_unsat starts as the target and is toggled by z0 below
                for (int g = warp; g < words_m; g += warps)
                {
                    const int p = g * 32 + lane;
                    uint32_t sb = 0;
                    if (p < m)
                    {
                        const uint32_t j = code.check_order[p];
                        sb = (args.syndrome_in[f * words_m + (j >> 5)] >> (j & 31)) & 1u;
                    }
                    const uint32_t word = __ballot_sync(0xffffffffu, sb);
                    if (lane == 0)
                        s_syn[g] = s_unsat[g] = word;
                }
            }
            __syncthreads();
            // ---- B: messages <- priors, unclamped (:182-190); z0 = the priors' own hard decision; the target syndrome (reconcile
            // mode: Alice's syndrome, :413-414) and s_unsat = syndrome(z0) ^ target from the BIT side: a bit toggles the bits of its
            // checks (a few thousand shared-memory reductions, no dependent walk over the checks' edge lists) -------------------------
            {
                // the Alice words of this warp's groups (group warp + l * warps in lane l), fetched in one go
                uint32_t my_alice = 0;
                int r = 0;
                for (int g = warp; g < words_n; g += warps, ++r) // n % 32 == 0: whole warps only
                {
                    if (kReconcile && (r & 31) == 0)
                        my_alice = warp + (r + lane) * warps < words_n ? args.alice[f * words_n + warp + (r + lane) * warps] : 0u;
                    const int i = g * 32 + lane;
                    uint32_t sl[kBW];
#pragma unroll
                    for (int a = 0; a < kBW; ++a)
                        sl[a] = bslot[a * n + i];
                    double prior;
                    if (kReconcile)
                        prior = __hiloint2double(__double2hiint(lp) ^ (int)(((s_bob[g] >> lane) & 1u) << 31), __double2loint(lp)); // :401-405
                    else
                        prior = llr_f[i];
                    const bool z0 = prior <= 0.;
                    const uint32_t word = __ballot_sync(0xffffffffu, z0);
                    if (lane == 0)
                        s_z[g] = word;
                    const bool ab = kReconcile && ((__shfl_sync(0xffffffffu, my_alice, r & 31) >> lane) & 1u);
#pragma unroll
                    for (int a = 0; a < kBW; ++a)
                    {
                        msg.st(sl[a], prior);
                        if (ab || z0)
                        {
                            const uint32_t p = check_of_slot64(sl[a], s_base, code.max_check_w);
                            if (ab)
                                toggle_bit(s_syn, p);
                            if (ab != z0)
                                toggle_bit(s_unsat, p);
                        }
                    }
                }
            }
            __syncthreads();
            if (kReconcile && args.syndrome_out) // Alice's syndrome in natural check order
            {
                for (int w = tid; w < words_m; w += kThreads)
                    args.syndrome_out[f * words_m + w] = 0;
                __syncthreads();
                for (int p = tid; p < m; p += kThreads)
                    if ((s_syn[p >> 5] >> (p & 31)) & 1u)
                    {
                        const uint32_t j = code.check_order[p];
                        atomicOr(&args.syndrome_out[f * words_m + (j >> 5)], 1u << (j & 31));
                    }
            }

            int it = 0; // completed bit passes
            bool success = false;
            while (it < args.max_it)
            {
                // ---- check pass (:220-249) -----------------------------------------------------------------------------------
                {
#pragma unroll 1
                    for (int g = warp; g < n_cg; g += warps)
                    {
                        const uint32_t ent = s_cg[g];
                        const uint32_t p = ((ent & 0x7ffu) << 5) + lane;
                        const bool active = lane >= (int)((ent >> 11) & 31u) && lane <= (int)((ent >> 16) & 31u);
                        const bool syn = ((s_syn[ent & 0x7ffu] >> lane) & 1u) != 0;
                        switch (ent >> 21)
                        {
#define QLB_GRP64(W_)                                                                                                       \
    case W_ * 4 + 0: check_group64<Math, kWantInf, W_, 0>(msg, Base64FromParams{args}, p, active, syn, thr_eff, s_exp_tab); break; \
    case W_ * 4 + 1: check_group64<Math, kWantInf, W_, 1>(msg, Base64FromParams{args}, p, active, syn, thr_eff, s_exp_tab); break; \
    case W_ * 4 + 3: check_group64<Math, kWantInf, W_, 3>(msg, Base64FromParams{args}, p, active, syn, thr_eff, s_exp_tab); break;
#define QLB_GRP64W(W_) \
    case W_ * 4 + 3: check_group64_wide<Math, kWantInf, W_>(msg, s_base, p, active, syn, thr_eff, s_exp_tab); break;
                            QLB_GRP64(1) QLB_GRP64(2) QLB_GRP64(3) QLB_GRP64(4) QLB_GRP64(5) QLB_GRP64(6) QLB_GRP64(7) QLB_GRP64(8)
                            QLB_GRP64W(9) QLB_GRP64W(10) QLB_GRP64W(11) QLB_GRP64W(12) QLB_GRP64W(13) QLB_GRP64W(14) QLB_GRP64W(15) QLB_GRP64W(16)
#undef QLB_GRP64
#undef QLB_GRP64W
                        default: // checks without edges send nothing
                            break;
                        }
                    }
                }
                __syncthreads();
                // ---- bit pass: total (:256-258), decision (:259-266), extrinsic + clamp (:300-316); a flipped decision toggles
                // the unsatisfied-bits of the bit's checks ------------------------------------------------------------------
                {
                    // this warp's groups: entries warp, warp + warps, ... of the table (slow groups first, so every warp gets its
                    // share of them); the slot indices (L2) of the group after next travel while a group is processed
                    uint32_t ent = warp < n_bg ? s_bg[warp] : 0u, ent1 = warp + warps < n_bg ? s_bg[warp + warps] : 0u;
                    uint32_t sl[kBW], sl1[kBW];
#pragma unroll
                    for (int a = 0; a < kBW; ++a)
                    {
                        sl[a] = bslot[a * n + (int)(ent & 0x7fffu) * 32 + lane];
                        sl1[a] = bslot[a * n + (int)(ent1 & 0x7fffu) * 32 + lane];
                    }
#pragma unroll 1
                    for (int g = warp; g < n_bg; g += warps)
                    {
                        const uint32_t ent2 = g + 2 * warps < n_bg ? s_bg[g + 2 * warps] : 0u;
                        uint32_t sl2[kBW];
#pragma unroll
                        for (int a = 0; a < kBW; ++a)
                            sl2[a] = bslot[a * n + (int)(ent2 & 0x7fffu) * 32 + lane];
                        const int grp = (int)(ent & 0x7fffu);
                        double prior;
                        if (kReconcile)
                            prior = __hiloint2double(__double2hiint(lp) ^ (int)(((s_bob[grp] >> lane) & 1u) << 31), __double2loint(lp));
                        else
                            prior = llr_f[grp * 32 + lane];
                        double c[kBW];
                        bool z;
                        if (ent & kR64BitGroupFast)
                        {
#pragma unroll
                            for (int a = 0; a < kBW; ++a)
                            {
                                QLB_CHECK_INDEX(sl[a], msg.smem_slots); // a `fast` group never leaves shared memory
                                c[a] = msg.smem[sl[a]];
                            }
                            double total = prior;
#pragma unroll
                            for (int a = 0; a < kBW; ++a)
                                total = total + c[a];
                            z = total <= 0.;
#pragma unroll
                            for (int a = 0; a < kBW; ++a)
                                msg.smem[sl[a]] = clamp_f64(total - c[a], thr_eff);
                        }
                        else
                        {
#pragma unroll
                            for (int a = 0; a < kBW; ++a)
                                c[a] = msg.ld(sl[a]);
                            double total = prior;
#pragma unroll
                            for (int a = 0; a < kBW; ++a)
                                total = total + c[a];
                            z = total <= 0.;
#pragma unroll
                            for (int a = 0; a < kBW; ++a)
                                msg.st(sl[a], clamp_f64(total - c[a], thr_eff));
                        }
                        const uint32_t word = __ballot_sync(0xffffffffu, z);
                        const uint32_t flips = word ^ s_z[grp];
                        if (flips) // warp-uniform
                        {
                            if ((flips >> lane) & 1u)
                            {
#pragma unroll 1
                                for (int a = 0; a < kBW; ++a)
                                    toggle_bit(s_unsat, check_of_slot64(sl[a], s_base, code.max_check_w));
                            }
                            __syncwarp();
                            if (lane == 0)
                                s_z[grp] = word;
                        }
                        ent = ent1;
                        ent1 = ent2;
#pragma unroll
                        for (int a = 0; a < kBW; ++a)
                        {
                            sl[a] = sl1[a];
                            sl1[a] = sl2[a];
                        }
                    }
                }
                ++it;
                __syncthreads();
                // calculate_syndrome + arrays_equal of :277-298: all checks satisfied?
                int open = 0;
                for (int w = tid; w < words_m; w += kThreads)
                    open |= s_unsat[w] != 0u;
                if (!__syncthreads_or(open))
                {
                    success = true; // :285-298
                    break;
                }
            }

            int differs = 0;
            for (int w = tid; w < words_n; w += kThreads)
            {
                const uint32_t zw = s_z[w];
                if (args.decoded)
                    args.decoded[f * words_n + w] = zw;
                if (kReconcile)
                    differs |= (zw != args.alice[f * words_n + w]);
            }
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
}
