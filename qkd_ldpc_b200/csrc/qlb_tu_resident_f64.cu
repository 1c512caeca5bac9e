#include "qlb_internal.hpp"
using namespace qlb;
#include "qlb_resident_f64.cuh"

namespace
{
    // Upper bound of the check walk's group count: one group per started 32 positions, plus one per cut (weight classes, split sides).
    int check_group_cap(const CodeDev &c) { return (c.m + 31) / 32 + 3 * c.max_check_w + 4; }

    // Message slots kept in shared memory: what is left beside the small arrays and the group tables, a multiple of 32 (rows start
    // on multiples of 32, so the split then falls on a 32-aligned sorted position in every row).
    uint32_t resident64_smem_slots(const qlb_ctx *ctx, const CodeDev &c)
    {
        const size_t fixed = kResident64StaticSmem + resident64_small_bytes(c.n, c.m, check_group_cap(c), (c.n + 31) / 32);
        if ((size_t)ctx->smem_optin <= fixed + 8192)
            return 0;
        const size_t fit = ((size_t)ctx->smem_optin - fixed) / 8 / 32 * 32;
        return (uint32_t)std::min<size_t>(fit, (size_t)c.slots);
    }

    template <typename Math, bool kReconcile, int kBW>
    int launch_resident64(qlb_ctx *ctx, DecodeArgs &args, int block_threads)
    {
        // the infinity of a saturated product is only materialised where the clamp cannot hide it (MathF64::check_fast); the fused
        // rule produces it either way and has the one instantiation
        const double thr_eff = args.enable_thr ? args.thr : __builtin_huge_val();
        auto kern = decode_resident_f64_kernel<Math, kReconcile, kBW, kResident64Threads, false>;
        if constexpr (std::is_same<Math, MathF64>::value)
            if (!(thr_eff <= 700.))
                kern = decode_resident_f64_kernel<Math, kReconcile, kBW, kResident64Threads, true>;
        const CodeDev &c = args.code;
        int kThreads = kResident64Threads;
        if (const int t = block_threads / 32 * 32) // qlb_decode_params.block_threads
            if (t >= 32 && t <= kResident64Threads)
                kThreads = t;
        const size_t smem = (size_t)c.r64_smem_slots * 8 + resident64_small_bytes(c.n, c.m, c.r64_check_groups, c.r64_bit_groups);
        const size_t tail = align_up((size_t)(c.slots - c.r64_smem_slots) * 8 + 16, 256); // the slots beyond r64_smem_slots
        char name[sizeof(qlb_ctx::last_decoder)];
        std::snprintf(name, sizeof name, "resident_f64%s bw=%d threads=%d smem_slots=%u/%d",
                      std::is_same<Math, MathF64Fused>::value ? "fused" : "", kBW, kThreads, c.r64_smem_slots, c.slots);
        return launch_persistent(ctx, args, kern, kThreads, smem, 1, tail, name); // one resident CTA per SM
    }
}
namespace qlb
{
    // The group tables of the two walks (see qlb_resident_f64.cuh). `bit_slots`: [max_bit_w][n] physical slot of every edge of every bit.
    // Returns false (outputs unspecified) when the kernel does not take the code on this device: the kernel's admission test.
    bool resident64_build_tables(const qlb_ctx *ctx, const CodeDev &c, const uint32_t *bit_slots, std::vector<uint32_t> &check_groups,
                                 std::vector<uint16_t> &bit_groups, uint32_t &smem_slots)
    {
        smem_slots = resident64_smem_slots(ctx, c);
        if (!(c.slots < 65535 && c.n < 65536 && c.m < 65536 && c.bit_slots16 && c.col_of_slot16 && c.uniform_bit_w >= 2 && c.uniform_bit_w <= 4 &&
              c.max_check_w <= kResidentMaxCW && c.n % 32 == 0 && smem_slots >= (uint32_t)c.slots / 2))
            return false;
        std::vector<uint32_t> slow, fast;
        auto push_run = [&](uint32_t lo, uint32_t hi, int w, int tail)
        {
            for (uint32_t p0 = lo / 32 * 32; p0 < hi; p0 += 32)
            {
                const int l0 = (int)(std::max(lo, p0) - p0), l1 = (int)(std::min(hi, p0 + 32) - p0) - 1;
                (tail == 0 ? fast : slow).push_back(r64_pack_group(p0, l0, l1, w, tail));
            }
        };
        for (int w = c.max_check_w; w >= 1; --w)
        {
            const uint32_t lo = (w < c.max_check_w) ? c.cnt[w] : 0u, hi = c.cnt[w - 1];
            if (lo >= hi)
                continue;
            if (w > kResident64FastW)
            {
                push_run(lo, hi, w, 3);
                continue;
            }
            // positions below split(k) keep row k in shared memory; rows are laid out in increasing k, so split(k) decreases with k
            auto split = [&](int k) -> uint32_t
            {
                const long long s = (long long)smem_slots - (long long)c.base[k];
                return (uint32_t)std::min<long long>(hi, std::max<long long>(lo, s));
            };
            const uint32_t s1 = split(w - 1), s2 = w >= 2 ? split(w - 2) : hi; // [lo, s1): all rows shared; [s1, s2): the last row in the tail
            push_run(lo, s1, w, 0);
            push_run(s1, s2, w, 1);
            push_run(s2, hi, w, 3);
        }
        // the groups that reach into the global tail first: their latency is then covered by the others
        check_groups = slow;
        check_groups.insert(check_groups.end(), fast.begin(), fast.end());
        if ((int)check_groups.size() > check_group_cap(c))
            return false;
        std::vector<uint16_t> bslow, bfast;
        for (int g = 0; g < c.n / 32; ++g)
        {
            bool all_smem = true;
            for (int a = 0; a < c.max_bit_w && all_smem; ++a)
                for (int l = 0; l < 32; ++l)
                    if (bit_slots[(size_t)a * c.n + g * 32 + l] >= smem_slots)
                    {
                        all_smem = false;
                        break;
                    }
            (all_smem ? bfast : bslow).push_back((uint16_t)(g | (all_smem ? kR64BitGroupFast : 0)));
        }
        bit_groups = bslow;
        bit_groups.insert(bit_groups.end(), bfast.begin(), bfast.end());
        return true;
    }

    int launch_resident_f64(qlb_ctx *ctx, DecodeArgs &args, const Route &r)
    {
        return with_rule<Rule::F64, Rule::F64Fused>(r, [&](auto rule, auto reconcile) -> int
        {
            typedef MathOf<decltype(rule)::value> Math;
            constexpr bool kReconcile = decltype(reconcile)::value;
            switch (args.code.uniform_bit_w)
            {
#ifndef QLB_R64_LEAN // kernel-tuning builds (scripts/build_stream_variants.py) compile the bit weight of the benchmark code only
            case 2: return launch_resident64<Math, kReconcile, 2>(ctx, args, r.block_threads);
            case 4: return launch_resident64<Math, kReconcile, 4>(ctx, args, r.block_threads);
#endif
            case 3: return launch_resident64<Math, kReconcile, 3>(ctx, args, r.block_threads);
            default: return fail(QLB_ERR_UNSUPPORTED, "fp64 resident kernel: unsupported bit weight");
            }
        });
    }
}
