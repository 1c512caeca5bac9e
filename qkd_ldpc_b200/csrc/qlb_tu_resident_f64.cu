#include "qlb_internal.hpp"
#include <algorithm>
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

    bool resident64_eligible_impl(const qlb_ctx *ctx, const CodeDev &c)
    {
        return c.slots < 65535 && c.n < 65536 && c.m < 65536 && c.bit_slots16 && c.col_of_slot16 && c.uniform_bit_w >= 2 && c.uniform_bit_w <= 4 &&
               c.max_check_w <= kResidentMaxCW && c.n % 32 == 0 && resident64_smem_slots(ctx, c) >= (uint32_t)c.slots / 2;
    }

    template <typename Math, bool kReconcile, int kBW>
    int launch_resident64(qlb_ctx *ctx, DecodeArgs &args)
    {
        auto kern = decode_resident_f64_kernel<Math, kReconcile, kBW, kResident64Threads>;
        const CodeDev &c = args.code;
        if (!c.r64_check_group_table || !c.r64_bit_group_table)
            return fail(QLB_ERR_UNSUPPORTED, "fp64 resident kernel: the code carries no group tables");
        int kThreads = kResident64Threads;
        if (const int t = args.block_threads / 32 * 32) // qlb_decode_params.block_threads
            if (t >= 32 && t <= kResident64Threads)
                kThreads = t;
        const size_t smem = (size_t)c.r64_smem_slots * 8 + resident64_small_bytes(c.n, c.m, c.r64_check_groups, c.r64_bit_groups);
        QLB_CUDA(allow_full_dynamic_smem(ctx, kern));
        long long grid = ctx->sm_count;
        if (grid > args.n_frames)
            grid = args.n_frames;
        const size_t tail = align_up((size_t)(c.slots - c.r64_smem_slots) * 8 + 16, 256);
        QLB_CUDA(ctx->scratch.reserve((size_t)grid * tail));
        args.scratch = static_cast<unsigned char *>(ctx->scratch.p);
        args.scratch_stride = tail;
#ifdef QLB_DEBUG_LAUNCH
        std::fprintf(stderr, "[qlb] decode_resident_f64_kernel: %d threads, %u of %d slots in shared memory (%zu B), %zu B tail scratch per CTA, grid=%lld, "
                             "%d check groups, %d bit groups\n", kThreads, c.r64_smem_slots, c.slots, smem, tail, grid, c.r64_check_groups, c.r64_bit_groups);
#endif
        QLB_CUDA(cudaMemsetAsync(ctx->d_counters, 0, sizeof(unsigned long long), ctx->stream));
        args.queue = ctx->d_counters;
        args.iter_total = ctx->d_counters + 1;
        std::snprintf(ctx->last_decoder, sizeof ctx->last_decoder, "resident_f64%s bw=%d threads=%d smem_slots=%u/%d",
                      std::is_same<Math, MathF64Fused>::value ? "fused" : "", kBW, kThreads, c.r64_smem_slots, c.slots);
        kern<<<(unsigned)grid, kThreads, smem, ctx->stream>>>(args);
        QLB_CUDA(cudaGetLastError());
        ++ctx->launches;
        return QLB_OK;
    }
    template <typename Math, bool kReconcile>
    int launch_resident64_bw(qlb_ctx *ctx, DecodeArgs &args)
    {
        switch (args.code.uniform_bit_w)
        {
#ifndef QLB_R64_LEAN // kernel-tuning builds (scripts/build_stream_variants.py) compile the bit weight of the benchmark code only
        case 2: return launch_resident64<Math, kReconcile, 2>(ctx, args);
        case 4: return launch_resident64<Math, kReconcile, 4>(ctx, args);
#endif
        case 3: return launch_resident64<Math, kReconcile, 3>(ctx, args);
        default: return fail(QLB_ERR_UNSUPPORTED, "fp64 resident kernel: unsupported bit weight");
        }
    }
}
namespace qlb
{
    bool resident_f64_eligible(const qlb_ctx *ctx, const CodeDev &c) { return resident64_eligible_impl(ctx, c) && c.r64_check_group_table; }

    // The group tables of the two walks (see qlb_resident_f64.cuh). `bit_slots`: [max_bit_w][n] physical slot of every edge of every bit.
    // Returns false (and leaves the outputs empty) when the kernel does not take the code on this device.
    bool resident64_build_tables(const qlb_ctx *ctx, const CodeDev &c, const uint32_t *bit_slots, std::vector<uint32_t> &check_groups,
                                 std::vector<uint16_t> &bit_groups, uint32_t &smem_slots)
    {
        check_groups.clear();
        bit_groups.clear();
        smem_slots = 0;
        if (!resident64_eligible_impl(ctx, c))
            return false;
        smem_slots = resident64_smem_slots(ctx, c);
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
        {
            check_groups.clear();
            return false;
        }
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

    int launch_resident_f64(qlb_ctx *ctx, DecodeArgs &args, bool reconcile, bool fused)
    {
        if (fused)
            return reconcile ? launch_resident64_bw<MathF64Fused, true>(ctx, args) : launch_resident64_bw<MathF64Fused, false>(ctx, args);
        return reconcile ? launch_resident64_bw<MathF64, true>(ctx, args) : launch_resident64_bw<MathF64, false>(ctx, args);
    }
}
