// Rate-adaptive reconciliation (qlb_rate_pattern, qlb_reconcile_adapted_packed, qlb_run_trials_adapted; defined in the header).
// A rate-adapted batch is turned on the device into the LLR-and-syndrome form of qlb_sum_product_batch, decoded by launch_decode
// in that mode -- the same decoders, rules and routing as every other decode -- and the decoded bits at the key positions are
// then compared with Alice's key on the device. The kernels here only move bits: embed, fill, and key extraction.
#include "qlb_internal.hpp"
#include "qlb_generate.cuh"
#include "qlb_layout.hpp"

#include <cmath>
#include <cstring>
#include <numeric>
#include <string>
#include <vector>

using namespace qlb;

namespace qlb
{
    // Position table entry: class in bits 30..31 (QLB_POS_*), key or fill index in bits 0..29.
    constexpr uint32_t kRateIndexMask = (1u << 30) - 1;

    // One warp per 32 positions of one frame: the LLR row (double[N]) and Alice's packed mother word.
    __global__ void __launch_bounds__(256) rate_embed_kernel(long long n_frames, int n_bits, int words_n, int words_key, int words_fill,
                                                             const uint32_t *__restrict__ pos_tab, const uint32_t *__restrict__ alice,
                                                             const uint32_t *__restrict__ bob, const uint32_t *__restrict__ fill,
                                                             const double *__restrict__ log_prior, double thr, double *__restrict__ llr_out,
                                                             uint32_t *__restrict__ word_out)
    {
        const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
        const int lane = threadIdx.x & 31;
        if (warp >= n_frames * words_n)
            return;
        const long long f = warp / words_n;
        const int w = (int)(warp - f * words_n), i = w * 32 + lane;
        uint32_t a = 0;
        if (i < n_bits)
        {
            const uint32_t t = pos_tab[i], k = t & kRateIndexMask, cls = t >> 30;
            double l;
            if (cls == QLB_POS_KEY)
            {
                a = (alice[f * words_key + (k >> 5)] >> (k & 31)) & 1u;
                const double lp = log_prior[f];
                l = (bob[f * words_key + (k >> 5)] >> (k & 31)) & 1u ? -lp : lp;
            }
            else
            {
                a = (fill[f * words_fill + (k >> 5)] >> (k & 31)) & 1u;
                l = cls == QLB_POS_PUNCTURED ? 0.0 : (a ? -thr : thr);
            }
            llr_out[f * n_bits + i] = l;
        }
        const uint32_t word = __ballot_sync(0xFFFFFFFFu, a);
        if (lane == 0)
            word_out[f * words_n + w] = word;
    }

    // One CTA per frame: the decoded bits at the key positions, packed; QLB_RES_KEYS_MATCH when they equal Alice's key.
    __global__ void __launch_bounds__(256) rate_extract_kernel(int n_key, int words_n, int words_key, const uint32_t *__restrict__ key_pos,
                                                               const uint32_t *__restrict__ decoded, const uint32_t *__restrict__ alice,
                                                               uint8_t *__restrict__ result, uint32_t *__restrict__ key_out)
    {
        const long long f = blockIdx.x;
        const int lane = threadIdx.x & 31;
        const uint32_t *dec = decoded + f * words_n;
        int mismatch = 0;
        for (int w = threadIdx.x >> 5; w < words_key; w += blockDim.x >> 5)
        {
            const int k = w * 32 + lane;
            uint32_t b = 0;
            if (k < n_key)
            {
                const uint32_t i = key_pos[k];
                b = (dec[i >> 5] >> (i & 31)) & 1u;
            }
            const uint32_t word = __ballot_sync(0xFFFFFFFFu, b);
            const uint32_t valid = n_key - w * 32 >= 32 ? 0xFFFFFFFFu : (1u << (n_key - w * 32)) - 1u;
            if (lane == 0)
            {
                mismatch |= ((word ^ alice[f * words_key + w]) & valid) != 0;
                if (key_out)
                    key_out[f * words_key + w] = word;
            }
        }
        if (__syncthreads_or(mismatch) == 0 && threadIdx.x == 0)
            result[f] |= QLB_RES_KEYS_MATCH;
    }

    // One thread per frame: fill bit k = top bit of the k-th output of Xoshiro256PlusPlus(~(seeds[f] + seed_offset)).
    __global__ void __launch_bounds__(128) rate_fill_kernel(long long n_frames, int n_fill, int words_fill, const uint64_t *__restrict__ seeds,
                                                            uint64_t seed_offset, uint32_t *__restrict__ fill_out)
    {
        const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
        if (f >= n_frames)
            return;
        Xoshiro256pp rng(~(seeds[f] + seed_offset));
        for (int w = 0; w < words_fill; ++w)
        {
            uint32_t word = 0;
            const int lim = min(32, n_fill - w * 32);
            for (int b = 0; b < lim; ++b)
                word |= (uint32_t)(rng.next() >> 63) << b;
            fill_out[f * words_fill + w] = word;
        }
    }
}

namespace
{
    struct RatePattern
    {
        int32_t n_key = 0, n_punct = 0, n_short = 0;
        std::vector<uint32_t> tab; // [N] pos_tab entries, then [n_key] key positions
        int words_key() const { return (n_key + 31) / 32; }
        int words_fill() const { return (n_punct + n_short + 31) / 32; }
    };

    // Scans the class array into the device tables and checks the pattern against the decode parameters.
    int scan_pattern(const CodeLayout &L, const qlb_decode_params &p, const uint8_t *pos_class, RatePattern &out)
    {
        if (!pos_class)
            return fail(QLB_ERR_INVALID, "rate adaptation: pos_class is null");
        out.tab.assign((size_t)L.n, 0);
        std::vector<uint32_t> key_pos;
        uint32_t n_fill = 0;
        for (int32_t i = 0; i < L.n; ++i)
        {
            const uint8_t c = pos_class[i];
            if (c == QLB_POS_KEY)
            {
                out.tab[i] = (uint32_t)key_pos.size();
                key_pos.push_back((uint32_t)i);
            }
            else if (c == QLB_POS_PUNCTURED || c == QLB_POS_SHORTENED)
            {
                out.tab[i] = (uint32_t)c << 30 | n_fill++;
                ++(c == QLB_POS_PUNCTURED ? out.n_punct : out.n_short);
            }
            else
                return fail(QLB_ERR_INVALID, "rate adaptation: pos_class[" + std::to_string(i) + "] = " + std::to_string(c) +
                                                 " is not QLB_POS_KEY, QLB_POS_PUNCTURED or QLB_POS_SHORTENED");
        }
        out.n_key = (int32_t)key_pos.size();
        if (out.n_key == 0)
            return fail(QLB_ERR_INVALID, "rate adaptation: pos_class has no key position");
        out.tab.insert(out.tab.end(), key_pos.begin(), key_pos.end());
        if (out.n_short > 0 && !p.enable_threshold)
            return fail(QLB_ERR_INVALID, "rate adaptation: shortened positions take the prior +-threshold and need enable_threshold");
        if (out.n_punct > 0)
        {
            if (p.precision == QLB_PRECISION_F64)
                return fail(QLB_ERR_UNSUPPORTED, std::string("rate adaptation: punctured positions need a check rule defined at a zero message; ") +
                                                     (p.flags & QLB_FLAG_F64_FUSED_RATIO ? "fp64 fused" : "fp64") +
                                                     " divides by the edge's own tanh(m/2) and gives 0/0 there (use fp32 or fp32 min-sum)");
            if (p.flags & QLB_FLAG_F32_FAST_MATH)
                return fail(QLB_ERR_UNSUPPORTED, "rate adaptation: punctured positions need a check rule defined at a zero message; "
                                                 "fp32 fast math gives (S-D)/(D-S) = 0/0 there (use fp32 or fp32 min-sum)");
        }
        return QLB_OK;
    }

    // Embed, syndrome, decode (sum-product mode), key extraction: on the context's stream, device buffers, no synchronisation.
    int decode_adapted(qlb_ctx *ctx, const CodeDev &dev, const qlb_decode_params &p, const RatePattern &pat, int64_t n_frames,
                       const uint32_t *d_alice, const uint32_t *d_bob, const uint32_t *d_fill, const double *d_log_prior,
                       uint32_t *d_iterations, uint8_t *d_result, uint32_t *d_key_out)
    {
        const size_t F = (size_t)n_frames, tab_bytes = pat.tab.size() * 4;
        QLB_CUDA(ctx->rate_tab.reserve(tab_bytes));
        QLB_CUDA(ctx->in_llr.reserve(F * dev.n * 8));
        QLB_CUDA(ctx->rate_word.reserve(F * dev.words_n * 4));
        QLB_CUDA(ctx->in_syn.reserve(F * dev.words_m * 4));
        QLB_CUDA(ctx->out_dec.reserve(F * dev.words_n * 4));
        QLB_CUDA(cudaMemcpyAsync(ctx->rate_tab.p, pat.tab.data(), tab_bytes, cudaMemcpyHostToDevice, ctx->stream));
        const uint32_t *d_pos_tab = (const uint32_t *)ctx->rate_tab.p, *d_key_pos = d_pos_tab + dev.n;
        double *d_llr = (double *)ctx->in_llr.p;
        uint32_t *d_word = (uint32_t *)ctx->rate_word.p, *d_syn = (uint32_t *)ctx->in_syn.p, *d_dec = (uint32_t *)ctx->out_dec.p;

        const long long warps = (long long)n_frames * dev.words_n;
        rate_embed_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, ctx->stream>>>(n_frames, dev.n, dev.words_n, pat.words_key(), pat.words_fill(),
                                                                                 d_pos_tab, d_alice, d_bob, d_fill, d_log_prior, p.threshold,
                                                                                 d_llr, d_word);
        QLB_CUDA(cudaGetLastError());
        if (const int rc = launch_syndrome(ctx, dev, n_frames, d_word, d_syn))
            return rc;
        DecodeArgs args{};
        args.code = dev;
        args.n_frames = n_frames;
        args.llr = d_llr;
        args.syndrome_in = d_syn;
        args.iterations = d_iterations;
        args.result = d_result;
        args.decoded = d_dec;
        if (const int rc = launch_decode(ctx, p, false, args))
            return rc;
        const int threads = std::min(256, pat.words_key() * 32); // one warp per key word
        rate_extract_kernel<<<(unsigned)n_frames, threads, 0, ctx->stream>>>(pat.n_key, dev.words_n, pat.words_key(), d_key_pos, d_dec, d_alice,
                                                                             d_result, d_key_out);
        QLB_CUDA(cudaGetLastError());
        return QLB_OK;
    }
}

extern "C"
{
    int qlb_rate_pattern(const qlb_code *code, int32_t n_punctured, int32_t n_shortened, uint64_t seed, uint8_t *class_out)
    {
        if (!code || !class_out)
            return fail(QLB_ERR_INVALID, "qlb_rate_pattern: null code or output");
        const CodeLayout &L = layout_of(code);
        const int32_t N = L.n;
        if (n_punctured < 0 || n_shortened < 0 || (int64_t)n_punctured + n_shortened >= N)
            return fail(QLB_ERR_INVALID, "qlb_rate_pattern: need p >= 0, s >= 0 and p + s < N (p = " + std::to_string(n_punctured) +
                                             ", s = " + std::to_string(n_shortened) + ", N = " + std::to_string(N) + ")");
        std::vector<uint64_t> r((size_t)N);
        Xoshiro256pp rng(seed);
        for (auto &x : r)
            x = rng.next();
        std::vector<int32_t> order((size_t)N);
        std::iota(order.begin(), order.end(), 0);
        std::sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return r[a] != r[b] ? r[a] < r[b] : a < b; });
        // checks of each bit (the code keeps the check half)
        std::vector<int32_t> bit_ptr((size_t)N + 1, 0), bit_checks((size_t)L.e);
        for (int32_t q = 0; q < L.e; ++q)
            ++bit_ptr[L.col_idx[q] + 1];
        std::partial_sum(bit_ptr.begin(), bit_ptr.end(), bit_ptr.begin());
        {
            std::vector<int32_t> fillp(bit_ptr.begin(), bit_ptr.end() - 1);
            for (int32_t j = 0; j < L.m; ++j)
                for (int32_t q = L.row_ptr[j]; q < L.row_ptr[j + 1]; ++q)
                    bit_checks[fillp[L.col_idx[q]]++] = j;
        }
        std::vector<uint8_t> tainted((size_t)L.m, 0), cls((size_t)N, QLB_POS_KEY);
        int32_t punctured = 0;
        for (size_t q = 0; q < order.size() && punctured < n_punctured; ++q)
        {
            const int32_t i = order[q];
            bool free = true;
            for (int32_t k = bit_ptr[i]; k < bit_ptr[i + 1] && free; ++k)
                free = !tainted[bit_checks[k]];
            if (!free)
                continue;
            cls[i] = QLB_POS_PUNCTURED;
            ++punctured;
            for (int32_t k = bit_ptr[i]; k < bit_ptr[i + 1]; ++k)
                tainted[bit_checks[k]] = 1;
        }
        if (punctured < n_punctured) // the walk went through every position
            return fail(QLB_ERR_UNSUPPORTED, "qlb_rate_pattern: " + std::to_string(n_punctured) + " punctured positions requested, the untainted walk of this seed finds " +
                                                 std::to_string(punctured));
        int32_t shortened = 0;
        for (size_t q = 0; q < order.size() && shortened < n_shortened; ++q)
            if (cls[order[q]] == QLB_POS_KEY)
            {
                cls[order[q]] = QLB_POS_SHORTENED;
                ++shortened;
            }
        std::memcpy(class_out, cls.data(), (size_t)N);
        return QLB_OK;
    }

    int qlb_reconcile_adapted_packed(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, const uint8_t *pos_class,
                                     int64_t n_frames, const uint32_t *alice_key_packed, const uint32_t *bob_key_packed,
                                     const uint32_t *fill_packed, const double *qber, uint32_t *iterations_out, uint8_t *result_out,
                                     uint32_t *decoded_key_packed_out)
    {
        if (!ctx || !code || n_frames < 0)
            return fail(QLB_ERR_INVALID, "qlb_reconcile_adapted_packed: null context/code or negative frame count");
        int rc = check_params(params);
        if (rc)
            return rc;
        RatePattern pat;
        if ((rc = scan_pattern(layout_of(code), *params, pos_class, pat)))
            return rc;
        if (n_frames == 0)
            return QLB_OK;
        if (!alice_key_packed || !bob_key_packed || !qber || !iterations_out || !result_out || (pat.words_fill() && !fill_packed))
            return fail(QLB_ERR_INVALID, "qlb_reconcile_adapted_packed: null host buffer");
        ctx->host_logp.resize((size_t)n_frames);
        for (int64_t f = 0; f < n_frames; ++f)
        {
            const double q = qber[f];
            if (q == 0.)
                return fail(QLB_ERR_KEY_TOO_SMALL, "Key size '" + std::to_string(pat.n_key) + "' is too small for QBER.");
            if (!(q > 0. && q < 1.))
                return fail(QLB_ERR_INVALID, "QBER must be: 0 < QBER < 1");
            ctx->host_logp[(size_t)f] = std::log((1. - q) / q);
        }
        QLB_CUDA(cudaSetDevice(ctx->device));
        const CodeDev *dev;
        if ((rc = get_device_code(ctx, code, &dev)))
            return rc;
        const size_t F = (size_t)n_frames, key_bytes = F * pat.words_key() * 4, fill_bytes = F * pat.words_fill() * 4;
        QLB_CUDA(ctx->in_a.reserve(key_bytes));
        QLB_CUDA(ctx->in_b.reserve(key_bytes));
        QLB_CUDA(ctx->rate_fill.reserve(fill_bytes + 4));
        QLB_CUDA(ctx->in_q.reserve(F * 8));
        QLB_CUDA(ctx->out_it.reserve(F * 4));
        QLB_CUDA(ctx->out_res.reserve(F));
        if (decoded_key_packed_out)
            QLB_CUDA(ctx->rate_key.reserve(key_bytes));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_a.p, alice_key_packed, key_bytes, cudaMemcpyHostToDevice, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_b.p, bob_key_packed, key_bytes, cudaMemcpyHostToDevice, ctx->stream));
        if (fill_bytes)
            QLB_CUDA(cudaMemcpyAsync(ctx->rate_fill.p, fill_packed, fill_bytes, cudaMemcpyHostToDevice, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_q.p, ctx->host_logp.data(), F * 8, cudaMemcpyHostToDevice, ctx->stream));
        if ((rc = decode_adapted(ctx, *dev, *params, pat, n_frames, (const uint32_t *)ctx->in_a.p, (const uint32_t *)ctx->in_b.p,
                                 (const uint32_t *)ctx->rate_fill.p, (const double *)ctx->in_q.p, (uint32_t *)ctx->out_it.p,
                                 (uint8_t *)ctx->out_res.p, decoded_key_packed_out ? (uint32_t *)ctx->rate_key.p : nullptr)))
            return rc;
        QLB_CUDA(cudaMemcpyAsync(iterations_out, ctx->out_it.p, F * 4, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(result_out, ctx->out_res.p, F, cudaMemcpyDeviceToHost, ctx->stream));
        if (decoded_key_packed_out)
            QLB_CUDA(cudaMemcpyAsync(decoded_key_packed_out, ctx->rate_key.p, key_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        return QLB_OK;
    }

    int qlb_run_trials_adapted(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, const uint8_t *pos_class,
                               int64_t n_frames, const uint64_t *seeds, uint64_t seed_offset, double qber, uint32_t *iterations_out,
                               uint8_t *result_out, double *exact_qber_out)
    {
        if (!ctx || !code || n_frames < 0 || (n_frames > 0 && (!seeds || !iterations_out || !result_out)))
            return fail(QLB_ERR_INVALID, "qlb_run_trials_adapted: bad arguments");
        int rc = check_params(params);
        if (rc)
            return rc;
        RatePattern pat;
        if ((rc = scan_pattern(layout_of(code), *params, pos_class, pat)))
            return rc;
        QLB_CUDA(cudaSetDevice(ctx->device));
        const size_t F = (size_t)n_frames, key_bytes = F * pat.words_key() * 4;
        QLB_CUDA(ctx->gen_seeds.reserve(F * 8 + 8));
        QLB_CUDA(ctx->in_a.reserve(key_bytes + 4));
        QLB_CUDA(ctx->in_b.reserve(key_bytes + 4));
        QLB_CUDA(ctx->rate_fill.reserve(F * pat.words_fill() * 4 + 4));
        QLB_CUDA(ctx->in_q.reserve(F * 8 + 8));
        QLB_CUDA(ctx->out_it.reserve(F * 4 + 4));
        QLB_CUDA(ctx->out_res.reserve(F + 4));
        if (n_frames)
            QLB_CUDA(cudaMemcpyAsync(ctx->gen_seeds.p, seeds, F * 8, cudaMemcpyHostToDevice, ctx->stream));
        double exact = 0.;
        const uint64_t *d_seeds = (const uint64_t *)ctx->gen_seeds.p;
        rc = qlb_generate_device(ctx, pat.n_key, n_frames, d_seeds, seed_offset, qber, (uint32_t *)ctx->in_a.p, (uint32_t *)ctx->in_b.p, &exact);
        if (exact_qber_out)
            *exact_qber_out = exact;
        if (rc || n_frames == 0)
            return rc;
        if (pat.words_fill())
        {
            rate_fill_kernel<<<(unsigned)((n_frames + 127) / 128), 128, 0, ctx->stream>>>(n_frames, pat.n_punct + pat.n_short, pat.words_fill(),
                                                                                           d_seeds, seed_offset, (uint32_t *)ctx->rate_fill.p);
            QLB_CUDA(cudaGetLastError());
        }
        // ln((1-q)/q) of the exact ratio over the n key bits, on the host in double (as qlb_run_trials)
        ctx->host_logp.assign(F, std::log((1. - exact) / exact));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_q.p, ctx->host_logp.data(), F * 8, cudaMemcpyHostToDevice, ctx->stream));
        const CodeDev *dev;
        if ((rc = get_device_code(ctx, code, &dev)))
            return rc;
        if ((rc = decode_adapted(ctx, *dev, *params, pat, n_frames, (const uint32_t *)ctx->in_a.p, (const uint32_t *)ctx->in_b.p,
                                 (const uint32_t *)ctx->rate_fill.p, (const double *)ctx->in_q.p, (uint32_t *)ctx->out_it.p,
                                 (uint8_t *)ctx->out_res.p, nullptr)))
            return rc;
        QLB_CUDA(cudaMemcpyAsync(iterations_out, ctx->out_it.p, F * 4, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(result_out, ctx->out_res.p, F, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        return QLB_OK;
    }
}
