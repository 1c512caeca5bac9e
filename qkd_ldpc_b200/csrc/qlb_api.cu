// C-ABI of libqkdldpc_b200.so (declared in include/qkd_ldpc_b200.h): code handles, per-GPU contexts, and the batch
// entry points that replace the reference's per-frame hot-path functions. No CPU compute path exists here: every
// entry that does work launches the sm_100a kernels in qlb_kernels.cuh or fails.
#include "qlb_internal.hpp"
#include "qlb_generate.cuh"
#include "qlb_trace_f64.cuh"
#include "qlb_layout.hpp"

#include <atomic>
#include <dlfcn.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

using namespace qlb;

namespace qlb
{
    // Test probe: the fp64 building blocks of the check rule, element-wise (see qlb_test_f64_math in the header).
    __global__ void f64_math_probe_kernel(int op, long long n, const double *__restrict__ a, const double *__restrict__ b, double *__restrict__ out)
    {
        const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
            return;
        const double x = a[i], y = b ? b[i] : 0.;
        double r;
        switch (op)
        {
        case 0: r = MathF64::quotient(x, y); break;
        case 1: r = f64m::exp_neg(x); break;
        case 2: r = f64m::log_ratio(x, y); break;
        case 3: r = MathF64::tanh_half(x); break;
        case 4: r = MathF64::two_atanh(x, y != 0.); break;
        case 5: r = f64m::exp_neg_abs(x); break;
        default: r = 0.; break;
        }
        out[i] = r;
    }
    // op 6: the whole check rule as the resident fp64 kernel runs it (MathF64::check_fast with the exp table in shared memory and
    // want_inf routed at compile time), one check per record of 8 doubles: a = the W messages, b = {W, syndrome bit, thr_eff}
    template <int W>
    __device__ __forceinline__ void f64_rule_probe(const double *a, double s, double thr_eff, const double2 *s_tab, double *out)
    {
        double v[W];
#pragma unroll
        for (int k = 0; k < W; ++k)
            v[k] = a[k];
        if (!(thr_eff <= 700.))
            MathF64::check_fast<W, true>(v, s != 0., thr_eff, s_tab);
        else
            MathF64::check_fast<W, false>(v, s != 0., thr_eff, s_tab);
#pragma unroll
        for (int k = 0; k < W; ++k)
            out[k] = v[k];
    }
    __global__ void f64_rule_probe_kernel(long long checks, const double *__restrict__ a, const double *__restrict__ b, double *__restrict__ out)
    {
        __shared__ double2 s_tab[32];
        if (threadIdx.x < 32)
            s_tab[threadIdx.x] = f64m::kExpTab[threadIdx.x];
        __syncthreads();
        const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
        if (c >= checks)
            return;
        const double *x = a + 8 * c, *p = b + 8 * c;
        double *o = out + 8 * c;
        switch ((int)p[0])
        {
        case 3: f64_rule_probe<3>(x, p[1], p[2], s_tab, o); break;
        case 4: f64_rule_probe<4>(x, p[1], p[2], s_tab, o); break;
        case 5: f64_rule_probe<5>(x, p[1], p[2], s_tab, o); break;
        case 6: f64_rule_probe<6>(x, p[1], p[2], s_tab, o); break;
        case 7: f64_rule_probe<7>(x, p[1], p[2], s_tab, o); break;
        case 8: f64_rule_probe<8>(x, p[1], p[2], s_tab, o); break;
        default: break;
        }
    }
}

namespace
{
    thread_local std::string g_error;
    std::atomic<uint64_t> g_next_code_id{1};
}
namespace qlb
{
    int fail(int code, const std::string &msg)
    {
        g_error = msg;
        return code;
    }
    int cuda_fail(cudaError_t e, const char *what)
    {
        return fail(QLB_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
    }
}

struct qlb_code
{
    uint64_t id;
    CodeLayout L;
};

namespace
{
    int upload(const void *src, size_t bytes, DeviceCode &dc, const void **dst_out)
    {
        void *d = nullptr;
        QLB_CUDA(cudaMalloc(&d, bytes ? bytes : 4));
        dc.allocs.push_back(d);
        if (bytes)
            QLB_CUDA(cudaMemcpy(d, src, bytes, cudaMemcpyHostToDevice));
        *dst_out = d;
        return QLB_OK;
    }
}

namespace qlb
{
    const CodeLayout &layout_of(const qlb_code *code) { return code->L; }

    int get_device_code(qlb_ctx *ctx, const qlb_code *code, const CodeDev **out)
    {
        auto it = ctx->codes.find(code->id);
        if (it != ctx->codes.end())
        {
            *out = &it->second.dev;
            return QLB_OK;
        }
        const CodeLayout &L = code->L;
        DeviceCode dc;
        CodeDev &d = dc.dev;
        d.n = L.n;
        d.m = L.m;
        d.e = L.e;
        d.words_n = L.words_n;
        d.words_m = L.words_m;
        d.max_check_w = L.max_check_w;
        d.max_bit_w = L.max_bit_w;
        for (int k = 0; k < kMaxCW; ++k)
        {
            d.cnt[k] = k < L.max_check_w ? L.cnt[k] : 0;
            d.base[k] = k < L.max_check_w ? L.base[k] : 0;
        }
        for (int k = 0; k < 16; ++k)
            d.base4[k] = 4u * d.base[k];
        d.uniform_bit_w = L.uniform_bit_w;
        d.slots = L.slots;
        int rc;
        const void *p = nullptr;
        if (L.slots < 65535)
        {
            std::vector<uint16_t> s16((L.bit_slots.size() + 7) / 8 * 8, 0xFFFFu); // 16-byte padded for the TMA bulk copy
            for (size_t i = 0; i < L.bit_slots.size(); ++i)
                s16[i] = L.bit_slots[i] == kNoSlot ? 0xFFFFu : static_cast<uint16_t>(L.bit_slots[i]);
            if ((rc = upload(s16.data(), s16.size() * 2, dc, &p)))
                return rc;
            d.bit_slots16 = static_cast<const uint16_t *>(p);
        }
        if ((rc = upload(L.bit_slots.data(), L.bit_slots.size() * 4, dc, &p)))
            return rc;
        d.bit_slots32 = static_cast<const uint32_t *>(p);
        if (L.n < 65536)
        {
            std::vector<uint16_t> c16(L.col_of_slot.size());
            for (size_t i = 0; i < c16.size(); ++i)
                c16[i] = L.col_of_slot[i] == kNoSlot ? 0xFFFFu : static_cast<uint16_t>(L.col_of_slot[i]);
            if ((rc = upload(c16.data(), c16.size() * 2, dc, &p)))
                return rc;
            d.col_of_slot16 = static_cast<const uint16_t *>(p);
        }
        if ((rc = upload(L.col_of_slot.data(), L.col_of_slot.size() * 4, dc, &p)))
            return rc;
        d.col_of_slot32 = static_cast<const uint32_t *>(p);
        if ((rc = upload(L.check_order.data(), L.check_order.size() * 4, dc, &p)))
            return rc;
        d.check_order = static_cast<const uint32_t *>(p);
        if ((rc = upload(L.row_ptr.data(), L.row_ptr.size() * 4, dc, &p)))
            return rc;
        d.row_ptr = static_cast<const int32_t *>(p);
        if ((rc = upload(L.col_idx.data(), L.col_idx.size() * 4, dc, &p)))
            return rc;
        d.col_idx = static_cast<const int32_t *>(p);
        {
            std::vector<uint32_t> cg;
            std::vector<uint16_t> bg;
            uint32_t smem_slots = 0;
            if (resident64_build_tables(ctx, d, L.bit_slots.data(), cg, bg, smem_slots))
            {
                if ((rc = upload(cg.data(), cg.size() * 4, dc, &p)))
                    return rc;
                d.r64_check_group_table = static_cast<const uint32_t *>(p);
                if ((rc = upload(bg.data(), bg.size() * 2, dc, &p)))
                    return rc;
                d.r64_bit_group_table = static_cast<const uint16_t *>(p);
                d.r64_check_groups = (int32_t)cg.size();
                d.r64_bit_groups = (int32_t)bg.size();
                d.r64_smem_slots = smem_slots;
            }
        }
        auto ins = ctx->codes.emplace(code->id, std::move(dc));
        *out = &ins.first->second.dev;
        return QLB_OK;
    }

    int check_params(const qlb_decode_params *p)
    {
        if (!p)
            return fail(QLB_ERR_INVALID, "decode params are null");
        if (p->precision != QLB_PRECISION_F64 && p->precision != QLB_PRECISION_F32)
            return fail(QLB_ERR_INVALID, "precision must be 64 or 32");
        if (p->max_iterations < 1)
            return fail(QLB_ERR_INVALID, "Minimum number of sum-product iterations must be >= 1!");
        if (p->enable_threshold && !(p->threshold > 0.))
            return fail(QLB_ERR_INVALID, "Sum-product message LLR threshold must be > 0!");
        if ((p->flags & QLB_FLAG_F32_FAST_MATH) && p->precision != QLB_PRECISION_F32)
            return fail(QLB_ERR_INVALID, "QLB_FLAG_F32_FAST_MATH requires fp32 precision");
        if ((p->flags & QLB_FLAG_F64_FUSED_RATIO) && p->precision != QLB_PRECISION_F64)
            return fail(QLB_ERR_INVALID, "QLB_FLAG_F64_FUSED_RATIO requires fp64 precision");
        if (p->stream_max_bundles < 0 || p->block_threads < 0)
            return fail(QLB_ERR_INVALID, "qlb_decode_params: negative execution knob");
        if (p->flags & QLB_FLAG_F32_MIN_SUM)
        {
            if (p->precision != QLB_PRECISION_F32)
                return fail(QLB_ERR_INVALID, "QLB_FLAG_F32_MIN_SUM requires fp32 precision");
            if (p->flags & QLB_FLAG_F32_FAST_MATH)
                return fail(QLB_ERR_INVALID, "QLB_FLAG_F32_MIN_SUM and QLB_FLAG_F32_FAST_MATH exclude each other");
            if (!(p->min_sum_scale > 0.f && p->min_sum_scale <= 1.f))
                return fail(QLB_ERR_INVALID, "qlb_decode_params.min_sum_scale must be in (0, 1] with QLB_FLAG_F32_MIN_SUM");
        }
        else if (p->min_sum_scale != 0.f) // also a NaN
            return fail(QLB_ERR_INVALID, "qlb_decode_params.min_sum_scale must be 0 without QLB_FLAG_F32_MIN_SUM");
        if (((p->flags >> QLB_FLAG_TEST_TIER_SHIFT) & 0xF) > 4)
            return fail(QLB_ERR_INVALID, "qlb_decode_params.flags: the test hook (bits 8..11) must be 0 (none) or 1 + hook, hook 0 ... 3");
        return QLB_OK;
    }

    int launch_syndrome(qlb_ctx *ctx, const CodeDev &dev, long long n_frames, const uint32_t *d_bits, uint32_t *d_out)
    {
        const size_t per_frame = (size_t)dev.words_n * 4;
        int group = kSynFrames, stage = 1;
        const size_t budget = 96 * 1024;
        if (per_frame > budget)
        {
            group = 1;
            stage = 0;
        }
        else
            while ((size_t)group * per_frame > budget)
                group >>= 1;
        const size_t smem = stage ? (size_t)group * per_frame : 0;
        QLB_CUDA(allow_full_dynamic_smem(ctx, syndrome_kernel<kSynThreads>));
        const long long grid = (n_frames + group - 1) / group;
        syndrome_kernel<kSynThreads><<<(unsigned)grid, kSynThreads, smem, ctx->stream>>>(dev, n_frames, group, stage, d_bits, d_out);
        QLB_CUDA(cudaGetLastError());
        return QLB_OK;
    }

}

namespace
{
    void pack_frames(const int32_t *bits, int64_t frames, int n, int words, uint32_t *out)
    {
        for (int64_t f = 0; f < frames; ++f)
        {
            const int32_t *src = bits + f * n;
            uint32_t *dst = out + f * words;
            for (int w = 0; w < words; ++w)
            {
                uint32_t v = 0;
                const int lim = n - w * 32 < 32 ? n - w * 32 : 32;
                for (int b = 0; b < lim; ++b)
                    v |= static_cast<uint32_t>(src[w * 32 + b] & 1) << b;
                dst[w] = v;
            }
        }
    }
    void unpack_frames(const uint32_t *packed, int64_t frames, int n, int words, int32_t *out)
    {
        for (int64_t f = 0; f < frames; ++f)
            for (int i = 0; i < n; ++i)
                out[f * n + i] = static_cast<int32_t>((packed[f * words + (i >> 5)] >> (i & 31)) & 1u);
    }
}

extern "C"
{
    int qlb_version(void) { return QLB_VERSION; }
    const char *qlb_last_error(void) { return g_error.c_str(); }

    int qlb_device_count(void)
    {
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess)
        {
            cudaGetLastError();
            return 0;
        }
        return n;
    }

    int qlb_code_create(int32_t n_bits, int32_t n_checks, const int32_t *row_ptr, const int32_t *col_idx,
                        const int32_t *col_ptr, const int32_t *row_idx, qlb_code **code_out)
    {
        if (!code_out)
            return fail(QLB_ERR_INVALID, "code_out is null");
        *code_out = nullptr;
        qlb_code *c = new qlb_code();
        const std::string err = c->L.build(n_bits, n_checks, row_ptr, col_idx, col_ptr, row_idx);
        if (!err.empty())
        {
            delete c;
            return fail(QLB_ERR_INVALID, err);
        }
        c->id = g_next_code_id.fetch_add(1);
        *code_out = c;
        return QLB_OK;
    }
    void qlb_code_destroy(qlb_code *code) { delete code; }
    int32_t qlb_code_n(const qlb_code *c) { return c ? c->L.n : 0; }
    int32_t qlb_code_m(const qlb_code *c) { return c ? c->L.m : 0; }
    int32_t qlb_code_edges(const qlb_code *c) { return c ? c->L.e : 0; }
    int32_t qlb_code_words_n(const qlb_code *c) { return c ? c->L.words_n : 0; }
    int32_t qlb_code_words_m(const qlb_code *c) { return c ? c->L.words_m : 0; }
    int32_t qlb_code_max_bit_weight(const qlb_code *c) { return c ? c->L.max_bit_w : 0; }
    int32_t qlb_code_max_check_weight(const qlb_code *c) { return c ? c->L.max_check_w : 0; }
    int32_t qlb_code_slots(const qlb_code *c) { return c ? c->L.slots : 0; }
    int qlb_code_layout(const qlb_code *c, uint32_t *slot_of_edge, uint32_t *bit_slots, uint32_t *check_order)
    {
        if (!c)
            return fail(QLB_ERR_INVALID, "code is null");
        if (slot_of_edge)
            std::memcpy(slot_of_edge, c->L.slot_of_edge.data(), c->L.slot_of_edge.size() * 4);
        if (bit_slots)
            std::memcpy(bit_slots, c->L.bit_slots.data(), c->L.bit_slots.size() * 4);
        if (check_order)
            std::memcpy(check_order, c->L.check_order.data(), c->L.check_order.size() * 4);
        return QLB_OK;
    }

    int qlb_code_gather_wavefronts(const qlb_code *c, double *naive_out, double *placed_out)
    {
        if (!c)
            return fail(QLB_ERR_INVALID, "code is null");
        if (naive_out)
            *naive_out = c->L.gather_wavefronts_naive;
        if (placed_out)
            *placed_out = c->L.gather_wavefronts_opt;
        return QLB_OK;
    }

    int qlb_ctx_create(int device, qlb_ctx **ctx_out)
    {
        if (!ctx_out)
            return fail(QLB_ERR_INVALID, "ctx_out is null");
        *ctx_out = nullptr;
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0)
        {
            cudaGetLastError();
            return fail(QLB_ERR_CUDA, "no CUDA device is available: libqkdldpc_b200 has no CPU path");
        }
        if (device < 0 || device >= count)
            return fail(QLB_ERR_INVALID, "device index out of range");
        cudaDeviceProp prop;
        QLB_CUDA(cudaGetDeviceProperties(&prop, device));
        if (prop.major < 10)
            return fail(QLB_ERR_CUDA, std::string("device '") + prop.name + "' is not sm_100-class; the kernels are built for sm_100a only");
        QLB_CUDA(cudaSetDevice(device));
        qlb_ctx *ctx = new qlb_ctx();
        ctx->device = device;
        ctx->sm_count = prop.multiProcessorCount;
        ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
        if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaEventCreate(&ctx->ev_start)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev_stop)) != cudaSuccess ||
            (e = cudaMalloc(&ctx->d_counters, 2 * sizeof(unsigned long long))) != cudaSuccess ||
            (e = cudaMemset(ctx->d_counters, 0, 2 * sizeof(unsigned long long))) != cudaSuccess)
        {
            qlb_ctx_destroy(ctx);
            return cuda_fail(e, "context setup");
        }
        *ctx_out = ctx;
        return QLB_OK;
    }

    void qlb_ctx_destroy(qlb_ctx *ctx)
    {
        if (!ctx)
            return;
        cudaSetDevice(ctx->device);
        if (ctx->stream)
            cudaStreamSynchronize(ctx->stream);
        for (auto &kv : ctx->codes)
            for (void *p : kv.second.allocs)
                cudaFree(p);
        for (DevBuf *b : {&ctx->scratch, &ctx->in_a, &ctx->in_b, &ctx->in_q, &ctx->in_llr, &ctx->in_syn, &ctx->out_it,
                          &ctx->out_res, &ctx->out_dec, &ctx->out_syn, &ctx->gen_perm, &ctx->gen_seeds, &ctx->rate_tab,
                          &ctx->rate_fill, &ctx->rate_word, &ctx->rate_key})
            b->release();
        if (ctx->d_counters)
            cudaFree(ctx->d_counters);
        if (ctx->ev_start)
            cudaEventDestroy(ctx->ev_start);
        if (ctx->ev_stop)
            cudaEventDestroy(ctx->ev_stop);
        if (ctx->stream)
            cudaStreamDestroy(ctx->stream);
        delete ctx;
    }

    int qlb_ctx_device(const qlb_ctx *ctx) { return ctx ? ctx->device : -1; }
    int qlb_ctx_sm_count(const qlb_ctx *ctx) { return ctx ? ctx->sm_count : 0; }
    void *qlb_ctx_stream(const qlb_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
    const char *qlb_ctx_last_decoder(const qlb_ctx *ctx) { return ctx ? ctx->last_decoder : ""; }
    int qlb_ctx_synchronize(qlb_ctx *ctx)
    {
        if (!ctx)
            return fail(QLB_ERR_INVALID, "ctx is null");
        QLB_CUDA(cudaSetDevice(ctx->device));
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        return QLB_OK;
    }
    int qlb_ctx_counters(qlb_ctx *ctx, uint64_t *kernel_launches, uint64_t *frame_iterations, int reset)
    {
        if (!ctx)
            return fail(QLB_ERR_INVALID, "ctx is null");
        QLB_CUDA(cudaSetDevice(ctx->device));
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        unsigned long long it = 0;
        QLB_CUDA(cudaMemcpy(&it, ctx->d_counters + 1, sizeof(it), cudaMemcpyDeviceToHost));
        if (kernel_launches)
            *kernel_launches = ctx->launches;
        if (frame_iterations)
            *frame_iterations = it;
        if (reset)
        {
            ctx->launches = 0;
            QLB_CUDA(cudaMemset(ctx->d_counters + 1, 0, sizeof(unsigned long long)));
        }
        return QLB_OK;
    }
    int qlb_ctx_timer_start(qlb_ctx *ctx)
    {
        if (!ctx)
            return fail(QLB_ERR_INVALID, "ctx is null");
        QLB_CUDA(cudaSetDevice(ctx->device));
        QLB_CUDA(cudaEventRecord(ctx->ev_start, ctx->stream));
        return QLB_OK;
    }
    int qlb_ctx_timer_stop(qlb_ctx *ctx, float *elapsed_ms_out)
    {
        if (!ctx || !elapsed_ms_out)
            return fail(QLB_ERR_INVALID, "ctx or output is null");
        QLB_CUDA(cudaSetDevice(ctx->device));
        QLB_CUDA(cudaEventRecord(ctx->ev_stop, ctx->stream));
        QLB_CUDA(cudaEventSynchronize(ctx->ev_stop));
        QLB_CUDA(cudaEventElapsedTime(elapsed_ms_out, ctx->ev_start, ctx->ev_stop));
        return QLB_OK;
    }

    // ---- syndrome ---------------------------------------------------------------------------------------------------
    int qlb_syndrome_batch_packed(qlb_ctx *ctx, const qlb_code *code, int64_t n_frames, const uint32_t *bits_packed,
                                  uint32_t *syndrome_packed_out)
    {
        if (!ctx || !code || n_frames < 0 || (n_frames > 0 && (!bits_packed || !syndrome_packed_out)))
            return fail(QLB_ERR_INVALID, "qlb_syndrome_batch_packed: null argument or negative frame count");
        if (n_frames == 0)
            return QLB_OK;
        QLB_CUDA(cudaSetDevice(ctx->device));
        const CodeDev *dev;
        int rc = get_device_code(ctx, code, &dev);
        if (rc)
            return rc;
        const size_t in_bytes = (size_t)n_frames * dev->words_n * 4, out_bytes = (size_t)n_frames * dev->words_m * 4;
        QLB_CUDA(ctx->in_a.reserve(in_bytes));
        QLB_CUDA(ctx->out_syn.reserve(out_bytes));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_a.p, bits_packed, in_bytes, cudaMemcpyHostToDevice, ctx->stream));
        if ((rc = launch_syndrome(ctx, *dev, n_frames, (const uint32_t *)ctx->in_a.p, (uint32_t *)ctx->out_syn.p)))
            return rc;
        QLB_CUDA(cudaMemcpyAsync(syndrome_packed_out, ctx->out_syn.p, out_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        return QLB_OK;
    }

    int qlb_syndrome_batch(qlb_ctx *ctx, const qlb_code *code, int64_t n_frames, const int32_t *bits, int32_t *syndrome_out)
    {
        if (!ctx || !code || n_frames < 0 || (n_frames > 0 && (!bits || !syndrome_out)))
            return fail(QLB_ERR_INVALID, "qlb_syndrome_batch: null argument or negative frame count");
        if (n_frames == 0)
            return QLB_OK;
        const CodeLayout &L = code->L;
        ctx->host_pack_a.resize((size_t)n_frames * L.words_n);
        ctx->host_pack_out.resize((size_t)n_frames * L.words_m);
        pack_frames(bits, n_frames, L.n, L.words_n, ctx->host_pack_a.data());
        int rc = qlb_syndrome_batch_packed(ctx, code, n_frames, ctx->host_pack_a.data(), ctx->host_pack_out.data());
        if (rc)
            return rc;
        unpack_frames(ctx->host_pack_out.data(), n_frames, L.m, L.words_m, syndrome_out);
        return QLB_OK;
    }

    // ---- reconcile --------------------------------------------------------------------------------------------------
    int qlb_reconcile_device(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, int64_t n_frames,
                             const uint32_t *d_alice_packed, const uint32_t *d_bob_packed, const double *d_log_prior,
                             uint32_t *d_iterations_out, uint8_t *d_result_out, uint32_t *d_decoded_packed_out,
                             uint32_t *d_syndrome_packed_out)
    {
        if (!ctx || !code || n_frames < 0)
            return fail(QLB_ERR_INVALID, "qlb_reconcile_device: null context/code or negative frame count");
        int rc = check_params(params);
        if (rc)
            return rc;
        if (n_frames == 0)
            return QLB_OK;
        if (!d_alice_packed || !d_bob_packed || !d_log_prior || !d_iterations_out || !d_result_out)
            return fail(QLB_ERR_INVALID, "qlb_reconcile_device: null device buffer");
        QLB_CUDA(cudaSetDevice(ctx->device));
        const CodeDev *dev;
        if ((rc = get_device_code(ctx, code, &dev)))
            return rc;
        DecodeArgs args{};
        args.code = *dev;
        args.n_frames = n_frames;
        args.alice = d_alice_packed;
        args.bob = d_bob_packed;
        args.log_prior = d_log_prior;
        args.iterations = d_iterations_out;
        args.result = d_result_out;
        args.decoded = d_decoded_packed_out;
        args.syndrome_out = d_syndrome_packed_out;
        return launch_decode(ctx, *params, true, args);
    }

    int qlb_reconcile_batch_packed(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, int64_t n_frames,
                                   const uint32_t *alice_packed, const uint32_t *bob_packed, const double *qber,
                                   uint32_t *iterations_out, uint8_t *result_out, uint32_t *decoded_packed_out,
                                   uint32_t *syndrome_packed_out)
    {
        if (!ctx || !code || n_frames < 0)
            return fail(QLB_ERR_INVALID, "qlb_reconcile_batch_packed: null context/code or negative frame count");
        int rc = check_params(params);
        if (rc)
            return rc;
        if (n_frames == 0)
            return QLB_OK;
        if (!alice_packed || !bob_packed || !qber || !iterations_out || !result_out)
            return fail(QLB_ERR_INVALID, "qlb_reconcile_batch_packed: null host buffer");
        const CodeLayout &L = code->L;
        // ln((1-q)/q) on the host in double, exactly as the reference forms it (src/qkd_ldpc_algorithm.cpp:400)
        ctx->host_logp.resize((size_t)n_frames);
        for (int64_t f = 0; f < n_frames; ++f)
        {
            const double q = qber[f];
            if (q == 0.)
                return fail(QLB_ERR_KEY_TOO_SMALL, "Key size '" + std::to_string(L.n) + "' is too small for QBER.");
            if (!(q > 0. && q < 1.))
                return fail(QLB_ERR_INVALID, "QBER must be: 0 < QBER < 1");
            ctx->host_logp[(size_t)f] = std::log((1. - q) / q);
        }
        QLB_CUDA(cudaSetDevice(ctx->device));
        const size_t key_bytes = (size_t)n_frames * L.words_n * 4, syn_bytes = (size_t)n_frames * L.words_m * 4;
        QLB_CUDA(ctx->in_a.reserve(key_bytes));
        QLB_CUDA(ctx->in_b.reserve(key_bytes));
        QLB_CUDA(ctx->in_q.reserve((size_t)n_frames * 8));
        QLB_CUDA(ctx->out_it.reserve((size_t)n_frames * 4));
        QLB_CUDA(ctx->out_res.reserve((size_t)n_frames));
        if (decoded_packed_out)
            QLB_CUDA(ctx->out_dec.reserve(key_bytes));
        if (syndrome_packed_out)
            QLB_CUDA(ctx->out_syn.reserve(syn_bytes));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_a.p, alice_packed, key_bytes, cudaMemcpyHostToDevice, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_b.p, bob_packed, key_bytes, cudaMemcpyHostToDevice, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_q.p, ctx->host_logp.data(), (size_t)n_frames * 8, cudaMemcpyHostToDevice, ctx->stream));
        rc = qlb_reconcile_device(ctx, code, params, n_frames, (const uint32_t *)ctx->in_a.p, (const uint32_t *)ctx->in_b.p,
                                  (const double *)ctx->in_q.p, (uint32_t *)ctx->out_it.p, (uint8_t *)ctx->out_res.p,
                                  decoded_packed_out ? (uint32_t *)ctx->out_dec.p : nullptr,
                                  syndrome_packed_out ? (uint32_t *)ctx->out_syn.p : nullptr);
        if (rc)
            return rc;
        QLB_CUDA(cudaMemcpyAsync(iterations_out, ctx->out_it.p, (size_t)n_frames * 4, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(result_out, ctx->out_res.p, (size_t)n_frames, cudaMemcpyDeviceToHost, ctx->stream));
        if (decoded_packed_out)
            QLB_CUDA(cudaMemcpyAsync(decoded_packed_out, ctx->out_dec.p, key_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        if (syndrome_packed_out)
            QLB_CUDA(cudaMemcpyAsync(syndrome_packed_out, ctx->out_syn.p, syn_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        return QLB_OK;
    }

    int qlb_reconcile_batch(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, int64_t n_frames,
                            const int32_t *alice, const int32_t *bob, const double *qber, uint32_t *iterations_out,
                            uint8_t *result_out, int32_t *decoded_out, int32_t *syndrome_out)
    {
        if (!ctx || !code || n_frames < 0)
            return fail(QLB_ERR_INVALID, "qlb_reconcile_batch: null context/code or negative frame count");
        if (n_frames == 0)
            return check_params(params);
        if (!alice || !bob)
            return fail(QLB_ERR_INVALID, "qlb_reconcile_batch: null key buffer");
        const CodeLayout &L = code->L;
        ctx->host_pack_a.resize((size_t)n_frames * L.words_n);
        ctx->host_pack_b.resize((size_t)n_frames * L.words_n);
        pack_frames(alice, n_frames, L.n, L.words_n, ctx->host_pack_a.data());
        pack_frames(bob, n_frames, L.n, L.words_n, ctx->host_pack_b.data());
        std::vector<uint32_t> dec, syn;
        if (decoded_out)
            dec.resize((size_t)n_frames * L.words_n);
        if (syndrome_out)
            syn.resize((size_t)n_frames * L.words_m);
        int rc = qlb_reconcile_batch_packed(ctx, code, params, n_frames, ctx->host_pack_a.data(), ctx->host_pack_b.data(), qber,
                                            iterations_out, result_out, decoded_out ? dec.data() : nullptr,
                                            syndrome_out ? syn.data() : nullptr);
        if (rc)
            return rc;
        if (decoded_out)
            unpack_frames(dec.data(), n_frames, L.n, L.words_n, decoded_out);
        if (syndrome_out)
            unpack_frames(syn.data(), n_frames, L.m, L.words_m, syndrome_out);
        return QLB_OK;
    }

    // ---- sum-product ------------------------------------------------------------------------------------------------
    int qlb_sum_product_batch(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, int64_t n_frames,
                              const double *llr, const int32_t *syndrome, int32_t *bits_out, uint32_t *iterations_out,
                              uint8_t *result_out)
    {
        if (!ctx || !code || n_frames < 0)
            return fail(QLB_ERR_INVALID, "qlb_sum_product_batch: null context/code or negative frame count");
        int rc = check_params(params);
        if (rc)
            return rc;
        if (n_frames == 0)
            return QLB_OK;
        if (!llr || !syndrome || !iterations_out || !result_out)
            return fail(QLB_ERR_INVALID, "qlb_sum_product_batch: null host buffer");
        const CodeLayout &L = code->L;
        QLB_CUDA(cudaSetDevice(ctx->device));
        const CodeDev *dev;
        if ((rc = get_device_code(ctx, code, &dev)))
            return rc;
        ctx->host_pack_a.resize((size_t)n_frames * L.words_m);
        pack_frames(syndrome, n_frames, L.m, L.words_m, ctx->host_pack_a.data());
        const size_t llr_bytes = (size_t)n_frames * L.n * 8, syn_bytes = (size_t)n_frames * L.words_m * 4,
                     key_bytes = (size_t)n_frames * L.words_n * 4;
        QLB_CUDA(ctx->in_llr.reserve(llr_bytes));
        QLB_CUDA(ctx->in_syn.reserve(syn_bytes));
        QLB_CUDA(ctx->out_it.reserve((size_t)n_frames * 4));
        QLB_CUDA(ctx->out_res.reserve((size_t)n_frames));
        QLB_CUDA(ctx->out_dec.reserve(key_bytes));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_llr.p, llr, llr_bytes, cudaMemcpyHostToDevice, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_syn.p, ctx->host_pack_a.data(), syn_bytes, cudaMemcpyHostToDevice, ctx->stream));
        DecodeArgs args{};
        args.code = *dev;
        args.n_frames = n_frames;
        args.llr = (const double *)ctx->in_llr.p;
        args.syndrome_in = (const uint32_t *)ctx->in_syn.p;
        args.iterations = (uint32_t *)ctx->out_it.p;
        args.result = (uint8_t *)ctx->out_res.p;
        args.decoded = (uint32_t *)ctx->out_dec.p;
        if ((rc = launch_decode(ctx, *params, false, args)))
            return rc;
        QLB_CUDA(cudaMemcpyAsync(iterations_out, ctx->out_it.p, (size_t)n_frames * 4, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(result_out, ctx->out_res.p, (size_t)n_frames, cudaMemcpyDeviceToHost, ctx->stream));
        if (bits_out)
        {
            ctx->host_pack_out.resize((size_t)n_frames * L.words_n);
            QLB_CUDA(cudaMemcpyAsync(ctx->host_pack_out.data(), ctx->out_dec.p, key_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        }
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        if (bits_out)
            unpack_frames(ctx->host_pack_out.data(), n_frames, L.n, L.words_n, bits_out);
        return QLB_OK;
    }

    // ---- trace form of one decode (qlb_trace_f64.cuh) ------------------------------------------------------------------
    int qlb_sum_product_trace(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, const double *llr,
                              const int32_t *syndrome, int32_t capacity, double *e_out, double *l_out, int32_t *z_out,
                              int32_t *s_out, double *m_out, int32_t *bits_out, uint32_t *iterations_out, uint8_t *result_out)
    {
        if (!ctx || !code || capacity < 0)
            return fail(QLB_ERR_INVALID, "qlb_sum_product_trace: null context/code or negative capacity");
        int rc = check_params(params);
        if (rc)
            return rc;
        if (params->precision != QLB_PRECISION_F64)
            return fail(QLB_ERR_UNSUPPORTED, "qlb_sum_product_trace: the trace exists for the reference's arithmetic (fp64) only");
        if (!llr || !syndrome || !iterations_out || !result_out)
            return fail(QLB_ERR_INVALID, "qlb_sum_product_trace: null host buffer");
        const CodeLayout &L = code->L;
        QLB_CUDA(cudaSetDevice(ctx->device));
        const CodeDev *dev;
        if ((rc = get_device_code(ctx, code, &dev)))
            return rc;
        if (capacity > params->max_iterations)
            capacity = params->max_iterations;
        const size_t slots = (size_t)L.slots, n = (size_t)L.n, m = (size_t)L.m, cap = (size_t)capacity;
        // device scratch: msg[slots] | snap_e[cap][slots] | snap_m[cap][slots] | tot[cap][n] (doubles) | z_cur[n] | z[cap][n] | s[cap][m] (int32)
        const size_t n_f64 = slots + 2 * cap * slots + cap * n, n_i32 = n + cap * n + cap * m;
        QLB_CUDA(ctx->scratch.reserve(n_f64 * 8 + n_i32 * 4));
        double *d_msg = static_cast<double *>(ctx->scratch.p), *d_e = d_msg + slots, *d_m = d_e + cap * slots, *d_tot = d_m + cap * slots;
        int32_t *d_zcur = reinterpret_cast<int32_t *>(d_tot + cap * n), *d_z = d_zcur + n, *d_s = d_z + cap * n;
        ctx->host_pack_a.resize(L.words_m);
        pack_frames(syndrome, 1, L.m, L.words_m, ctx->host_pack_a.data());
        QLB_CUDA(ctx->in_llr.reserve(n * 8));
        QLB_CUDA(ctx->in_syn.reserve((size_t)L.words_m * 4));
        QLB_CUDA(ctx->out_it.reserve(4));
        QLB_CUDA(ctx->out_res.reserve(1));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_llr.p, llr, n * 8, cudaMemcpyHostToDevice, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_syn.p, ctx->host_pack_a.data(), (size_t)L.words_m * 4, cudaMemcpyHostToDevice, ctx->stream));
        QLB_CUDA(cudaMemsetAsync(d_msg, 0, n_f64 * 8 + n_i32 * 4, ctx->stream));
        trace_f64_kernel<<<1, kTraceThreads, 0, ctx->stream>>>(*dev, (const double *)ctx->in_llr.p, (const uint32_t *)ctx->in_syn.p,
                                                                params->max_iterations, params->enable_threshold, params->threshold,
                                                                capacity, d_msg, d_zcur, d_e, d_m, d_tot, d_z, d_s,
                                                                (uint32_t *)ctx->out_it.p, (uint8_t *)ctx->out_res.p);
        QLB_CUDA(cudaGetLastError());
        ++ctx->launches;
        std::vector<double> h_e(e_out ? cap * slots : 0), h_m(m_out ? cap * slots : 0);
        std::vector<int32_t> h_z(bits_out ? n : 0);
        if (e_out && cap)
            QLB_CUDA(cudaMemcpyAsync(h_e.data(), d_e, cap * slots * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (m_out && cap)
            QLB_CUDA(cudaMemcpyAsync(h_m.data(), d_m, cap * slots * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (l_out && cap)
            QLB_CUDA(cudaMemcpyAsync(l_out, d_tot, cap * n * 8, cudaMemcpyDeviceToHost, ctx->stream));
        if (z_out && cap)
            QLB_CUDA(cudaMemcpyAsync(z_out, d_z, cap * n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (s_out && cap)
            QLB_CUDA(cudaMemcpyAsync(s_out, d_s, cap * m * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (bits_out)
            QLB_CUDA(cudaMemcpyAsync(bits_out, d_zcur, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(iterations_out, ctx->out_it.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(result_out, ctx->out_res.p, 1, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        // slot snapshots -> the reference's jagged rows (plain re-indexing, no arithmetic)
        const size_t E = (size_t)L.e;
        for (size_t t = 0; t < cap; ++t)
        {
            if (e_out) // check_to_bit_msg[i][a]: bit-major, a-th arrival at bit i
            {
                size_t q = 0;
                for (size_t i = 0; i < n; ++i)
                    for (int a = 0; a < L.max_bit_w; ++a)
                    {
                        const uint32_t sl = L.bit_slots[(size_t)a * n + i];
                        if (sl != kNoSlot)
                            e_out[t * E + q++] = h_e[t * slots + sl];
                    }
            }
            if (m_out) // bit_to_check_msg[j][k]: check-major, CSR order
                for (size_t q = 0; q < E; ++q)
                    m_out[t * E + q] = h_m[t * slots + L.slot_of_edge[q]];
        }
        return QLB_OK;
    }

    // ---- test probe of the fp64 building blocks -----------------------------------------------------------------------------
    int qlb_test_f64_math(qlb_ctx *ctx, int op, int64_t n, const double *a, const double *b, double *out)
    {
        if (!ctx || n < 0 || op < 0 || op > 6 || (n > 0 && (!a || !out)) || (op == 6 && (n % 8 != 0 || !b)))
            return fail(QLB_ERR_INVALID, "qlb_test_f64_math: bad arguments");
        if (n == 0)
            return QLB_OK;
        QLB_CUDA(cudaSetDevice(ctx->device));
        const size_t bytes = (size_t)n * 8;
        QLB_CUDA(ctx->in_llr.reserve(2 * bytes));
        QLB_CUDA(ctx->scratch.reserve(bytes));
        double *d_a = static_cast<double *>(ctx->in_llr.p), *d_b = b ? d_a + n : nullptr, *d_o = static_cast<double *>(ctx->scratch.p);
        QLB_CUDA(cudaMemcpyAsync(d_a, a, bytes, cudaMemcpyHostToDevice, ctx->stream));
        if (b)
            QLB_CUDA(cudaMemcpyAsync(d_b, b, bytes, cudaMemcpyHostToDevice, ctx->stream));
        if (op == 6)
            QLB_CUDA(cudaMemsetAsync(d_o, 0, bytes, ctx->stream)); // the slots of a record beyond its W messages come back as 0
        if (op == 6)
            f64_rule_probe_kernel<<<(unsigned)((n / 8 + 255) / 256), 256, 0, ctx->stream>>>(n / 8, d_a, d_b, d_o);
        else
            f64_math_probe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(op, n, d_a, d_b, d_o);
        QLB_CUDA(cudaGetLastError());
        QLB_CUDA(cudaMemcpyAsync(out, d_o, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        return QLB_OK;
    }

    // ---- statistics all-reduce over the GPUs of this process (NCCL, loaded lazily) ---------------------------------------
    namespace
    {
        typedef void *nccl_comm_t;
        struct nccl_api
        {
            typedef int (*init_all_t)(nccl_comm_t *, int, const int *);
            typedef int (*allreduce_t)(const void *, void *, size_t, int, int, nccl_comm_t, cudaStream_t);
            typedef int (*group_t)(void);
            typedef const char *(*errstr_t)(int);
            void *lib = nullptr;
            init_all_t init_all = nullptr;
            allreduce_t allreduce = nullptr;
            group_t group_start = nullptr, group_end = nullptr;
            errstr_t errstr = nullptr;
            std::map<std::vector<int>, std::vector<nccl_comm_t>> comms;
            std::mutex mu;
            int fail_with(int rc, const char *what) const { return fail(QLB_ERR_NCCL, std::string(what) + ": " + (errstr ? errstr(rc) : "NCCL error")); }
        };
        nccl_api g_nccl;

        // The communicators of a device list (created once, kept for the life of the process). Caller holds g_nccl.mu.
        int nccl_comms_for(const std::vector<int> &devs, std::vector<nccl_comm_t> **out)
        {
            const int n_ctx = (int)devs.size();
            nccl_api &api = g_nccl;
            if (!api.lib)
            {
                api.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
                if (!api.lib)
                    return fail(QLB_ERR_NCCL, std::string("cannot load libnccl.so.2: ") + dlerror());
                api.init_all = (nccl_api::init_all_t)dlsym(api.lib, "ncclCommInitAll");
                api.allreduce = (nccl_api::allreduce_t)dlsym(api.lib, "ncclAllReduce");
                api.group_start = (nccl_api::group_t)dlsym(api.lib, "ncclGroupStart");
                api.group_end = (nccl_api::group_t)dlsym(api.lib, "ncclGroupEnd");
                api.errstr = (nccl_api::errstr_t)dlsym(api.lib, "ncclGetErrorString");
                if (!api.init_all || !api.allreduce || !api.group_start || !api.group_end)
                    return fail(QLB_ERR_NCCL, "libnccl.so.2 lacks the expected entry points");
            }
            auto it = api.comms.find(devs);
            if (it == api.comms.end())
            {
                std::vector<nccl_comm_t> comms(n_ctx, nullptr);
                int rc = api.init_all(comms.data(), n_ctx, devs.data());
                if (rc != 0)
                    return api.fail_with(rc, "ncclCommInitAll");
                // NCCL connects its channels lazily, inside the first collective (0.1 ... 0.9 s measured on 2 GPUs): run one tiny
                // all-reduce now, while the set-up is still off the sweep's critical path
                std::vector<void *> buf(n_ctx, nullptr);
                std::vector<cudaStream_t> str(n_ctx, nullptr);
                for (int g = 0; g < n_ctx; ++g)
                {
                    QLB_CUDA(cudaSetDevice(devs[g]));
                    QLB_CUDA(cudaMalloc(&buf[g], 64));
                    QLB_CUDA(cudaMemset(buf[g], 0, 64));
                    QLB_CUDA(cudaStreamCreateWithFlags(&str[g], cudaStreamNonBlocking));
                }
                rc = api.group_start();
                for (int g = 0; g < n_ctx && rc == 0; ++g)
                {
                    QLB_CUDA(cudaSetDevice(devs[g]));
                    rc = api.allreduce(buf[g], buf[g], 8, /*ncclUint64*/ 5, /*ncclSum*/ 0, comms[g], str[g]);
                }
                const int rc_end = api.group_end();
                for (int g = 0; g < n_ctx; ++g)
                {
                    QLB_CUDA(cudaSetDevice(devs[g]));
                    QLB_CUDA(cudaStreamSynchronize(str[g]));
                    cudaStreamDestroy(str[g]);
                    cudaFree(buf[g]);
                }
                if (rc != 0 || rc_end != 0)
                    return api.fail_with(rc != 0 ? rc : rc_end, "first ncclAllReduce");
                it = api.comms.emplace(devs, comms).first;
            }
            *out = &it->second;
            return QLB_OK;
        }
    }

    int qlb_stats_comm_prepare(const int32_t *devices, int n_devices)
    {
        if (!devices || n_devices < 1)
            return fail(QLB_ERR_INVALID, "qlb_stats_comm_prepare: bad arguments");
        std::lock_guard<std::mutex> lk(g_nccl.mu);
        std::vector<nccl_comm_t> *comms = nullptr;
        return nccl_comms_for(std::vector<int>(devices, devices + n_devices), &comms);
    }

    int qlb_stats_allreduce(qlb_ctx *const *ctxs, int n_ctx, uint64_t *const *vectors, size_t count)
    {
        if (!ctxs || !vectors || n_ctx < 1 || count == 0)
            return fail(QLB_ERR_INVALID, "qlb_stats_allreduce: bad arguments");
        nccl_api &api = g_nccl;
        std::lock_guard<std::mutex> lk(api.mu);
        std::vector<int> devs;
        for (int g = 0; g < n_ctx; ++g)
        {
            if (!ctxs[g] || !vectors[g])
                return fail(QLB_ERR_INVALID, "qlb_stats_allreduce: null context or vector");
            devs.push_back(ctxs[g]->device);
        }
        std::vector<nccl_comm_t> *comms = nullptr;
        if (const int rc0 = nccl_comms_for(devs, &comms))
            return rc0;
        auto nccl_fail = [&](int rc, const char *what) { return api.fail_with(rc, what); };
        const size_t bytes = count * sizeof(uint64_t);
        for (int g = 0; g < n_ctx; ++g)
        {
            QLB_CUDA(cudaSetDevice(ctxs[g]->device));
            QLB_CUDA(ctxs[g]->in_q.reserve(bytes));
            QLB_CUDA(cudaMemcpyAsync(ctxs[g]->in_q.p, vectors[g], bytes, cudaMemcpyHostToDevice, ctxs[g]->stream));
        }
        int rc = api.group_start();
        if (rc != 0)
            return nccl_fail(rc, "ncclGroupStart");
        for (int g = 0; g < n_ctx; ++g)
        {
            QLB_CUDA(cudaSetDevice(ctxs[g]->device));
            rc = api.allreduce(ctxs[g]->in_q.p, ctxs[g]->in_q.p, count, /*ncclUint64*/ 5, /*ncclSum*/ 0, (*comms)[g], ctxs[g]->stream);
            if (rc != 0)
            {
                api.group_end();
                return nccl_fail(rc, "ncclAllReduce");
            }
        }
        rc = api.group_end();
        if (rc != 0)
            return nccl_fail(rc, "ncclGroupEnd");
        for (int g = 0; g < n_ctx; ++g)
        {
            QLB_CUDA(cudaSetDevice(ctxs[g]->device));
            QLB_CUDA(cudaMemcpyAsync(vectors[g], ctxs[g]->in_q.p, bytes, cudaMemcpyDeviceToHost, ctxs[g]->stream));
            QLB_CUDA(cudaStreamSynchronize(ctxs[g]->stream));
        }
        return QLB_OK;
    }

    // ---- on-device key generation -----------------------------------------------------------------------------------------
    int qlb_generate_device(qlb_ctx *ctx, int32_t n_bits, int64_t n_frames, const uint64_t *d_seeds, uint64_t seed_offset, double qber,
                            uint32_t *d_alice_packed_out, uint32_t *d_bob_packed_out, double *exact_qber_out)
    {
        if (!ctx || n_bits < 1 || n_frames < 0)
            return fail(QLB_ERR_INVALID, "qlb_generate_device: null context, non-positive key length or negative frame count");
        if (!(qber >= 0. && qber < 1.))
            return fail(QLB_ERR_INVALID, "QBER must be: 0 <= QBER < 1");
        // floor(N * q) exactly as the reference forms it (src/array_and_matrix_operations.cpp:436)
        const size_t n_err = static_cast<size_t>(static_cast<size_t>(n_bits) * qber);
        if (exact_qber_out)
            *exact_qber_out = static_cast<double>(n_err) / static_cast<size_t>(n_bits);
        if (n_err == 0)
            return fail(QLB_ERR_KEY_TOO_SMALL, "Key size '" + std::to_string(n_bits) + "' is too small for QBER.");
        if (n_frames == 0)
            return QLB_OK;
        if (!d_seeds || !d_alice_packed_out || !d_bob_packed_out)
            return fail(QLB_ERR_INVALID, "qlb_generate_device: null device buffer");
        QLB_CUDA(cudaSetDevice(ctx->device));
        if (n_err > 0x7fffffffULL)
            return fail(QLB_ERR_UNSUPPORTED, "qlb_generate_device: more than 2^31 - 1 flipped positions per key");
        const int words = (n_bits + 31) / 32;
        const size_t pos_bytes = n_bits <= 65536 ? 2 : 4, state_bytes = n_err * pos_bytes; // per trial: the K-entry shuffle prefix
        // Trials do not cooperate, so CTAs are small (64 or 32 threads) and the SM packs as many as its shared memory holds (each
        // CTA also pays 1 KB of system shared memory); when not even one warp's prefixes fit they go to global memory.
        const size_t smem_budget = (size_t)ctx->smem_optin - 1024;
        int threads = 64;
        if (threads * state_bytes > smem_budget)
            threads = 32;
        const bool shared = threads * state_bytes <= smem_budget;
        if (!shared)
            threads = 128;
        const size_t smem = shared ? state_bytes * threads : 0;
        int64_t slice = n_frames;
        if (!shared)
        {
            slice = std::max<int64_t>(1, std::min<int64_t>(n_frames, (int64_t)((1ull << 30) / state_bytes))); // bound the scratch
            QLB_CUDA(ctx->gen_perm.reserve((size_t)slice * state_bytes));
        }
        auto launch = [&](auto kern, auto *state) -> int
        {
            QLB_CUDA(allow_full_dynamic_smem(ctx, kern));
            for (int64_t f0 = 0; f0 < n_frames; f0 += slice)
            {
                const int64_t nf = std::min(slice, n_frames - f0);
                kern<<<(unsigned)((nf + threads - 1) / threads), threads, smem, ctx->stream>>>(nf, n_bits, words, (int)n_err, d_seeds + f0, seed_offset, state,
                                                                                                 d_alice_packed_out + f0 * words, d_bob_packed_out + f0 * words);
                QLB_CUDA(cudaGetLastError());
            }
            return QLB_OK;
        };
        if (pos_bytes == 2)
            return shared ? launch(generate_keys_kernel<uint16_t, true>, (uint16_t *)nullptr) : launch(generate_keys_kernel<uint16_t, false>, (uint16_t *)ctx->gen_perm.p);
        return shared ? launch(generate_keys_kernel<uint32_t, true>, (uint32_t *)nullptr) : launch(generate_keys_kernel<uint32_t, false>, (uint32_t *)ctx->gen_perm.p);
    }

    int qlb_generate_batch_packed(qlb_ctx *ctx, int32_t n_bits, int64_t n_frames, const uint64_t *seeds, uint64_t seed_offset, double qber,
                                  uint32_t *alice_packed_out, uint32_t *bob_packed_out, double *exact_qber_out)
    {
        if (!ctx || n_bits < 1 || n_frames < 0 || (n_frames > 0 && (!seeds || !alice_packed_out || !bob_packed_out)))
            return fail(QLB_ERR_INVALID, "qlb_generate_batch_packed: bad arguments");
        QLB_CUDA(cudaSetDevice(ctx->device));
        const size_t key_bytes = (size_t)n_frames * ((n_bits + 31) / 32) * 4;
        QLB_CUDA(ctx->gen_seeds.reserve((size_t)n_frames * 8 + 8));
        QLB_CUDA(ctx->in_a.reserve(key_bytes + 4));
        QLB_CUDA(ctx->in_b.reserve(key_bytes + 4));
        if (n_frames)
            QLB_CUDA(cudaMemcpyAsync(ctx->gen_seeds.p, seeds, (size_t)n_frames * 8, cudaMemcpyHostToDevice, ctx->stream));
        int rc = qlb_generate_device(ctx, n_bits, n_frames, (const uint64_t *)ctx->gen_seeds.p, seed_offset, qber, (uint32_t *)ctx->in_a.p,
                                     (uint32_t *)ctx->in_b.p, exact_qber_out);
        if (rc || n_frames == 0)
            return rc;
        QLB_CUDA(cudaMemcpyAsync(alice_packed_out, ctx->in_a.p, key_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(bob_packed_out, ctx->in_b.p, key_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        return QLB_OK;
    }

    int qlb_run_trials(qlb_ctx *ctx, const qlb_code *code, const qlb_decode_params *params, int64_t n_frames, const uint64_t *seeds,
                       uint64_t seed_offset, double qber, uint32_t *iterations_out, uint8_t *result_out, double *exact_qber_out)
    {
        if (!ctx || !code || n_frames < 0 || (n_frames > 0 && (!seeds || !iterations_out || !result_out)))
            return fail(QLB_ERR_INVALID, "qlb_run_trials: bad arguments");
        int rc = check_params(params);
        if (rc)
            return rc;
        const CodeLayout &L = code->L;
        QLB_CUDA(cudaSetDevice(ctx->device));
        const size_t key_bytes = (size_t)n_frames * L.words_n * 4;
        QLB_CUDA(ctx->gen_seeds.reserve((size_t)n_frames * 8 + 8));
        QLB_CUDA(ctx->in_a.reserve(key_bytes + 4));
        QLB_CUDA(ctx->in_b.reserve(key_bytes + 4));
        QLB_CUDA(ctx->in_q.reserve((size_t)n_frames * 8 + 8));
        QLB_CUDA(ctx->out_it.reserve((size_t)n_frames * 4 + 4));
        QLB_CUDA(ctx->out_res.reserve((size_t)n_frames + 4));
        if (n_frames)
            QLB_CUDA(cudaMemcpyAsync(ctx->gen_seeds.p, seeds, (size_t)n_frames * 8, cudaMemcpyHostToDevice, ctx->stream));
        double exact = 0.;
        rc = qlb_generate_device(ctx, L.n, n_frames, (const uint64_t *)ctx->gen_seeds.p, seed_offset, qber, (uint32_t *)ctx->in_a.p,
                                 (uint32_t *)ctx->in_b.p, &exact);
        if (exact_qber_out)
            *exact_qber_out = exact;
        if (rc || n_frames == 0)
            return rc;
        // ln((1-q)/q) of the exact ratio, on the host in double as the reference forms it (src/qkd_ldpc_algorithm.cpp:400)
        ctx->host_logp.assign((size_t)n_frames, std::log((1. - exact) / exact));
        QLB_CUDA(cudaMemcpyAsync(ctx->in_q.p, ctx->host_logp.data(), (size_t)n_frames * 8, cudaMemcpyHostToDevice, ctx->stream));
        rc = qlb_reconcile_device(ctx, code, params, n_frames, (const uint32_t *)ctx->in_a.p, (const uint32_t *)ctx->in_b.p, (const double *)ctx->in_q.p,
                                  (uint32_t *)ctx->out_it.p, (uint8_t *)ctx->out_res.p, nullptr, nullptr);
        if (rc)
            return rc;
        QLB_CUDA(cudaMemcpyAsync(iterations_out, ctx->out_it.p, (size_t)n_frames * 4, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaMemcpyAsync(result_out, ctx->out_res.p, (size_t)n_frames, cudaMemcpyDeviceToHost, ctx->stream));
        QLB_CUDA(cudaStreamSynchronize(ctx->stream));
        return QLB_OK;
    }
}
