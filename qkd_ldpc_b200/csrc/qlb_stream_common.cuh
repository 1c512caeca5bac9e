// Shared pieces of the frame-interleaved "streaming" decoder (qlb_stream_split.cuh), fp32 and fp64: the kernels for codes whose
// messages do not fit in shared memory (BASELINE.json configs[3]: N = 100 000 ... 1 000 000) -- the HBM-bound design point
// of SURVEY.md 8d.
//
// Frames are decoded in GROUPS of G = 32 * VEC (128-bit accesses: VEC = 4 floats or 2 doubles). Messages are stored slot-major,
// frame-minor: msg[slot][G]. A WARP works on one node at a time and lane l owns frames VEC*l ... VEC*l+VEC-1 of the group, so
// whatever the Tanner graph looks like, every message access of the warp is one fully coalesced 512-byte row,
// and the graph indices are warp-uniform (one broadcast load per node, amortised over the G frames). Traffic per executed
// iteration is the algorithmic 16 B (fp32) / 32 B (fp64) per edge and frame (read + write in the check pass, read + write in the
// bit pass) plus < 3 % of indices and packed bits. Keys, decisions and syndromes are kept bit-transposed per group ([node][VEC]
// words, word j bit l = frame VEC*l + j) so a lane extracts its frames' bits with one shift; the transposes run once per group
// with __ballot_sync. fp32: node arithmetic, the decision-in-LSB trick and the convergence rule are those of the SM-resident
// kernel (qlb_resident_f32.cuh). fp64: the reference's arithmetic and order (MathF64 / MathF64Fused::check_fast, the bit rule of
// qlb_resident_f64.cuh); its messages have no spare mantissa bit, so a check's parity comes from the packed decisions of its
// bits (slot -> bit table + one warp-uniform word per bit and frame word). A converged frame is frozen (decisions and counters
// kept) while its group finishes.
#pragma once
#include "qlb_resident_f32.cuh"
#include "qlb_resident_f64.cuh"

namespace qlb
{

    // How a precision rides through the streaming kernels: the message type, the widest group (128-bit accesses), whether the
    // bit's hard decision travels in the mantissa LSB of its outgoing messages (fp32: the bar is statistical) or is read from
    // the packed decisions (fp64: outcome-exact).
    template <typename Rule_>
    struct StreamF32
    {
        typedef float real;
        typedef Rule_ Rule;
        static constexpr bool kLsbDecision = true;
        static constexpr int kVecWide = 4;
    };
    template <typename Math_>
    struct StreamF64
    {
        typedef double real;
        typedef Math_ Math;
        static constexpr bool kLsbDecision = false;
#ifndef QLB_STREAM64_VEC
#define QLB_STREAM64_VEC 2
#endif
        static constexpr int kVecWide = QLB_STREAM64_VEC;
    };

    template <typename Real, int VEC>
    struct VecIO;
    template <>
    struct VecIO<float, 4>
    {
        static __device__ __forceinline__ void load(const float *p, float (&v)[4])
        {
#ifdef QLB_STREAM_CS
            const float4 t = __ldcs(reinterpret_cast<const float4 *>(p));
#else
            const float4 t = *reinterpret_cast<const float4 *>(p);
#endif
            v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        }
        static __device__ __forceinline__ void store(float *p, const float (&v)[4])
        {
#ifdef QLB_STREAM_CS
            __stcs(reinterpret_cast<float4 *>(p), make_float4(v[0], v[1], v[2], v[3]));
#else
            *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
#endif
        }
    };
    template <>
    struct VecIO<double, 2>
    {
        static __device__ __forceinline__ void load(const double *p, double (&v)[2])
        {
            const double2 t = *reinterpret_cast<const double2 *>(p);
            v[0] = t.x; v[1] = t.y;
        }
        static __device__ __forceinline__ void store(double *p, const double (&v)[2]) { *reinterpret_cast<double2 *>(p) = make_double2(v[0], v[1]); }
    };
    template <typename Real>
    struct VecIO<Real, 1>
    {
        static __device__ __forceinline__ void load(const Real *p, Real (&v)[1]) { v[0] = *p; }
        static __device__ __forceinline__ void store(Real *p, const Real (&v)[1]) { *p = v[0]; }
    };

    // Software prefetch into L2: registers bound how many demand loads a warp can keep in flight (W rows of 512 B), which is
    // not enough to cover HBM latency at 16 warps per SM; prefetching the NEXT node's rows costs no registers and turns the
    // demand loads that follow into L2 hits.
    __device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

    // per-group scratch carve-up (bytes); G = 32 * VEC
    struct StreamCarve
    {
        size_t msg, bobT, aliceT, zT, synT, total;
    };
    __host__ __device__ inline StreamCarve stream_carve(int n, int m, int slots, int vec)
    {
        StreamCarve c{};
        const size_t G = 32 * (size_t)vec;
        size_t o = 0;
        c.msg = o; o += align_up((size_t)slots * G * 4, 256);
        c.bobT = o; o += align_up((size_t)n * vec * 4, 256);
        c.aliceT = o; o += align_up((size_t)n * vec * 4, 256);
        c.zT = o; o += align_up((size_t)n * vec * 4, 256);
        c.synT = o; o += align_up((size_t)m * vec * 4, 256);
        c.total = o;
        return c;
    }

    // One check of weight exactly W for the VEC frames of this lane.
    // row_stride: floats between the rows of consecutive slots (G, or B * G when B groups are interleaved slot by slot)
    template <typename Rule, int W, int VEC>
    __device__ __forceinline__ void stream_check(float *__restrict__ msg, const CodeDev &code, uint32_t p, int lane, uint32_t *__restrict__ synT,
                                                 typename Rule::Arg cap, bool first, uint32_t (&bad)[VEC], uint32_t row_stride)
    {
        float v[VEC][W];
        float *row[W];
#pragma unroll
        for (int k = 0; k < W; ++k)
        {
            QLB_CHECK_INDEX(code.base[k] + p, code.slots);
            QLB_CHECK_INDEX(p, code.cnt[k]);
            row[k] = msg + VEC * lane + (size_t)((code.base[k] + p) * row_stride); // 32-bit product (slots * row_stride < 2^32)
            float t[VEC];
            VecIO<float, VEC>::load(row[k], t);
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                v[j][k] = t[j];
        }
        uint32_t syn_words[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j)
            syn_words[j] = first ? 0u : synT[(size_t)p * VEC + j];
#pragma unroll
        for (int j = 0; j < VEC; ++j)
        {
            uint32_t xr = 0;
#pragma unroll
            for (int k = 0; k < W; ++k)
                xr ^= __float_as_uint(v[j][k]);
            uint32_t sb;
            if (first)
            {
                sb = xr & 1u; // Alice's bits ride in bit 0 during the first pass: their parity IS her syndrome bit
                const uint32_t word = __ballot_sync(0xffffffffu, sb != 0);
                if (lane == 0)
                    synT[(size_t)p * VEC + j] = word;
            }
            else
            {
                sb = (syn_words[j] >> lane) & 1u;
                bad[j] |= (xr ^ sb) & 1u;
            }
            xr ^= sb << 31;
            Rule::template apply<W>(v[j], xr, cap);
        }
#pragma unroll
        for (int k = 0; k < W; ++k)
        {
            float t[VEC];
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                t[j] = v[j][k];
            VecIO<float, VEC>::store(row[k], t);
        }
    }

    // fp64: one check of weight exactly W for the VEC frames of this lane, the reference's rule (Math::check_fast). bitsT: the
    // bit-transposed words the check's parity is formed from -- Alice's key in the first pass of a reconciliation (the parity IS
    // her syndrome bit, src/qkd_ldpc_algorithm.cpp:413-414), the decisions of the last bit pass afterwards (:277-298).
    template <typename Math, int W, int VEC>
    __device__ __forceinline__ void stream_check64(double *__restrict__ msg, const CodeDev &code, uint32_t p, int lane, uint32_t *__restrict__ synT,
                                                   const uint32_t *__restrict__ bitsT, double thr_eff, bool want_inf, bool first, uint32_t (&bad)[VEC],
                                                   uint32_t row_stride)
    {
        double v[VEC][W];
        double *row[W];
        uint32_t par[VEC], synw[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j)
        {
            par[j] = 0;
            synw[j] = first ? 0u : synT[(size_t)p * VEC + j];
        }
#pragma unroll
        for (int k = 0; k < W; ++k)
        {
            QLB_CHECK_INDEX(code.base[k] + p, code.slots);
            QLB_CHECK_INDEX(p, code.cnt[k]);
            row[k] = msg + VEC * lane + (size_t)((code.base[k] + p) * row_stride); // 32-bit product (slots * row_stride < 2^32)
            double t[VEC];
            VecIO<double, VEC>::load(row[k], t);
            const uint32_t bit = code.col_of_slot32[code.base[k] + p];
            QLB_CHECK_INDEX(bit, code.n);
#pragma unroll
            for (int j = 0; j < VEC; ++j)
            {
                v[j][k] = t[j];
                par[j] ^= bitsT[(size_t)bit * VEC + j]; // warp-uniform
            }
        }
#pragma unroll
        for (int j = 0; j < VEC; ++j)
        {
            if (first)
            {
                synw[j] = par[j];
                if (lane == 0)
                    synT[(size_t)p * VEC + j] = par[j];
            }
            else
                bad[j] |= ((par[j] ^ synw[j]) >> lane) & 1u; // parity of the decisions != target: this frame's check is unsatisfied
            const bool syn = ((synw[j] >> lane) & 1u) != 0;
            Math::template check_fast<W>(v[j], syn, thr_eff, want_inf);
        }
#pragma unroll
        for (int k = 0; k < W; ++k)
        {
            double t[VEC];
#pragma unroll
            for (int j = 0; j < VEC; ++j)
                t[j] = v[j][k];
            VecIO<double, VEC>::store(row[k], t);
        }
    }

    // 32 x 32 bit transposes between frame-major packed words and the per-group node-major layout.
    // in:  word `wd` of frames f0 + VEC*l + j (lane l)      out: T[(32*wd + b) * VEC + j] = word whose bit l is bit b of that frame's word
    template <int VEC>
    __device__ __forceinline__ void transpose_in(const uint32_t *__restrict__ frames, long long f0, long long n_frames, int words, int n, uint32_t *__restrict__ T)
    {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
        for (int item = warp; item < words * VEC; item += nwarps)
        {
            const int wd = item / VEC, j = item % VEC;
            const long long f = f0 + (long long)VEC * lane + j;
            const uint32_t x = f < n_frames ? frames[f * words + wd] : 0u;
            uint32_t mine = 0;
#pragma unroll
            for (int b = 0; b < 32; ++b)
            {
                const uint32_t col = __ballot_sync(0xffffffffu, (x >> b) & 1u);
                if (lane == b)
                    mine = col;
            }
            const int bit = 32 * wd + lane;
            if (bit < n)
                T[(size_t)bit * VEC + j] = mine;
        }
    }
    // fmap_g (optional): frame index of each of the group's 32 * VEC columns (0xFFFFFFFF = none) instead of f0 + column;
    // keep[j] (with fmap_g): only the columns whose bit is set in keep[j] are written
    template <int VEC>
    __device__ __forceinline__ void transpose_out(const uint32_t *__restrict__ T, long long f0, long long n_frames, int words, int n, uint32_t *__restrict__ frames,
                                                  const uint32_t *__restrict__ fmap_g = nullptr, const uint32_t *keep = nullptr)
    {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
        for (int item = warp; item < words * VEC; item += nwarps)
        {
            const int wd = item / VEC, j = item % VEC;
            const int bit = 32 * wd + lane;
            const uint32_t x = bit < n ? T[(size_t)bit * VEC + j] : 0u;
            uint32_t mine = 0;
#pragma unroll
            for (int l = 0; l < 32; ++l)
            {
                const uint32_t row = __ballot_sync(0xffffffffu, (x >> l) & 1u);
                if (lane == l)
                    mine = row;
            }
            long long f = f0 + (long long)VEC * lane + j;
            if (fmap_g)
            {
                const uint32_t fm = fmap_g[VEC * lane + j];
                f = (fm == 0xFFFFFFFFu || (keep && !((keep[j] >> lane) & 1u))) ? n_frames : (long long)fm;
            }
            if (f < n_frames)
                frames[f * words + wd] = mine;
        }
    }

}
