// On-device key / error generator, bit-exact with the reference's run_trial inputs (SURVEY.md 8f-1).
//
// The reference draws, per trial, from one xoshiro256++ stream seeded through SplitMix64 (third-party module
// Reputeless/Xoshiro-cpp v1.1; reference src/simulation.cpp:163):
//   Alice  : generate_random_bit_array (src/array_and_matrix_operations.cpp:424-431) -- uniform_int_distribution<int>(0,1)
//            per bit: libstdc++ 13.3 maps a 64-bit draw to [0, 2) by Lemire's multiply-shift, i.e. the draw's top bit;
//   Bob    : introduce_errors (:434-460) -- std::shuffle of 0..N-1 (libstdc++ 13.3 bits/stl_algo.h:3742-3806: one optional
//            single swap, then two swap positions per draw from uniform_int_distribution{0, (i+1)(i+2)-1}, with the
//            rejection loop of bits/uniform_int_dist.h:257-280), the first floor(N*q) entries are flipped.
// One thread replays one trial's stream sequentially (the stream and the Fisher-Yates chain are inherently serial); thousands
// of trials run side by side.
//
// Only the first K = floor(N*q) entries of the shuffled order are ever used, and the forward Fisher-Yates never moves a
// value from a position >= K back below K: step i swaps a[i] (still holding i) with a[j], j <= i. So
//   steps i <  K : a plain swap inside the K-entry prefix                      a[i] = a[j], a[j] = i
//   steps i >= K : only "a[j] = i when j < K" matters -- the value that leaves the prefix can never return, and what later
//                  steps do among the positions >= K is invisible
// and the per-trial state is K entries (<= 2.2 KB at q = 0.11, N = 10240) instead of N: it lives in SHARED memory (global
// memory only for keys so long that not even one warp's prefixes fit), every draw of the reference's stream is still made
// (Lemire rejection loop and pair draws included), and phase 2 is write-only. The first version kept a full N-entry permutation per
// trial in global memory and was bound by its random 2-byte read-modify-writes (2.2 M trials/s).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace qlb
{
    struct Xoshiro256pp
    {
        uint64_t s0, s1, s2, s3;
        __host__ __device__ __forceinline__ explicit Xoshiro256pp(uint64_t seed)
        {
            uint64_t x = seed;
            s0 = splitmix(x);
            s1 = splitmix(x);
            s2 = splitmix(x);
            s3 = splitmix(x);
        }
        static __host__ __device__ __forceinline__ uint64_t splitmix(uint64_t &x)
        {
            uint64_t z = (x += 0x9e3779b97f4a7c15ULL);
            z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL;
            z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL;
            return z ^ (z >> 31);
        }
        static __host__ __device__ __forceinline__ uint64_t rotl(uint64_t v, int k) { return (v << k) | (v >> (64 - k)); }
        __host__ __device__ __forceinline__ uint64_t next()
        {
            const uint64_t out = rotl(s0 + s3, 23) + s0;
            const uint64_t t = s1 << 17;
            s2 ^= s0;
            s3 ^= s1;
            s1 ^= s2;
            s0 ^= s3;
            s2 ^= t;
            s3 = rotl(s3, 45);
            return out;
        }
        // uniform on [0, range): Lemire's method as libstdc++ 13.3 implements it (bits/uniform_int_dist.h:257-280)
        __device__ __forceinline__ uint64_t below(uint64_t range)
        {
            uint64_t g = next();
            uint64_t lo = g * range, hi = __umul64hi(g, range);
            if (lo < range)
            {
                const uint64_t threshold = (0 - range) % range;
                while (lo < threshold)
                {
                    g = next();
                    lo = g * range;
                    hi = __umul64hi(g, range);
                }
            }
            return hi;
        }
    };

    // State: K = n_err entries of PosT per trial -- shared memory (kShared; dynamic, blockDim.x * n_err entries, trial-major) or
    // `state_global` ([n_frames][n_err]). n_err = floor(n * q) >= 1, computed by the host in double as the reference does.
    template <typename PosT, bool kShared>
    __global__ void __launch_bounds__(256) generate_keys_kernel(long long n_frames, int n, int words, int n_err, const uint64_t *__restrict__ seeds,
                                                                uint64_t seed_offset, PosT *__restrict__ state_global, uint32_t *__restrict__ alice_out,
                                                                uint32_t *__restrict__ bob_out)
    {
        extern __shared__ __align__(16) unsigned char gen_smem[];
        const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
        if (f >= n_frames)
            return;
        Xoshiro256pp rng(seeds[f] + seed_offset);
        uint32_t *alice = alice_out + f * words, *bob = bob_out + f * words;

        // Alice: bit i = top bit of draw i; Bob starts as a copy. Four words per store when the rows are 16-byte aligned.
        if ((words & 3) == 0 && n == words * 32)
        {
            for (int w = 0; w < words; w += 4)
            {
                uint32_t v[4];
#pragma unroll
                for (int q = 0; q < 4; ++q)
                {
                    uint32_t word = 0;
#pragma unroll 8
                    for (int b = 0; b < 32; ++b)
                        word |= (uint32_t)(rng.next() >> 63) << b;
                    v[q] = word;
                }
                const uint4 t = make_uint4(v[0], v[1], v[2], v[3]);
                *reinterpret_cast<uint4 *>(alice + w) = t;
                *reinterpret_cast<uint4 *>(bob + w) = t;
            }
        }
        else
            for (int w = 0; w < words; ++w)
            {
                uint32_t word = 0;
                const int lim = min(32, n - w * 32);
                for (int b = 0; b < lim; ++b)
                    word |= (uint32_t)(rng.next() >> 63) << b;
                alice[w] = word;
                bob[w] = word;
            }

        // std::shuffle of 0..n-1, restricted to the prefix that is used (see the header comment)
        const int K = n_err;
        PosT *a = kShared ? reinterpret_cast<PosT *>(gen_smem) + (size_t)threadIdx.x * K : state_global + (size_t)f * K;
        a[0] = 0;
        auto step = [&](int pos, uint64_t j)
        {
            if (pos < K) // swap(a[pos], a[j]) with a[pos] == pos still untouched
            {
                if ((int)j == pos)
                    a[pos] = (PosT)pos;
                else
                {
                    a[pos] = a[j];
                    a[j] = (PosT)pos;
                }
            }
            else if (j < (uint64_t)K)
                a[j] = (PosT)pos;
        };
        if (n > 1)
        {
            int i = 1;
            if ((n & 1) == 0)
            {
                step(1, rng.below(2));
                i = 2;
            }
            for (; i < n; i += 2)
            {
                const uint64_t swap_range = (uint64_t)i + 1, b1 = swap_range + 1;
                const uint64_t x = rng.below(swap_range * b1);
                uint64_t j0, j1;
                if (swap_range * b1 <= 0xffffffffULL)
                {
                    j0 = (uint32_t)x / (uint32_t)b1;
                    j1 = (uint32_t)x % (uint32_t)b1;
                }
                else
                {
                    j0 = x / b1;
                    j1 = x % b1;
                }
                step(i, j0);
                step(i + 1, j1);
            }
        }
        // flip the first floor(n*q) positions of the shuffled order (distinct positions: the XORs commute). The reductions are
        // fire-and-forget (no value returns to the thread) and ordered after this thread's own stores to the same words.
        for (int k = 0; k < K; ++k)
        {
            const uint32_t pos = (uint32_t)a[k];
            atomicXor(&bob[pos >> 5], 1u << (pos & 31));
        }
    }
}
