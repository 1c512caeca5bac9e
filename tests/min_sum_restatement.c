/* TEST INFRASTRUCTURE ONLY: the CPU restatement of the fp32 normalized min-sum decoder (QLB_FLAG_F32_MIN_SUM).
 *
 * It follows the rule as include/qkd_ldpc_b200.h defines it, in plain C with one message array per direction and the
 * reference's positional routing (arrival counters, src/qkd_ldpc_algorithm.cpp:228-243, 300-311), as the pinned sum-product
 * restatement in oracle/restatement/ does. Key generation, trial seeds and the syndrome are that restatement's, linked in
 * unchanged. Every operation of the rule is exact or one IEEE fp32 rounding, so the GPU decoders must equal this code on
 * every frame. Build: cc -std=c11 -O2 -fPIC -shared -ffp-contract=off -fopenmp (no -ffast-math: subnormals and NaN matter).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../oracle/restatement/sp_oracle.h"

static uint32_t f2u(float f)
{
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
}
static float u2f(uint32_t u)
{
    float f;
    memcpy(&f, &u, 4);
    return f;
}

/* The decode from fp32 priors. lsb0[i]: bit 0 of bit i's first messages (Alice's bit, or 0). cap: the clamp, +inf when off. */
static orc_sp_result msr_decode(const orc_graph *g, const float *prior, const int32_t *lsb0, const int32_t *syndrome,
                                uint64_t max_it, float cap, float scale, int32_t *bits_out)
{
    const int32_t n = g->n, m = g->m, e = g->e;
    uint32_t *b2c = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)(e > 0 ? e : 1)); /* check-major words */
    float *c2b = (float *)malloc(sizeof(float) * (size_t)(e > 0 ? e : 1));          /* bit-major          */
    int32_t *arr_bit = (int32_t *)malloc(sizeof(int32_t) * (size_t)(n > 0 ? n : 1));
    int32_t *arr_chk = (int32_t *)malloc(sizeof(int32_t) * (size_t)(m > 0 ? m : 1));
    int32_t *dec_syn = (int32_t *)malloc(sizeof(int32_t) * (size_t)(m > 0 ? m : 1));
    orc_sp_result res;
    res.iterations_num = max_it;
    res.syndromes_match = 0;

    for (int32_t j = 0; j < m; ++j)
        for (int32_t p = g->row_ptr[j]; p < g->row_ptr[j + 1]; ++p) {
            const int32_t b = g->col_idx[p];
            b2c[p] = (f2u(prior[b]) & ~1u) | (uint32_t)(lsb0 ? lsb0[b] & 1 : 0);
        }

    for (uint64_t it = 0; it != max_it; ++it) {
        /* check pass: the minimum over the other edges, taken literally (no min1 / min2) */
        memset(arr_bit, 0, sizeof(int32_t) * (size_t)n);
        for (int32_t j = 0; j < m; ++j) {
            const int32_t lo = g->row_ptr[j], hi = g->row_ptr[j + 1];
            uint32_t x = syndrome[j] ? 0x80000000u : 0u;
            for (int32_t p = lo; p < hi; ++p)
                x ^= b2c[p];
            for (int32_t p = lo; p < hi; ++p) {
                uint32_t mu = 0x7F800000u; /* the empty minimum: +inf */
                int first = 1;
                for (int32_t q = lo; q < hi; ++q)
                    if (q != p) {
                        const uint32_t a = b2c[q] & 0x7FFFFFFFu;
                        if (first || a < mu)
                            mu = a;
                        first = 0;
                    }
                const float prod = scale * u2f(mu);
                const float mag = fminf(prod, cap);
                const int32_t b = g->col_idx[p];
                c2b[g->col_ptr[b] + arr_bit[b]++] = u2f(((x ^ b2c[p]) & 0x80000000u) | f2u(mag));
            }
        }

        /* bit pass: total from the prior in arrival order, hard decision, clamped extrinsic with the decision in bit 0 */
        memset(arr_chk, 0, sizeof(int32_t) * (size_t)m);
        for (int32_t i = 0; i < n; ++i) {
            float total = prior[i];
            for (int32_t p = g->col_ptr[i]; p < g->col_ptr[i + 1]; ++p)
                total = total + c2b[p];
            const int z = total <= 0.f;
            bits_out[i] = z;
            for (int32_t p = g->col_ptr[i]; p < g->col_ptr[i + 1]; ++p) {
                const int32_t c = g->row_idx[p];
                const float v = fminf(fmaxf(total - c2b[p], -cap), cap);
                b2c[g->row_ptr[c] + arr_chk[c]++] = (f2u(v) & ~1u) | (uint32_t)z;
            }
        }

        orc_syndrome(g, bits_out, dec_syn);
        if (orc_arrays_equal(syndrome, dec_syn, (size_t)m)) {
            res.iterations_num = it + 1;
            res.syndromes_match = 1;
            break;
        }
    }
    free(b2c); free(c2b); free(arr_bit); free(arr_chk); free(dec_syn);
    return res;
}

static float msr_cap(int enable_threshold, double thr) { return enable_threshold ? (float)thr : INFINITY; }

/* Sum-product entry: prior = (float)llr, a NaN entering as 0x7FFFFFFF. */
orc_sp_result msr_sum_product(const orc_graph *g, const double *llr, const int32_t *syndrome, uint64_t max_it, int enable_threshold,
                              double thr, float scale, int32_t *bits_out)
{
    const int32_t n = g->n;
    float *prior = (float *)malloc(sizeof(float) * (size_t)(n > 0 ? n : 1));
    for (int32_t i = 0; i < n; ++i)
        prior[i] = isnan(llr[i]) ? u2f(0x7FFFFFFFu) : (float)llr[i];
    const orc_sp_result r = msr_decode(g, prior, NULL, syndrome, max_it, msr_cap(enable_threshold, thr), scale, bits_out);
    free(prior);
    return r;
}

/* Reconcile entry: prior = +-(float)ln((1 - q) / q), Alice's syndrome, decode, key compare. */
orc_ldpc_result msr_qkd_ldpc(const orc_graph *g, const int32_t *alice, const int32_t *bob, double qber, uint64_t max_it,
                             int enable_threshold, double thr, float scale, int32_t *syndrome_out, int32_t *decoded_out)
{
    const int32_t n = g->n, m = g->m;
    int32_t *syn = syndrome_out ? syndrome_out : (int32_t *)malloc(sizeof(int32_t) * (size_t)(m > 0 ? m : 1));
    int32_t *dec = decoded_out ? decoded_out : (int32_t *)malloc(sizeof(int32_t) * (size_t)(n > 0 ? n : 1));
    float *prior = (float *)malloc(sizeof(float) * (size_t)(n > 0 ? n : 1));
    const float lp = (float)log((1. - qber) / qber);
    for (int32_t i = 0; i < n; ++i)
        prior[i] = bob[i] ? -lp : lp;
    orc_syndrome(g, alice, syn);
    orc_ldpc_result r;
    r.sp_res = msr_decode(g, prior, alice, syn, max_it, msr_cap(enable_threshold, thr), scale, dec);
    r.keys_match = orc_arrays_equal(alice, dec, (size_t)n);
    free(prior);
    if (!syndrome_out) free(syn);
    if (!decoded_out) free(dec);
    return r;
}

/* One trial per seed (keys from the reference's generator, reconciled at the exact QBER) on `threads` OpenMP threads;
 * out3[3k + {0, 1, 2}] = {iterations, syndromes_match, keys_match}; decoded_out (may be NULL): count * n bits.
 * Returns -1 when floor(n * qber) == 0. */
int msr_run_trials(const orc_graph *g, double qber, const uint64_t *seeds, uint64_t count, int threads, uint64_t max_it,
                   int enable_threshold, double thr, float scale, uint64_t *out3, int32_t *decoded_out)
{
    const size_t n = (size_t)g->n;
    int status = 0;
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads < 1 ? 1 : threads)
    for (int64_t k = 0; k < (int64_t)count; ++k) {
        int32_t *alice = (int32_t *)malloc(sizeof(int32_t) * (n ? n : 1));
        int32_t *bob = (int32_t *)malloc(sizeof(int32_t) * (n ? n : 1));
        const double exact = orc_generate(seeds[k], n, qber, alice, bob);
        if (exact == 0.) {
#pragma omp atomic write
            status = -1;
        } else {
            const orc_ldpc_result r = msr_qkd_ldpc(g, alice, bob, exact, max_it, enable_threshold, thr, scale, NULL,
                                                   decoded_out ? decoded_out + (size_t)k * n : NULL);
            out3[3 * k] = r.sp_res.iterations_num;
            out3[3 * k + 1] = (uint64_t)r.sp_res.syndromes_match;
            out3[3 * k + 2] = (uint64_t)r.keys_match;
        }
        free(alice);
        free(bob);
    }
    return status;
}
