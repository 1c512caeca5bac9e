/* TEST INFRASTRUCTURE ONLY: replays the random stream of one key generation as the pinned restatement draws it
 * (orc_generate, oracle/restatement/sp_oracle.c) and reports where the shuffle's Lemire rejection loop draws again.
 *
 * A shuffle draw for the pair of positions (i, i+1) takes one value uniform on [0, (i+1)(i+2)) by Lemire's multiply-shift;
 * when the low product word falls below (2^64 - range) % range the draw is rejected and the next raw value is used
 * (libstdc++ 13.3 bits/uniform_int_dist.h:257-280). The chance per draw is below range / 2^64, so redraws only show at long
 * keys (about 4 trials in 1 000 at n = 10^6). Which trials redraw depends on the seed and n alone, not on the QBER: the
 * shuffle makes every draw whatever number of positions is flipped afterwards.
 * Build: cc -std=c11 -O2 -fPIC -shared, linked with sp_oracle.c for the PRNG.
 */
#include <stdint.h>

#include "../oracle/restatement/sp_oracle.h"

/* Returns the number of rejected draws of the shuffle of an n-bit key from `seed` (n * n < 2^64, where every step after the
 * first takes a pair of positions from one draw), or UINT64_MAX for a longer key. pos_out[k], k < cap, receives the first
 * position i of the pair whose draw was rejected for the k-th time. */
uint64_t gr_redraws(uint64_t seed, uint64_t n, uint64_t *pos_out, uint64_t cap)
{
    if (n > 1 && UINT64_MAX / n < n)
        return UINT64_MAX;
    orc_prng p;
    orc_prng_seed(&p, seed);
    /* Alice: one draw on [0, 2) per bit; (2^64 - 2) % 2 = 0, so these are never rejected. The single swap of an even n draws
     * on [0, 2) as well. */
    for (uint64_t i = 0; i < n; ++i)
        orc_prng_next(&p);
    uint64_t i = 1, count = 0;
    if (n > 1 && (n % 2) == 0) {
        orc_prng_next(&p);
        i = 2;
    }
    for (; n > 1 && i < n; i += 2) {
        const uint64_t range = (i + 1) * (i + 2);
        unsigned __int128 product = (unsigned __int128)orc_prng_next(&p) * range;
        if ((uint64_t)product < range) {
            const uint64_t threshold = (0 - range) % range;
            while ((uint64_t)product < threshold) {
                if (count < cap)
                    pos_out[count] = i;
                ++count;
                product = (unsigned __int128)orc_prng_next(&p) * range;
            }
        }
    }
    return count;
}
