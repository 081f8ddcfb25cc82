/*
 * me_oracle_ladder.c — temperature ladders (parallel tempering) on top of the scalar oracle.  TEST INFRASTRUCTURE ONLY.
 *
 * Compiled as one translation unit with oracle/me_oracle.c (included below), so that a ladder runs each rung through the
 * unchanged meo_run_group with the same Philox streams.  Nothing in the product links, loads or calls this file; the tests
 * compare the PT instantiation of the fused kernel (me_device.cuh, run_body / swap_round) against it chain by chain.
 *
 * Build: gcc -O2 -ffp-contract=off -fPIC -shared  (as me_oracle.c).
 */
#include "me_oracle.c"

/* ------------------------------------------------------------------ ladders
 * Stream definition shared with the CUDA kernels (me_device.cuh, swap_round): the R chains of one ladder are the global
 * chains chain0 .. chain0 + R - 1, rung r running at temps[r].  After the measure of every period whose counter n is a
 * multiple of swap_every, round k = n / swap_every pairs rungs (r, r + 1) with r = k (mod 2); the pair swaps iff
 * u <= exp((1/T_lo - 1/T_hi)(E_lo - E_hi)), u = (K + 1/2) 2^-52, K = y : x[31:12] of the Philox call with counter
 * (lo(chain0 + r), hi(chain0 + r), lo32(n), 0xFFFFFFFF).  A swap exchanges x and E (and the walker labels); sigma, means,
 * covariances, factors, observable means, NACC and STATUS stay with the rung. */
double meo_swap_uniform(uint64_t seed, uint64_t chain, int64_t n) {
    uint32_t r[4];
    meo_philox(seed, chain, (uint32_t)n, 0xFFFFFFFFu, r);
    uint64_t K = ((uint64_t)r[1] << 20) | (uint64_t)(r[0] >> 12);
    return ((double)K + 0.5) * (1.0 / 4503599627370496.0);
}

/* states: R consecutive state columns of `words` doubles; walker[R], swap_acc[R] (accepted swaps between rung r and r + 1)
 * and swap_att[R] (attempts of that pair) are in / out.  do_measure = 0: n_blocks x spm steps, no measure, no swap. */
int meo_run_ladder(const meo_config *c, int R, const double *temps, double *states, int64_t swap_every, int64_t n_blocks,
                   int64_t spm, int do_measure, int64_t *n_measure, uint64_t seed, uint64_t chain0, uint64_t step0,
                   int32_t *walker, uint32_t *swap_acc, uint32_t *swap_att) {
    meo_offsets o;
    const int d = c->n_r + 2 * c->n_c;
    meo_layout(c->n_r, c->n_c, &o);
    int64_t n = *n_measure;
    for (int64_t b = 0; b < n_blocks; b++) {
        int64_t n_after = n;
        for (int r = 0; r < R; r++) {
            meo_config cr = *c;
            cr.temp = temps[r];
            int64_t nr_ = n;
            int rc = meo_run_group(&cr, states + (size_t)r * o.WORDS, MEO_PHILOX, 1, spm, do_measure, &nr_, NULL, NULL,
                                   seed, chain0 + (uint64_t)r, step0 + (uint64_t)(b * spm), NULL, NULL, 0);
            if (rc) return rc;
            n_after = nr_;
        }
        n = n_after;
        if (!do_measure || swap_every <= 0 || n % swap_every != 0) continue;
        const int64_t k = n / swap_every;
        for (int lo = (int)(k & 1); lo + 1 < R; lo += 2) {
            double *a = states + (size_t)lo * o.WORDS, *h = states + (size_t)(lo + 1) * o.WORDS;
            const double delta = (1.0 / temps[lo] - 1.0 / temps[lo + 1]) * (a[o.E] - h[o.E]);
            swap_att[lo] += 1;
            if (meo_swap_uniform(seed, chain0 + (uint64_t)lo, n) <= exp(delta)) {
                for (int i = 0; i < d; i++) { double t = a[o.X + i]; a[o.X + i] = h[o.X + i]; h[o.X + i] = t; }
                double te = a[o.E]; a[o.E] = h[o.E]; h[o.E] = te;
                int32_t tw = walker[lo]; walker[lo] = walker[lo + 1]; walker[lo + 1] = tw;
                swap_acc[lo] += 1;
            }
        }
    }
    *n_measure = n;
    return 0;
}
