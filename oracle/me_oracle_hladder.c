/*
 * me_oracle_hladder.c — Hamiltonian ladders (per-rung functor constants, H-REMD) on top of the ladder oracle.  TEST
 * INFRASTRUCTURE ONLY.
 *
 * Compiled as one translation unit with oracle/me_oracle_ladder.c (and through it oracle/me_oracle.c), so that every rung
 * runs through the unchanged meo_run_group with its own meo_config and the swaps use the same meo_swap_uniform.  Nothing in
 * the product links, loads or calls this file; the tests compare the HX instantiation of the fused kernel (me_device.cuh,
 * run_body / swap_round) against it chain by chain.
 *
 * Build: gcc -O2 -ffp-contract=off -fPIC -shared  (as me_oracle.c).
 */
#include "me_oracle_ladder.c"

/* ------------------------------------------------------------------ Hamiltonian ladders
 * Stream definition shared with the CUDA kernels (me_device.cuh, swap_round, HX instantiation): rung r has temperature T_r
 * and constant vector k_r[0..K), 1 <= K <= 16 (here: cfgs[r], whose temp, consts and wall are the rung's); every step
 * evaluates the functor (eval and reject) with k_r of the chain's rung.  The swap uniform, the pairing schedule and what
 * moves or stays are those of meo_run_ladder.  With a the lower and b the upper rung of a pair and E_a(x) rung a's functor
 * with k_a at x, the pair swaps iff u <= exp(-D) with
 *     D = (1/T_a) (E_a(x_b) - E_a(x_a)) + (1/T_b) (E_b(x_a) - E_b(x_b)),
 * which both lanes evaluate from the same four energies in this operand order, so they agree bit for bit.  The pair does
 * not swap if either cross-configuration is walled (reject(x_b; k_a) or reject(x_a; k_b)).  A NaN cross-energy refuses the
 * swap and sets ME_STATUS_ENERGY_NAN on the lane that computed it (a lane that pairs and whose own wall passes its
 * partner's configuration).  After a swap a chain holds its own rung's energy of the new configuration, E_a(x_b), not its
 * partner's E.  Temperatures: finite and > 0 in any order with swaps (equal ones are the usual case), >= 0 without. */
static void hladder_cross(const meo_config *c, const double *x, double *st, const meo_offsets *o, double *e, int *wall) {
    *wall = reject_eval(c, x);
    *e = energy_eval(c, x);
    if (!*wall && *e != *e) st[o->STATUS] = (double)((int)st[o->STATUS] | 4);
}

int meo_run_hladder(const meo_config *cfgs, int R, double *states, int64_t swap_every, int64_t n_blocks, int64_t spm,
                    int do_measure, int64_t *n_measure, uint64_t seed, uint64_t chain0, uint64_t step0, int32_t *walker,
                    uint32_t *swap_acc, uint32_t *swap_att) {
    meo_offsets o;
    const int d = cfgs[0].n_r + 2 * cfgs[0].n_c;
    meo_layout(cfgs[0].n_r, cfgs[0].n_c, &o);
    int64_t n = *n_measure;
    for (int64_t b = 0; b < n_blocks; b++) {
        int64_t n_after = n;
        for (int r = 0; r < R; r++) {
            int64_t nr_ = n;
            int rc = meo_run_group(&cfgs[r], states + (size_t)r * o.WORDS, MEO_PHILOX, 1, spm, do_measure, &nr_, NULL,
                                   NULL, seed, chain0 + (uint64_t)r, step0 + (uint64_t)(b * spm), NULL, NULL, 0);
            if (rc) return rc;
            n_after = nr_;
        }
        n = n_after;
        if (!do_measure || swap_every <= 0 || n % swap_every != 0) continue;
        const int64_t k = n / swap_every;
        for (int lo = (int)(k & 1); lo + 1 < R; lo += 2) {
            const meo_config *ca = &cfgs[lo], *cb = &cfgs[lo + 1];
            double *a = states + (size_t)lo * o.WORDS, *h = states + (size_t)(lo + 1) * o.WORDS;
            double xa[MEO_MAX_D], xb[MEO_MAX_D], e_a_xb, e_b_xa;
            int wall_a, wall_b;
            for (int i = 0; i < d; i++) { xa[i] = a[o.X + i]; xb[i] = h[o.X + i]; }
            hladder_cross(ca, xb, a, &o, &e_a_xb, &wall_a);          /* rung a at x_b, computed by a's lane */
            hladder_cross(cb, xa, h, &o, &e_b_xa, &wall_b);          /* rung b at x_a, computed by b's lane */
            const double delta = (1.0 / ca->temp) * (e_a_xb - a[o.E]) + (1.0 / cb->temp) * (e_b_xa - h[o.E]);
            swap_att[lo] += 1;
            if (!wall_a && !wall_b && meo_swap_uniform(seed, chain0 + (uint64_t)lo, n) <= exp(-delta)) {
                for (int i = 0; i < d; i++) { a[o.X + i] = xb[i]; h[o.X + i] = xa[i]; }
                a[o.E] = e_a_xb;
                h[o.E] = e_b_xa;
                int32_t tw = walker[lo]; walker[lo] = walker[lo + 1]; walker[lo + 1] = tw;
                swap_acc[lo] += 1;
            }
        }
    }
    *n_measure = n;
    return 0;
}
