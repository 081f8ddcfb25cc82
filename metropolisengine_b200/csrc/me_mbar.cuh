/* me_mbar.cuh — one MBAR pass (Shirts & Chodera, J. Chem. Phys. 129, 124105, 2008) over recorded time-series rows
 * (DESIGN §3 "MBAR over recorded ladder rows").
 *
 * Given the rungs' reduced free energies f[R], every sample x_n (one recorded row of one chain) contributes
 *     L_n  = ln sum_k N_k exp(f_k - u_k(x_n))                 (k over the R rungs, max-shifted log-sum-exp)
 *     w_ns = exp(f_s - u_s(x_n) - L_n)                        (s over the S output states; f = 0 for the targets)
 * with u_s(x) = E(x; k_s) / T_s re-evaluated from the stored x columns (the stored E column is not read) and u_s = +inf
 * where the functor's wall rejects x under k_s.  A pass returns the fixed-order sums
 *     sum_n L_n,  s_s = sum_n w_ns,  G_st = sum_n w_ns w_nt,  sum_n w_ns [x, x^2, E_s, E_s^2]  (the latter optional)
 * and the counts of samples with a NaN energy or a non-finite L_n, and of samples whose target weight exceeds 1e140
 * (a target without overlap); such samples enter no sum.
 *
 * One thread per sample, chain-fastest, so the loads of each x column coalesce as the rows were written.  The energies
 * and weights of a warp's 32 samples are staged column-wise in shared memory (z[row][lane], one column per lane), and all
 * sums over samples are products with the 32 samples as the K dimension on the FP64 tensor cores (mma.m8n8k4, as
 * pool_mma_update): tile (a, b) accumulates Z_a Z_b^T of two 8-row blocks of z.  Row blocks of z:
 *     [0, nb)            w_s           (rows s < S; the rest stay 0)
 *     nb                 ONE           (row 0 = 1, rows 1..7 = 0: a product with it is a plain sum over the samples)
 *     [nb+1, 2nb+1)      E_s, then w_s E_s
 *     [2nb+1, 3nb+1)     w_s E_s^2                            (observables only)
 *     [3nb+1, 3nb+1+nx)  x_0..x_{D-1}, x_0^2..x_{D-1}^2      (observables only)
 * Each warp adds its tile products to its own rows of shared memory after every 32 samples; at the end the CTA sums its
 * warps in order and writes one partial row [sum L, n_nan, n_overflow, tiles[n_tiles][8][8]], which the host reduces
 * with the fixed-order k_pool_reduce.  Every sum therefore has a fixed order for a given (samples, grid, block): a pass
 * is bit-identical from run to run on one device.
 *
 * mbar_hist_body (k_mbar_hist, me_mbar_hist_pass) is the histogram pass of free-energy profiles over the same samples
 * and weights, mbar_cov_body (k_mbar_cov, me_mbar_cov_pass) the covariance pass of expectation uncertainties; mbar_sample
 * is the per-sample evaluation all three passes share. */
#ifndef ME_MBAR_CUH
#define ME_MBAR_CUH

#include "me_device.cuh"

#define ME_MBAR_LD 36                /* doubles per staged row: 32 samples + 4 of padding (fragment reads: two wavefronts) */
#define ME_MBAR_HEAD 64              /* f[32], then [ME_MBAR_MAX_WARPS][4] per-warp scalar sums */
#define ME_MBAR_MAX_WARPS 4
#define ME_MBAR_OVERFLOW 1e140       /* w^2 summed over 10^10 samples stays finite */

namespace me {

template <bool WIDE> struct MbarMask { typedef unsigned T; };
template <> struct MbarMask<true> { typedef unsigned long long T; };

/* One sample's share of a pass, common to k_mbar and k_mbar_hist: load x_n (sample n < hi: row n / ld, chain n % ld;
 * x = 0 and live = false past hi), evaluate the wall and energy of every output state (wall first, as in the step) into
 * z[E0 + s][lane], then L_n into l and the weights w_ns into z[W0 + s][lane].  bad: a NaN energy or a non-finite L_n;
 * ovf: some weight exceeds ME_MBAR_OVERFLOW.  States s < R are the rungs.  HIST: S = R + 1 and the last state is the
 * histogram pass's target, whose temperature and constants are t_inv_temp / t_consts (so R = 32 still fits). */
template <class C, bool HIST>
__device__ __forceinline__ void mbar_sample(const MeMbarParams &q, const double *fs, double (*z)[ME_MBAR_LD], int W0,
                                            int E0, int lane, long long n, long long hi, double *x, bool &live,
                                            bool &bad, bool &ovf, double &l) {
    using L = Lay<C::NR, C::NC>;
    using Energy = typename C::Energy;
    using Mask = typename MbarMask<HIST>::T;
    constexpr int D = L::D, NR = L::NR, NC = L::NC;
    const int S = q.n_states, R = q.n_rungs;
    live = n < hi;
    if (live) {
        const long long i = n / q.ld, ch = n - i * q.ld;
        const double *xp = q.ts + (q.row0 + i * q.stride) * (long long)q.ts_cols * q.ld + ch;
#pragma unroll
        for (int d = 0; d < D; d++) x[d] = xp[(long long)d * q.ld];
    } else {
#pragma unroll
        for (int d = 0; d < D; d++) x[d] = 0.0;
    }
    /* energies of every output state (wall first, as in the step), staged in this lane's column */
    bad = false;
    Mask walled = 0u;
    if (live) {
        for (int s = 0; s < S; s++) {
            const double *k = (HIST && s == R) ? q.t_consts : q.consts[s];
            const bool w = q.use_reject && Energy::reject(x, x + NR, x + NR + NC, k);
            const double e = w ? 0.0 : Energy::eval(x, x + NR, x + NR + NC, k);
            bad = bad || e != e;
            walled |= (Mask)w << s;
            z[E0 + s][lane] = e;
        }
    }
    /* L_n = ln N + m + ln sum_k exp(a_k - m),  a_k = f_k - u_k */
    double m = -__longlong_as_double(0x7ff0000000000000LL);   /* -inf */
    if (live && !bad)
        for (int k = 0; k < R; k++)
            if (!((walled >> k) & 1u)) m = fmax(m, fs[k] - z[E0 + k][lane] * q.inv_temp[k]);
    double sum = 0.0;
    if (live && !bad)
        for (int k = 0; k < R; k++) {
            const double ek = ((walled >> k) & 1u) ? 0.0 : exp(fs[k] - z[E0 + k][lane] * q.inv_temp[k] - m);
            z[W0 + k][lane] = ek;
            sum += ek;
        }
    l = q.log_n + m + log(sum);
    if (live && !bad && !(fabs(l) <= 1.79e308)) bad = true;   /* every rung walled, or an infinite energy */
    ovf = false;
    if (live && !bad) {
        const double sc = 1.0 / (q.n_per_state * sum);
        for (int s = 0; s < S; s++) {
            double w;
            if (s < R) w = z[W0 + s][lane] * sc;
            else w = ((walled >> s) & 1u) ? 0.0 : exp(-z[E0 + s][lane] * (HIST ? q.t_inv_temp : q.inv_temp[s]) - l);
            if (!(w <= ME_MBAR_OVERFLOW)) ovf = true;
            z[W0 + s][lane] = w;
        }
    }
}

template <class C>
__device__ __forceinline__ void mbar_pass_body(const MeMbarParams &q) {
    constexpr int D = Lay<C::NR, C::NC>::D;
    extern __shared__ __align__(16) double me_mbar_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int r8 = lane >> 2, k4 = lane & 3;
    const int S = q.n_states, R = q.n_rungs, nb = q.nb;
    double *fs = me_mbar_smem, *scal = me_mbar_smem + 32;
    double *acc = me_mbar_smem + ME_MBAR_HEAD + (long long)warp * q.n_tiles * 64;
    double(*z)[ME_MBAR_LD] =
        reinterpret_cast<double(*)[ME_MBAR_LD]>(me_mbar_smem + ME_MBAR_HEAD + (long long)nw * q.n_tiles * 64) +
        (long long)warp * q.z_rows;
    const int W0 = 0, ONE = 8 * nb, E0 = 8 * (nb + 1), E20 = 8 * (2 * nb + 1), X0 = 8 * (3 * nb + 1);
    const bool obs = q.nx > 0;

    for (int i = threadIdx.x; i < 32; i += blockDim.x) fs[i] = i < R ? q.f[i] : 0.0;
    for (int i = lane; i < q.n_tiles * 64; i += 32) acc[i] = 0.0;
    for (int r = 0; r < q.z_rows; r++) z[r][lane] = r == ONE ? 1.0 : 0.0;
    __syncthreads();

    const long long per = (q.n_samples + gridDim.x - 1) / gridDim.x;
    const long long lo = (long long)blockIdx.x * per;
    const long long hi = lo + per < q.n_samples ? lo + per : q.n_samples;
    double sum_l = 0.0, n_bad = 0.0, n_ovf = 0.0;
    for (long long base = lo + 32LL * warp; base < hi; base += 32LL * nw) {   /* warp-uniform trip count */
        const long long n = base + lane;
        double x[D];
        bool live, bad, ovf;
        double l;
        mbar_sample<C, false>(q, fs, z, W0, E0, lane, n, hi, x, live, bad, ovf, l);
        live = live && !bad && !ovf;
        if (live) {
            sum_l += l;
            for (int s = 0; s < S; s++) {
                const double w = z[W0 + s][lane], e = z[E0 + s][lane];
                z[E0 + s][lane] = w * e;
                if (obs) z[E20 + s][lane] = (w * e) * e;
            }
            if (obs) {
#pragma unroll
                for (int d = 0; d < D; d++) {
                    z[X0 + d][lane] = x[d];
                    z[X0 + D + d][lane] = x[d] * x[d];
                }
            }
        } else {
            n_bad += bad ? 1.0 : 0.0;
            n_ovf += (!bad && ovf) ? 1.0 : 0.0;
            for (int s = 0; s < S; s++) {
                z[W0 + s][lane] = 0.0;
                z[E0 + s][lane] = 0.0;
                if (obs) z[E20 + s][lane] = 0.0;
            }
            if (obs)
                for (int d = 0; d < 2 * D; d++) z[X0 + d][lane] = 0.0;
        }
        __syncwarp();
        for (int t = 0; t < q.n_tiles; t++) {
            const int ra = 8 * q.tile_a[t] + r8, rb = 8 * q.tile_b[t] + r8;
            double c0 = 0.0, c1 = 0.0;
#pragma unroll
            for (int kk = 0; kk < 8; kk++) dmma_8x8x4(c0, c1, z[ra][4 * kk + k4], z[rb][4 * kk + k4]);
            acc[t * 64 + 2 * lane] += c0;            /* C[r8][2 k4 + i] at r8 * 8 + 2 k4 + i: tiles are row-major */
            acc[t * 64 + 2 * lane + 1] += c1;
        }
        __syncwarp();
    }
    sum_l = warp_sum(sum_l);
    n_bad = warp_sum(n_bad);
    n_ovf = warp_sum(n_ovf);
    if (lane == 0) {
        scal[4 * warp] = sum_l;
        scal[4 * warp + 1] = n_bad;
        scal[4 * warp + 2] = n_ovf;
    }
    __syncthreads();
    double *row = q.partial + (long long)blockIdx.x * q.rw;
    for (int w = threadIdx.x; w < q.rw; w += blockDim.x) {
        double v = 0.0;
        if (w < 3) {
            for (int j = 0; j < nw; j++) v += scal[4 * j + w];
        } else {
            const double *a0 = me_mbar_smem + ME_MBAR_HEAD + (w - 3);
            for (int j = 0; j < nw; j++) v += a0[(long long)j * q.n_tiles * 64];
        }
        row[w] = v;
    }
}

/* Histogram pass (me_mbar_hist_pass, DESIGN §3 "MBAR free-energy profiles"): the same samples and weights as
 * mbar_pass_body with the R rungs and one target t (S = R + 1), and per sample the bin of one or two coordinates.  Per
 * bin b the pass sums h_b = sum w_nt, q_b = sum w_nt^2 and c_bk = sum w_nt w_nk; out-of-range samples go to w_out and
 * n_out.  Each warp owns a histogram of hw = B (R + 2) doubles in shared memory.  After every 32 samples,
 * __match_any_sync on the bin groups the lanes; the lowest lane of each group sums the group's staged weights in lane
 * order and adds them to the warp's histogram, so no two lanes ever write one bin.  At the end the CTA sums its warps
 * in order into one partial row [n_nan, n_overflow, w_out, n_out, hist[hw]] (the layout of the sums vector), and
 * k_pool_reduce sums the rows in fixed order: a pass is bit-identical from run to run on one device.
 *
 * The coordinate, its modulus and the bin index use explicit round-to-nearest intrinsics, so FMA contraction in the
 * fast build cannot move a sample across a bin edge: i = floor((c - lo) * inv_w), in range iff lo <= c < hi (NaN is
 * not), i = n rounds to n - 1. */
template <class C>
__device__ __forceinline__ void mbar_hist_body(const MeMbarParams &q) {
    using L = Lay<C::NR, C::NC>;
    constexpr int D = L::D, NR = L::NR, NC = L::NC;
    extern __shared__ __align__(16) double me_mbar_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int R = q.n_rungs, S = R + 1, J = R + 2;
    double *fs = me_mbar_smem, *scal = me_mbar_smem + 32;
    double *hist = me_mbar_smem + ME_MBAR_HEAD + (long long)warp * q.hw;
    double(*z)[ME_MBAR_LD] =
        reinterpret_cast<double(*)[ME_MBAR_LD]>(me_mbar_smem + ME_MBAR_HEAD + (long long)nw * q.hw) +
        (long long)warp * q.z_rows;                       /* rows [0, S): w_s (w_t at row R); rows [S, 2S): E_s */

    for (int i = threadIdx.x; i < 32; i += blockDim.x) fs[i] = i < R ? q.f[i] : 0.0;
    for (int i = lane; i < q.hw; i += 32) hist[i] = 0.0;
    __syncthreads();

    const long long per = (q.n_samples + gridDim.x - 1) / gridDim.x;
    const long long lo = (long long)blockIdx.x * per;
    const long long hi = lo + per < q.n_samples ? lo + per : q.n_samples;
    double n_bad = 0.0, n_ovf = 0.0, w_out = 0.0, n_out = 0.0;
    for (long long base = lo + 32LL * warp; base < hi; base += 32LL * nw) {   /* warp-uniform trip count */
        const long long n = base + lane;
        double x[D];
        bool live, bad, ovf;
        double l;
        mbar_sample<C, true>(q, fs, z, 0, S, lane, n, hi, x, live, bad, ovf, l);
        live = live && !bad && !ovf;
        int b = -2;                                       /* -2: no sample, -1: out of range, else the bin */
        if (live) {
            b = 0;
            for (int a = 0; a < q.n_axes; a++) {
                const int j = q.axis_index[a];
                double c = 0.0;
                if (q.axis_kind[a] == 0) {
#pragma unroll
                    for (int d = 0; d < D; d++)
                        if (d == j) c = x[d];
                } else {
                    double re = 0.0, im = 0.0;
#pragma unroll
                    for (int d = 0; d < NC; d++)
                        if (d == j) re = x[NR + d], im = x[NR + NC + d];
                    c = __dsqrt_rn(__dadd_rn(__dmul_rn(re, re), __dmul_rn(im, im)));
                }
                if (!(c >= q.axis_lo[a] && c < q.axis_hi[a])) {
                    b = -1;
                    break;
                }
                int i = (int)floor(__dmul_rn(__dsub_rn(c, q.axis_lo[a]), q.axis_inv_w[a]));
                if (i >= q.n_bins[a]) i = q.n_bins[a] - 1;
                b = b * q.n_bins[a] + i;
            }
            if (b < 0) {
                w_out += z[R][lane];
                n_out += 1.0;
            }
        } else {
            n_bad += bad ? 1.0 : 0.0;
            n_ovf += (!bad && ovf) ? 1.0 : 0.0;
        }
        __syncwarp();
        const unsigned grp = __match_any_sync(0xffffffffu, b);
        if (b >= 0 && lane == __ffs(grp) - 1) {
            double *hb = hist + (long long)b * J;
            for (int k = 0; k < J; k++) {                 /* [h, q, c_0 .. c_{R-1}] */
                double v = 0.0;
                for (unsigned mk = grp; mk; mk &= mk - 1) {
                    const int ln = __ffs(mk) - 1;
                    const double wt = z[R][ln];
                    v += k == 0 ? wt : wt * (k == 1 ? wt : z[k - 2][ln]);
                }
                hb[k] += v;
            }
        }
        __syncwarp();
    }
    n_bad = warp_sum(n_bad);
    n_ovf = warp_sum(n_ovf);
    w_out = warp_sum(w_out);
    n_out = warp_sum(n_out);
    if (lane == 0) {
        scal[4 * warp] = n_bad;
        scal[4 * warp + 1] = n_ovf;
        scal[4 * warp + 2] = w_out;
        scal[4 * warp + 3] = n_out;
    }
    __syncthreads();
    double *row = q.partial + (long long)blockIdx.x * q.rw;
    for (int w = threadIdx.x; w < q.rw; w += blockDim.x) {
        double v = 0.0;
        if (w < 4) {
            for (int j = 0; j < nw; j++) v += scal[4 * j + w];
        } else {
            const double *a0 = me_mbar_smem + ME_MBAR_HEAD + (w - 4);
            for (int j = 0; j < nw; j++) v += a0[(long long)j * q.hw];
        }
        row[w] = v;
    }
}

/* Covariance pass (me_mbar_cov_pass, DESIGN §3 "Uncertainties of reweighted expectations"): the samples and weights of
 * mbar_pass_body with the same R rungs and targets, and for each covered state s = cov_first + c (c < n_cov) the centred
 * observables a~ = a_s - c_s, a_s = [x_0..x_{D-1}, x_0^2..x_{D-1}^2, E_s, E_s^2] (m = 2D + 2).  Row blocks of z:
 *     [0, nb)                 w_s           (rows s < S; the rest stay 0)
 *     nb                      ONE
 *     [nb+1, 2nb+1)           E_s           (mbar_sample's staging only)
 *     2nb+1 + c mb + [0, mb)  w_s a~        (rows a < m of covered state c; mb = ceil(m / 8) blocks, padding rows 0)
 * The host's tile list (me_api.cu, mbar_cov_layout) pairs each covered state's blocks with ONE (o_a), with every w block
 * (C_ak against the rungs and the self column C_a* = sum w_s^2 a~) and with each other (Q_ab, b <= a).  Tiles accumulate
 * per warp in shared memory as in mbar_pass_body; the CTA writes [n_nan, n_overflow, tiles[n_tiles][8][8]] and
 * k_pool_reduce sums the rows in fixed order, so a pass is bit-identical from run to run on one device.
 * Shared memory: 512 + 512 n_tiles + 288 z_rows bytes for one warp, at most the 227 KB opt-in (the host refuses larger
 * ranges).  One covered state always fits: at D = 32 and S = 32 it takes 90 tiles and 144 rows, 88 KB. */
template <class C>
__device__ __forceinline__ void mbar_cov_body(const MeMbarParams &q) {
    constexpr int D = Lay<C::NR, C::NC>::D, M = 2 * D + 2;
    extern __shared__ __align__(16) double me_mbar_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int r8 = lane >> 2, k4 = lane & 3;
    const int S = q.n_states, R = q.n_rungs, nb = q.nb, mb = q.cov_mb;
    double *fs = me_mbar_smem, *scal = me_mbar_smem + 32;
    double *acc = me_mbar_smem + ME_MBAR_HEAD + (long long)warp * q.n_tiles * 64;
    double(*z)[ME_MBAR_LD] =
        reinterpret_cast<double(*)[ME_MBAR_LD]>(me_mbar_smem + ME_MBAR_HEAD + (long long)nw * q.n_tiles * 64) +
        (long long)warp * q.z_rows;
    const int W0 = 0, ONE = 8 * nb, E0 = 8 * (nb + 1), V0 = 8 * (2 * nb + 1);

    for (int i = threadIdx.x; i < 32; i += blockDim.x) fs[i] = i < R ? q.f[i] : 0.0;
    for (int i = lane; i < q.n_tiles * 64; i += 32) acc[i] = 0.0;
    for (int r = 0; r < q.z_rows; r++) z[r][lane] = r == ONE ? 1.0 : 0.0;
    __syncthreads();

    const long long per = (q.n_samples + gridDim.x - 1) / gridDim.x;
    const long long lo = (long long)blockIdx.x * per;
    const long long hi = lo + per < q.n_samples ? lo + per : q.n_samples;
    double n_bad = 0.0, n_ovf = 0.0;
    for (long long base = lo + 32LL * warp; base < hi; base += 32LL * nw) {   /* warp-uniform trip count */
        const long long n = base + lane;
        double x[D];
        bool live, bad, ovf;
        double l;
        mbar_sample<C, false>(q, fs, z, W0, E0, lane, n, hi, x, live, bad, ovf, l);
        live = live && !bad && !ovf;
        if (live) {
            for (int c = 0; c < q.n_cov; c++) {
                const int s = q.cov_first + c;
                const double w = z[W0 + s][lane], e = z[E0 + s][lane];
                const double *ce = q.centers + (long long)c * M;
                double *v = &z[V0 + 8 * mb * c][0] + lane;
#pragma unroll
                for (int d = 0; d < D; d++) {
                    v[d * ME_MBAR_LD] = w * (x[d] - ce[d]);
                    v[(D + d) * ME_MBAR_LD] = w * (x[d] * x[d] - ce[D + d]);
                }
                v[2 * D * ME_MBAR_LD] = w * (e - ce[2 * D]);
                v[(2 * D + 1) * ME_MBAR_LD] = w * (e * e - ce[2 * D + 1]);
            }
        } else {
            n_bad += bad ? 1.0 : 0.0;
            n_ovf += (!bad && ovf) ? 1.0 : 0.0;
            for (int s = 0; s < S; s++) z[W0 + s][lane] = 0.0;
            for (int c = 0; c < q.n_cov; c++)
                for (int a = 0; a < M; a++) z[V0 + 8 * mb * c + a][lane] = 0.0;
        }
        __syncwarp();
        for (int t = 0; t < q.n_tiles; t++) {
            const int ra = 8 * q.cov_tile_a[t] + r8, rb = 8 * q.cov_tile_b[t] + r8;
            double c0 = 0.0, c1 = 0.0;
#pragma unroll
            for (int kk = 0; kk < 8; kk++) dmma_8x8x4(c0, c1, z[ra][4 * kk + k4], z[rb][4 * kk + k4]);
            acc[t * 64 + 2 * lane] += c0;
            acc[t * 64 + 2 * lane + 1] += c1;
        }
        __syncwarp();
    }
    n_bad = warp_sum(n_bad);
    n_ovf = warp_sum(n_ovf);
    if (lane == 0) {
        scal[4 * warp] = n_bad;
        scal[4 * warp + 1] = n_ovf;
    }
    __syncthreads();
    double *row = q.partial + (long long)blockIdx.x * q.rw;
    for (int w = threadIdx.x; w < q.rw; w += blockDim.x) {
        double v = 0.0;
        if (w < 2) {
            for (int j = 0; j < nw; j++) v += scal[4 * j + w];
        } else {
            const double *a0 = me_mbar_smem + ME_MBAR_HEAD + (w - 2);
            for (int j = 0; j < nw; j++) v += a0[(long long)j * q.n_tiles * 64];
        }
        row[w] = v;
    }
}

}  // namespace me

#endif
