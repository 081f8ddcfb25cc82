/* me_device.cuh — device side of the fused Metropolis hot path (sm_100a).
 *
 * One thread owns one chain; the chain's parameters, energy, sampling width and proposal factors live in
 * registers for the whole launch, which runs  n_blocks x (spm steps [+ one measure])  without touching HBM except
 * for the time-series rows.  This is the B200 counterpart of the reference's user loop
 *     for ...: for ...: engine.step_all()         (metropolis_engine.py:241-259 / 225-239 / 209-223)
 *              engine.measure()                   (metropolis_engine.py:342-427)
 * (README.md:39-44, demo/toymodel_xypotentialwell.py:39-44).
 *
 * The same text is compiled three ways: ahead of time for the named workloads (me_aot_fast.cu with FMA
 * contraction, me_aot_strict.cu with -fmad=false and the reference's operation order for draw-injected parity),
 * and at run time by NVRTC for user energy functors / shapes that were not instantiated ahead of time.
 * Therefore: no #include of anything but the sibling headers (handed to NVRTC as in-memory includes),
 * built-in types only.
 *
 * State layout (chain-minor, `state[word*ld + chain]`), D = NR + 2 NC, parameter order [real, Re c, Im c]
 * (the reference's embedding order, metropolis_engine.py:288):
 *   X D | E 1 | SIG 2 | MEAN D | COVR NR(NR+1)/2 | COVC NC^2 | OBSM 2NR+NC | FACR NR(NR+1)/2 | FACC NC^2 | NACC | STATUS
 * Hermitian packing: strictly-lower pairs p=i(i-1)/2+j at [2p]=Re,[2p+1]=Im, then NC real diagonal entries.
 */
#ifndef ME_DEVICE_CUH
#define ME_DEVICE_CUH

#include "me_params.h"
#include "me_math.cuh"

#define ME_MAX_BLOCK 256
#ifndef ME_PAIR_BIG
#define ME_PAIR_BIG 0          /* shapes with D > 4: 1 = process the steps in pairs too (see run_body) */
#endif
#ifndef ME_BIG_LOOKAHEAD
#define ME_BIG_LOOKAHEAD 0     /* shapes with D > 4: 1 = generate the draws of step s+1 during step s (costs D+2 doubles of
                                  registers).  Measured on the 3r+4c shape, 262,144 chains: pairs + look-ahead 1.51e10,
                                  single steps + look-ahead 1.55e10, single steps without look-ahead 1.70e10 chain-steps/s
                                  (ceil(D/2) independent generator calls per step already give the warp its ILP; the
                                  27 KB pair-unrolled loop stalls on instruction fetch) */
#endif
#define ME_FULL 0xffffffffu
#define ME_SEG_MAX_D 4         /* shapes up to this D = n_real + 2 n_complex support work-queue time segmentation */
#define ME_MAX_POOLW 600

namespace me {

template <bool SMEM> struct TabSelect { typedef LogTabGlobal type; };
template <> struct TabSelect<true> { typedef LogTabShared type; };

template <int NR_, int NC_>
struct Lay {
    static constexpr int NR = NR_, NC = NC_;
    static constexpr int D = NR + 2 * NC;
    static constexpr int NCOVR = NR * (NR + 1) / 2;
    static constexpr int NCOVC = NC * NC;
    static constexpr int NOBS = 2 * NR + NC;
    static constexpr int X = 0;
    static constexpr int E = D;
    static constexpr int SIG = D + 1;
    static constexpr int MEAN = D + 3;
    static constexpr int COVR = MEAN + D;
    static constexpr int COVC = COVR + NCOVR;
    static constexpr int OBSM = COVC + NCOVC;
    static constexpr int FACR = OBSM + NOBS;
    static constexpr int FACC = FACR + NCOVR;
    static constexpr int NACC = FACC + NCOVC;
    static constexpr int STATUS = NACC + 1;
    static constexpr int WORDS = STATUS + 1;
    static constexpr int NSIGCOL = (NR > 0 && NC > 0) ? 2 : 1;  /* mixed engines record both group widths */
    static constexpr int TSCOLS = D + 1 + NSIGCOL;             /* x[D], E, sigma(s) */
    static constexpr int POOLW = D + D * (D + 1) / 2 + NOBS;   /* sum(x-s), sum (x-s)(x-s)^T lower, sum obs */
    static constexpr int KIND = (NR > 0 && NC > 0) ? 0 : (NR > 0 ? 1 : 2);   /* 0 mixed, 1 all-real, 2 all-complex */
    static constexpr int SIGIDX = (KIND == 2) ? 1 : 0;         /* which width step_all adapts (ME:46,56) */
};

__host__ __device__ constexpr int nz(int n) { return n > 0 ? n : 1; }
__device__ __forceinline__ constexpr int herm_lo(int i, int j) { return 2 * (i * (i - 1) / 2 + j); }
__device__ __forceinline__ constexpr int tri(int i, int j) { return i * (i + 1) / 2 + j; }

/* ------------------------------------------------------------------------------------------ Philox4x32-7 */
struct U4 { unsigned x, y, z, w; };

/* Philox4x32 with ME_PHILOX_ROUNDS = 7 rounds: the smallest round count Random123 (Salmon et al., SC'11, table 2) reports
 * as passing the full BigCrush battery ("Crush-resistant"); 10 is that library's default with a safety margin.  The
 * generator's IMAD.WIDE rounds contend with the FP64 pipe (profiles/r01_microbench_issue_mix.txt), so three rounds less
 * are six quarter-rate instructions less per Gaussian pair.  The C oracle uses the same count and is pinned against the
 * Random123 known-answer vectors for both 7 and 10 rounds.
 * rk: the round-key pairs (k0 + r*0x9E3779B9, k1 + r*0xBB67AE85), precomputed on the host: they are the same
 * for every chain and step, and as kernel parameters they are constant-bank operands of the XORs. */
#define ME_PHILOX_ROUNDS 7
__device__ __forceinline__ U4 philox4x32(unsigned c0, unsigned c1, unsigned c2, unsigned c3,
                                         const unsigned *rk) {
#pragma unroll
    for (int r = 0; r < ME_PHILOX_ROUNDS; r++) {
        const unsigned k0 = rk[2 * r], k1 = rk[2 * r + 1];
        const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;   /* one IMAD.WIDE each */
        const unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
        const unsigned n0 = (unsigned)(p1 >> 32) ^ c1 ^ k0;
        const unsigned n2 = (unsigned)(p0 >> 32) ^ c3 ^ k1;
        c0 = n0; c1 = (unsigned)p1; c2 = n2; c3 = (unsigned)p0;
    }
    U4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3;
    return o;
}

/* Stream definition (identical in oracle/me_oracle.c): per step and chain, Philox call q = 0..ceil(D/2)-1 with
 * counter (chain_lo, chain_hi, step, q), key = seed, output words (x, y, z, w):
 *   radius uniform  u1 = (K + 1/2) 2^-52 in (0,1),  K = y : x[31:12]  (52 bits);   angle t = z 2^-31 in [0,2);
 *   z_{2q} = sqrt(-2 ln u1) cos(pi t), z_{2q+1} = sqrt(-2 ln u1) sin(pi t);
 *   accept uniform  u = (A + 1/2) 2^-44 in (0,1),  A = w_0 : x_0[11:0]  (44 bits of call 0 the normals do not use).
 *   The throughput build never exponentiates: u <= exp(-dE/T)  <=>  dE <= -T ln u, and the threshold -T ln u does not
 *   depend on the chain's state, so it is computed in the draw stage (one table-driven log, off the critical path)
 *   and the Metropolis test of the state-dependent chain is a single comparison.
 * One Philox call per Gaussian pair, nothing else.  Both uniforms are assembled as the mantissa of a double in
 * [1,2) and shifted down with ONE exact subtraction (no integer->double conversion, no magic-number pairs). */
struct Spare { unsigned w0, x0; };

/* One-parameter shapes (D = 1; the README configuration) would throw away the second normal of every Box-Muller pair and
 * most of the call's spare bits, so there ONE Philox call serves TWO consecutive steps: steps 2P and 2P + 1 use the call with
 * counter (chain_lo, chain_hi, P, 0):
 *   radius uniform  u1 = (K + 1/2) 2^-52,  K = y : 0x80000  (the 32 bits of y; the low 20 mantissa bits are the constant mid-point);
 *   angle t = z 2^-31;   step 2P proposes with sqrt(-2 ln u1) cos(pi t),  step 2P + 1 with sqrt(-2 ln u1) sin(pi t);
 *   accept uniform  u = (A + 1/2) 2^-44,  A = w : 0x800 for step 2P,  A = x : 0x800 for step 2P + 1  (32 random bits each).
 * The two normals of a pair are independent, and so are the four output words, so the chain sees the same law as before;
 * |z| <= 6.8 and u >= 2^-33 (both ends beyond anything 10^12 steps resolve).  The step loop computes the pair at the even
 * step and carries the second half to the odd one: -15 % instructions per step at D = 1. */
template <class L> struct ShareCall { static constexpr bool value = L::D == 1; };
/* (The same idea for the one spare normal of larger odd shapes — the last pair of the 3r+4c shape shared by two steps — was
 * measured and lost: 10.0 against 9.8 ms per pass; the conditional pair costs the unrolled draw stage more overlap than half
 * a call saves.) */
__device__ __forceinline__ U4 share_radius_bits(const U4 &r) { U4 o = r; o.x = 0x80000000u; return o; }
__device__ __forceinline__ Spare share_spare(const U4 &r, unsigned step) {
    Spare sp;
    sp.w0 = (step & 1u) ? r.x : r.w;
    sp.x0 = 0x800u;
    return sp;
}

struct Rng {
    unsigned c0, c1;
    const unsigned *rk;
    __device__ __forceinline__ Rng(const MeParams &p, unsigned long long gchain)
        : c0((unsigned)gchain), c1((unsigned)(gchain >> 32)), rk(p.rk) {}
    __device__ __forceinline__ U4 bits(unsigned step, unsigned slot) const {
        return philox4x32(c0, c1, step, slot, rk);
    }
    template <bool STRICT, class Tab = LogTabGlobal>
    __device__ __forceinline__ static void box_muller(const U4 &r, const MathTables &T, double &z0, double &z1,
                                                      const double unit = ME_C_UNIT, const double angle = ME_C_ANGLE_TAB,
                                                      const Tab logtab = Tab{nullptr}) {
        const double d = __hiloint2double((int)(0x3ff00000u | (r.y >> 12)), (int)((r.y << 20) | (r.x >> 12)));
        const double u1 = d - unit;                                                     /* d - (1 - 2^-53), exact */
        double s, c, rad;
        if (STRICT) {           /* parity build: libdevice log / sqrt and the full-accuracy polynomial sin/cos */
            rad = sqrt(-2.0 * log(u1));
            sincospi_bits(r.z, s, c);
        } else {                /* throughput build: table-driven log and sin/cos, accuracy budget 1e-10 */
            rad = sqrt_pos(neg2log_unit(u1, logtab));
            sincospi_tab(r.z, s, c, logtab, angle);
        }
        z0 = rad * c;
        z1 = rad * s;
    }
    __device__ __forceinline__ static void keep_spare(const U4 &r, int q, Spare &sp) {
        if (q == 0) { sp.w0 = r.w; sp.x0 = r.x; }
    }
    __device__ __forceinline__ static double accept_uniform(const Spare &sp) {
        const double d = __hiloint2double((int)(0x3ff00000u | (sp.w0 >> 12)),
                                          (int)((sp.w0 << 20) | ((sp.x0 & 0xfffu) << 8) | 0x80u));
        return d - 1.0;
    }
    /* -T ln u = (T/2) (-2 ln u) >= 0; T == 0 gives 0: only moves with dE <= 0 are accepted (ME:331-332) */
    template <class Tab>
    __device__ __forceinline__ static double accept_threshold(const Spare &sp, const Tab &logtab, double half_temp) {
        return half_temp * neg2log_unit(accept_uniform(sp), logtab);
    }
    /* A window [lo, hi] around the threshold -T ln u, from FP32 arithmetic only: the FP64 pipe is what bounds the step
     * kernel and the exact threshold costs it 12 instructions per step, while almost every decision is far from the
     * threshold.  u 2^32 lies in [w0, w0 + 1); with w0 >= 2^18 the estimate ln u ~ ln((w0 + 1/2) 2^-32) is off by at most
     * 1.9e-6, MUFU.LG2 by 2^-22 relative of |log2 u| <= 14 (7.7e-6 ln2 in ln u at worst over the full range), the
     * conversion and the FP32 FMA / adds by < 4e-6 T: |estimate - (-T ln u)| < 1.1e-5 T; the window half-width is 4e-5 T.
     * The caller decides: dE <= lo accepts, dE > hi rejects, anything else — in between (probability ~2e-5 per step) or
     * NaN — takes the exact test dE <= -T ln u.
     * Invariant: every decision equals the exact test, so the chains are those of an exact FP64 comparison, bit for bit.
     *   1e-30 <= T <= 1e30 (t_ln2 = T ln2, t_band = 4e-5 T, both rounded once on the host): |thr| <= 9.8 T, so the
     *   rounding of lo / hi (relative 2^-24, absolute 2^-150 below the normal range) adds < 6e-7 T + 2^-150 to the
     *   1.1e-5 T of the estimate, well inside the half-width.  A NaN dE fails both comparisons.
     *   w0 < 2^18 (probability 2^-14): [-2^-149, inf), i.e. only dE <= -2^-149 (< 0 <= -T ln u) is decided here.
     *   T == 0 (t_ln2 = 0, t_band = 2^-149): [-2^-149, 2^-149], so a dE of magnitude below 2^-149 is exact.
     *   Any other T (t_band = inf): (-inf, inf), every decision is exact. */
    __device__ __forceinline__ static void accept_window(unsigned w0, float t_ln2, float t_band, float &lo, float &hi) {
        float lg;
        const float f = __uint2float_rn(w0) + 0.5f;
        asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(f));
        const float thr = (32.0f - lg) * t_ln2;                   /* T ln2 (32 - log2(w0 + 1/2)) */
        const bool wide = w0 < 0x40000u;
        lo = wide ? -0x1p-149f : thr - t_band;
        hi = wide ? __int_as_float(0x7f800000) : thr + t_band;
    }
};

/* The temperature of a chain on a ladder (run_body's PT instantiation): its rung's T and FP32 window constants, loaded once
 * per launch.  Functions that take `const LaneTemp *lt` use the launch's scalar temperature (MeParams::temp, t_ln2, t_band)
 * when it is null, which is what every other instantiation passes. */
struct LaneTemp {
    double temp;
    float t_ln2, t_band;
};

/* Ladder mode of run_body: none (one temperature and one constant vector for every chain), a temperature ladder (PT), or
 * a Hamiltonian ladder (HX: every rung also has its own functor constants, and a swap evaluates each rung's energy at its
 * partner's configuration). */
enum LadderMode { LADDER_NONE = 0, LADDER_TEMP = 1, LADDER_HAM = 2 };

/* ------------------------------------------------------------------------------------------ per-chain registers */
template <class L>
struct Chain {
    double x[L::D];
    double e;
    double sig[2];
    double facr[nz(L::NCOVR)];
    double facc[nz(L::NCOVC)];
    double nacc;
    unsigned nacc_new;      /* acceptances of this launch (integer add in the step loop; folded into nacc on store) */
    int status;
};

template <class L>
struct Stats {
    double mean[L::D];
    double covr[nz(L::NCOVR)];
    double covc[nz(L::NCOVC)];
    double obsm[L::NOBS];
};

/* State loads bypass L1 (__ldcg): consecutive time segments of one chain group run as different CTAs, possibly on
 * different SMs, and hand the state over through global memory (see run_body). */
template <class L>
__device__ __forceinline__ void load_chain(Chain<L> &c, const double *st, long long ld, long long ch) {
#pragma unroll
    for (int i = 0; i < L::D; i++) c.x[i] = __ldcg(st + (long long)(L::X + i) * ld + ch);
    c.e = __ldcg(st + (long long)L::E * ld + ch);
    c.sig[0] = __ldcg(st + (long long)L::SIG * ld + ch);
    c.sig[1] = __ldcg(st + (long long)(L::SIG + 1) * ld + ch);
#pragma unroll
    for (int i = 0; i < L::NCOVR; i++) c.facr[i] = __ldcg(st + (long long)(L::FACR + i) * ld + ch);
#pragma unroll
    for (int i = 0; i < L::NCOVC; i++) c.facc[i] = __ldcg(st + (long long)(L::FACC + i) * ld + ch);
    c.nacc = __ldcg(st + (long long)L::NACC * ld + ch);
    c.nacc_new = 0u;
    c.status = (int)__ldcg(st + (long long)L::STATUS * ld + ch);
}

template <class L>
__device__ __forceinline__ void store_chain(const Chain<L> &c, double *st, long long ld, long long ch) {
#pragma unroll
    for (int i = 0; i < L::D; i++) st[(long long)(L::X + i) * ld + ch] = c.x[i];
    st[(long long)L::E * ld + ch] = c.e;
    st[(long long)L::SIG * ld + ch] = c.sig[0];
    st[(long long)(L::SIG + 1) * ld + ch] = c.sig[1];
#pragma unroll
    for (int i = 0; i < L::NCOVR; i++) st[(long long)(L::FACR + i) * ld + ch] = c.facr[i];
#pragma unroll
    for (int i = 0; i < L::NCOVC; i++) st[(long long)(L::FACC + i) * ld + ch] = c.facc[i];
    st[(long long)L::NACC * ld + ch] = c.nacc + (double)c.nacc_new;
    st[(long long)L::STATUS * ld + ch] = (double)c.status;
}

template <class L>
__device__ __forceinline__ void load_stats(Stats<L> &s, const double *st, long long ld, long long ch) {
#pragma unroll
    for (int i = 0; i < L::D; i++) s.mean[i] = __ldcg(st + (long long)(L::MEAN + i) * ld + ch);
#pragma unroll
    for (int i = 0; i < L::NCOVR; i++) s.covr[i] = __ldcg(st + (long long)(L::COVR + i) * ld + ch);
#pragma unroll
    for (int i = 0; i < L::NCOVC; i++) s.covc[i] = __ldcg(st + (long long)(L::COVC + i) * ld + ch);
#pragma unroll
    for (int i = 0; i < L::NOBS; i++) s.obsm[i] = __ldcg(st + (long long)(L::OBSM + i) * ld + ch);
}

template <class L>
__device__ __forceinline__ void store_stats(const Stats<L> &s, double *st, long long ld, long long ch) {
#pragma unroll
    for (int i = 0; i < L::D; i++) st[(long long)(L::MEAN + i) * ld + ch] = s.mean[i];
#pragma unroll
    for (int i = 0; i < L::NCOVR; i++) st[(long long)(L::COVR + i) * ld + ch] = s.covr[i];
#pragma unroll
    for (int i = 0; i < L::NCOVC; i++) st[(long long)(L::COVC + i) * ld + ch] = s.covc[i];
#pragma unroll
    for (int i = 0; i < L::NOBS; i++) st[(long long)(L::OBSM + i) * ld + ch] = s.obsm[i];
}

/* ------------------------------------------------------------------------------------------ Cholesky factors
 * Replaces the SVD hidden inside np.random.multivariate_normal (metropolis_engine.py:268,300): the factor only
 * changes when measure() changes the covariance, so it is recomputed there, not per step.
 * Real block C_r = L L^T; complex block C_c = G G^H.  Returns nonzero if a pivot was not positive. */
template <class L, bool FAST = false>
__device__ __forceinline__ int refactor(const Stats<L> &s, Chain<L> &c) {
    int bad = 0;
    /* FAST (throughput build): one reciprocal square root per pivot — L_ii = a r, L_ij = a_ij r_j with r = a^-1/2 —
       instead of a libdevice sqrt plus a division per off-diagonal entry */
    double rinv[nz(L::NR)];
#pragma unroll
    for (int i = 0; i < L::NR; i++) {
#pragma unroll
        for (int j = 0; j <= i; j++) {
            double a = s.covr[tri(i, j)];
#pragma unroll
            for (int k = 0; k < j; k++) a -= c.facr[tri(i, k)] * c.facr[tri(j, k)];
            if (i == j) {
                if (FAST) {
                    const bool ok = a > 0.0;
                    if (!ok) bad = 1;
                    const double r = rsqrt_pos(ok ? a : 1.0);
                    rinv[i] = ok ? r : 0.0;
                    c.facr[tri(i, i)] = ok ? a * r : 0.0;
                } else {
                    if (!(a > 0.0)) { bad = 1; a = 0.0; }
                    c.facr[tri(i, i)] = sqrt(a);
                }
            } else if (FAST) {
                c.facr[tri(i, j)] = a * rinv[j];
            } else {
                const double piv = c.facr[tri(j, j)];
                c.facr[tri(i, j)] = piv > 0.0 ? a / piv : 0.0;
            }
        }
    }
    constexpr int dg = L::NC * (L::NC - 1);
    double cinv[nz(L::NC)];
#pragma unroll
    for (int i = 0; i < L::NC; i++) {
#pragma unroll
        for (int j = 0; j <= i; j++) {
            if (i == j) {
                double a = s.covc[dg + i];
#pragma unroll
                for (int k = 0; k < j; k++) {
                    const double re = c.facc[herm_lo(i, k)], im = c.facc[herm_lo(i, k) + 1];
                    a -= re * re + im * im;
                }
                if (FAST) {
                    const bool ok = a > 0.0;
                    if (!ok) bad = 1;
                    const double r = rsqrt_pos(ok ? a : 1.0);
                    cinv[i] = ok ? r : 0.0;
                    c.facc[dg + i] = ok ? a * r : 0.0;
                } else {
                    if (!(a > 0.0)) { bad = 1; a = 0.0; }
                    c.facc[dg + i] = sqrt(a);
                }
            } else {
                double are = s.covc[herm_lo(i, j)], aim = s.covc[herm_lo(i, j) + 1];
#pragma unroll
                for (int k = 0; k < j; k++) {   /* a -= G_ik conj(G_jk) */
                    const double pr = c.facc[herm_lo(i, k)], pi = c.facc[herm_lo(i, k) + 1];
                    const double qr = c.facc[herm_lo(j, k)], qi = c.facc[herm_lo(j, k) + 1];
                    are -= pr * qr + pi * qi;
                    aim -= pi * qr - pr * qi;
                }
                if (FAST) {
                    c.facc[herm_lo(i, j)] = are * cinv[j];
                    c.facc[herm_lo(i, j) + 1] = aim * cinv[j];
                } else {
                    const double piv = c.facc[dg + j];
                    c.facc[herm_lo(i, j)] = piv > 0.0 ? are / piv : 0.0;
                    c.facc[herm_lo(i, j) + 1] = piv > 0.0 ? aim / piv : 0.0;
                }
            }
        }
    }
    return bad;
}

/* ------------------------------------------------------------------------------------------ proposal
 * real block   x' = x + sigma_r L z                         ~ N(x, sigma_r^2 C_r)          (ME:268-270)
 * complex      c' = c + sigma_c conj(G) xi, xi=(z+iz')/sqrt2 ~ CN(c, sigma_c^2 conj(C_c))   (ME:288-302; App. B-8)
 * Draw order per step: real block first, then complex (ME:246).  Normals (2q, 2q+1) come from Philox slot q. */
template <class L>
struct Draws {                 /* everything random one step consumes; independent of the chain's state */
    double z[(L::D + 1) / 2 * 2];
    double u;                  /* parity build: the accept uniform */
    float lo, hi;              /* throughput build: the threshold window (Rng::accept_window) */
    double u2;                 /* D = 1 (ShareCall): the same for the odd step of the pair; z[1] is its normal */
    float lo2, hi2;
};

template <class L>
struct Raw {                   /* the generator output one step consumes: one Philox call per Gaussian pair */
    U4 r[(L::D + 1) / 2];
};

template <class L>
__device__ __forceinline__ void gen_bits(const Rng &rng, unsigned step, Raw<L> &raw) {
    if (ShareCall<L>::value) { raw.r[0] = rng.bits(step >> 1, 0u); return; }
#pragma unroll
    for (int q = 0; q < (L::D + 1) / 2; q++) raw.r[q] = rng.bits(step, (unsigned)q);
}

/* D = 1: everything the two steps of a pair consume, from the pair's call: z[0] / (u | lo, hi) for the even step, z[1] /
   (u2 | lo2, hi2) for the odd one */
template <class L, bool STRICT, class Tab>
__device__ __forceinline__ void shape_pair(const Raw<L> &raw, const MathTables &T, Draws<L> &d, const Pins &pins,
                                           const MeParams &p, const Tab &logtab, const LaneTemp *lt = nullptr) {
    const float t_ln2 = lt ? lt->t_ln2 : p.t_ln2, t_band = lt ? lt->t_band : p.t_band;
    const U4 r = raw.r[0];
    Rng::box_muller<STRICT, Tab>(share_radius_bits(r), T, d.z[0], d.z[1], pins.unit, pins.angle, logtab);
    const Spare se = share_spare(r, 0u), so = share_spare(r, 1u);
    if (STRICT) {
        d.u = Rng::accept_uniform(se);
        d.u2 = Rng::accept_uniform(so);
    } else {
        Rng::accept_window(se.w0, t_ln2, t_band, d.lo, d.hi);
        Rng::accept_window(so.w0, t_ln2, t_band, d.lo2, d.hi2);
    }
}
/* the odd step of a pair takes over what the even step carried */
template <class L>
__device__ __forceinline__ void take_second_half(const Draws<L> &even, Draws<L> &odd) {
    odd.z[0] = even.z[1]; odd.z[1] = even.z[1];
    odd.u = even.u2; odd.u2 = even.u2;
    odd.lo = even.lo2; odd.hi = even.hi2; odd.lo2 = even.lo2; odd.hi2 = even.hi2;
}

template <class L, bool STRICT, class Tab>
__device__ __forceinline__ void shape_draws(const Raw<L> &raw, const MathTables &T, Draws<L> &d, const Pins &pins,
                                            const MeParams &p, const Tab &logtab, unsigned step = 0u,
                                            const LaneTemp *lt = nullptr) {
    constexpr int NQ = (L::D + 1) / 2;
    if (ShareCall<L>::value) {            /* stateless form: the draws of `step` from its pair's call */
        shape_pair<L, STRICT, Tab>(raw, T, d, pins, p, logtab, lt);
        if (step & 1u) { const Draws<L> e = d; take_second_half<L>(e, d); }
        return;
    }
    Spare sp;
    sp.w0 = sp.x0 = 0;
#pragma unroll
    for (int q = 0; q < NQ; q++) {
        Rng::keep_spare(raw.r[q], q, sp);
        Rng::box_muller<STRICT, Tab>(raw.r[q], T, d.z[2 * q], d.z[2 * q + 1], pins.unit, pins.angle, logtab);
    }
    /* strict build: the uniform itself; throughput build: a window around the energy threshold -T ln u */
    if (STRICT) d.u = Rng::accept_uniform(sp);
    else Rng::accept_window(sp.w0, lt ? lt->t_ln2 : p.t_ln2, lt ? lt->t_band : p.t_band, d.lo, d.hi);
    d.u2 = 0.0;
    d.lo2 = d.hi2 = 0.0f;
}

template <class L, bool STRICT, class Tab>
__device__ __forceinline__ void gen_draws(const Rng &rng, unsigned step, const MathTables &T, Draws<L> &d,
                                          const Pins &pins, const MeParams &p, const Tab &logtab,
                                          const LaneTemp *lt = nullptr) {
    Raw<L> raw;
    gen_bits<L>(rng, step, raw);
    shape_draws<L, STRICT, Tab>(raw, T, d, pins, p, logtab, step, lt);
}

template <class L>
__device__ __forceinline__ void apply_proposal(const Chain<L> &c, const double *z, double (&prop)[L::D]) {
#pragma unroll
    for (int i = 0; i < L::NR; i++) {
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j <= i; j++) acc = acc + c.facr[tri(i, j)] * z[j];
        prop[i] = c.x[i] + c.sig[0] * acc;
    }
    constexpr int dg = L::NC * (L::NC - 1);
    const double sc = c.sig[1] * 0.70710678118654752440;
#pragma unroll
    for (int i = 0; i < L::NC; i++) {
        double are = 0.0, aim = 0.0;
#pragma unroll
        for (int j = 0; j < i; j++) {
            const double lre = c.facc[herm_lo(i, j)], lim = -c.facc[herm_lo(i, j) + 1];
            const double zre = z[L::NR + 2 * j], zim = z[L::NR + 2 * j + 1];
            are = are + (lre * zre - lim * zim);
            aim = aim + (lre * zim + lim * zre);
        }
        are = are + c.facc[dg + i] * z[L::NR + 2 * i];
        aim = aim + c.facc[dg + i] * z[L::NR + 2 * i + 1];
        prop[L::NR + i] = c.x[L::NR + i] + sc * are;
        prop[L::NR + L::NC + i] = c.x[L::NR + L::NC + i] + sc * aim;
    }
}

/* Magnitude-phase complex moves (complex_sample_method="magnitude-phase", ME:129-130, 168-207, 304-317): the
 * reference's step_complex_group becomes a Gaussian move of every modulus at fixed phase followed by a uniform redraw of
 * every phase at fixed modulus, each with its own Metropolis test.  group 3 = magnitudes, group 4 = phases.
 *   magnitude: |c_j|' = |c_j| + s_j z_j with s_j = sigma_c^2 C_jj — the reference hands this VARIANCE to
 *              random.gauss as the standard deviation (ME:305,310); reproduced.  C_jj = sum_k |G_jk|^2.
 *   phase:     c_j' = |c_j| e^{i theta}, theta = pi t - pi, t = 2^-31 x (angle word of Philox call j). */
template <class L>
__device__ __forceinline__ void propose_magnitudes(const Chain<L> &c, const double *z, double (&prop)[L::D]) {
    constexpr int NR = L::NR, NC = L::NC, dg = NC * (NC - 1);
#pragma unroll
    for (int i = 0; i < NR; i++) prop[i] = c.x[i];
#pragma unroll
    for (int j = 0; j < NC; j++) {
        double cjj = c.facc[dg + j] * c.facc[dg + j];
#pragma unroll
        for (int k = 0; k < j; k++)
            cjj += c.facc[herm_lo(j, k)] * c.facc[herm_lo(j, k)] + c.facc[herm_lo(j, k) + 1] * c.facc[herm_lo(j, k) + 1];
        const double re = c.x[NR + j], im = c.x[NR + NC + j];
        const double mag = hypot(re, im);
        const double nm = mag + z[j] * ((c.sig[1] * c.sig[1]) * cjj);
        const double ratio = nm / mag;
        /* zero modulus: cmath.polar keeps atan2's signed zeros — arg(+0 +-0i) = +-0, arg(-0 +-0i) = +-pi (a rejected
         * first move followed by a phase redraw leaves 0 x -cos(theta) = -0 behind) */
        const bool neg0 = __double2hiint(re) < 0;
        prop[NR + j] = mag > 0.0 ? re * ratio : (neg0 ? -nm : nm);
        prop[NR + NC + j] = mag > 0.0 ? im * ratio : nm * copysign(neg0 ? 1.2246467991473532e-16 : 0.0, im);
    }
}

template <class L>
__device__ __forceinline__ void propose_phases(const Chain<L> &c, const Rng &rng, unsigned step, double (&prop)[L::D]) {
    constexpr int NR = L::NR, NC = L::NC;
#pragma unroll
    for (int i = 0; i < NR; i++) prop[i] = c.x[i];
#pragma unroll
    for (int j = 0; j < NC; j++) {
        const U4 r = rng.bits(step, (unsigned)j);
        double sn, cs;
        sincospi_bits(r.z, sn, cs);
        const double mag = hypot(c.x[NR + j], c.x[NR + NC + j]);
        prop[NR + j] = mag * -cs;
        prop[NR + NC + j] = mag * -sn;
    }
}

/* ------------------------------------------------------------------------------------------ decision + adaptation */
struct Gains {            /* per measure-block constants of the Robbins-Monro update (ME:429-456) */
    double f;             /* max(n_measure / m, 200) */
    double up, ndown;     /* fast mode: ratio (1 - target) / f and -ratio target / f */
    double k64;           /* pinned 64/ln2 of exp_nonpos */
    bool hot;             /* temp != 0 */
};

template <bool FAST = false>
__device__ __forceinline__ Gains make_gains(long long n_meas, const MeParams &p, double inv_n = 0.0) {
    Gains g;
    if (FAST) {
        /* 1/f = min(m / n, 1/200): no FP64 division (the measure block runs once per few steps; three divisions with
           their slow-path calls were a tenth of the C2 step cost); inv_n = 1/n from the measure clock */
        const double invf = n_meas > 200LL * p.m ? (double)p.m * inv_n : 0.005;
        g.f = 0.0;
        g.up = (p.ratio * (1 - p.target)) * invf;
        g.ndown = -((p.ratio * p.target) * invf);
        asm volatile("" : "+d"(g.up), "+d"(g.ndown));
        g.hot = p.temp != 0;
        g.k64 = ME_C_64_LN2;
        return g;
    }
    double f = (double)n_meas / (double)p.m;
    if (!(f > 200.0)) f = 200.0;
    g.f = f;
    g.up = p.ratio * (1 - p.target) / f;
    g.ndown = -(p.ratio * p.target / f);
    /* keep the two quotients as values: without this the compiler sinks the division into the step loop
       (select the numerator by `accept`, divide once per step) */
    asm volatile("" : "+d"(g.up), "+d"(g.ndown));
    g.hot = p.temp != 0;
    g.k64 = ME_C_64_LN2;
    return g;
}

/* Metropolis test (ME:319-338): ties accept; T == 0 rejects every uphill move; otherwise u <= exp(-1*diff/T). */
template <bool STRICT>
__device__ __forceinline__ bool decide(double diff, double u, const MeParams &p, const MathTables &T, bool hot,
                                       const double k64 = ME_C_64_LN2, const LaneTemp *lt = nullptr) {
    if (STRICT) {
        const double temp = lt ? lt->temp : p.temp;
        if (diff <= 0) return true;
        if (temp == 0) return false;
        return u <= exp(-1 * diff / temp);
    }
    /* throughput build: `u` is the precomputed threshold -T ln u >= 0 (see the stream definition): one comparison;
       ties accept, NaN rejects, T == 0 accepts only dE <= 0 */
    return diff <= u;
}

template <bool STRICT>
__device__ __forceinline__ double adapt_sigma(double sig, bool accept, const Gains &g, const MeParams &p) {
    if (STRICT) {
        const double c = sig * p.ratio;
        return accept ? sig + (c * (1 - p.target)) / g.f : sig - (c * p.target) / g.f;
    }
    return fma(sig, accept ? g.up : g.ndown, sig);
}

/* |c_j| of the observables: libdevice hypot in the parity build; in the throughput build sqrt(re^2 + im^2) through
 * MUFU.RSQ64H + Newton (relative error < 2^-52.5; |c| < 1e-140 reads as 0, an overflowing sum of squares as NaN). */
template <bool FAST>
__device__ __forceinline__ double cabs2(double re, double im) {
    if (!FAST) return hypot(re, im);
    const double w = fma(re, re, im * im);
    return w >= 1e-280 ? sqrt_pos_full(w) : 0.0;
}

/* ------------------------------------------------------------------------------------------ measure (ME:342-427)
 * Running means, Haario recursion + sigma^2/n regulariser once n > 50, observable means; evaluation order as in
 * the reference (SURVEY Appendix A).  numpy divides a complex array by a real as multiplication by the reciprocal,
 * so the complex block uses inv_n / inv_n1 where the real block divides (strict build); the throughput build
 * uses the reciprocals everywhere. */
/* Counter of the measure loop as the throughput build wants it: n as a double and its reciprocal.  The reciprocals of
 * consecutive counters are all the measure block needs (1/n, 1/(n-1), and m/n for the Robbins-Monro gain), so ONE
 * reciprocal is computed per measure and the previous one is kept; the counter itself is advanced in floating point
 * (exact below 2^53) instead of three 64-bit integer->double conversions. */
struct MeasureClock {
    double dn, inv_dn;
    __device__ __forceinline__ void start(long long n) { dn = (double)n; inv_dn = __drcp_rn(dn); }
};

/* Everything of one measure period of the throughput build that depends on the measure counter alone, i.e. is the same
 * for every chain of the launch: the Robbins-Monro gains of the period's steps and the coefficients of the measure that
 * ends it.  run_body has the threads of a CTA compute a chunk of these rows into shared memory once, instead of every
 * thread recomputing its row (two reciprocals with their slow-path tests, the gains) in every period. */
struct MeasureRow {
    double up, ndown;                          /* Gains::up / ndown of the period's steps */
    double inv_n, inv_n1, shrink, decay, grow; /* the measure: counter n0 -> n0 + 1 */
    double pad;
};
static_assert(sizeof(MeasureRow) == 64, "run_body's shared-memory budget counts 64 bytes per MeasureRow");

/* the row of the period that starts at counter n0 (the same values as a MeasureClock started at n0 and advanced by
   one measure) */
__device__ __forceinline__ void fill_measure_row(long long n0, const MeParams &p, MeasureRow &r) {
    MeasureClock clk;
    clk.start(n0);
    const Gains g = make_gains<true>(n0, p, clk.inv_dn);
    const double dn1 = clk.dn, dn = dn1 + 1.0, dn2 = dn1 - 1.0;
    const double inv_n = __drcp_rn(dn), inv_n1 = clk.inv_dn;
    r.up = g.up; r.ndown = g.ndown;
    r.inv_n = inv_n; r.inv_n1 = inv_n1;
    r.shrink = dn1 * inv_n; r.decay = dn2 * inv_n1; r.grow = dn * inv_n1;
    r.pad = 0.0;
}

template <class L, bool STRICT>
__device__ __forceinline__ void measure_update(Chain<L> &c, Stats<L> &s, long long n, const MeasureRow *row = nullptr) {
    constexpr int NR = L::NR, NC = L::NC;
    double dn = 0.0, dn1 = 0.0, inv_n, inv_n1, shrink, decay, grow;
    if (!STRICT && row != nullptr) {          /* the row of the period this measure ends (counter n - 1 -> n) */
        inv_n = row->inv_n; inv_n1 = row->inv_n1;
        shrink = row->shrink; decay = row->decay; grow = row->grow;
    } else {
        dn = (double)n; dn1 = (double)(n - 1);
        const double dn2 = (double)(n - 2);
        /* throughput build: two reciprocals per measure instead of a division per element */
        inv_n = STRICT ? 1.0 / dn : __drcp_rn(dn); inv_n1 = STRICT ? 1.0 / dn1 : __drcp_rn(dn1);
        shrink = STRICT ? dn1 / dn : dn1 * inv_n;
        decay = STRICT ? dn2 / dn1 : dn2 * inv_n1;
        grow = STRICT ? dn / dn1 : dn * inv_n1;
    }
    const bool adapt_cov = n > 50;
    if (NR > 0) {
        double old[nz(NR)];
#pragma unroll
        for (int i = 0; i < NR; i++) old[i] = s.mean[i];
#pragma unroll
        for (int i = 0; i < NR; i++) {
            s.mean[i] = s.mean[i] * shrink;
            s.mean[i] = s.mean[i] + (STRICT ? c.x[i] / dn : c.x[i] * inv_n);
        }
        if (adapt_cov) {
            const double small = STRICT ? (c.sig[0] * c.sig[0]) / dn : (c.sig[0] * c.sig[0]) * inv_n;
#pragma unroll
            for (int i = 0; i < NR; i++)
#pragma unroll
                for (int j = 0; j <= i; j++) {
                    const double v = s.covr[tri(i, j)] * decay;
                    const double xx = STRICT ? (c.x[i] * c.x[j]) / dn1 : (c.x[i] * c.x[j]) * inv_n1;
                    const double add = ((old[i] * old[j] - grow * (s.mean[i] * s.mean[j])) + xx) + (i == j ? small : 0.0);
                    s.covr[tri(i, j)] = v + add;
                }
        }
    }
    if (NC > 0) {
        double *xr = c.x + NR, *xi = c.x + NR + NC, *mr = s.mean + NR, *mi = s.mean + NR + NC;
        double orr[nz(NC)], oi[nz(NC)];
#pragma unroll
        for (int j = 0; j < NC; j++) { orr[j] = mr[j]; oi[j] = mi[j]; }
#pragma unroll
        for (int j = 0; j < NC; j++) {
            mr[j] = mr[j] * shrink; mi[j] = mi[j] * shrink;
            mr[j] = mr[j] + xr[j] * inv_n; mi[j] = mi[j] + xi[j] * inv_n;
        }
        if (adapt_cov) {
            const double small = STRICT ? (c.sig[1] * c.sig[1]) / dn : (c.sig[1] * c.sig[1]) * inv_n;
            constexpr int dg = NC * (NC - 1);
#pragma unroll
            for (int i = 0; i < NC; i++)
#pragma unroll
                for (int j = 0; j <= i; j++) {
                    const double o_re = orr[i] * orr[j] + oi[i] * oi[j], o_im = oi[i] * orr[j] - orr[i] * oi[j];
                    const double m_re = mr[i] * mr[j] + mi[i] * mi[j], m_im = mi[i] * mr[j] - mr[i] * mi[j];
                    const double x_re = xr[i] * xr[j] + xi[i] * xi[j], x_im = xi[i] * xr[j] - xr[i] * xi[j];
                    const double a_re = ((o_re - grow * m_re) + x_re * inv_n1) + (i == j ? small : 0.0);
                    const double a_im = ((o_im - grow * m_im) + x_im * inv_n1);
                    if (i == j) {
                        s.covc[dg + i] = s.covc[dg + i] * decay + a_re;
                    } else {
                        s.covc[herm_lo(i, j)] = s.covc[herm_lo(i, j)] * decay + a_re;
                        s.covc[herm_lo(i, j) + 1] = s.covc[herm_lo(i, j) + 1] * decay + a_im;
                    }
                }
        }
    }
    /* observables |x_i|, |c_j|, x_i^2 (ME:458-463) and their running mean (ME:412-414) */
#pragma unroll
    for (int i = 0; i < NR; i++)
        s.obsm[i] = s.obsm[i] * shrink + (STRICT ? fabs(c.x[i]) / dn : fabs(c.x[i]) * inv_n);
#pragma unroll
    for (int j = 0; j < NC; j++) {
        const double a = cabs2<!STRICT>(c.x[NR + j], c.x[NR + NC + j]);
        s.obsm[NR + j] = s.obsm[NR + j] * shrink + (STRICT ? a / dn : a * inv_n);
    }
#pragma unroll
    for (int i = 0; i < NR; i++) {
        const double q = c.x[i] * c.x[i];
        s.obsm[NR + NC + i] = s.obsm[NR + NC + i] * shrink + (STRICT ? q / dn : q * inv_n);
    }
    if (adapt_cov && refactor<L, !STRICT>(s, c)) c.status |= ME_STATUS_NOT_PSD;
}

/* ------------------------------------------------------------------------------------------ pooled moments
 * Ensemble-level shifted raw moments  sum(x-s), sum (x-s)(x-s)^T, sum obs  over every (chain, measure) sample —
 * the quantity the pooled-statistics all-reduce sums across GPUs (SURVEY §8e).  No reference counterpart
 * (the reference is one chain); pooled mean/covariance are derived on the host. */
template <class L, class F>
__device__ __forceinline__ void for_each_pool_word(const Chain<L> &c, const double (&sh)[L::D], F &&f) {
    constexpr int D = L::D, NR = L::NR, NC = L::NC;
    double dx[D];
#pragma unroll
    for (int i = 0; i < D; i++) dx[i] = c.x[i] - sh[i];
#pragma unroll
    for (int i = 0; i < D; i++) f(i, dx[i]);
#pragma unroll
    for (int i = 0; i < D; i++)
#pragma unroll
        for (int j = 0; j <= i; j++) f(D + tri(i, j), dx[i] * dx[j]);
    constexpr int O = D + D * (D + 1) / 2;
#pragma unroll
    for (int i = 0; i < NR; i++) f(O + i, fabs(c.x[i]));
#pragma unroll
    for (int j = 0; j < NC; j++) f(O + NR + j, hypot(c.x[NR + j], c.x[NR + NC + j]));
#pragma unroll
    for (int i = 0; i < NR; i++) f(O + NR + NC + i, c.x[i] * c.x[i]);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(ME_FULL, v, o);
    return v;
}

/* Pooled moments of mid-sized shapes (9 < POOLW, D <= 15) on the FP64 tensor cores.  The sums over the 32 chains of a warp
 * of y y^T, y = [x - s, 1], are a matrix product with the chains as the K dimension: per measure the warp stages y in shared
 * memory (row = coordinate, column = chain; two rounds of 16 chains), reads it back in mma.m8n8k4 fragment order — the A
 * and the B fragment of a thread are the same word when the row block equals the column block — and issues
 * 8 x NBX (NBX + 1) / 2 DMMAs (C3: 24); the observable sums are a second product against a unit vector.  No shuffles and
 * no CTA barrier: the 87 warp_sum reductions of the 3r+4c shape (870 SHFL + two __syncthreads per measure) were 39 % of
 * that kernel's time (tests/scripts/c3_probe.py: 13.9 ms with them, 8.5 ms without).  Each accumulator element belongs to
 * one thread, which adds it to its word of the warp's row of pooled sums (pw). */
#define ME_YB_LD 20            /* doubles per staged row: 16 chains + 4 of padding (fragment reads take two wavefronts) */
/* staging rows (a multiple of 8 holding [x - s, 1]) and the CTA size that keeps the per-warp staging + the warp's row of sums
   + the math tables inside the 48 KB of static shared memory: D <= 15 -> 16 rows, 128 threads; D <= 23 -> 24 rows, 64
   threads; D <= 31 -> 32 rows, 32 threads.  choose_dims (me_api.cu) applies the same rule on the host. */
__host__ __device__ constexpr int me_pool_mma_rows(int d) { return (d + 1 + 7) / 8 * 8; }
__host__ __device__ constexpr int me_pool_mma_max_block(int d) { return d + 1 <= 16 ? 128 : (d + 1 <= 24 ? 64 : 32); }
__host__ __device__ constexpr bool me_pool_mma_shape(int d, int poolw) { return poolw > 9 && d + 1 <= 32; }

__device__ __forceinline__ void dmma_8x8x4(double &d0, double &d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};"
                 : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

template <class L, bool FAST>
__device__ __forceinline__ void pool_mma_update(const Chain<L> &c, const double (&sh)[L::D], bool active,
                                                double (*yb)[ME_YB_LD], double *pw) {
    constexpr int D = L::D, NR = L::NR, NC = L::NC, NOBS = L::NOBS;
    /* row blocks of [x - s, 1] (instantiated, never executed, for larger shapes: their block count is clamped) */
    constexpr int NBX = (D + 1 + 7) / 8 <= 4 ? (D + 1 + 7) / 8 : 4;
    constexpr int NBO = (NOBS + 7) / 8;            /* row blocks of the observables */
    const int lane = threadIdx.x & 31, r8 = lane >> 2, k4 = lane & 3, half = lane >> 4, colw = lane & 15;
    double acc[NBX * (NBX + 1) / 2][2];
#pragma unroll
    for (int i = 0; i < NBX * (NBX + 1) / 2; i++) acc[i][0] = acc[i][1] = 0.0;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        __syncwarp();
        if (half == h) {
#pragma unroll
            for (int i = 0; i < D; i++) yb[i][colw] = active ? c.x[i] - sh[i] : 0.0;
            yb[D][colw] = active ? 1.0 : 0.0;
        }
        __syncwarp();
#pragma unroll
        for (int t = 0; t < 4; t++) {
            double a[NBX];
#pragma unroll
            for (int b = 0; b < NBX; b++) {
                const double v = yb[8 * b + r8][4 * t + k4];
                a[b] = (8 * b + r8 <= D) ? v : 0.0;          /* rows beyond the constant 1 are never written */
            }
#pragma unroll
            for (int i = 0; i < NBX; i++)
#pragma unroll
                for (int j = 0; j <= i; j++) dmma_8x8x4(acc[tri(i, j)][0], acc[tri(i, j)][1], a[i], a[j]);
        }
    }
    /* observables |x_i|, |c_j|, x_i^2: sums over the chains = product with the unit vector e_0 (result column 0) */
    double ob[NOBS];
#pragma unroll
    for (int i = 0; i < NR; i++) ob[i] = active ? fabs(c.x[i]) : 0.0;
#pragma unroll
    for (int j = 0; j < NC; j++) ob[NR + j] = active ? cabs2<FAST>(c.x[NR + j], c.x[NR + NC + j]) : 0.0;
#pragma unroll
    for (int i = 0; i < NR; i++) ob[NR + NC + i] = active ? c.x[i] * c.x[i] : 0.0;
    double acco[NBO][2];
    const double e0 = r8 == 0 ? 1.0 : 0.0;
#pragma unroll
    for (int cb = 0; cb < NBO; cb++) {
        acco[cb][0] = acco[cb][1] = 0.0;
#pragma unroll
        for (int h = 0; h < 2; h++) {
            __syncwarp();
            if (half == h) {
#pragma unroll
                for (int r = 0; r < 8; r++)
                    if (8 * cb + r < NOBS) yb[r][colw] = ob[8 * cb + r];
            }
            __syncwarp();
#pragma unroll
            for (int t = 0; t < 4; t++) {
                const double v = yb[r8][4 * t + k4];
                dmma_8x8x4(acco[cb][0], acco[cb][1], (8 * cb + r8 < NOBS) ? v : 0.0, e0);
            }
        }
    }
    /* every needed element of the products has exactly one owner in the warp */
#pragma unroll
    for (int i = 0; i < NBX; i++)
#pragma unroll
        for (int j = 0; j <= i; j++)
#pragma unroll
            for (int e = 0; e < 2; e++) {
                const int r = 8 * i + r8, cc = 8 * j + 2 * k4 + e;
                if (r < D && cc <= r) pw[D + r * (r + 1) / 2 + cc] += acc[tri(i, j)][e];
                else if (r == D && cc < D) pw[cc] += acc[tri(i, j)][e];
            }
#pragma unroll
    for (int cb = 0; cb < NBO; cb++)
        if (k4 == 0 && 8 * cb + r8 < NOBS) pw[D + D * (D + 1) / 2 + 8 * cb + r8] += acco[cb][0];
}

/* ------------------------------------------------------------------------------------------ one state-dependent step
 * proposal (already formed in `prop`) -> hard wall (ME:247) -> energy (ME:250) -> decision (ME:252) -> select
 * (ME:253-257) -> width adaptation (ME:258 / group variants ME:440-456). */
template <class Cfg, class Tab = LogTabGlobal>
__device__ __forceinline__ bool finish_step(Chain<Lay<Cfg::NR, Cfg::NC>> &c, double (&prop)[Lay<Cfg::NR, Cfg::NC>::D],
                                            const Draws<Lay<Cfg::NR, Cfg::NC>> &d, const Gains &g, const MeParams &p,
                                            const MathTables &tables, int group, const Rng &rng, unsigned step,
                                            const Tab &logtab, const LaneTemp *lt = nullptr,
                                            const double *krung = nullptr) {
    using L = Lay<Cfg::NR, Cfg::NC>;
    using Energy = typename Cfg::Energy;
    constexpr bool STRICT = Cfg::STRICT;
    constexpr int D = L::D;
    const double *k = krung ? krung : p.consts;      /* the chain's rung constants on a Hamiltonian ladder */
    if (L::KIND == 0 && group != 0) {       /* group-wise step: the other block keeps its value */
#pragma unroll
        for (int i = 0; i < D; i++) {
            const bool real_block = i < L::NR;
            if (real_block != (group == 1)) prop[i] = c.x[i];
        }
    }
    bool accept = false;
    const bool wall = p.use_reject && Energy::reject(prop, prop + L::NR, prop + L::NR + L::NC, k);
    if (STRICT) {
        if (!wall) {
            const double e_new = Energy::eval(prop, prop + L::NR, prop + L::NR + L::NC, k);
            if (e_new != e_new) c.status |= ME_STATUS_ENERGY_NAN;
            accept = decide<STRICT>(e_new - c.e, d.u, p, tables, g.hot, g.k64, lt);
            if (accept) {
                c.e = e_new;
#pragma unroll
                for (int i = 0; i < D; i++) c.x[i] = prop[i];
                c.nacc_new += 1u;
            }
        }
    } else {
        /* throughput build: dE against the FP32 window (Rng::accept_window).  The comparison stays in FP64: deciding on
           FP32(dE) instead was measured slower on the B200 (C2: 41.2 against 40.1 ms per pass), the conversion sits on
           the step's dependent chain */
        double e_new = 0.0, diff = 0.0;
        bool inside = false;
        if (!wall) {
            e_new = Energy::eval(prop, prop + L::NR, prop + L::NR + L::NC, k);
            diff = e_new - c.e;
            accept = diff <= (double)d.lo;
            inside = !accept && !(diff > (double)d.hi);
        }
        /* inside the window (about 2 steps in 10^5) or NaN: the exact threshold from the same random bits.  The branch
           is taken by the whole warp on a vote, so the common path stays straight-line code that the compiler can
           interleave with the draw stages of the following steps.  The warp is converged here: the step loop has
           uniform trip counts, lanes without a chain run it too, and the vote sits outside the wall's branch. */
        if (__any_sync(ME_FULL, inside)) {
            /* a NaN energy gives a NaN dE, which is always inside: the status bit needs no test on the common path */
            if (inside && e_new != e_new) c.status |= ME_STATUS_ENERGY_NAN;
            Spare sp;
            if (ShareCall<L>::value) sp = share_spare(rng.bits(step >> 1, 0u), step);
            else Rng::keep_spare(rng.bits(step, 0u), 0, sp);
            const double thr = Rng::accept_threshold(sp, logtab, 0.5 * (lt ? lt->temp : p.temp));
            accept = accept | (inside & (diff <= thr));
        }
        /* selects, not a divergent branch — a reconvergence region in the middle of the step would stop the compiler from
           interleaving the state update with the draw stages of the following steps */
        c.e = accept ? e_new : c.e;
#pragma unroll
        for (int i = 0; i < D; i++) c.x[i] = accept ? prop[i] : c.x[i];
        c.nacc_new += accept ? 1u : 0u;
    }
    if (L::NC > 0 && group == 4) {
        /* phase redraw: no width adapts, on the wall or otherwise (ME:194-207) */
    } else if (L::KIND == 0 && group != 0) {       /* ME:440-456: only the stepped group's width adapts */
        /* (selects, not c.sig[group - 1]: a run-time index would move the whole chain struct to local memory) */
        const double sg = adapt_sigma<STRICT>(group == 1 ? c.sig[0] : c.sig[1], accept, g, p);
        if (group == 1) c.sig[0] = sg; else c.sig[1] = sg;
    } else {
        const double sg = adapt_sigma<STRICT>(c.sig[L::SIGIDX], accept, g, p);
        c.sig[L::SIGIDX] = sg;
        if (L::KIND == 0) { c.sig[1] = sg; if (!(sg > 0)) c.status |= ME_STATUS_SIGMA_NONPOS; }
    }
    return accept;
}

/* ------------------------------------------------------------------------------------------ replica exchange
 * Stream definition (identical in oracle/me_oracle_ladder.c, meo_run_ladder).  A ladder of R rungs (a power of two <= 32) lives in
 * R consecutive lanes of a warp: global chain g is rung g % R.  Round k = n / swap_every, at a measure whose counter n (after
 * its increment) is a multiple of swap_every, pairs rungs (r, r + 1) with r = k (mod 2) (deterministic even/odd).  With
 * lo / hi the colder / hotter rung of a pair, the pair swaps iff  u <= exp((1/T_lo - 1/T_hi) (E_lo - E_hi)),  where u is
 * built like the radius uniform, (K + 1/2) 2^-52 with K = y : x[31:12], from the Philox call with counter
 * (lo(g_lo), hi(g_lo), lo32(n), 0xFFFFFFFF) and key = seed, g_lo the global id of the lower rung's chain (step draws use
 * slots < 16).  Both lanes of a pair compute the test from the same operands, so they agree.  A swap exchanges the
 * configuration, the energy and the walker label; everything adapted to a temperature (widths, means, covariances and
 * factors, observable means, counters) stays with the rung.
 *
 * Hamiltonian ladders (identical in oracle/me_oracle_hladder.c, meo_run_hladder).  Rung r has temperature T_r and constant
 * vector k_r[0..K), 1 <= K <= 16; every step evaluates the functor (eval and reject) with k_r of the chain's rung.  The
 * swap uniform, the pairing schedule and what moves or stays are those above.  With a the lower and b the upper rung of a
 * pair and E_a(x) rung a's functor with k_a at x, the pair swaps iff u <= exp(-D) with
 *     D = (1/T_a) (E_a(x_b) - E_a(x_a)) + (1/T_b) (E_b(x_a) - E_b(x_b)),
 * which both lanes evaluate from the same four energies in this operand order, so they agree bit for bit.  The pair does
 * not swap if either cross-configuration is walled (reject(x_b; k_a) or reject(x_a; k_b)).  A NaN cross-energy refuses the
 * swap and sets ME_STATUS_ENERGY_NAN on the lane that computed it (a lane that pairs and whose own wall passes its
 * partner's configuration).  After a swap a chain holds its own rung's energy of the new configuration, E_a(x_b), not its
 * partner's E.  Temperatures: finite and > 0 in any order with swaps (equal ones are the usual case), >= 0 without. */
__device__ __forceinline__ double swap_uniform(const U4 &r) {
    const double d = __hiloint2double((int)(0x3ff00000u | (r.y >> 12)), (int)((r.y << 20) | (r.x >> 12)));
    return d - (1.0 - 0x1p-53);                                               /* exact */
}

/* the rung a lane of rung r pairs with in an even / odd round; r itself when it sits out (odd rounds: the end rungs) */
__device__ __forceinline__ int swap_partner(int r, int R, bool odd) {
    const int pr = odd ? ((r + 1) ^ 1) - 1 : r ^ 1;
    return pr >= 0 && pr < R ? pr : r;
}

/* 1/T_lo - 1/T_hi of the pair a lane of rung r belongs to in an even / odd round (0 when it sits out); computed once per
   launch, so that the global loads and divisions stay off the swap's dependent chain */
__device__ __forceinline__ double swap_dbeta(const MeParams &p, int r, bool odd) {
    const int q = swap_partner(r, p.n_rungs, odd);
    const int rlo = q > r ? r : q, rhi = q > r ? q : r;
    return 1.0 / p.rung_temp[rlo] - 1.0 / p.rung_temp[rhi];
}

/* 1/T of the rung a lane of rung r pairs with in an even / odd round (Hamiltonian ladders; its own 1/T when it sits out),
   computed once per launch like swap_dbeta */
__device__ __forceinline__ double swap_beta(const MeParams &p, int r, bool odd) {
    return 1.0 / p.rung_temp[swap_partner(r, p.n_rungs, odd)];
}

/* One round.  Temperature ladders: dbeta = swap_dbeta.  Hamiltonian ladders: dbeta = swap_beta, beta = 1/T of the lane's
   own rung, krung = its rung's constants. */
template <class Cfg, int LM>
__device__ __forceinline__ void swap_round(Chain<Lay<Cfg::NR, Cfg::NC>> &c, int &walker, unsigned &swap_acc, bool odd,
                                           double dbeta, long long n, unsigned long long gid, const MeParams &p,
                                           double beta = 0.0, const double *krung = nullptr) {
    using L = Lay<Cfg::NR, Cfg::NC>;
    using Energy = typename Cfg::Energy;
    const int R = p.n_rungs;
    const int lane = threadIdx.x & 31, r = lane & (R - 1);
    const int q = swap_partner(r, R, odd);
    const bool pairs = q != r;
    const int partner = lane - r + q;
    double xo[L::D];
#pragma unroll
    for (int i = 0; i < L::D; i++) xo[i] = __shfl_sync(ME_FULL, c.x[i], partner);
    const double eo = __shfl_sync(ME_FULL, c.e, partner);
    const int wo = __shfl_sync(ME_FULL, walker, partner);
    const bool lower = q > r;
    const int rlo = lower ? r : q;
    double e_new = eo;
    bool ok = pairs;
    double delta;
    if (LM == LADDER_HAM) {
        /* own rung at the partner's configuration; the partner's rung at this one comes back by shuffle */
        const bool wall = p.use_reject && Energy::reject(xo, xo + L::NR, xo + L::NR + L::NC, krung);
        const double ec = Energy::eval(xo, xo + L::NR, xo + L::NR + L::NC, krung);
        if (pairs && !wall && ec != ec) c.status |= ME_STATUS_ENERGY_NAN;
        const double eco = __shfl_sync(ME_FULL, ec, partner);
        const bool wall_o = __shfl_sync(ME_FULL, (int)wall, partner) != 0;
        const double d_own = ec - c.e, d_other = eco - eo;
        const double b_lo = lower ? beta : dbeta, b_hi = lower ? dbeta : beta;
        const double d_lo = lower ? d_own : d_other, d_hi = lower ? d_other : d_own;
        delta = -(b_lo * d_lo + b_hi * d_hi);
        ok = ok && !wall && !wall_o;
        e_new = ec;
    } else {
        const double e_lo = lower ? c.e : eo, e_hi = lower ? eo : c.e;
        delta = dbeta * (e_lo - e_hi);
    }
    const unsigned long long glo = gid - (unsigned long long)r + (unsigned long long)rlo;
    const U4 b = philox4x32((unsigned)glo, (unsigned)(glo >> 32), (unsigned)n, 0xFFFFFFFFu, p.rk);
    const bool acc = ok && swap_uniform(b) <= exp(delta);
#pragma unroll
    for (int i = 0; i < L::D; i++) c.x[i] = acc ? xo[i] : c.x[i];
    c.e = acc ? e_new : c.e;
    walker = acc ? wo : walker;
    swap_acc += (acc && lower) ? 1u : 0u;
}

/* sum of v over the lanes of the same rung of a warp (xor offsets >= R): lane r < R then holds its rung's sum */
__device__ __forceinline__ double rung_sum(double v, int R) {
    for (int o = 16; o >= R; o >>= 1) v += __shfl_xor_sync(ME_FULL, v, o);
    return v;
}

/* ------------------------------------------------------------------------------------------ the fused kernel body
 * Cfg:  NR, NC, Energy (functor with eval / reject), STRICT (reference operation order + draw injection).   */
/* MP: instantiation that also serves the magnitude / phase moves (groups 3, 4).  They are kept out of the default
 * instantiation so that their code (a second set of generator calls, hypot) does not sit in the hot step loop.
 * PT: instantiation for temperature ladders (MeParams::n_rungs ...): every chain runs at its rung's temperature, swaps
 * configurations with its neighbour rungs at the measures (swap_round) and pools its moments into its rung's row.  A ladder
 * with swaps is R <= 32 consecutive lanes of one warp, so a launch needs chain_offset and the chain count to be multiples
 * of R (me_set_ladder); the lanes without a chain then form whole ladders of their own.
 * LM selects the ladder mode: LADDER_TEMP is the PT instantiation above; LADDER_HAM (HX) is the same with each rung's
 * functor constants (MeParams::rung_consts) held per lane for the whole launch, and a swap round that evaluates each
 * rung's energy at its partner's configuration (swap_round). */
template <class Cfg, bool MP = false, int LM = LADDER_NONE>
__device__ __forceinline__ void run_body(const MeParams &p) {
    using L = Lay<Cfg::NR, Cfg::NC>;
    using Energy = typename Cfg::Energy;
    constexpr bool STRICT = Cfg::STRICT;
    constexpr int D = L::D;
    constexpr bool PT = LM != LADDER_NONE, HAM = LM == LADDER_HAM;
    /* small problems keep running statistics and pooled accumulators in registers for the whole launch;
       larger ones touch them in global memory at measure time only */
#ifndef ME_STATS_REG_MAX
#define ME_STATS_REG_MAX 12      /* build-time experiment knobs (tests/scripts/nreg_probe.py) */
#endif
#ifndef ME_POOL_REG_MAX
#define ME_POOL_REG_MAX 9
#endif
    constexpr bool STATS_REG = (L::D + L::NCOVR + L::NCOVC + L::NOBS) <= ME_STATS_REG_MAX;
    constexpr bool POOL_REG = L::POOLW <= ME_POOL_REG_MAX;
    constexpr bool POOL_OK = L::POOLW <= ME_MAX_POOLW;        /* static shared-memory budget */
    constexpr int PW = POOL_OK ? L::POOLW : 1;
#ifndef ME_POOL_MMA
#define ME_POOL_MMA 1            /* build-time experiment knob: 0 = warp_sum reductions for every shape beyond POOL_REG */
#endif
    /* mid-sized shapes: pooled moments on the FP64 tensor cores (pool_mma_update); their CTAs are at most
       me_pool_mma_max_block(D) threads (choose_dims in me_api.cu follows the same rule) */
    constexpr bool POOL_MMA = !PT && ME_POOL_MMA && !POOL_REG && POOL_OK && me_pool_mma_shape(L::D, L::POOLW);
    constexpr int POOL_MMA_BLOCK = me_pool_mma_max_block(L::D), YB_ROWS = POOL_MMA ? me_pool_mma_rows(L::D) : 1;
    constexpr int POOL_WARPS = (POOL_MMA ? POOL_MMA_BLOCK : ME_MAX_BLOCK) / 32;
    /* ladders stage nothing in shared memory (it would cost one-warp CTAs occupancy): register-pooled shapes add their rung
       rows to the CTA's rows in global memory warp by warp at the end of the launch; the others add every measure's rung
       sums straight into the CTA's rows, which the host allows with one-warp CTAs only (me_set_ladder) */
    __shared__ double pool_warp[PT ? 1 : POOL_WARPS][PT ? 1 : PW];
    __shared__ double pool_cta[POOL_MMA || PT ? 1 : PW];
    __shared__ double ybuf[POOL_MMA ? POOL_WARPS : 1][YB_ROWS][ME_YB_LD];
    __shared__ MathTables tables;
    init_math_tables(tables);
    __syncthreads();

    /* Time segmentation with a work queue (p.seg_count > 1).  A fused launch of an ensemble that fits the device in
       about one wave is badly balanced: the CTAs that are resident at once are an integer number per SM sub-partition
       (1-warp CTAs at 129..160 registers: 12 per SM = 3 per sub-partition), 65,536 chains are 2048 of them against
       1776 slots, so a static launch runs a full first wave and then a second one at a sixth of the occupancy
       (tests/scripts/scale_probe.py: 3 warps per sub-partition saturate its pipes).  Instead the launch is cut into
       seg_count (<= 64) time segments per chain group (= the 32..128 chains of one CTA) and launched as groups x seg_count
       CTAs, each of which takes ONE item from a FIFO of ready (group, segment) items when it starts: it loads that
       group's state, runs the segment, stores the state and pushes the group's next segment.  Which CTA index runs which
       item is decided at run time, so the hardware CTA scheduler — which refills a slot the moment it frees — becomes
       a work-conserving scheduler: every slot is busy until the work runs out, all groups advance at the same rate,
       and the last, partly filled round costs 1/seg_count of the launch instead of a whole wave.  Progress: an item is
       only ever pushed by a CTA that already holds its own item (resident or finished), so the CTA holding the lowest
       unserved ticket never waits on an undispatched CTA.
       Results do not depend on the schedule: a segment is a pure function of the group's stored state.
       Queue memory (p.seg_flags, written by the host before the launch): [0] tickets handed out, [1] pushes made,
       [2 .. 2 + cap) ring of entries (segment << 32 | group) + 1, 0 = empty, pre-filled with segment 0 of every group;
       cap = p.seg_base is a power of two >= groups x 64 >= the number of items, so no two tickets share a slot.
       (A persistent-worker loop around this body was measured first: it costs 7 % in the step loop, because the
       compiler no longer proves the control flow uniform and reloads its uniform-register operands every iteration.) */
    constexpr bool SEGMENTED = L::D <= ME_SEG_MAX_D;     /* larger shapes run at 255 registers: not worth the pressure */
    __shared__ unsigned long long next_item;
    long long cgroup = blockIdx.x, b_first = 0, n_blocks = p.n_blocks;
    int seg = 0;
    if (SEGMENTED && p.seg_count > 1) {
        if (threadIdx.x == 0) {
            unsigned long long *q = p.seg_flags;
            const unsigned long long ticket = atomicAdd(q, 1ull);       /* < groups x seg_count = the grid size */
            unsigned long long *entry = q + 2 + (ticket & (p.seg_base - 1));
            unsigned long long got = 0;
            unsigned spin = 0;
            for (;;) {
                asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(got) : "l"(entry) : "memory");
                if (got != 0) break;
                __nanosleep(spin < 4096u ? 200u : 2000u);
                if (++spin > (1u << 28)) __trap();       /* > 8 minutes: a broken queue must not hang the GPU for good */
            }
            atomicExch(entry, 0ull);
            next_item = got;
        }
        __syncthreads();
        const unsigned long long it = next_item;
        cgroup = (long long)((it - 1ull) & 0xffffffffull);
        seg = (int)((it - 1ull) >> 32);
        const long long per = (p.n_blocks + p.seg_count - 1) / p.seg_count;
        b_first = seg * per;
        n_blocks = p.n_blocks - b_first < per ? p.n_blocks - b_first : per;
        if (n_blocks < 0) n_blocks = 0;
    }
    const long long tid = cgroup * blockDim.x + threadIdx.x;
    const bool active = tid < p.n_chains;
    const long long ch = active ? tid : p.n_chains - 1;
    const long long ld = p.ld;
    double *st = p.state;

    Chain<L> c;
    load_chain<L>(c, st, ld, ch);
    Stats<L> sreg;
    if (STATS_REG) load_stats<L>(sreg, st, ld, ch);
    double pacc[nz(POOL_REG ? L::POOLW : 0)];
    if (POOL_REG) {
#pragma unroll
        for (int w = 0; w < L::POOLW; w++) pacc[w] = 0.0;
    }
#ifndef ME_EXPERIMENT_NO_POOL
#define ME_EXPERIMENT_NO_POOL 0   /* build-time experiment knob (tests/scripts/c3_probe.py): what the pooled moments cost */
#endif
    const bool pooling = POOL_OK && p.pool != nullptr && p.do_measure && !ME_EXPERIMENT_NO_POOL;
    if (POOL_MMA && blockDim.x > POOL_MMA_BLOCK) __trap();       /* the host never launches this (choose_dims) */
    if (pooling && POOL_MMA) {
        for (int w = threadIdx.x; w < POOL_WARPS * PW; w += blockDim.x) (&pool_warp[0][0])[w] = 0.0;
        __syncthreads();
    } else if (pooling && !POOL_REG && !PT) {
        for (int w = threadIdx.x; w < L::POOLW; w += blockDim.x) pool_cta[w] = 0.0;
        __syncthreads();
    }
    double shift[D];
#pragma unroll
    for (int i = 0; i < D; i++) shift[i] = pooling ? p.shift[i] : 0.0;

    const Rng rng(p, p.chain_offset + (unsigned long long)ch);
    LaneTemp lane_temp;
    int walker = 0;
    unsigned swap_acc = 0u;
    /* Hamiltonian ladders: the rung's constants in registers for the whole launch (the functor indexes them with
       constants, so only the ones it reads stay live), zero beyond K as p.consts is */
    double krung[HAM ? ME_MAX_CONSTS : 1];
    if (PT) {
        const long long rung = (long long)((p.chain_offset + (unsigned long long)ch) % (unsigned long long)p.n_rungs);
        lane_temp.temp = p.rung_temp[rung];
        lane_temp.t_ln2 = p.rung_window[2 * rung];
        lane_temp.t_band = p.rung_window[2 * rung + 1];
        walker = __ldcg(p.walker + ch);
        swap_acc = __ldcg(p.swap_acc + ch);
        if (HAM) {
            const double *row = p.rung_consts + rung * p.n_consts;
#pragma unroll
            for (int i = 0; i < (HAM ? ME_MAX_CONSTS : 1); i++) krung[i] = i < p.n_consts ? row[i] : 0.0;
        }
    }
    const LaneTemp *lt = PT ? &lane_temp : nullptr;
    const double *kr = HAM ? krung : nullptr;
    const bool inject = STRICT && p.inj_delta != nullptr;
    const int group = p.group;
    /* under CUDA-graph replay the kernel parameters are frozen: the step index and the measure counter then come from
       the device copy that the library advances in-stream after every launch (MeParams::ctr_dev) */
    unsigned long long step0 = p.step0;
    long long n_meas0 = p.n_meas0;
    if (p.ctr_dev != nullptr) { step0 = __ldcg(p.ctr_dev); n_meas0 = (long long)__ldcg(p.ctr_dev + 1); }
    long long n = n_meas0 + (p.do_measure ? b_first : 0);
    /* ladders: measures left until the next swap round, and that round's parity */
    long long swap_in = 0;
    bool swap_odd = false;
    double dbeta_even = 0.0, dbeta_odd = 0.0, beta = 0.0;      /* Hamiltonian ladders: the partner's 1/T, and the own 1/T */
    if (PT && p.swap_every > 0) {
        swap_in = p.swap_every - n % p.swap_every;
        swap_odd = ((n / p.swap_every + 1) & 1) != 0;
        const int r = (int)(threadIdx.x & 31) & (p.n_rungs - 1);
        if (HAM) {
            dbeta_even = swap_beta(p, r, false);
            dbeta_odd = swap_beta(p, r, true);
            beta = 1.0 / lane_temp.temp;
        } else {
            dbeta_even = swap_dbeta(p, r, false);
            dbeta_odd = swap_dbeta(p, r, true);
        }
    }
    const unsigned step_first = (unsigned)(step0 + (unsigned long long)(b_first * p.spm));
    long long s_local = 0;
    bool accept = false;

    /* Software pipelining: the random draws do not depend on the chain's state, so they are produced ahead of the
       state-dependent chain (proposal -> energy -> exp -> select) of the step that consumes them.  An ensemble of
       65,536 chains gives each SM sub-partition only 3-4 warps, so the kernel is bound by dependent-issue latency,
       not by issue slots (tests/scripts/issue_mix.cu: FP64 and integer instructions overlap on sm_100a), and what
       counts is how many independent dependency chains one warp has in flight.  Small shapes run THREE stages per
       iteration — Philox rounds of step s+2 (10 dependent IMAD.WIDE/LOP3 rounds, ~180 cycles), Box-Muller of step
       s+1 (log -> rsqrt -> multiply, ~200 cycles), state update of step s (~190 cycles); larger shapes already
       have ceil(D/2) independent generator calls per step and keep two stages (registers). */
    constexpr bool DEEP = L::D <= 4;
    constexpr bool AHEAD = DEEP || (ME_BIG_LOOKAHEAD != 0);
    Draws<L> cur;
    Raw<L> raw_a, raw_b;
    const Pins pins = load_pins(tables);
    /* log table: read-only global path for small shapes, per-CTA shared copy for larger ones (see me_math.cuh) */
    /* static shared-memory budget (48 KB): the pooled-moment staging of a large shape (9 x POOLW doubles, up to 43 KB at
       ME_MAX_POOLW) and the 16 KB table copy do not both fit; such shapes read the table through the read-only path */
    constexpr int TAB_ENTRIES = ME_LOGTAB_ENTRIES + ME_SINTAB_ENTRIES;       /* log table, then the sin/cos table */
    constexpr int POOL_SMEM = POOL_MMA ? POOL_WARPS * (PW + YB_ROWS * ME_YB_LD) * 8 : (ME_MAX_BLOCK / 32 + 1) * PW * 8;
    constexpr bool TAB_FITS = POOL_SMEM + TAB_ENTRIES * 16 + 1024 <= 48 * 1024;
    constexpr bool TAB_SMEM = !PT && !STRICT && L::D > ME_SEG_MAX_D && TAB_FITS;   /* ladders of larger shapes run one-warp
                                                                                      CTAs: a per-CTA copy would cost occupancy */
    __shared__ double2 logtab_s[TAB_SMEM ? TAB_ENTRIES : 1];
    if (TAB_SMEM) {
        for (int i = threadIdx.x; i < TAB_ENTRIES; i += blockDim.x)
            logtab_s[i] = __ldg(reinterpret_cast<const double2 *>(p.logtab) + i);
        __syncthreads();
    }
    typedef typename TabSelect<TAB_SMEM>::type Tab;
    const Tab logtab{TAB_SMEM ? logtab_s : reinterpret_cast<const double2 *>(p.logtab)};
    if (!inject && p.spm > 0 && AHEAD) {
        gen_draws<L, STRICT, Tab>(rng, step_first, tables, cur, pins, p, logtab, lt);
        if (DEEP) gen_bits<L>(rng, step_first + 1u, raw_a);
    }

    /* one step: consumes the draws in `use`, generates the draws of the following step into `make` */
    unsigned step32 = step_first;
    auto one_step = [&](const Gains &g, Draws<L> &use, Draws<L> &make, Raw<L> &raw_in, Raw<L> &raw_out) {
        double prop[D];
        if (inject) {
            const bool absolute = MP && L::NC > 0 && group >= 3;      /* magnitude / phase records hold the proposal itself */
#pragma unroll
            for (int i = 0; i < D; i++)
                prop[i] = p.inj_delta[(s_local * D + i) * ld + ch] + (absolute ? 0.0 : c.x[i]);
            use.u = p.inj_u[s_local * ld + ch];
            s_local++;
        } else {
            if (DEEP && ShareCall<L>::value) {
                /* one call per pair of steps.  Invariant: `use` holds the draws of this step (with the pair's second half
                   when the step is even), raw_in the bits of the pair of the NEXT step */
                if ((step32 & 1u) == 0u) {           /* next step: second half of this pair; step + 2 opens a new pair */
                    gen_bits<L>(rng, step32 + 2u, raw_out);
                    take_second_half<L>(use, make);
                } else {                             /* next step opens the pair whose bits are waiting; step + 2 shares it */
                    raw_out = raw_in;
                    shape_pair<L, STRICT, Tab>(raw_in, tables, make, pins, p, logtab, lt);
                }
            } else if (DEEP) {
                gen_bits<L>(rng, step32 + 2u, raw_out);
                shape_draws<L, STRICT, Tab>(raw_in, tables, make, pins, p, logtab, 0u, lt);
            } else if (AHEAD) {
                gen_draws<L, STRICT, Tab>(rng, step32 + 1u, tables, make, pins, p, logtab, lt);
            } else {
                gen_draws<L, STRICT, Tab>(rng, step32, tables, use, pins, p, logtab, lt);
            }
            apply_proposal<L>(c, use.z, prop);
            if (MP && L::NC > 0 && group >= 3) {
                if (group == 3) propose_magnitudes<L>(c, use.z, prop);
                else propose_phases<L>(c, rng, step32, prop);
            }
        }
        accept = finish_step<Cfg, Tab>(c, prop, use, g, p, tables, group, rng, step32, logtab, lt, kr);
        step32++;
    };
    const unsigned spm = (unsigned)p.spm;
    /* running row pointer of the time series (one 64-bit add per measure instead of the full index arithmetic) */
    double *row = p.record ? p.ts + (p.ts_row0 + b_first) * (long long)L::TSCOLS * ld + ch : nullptr;
    const long long row_stride = (long long)L::TSCOLS * ld;

    /* per-measure values (MeasureRow) from a per-CTA table, a chunk of periods at a time; larger shapes (254 registers)
       keep computing them per thread, the loop nest would cost them spills */
    constexpr bool MTAB = !STRICT && SEGMENTED;
    constexpr int MCHUNK = 32;
    __shared__ MeasureRow mrow[MTAB ? MCHUNK : 1];
    for (long long b0 = 0; b0 < n_blocks; b0 += MCHUNK) {
        const int nb = n_blocks - b0 < MCHUNK ? (int)(n_blocks - b0) : MCHUNK;
        if (MTAB) {
            __syncthreads();                   /* every thread is done with the previous chunk */
            for (int j = threadIdx.x; j < nb; j += blockDim.x) fill_measure_row(n + (p.do_measure ? j : 0), p, mrow[j]);
            __syncthreads();
        }
        for (int j = 0; j < nb; j++) {
            Gains g;
            if (!MTAB) {
                g = make_gains<!STRICT>(n, p, STRICT ? 0.0 : __drcp_rn((double)n));
            } else {
                g = Gains{};
                g.up = mrow[j].up;
                g.ndown = mrow[j].ndown;
            }
            g.k64 = pins.k64;
            /* steps in pairs so that the two draw buffers swap roles by name instead of by register moves */
            Draws<L> nxt;
            unsigned k = 0;
            if (ME_PAIR_BIG || DEEP) {
                for (; k + 1 < spm; k += 2) {
                    one_step(g, cur, nxt, raw_a, raw_b);
                    one_step(g, nxt, cur, raw_b, raw_a);
                }
                if (k < spm) {
                    one_step(g, cur, nxt, raw_a, raw_b);
                    if (!inject) { cur = nxt; if (DEEP) raw_a = raw_b; }
                }
            } else {
                /* larger shapes: one step per iteration (the pair-unrolled loop of a 3r+4c shape is 27 KB of code) */
#pragma unroll 1
                for (; k < spm; k++) {
                    one_step(g, cur, nxt, raw_a, raw_b);
                    if (!inject && AHEAD) cur = nxt;
                }
            }
            if (p.do_measure) {
                n += 1;
                if (STATS_REG) {
                    measure_update<L, STRICT>(c, sreg, n, MTAB ? &mrow[j] : nullptr);
                } else {
                    Stats<L> s;
                    load_stats<L>(s, st, ld, ch);
                    measure_update<L, STRICT>(c, s, n, MTAB ? &mrow[j] : nullptr);
                    if (active) store_stats<L>(s, st, ld, ch);
                }
                if (p.record && active) {
#pragma unroll
                    for (int i = 0; i < D; i++) __stcs(row + (long long)i * ld, c.x[i]);
                    __stcs(row + (long long)D * ld, c.e);
                    if (L::KIND == 0) {
                        __stcs(row + (long long)(D + 1) * ld, c.sig[0]);
                        __stcs(row + (long long)(D + 2) * ld, c.sig[1]);
                    } else {
                        __stcs(row + (long long)(D + 1) * ld, c.sig[L::SIGIDX]);
                    }
                }
                if (p.record) row += row_stride;
                if (pooling) {
                    if (POOL_REG) {
                        for_each_pool_word<L>(c, shift, [&](int w, double v) { pacc[w] += v; });
                    } else if (PT) {
                        const int lane = threadIdx.x & 31, R = p.n_rungs;
                        double *row_pool = p.pool + cgroup * (long long)(R * L::POOLW) + lane * L::POOLW;
                        for_each_pool_word<L>(c, shift, [&](int w, double v) {
                            v = rung_sum(active ? v : 0.0, R);
                            if (lane < R) row_pool[w] = __ldcg(row_pool + w) + v;
                        });
                    } else if (POOL_MMA) {
                        const int warp = threadIdx.x >> 5;
                        pool_mma_update<L, !STRICT>(c, shift, active, ybuf[warp], pool_warp[warp]);
                    } else {
                        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
                        for_each_pool_word<L>(c, shift, [&](int w, double v) {
                            v = warp_sum(active ? v : 0.0);
                            if (lane == 0) pool_warp[warp][w] = v;
                        });
                        __syncthreads();
                        const int nw = (blockDim.x + 31) >> 5;
                        for (int w = threadIdx.x; w < L::POOLW; w += blockDim.x) {
                            double t = 0.0;
                            for (int q = 0; q < nw; q++) t += pool_warp[q][w];
                            pool_cta[w] += t;
                        }
                        __syncthreads();
                    }
                }
                if (PT && p.swap_every > 0 && --swap_in == 0) {
                    swap_round<Cfg, LM>(c, walker, swap_acc, swap_odd, swap_odd ? dbeta_odd : dbeta_even, n,
                                        p.chain_offset + (unsigned long long)ch, p, beta, kr);
                    swap_in = p.swap_every;
                    swap_odd = !swap_odd;
                }
            }
        }
    }

    if (active) {
        store_chain<L>(c, st, ld, ch);
        if (STATS_REG && p.do_measure) store_stats<L>(sreg, st, ld, ch);
        if (p.last_accept && p.spm > 0 && n_blocks > 0) p.last_accept[ch] = (unsigned char)accept;
        if (PT) { p.walker[ch] = walker; p.swap_acc[ch] = swap_acc; }
    }
    if (PT && pooling && POOL_REG) {       /* lanes 0..R-1 of every warp hold their rung's sums; rows rung-major */
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, R = p.n_rungs;
        double v[L::POOLW];
#pragma unroll
        for (int w = 0; w < L::POOLW; w++) v[w] = rung_sum(active ? pacc[w] : 0.0, R);
        double *rows = p.pool + cgroup * (long long)(R * L::POOLW) + lane * L::POOLW;
        const int nw = (blockDim.x + 31) >> 5;
        for (int q = 0; q < nw; q++) {            /* warps in order: the sums do not depend on the schedule */
            if (warp == q && lane < R) {
#pragma unroll
                for (int w = 0; w < L::POOLW; w++) rows[w] = __ldcg(rows + w) + v[w];
            }
            __syncthreads();
        }
    } else if (PT) {
        /* other shapes added every measure's sums to the CTA's rows already */
    } else if (pooling) {
        if (POOL_REG || POOL_MMA) {
            if (POOL_REG) {
                const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
                for (int w = 0; w < L::POOLW; w++) {
                    const double v = warp_sum(active ? pacc[w] : 0.0);
                    if (lane == 0) pool_warp[warp][w] = v;
                }
            }
            __syncthreads();
            const int nw = (blockDim.x + 31) >> 5;
            for (int w = threadIdx.x; w < L::POOLW; w += blockDim.x) {
                double t = 0.0;
                for (int q = 0; q < nw; q++) t += pool_warp[q][w];
                p.pool[cgroup * L::POOLW + w] = __ldcg(p.pool + cgroup * L::POOLW + w) + t;
            }
        } else {
            for (int w = threadIdx.x; w < L::POOLW; w += blockDim.x)
                p.pool[cgroup * L::POOLW + w] = __ldcg(p.pool + cgroup * L::POOLW + w) + pool_cta[w];
        }
    }
    if (SEGMENTED && p.seg_count > 1 && seg + 1 < p.seg_count) {      /* hand the chain group over: publish its next segment */
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long *q = p.seg_flags;
            __threadfence();                           /* the group's state is visible before its next segment is */
            const unsigned long long slot = atomicAdd(q + 1, 1ull);
            const unsigned long long item = (((unsigned long long)(seg + 1) << 32) | (unsigned long long)cgroup) + 1ull;
            asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(q + 2 + (slot & (p.seg_base - 1))), "l"(item) : "memory");
        }
    }
}

/* ------------------------------------------------------------------------------------------ initialisation (ME:40-125)
 * x <- x0; means <- x0; covariances <- identity or the constructor-supplied matrices (ME:63-70); observable means
 * <- observables of x0 (ME:80-81); widths <- sampling_width (ME:93-99); energy <- functor(x0) (ME:123-125). */
template <class Cfg>
__device__ __forceinline__ void init_body(const MeParams &p) {
    using L = Lay<Cfg::NR, Cfg::NC>;
    using Energy = typename Cfg::Energy;
    constexpr int NR = L::NR, NC = L::NC, D = L::D;
    const long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_chains) return;
    const long long ld = p.ld;
    Chain<L> c;
    Stats<L> s;
#pragma unroll
    for (int i = 0; i < D; i++) {
        c.x[i] = p.x0_broadcast ? p.x0[i] : p.x0[(long long)i * ld + ch];
        s.mean[i] = c.x[i];
    }
    c.sig[0] = c.sig[1] = p.sigma0;
#pragma unroll
    for (int i = 0; i < NR; i++)
#pragma unroll
        for (int j = 0; j <= i; j++) s.covr[tri(i, j)] = p.cov_r0 ? p.cov_r0[i * NR + j] : (i == j ? 1.0 : 0.0);
    constexpr int dg = NC * (NC - 1);
#pragma unroll
    for (int i = 0; i < NC; i++) {
        s.covc[dg + i] = p.cov_c0_re ? p.cov_c0_re[i * NC + i] : 1.0;
#pragma unroll
        for (int j = 0; j < i; j++) {
            s.covc[herm_lo(i, j)] = p.cov_c0_re ? p.cov_c0_re[i * NC + j] : 0.0;
            s.covc[herm_lo(i, j) + 1] = p.cov_c0_im ? p.cov_c0_im[i * NC + j] : 0.0;
        }
    }
#pragma unroll
    for (int i = 0; i < NR; i++) s.obsm[i] = fabs(c.x[i]);
#pragma unroll
    for (int j = 0; j < NC; j++) s.obsm[NR + j] = hypot(c.x[NR + j], c.x[NR + NC + j]);
#pragma unroll
    for (int i = 0; i < NR; i++) s.obsm[NR + NC + i] = c.x[i] * c.x[i];
    /* a Hamiltonian ladder's chain starts with its rung's energy */
    double k[ME_MAX_CONSTS];
    const bool rungs = p.rung_consts != nullptr;
    const long long rung = rungs ? (long long)((p.chain_offset + (unsigned long long)ch) % (unsigned long long)p.n_rungs) : 0;
#pragma unroll
    for (int i = 0; i < ME_MAX_CONSTS; i++)
        k[i] = rungs ? (i < p.n_consts ? p.rung_consts[rung * p.n_consts + i] : 0.0) : p.consts[i];
    c.e = p.have_e0 ? p.e_new[ch] : Energy::eval(c.x, c.x + NR, c.x + NR + NC, k);
    c.nacc = 0.0;
    c.nacc_new = 0u;
    c.status = 0;
    if (c.e != c.e) c.status |= ME_STATUS_ENERGY_NAN;
    if (refactor<L>(s, c)) c.status |= ME_STATUS_NOT_PSD;
    store_chain<L>(c, p.state, ld, ch);
    store_stats<L>(s, p.state, ld, ch);
}

/* ------------------------------------------------------------------------------------------ unfused path
 * For energies given as a torch-vectorised callable: propose -> (callable on the proposal block) -> accept.
 * Same proposal / decision / adaptation code as the fused kernel, with one HBM round trip in between. */
template <class Cfg>
__device__ __forceinline__ void propose_body(const MeParams &p) {
    using L = Lay<Cfg::NR, Cfg::NC>;
    constexpr int D = L::D;
    __shared__ MathTables tables;
    init_math_tables(tables);
    __syncthreads();
    const long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_chains) return;
    Chain<L> c;
    load_chain<L>(c, p.state, p.ld, ch);
    double prop[D];
    if (Cfg::STRICT && p.inj_delta != nullptr) {
        const bool absolute = L::NC > 0 && p.group >= 3;
#pragma unroll
        for (int i = 0; i < D; i++) prop[i] = p.inj_delta[(long long)i * p.ld + ch] + (absolute ? 0.0 : c.x[i]);
    } else {
        const Rng rng(p, p.chain_offset + (unsigned long long)ch);
        Draws<L> d;
        const unsigned step = p.ctr_dev ? (unsigned)p.ctr_dev[0] : (unsigned)p.step0;
        gen_draws<L, Cfg::STRICT, LogTabGlobal>(rng, step, tables, d, load_pins(tables), p,
                                                LogTabGlobal{reinterpret_cast<const double2 *>(p.logtab)});
        apply_proposal<L>(c, d.z, prop);
        if (L::NC > 0 && p.group >= 3) {
            if (p.group == 3) propose_magnitudes<L>(c, d.z, prop);
            else propose_phases<L>(c, rng, step, prop);
        }
    }
    if (L::KIND == 0 && p.group != 0) {
#pragma unroll
        for (int i = 0; i < D; i++)
            if ((i < L::NR) != (p.group == 1)) prop[i] = c.x[i];
    }
#pragma unroll
    for (int i = 0; i < D; i++) p.prop[(long long)i * p.ld + ch] = prop[i];
}

/* Energy (and hard wall) of a proposal block with the engine's device functor: lets a host-side predicate (a python
 * reject_condition, ME:142-146) sit between the proposal and the decision of a functor engine. */
template <class Cfg>
__device__ __forceinline__ void energy_body(const MeParams &p) {
    using L = Lay<Cfg::NR, Cfg::NC>;
    using Energy = typename Cfg::Energy;
    constexpr int D = L::D;
    const long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_chains) return;
    double x[D];
#pragma unroll
    for (int i = 0; i < D; i++) x[i] = p.prop[(long long)i * p.ld + ch];
    p.e_out[ch] = Energy::eval(x, x + L::NR, x + L::NR + L::NC, p.consts);
    if (p.rej_out)
        p.rej_out[ch] = (p.use_reject && Energy::reject(x, x + L::NR, x + L::NR + L::NC, p.consts)) ? 1 : 0;
}

template <class Cfg>
__device__ __forceinline__ void accept_body(const MeParams &p) {
    using L = Lay<Cfg::NR, Cfg::NC>;
    constexpr bool STRICT = Cfg::STRICT;
    constexpr int D = L::D;
    __shared__ MathTables tables;
    init_math_tables(tables);
    __syncthreads();
    const long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_chains) return;
    const long long ld = p.ld;
    double *st = p.state;
    double e = st[(long long)L::E * ld + ch];
    const bool grouped = L::KIND == 0 && p.group != 0;
    const int sidx = grouped ? (p.group == 1 ? 0 : 1) : L::SIGIDX;
    double sg = st[(long long)(L::SIG + sidx) * ld + ch];
    int status = (int)st[(long long)L::STATUS * ld + ch];
    const Gains g = make_gains(p.ctr_dev ? (long long)p.ctr_dev[1] : p.n_meas0, p);
    bool accept = false;
    const bool wall = p.rej != nullptr && p.rej[ch] != 0;
    if (!wall) {
        const double e_new = p.e_new[ch];
        if (e_new != e_new) status |= ME_STATUS_ENERGY_NAN;
        const double diff = e_new - e;
        double u = 0.0;
        if (STRICT && p.inj_u != nullptr) u = p.inj_u[ch];
        else if (diff > 0 && p.temp != 0) {      /* regenerate the spare words of Philox calls 0 (and 1) */
            const Rng rng(p, p.chain_offset + (unsigned long long)ch);
            Spare sp;
            const unsigned step_now = p.ctr_dev ? (unsigned)p.ctr_dev[0] : (unsigned)p.step0;
            if (ShareCall<L>::value) sp = share_spare(rng.bits(step_now >> 1, 0u), step_now);
            else Rng::keep_spare(rng.bits(step_now, 0u), 0, sp);
            u = STRICT ? Rng::accept_uniform(sp)
                       : Rng::accept_threshold(sp, LogTabGlobal{reinterpret_cast<const double2 *>(p.logtab)}, 0.5 * p.temp);
        }
        accept = decide<STRICT>(diff, u, p, tables, g.hot);
        if (accept) {
            st[(long long)L::E * ld + ch] = e_new;
#pragma unroll
            for (int i = 0; i < D; i++) st[(long long)(L::X + i) * ld + ch] = p.prop[(long long)i * ld + ch];
            st[(long long)L::NACC * ld + ch] += 1.0;
        }
    }
    if (!(L::NC > 0 && p.group == 4)) sg = adapt_sigma<STRICT>(sg, accept, g, p);     /* phase redraw: ME:194-207 */
    st[(long long)(L::SIG + sidx) * ld + ch] = sg;
    if (L::KIND == 0 && !grouped) {
        st[(long long)(L::SIG + 1) * ld + ch] = sg;
        if (!(sg > 0)) status |= ME_STATUS_SIGMA_NONPOS;
    }
    st[(long long)L::STATUS * ld + ch] = (double)status;
    if (p.last_accept) p.last_accept[ch] = (unsigned char)accept;
}

}  // namespace me

#endif
