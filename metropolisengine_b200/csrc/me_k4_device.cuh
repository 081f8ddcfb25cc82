/* me_k4_device.cuh — shared-covariance step kernel, version 2: a warp-specialised tcgen05 pipeline (sm_100a).
 *
 * One Metropolis step of an ensemble whose complex block shares ONE proposal covariance (pooled over the chains at
 * measure boundaries; reference step: metropolis_engine.py:241-259, proposal law ME:274-302, hard wall ME:247, decision
 * ME:319-338, Robbins-Monro width ME:429-438).  For a tile of 128 chains the proposal increments are one contraction
 *        Delta[128 chains x N] = Z[128 x K normals] . B^T[K x N],     N = K = 2 n_c,
 * B the real embedding of conj(G)/sqrt2 in interleaved (Re, Im) coordinates, C_c = G G^H.
 *
 * Roles inside a CTA of 16 warps (no CTA-wide barrier in the step loop):
 *   warps 8..15  GENERATORS  Philox4x32-7 -> BF16 normals by table (inverse CDF), written straight into the UMMA canonical K-major
 *                            operand layout.  The K dimension is produced in two halves, each its own pipeline stage
 *                            (mbarriers z_full / z_empty), so the generators of step s+1 start as soon as the MMAs of step
 *                            s have consumed the FIRST half of the operand: they never wait for the epilogue.
 *   warp 8 lane 0 MMA ISSUER after its warp's share of an operand half: K/32 x tcgen05.mma (M128, N, K16, kind::f16) into one
 *                            of TWO FP32 accumulators in TMEM (lane = chain), tcgen05.commit -> mbarriers.  The shared
 *                            factor B is brought in once per CTA by TMA (cp.async.bulk.tensor through a tensor map).
 *                            (A 17th warp for this role would cost four warps of registers: they are granted in fours.)
 *   warps 0..7   EPILOGUE    thread (chain m, column group g) owns the coordinates [g N/2, (g+1) N/2) of chain m for the whole
 *                            launch: tcgen05.ld -> x' = x + sigma Delta (FP64) -> the energy functor's per-mode sums -> ONE
 *                            64-thread named barrier with the other column group -> both evaluate the (identical)
 *                            Metropolis decision -> accepted chains write x' (their own words of the shared-memory state
 *                            tile).  Chain scalars (a, E, sigma, count) live in registers of both threads.
 * The only serial dependency is the state inside the epilogue; generation and contraction run ahead of it.
 *
 * Stream definition (restated by oracle/me_oracle_k4.c): chain g, step s —
 *   normals 8c .. 8c+7 of the chain's row of Z: Philox4x32-7(counter (g_lo, g_hi, s, c), key seed) -> words x, y, z, w; each
 *   word gives two normals, from its low and its high half: 12 bits index a table of the 4096 quantiles
 *   Phi^-1(1/2 + (i + 1/2) / 8192) of the half-normal law (rounded to BF16 — the operand's own format, which resolves only
 *   ~900 magnitudes anyway), bit 15 of the half is the sign.  Inverse-CDF sampling straight in the operand's precision: 8
 *   instructions per pair instead of the ~30 of an FP32 Box-Muller (the generator was more than half of the kernel's
 *   instructions), exactly symmetric, |z| <= 3.84.
 *   scalar draws: Philox call with slot 0x10000: low half of word x -> the real parameter's normal (same table), words z, w ->
 *   the accept uniform (53 bits).
 * Energy plugin: the functor supplies per-mode contributions to two sums and the total, i.e. energies of the form
 *   E = total(a, sum_j f0_j(c_j), sum_j f1_j(c_j)) — the Fourier-mode field energies this path is for:
 *     static void   mode(double q, double re, double im, const double *k, double &s0, double &s1);   q = j - n_c/2
 *     static double total(double a, double s0, double s1, const double *k, int n_c);
 *     static bool   reject(double a, const double *k);
 * Fed to NVRTC as text for user functors: no #include of anything but the sibling headers.
 */
#ifndef ME_K4_DEVICE_CUH
#define ME_K4_DEVICE_CUH

#include "me_params.h"
#include "me_math.cuh"

namespace k4 {

typedef unsigned int u32;
typedef unsigned long long u64;

constexpr int TILE = 128;               /* chains per tile = MMA M = TMEM lanes */
/* CTA shape: 16 warps = 8 epilogue warps (2 column groups x 4 lane quarters) + 8 generator warps, 128 registers each.
 * It beat a 32-warp layout (16 + 16, launched at 64 registers, epilogue warpgroups grown to 80 and generator warpgroups
 * shrunk to 48 with setmaxnreg) on B200 (profiles/r02_k4_probe_*.txt, 32,768 chains, 10 / 100 steps per launch):
 * 16 warps 90.5 / 766 us, 32 warps 96.2 / 832 us — with twice the warps the issue slots fill up (52 -> 58 %) but the
 * four threads of a chain repeat the decision and the scalar draws, the mbarrier polls double, and the shared-memory
 * pipe (state tile, partial sums, the generator's table) becomes the limiter (51 % of its cycles, MIO-throttle stalls). */
/* Two instantiations of the step kernel (template parameter XP):
 *   XP = true   the proposed state x' = x + sigma Delta of a step is parked in TMEM (FP64 = two 32-bit columns per coordinate,
 *               the thread's own lane) between the energy pass and the accept pass, which then is a TMEM load + the stores of
 *               the accepted chains (measured: 10 steps of 32,768 chains 92.1 -> 85.7 us).  With n_c = 64 the two step
 *               accumulators and x' fill all 512 TMEM columns, so the measure tail's accumulators reuse the step accumulators
 *               and hand their sums over to global memory after EVERY tile (s_read): used for launches without a measure
 *               tail and for CTAs of a single tile, where that costs nothing.
 *   XP = false  the accept pass recomputes x' from the increments and the state tile; the tail's accumulators have their own
 *               TMEM columns, accumulate over all tiles of the CTA and are written once (+14 us per measure otherwise at
 *               two tiles per CTA). */
constexpr int EPI_GROUPS = 2;                               /* threads per chain in the epilogue (column groups) */
constexpr int EPI_WARPS = 4 * EPI_GROUPS, GEN_WARPS = 8;
constexpr int GEN_PAR = GEN_WARPS * 32 / TILE;              /* generator threads per operand row */
/* the measure tail pairs generator thread (chain m, c_par) with epilogue thread (chain m, column group c_par): it takes the
   per-chain measurement of the second half of that thread's modes */
static_assert(EPI_GROUPS == GEN_PAR, "one generator thread per epilogue column group");
constexpr int GEN_WARP0 = EPI_WARPS, MMA_WARP = GEN_WARP0;  /* lane 0 of the first generator warp also issues the MMAs: registers
                                                               are granted in groups of four warps, a 33rd warp would cost four */
constexpr int THREADS = 32 * (EPI_WARPS + GEN_WARPS);
constexpr u32 SCALAR_SLOT = 0x10000u;   /* Philox slot of the per-chain scalar draws (beyond any operand chunk) */
constexpr int PHILOX_ROUNDS = 7;

struct TensorMap { alignas(64) u64 opaque[16]; };      /* a CUtensorMap, opaque to device code */

struct StepParams {
    double *state;
    long long ld, n_chains;
    u64 chain_offset;
    u32 rk[20];
    u64 step0;
    long long n_steps;
    long long chains_per_cta;      /* contiguous chains per CTA (a multiple of 32) */
    long long n_meas;              /* measure_step_counter (for the Robbins-Monro gain) */
    double temp, inv_temp, target, ratio;
    int m;                         /* n_real + n_complex */
    int n_c;
    double consts[ME_MAX_CONSTS];  /* energy functor constants */
    int use_wall;
    int use_tma;                   /* 1: B arrives through the tensor map; 0: plain loads from `factor` */
    const void *factor;            /* B operand, BF16, UMMA canonical K-major layout [K/8 chunks][N rows][8] */
    const unsigned short *ztab;    /* [4096] BF16 quantiles of the half-normal law (device memory owned by the library) */
    const double *s_a;             /* device scalar: shared proposal std of the real parameter */
    unsigned char *last_accept;
    float *dbg_z;                  /* optional [K][ld]: the normals of the FIRST step of the launch (tests / oracle taps) */
    float *dbg_delta;              /* optional [N][ld]: the tensor-core increments of the first step */
    double *dbg_scal;              /* optional [2][ld]: real-parameter normal and accept uniform of the first step */
    /* fused measure tail (do_measure != 0): after the last step of every tile the epilogue warps take the measurement
       (means, observable means, time-series row: ME:342-356, 404-414) and the CTA leaves its partial of the pooled moments
       in mom_part[blockIdx.x] (layout of k4_moments_stage1 in me_k4.cu) */
    int do_measure, record;
    long long n_meas_after;        /* measure_step_counter after the increment */
    double *ts;                    /* time-series block [rows][D + 2][ld] (record != 0) */
    long long ts_row;
    const double *shift;           /* [1 + 2 n_c] fixed shift of the pooled moments */
    double *mom_part;              /* [gridDim.x][4 + N + N N] */
};

/* state-block word offsets for n_c complex parameters: X (1 + 2 n_c) | E | SIG | MEAN (1 + 2 n_c) | OBSM (2 + n_c) | NACC | STATUS */
struct Layout {
    int D, X, E, SIG, MEAN, OBSM, NOBS, NACC, STATUS, WORDS;
    __host__ __device__ explicit Layout(int nc) {
        D = 1 + 2 * nc; X = 0; E = D; SIG = D + 1; MEAN = D + 2; OBSM = MEAN + D; NOBS = 2 + nc; NACC = OBSM + NOBS;
        STATUS = NACC + 1; WORDS = STATUS + 1;
    }
};

/* -------------------------------------------------------------------------------------------- PTX helpers */
__device__ __forceinline__ u32 smem_u32(const void *p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64 *bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ bool mbar_try_wait(u64 *bar, u32 parity) {
    u32 ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
/* bounded wait: a protocol error must not hang the GPU — trap instead */
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity) {
    for (u32 spin = 0; !mbar_try_wait(bar, parity); ++spin)
        if (spin > (1u << 26)) __trap();
}
__device__ __forceinline__ void mbar_arrive(u64 *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64 *bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void named_barrier(int id, int threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void *dst, const TensorMap *map, u64 *bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"((u64)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc(u32 *slot, u32 cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(u32 addr, u32 cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

/* D[tmem] (+)= A[smem] . B[smem]^T, BF16 inputs, FP32 accumulate, M = 128, K = 16 */
__device__ __forceinline__ void umma_bf16(u32 tmem_d, u64 desc_a, u64 desc_b, u32 idesc, u32 accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(u64 *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
/* K-major, no swizzle: core matrix = 8 rows x 16 B contiguous; row groups 128 B apart (SBO); the two 16-byte K chunks of
 * one K=16 MMA `lbo` bytes apart; descriptor fields in 16-byte units; version 1 (Blackwell). */
__device__ __forceinline__ u64 umma_desc(u32 smem_addr, u32 lbo) {
    return (u64)((smem_addr & 0x3ffffu) >> 4) | ((u64)(lbo >> 4) << 16) | ((u64)(128 >> 4) << 32) | (1ull << 46);
}
/* instruction descriptor: D = F32, A = B = BF16, both K-major, N, M = 128 */
__host__ __device__ constexpr u32 umma_idesc(int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((u32)(n >> 3) << 17) | ((u32)(TILE >> 4) << 24);
}

template <int CNT> struct TmemLd;
template <> struct TmemLd<4> {
    __device__ __forceinline__ static void ld(u32 taddr, u32 *r) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
    }
};
template <> struct TmemLd<8> {
    __device__ __forceinline__ static void ld(u32 taddr, u32 *r) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                     : "r"(taddr) : "memory");
    }
};
template <> struct TmemLd<16> {
    __device__ __forceinline__ static void ld(u32 taddr, u32 *r) {
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
                     "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                     : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                       "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                     : "r"(taddr) : "memory");
    }
};
template <> struct TmemLd<32> {
    __device__ __forceinline__ static void ld(u32 taddr, u32 *r) {
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
              "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
              "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
              "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
            : "r"(taddr) : "memory");
    }
};
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

/* registers -> this thread's TMEM lane, CNT consecutive 32-bit columns */
template <int CNT> struct TmemSt;
template <> struct TmemSt<8> {
    __device__ __forceinline__ static void st(u32 taddr, const u32 *r) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                     :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                     : "memory");
    }
};
template <> struct TmemSt<16> {
    __device__ __forceinline__ static void st(u32 taddr, const u32 *r) {
        asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
                     "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
                     :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
                        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
                     : "memory");
    }
};
template <> struct TmemSt<32> {
    __device__ __forceinline__ static void st(u32 taddr, const u32 *r) {
        asm volatile(
            "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
            "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
            "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
            :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
               "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
               "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
               "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
            : "memory");
    }
};
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

/* -------------------------------------------------------------------------------------------- RNG (FP32 path) */
struct U4 { u32 x, y, z, w; };
__device__ __forceinline__ U4 philox(u32 c0, u32 c1, u32 c2, u32 c3, const u32 *rk) {
#pragma unroll
    for (int r = 0; r < PHILOX_ROUNDS; r++) {
        const u64 p0 = (u64)0xD2511F53u * c0;
        const u64 p1 = (u64)0xCD9E8D57u * c2;
        const u32 n0 = (u32)(p1 >> 32) ^ c1 ^ rk[2 * r];
        const u32 n2 = (u32)(p0 >> 32) ^ c3 ^ rk[2 * r + 1];
        c0 = n0; c1 = (u32)p1; c2 = n2; c3 = (u32)p0;
    }
    U4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3;
    return o;
}
constexpr int ZTAB_ENTRIES = 4096;
/* two BF16 normals (packed: low half = first) from one 32-bit random word and the quantile table in shared memory */
__device__ __forceinline__ u32 normal_pair_bf16(u32 w, const unsigned short *ztab) {
    const u32 t0 = *reinterpret_cast<const unsigned short *>(reinterpret_cast<const char *>(ztab) + ((w << 1) & 0x1ffeu));
    const u32 t1 = *reinterpret_cast<const unsigned short *>(reinterpret_cast<const char *>(ztab) + ((w >> 15) & 0x1ffeu));
    return (t0 | (t1 << 16)) | (w & 0x80008000u);
}
__device__ __forceinline__ float bf16_lo_to_float(u32 packed) { return __uint_as_float(packed << 16); }
__device__ __forceinline__ float bf16_hi_to_float(u32 packed) { return __uint_as_float(packed & 0xffff0000u); }
__device__ __forceinline__ double u53(u32 hi, u32 lo) {
    const double a = __hiloint2double(0x43300000 - (27 << 20), (int)(hi >> 5)) - 33554432.0;
    const double b = __hiloint2double(0x43300000 - (53 << 20), (int)(lo >> 6)) - 0.5;
    return a + b;
}
/* |c| of a complex parameter for the observable means (ME:412-414): sqrt(re^2 + im^2) through MUFU.RSQ64H + Newton
 * (relative error < 2^-52.5).  |c| < 1e-140 reads as 0; an overflowing sum of squares (|c| > 1e154) as NaN. */
__device__ __forceinline__ double cabs_fast(double re, double im) {
    const double w = fma(re, re, im * im);
    return w >= 1e-280 ? me::sqrt_pos_full(w) : 0.0;
}
/* two floats -> packed BF16 pair, round to nearest even (low half = first) */
__device__ __forceinline__ u32 bf16x2_rn(float first, float second) {
    u32 d;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(second), "f"(first));
    return d;
}
/* FP32 accumulator word -> double (F2F.F64.F32, exact) */
__device__ __forceinline__ double f32_bits_to_f64(u32 f) { return (double)__uint_as_float(f); }

/* -------------------------------------------------------------------------------------------- built-in functor */
/* cylinder-style Fourier-mode field (SURVEY §8d C4; shape from legacy metropolis_engine.py:103,139-143):
 * E = k0 a^2 + sum_q (k1 + k2 q^2 (1+a^2)) |c_q|^2 + (k3/(2 n_c)) (sum_q |c_q|^2)^2, q = j - n_c/2; hard wall |a| >= 1 */
struct EnergyCylinder {
    __device__ __forceinline__ static void mode(double q, double re, double im, const double *, double &s0, double &s1) {
        const double m2 = fma(re, re, im * im);
        s0 += m2;
        s1 = fma(q * q, m2, s1);
    }
    /* written with explicit fma so that the compiler's contraction choices cannot change the bits (the C oracle
       restates exactly this sequence) */
    __device__ __forceinline__ static double total(double a, double s0, double s1, const double *k, int nc) {
        const double a2 = a * a;
        const double inner = fma(k[1], s0, (k[2] * (1.0 + a2)) * s1);
        const double quad = fma(k[0], a2, inner);
        return fma(k[3] / (2.0 * (double)nc), s0 * s0, quad);
    }
    __device__ __forceinline__ static bool reject(double a, const double *) { return fabs(a) >= 1.0; }
};

/* -------------------------------------------------------------------------------------------- shared memory */
template <int NC>
struct Smem {
    static constexpr int N = 2 * NC;
    static constexpr int CHUNKS = N / 8;                                   /* 16-byte K chunks per operand row */
    static constexpr int HALVES = (CHUNKS >= 2 * GEN_PAR) ? 2 : 1;         /* operand pipeline stages */
    double xs[N][TILE];                                     /* complex block, interleaved [n][chain]      N KB   */
    alignas(1024) unsigned char zs[TILE * N * 2];           /* A operand (normals), BF16, HALVES stages            */
    alignas(1024) unsigned char ls[N * N * 2];              /* B operand (factor), BF16                            */
    double part[2][EPI_GROUPS][2][TILE];                    /* [step parity][column group][sum][chain] partial sums */
    alignas(128) unsigned short ones[TILE / 8][16][8];      /* measure tail: a B operand of ones (first moments = Y . 1)     */
    double cscal[4][4];                                     /*               per lane quarter, sums of a, a^2, sigma         */
    double shift_s[N + 2];                                  /*               the moments' shift: [Re/Im interleaved N | a]   */
    alignas(16) unsigned short ztab[ZTAB_ENTRIES];          /* BF16 quantile table of the generator               8 KB   */
    me::MathTables tables;
    u64 z_full[2], z_empty[2], acc_full[2], acc_empty[2], b_full;
    u64 y_full, s_done, x_final, x_free, s_read;            /* measure tail: operands written / moment MMAs complete / final
                                                               states of the tile in xs / epilogue done reading xs / the
                                                               tile's moment sums have left TMEM */
    u32 tmem_slot;
};

static_assert(sizeof(Smem<64>) + 1024 <= 227 * 1024, "the 1 real + 64 complex tile must fit the 227 KB of one SM");

__device__ __forceinline__ void cp_async_8(void *smem_dst, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

/* Per-chain measurement of CNT complex modes j0 .. j0 + CNT - 1 of chain `m` of the tile (global chain `ch`): running means
 * and observable means (ME:404-414) of the chain's words in the state block, and the modes' columns of the time-series row.
 * Called by the epilogue threads for the first half of their modes and by the generator threads — idle at that point — for the
 * second half, so twice as many threads keep the read-modify-write traffic of the tail in flight. */
template <int NC, int CNT>
__device__ __forceinline__ void measure_modes(const StepParams &p, const Layout &L, const double (*xs)[TILE], int m,
                                              long long ch, long long ld, int j0, double inv_n, double shrink, double *row) {
    constexpr int JB = CNT < 8 ? CNT : 8;     /* modes per batch: the batch's global loads are all in flight before the first
                                                 store (stores to the state block may alias) */
    /* running pointers (one 64-bit add per mode each) instead of a 64-bit multiply per address */
    double *pmr = p.state + (long long)(L.MEAN + 1 + j0) * ld + ch, *pmi = pmr + (long long)NC * ld;
    double *pob = p.state + (long long)(L.OBSM + 1 + j0) * ld + ch;
    double *prr = row ? row + (long long)(1 + j0) * ld : nullptr, *pri = row ? prr + (long long)NC * ld : nullptr;
#pragma unroll
    for (int jb = 0; jb < CNT; jb += JB) {
        double mr[JB], mi[JB], ob[JB];
#pragma unroll
        for (int b = 0; b < JB; b++) { mr[b] = pmr[b * ld]; mi[b] = pmi[b * ld]; ob[b] = pob[b * ld]; }
#pragma unroll
        for (int b = 0; b < JB; b++) {
            const int j = j0 + jb + b;
            const double re = xs[2 * j][m], im = xs[2 * j + 1][m];
            *pmr = fma(re, inv_n, mr[b] * shrink);
            *pmi = fma(im, inv_n, mi[b] * shrink);
            *pob = fma(cabs_fast(re, im), inv_n, ob[b] * shrink);
            pmr += ld; pmi += ld; pob += ld;
            if (row) {
                __stcs(prr, re);
                __stcs(pri, im);
                prr += ld; pri += ld;
            }
        }
    }
}

/* -------------------------------------------------------------------------------------------- the step kernel */
template <int NC, class Energy, bool XP = false>
__device__ __forceinline__ void steps_body(const StepParams &p, const TensorMap *bmap) {
    typedef Smem<NC> S_t;
    constexpr int N = S_t::N, K = N, HALVES = S_t::HALVES, CHUNKS = S_t::CHUNKS;
    constexpr int CS = CHUNKS / HALVES;           /* chunks per pipeline stage (even) */
    constexpr u32 A_LBO = TILE * 16, B_LBO = N * 16;
    constexpr u32 TCOLS = N < 32 ? 32 : N;        /* TMEM columns per accumulator */
    constexpr u32 IDESC = umma_idesc(N);
    /* TMEM columns: two step accumulators [0, 2 TCOLS).  XP: the proposed state [2 TCOLS, 2 TCOLS + 2 N); the accumulators
       of the measure tail — S (N columns) and 16 (identical) columns of first moments — reuse the step accumulators, which
       are dead between the last step of a tile and the first step of the next one, and are emptied after every tile.
       Otherwise S and the first moments follow the step accumulators and live for the whole launch.  A power of two. */
    constexpr u32 XPCOL = 2 * TCOLS;
    constexpr u32 SCOL = XP ? 0 : 2 * TCOLS, CCOL = XP ? TCOLS : SCOL + N;
    constexpr u32 TUSED = XP ? 2 * TCOLS + 2 * N : CCOL + 16;
    constexpr u32 TALLOC = TUSED <= 128 ? 128 : (TUSED <= 256 ? 256 : 512);
    static_assert(TUSED <= 512 && N <= TCOLS && 16 <= TCOLS, "TMEM budget");
    constexpr u32 Y_LBO = N * 16;                 /* moment operands: [TILE / 8 chain chunks][N rows][8 chains] */
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    S_t &S = *reinterpret_cast<S_t *>(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long ld = p.ld;
    const Layout L(NC);

    me::init_math_tables(S.tables);
    if (tid == 0) {
        for (int i = 0; i < 2; i++) {
            mbar_init(&S.z_full[i], GEN_WARPS);
            mbar_init(&S.z_empty[i], 1);
            mbar_init(&S.acc_full[i], 1);
            mbar_init(&S.acc_empty[i], EPI_WARPS);
        }
        mbar_init(&S.b_full, 1);
        mbar_init(&S.y_full, GEN_WARPS);
        mbar_init(&S.s_done, 1);
        mbar_init(&S.x_final, EPI_WARPS);
        mbar_init(&S.x_free, EPI_WARPS);
        mbar_init(&S.s_read, EPI_WARPS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == MMA_WARP) tmem_alloc(&S.tmem_slot, TALLOC);
    {                                             /* the generator's quantile table */
        const uint4 *src = reinterpret_cast<const uint4 *>(p.ztab);
        uint4 *dst = reinterpret_cast<uint4 *>(S.ztab);
        for (int i = tid; i < ZTAB_ENTRIES * 2 / 16; i += THREADS) dst[i] = src[i];
    }
    if (p.do_measure) {                           /* the moments' shift, in the interleaved coordinate order of the tile */
        for (int i = tid; i < (TILE / 8) * 16 * 8; i += THREADS) (&S.ones[0][0][0])[i] = 0x3f80;     /* BF16 1.0 */
        for (int i = tid; i < N; i += THREADS) S.shift_s[i] = p.shift[1 + ((i & 1) ? NC + (i >> 1) : (i >> 1))];
        if (tid == 0) S.shift_s[N] = p.shift[0];
        fence_async_smem();
    }
    if (!p.use_tma) {                             /* plain staging of the factor (tensor map not available) */
        const uint4 *src = reinterpret_cast<const uint4 *>(p.factor);
        uint4 *dst = reinterpret_cast<uint4 *>(S.ls);
        for (int i = tid; i < N * N * 2 / 16; i += THREADS) dst[i] = src[i];
        fence_async_smem();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const u32 tmem_base = S.tmem_slot;

    /* the chains of this CTA, walked in tiles of up to 128; iteration it = tile * n_steps + s */
    const long long range_lo = (long long)blockIdx.x * p.chains_per_cta;
    const long long range_hi = range_lo + p.chains_per_cta < p.n_chains ? range_lo + p.chains_per_cta : p.n_chains;
    const long long n_tiles = range_hi > range_lo ? (range_hi - range_lo + TILE - 1) / TILE : 0;
    const long long n_steps = p.n_steps;

    if (warp >= GEN_WARP0) {
        /* ================================================================== generators (+ the MMA issuer) */
        const bool issuer = warp == MMA_WARP && lane == 0;
        if (issuer && p.use_tma) {
            constexpr int ROWS = CHUNKS * N;                 /* rows of 16 bytes */
            constexpr int BOX = ROWS < 256 ? ROWS : 256;
            mbar_expect_tx(&S.b_full, (u32)(N * N * 2));
            for (int r = 0; r < ROWS; r += BOX) tma_load_2d(S.ls + r * 16, bmap, &S.b_full, 0, r);
            mbar_wait(&S.b_full, 0);
        }
        const u32 zs_addr = smem_u32(S.zs), ls_addr = smem_u32(S.ls);
        const int gt = tid - 32 * GEN_WARP0;
        const int m = gt & (TILE - 1);                /* operand row = chain within the tile */
        const int c_par = gt >> 7;                    /* this thread takes the chunks c_par, c_par + GEN_PAR, ... of a stage */
        long long it = 0;
        for (long long t = 0; t < n_tiles; t++) {
            const long long base = range_lo + t * TILE;
            const int cnt = (int)(range_hi - base < TILE ? range_hi - base : TILE);      /* multiple of 32 */
            const bool act = m < cnt;                                                    /* warp-uniform */
            const u64 gch = p.chain_offset + (u64)(act ? base + m : base);
            const u32 c0 = (u32)gch, c1 = (u32)(gch >> 32);
            for (long long s = 0; s < n_steps; s++, it++) {
                const u32 step = (u32)(p.step0 + (u64)s);
                const u32 a = (u32)(it & 1);
                for (int h = 0; h < HALVES; h++) {
                    if (it >= 1) mbar_wait(&S.z_empty[h], (u32)((it - 1) & 1));
                    if (act) {
#pragma unroll
                        for (int cc = 0; cc < CS; cc += GEN_PAR) {
                            if (cc + c_par < CS) {
                                const int c = h * CS + cc + c_par;
                                const U4 r = philox(c0, c1, step, (u32)c, p.rk);
                                uint4 v;
                                v.x = normal_pair_bf16(r.x, S.ztab);
                                v.y = normal_pair_bf16(r.y, S.ztab);
                                v.z = normal_pair_bf16(r.z, S.ztab);
                                v.w = normal_pair_bf16(r.w, S.ztab);
                                *reinterpret_cast<uint4 *>(S.zs + c * A_LBO + m * 16) = v;
                                if (s == 0 && p.dbg_z != nullptr) {
                                    const u32 w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                                    for (int k = 0; k < 4; k++) {
                                        p.dbg_z[(long long)(8 * c + 2 * k) * ld + base + m] = bf16_lo_to_float(w4[k]);
                                        p.dbg_z[(long long)(8 * c + 2 * k + 1) * ld + base + m] = bf16_hi_to_float(w4[k]);
                                    }
                                }
                            }
                        }
                    }
                    fence_async_smem();          /* generic-proxy stores -> visible to the tensor-core (async) proxy */
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&S.z_full[h]);
                    if (issuer) {
                        /* Delta (+)= Z_stage . B_stage^T: CS / 2 x (M128, N, K16), accumulator `a` in TMEM */
                        if (h == 0 && it >= 2) mbar_wait(&S.acc_empty[a], (u32)(((it >> 1) - 1) & 1));
                        /* the previous tile's moment sums sit in the accumulators until the epilogue has read them */
                        if (XP && p.do_measure && t > 0 && s == 0 && h == 0) mbar_wait(&S.s_read, (u32)((t - 1) & 1));
                        mbar_wait(&S.z_full[h], (u32)(it & 1));
                        tc_fence_after();
#pragma unroll
                        for (int k = 0; k < CS / 2; k++) {
                            const int c = h * CS + 2 * k;            /* first of the two K chunks of this MMA */
                            umma_bf16(tmem_base + a * TCOLS, umma_desc(zs_addr + c * A_LBO, A_LBO),
                                      umma_desc(ls_addr + c * B_LBO, B_LBO), IDESC, (h > 0 || k > 0) ? 1u : 0u);
                        }
                        umma_commit(&S.z_empty[h]);                  /* the operand stage may be overwritten */
                        if (h == HALVES - 1) umma_commit(&S.acc_full[a]);   /* the accumulator is complete */
                    }
                    __syncwarp();
                }
            }
            if (p.do_measure) {
                /* measure tail.  While the epilogue warps take the per-chain measurement, the generator warps prepare the
                   operands of the pooled moments: Y = final state - shift of the tile's chains, split into two BF16 words,
                   in the K-major layout [chain chunk][coordinate row][8 chains].  Yh goes into the normals' buffer (free:
                   the last step's MMAs have completed), Yl into the state tile once the epilogue has stopped reading it.
                   Then S (+)= Yh Yh^T + Yh Yl^T + Yl Yh^T and the first moments (Yh + Yl) . 1 on the tensor cores.  Nobody
                   touches either buffer again before those MMAs have completed (s_done). */
                constexpr int GM = NC / GEN_PAR;              /* modes per generator thread */
                u32 ylp[GM];
                unsigned char *yh_row = S.zs + (m >> 3) * Y_LBO + (m & 7) * 2;
                unsigned char *yl_row = reinterpret_cast<unsigned char *>(&S.xs[0][0]) + (m >> 3) * Y_LBO + (m & 7) * 2;
                mbar_wait(&S.x_final, (u32)(t & 1));          /* the tile's last step has been decided */
#pragma unroll
                for (int jj = 0; jj < GM; jj++) {
                    const int j = c_par * GM + jj;
                    float yr = 0.f, yi = 0.f;
                    if (act) {
                        yr = (float)(S.xs[2 * j][m] - S.shift_s[2 * j]);
                        yi = (float)(S.xs[2 * j + 1][m] - S.shift_s[2 * j + 1]);
                    }
                    const u32 hi_pair = bf16x2_rn(yr, yi);
                    *reinterpret_cast<unsigned short *>(yh_row + (2 * j) * 16) = (unsigned short)hi_pair;
                    *reinterpret_cast<unsigned short *>(yh_row + (2 * j + 1) * 16) = (unsigned short)(hi_pair >> 16);
                    ylp[jj] = bf16x2_rn(yr - bf16_lo_to_float(hi_pair), yi - bf16_hi_to_float(hi_pair));
                }
                if (act) {
                    /* the second half of the modes of (chain m, column group c_par): their per-chain measurement */
                    constexpr int EM = NC / EPI_GROUPS, SHARE = EM / 2;
                    const double dn = (double)p.n_meas_after, inv_n = 1.0 / dn, shrink = (dn - 1.0) * inv_n;
                    const long long chg = base + m;
                    double *row = p.record ? p.ts + p.ts_row * (long long)(L.D + 2) * ld + chg : nullptr;
                    measure_modes<NC, SHARE>(p, L, S.xs, m, chg, ld, c_par * EM + (EM - SHARE), inv_n, shrink, row);
                }
                mbar_wait(&S.x_free, (u32)(t & 1));           /* every epilogue thread is done with the state tile */
#pragma unroll
                for (int jj = 0; jj < GM; jj++) {
                    const int j = c_par * GM + jj;
                    *reinterpret_cast<unsigned short *>(yl_row + (2 * j) * 16) = (unsigned short)(ylp[jj] & 0xffffu);
                    *reinterpret_cast<unsigned short *>(yl_row + (2 * j + 1) * 16) = (unsigned short)(ylp[jj] >> 16);
                }
                fence_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.y_full);
                if (issuer) {
                    mbar_wait(&S.y_full, (u32)(t & 1));
                    tc_fence_after();
                    const u32 yh = zs_addr, yl = smem_u32(S.xs), on = smem_u32(S.ones);
                    constexpr u32 IDESC1 = umma_idesc(16);
#pragma unroll
                    for (int k = 0; k < TILE / 16; k++) {
                        const u64 dh = umma_desc(yh + 2 * k * Y_LBO, Y_LBO), d1 = umma_desc(on + 2 * k * 256, 256);
                        umma_bf16(tmem_base + SCOL, dh, dh, IDESC, ((!XP && t > 0) || k > 0) ? 1u : 0u);
                        umma_bf16(tmem_base + CCOL, dh, d1, IDESC1, ((!XP && t > 0) || k > 0) ? 1u : 0u);
                    }
#pragma unroll
                    for (int k = 0; k < TILE / 16; k++) {
                        const u64 dh = umma_desc(yh + 2 * k * Y_LBO, Y_LBO), dl = umma_desc(yl + 2 * k * Y_LBO, Y_LBO);
                        umma_bf16(tmem_base + SCOL, dh, dl, IDESC, 1u);
                        umma_bf16(tmem_base + SCOL, dl, dh, IDESC, 1u);
                        umma_bf16(tmem_base + CCOL, dl, umma_desc(on + 2 * k * 256, 256), IDESC1, 1u);
                    }
                    umma_commit(&S.s_done);
                }
                __syncwarp();
                mbar_wait(&S.s_done, (u32)(t & 1));
            }
        }
    } else {
        /* ================================================================== epilogue */
        const int q4 = warp & 3, g = warp >> 2;        /* lane quarter (TMEM lanes 32 q4 ..), column group */
        const int m = 32 * q4 + lane;                  /* chain within the tile = TMEM lane */
        constexpr int MODES = NC / EPI_GROUPS;         /* modes per thread */
        constexpr int GEN_SHARE = MODES / 2;           /* modes whose measurement the generators take */
        constexpr int COLS = 2 * MODES;                /* accumulator columns per thread */
        constexpr int LDCH = COLS < 32 ? COLS : 32;    /* columns per tcgen05.ld */
        constexpr int LD1 = XP ? (COLS < 16 ? COLS : 16) : LDCH;     /* energy pass: increments per load (x' words are held
                                                                        until their store: 2 x LD1 registers) */
        constexpr int LD2 = 2 * COLS < 32 ? 2 * COLS : 32;           /* accept pass: words of x' per load */
        const double s_a = *p.s_a;
        double f = (double)p.n_meas / (double)p.m;
        if (!(f > 200.0)) f = 200.0;
        const double g_up = p.ratio * (1 - p.target) / f, g_down = p.ratio * p.target / f;
        const double q_first = (double)(g * MODES - NC / 2);     /* wavenumber of this thread's first mode */
        double sc_acc[4] = {0.0, 0.0, 0.0, 0.0};                 /* measure tail: scalar sums over this CTA's tiles */
        long long it = 0;
        for (long long t = 0; t < n_tiles; t++) {
            const long long base = range_lo + t * TILE;
            const int cnt = (int)(range_hi - base < TILE ? range_hi - base : TILE);
            const bool act = 32 * q4 < cnt;                                              /* warp-uniform */
            const long long ch = act ? base + m : base;
            const u64 gch = p.chain_offset + (u64)ch;
            const u32 c0 = (u32)gch, c1 = (u32)(gch >> 32);
            /* this thread's words of the tile's state (asynchronous copies: all of them in flight at once), and — every
               thread of the chain redundantly — the chain's scalars */
            double a = 0, e = 0, sig = 0, nacc = 0;
            int status = 0, accepted_last = 0;
            if (act) {
#pragma unroll
                for (int jj = 0; jj < MODES; jj++) {
                    const int j = g * MODES + jj;
                    cp_async_8(&S.xs[2 * j][m], p.state + (long long)(L.X + 1 + j) * ld + ch);
                    cp_async_8(&S.xs[2 * j + 1][m], p.state + (long long)(L.X + 1 + NC + j) * ld + ch);
                }
                a = p.state[(long long)L.X * ld + ch];
                e = p.state[(long long)L.E * ld + ch];
                sig = p.state[(long long)L.SIG * ld + ch];
                nacc = p.state[(long long)L.NACC * ld + ch];
                status = (int)p.state[(long long)L.STATUS * ld + ch];
                cp_async_wait_all();
            }
            for (long long s = 0; s < n_steps; s++, it++) {
                const u32 step = (u32)(p.step0 + (u64)s);
                const u32 acc = (u32)(it & 1);
                /* scalar draws of this (chain, step): independent of the state, computed while the MMA is in flight */
                double za = 0.0, u = 0.0;
                if (act) {
                    const U4 r = philox(c0, c1, step, SCALAR_SLOT, p.rk);
                    za = (double)bf16_lo_to_float(normal_pair_bf16(r.x, S.ztab));
                    u = u53(r.z, r.w);
                }
                mbar_wait(&S.acc_full[acc], (u32)((it >> 1) & 1));
                tc_fence_after();
                const u32 tcol = tmem_base + acc * TCOLS + ((u32)(32 * q4) << 16) + (u32)(g * COLS);
                const u32 xcol = tmem_base + XPCOL + ((u32)(32 * q4) << 16) + (u32)(2 * g * COLS);
                bool accept = false;
                double sg = sig;
                if (act) {
                    /* ---- pass 1: proposed coordinates of this column group, the functor's two sums.  The increments are
                       read from TMEM in chunks of LDCH columns (and read again in pass 2) instead of being held in
                       registers across the decision */
                    double s0 = 0.0, s1 = 0.0, q = q_first;
#pragma unroll
                    for (int c = 0; c < COLS; c += LD1) {
                        u32 raw[LD1];
                        TmemLd<LD1>::ld(tcol + (u32)c, raw);
                        tmem_ld_wait();
                        if (s == 0 && p.dbg_delta != nullptr) {
#pragma unroll
                            for (int k = 0; k < LD1; k++)
                                p.dbg_delta[(long long)(g * COLS + c + k) * ld + ch] = __uint_as_float(raw[k]);
                        }
                        u32 xw[2 * LD1];
#pragma unroll
                        for (int jj = 0; jj < LD1 / 2; jj++) {
                            const int j = g * MODES + c / 2 + jj;
                            const double re = fma(sig, f32_bits_to_f64(raw[2 * jj]), S.xs[2 * j][m]);
                            const double im = fma(sig, f32_bits_to_f64(raw[2 * jj + 1]), S.xs[2 * j + 1][m]);
                            Energy::mode(q, re, im, p.consts, s0, s1);
                            q += 1.0;
                            xw[4 * jj] = (u32)__double2loint(re); xw[4 * jj + 1] = (u32)__double2hiint(re);
                            xw[4 * jj + 2] = (u32)__double2loint(im); xw[4 * jj + 3] = (u32)__double2hiint(im);
                        }
                        if (XP) TmemSt<XP ? 2 * LD1 : 8>::st(xcol + (u32)(2 * c), xw);   /* x' parked in this thread's TMEM lane */
                    }
                    S.part[it & 1][g][0][m] = s0;
                    S.part[it & 1][g][1][m] = s1;
                }
                named_barrier(1 + q4, 32 * EPI_GROUPS);      /* the column groups of this lane quarter exchange their sums */
                if (act) {
                    /* ---- decision, evaluated identically by every thread of the chain (ME:247-258) */
                    const double t0 = S.part[it & 1][0][0][m] + S.part[it & 1][1][0][m];
                    const double t1 = S.part[it & 1][0][1][m] + S.part[it & 1][1][1][m];
                    const double a_new = fma(sig * s_a, za, a);
                    const bool wall = p.use_wall && Energy::reject(a_new, p.consts);
                    if (!wall) {
                        const double e_new = Energy::total(a_new, t0, t1, p.consts, NC);
                        if (e_new != e_new) status |= ME_STATUS_ENERGY_NAN;
                        const double diff = e_new - e;
                        const double prob = me::exp_nonpos(fmin(-diff * p.inv_temp, 0.0), S.tables);
                        /* a NaN difference rejects, as in the reference (`uniform <= exp(nan)` is False, ME:327-338) */
                        accept = (diff <= 0) | ((p.temp != 0) & (diff == diff) & (u <= prob));
                        if (accept) { e = e_new; a = a_new; nacc += 1.0; }
                    }
                    sg = accept ? fma(sig, g_up, sig) : fma(sig, -g_down, sig);
                    if (!(sg > 0)) status |= ME_STATUS_SIGMA_NONPOS;
                    if (s == 0 && g == 0 && p.dbg_scal != nullptr) { p.dbg_scal[ch] = za; p.dbg_scal[ld + ch] = u; }
                    /* ---- pass 2: accepted chains take the proposal (the same fma as pass 1: the accepted state is
                       bit-for-bit the one whose energy was evaluated) */
                    if (XP) {
                        /* the very words whose energy was evaluated come back from TMEM */
                        tmem_st_wait();
                        if (__any_sync(0xffffffffu, accept)) {
#pragma unroll
                            for (int c = 0; c < 2 * COLS; c += LD2) {
                                u32 w[LD2];
                                TmemLd<LD2>::ld(xcol + (u32)c, w);
                                tmem_ld_wait();
                                if (accept) {
#pragma unroll
                                    for (int k = 0; k < LD2 / 2; k++)
                                        S.xs[g * COLS + c / 2 + k][m] = __hiloint2double((int)w[2 * k + 1], (int)w[2 * k]);
                                }
                            }
                        }
                    } else if (__any_sync(0xffffffffu, accept)) {
#pragma unroll
                        for (int c = 0; c < COLS; c += LDCH) {
                            u32 raw[LDCH];
                            TmemLd<LDCH>::ld(tcol + (u32)c, raw);
                            tmem_ld_wait();
                            if (accept) {
#pragma unroll
                                for (int jj = 0; jj < LDCH / 2; jj++) {
                                    const int j = g * MODES + c / 2 + jj;
                                    S.xs[2 * j][m] = fma(sig, f32_bits_to_f64(raw[2 * jj]), S.xs[2 * j][m]);
                                    S.xs[2 * j + 1][m] = fma(sig, f32_bits_to_f64(raw[2 * jj + 1]), S.xs[2 * j + 1][m]);
                                }
                            }
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.acc_empty[acc]);       /* this warp is done with the accumulator */
                if (act) {
                    sig = sg;
                    accepted_last = accept ? 1 : 0;
                }
            }
            if (p.do_measure) {                               /* the generators may read the tile's final states */
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.x_final);
            }
            /* store this thread's words of the tile */
            if (act) {
#pragma unroll 8
                for (int jj = 0; jj < MODES; jj++) {
                    const int j = g * MODES + jj;
                    p.state[(long long)(L.X + 1 + j) * ld + ch] = S.xs[2 * j][m];
                    p.state[(long long)(L.X + 1 + NC + j) * ld + ch] = S.xs[2 * j + 1][m];
                }
                if (g == 0) {
                    p.state[(long long)L.X * ld + ch] = a;
                    p.state[(long long)L.E * ld + ch] = e;
                    p.state[(long long)L.SIG * ld + ch] = sig;
                    p.state[(long long)L.NACC * ld + ch] = nacc;
                    p.state[(long long)L.STATUS * ld + ch] = (double)status;
                    if (p.last_accept && n_steps > 0) p.last_accept[ch] = (unsigned char)accepted_last;
                }
            }
            if (p.do_measure) {
                /* ---------------------------------------------------------------- measure tail of this tile */
                const double dn = (double)p.n_meas_after, inv_n = 1.0 / dn, shrink = (dn - 1.0) * inv_n;
                double *row = p.record ? p.ts + p.ts_row * (long long)(L.D + 2) * ld + ch : nullptr;
                /* the first half of this thread's modes; the generator thread (m, c_par = g) takes the second half */
                if (act) measure_modes<NC, MODES - GEN_SHARE>(p, L, S.xs, m, ch, ld, g * MODES, inv_n, shrink, row);
                if (g == 0) {
                    double va = 0.0, va2 = 0.0, vs = 0.0;
                    if (act) {
                        double *mp = &p.state[(long long)L.MEAN * ld + ch];
                        double *o0 = &p.state[(long long)L.OBSM * ld + ch], *o1 = &p.state[(long long)(L.OBSM + 1 + NC) * ld + ch];
                        const double vm = *mp, v0 = *o0, v1 = *o1;
                        *mp = fma(a, inv_n, vm * shrink);
                        *o0 = fma(fabs(a), inv_n, v0 * shrink);
                        *o1 = fma(a * a, inv_n, v1 * shrink);
                        if (row) {
                            __stcs(row, a);
                            __stcs(row + (long long)L.D * ld, e);
                            __stcs(row + (long long)(L.D + 1) * ld, sig);
                        }
                        va = a - S.shift_s[N]; va2 = va * va; vs = sig;
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        va += __shfl_xor_sync(0xffffffffu, va, o);
                        va2 += __shfl_xor_sync(0xffffffffu, va2, o);
                        vs += __shfl_xor_sync(0xffffffffu, vs, o);
                    }
                    if (lane == 0) { S.cscal[q4][0] = va; S.cscal[q4][1] = va2; S.cscal[q4][2] = vs; }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.x_free);       /* this warp is done with the state tile */
                named_barrier(6, 32 * EPI_WARPS);            /* the lane quarters' scalar sums are in place */
                /* the CTA's running scalar sums (fixed order) */
                if (tid == 0) {
                    sc_acc[0] += (double)cnt;
                    sc_acc[1] += (S.cscal[0][2] + S.cscal[1][2]) + (S.cscal[2][2] + S.cscal[3][2]);
                    sc_acc[2] += (S.cscal[0][0] + S.cscal[1][0]) + (S.cscal[2][0] + S.cscal[3][0]);
                    sc_acc[3] += (S.cscal[0][1] + S.cscal[1][1]) + (S.cscal[2][1] + S.cscal[3][1]);
                }
                mbar_wait(&S.s_done, (u32)(t & 1));           /* the moment MMAs have read both operand buffers */
                /* ---------------------------------------------------- the CTA's pooled-moment partial.  XP: this tile's sums
                   leave TMEM now (the accumulators are the next tile's step accumulators) and the later tiles of the CTA add
                   theirs to the row; otherwise the sums of all tiles are written once, after the last tile */
                if (XP || t == n_tiles - 1) {
                    double *out = p.mom_part + (long long)blockIdx.x * (4 + N + N * N);
                    auto stage_row = [](int i) { return (i & 1) ? NC + (i >> 1) : (i >> 1); };   /* interleaved -> [Re; Im] */
                    tc_fence_after();
                    const int n_row = 32 * q4 + lane;                  /* TMEM lane = row of S (interleaved coordinate) */
                    if (32 * q4 < N) {
                        if (g == 0) {                                  /* first moments: column CCOL of this lane */
                            u32 raw[4];
                            TmemLd<4>::ld(tmem_base + CCOL + ((u32)(32 * q4) << 16), raw);
                            tmem_ld_wait();
                            if (n_row < N) {
                                double *o = out + 4 + stage_row(n_row);
                                *o = f32_bits_to_f64(raw[0]) + ((XP && t > 0) ? *o : 0.0);
                            }
                        }
                        /* S is symmetric: lane n writes S[n][c] to the transposed place, so that the 32 lanes of a store fall
                           into two contiguous runs of 16 doubles */
                        const u32 scol = tmem_base + SCOL + ((u32)(32 * q4) << 16) + (u32)(g * COLS);
#pragma unroll
                        for (int c = 0; c < COLS; c += LDCH) {
                            u32 raw[LDCH];
                            TmemLd<LDCH>::ld(scol + (u32)c, raw);
                            tmem_ld_wait();
                            if (n_row < N) {
#pragma unroll
                                for (int k = 0; k < LDCH; k++) {
                                    double *o = out + 4 + N + stage_row(g * COLS + c + k) * N + stage_row(n_row);
                                    *o = f32_bits_to_f64(raw[k]) + ((XP && t > 0) ? *o : 0.0);
                                }
                            }
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (XP && lane == 0) mbar_arrive(&S.s_read);       /* the accumulators may take the next tile's steps */
                }
            }
        }
        if (p.do_measure) {
            double *out = p.mom_part + (long long)blockIdx.x * (4 + N + N * N);
            if (tid == 0) { out[0] = sc_acc[0]; out[1] = sc_acc[1]; out[2] = sc_acc[2]; out[3] = sc_acc[3]; }
            if (n_tiles == 0)                                 /* a CTA without chains contributes zeros */
                for (int i = tid; i < N + N * N; i += 32 * EPI_WARPS) out[4 + i] = 0.0;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) tmem_dealloc(tmem_base, TALLOC);
}

/* -------------------------------------------------------------------------------------------- initialisation (ME:40-125) */
template <class Energy>
__device__ __forceinline__ void init_body(const StepParams &p, const double *x0, int broadcast, double sigma0) {
    const long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (ch >= p.n_chains) return;
    const long long ld = p.ld;
    const int nc = p.n_c;
    const Layout L(nc);
    double s0 = 0.0, s1 = 0.0;
    const double a = broadcast ? x0[0] : x0[ch];
    p.state[(long long)L.X * ld + ch] = a;
    p.state[(long long)L.MEAN * ld + ch] = a;
    for (int j = 0; j < nc; j++) {
        const double re = broadcast ? x0[1 + j] : x0[(long long)(1 + j) * ld + ch];
        const double im = broadcast ? x0[1 + nc + j] : x0[(long long)(1 + nc + j) * ld + ch];
        p.state[(long long)(L.X + 1 + j) * ld + ch] = re;
        p.state[(long long)(L.X + 1 + nc + j) * ld + ch] = im;
        p.state[(long long)(L.MEAN + 1 + j) * ld + ch] = re;
        p.state[(long long)(L.MEAN + 1 + nc + j) * ld + ch] = im;
        Energy::mode((double)(j - nc / 2), re, im, p.consts, s0, s1);
        p.state[(long long)(L.OBSM + 1 + j) * ld + ch] = hypot(re, im);
    }
    p.state[(long long)L.OBSM * ld + ch] = fabs(a);
    p.state[(long long)(L.OBSM + 1 + nc) * ld + ch] = a * a;
    p.state[(long long)L.E * ld + ch] = Energy::total(a, s0, s1, p.consts, nc);
    p.state[(long long)L.SIG * ld + ch] = sigma0;
    p.state[(long long)L.NACC * ld + ch] = 0.0;
    p.state[(long long)L.STATUS * ld + ch] = 0.0;
}

}  // namespace k4

#endif
