/* me_b200.h — C ABI of the B200-native ensemble Metropolis hot path (libme_b200.so).
 *
 * This is the drop-in boundary for ONE path of jklebes/MetropolisEngine: the user's loop
 *     engine.step_all() ... engine.measure()                 (README.md:39-44)
 * over an ensemble of independent chains.  The reference has no native interface (it is one Python class,
 * metropolisengine/metropolis_engine.py "ME"), so every entry point below cites the Python method it
 * replaces.  The reference-side binding a maintainer would add is the ctypes stub in INTEGRATION.md.
 *
 * Conventions
 *   - plain C: pointers, sizes, int return codes (0 = ME_OK); no exceptions cross the boundary;
 *     me_last_error() returns the message of the last failing call on that handle (or of me_create).
 *   - every `double*` / `unsigned char*` argument is a DEVICE pointer owned by the caller (torch tensors in
 *     the Python host); the library borrows it for the duration of the call and never frees it.
 *   - all work is stream-ordered on the `stream` argument (a cudaStream_t; NULL = default stream);
 *     no call synchronises the device except me_create / me_set_energy_source (compilation, no GPU work).
 *   - one handle per GPU (rank); calls on one handle are not thread-safe (the reference is single-threaded).
 *   - arrays over chains are chain-minor: a[word * ld + chain], ld = cfg.n_chains.
 *     Parameter order inside a chain: [real..., Re c..., Im c...]  (ME:288).
 */
#ifndef ME_B200_H
#define ME_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ME_ABI_VERSION 10

enum me_status_code {
    ME_OK = 0,
    ME_ERR_INVALID = 1,      /* bad argument (reference: ValueError, ME:37-39) */
    ME_ERR_CUDA = 2,         /* CUDA runtime / driver error */
    ME_ERR_COMPILE = 3,      /* NVRTC compilation of a user functor failed (log in me_last_error) */
    ME_ERR_UNSUPPORTED = 4,  /* shape / functor not available (e.g. NVRTC missing) */
    ME_ERR_STATE = 5         /* call order (nothing bound, no energy set, ...) */
};

/* built-in device energy functors (me_energies.cuh).  The energy function is the reference's plugin
 * surface (ME:20, ME:110-120, call sites ME:231, ME:250). */
enum me_energy_id {
    ME_ENERGY_X2 = 0,          /* README.md:26-27            E = x^2                           consts: -            */
    ME_ENERGY_XY_WELL = 1,     /* demo/toymodel_xypotentialwell.py:13-18  E = k0 (x^2+y^2)     consts: k0           */
    ME_ENERGY_MIXED_WELL = 2,  /* demo/toymodel_complex_and_real.py:17-26 and its 3r+4c scale-up consts: k, alpha, beta[, bounded] */
    ME_ENERGY_CYLINDER = 3,    /* cylinder-style Fourier-mode field, wall |a|>=1               consts: kappa, alpha, gamma, beta */
    ME_ENERGY_EXTERNAL = 99,   /* energy evaluated by the caller between me_propose and me_accept (torch callable) */
    ME_ENERGY_USER = 100       /* CUDA source given to me_set_energy_source */
};

/* per-chain status bits (STATUS word of the state block); the reference's failure modes, SURVEY.md §5 */
#define ME_STATUS_NOT_PSD 1        /* numpy "covariance is not symmetric positive-semidefinite" (ME:270) */
#define ME_STATUS_SIGMA_NONPOS 2   /* assert sampling_width > 0 (ME:438) */
#define ME_STATUS_ENERGY_NAN 4

typedef struct me_engine me_engine;   /* opaque */

/* Replaces the scalar part of MetropolisEngine.__init__ (ME:17-133). */
typedef struct me_config {
    int32_t n_real;             /* ME:42  */
    int32_t n_complex;          /* ME:52  */
    int64_t n_chains;           /* chains owned by this handle (this GPU) */
    int64_t chain_offset;       /* global id of local chain 0; the RNG stream of a chain depends only on
                                   (seed, global id), so results do not depend on how chains are sharded */
    double temp;                /* ME:91  */
    double target_acceptance;   /* ME:101 */
    double ratio;               /* ME:105-107 (the host computes it: needs the normal quantile, ME:102) */
    uint64_t seed;              /* Philox4x32-10 key (reference: process-global MT19937 state) */
    int32_t device;             /* CUDA device ordinal */
    int32_t strict;             /* 1: reference operation order, no FMA contraction, draw injection available */
} me_config;

/* Word offsets of the per-chain state block (state[word * ld + chain]) and derived sizes. */
typedef struct me_layout {
    int32_t X;        /* D words: current parameters        (real_params ME:41, complex_params ME:51)          */
    int32_t E;        /* live energy                        (energy['total'] / energy_total, ME:125,236,255)   */
    int32_t SIG;      /* 2 words: real_group_sampling_width, complex_group_sampling_width (ME:97-99)           */
    int32_t MEAN;     /* D words: real_mean, complex_mean   (ME:77-78)                                         */
    int32_t COVR;     /* NR(NR+1)/2 lower-packed covariance_matrix_real    (ME:63-66)                          */
    int32_t COVC;     /* NC^2 Hermitian-packed covariance_matrix_complex   (ME:67-70)                          */
    int32_t OBSM;     /* 2NR+NC observables_mean            (ME:80-81)                                         */
    int32_t FACR;     /* Cholesky factor of COVR  (replaces the per-step SVD inside numpy, ME:268)             */
    int32_t FACC;     /* Cholesky factor of COVC  (ME:300)                                                     */
    int32_t NACC;     /* accepted-step count (the reference's commented-out accepted_counter, ME:71)           */
    int32_t STATUS;   /* ME_STATUS_* bits                                                                      */
    int32_t WORDS;    /* total words per chain                                                                 */
    int32_t D;        /* NR + 2 NC                                                                             */
    int32_t TS_COLS;  /* time-series columns per row: x[D], energy, sigma (mixed engines: sigma_real, sigma_complex)  */
    int32_t POOL_WORDS; /* pooled-moment words: sum(x-s)[D], sum (x-s)(x-s)^T [D(D+1)/2 lower], sum obs [2NR+NC];
                           0 when the shape is too large for in-kernel pooling                               */
} me_layout;

int me_abi_version(void);

/* Layout of the state block for a parameter-space shape (pure function, no GPU). */
int me_state_layout(int32_t n_real, int32_t n_complex, me_layout *out);

/* MetropolisEngine.__init__ (ME:17): creates the handle; no device memory is allocated. */
int me_create(const me_config *cfg, me_engine **out);
int me_destroy(me_engine *eng);

/* Energy plugin registration — replaces the `energy_functions` constructor argument / set_energy_function
 * (ME:110-120, ME:136-140) and set_reject_condition (ME:142-146).
 *   builtin : one of me_energy_id with its constants;
 *   source  : CUDA C++ text defining
 *                 __device__ double me_user_energy(const double* x, const double* c_re, const double* c_im, const double* k);
 *             and, when use_reject != 0,
 *                 __device__ bool   me_user_reject(const double* x, const double* c_re, const double* c_im, const double* k);
 *             compiled for sm_100a with NVRTC and fused into the step kernel — for D > 32 into the runtime-shape kernels,
 *             which hand the functor gathered arrays (ME_NR / ME_NC are predefined macros);
 *   external: the caller evaluates energies itself between me_propose and me_accept. */
int me_set_energy_builtin(me_engine *eng, int32_t energy_id, const double *consts, int32_t n_consts, int32_t use_reject);
int me_set_energy_source(me_engine *eng, const char *cuda_source, const double *consts, int32_t n_consts, int32_t use_reject);
int me_set_energy_external(me_engine *eng);

/* Compile-only check of a user functor (works without a GPU): 0 = compiles; log (may be NULL) receives the
 * NVRTC log. */
int me_check_energy_source(const char *cuda_source, int32_t n_real, int32_t n_complex, int32_t use_reject,
                           int32_t strict, char *log, int64_t log_cap);

/* CUDA-graph replay of me_run (fused launches) and of the unfused step (me_propose -> caller's energy -> me_accept).
 * Kernel parameters are frozen when a graph is captured, so with enable != 0 the step index and the measure counter
 * are read from a device copy that me_run / me_accept advance themselves in-stream; the call (re)loads that copy from
 * the handle's counters, so call it again before a replay whenever the handle's counters moved outside the graph
 * (me_set_counters, launches made with enable == 0), and advance the handle's own counters with me_set_counters after a
 * replay.  Fused shapes (D <= 32) only. */
int me_device_counters(me_engine *eng, int32_t enable, void *stream);

/* Group-wise stepping of mixed engines (SURVEY §8 row f1): subsequent me_run / me_run_injected / me_propose /
 * me_accept calls perform step_real_group (group 1, ME:225-239: only the real block is proposed, only
 * real_group_sampling_width adapts, ME:440-446) or step_complex_group (group 2, ME:209-223, ME:449-456) instead of
 * step_all (group 0).  For all-real / all-complex engines the three coincide (ME:46,56).
 * Groups 3 and 4 are the two halves of step_complex_group under complex_sample_method="magnitude-phase"
 * (SURVEY §8 row f4; ME:129-130, 168-207, 304-317): 3 = Gaussian move of every modulus at fixed phase
 * (step_complex_group_magnitude, ME:178-192, draw ME:304-310 — the reference's sigma^2 C_jj is used as the standard
 * deviation, reproduced), adapts complex_group_sampling_width; 4 = uniform redraw of every phase at fixed modulus
 * (step_complex_group_phase, ME:194-207, draw ME:312-317), adapts nothing.  In injected (parity) mode the complex
 * block of the records of groups 3 / 4 holds the ABSOLUTE proposed values, not increments. */
int me_set_group(me_engine *eng, int32_t group);

/* Temperature ladder (parallel tempering).  Global chain g runs at temps[g % n_rungs]; the handle's chains must be whole
 * ladders (chain_offset and n_chains multiples of n_rungs).  swap_every > 0: replica exchange — at every measure whose
 * counter is a multiple of swap_every, neighbour rungs (deterministic even/odd pairing) swap configurations, energies and
 * walker labels with probability min(1, exp((1/T_lo - 1/T_hi)(E_lo - E_hi))); then n_rungs is 2, 4, 8, 16 or 32 and the
 * temperatures are finite, > 0 and strictly increasing.  swap_every = 0: a temperature sweep, any n_rungs >= 2, temps >= 0.
 * walker[n_chains] (device, int32) holds each chain's walker label, swap_acc[n_chains] (device, uint32) the accepted swaps
 * between the chain's rung and the next one up; both are read and written by me_run.  Fused shapes (D <= 32) with a device
 * functor, group 0, Philox draws only.  Call before me_bind: it may change the launch geometry, and the pool buffer of a
 * ladder with a power-of-two n_rungs <= 32 holds n_rungs rows of POOL_WORDS per CTA (rung-major), other ladders pool
 * nothing.  The temperatures are copied. */
int me_set_ladder(me_engine *eng, const double *temps, int32_t n_rungs, int64_t swap_every, int32_t *walker,
                  uint32_t *swap_acc);

/* Hamiltonian ladder: me_set_ladder where every rung also has its own functor constants.  Rung r runs the handle's functor
 * (eval and reject) with consts[r * n_consts .. (r + 1) * n_consts), 1 <= n_consts <= 16, at temps[r]; me_set_energy_builtin /
 * me_set_energy_source must then be given n_consts constants (their values are not used by the ladder kernels).  With
 * swap_every > 0 a pair of neighbour rungs a < b swaps configurations and walker labels with probability min(1, exp(-D)),
 * D = (1/T_a)(E_a(x_b) - E_a(x_a)) + (1/T_b)(E_b(x_a) - E_b(x_b)), never when either cross-configuration is walled; a chain
 * that takes a new configuration takes its own rung's energy of it.  Temperatures: finite and > 0 in any order with swaps
 * (equal ones are the usual case), >= 0 without.  Chains, walkers, swap counts, pool rows and launch geometry as for
 * me_set_ladder, before me_bind; consts = NULL is me_set_ladder.  ME_ERR_INVALID (with a message) for non-finite constants,
 * n_consts outside [1, 16] or different from the registered functor's, and the temperature rules.  A handle with a rung
 * table refuses me_energy_builtin (ME_ERR_UNSUPPORTED): there is no single constant vector to evaluate with.  The
 * temperatures and constants are copied. */
int me_set_hamiltonian_ladder(me_engine *eng, const double *temps, const double *consts /* [n_rungs][n_consts] */,
                              int32_t n_consts, int32_t n_rungs, int64_t swap_every, int32_t *walker, uint32_t *swap_acc);

/* Launch geometry the handle uses; the pool buffer has grid * POOL_WORDS doubles (see me_set_ladder for ladders). */
int me_launch_dims(me_engine *eng, int32_t *grid, int32_t *block);

typedef struct me_buffers {
    double *state;              /* [WORDS][n_chains] */
    double *pool;               /* [grid][POOL_WORDS] pooled-moment accumulators (may be NULL: no pooling) */
    double *shift;              /* [D] shift of the pooled moments (required when pool != NULL) */
    unsigned char *last_accept; /* [n_chains] accept flag of the most recent step — the return value of step_all() (ME:259) */
    double *scratch;            /* [D][n_chains] work space, required when D = n_real + 2 n_complex > 32 (may be NULL otherwise) */
    double *prop;               /* [D][n_chains] proposal block of the one-launch schedule of large shapes (me_run with steps on
                                   a D > 32 handle); may be NULL: such handles then step through me_propose / me_accept only */
} me_buffers;
int me_bind(me_engine *eng, const me_buffers *buffers);

/* State initialisation (ME:40-125): x <- x0, means <- x0, covariances <- given or identity, widths <- sigma0,
 * observable means <- observables(x0), energy <- functor(x0) (or e0 for external energies), counters <- 1.
 *   x0: [D][n_chains], or [D] when x0_broadcast;  cov_r: [NR*NR];  cov_c_re / cov_c_im: [NC*NC] (NULL = identity) */
int me_init(me_engine *eng, const double *x0, int32_t x0_broadcast, double sigma0, const double *cov_r,
            const double *cov_c_re, const double *cov_c_im, const double *e0, void *stream);

/* The hot path.  One launch runs  n_blocks x ( steps_per_measure x step_all() [+ measure()] )  for every chain:
 *   step_all   ME:241-259 (mixed) / ME:225-239 (all-real) / ME:209-223 (all-complex): Philox Gaussian proposal
 *              through the Cholesky factors (ME:261-302), hard-wall predicate (ME:247), energy functor (ME:250),
 *              Metropolis test (ME:319-338), Robbins-Monro width update (ME:429-456);
 *   measure    ME:342-427: running means, covariance recursion (+ refactorisation), observable means, and, when
 *              ts != NULL, one time-series row per chain at ts[((ts_row0 + block) * TS_COLS + col) * n_chains + chain]
 *              (the lists of ME:31-35,350-356).
 *   me_run(e, 1, k, 0, ...) is k plain step_all() calls; me_run(e, 1, 0, 1, ...) is one measure().
 * Scheduling is internal and does not change results: when the ensemble is about one wave of CTAs the launch is cut
 * into time segments per chain group served from a work queue (bit-identical to the plain launch; ME_SEGMENTS=1 in the
 * environment switches it off).  The call is asynchronous on `stream`. */
int me_run(me_engine *eng, int64_t n_blocks, int64_t steps_per_measure, int32_t do_measure, double *ts,
           int64_t ts_row0, void *stream);

/* Parity mode (strict handles only): the same schedule driven by recorded draws instead of Philox —
 * delta[(step * D + k) * n_chains + chain] is added to the parameters, u[step * n_chains + chain] is the accept
 * uniform (NaN where the reference drew none).  SURVEY.md §8(c) level L-A. */
int me_run_injected(me_engine *eng, int64_t n_blocks, int64_t steps_per_measure, int32_t do_measure,
                    const double *delta, const double *u, double *ts, int64_t ts_row0, void *stream);

/* Unfused step for energies evaluated by the caller (torch-vectorised callable):
 *   me_propose writes the proposal block prop[D][n_chains]  (draw_real_group / draw_complex_group, ME:261-302);
 *   the caller computes e_new[n_chains] (and optionally a hard-wall mask rej[n_chains]);
 *   me_accept applies ME:247-258 and advances the step counter.
 * inj_delta [D][n_chains] / inj_u [n_chains] (strict handles, may be NULL) inject draws for one step. */
int me_propose(me_engine *eng, double *prop, const double *inj_delta, void *stream);
int me_accept(me_engine *eng, const double *prop, const double *e_new, const unsigned char *rej,
              const double *inj_u, void *stream);

/* Large parameter spaces (D > 32, e.g. 1 real + 64 complex with per-chain covariance — the reference's own
 * algorithm at the cylinder shape): runtime-shape kernels whose state stays in global memory (csrc/me_generic.cuh).  With a
 * device functor (built-in, or user CUDA text) me_run performs the whole schedule in one launch (me_buffers.prop required); with a caller-evaluated
 * energy, a host-side predicate, magnitude / phase moves or injected draws the step is me_propose -> energy -> me_accept
 * and me_run serves measure().
 * me_energy_builtin evaluates the handle's DEVICE functor (built-in, or user CUDA text) and its hard
 * wall on a proposal block: e_out[n_chains], rej_out[n_chains] (may be NULL).  Besides the large-shape step it lets a
 * host-side predicate — the reference's python reject_condition (ME:142-146) — sit between me_propose and me_accept
 * of a functor engine of any shape. */
int me_energy_builtin(me_engine *eng, const double *prop, double *e_out, unsigned char *rej_out, void *stream);

/* Pooled ensemble moments: out[POOL_WORDS] = sum over CTAs (fixed order, deterministic) of the accumulators
 * filled at every measure; reset != 0 zeroes the accumulators afterwards.  The caller all-reduces `out` across
 * ranks (NCCL) — the only collective of the path (SURVEY.md §8e).  No reference counterpart. */
int me_pool_reduce(me_engine *eng, double *out, int32_t reset, void *stream);

/* Pooled statistics across GPUs inside the library (SURVEY.md §8b, §8e) — the path's only collective.
 * me_comm wraps an NCCL communicator: either one the library creates (rank 0 obtains a 128-byte id with
 * me_comm_unique_id, distributes it by any means — the Python host broadcasts it through torch.distributed — and every
 * rank calls me_comm_create), or an existing ncclComm_t of the host application (me_comm_adopt; not destroyed by
 * me_comm_destroy).  NCCL itself is loaded at run time (the copy already in the process, else ME_NCCL_PATH /
 * me_comm_set_library).
 * me_allreduce_stats, all stream-ordered and without host synchronisation (so it can be captured in a CUDA graph
 * together with me_run):  inc[0..POOL_WORDS) = fixed-order sum of this handle's per-CTA accumulators (which are
 * reset), inc[POOL_WORDS] = n_samples (the (chain, measure) samples pooled since the previous call);  inc is summed
 * over the ranks of `comm` in place (comm == NULL or one rank: no collective);  totals[0..POOL_WORDS] += inc.
 * `totals` is the device-resident running moment vector the host reads once when statistics are wanted. */
typedef struct me_comm me_comm;
int me_comm_set_library(const char *libnccl_path);
int me_comm_unique_id(unsigned char *id128);
int me_comm_create(const unsigned char *id128, int32_t world, int32_t rank, int32_t device, me_comm **out);
int me_comm_adopt(void *nccl_comm, int32_t world, int32_t rank, int32_t device, me_comm **out);
int me_comm_destroy(me_comm *comm);
/* One-shot all-reduce over NVLink peer memory for the ranks of one box (SURVEY.md §5 / §8e): the pooled-moment vectors are
 * latency-bound, so each rank publishes its vector in a window of its own HBM that the other ranks open through CUDA IPC, and
 * ONE single-CTA kernel per rank waits for the peers' epoch flags and sums the windows in rank order (every rank gets
 * bitwise the same sum; replays inside CUDA graphs).  Set-up: me_comm_peer_init (allocates the window for vectors of up to
 * max_doubles, returns its 64-byte IPC handle) -> the host gathers the handles of all ranks -> me_comm_peer_connect(handles
 * [world][64]) -> once EVERY rank has connected, me_comm_peer_enable(1).  Vectors that do not fit, and communicators
 * without windows, go through NCCL.  me_comm_allreduce is the collective itself (sum, in place, stream-ordered). */
int me_comm_peer_init(me_comm *comm, int64_t max_doubles, unsigned char *handle64);
int me_comm_peer_connect(me_comm *comm, const unsigned char *handles);
int me_comm_peer_enable(me_comm *comm, int32_t enable);
int me_comm_allreduce(me_comm *comm, double *buf, int64_t n, void *stream);
const char *me_comm_last_error(void);
int me_allreduce_stats(me_engine *eng, me_comm *comm, double *inc, double *totals, int64_t n_samples, void *stream);
/* The two halves of me_allreduce_stats, for hosts that overlap the collective with the next stepping launch (SURVEY.md
 * §8e "overlap with the next stepping launch"): me_reduce_stats on the stepping stream (it reads and resets the per-CTA
 * accumulators the next me_run writes), then — ordered after it by an event — me_accumulate_stats on a side stream
 * (all-reduce of `inc` over the ranks, totals += inc).  Use one `inc` buffer per launch in flight. */
int me_reduce_stats(me_engine *eng, double *inc, int64_t n_samples, void *stream);
int me_accumulate_stats(me_engine *eng, me_comm *comm, double *inc, double *totals, void *stream);

/* measure_step_counter (ME:73) and the global step index (Philox counter); for checkpoint / resume. */
int me_get_counters(me_engine *eng, int64_t *n_measure, uint64_t *step);
int me_set_counters(me_engine *eng, int64_t n_measure, uint64_t step);

/* ------------------------------------------------------------------------------------------------------------
 * Shared-covariance tensor-core path (BASELINE config 4: 1 real + n_c complex Fourier-mode coefficients, n_c = 8, 16, 32
 * or 64).  Same step as me_run (ME:241-259), but the complex block's proposal covariance is pooled over the ensemble at
 * measure boundaries and shared by all chains, so the proposal increments of 128 chains are one BF16 tcgen05
 * contraction  Delta = Z . B^T  with the FP32 accumulator in TMEM (csrc/me_k4_device.cuh: warp-specialised pipeline of
 * generator warps, one MMA-issuing warp and epilogue warps; B arrives by TMA).  The caller owns the pooled covariance /
 * Cholesky factor (host side: engine_shared.py) and hands the factor over in `factor_bf16`:
 *   B[2i][2j] = Re G_ij / sqrt2, B[2i][2j+1] = Im G_ij / sqrt2, B[2i+1][2j] = -Im G_ij / sqrt2, B[2i+1][2j+1] = Re G_ij / sqrt2
 *   (C_c = G G^H; ME:288-302 samples CN(0, sigma^2 conj(C_c))), stored BF16 as [K/8 k-chunks][N n][8], N = K = 2 n_c (UMMA
 *   canonical K-major, no swizzle).
 * State block (me_k4_layout_for): X 1+2n_c (a, Re c, Im c) | E | SIG | MEAN 1+2n_c | OBSM 2+n_c | NACC | STATUS.
 * Energy plugin (ME:20, 110-120): the built-in cylinder-style functor (consts: kappa, alpha, gamma, beta; hard wall
 * |a| >= 1, legacy metropolis_engine.py:103,139), or CUDA text through me_k4_set_energy_source defining
 *     __device__ void   me_k4_mode(double q, double re, double im, const double *k, double &s0, double &s1);   q = j - n_c/2
 *     __device__ double me_k4_total(double a, double s0, double s1, const double *k, int n_c);
 *     __device__ bool   me_k4_reject(double a, const double *k);                  (only when use_reject != 0)
 * i.e. energies of the form E = total(a, sum_j f0_j(c_j), sum_j f1_j(c_j)); the per-mode sums are accumulated by the
 * epilogue threads in mode order (first half of the modes, second half, then added). */
typedef struct me_k4 me_k4;
typedef struct me_k4_config {
    int32_t n_real;             /* must be 1  */
    int32_t n_complex;          /* 8, 16, 32 or 64 */
    int64_t n_chains;           /* multiple of 128 */
    int64_t chain_offset;
    double temp;
    double target_acceptance;
    double ratio;               /* ME:105-107 with m = 1 + n_complex */
    uint64_t seed;
    int32_t device;
    int32_t use_reject;         /* hard wall of the functor */
    double consts[4];           /* built-in cylinder energy: kappa, alpha, gamma, beta */
} me_k4_config;
typedef struct me_k4_layout {
    int32_t X, E, SIG, MEAN, OBSM, NACC, STATUS, WORDS, D, TS_COLS, N_COMPLEX, TILE, FACTOR_BYTES, MOM_WORDS;
    int32_t MOM_SCRATCH_PER_SM;   /* doubles of me_k4_moments scratch per SM */
    int32_t SUM_GROUPS;           /* the functor's per-mode sums are accumulated over this many groups of consecutive modes
                                     (2: a + b; 4: (a + b) + (c + d)) — part of the arithmetic the oracle restates */
} me_k4_layout;
int me_k4_layout_get(me_k4_layout *out);                       /* n_complex = 64 */
int me_k4_layout_for(int32_t n_complex, me_k4_layout *out);
int me_k4_create(const me_k4_config *cfg, me_k4 **out);
int me_k4_destroy(me_k4 *eng);
int me_k4_set_energy_source(me_k4 *eng, const char *cuda_source, const double *consts, int32_t n_consts, int32_t use_reject);
int me_k4_check_energy_source(const char *cuda_source, int32_t n_complex, int32_t use_reject, char *log, int64_t log_cap);
int me_k4_bind(me_k4 *eng, double *state, const void *factor_bf16, unsigned char *last_accept);
int me_k4_init(me_k4 *eng, const double *x0, int32_t x0_broadcast, double sigma0, void *stream);
/* n_steps x step_all(); s_a = DEVICE scalar, shared proposal std of the real parameter.  Taps of the FIRST step of the launch
 * (may be NULL; tests and the oracle's injection protocol): dbg_z [2 n_c][n_chains] normals (BF16 values), dbg_delta
 * [2 n_c][n_chains] tensor-core increments (interleaved Re, Im), dbg_scal [2][n_chains] the real parameter's normal and
 * the accept uniform. */
int me_k4_step(me_k4 *eng, int64_t n_steps, const double *s_a, float *dbg_z, float *dbg_delta, double *dbg_scal, void *stream);
/* measure() without the covariance recursion (the caller pools it): means, observable means, one row
 * ts[(row * TS_COLS + col) * n_chains + chain]. */
int me_k4_measure(me_k4 *eng, double *ts, int64_t ts_row, void *stream);
/* Pooled moments of the current states of this handle's chains, deterministic (fixed summation order):
 * inc[MOM_WORDS] complex (double pairs) = [chains, sum sigma, sum a, sum a^2, sum c[64], sum c c^H[64x64]] about
 * shift[129] (a, Re c, Im c).  scratch needs (n_sm + 1) * MOM_SCRATCH_PER_SM doubles.  The caller all-reduces `inc` across
 * ranks (NCCL) and adds it to its running moments.
 * Single-GPU fast path: mom_accum (may be NULL) = running moments advanced in the same launch (mom[w] += inc[w], w != 1);
 * snapshot (may be NULL, needs MOM_WORDS + 2 complex) = [mom after the update | inc[0], inc[1]], the input of a factor
 * refresh that runs later on another stream. */
int me_k4_moments(me_k4 *eng, const double *shift, double *scratch, int64_t scratch_doubles, double *inc, double *mom_accum,
                  double *snapshot, void *stream);
/* Multi-GPU: after `inc` has been summed over the ranks (me_comm_allreduce), advance the running moments and write the
 * snapshot the factor refresh reads — on one GPU me_k4_moments / me_k4_step_measure do this themselves. */
int me_k4_accumulate_moments(me_k4 *eng, const double *inc, double *mom_accum, double *snapshot, void *stream);
/* Pooled moments -> shared covariance (+ sigma^2/n regulariser, ME:418,425) -> Cholesky -> BF16 operand, one
 * launch, no host sync.  mom / inc are complex (double pairs): mom = [N, -, sum a, sum a^2, sum c[64], sum c c^H
 * [64x64]] about a fixed shift, inc = [chains measured now, sum of their sigma]; cov_c receives the 64x64 complex
 * covariance, cov_a the variance of the real parameter, s_a its square root, status != 0 if not positive definite. */
int me_k4_refactor(me_k4 *eng, const double *mom, const double *inc, int64_t n_measure, double *cov_c, double *cov_a,
                   void *factor_bf16, double *s_a, int32_t *status, void *stream);   /* n_measure <= 0: the handle's counter */
/* The block a sampling loop repeats — n_steps x step_all(), then measure() (reference README loop; ME:241-259, 342-356)
 * — as ONE launch of the step kernel plus the two small reduction kernels of the pooled moments.  The per-chain
 * measurement equals me_k4_measure bit for bit.  The second moments sum Y Y^T are formed on the tensor cores from Y split
 * into two BF16 words (products accurate to ~2^-16 relative, FP32 accumulation per CTA, FP64 across CTAs); first moments
 * and scalar sums are FP64.  me_k4_measure + me_k4_moments remain the all-FP64 route.  Arguments as in me_k4_step,
 * me_k4_measure (ts may be NULL) and me_k4_moments; n_steps >= 1. */
int me_k4_step_measure(me_k4 *eng, int64_t n_steps, const double *s_a, double *ts, int64_t ts_row, const double *shift,
                       double *scratch, int64_t scratch_doubles, double *inc, double *mom_accum, double *snapshot,
                       void *stream);
/* The factor the next me_k4_step launches read (double-buffering: a refresh may be writing the other buffer), and the
 * number of SMs the step kernel leaves idle so that the one-CTA refresh can run beside it on another stream. */
int me_k4_set_factor(me_k4 *eng, const void *factor_bf16);
int me_k4_set_reserved_sms(me_k4 *eng, int32_t n);
/* The generator's quantile table (host copy): out[4096] BF16 bit patterns of Phi^-1(1/2 + (i + 1/2) / 8192); n must be 4096.
 * The kernel draws its BF16 normals by inverse CDF from it (12 index bits + 1 sign bit of a Philox half-word each). */
int me_k4_normal_table(uint16_t *out, int32_t n);
int me_k4_get_counters(me_k4 *eng, int64_t *n_measure, uint64_t *step);
const char *me_k4_last_error(me_k4 *eng);

/* Measurement aid (no reference counterpart): FP64 FMA throughput probe used as the roofline denominator of the
 * step kernels.  Launches n_sm*8 CTAs of 256 threads, 8 independent FMA streams each, `iters` iterations;
 * out needs n_sm*8*256 doubles; *flops receives the flop count of the launch.  Time it with CUDA events. */
int me_probe_fp64(int32_t device, int64_t iters, double *out, int64_t out_len, void *stream, int64_t *flops);

/* Statistical inefficiency g (pymbar's definition, reference statistics.py:36-38,46 via metropolis_engine.py:490)
 * of column `col` of a time-series block ts[row][cols][ld] for chains [chain0, chain0 + n_sel), using rows
 * [row0, rows); the autocorrelation sum stops at the first non-positive term or at max_lag (<= 0: no cap).
 * g_out[n_sel].  ESS = N / g.  SURVEY.md §8 row f3 / metric "ESS/sec". */
int me_statistical_inefficiency(const double *ts, int64_t rows, int64_t row0, int32_t cols, int64_t ld, int32_t col,
                                int64_t chain0, int64_t n_sel, int64_t max_lag, double *g_out, void *stream);

/* Equilibration detection (SURVEY.md §8 row f3): for chains [chain0, chain0 + n_sel) and column `col` of the block
 * ts[row][cols][ld], the start t0 of the production region, its statistical inefficiency g and
 * Neff_max = max_t0 (rows - t0 + 1) / g(t0) over t0 in range(0, rows - 1, nskip) — what the reference's
 * save_equilibrium_stats (metropolis_engine.py:481-504) obtains per data-frame column from
 * pymbar.timeseries.detectEquilibration through statistics.get_equilibration_points (statistics.py:25-48).
 * fast != 0: pymbar's growing lag increments (its default inside detectEquilibration).  scratch needs
 * 2 * ceil((rows - 1) / nskip) * n_sel doubles.  t_out / g_out / neff_out: [n_sel] doubles. */
int me_detect_equilibration(const double *ts, int64_t rows, int32_t cols, int64_t ld, int32_t col, int64_t chain0,
                            int64_t n_sel, int64_t nskip, int32_t fast, double *scratch, int64_t scratch_doubles,
                            double *t_out, double *g_out, double *neff_out, void *stream);

/* MBAR over recorded rows (Shirts & Chodera, J. Chem. Phys. 129, 124105, 2008; pymbar's MBAR): one pass of the
 * multistate Bennett acceptance ratio over the time-series rows [row0, rows) of one storage chunk ts[row][TS_COLS][n_chains]
 * of this handle, every stride-th row, every local chain.  Sample n = (row, chain) was drawn at rung
 * (chain_offset + chain) % R (R = 1 for a handle without a ladder); every rung has the same count N = n_per_state (the
 * global count: samples of all chunks and all ranks / R).  States: the R rungs (temps[r], the rung's constants, or the
 * handle's constants on a temperature ladder; the handle's temp when R = 1) followed by n_target targets
 * (target_temps[t], target_consts[t][K] with K the functor's constant count; target_consts = NULL: the handle's constants,
 * not allowed on a Hamiltonian ladder); S = R + n_target <= 32.  u_s(x) = E(x; k_s) / T_s is re-evaluated from the stored
 * x columns with the handle's device functor (wall first: a walled x has weight 0 in state s).  Given f[R] (device,
 * reduced free energies of the rungs; the targets take f = 0):
 *     L_n  = ln sum_k N exp(f_k - u_k(x_n)),   w_ns = exp(f_s - u_s(x_n) - L_n)
 * and the pass writes (accumulate = 0) or adds (accumulate != 0: a series kept in several chunks is passed chunk by chunk)
 * the fixed-order sums
 *     sums[0] = sum_n L_n,  sums[1] = samples with a NaN energy or a non-finite L_n,  sums[2] = samples whose target
 *     weight exceeds 1e140 (a target without overlap) — such samples enter no other sum;
 *     then s[S] (s_s = sum_n w_ns), then G lower-packed (G_st = sum_n w_ns w_nt at s(s+1)/2 + t, t <= s),
 *     then, with_obs != 0, per state s: sum_n w_ns [x_0..x_{D-1}, x_0^2..x_{D-1}^2, E_s(x_n), E_s(x_n)^2].
 * me_mbar_words gives the length.  The sums are plain FP64 sums: across ranks they all-reduce as they are
 * (me_comm_allreduce).  One pass is bit-identical from run to run on one device.
 * Finishing the computation on the host (S x S algebra, what metropolisengine_b200/mbar.py does):
 *     objective F(f) = sum L - N sum_k f_k (convex), gradient g_i = N (s_i - 1), Hessian H_ij = delta_ij N s_i - N^2 G_ij;
 *     gauge f_0 = 0; Newton on f_1..f_{R-1} from f = 0 with a backtracking line search on F (one pass per trial point),
 *     until max |s_i - 1| < tol; if the reduced Hessian is not positive definite, f_i <- f_i - ln s_i.
 *     Targets: f_t = -ln s_t;  <a>_t = (sum_n w_nt a_t) / s_t.
 *     Uncertainties (pymbar "svd-ew", uncorrelated samples: take stride ~ the statistical inefficiency of the E column):
 *     G = V Sigma^2 V^T,  Theta = V Sigma (I - Sigma V^T diag(N_s) V Sigma)^+ Sigma V^T with N_s = 0 for targets,
 *     d(f_j - f_i) = sqrt(Theta_ii + Theta_jj - 2 Theta_ij).
 * ME_ERR_INVALID (with a message): more than 32 rungs or states, a rung or target temperature not finite or not > 0,
 * non-finite constants, targets of a Hamiltonian ladder without target_consts, row0 outside [0, rows), stride < 1,
 * n_per_state < 1, null pointers.  ME_ERR_UNSUPPORTED: D > 32, caller-evaluated energies, group / magnitude-phase modes.
 * Arguments are checked before any device work. */
int me_mbar_words(me_engine *eng, int32_t n_target, int32_t with_obs, int64_t *words);
int me_mbar_pass(me_engine *eng, const double *ts, int64_t rows, int64_t row0, int64_t stride, const double *f,
                 int64_t n_per_state, int32_t n_target, const double *target_temps, const double *target_consts,
                 int32_t with_obs, double *sums, int32_t accumulate, void *stream);

/* MBAR free-energy profiles (pymbar's histogram FES: pymbar 4 FES, pymbar 3 computePMF): one histogram pass over the
 * samples of me_mbar_pass (rows [row0, rows) of one storage chunk, every stride-th row, every local chain) with its
 * weights at the rungs' f[R] (device):
 *     L_n = ln sum_k N exp(f_k - u_k(x_n)),  w_nt = exp(-u_t(x_n) - L_n),  w_nk = exp(f_k - u_k(x_n) - L_n)
 * for one target state t = (target_temp, target_consts[K]; NULL: the handle's constants, not allowed on a Hamiltonian
 * ladder).  A walled x has u = +inf.  Samples with a NaN energy or a non-finite L_n count in n_nan, samples whose
 * target weight exceeds 1e140 in n_overflow; neither enters a sum.
 * Coordinates: n_axes in {1, 2}; axis a is stored parameter column coord_index[a] in [0, D) (order real, Re c, Im c)
 * when coord_kind[a] = 0, or the modulus |c_j| = sqrt(Re c_j^2 + Im c_j^2) of complex parameter j = coord_index[a] in
 * [0, n_complex) when coord_kind[a] = 1.  Uniform bins on [lo[a], hi[a]) (finite, hi > lo), n_bins[a] >= 1:
 *     i = floor((c - lo) * inv_w),  inv_w = n / (hi - lo) rounded once;  in range iff lo <= c < hi (NaN is not);
 *     i = n becomes n - 1;  bin b = i_0 n_bins[1] + i_1 in 2-D;  B = prod n_bins.
 * The coordinate, modulus and index are computed with round-to-nearest operations (no FMA contraction), so every
 * sample falls in the same bin in both builds and in a restatement in IEEE FP64.
 * Sums (accumulate = 0: written; != 0: added), words = 4 + B (R + 2) (me_mbar_hist_words):
 *     sums[0] = n_nan, sums[1] = n_overflow, sums[2] = w_out = sum of w_nt over out-of-range samples, sums[3] = their
 *     count, then per bin b: h_b = sum_{n in b} w_nt, q_b = sum_{n in b} w_nt^2, c_bk = sum_{n in b} w_nt w_nk (k < R).
 * Plain FP64 sums: chunks accumulate and ranks all-reduce them as they are.  A pass is bit-identical from run to run on
 * one device.  B (R + 2) <= 24576.
 * Finishing on the host (metropolisengine_b200/mbar.py, pmf): f_b = -ln h_b reported as f_b - f_ref;
 * p_b = h_b / (sum h + w_out); uncertainties from Theta (me_mbar_pass) of the augmented Gram matrix over the R rungs
 * and the non-empty bins: G_RR = the rungs' G at the solution, G_bk = c_bk / h_b, G_bb = q_b / h_b^2, G_bb' = 0, with
 * N = [N .. N, 0 .. 0]: df_b = sqrt(Theta_bb + Theta_rr - 2 Theta_br) against the reference bin r (the lowest f, or a
 * given bin).  An empty bin has f = +inf and df = NaN and stays out of Theta.
 * ME_ERR_INVALID (with a message): n_axes not 1 or 2, an unknown coord_kind, a column outside [0, D) or a modulus index
 * outside [0, n_complex), non-finite lo or hi or hi <= lo, n_bins < 1 or B (R + 2) > 24576, a target temperature not
 * finite or not > 0, non-finite constants, no target_consts on a Hamiltonian ladder, the row0 / stride / n_per_state
 * rules and null pointers of me_mbar_pass.  ME_ERR_UNSUPPORTED as me_mbar_pass.  Arguments are checked before any
 * device work. */
int me_mbar_hist_words(me_engine *eng, int32_t n_axes, const int32_t *n_bins, int64_t *words);
int me_mbar_hist_pass(me_engine *eng, const double *ts, int64_t rows, int64_t row0, int64_t stride, const double *f,
                      int64_t n_per_state, double target_temp, const double *target_consts, int32_t n_axes,
                      const int32_t *coord_kind, const int32_t *coord_index, const double *lo, const double *hi,
                      const int32_t *n_bins, double *sums, int32_t accumulate, void *stream);

/* MBAR expectation uncertainties (pymbar's compute_expectations covariance): one covariance pass over the samples and
 * weights of me_mbar_pass (the same rows, rungs, targets, f[R] and S = R + n_target <= 32 states)
 *     w_ns = exp(f_s - u_s(x_n) - L_n)
 * for the covered states s in [cov_first, cov_first + cov_count) of those S.  The observables of state s are the ones
 * me_mbar_pass averages, a_s = [x_0..x_{D-1}, x_0^2..x_{D-1}^2, E_s, E_s^2] (m = 2D + 2), taken about host-given
 * centres: a~ = a_s - c_s with centers[c][m] (device) for covered state c = s - cov_first.  Samples with a NaN energy or
 * a non-finite L_n count in n_nan, samples whose target weight exceeds 1e140 in n_overflow; neither enters a sum.
 * Sums (accumulate = 0: written; != 0: added), words = 2 + cov_count (m + m (R + 1) + m (m + 1) / 2)
 * (me_mbar_cov_words):
 *     sums[0] = n_nan, sums[1] = n_overflow, then per covered state s:
 *     o[m]          o_a = sum_n w_ns a~_a
 *     C[m][R + 1]   C_ak = sum_n w_ns a~_a w_nk for the rungs k < R, then C_a* = sum_n w_ns^2 a~_a
 *     Q[m(m+1)/2]   Q_ab = sum_n w_ns^2 a~_a a~_b, b <= a, lower-packed at a (a + 1) / 2 + b.
 * Plain FP64 sums: chunks accumulate and ranks all-reduce them as they are.  A pass is bit-identical from run to run on
 * one device.
 * Finishing on the host (metropolisengine_b200/mbar.py, expectation_covariance), with s_s and G from me_mbar_pass at the
 * same f: delta_a = o_a / s_s, <a>_s = c_a + delta_a; the centred column v_a = w_s (a - <a>_s) / s_s has the Gram entries
 *     G(v_a, k)   = (C_ak - delta_a G_sk) / s_s
 *     G(v_a, v_b) = (Q_ab - delta_a C_b* - delta_b C_a* + delta_a delta_b G_ss) / s_s^2
 * and Theta (me_mbar_pass) over [the R rungs, v_0 .. v_{m-1}] with N = [N .. N, 0 .. 0] gives
 * Cov(<a>_s, <b>_s) = Theta(v_a, v_b), for any centres (they only keep Q from cancelling when |<a>| >> std(a)).
 * Uncorrelated samples are assumed, as for the free-energy errors.
 * ME_ERR_INVALID (with a message): the rules of me_mbar_pass; cov_count < 1 or a range outside [0, S); null centers;
 * a range whose tiles and staging for one warp exceed the 227 KB of shared memory (a single state always fits, so
 * callers split the covered states into passes: me_mbar_cov_words applies the same check).  ME_ERR_UNSUPPORTED as
 * me_mbar_pass.  Arguments are checked before any device work. */
int me_mbar_cov_words(me_engine *eng, int32_t n_target, int32_t cov_first, int32_t cov_count, int64_t *words);
int me_mbar_cov_pass(me_engine *eng, const double *ts, int64_t rows, int64_t row0, int64_t stride, const double *f,
                     int64_t n_per_state, int32_t n_target, const double *target_temps, const double *target_consts,
                     int32_t cov_first, int32_t cov_count, const double *centers, double *sums, int32_t accumulate,
                     void *stream);

const char *me_last_error(me_engine *eng);   /* eng may be NULL: error of the last failing me_create */

#ifdef __cplusplus
}
#endif
#endif /* ME_B200_H */
