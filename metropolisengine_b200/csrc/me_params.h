/* me_params.h — plain-old-data launch parameters shared by the host library, the ahead-of-time kernels and the
 * NVRTC-compiled user-functor kernels.  Built-in types only (this text is also fed to NVRTC, which has no libc
 * headers).  Any change here changes the ABI between libme_b200.so and runtime-compiled kernels: bump
 * ME_PARAMS_VERSION. */
#ifndef ME_PARAMS_H
#define ME_PARAMS_H

#define ME_PARAMS_VERSION 12
#define ME_MAX_CONSTS 16

/* status bits written to the per-chain STATUS word (SURVEY §5 "failure detection") */
#define ME_STATUS_NOT_PSD 1      /* covariance lost positive-definiteness (reference: numpy raises, ME:270) */
#define ME_STATUS_SIGMA_NONPOS 2 /* sampling width <= 0 (reference: assert, ME:438) */
#define ME_STATUS_ENERGY_NAN 4   /* energy functor returned NaN */

struct MeParams {
    double *state;                 /* [WORDS][ld] chain-minor state block (layout: me_state_layout) */
    long long ld;                  /* leading dimension of every [..][chain] array = local chain capacity */
    long long n_chains;            /* chains owned by this launch (<= ld) */
    unsigned long long chain_offset; /* global id of local chain 0: Philox counters carry GLOBAL chain ids */
    unsigned long long seed;       /* Philox key */
    unsigned rk[20];               /* Philox round keys: rk[2r] = lo(seed) + r*0x9E3779B9, rk[2r+1] = hi(seed) + r*0xBB67AE85 */
    unsigned long long step0;      /* global index of the first step of this launch */
    long long n_blocks;            /* schedule: n_blocks x (spm steps [+ measure]) */
    long long spm;
    long long n_meas0;             /* measure_step_counter before this launch (reference starts at 1, ME:73) */
    int do_measure;
    int use_reject;
    int m;                         /* n_real + n_complex (ME:103) */
    int record;                    /* 1: store a time-series row at every measure */
    double temp, inv_temp;
    float t_ln2, t_band;           /* throughput build's FP32 threshold window (me_device.cuh, Rng::accept_window): T ln2 and
                                      the half-width 4e-5 T, see me_api.cu base_params */
    double target;                 /* target acceptance p* (ME:101) */
    double ratio;                  /* ME:105-107 */
    double consts[ME_MAX_CONSTS];  /* energy-functor constants */
    double *ts;                    /* time series [row][TSCOLS][ld]; row = ts_row0 + block index */
    long long ts_row0;
    const double *inj_delta;       /* parity mode: increments [step][D][ld] (NULL = Philox) */
    const double *inj_u;           /* parity mode: uniforms [step][ld], NaN = "reference drew none" */
    unsigned char *last_accept;    /* [ld] accept flag of the last step of the launch (may be NULL) */
    double *pool;                  /* [gridDim.x][POOLW] per-CTA pooled-moment accumulators (may be NULL) */
    const double *shift;           /* [D] shift vector of the pooled moments */
    /* unfused path (torch-callable energies) */
    double *prop;                  /* [D][ld] proposals */
    const double *e_new;           /* [ld] energies of the proposals */
    const unsigned char *rej;      /* [ld] hard-constraint mask (may be NULL) */
    /* initialisation */
    const double *x0;              /* [D][ld] or [D] when x0_broadcast */
    int x0_broadcast;
    int have_e0;                   /* 1: take initial energies from e_new instead of the functor */
    double sigma0;
    const double *cov_r0;          /* [NR*NR] row-major, shared by all chains (NULL = identity) */
    const double *cov_c0_re;       /* [NC*NC] */
    const double *cov_c0_im;
    /* generic (runtime-shape) kernels for large parameter spaces: me_generic.cu */
    int n_real, n_complex;
    int energy_id;                 /* built-in functor evaluated by gk_energy */
    double *scratch;               /* [D][ld] per-chain scratch (old means during measure) */
    double *e_out;                 /* [ld] gk_energy output */
    unsigned char *rej_out;        /* [ld] gk_energy hard-wall output (may be NULL) */
    int group;                     /* mixed engines: 0 = step_all (ME:241), 1 = step_real_group (ME:225), 2 = step_complex_group (ME:209),
                                      3 / 4 = magnitude / phase half of the magnitude-phase complex move (ME:178-207) */
    const unsigned long long *ctr_dev; /* unfused path under CUDA-graph replay: [0] index of the step, [1] measure counter,
                                      read by k_propose / k_accept INSTEAD of step0 / n_meas0 (kernel parameters are
                                      frozen at capture; NULL = use the parameters) */
    const double *logtab;          /* [1024][2] table of the table-driven log (me_math.cuh), device memory owned by the library */
    /* time segmentation of a launch with a work queue (me_device.cuh, run_body) */
    int seg_count;                 /* segments per chain group; <= 1: off */
    long long seg_groups;          /* chain groups; the launch has seg_groups x seg_count CTAs, one work item each */
    unsigned long long seg_base;   /* ring capacity (a power of two >= seg_groups x seg_count) */
    unsigned long long *seg_flags; /* queue: [0] tickets, [1] pushes, [2 .. 2 + capacity) ring; the host writes the initial
                                      image (segment 0 of every group ready) before the launch */
    /* temperature ladder (me_set_ladder; read by the PT instantiation of run_body only): global chain g is rung g % n_rungs */
    int n_rungs;
    long long swap_every;          /* replica-exchange round at every measure whose counter is a multiple; 0 = no swaps */
    const double *rung_temp;       /* [n_rungs] temperatures */
    const float *rung_window;      /* [n_rungs][2] t_ln2, t_band of each rung (the same expressions as the scalar ones) */
    int *walker;                   /* [ld] walker label of the configuration a chain holds */
    unsigned *swap_acc;            /* [ld] accepted swaps between this chain's rung and the next one up
                                      (pooled moments of a ladder: n_rungs rows of POOLW words per CTA, rung-major) */
    /* Hamiltonian ladder (me_set_hamiltonian_ladder; read by the HX instantiation of run_body and by init_body) */
    const double *rung_consts;     /* [n_rungs][n_consts] functor constants of each rung (NULL: consts on every chain) */
    int n_consts;                  /* K, 1 <= K <= ME_MAX_CONSTS */
};

#endif
