/* me_k4.cu — host side and the measure / pooled-moment / factor kernels of the shared-covariance path
 * (BASELINE config 4: cylinder-style Fourier-mode field, 1 real + n_c complex coefficients, n_c in {8, 16, 32, 64}).
 *
 * The step kernel is the warp-specialised tcgen05 pipeline of me_k4_device.cuh (ahead-of-time for the built-in cylinder
 * functor, NVRTC for user functors).  This file adds what happens at measure boundaries (reference measure()
 * metropolis_engine.py:342-356, covariance recursion ME:416-427 replaced by the POOLED covariance of all chains):
 *   k4_measure           per-chain running means / observable means / time-series row
 *   k4_moments_stage1/2  deterministic pooled moments as a symmetric rank-k update of Y = [Re c; Im c]
 *   k4_refactor          pooled covariance + sigma^2/n regulariser (ME:418,425) -> complex Cholesky -> BF16 UMMA operand
 */
#include <cuda_runtime.h>
#include <cuda.h>
#include <cuda_bf16.h>

#include <cstdint>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/me_b200.h"
#include "me_k4_device.cuh"
#include "me_rt.h"

namespace {

using k4::Layout;
using k4::StepParams;

constexpr int MAX_NC = 64;
constexpr int MAX_N = 2 * MAX_NC;

/* -------------------------------------------------------------------------------------------- step / init entry points */
template <int NC, class Energy, bool XP>
__global__ void __launch_bounds__(k4::THREADS, 1) k4_steps(const __grid_constant__ StepParams p,
                                                           const __grid_constant__ k4::TensorMap bmap) {
    k4::steps_body<NC, Energy, XP>(p, &bmap);
}
template <class Energy>
__global__ void k4_init(const __grid_constant__ StepParams p, const double *x0, int broadcast, double sigma0) {
    k4::init_body<Energy>(p, x0, broadcast, sigma0);
}

/* measure (ME:342-356 without the per-chain covariance, which is shared): running means (ME:404-410), observable
 * means (ME:412-414, 458-463), one time-series row [D params, E, sigma].  n = counter after the increment. */
struct MeasureParams {
    double *state;
    long long ld, n_chains, n_meas;
    int n_c;
    double *ts;
    long long ts_row;
    int record;
};
__global__ void k4_measure(MeasureParams p) {
    /* one thread per (slot, chain): slot j < n_c = complex mode j, slot n_c = real parameter + energy + sigma */
    const long long ch = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;
    if (ch >= p.n_chains) return;
    const long long ld = p.ld;
    const int nc = p.n_c;
    const Layout L(nc);
    const double dn = (double)p.n_meas, inv_n = 1.0 / dn, shrink = (dn - 1.0) * inv_n;
    double *row = p.record ? p.ts + p.ts_row * (long long)(L.D + 2) * ld + ch : nullptr;
    if (j == nc) {
        const double a = p.state[(long long)L.X * ld + ch];
        double *mp = &p.state[(long long)L.MEAN * ld + ch];
        *mp = fma(a, inv_n, *mp * shrink);
        double *o0 = &p.state[(long long)L.OBSM * ld + ch], *o1 = &p.state[(long long)(L.OBSM + 1 + nc) * ld + ch];
        *o0 = fma(fabs(a), inv_n, *o0 * shrink);
        *o1 = fma(a * a, inv_n, *o1 * shrink);
        if (row) {
            __stcs(row, a);
            __stcs(row + (long long)L.D * ld, p.state[(long long)L.E * ld + ch]);
            __stcs(row + (long long)(L.D + 1) * ld, p.state[(long long)L.SIG * ld + ch]);
        }
        return;
    }
    const double re = p.state[(long long)(L.X + 1 + j) * ld + ch];
    const double im = p.state[(long long)(L.X + 1 + nc + j) * ld + ch];
    double *mr = &p.state[(long long)(L.MEAN + 1 + j) * ld + ch];
    double *mi = &p.state[(long long)(L.MEAN + 1 + nc + j) * ld + ch];
    *mr = fma(re, inv_n, *mr * shrink);
    *mi = fma(im, inv_n, *mi * shrink);
    double *ob = &p.state[(long long)(L.OBSM + 1 + j) * ld + ch];
    *ob = fma(k4::cabs_fast(re, im), inv_n, *ob * shrink);
    if (row) {
        __stcs(row + (long long)(1 + j) * ld, re);
        __stcs(row + (long long)(1 + nc + j) * ld, im);
    }
}

/* Pooled moments of the current states, deterministic two-stage reduction (no atomics: the covariance feeds the
 * proposals, so run-to-run bit reproducibility needs a fixed summation order).
 *
 * With Y = [Re c; Im c] (N = 2 n_c rows) about the shift, everything the complex second moment needs is in the LOWER
 * triangle of the real symmetric S = sum_chains Y Y^T (N x N):
 *     Re (c c^H)_ij = S[i][j] + S[nc+i][nc+j],    Im (c c^H)_ij = S[nc+i][j] - S[nc+j][i]
 * — a rank-k update with half the flops of the full complex outer product.
 * Stage 1: CTA b sums its slice of chains.  Chains are staged 32 at a time in shared memory as Ys[k][row]; thread t < T
 *          (T = lower-triangle tiles of the N/8 x N/8 tile grid, 136 for N = 128) owns the 8 x 8 register tile (ti, tj),
 *          tj <= ti, of S; threads 136..255 keep the column sums of Y.
 *          part[b]: [0] chains, [1] sum sigma, [2] sum a, [3] sum a^2, [4..4+N) sum Y, [4+N..) S row-major (lower part).
 * Stage 2: fixed-order sum over the CTAs (2a), emitted in the complex layout the host accumulates (2b):
 *          out[MOMW] (double2): [0] chains, [1] sum sigma, [2] sum a, [3] sum a^2, [4..4+nc) sum c, [4+nc..) sum c c^H. */
constexpr int MOM_CHUNK = 32;
__host__ __device__ inline int momw(int nc) { return 4 + nc + nc * nc; }
__host__ __device__ inline int partw(int nc) { return 4 + 2 * nc + 4 * nc * nc; }

__global__ void __launch_bounds__(256) k4_moments_stage1(const double *state, long long ld, long long n_chains, int nc,
                                                         const double *shift, double *part, long long chains_per_cta) {
    /* Ys[k][pos(row)]: every block of 8 rows is followed by 2 pad doubles, so that the 16-byte reads of lanes that own
       neighbouring tiles (80 B apart) fall into distinct banks; the row length 162 keeps the staging stores (same
       row, consecutive k) at 4-way instead of 32-way conflicts. */
    constexpr int YLD = MAX_N + 2 * (MAX_N / 8) + 2;       /* 162 */
    __shared__ __align__(16) double Ys[MOM_CHUNK][YLD];   /* 41 KB */
    auto pos = [](int row) { return row + 2 * (row >> 3); };
    __shared__ double red[256];
    const int tid = threadIdx.x;
    const int N = 2 * nc, nt = N / 8, n_tiles = nt * (nt + 1) / 2;
    const Layout L(nc);
    const long long lo = (long long)blockIdx.x * chains_per_cta;
    long long hi = lo + chains_per_cta;
    if (hi > n_chains) hi = n_chains;
    /* tile of thread t < n_tiles: row-major enumeration of the lower triangle of the tile grid */
    int ti = 0, tj = 0;
    {
        int t = tid < n_tiles ? tid : 0;
        while (t > ti) { t -= ti + 1; ti++; }
        tj = t;
    }
    const bool tile_thread = tid < n_tiles;
    double acc[8][8];
#pragma unroll
    for (int a = 0; a < 8; a++)
#pragma unroll
        for (int b = 0; b < 8; b++) acc[a][b] = 0.0;
    const int r0 = tid - 136;                             /* column sums: rows r0 and r0 + 120 */
    double colsum = 0.0, colsum2 = 0.0;
    double sa = 0.0, sa2 = 0.0, ssig = 0.0;               /* threads < 32 */
    for (long long base = lo; base < hi; base += MOM_CHUNK) {
        const int cnt = (int)((hi - base) < MOM_CHUNK ? (hi - base) : MOM_CHUNK);
        __syncthreads();
        /* stage: consecutive threads read consecutive chains of one state word (coalesced), write Ys[k][row] */
        for (int e = tid; e < N * MOM_CHUNK; e += 256) {
            const int row = e / MOM_CHUNK, k = e % MOM_CHUNK;
            Ys[k][pos(row)] = k < cnt ? state[(long long)(L.X + 1 + row) * ld + base + k] - shift[1 + row] : 0.0;
        }
        if (tid < cnt) {
            const double a = state[(long long)L.X * ld + base + tid] - shift[0];
            sa += a; sa2 += a * a; ssig += state[(long long)L.SIG * ld + base + tid];
        }
        __syncthreads();
        if (tile_thread) {
#pragma unroll 4
            for (int k = 0; k < MOM_CHUNK; k++) {
                double ya[8], yb[8];
                const double2 *pa = reinterpret_cast<const double2 *>(&Ys[k][10 * ti]);     /* pos(8 ti) */
                const double2 *pb = reinterpret_cast<const double2 *>(&Ys[k][10 * tj]);
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const double2 va = pa[q], vb = pb[q];
                    ya[2 * q] = va.x; ya[2 * q + 1] = va.y; yb[2 * q] = vb.x; yb[2 * q + 1] = vb.y;
                }
#pragma unroll
                for (int a = 0; a < 8; a++)
#pragma unroll
                    for (int b = 0; b < 8; b++) acc[a][b] = fma(ya[a], yb[b], acc[a][b]);
            }
        } else if (tid >= 136) {
            if (r0 < N)
                for (int k = 0; k < MOM_CHUNK; k++) colsum += Ys[k][pos(r0)];
            if (r0 + 120 < N)
                for (int k = 0; k < MOM_CHUNK; k++) colsum2 += Ys[k][pos(r0 + 120)];
        }
    }
    double *out = part + (long long)blockIdx.x * partw(nc);
    if (tile_thread) {
#pragma unroll
        for (int a = 0; a < 8; a++)
#pragma unroll
            for (int b = 0; b < 8; b++) out[4 + N + (8 * ti + a) * N + (8 * tj + b)] = acc[a][b];
    }
    if (tid >= 136) {
        if (r0 < N) out[4 + r0] = colsum;
        if (r0 + 120 < N) out[4 + r0 + 120] = colsum2;
    }
    /* the three scalar sums: fixed-order trees */
    for (int which = 0; which < 3; which++) {
        __syncthreads();
        red[tid] = (tid < MOM_CHUNK) ? (which == 0 ? ssig : (which == 1 ? sa : sa2)) : 0.0;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) { if (tid < o) red[tid] += red[tid + o]; __syncthreads(); }
        if (tid == 0) out[1 + which] = red[0];
    }
    if (tid == 0) out[0] = (double)(hi > lo ? hi - lo : 0);
}

/* stage 2a: total[idx] = sum over the CTA partials in CTA order (one thread per word, coalesced across threads;
 * the upper triangle of S is never read, its threads idle) */
__global__ void k4_moments_stage2a(const double *part, int n_parts, double *total, int nc) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = 2 * nc, pw = partw(nc);
    if (idx >= pw) return;
    if (idx >= 4 + N) {
        const int e = idx - 4 - N;
        if (e / N < e % N) return;
    }
    /* loads in batches of 16 (independent), adds in CTA order (fixed summation order) */
    double t = 0.0;
    int b = 0;
    for (; b + 16 <= n_parts; b += 16) {
        double v[16];
#pragma unroll
        for (int q = 0; q < 16; q++) v[q] = part[(long long)(b + q) * pw + idx];
#pragma unroll
        for (int q = 0; q < 16; q++) t += v[q];
    }
    for (; b < n_parts; b++) t += part[(long long)b * pw + idx];
    total[idx] = t;
}
/* stage 2b: the complex layout the host accumulates.  Optionally (single-GPU fast path) the running moments are
 * advanced here, mom[w] += inc[w] for w != 1, and a snapshot [mom (MOMW) | inc[0], inc[1]] is written for a factor
 * refresh that runs asynchronously on another stream. */
__global__ void k4_moments_stage2b(const double *total, double2 *out, double2 *mom, double2 *snap, int nc) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = 2 * nc, mw = momw(nc);
    if (w >= mw) return;
    double2 v;
    if (w < 4) v = make_double2(total[w], 0.0);
    else if (w < 4 + nc) { const int i = w - 4; v = make_double2(total[4 + i], total[4 + nc + i]); }
    else {
        const int e = w - 4 - nc, i = e / nc, j = e % nc;
        auto S = [&](int r, int c) { return total[4 + N + (r >= c ? r * N + c : c * N + r)]; };   /* symmetric */
        v = make_double2(S(i, j) + S(nc + i, nc + j), S(nc + i, j) - S(nc + j, i));
    }
    out[w] = v;
    if (mom != nullptr) {
        double2 m = mom[w];
        if (w != 1) { m.x += v.x; m.y += v.y; mom[w] = m; }
        if (snap != nullptr) {
            snap[w] = m;
            if (w < 2) snap[mw + w] = v;
        }
    }
}

/* 1 / sqrt(d) for a normal positive d: MUFU.RSQ64H seed + two Newton steps (relative error ~1e-16) */
__device__ __forceinline__ double k4_rsqrt(double d) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
    double e = fma(-d, y * y, 1.0);
    y = fma(0.5 * y, e, y);
    e = fma(-d, y * y, 1.0);
    return fma(0.5 * y, e, y);
}

/* Pooled covariance -> shared proposal factor, one CTA (runs once per measure after the 50th, ME:389,396).
 * mom (complex, as double pairs): [0] sample count, [2] sum a, [3] sum a^2, [4..4+nc) sum c, [4+nc..) sum c c^H
 * (about a fixed shift); inc: [0] chains measured now, [1] sum of their sigma.  Computes
 *   C_c = (S2 - S1 S1^H / N)/(N-1) + small I,  small = mean(sigma)^2 / n   (the regulariser of ME:418,425),
 * its Cholesky factor G, the BF16 UMMA operand of the step kernel, and the same for the real parameter.
 * Cholesky: left-looking by columns, 4 threads per row splitting the dot product (fixed order + shuffle tree), two
 * barriers per column, pivot through one reciprocal square root.  status: nonzero if a pivot was not positive. */
__global__ void __launch_bounds__(256) k4_refactor(const double2 *mom, const double2 *inc, long long n_meas, int nc,
                                                   double2 *cov_c, double *cov_a, __nv_bfloat16 *factor, double *s_a,
                                                   int *status) {
    const int LDA = nc + 1;                              /* padded row length (double2) */
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    double2 *A = reinterpret_cast<double2 *>(smem_raw);  /* A[i * LDA + j] */
    __shared__ double2 col[MAX_NC];
    __shared__ int bad;
    const int tid = threadIdx.x, row = tid >> 2, part = tid & 3;
    const int N2 = 2 * nc;
    const double N = mom[0].x;
    const double sm = inc[1].x / inc[0].x;
    const double small = sm * sm / (double)n_meas;
    const double inv_n = 1.0 / N, inv_n1 = 1.0 / (N - 1.0);
    const double2 *s1 = mom + 4, *s2 = mom + 4 + nc;
    if (tid == 0) bad = 0;
    for (int e = tid; e < nc * nc; e += blockDim.x) {
        const int i = e / nc, j = e % nc;
        /* s1_i conj(s1_j) */
        const double pr = s1[i].x * s1[j].x + s1[i].y * s1[j].y, pi = s1[i].y * s1[j].x - s1[i].x * s1[j].y;
        double2 v;
        v.x = (s2[e].x - pr * inv_n) * inv_n1 + (i == j ? small : 0.0);
        v.y = (s2[e].y - pi * inv_n) * inv_n1;
        A[i * LDA + j] = v;
        cov_c[e] = v;
    }
    if (tid == 0) {
        const double va = (mom[3].x - mom[2].x * mom[2].x * inv_n) * inv_n1 + small;
        *cov_a = va;
        *s_a = sqrt(va);
    }
    __syncthreads();
    for (int j = 0; j < nc; j++) {
        /* v_i = A_ij - sum_{k<j} G_ik conj(G_jk), rows i >= j; the four parts of a row are adjacent lanes */
        double ar = 0.0, ai = 0.0;
        if (row >= j && row < nc) {
            for (int k = part; k < j; k += 4) {
                const double2 pq = A[row * LDA + k], q = A[j * LDA + k];
                ar = fma(pq.x, q.x, fma(pq.y, q.y, ar));
                ai = fma(pq.y, q.x, fma(-pq.x, q.y, ai));
            }
        }
        ar += __shfl_xor_sync(0xffffffffu, ar, 1); ai += __shfl_xor_sync(0xffffffffu, ai, 1);
        ar += __shfl_xor_sync(0xffffffffu, ar, 2); ai += __shfl_xor_sync(0xffffffffu, ai, 2);
        if (part == 0 && row >= j && row < nc) {
            const double2 a0 = A[row * LDA + j];
            col[row] = make_double2(a0.x - ar, a0.y - ai);
        }
        __syncthreads();
        double d = col[j].x;
        if (!(d > 0.0)) { if (tid == 0) bad = 1; d = small > 0.0 ? small : 1e-300; }
        const double inv = k4_rsqrt(d);
        if (part == 0 && row >= j && row < nc) {
            const double2 v = col[row];
            A[row * LDA + j] = row == j ? make_double2(d * inv, 0.0) : make_double2(v.x * inv, v.y * inv);
        }
        __syncthreads();
    }
    /* B[2i][2j] = Gr/sqrt2, B[2i][2j+1] = Gi/sqrt2, B[2i+1][2j] = -Gi/sqrt2, B[2i+1][2j+1] = Gr/sqrt2; stored
       BF16 at [k/8][n][k%8] */
    const double rs = 0.70710678118654752440;
    for (int e = tid; e < N2 * N2; e += blockDim.x) {
        const int nrow = e / N2, k = e % N2;
        const int i = nrow >> 1, jj = k >> 1;
        double v = 0.0;
        if (jj <= i) {
            const double2 gij = A[i * LDA + jj];
            const bool ro = nrow & 1, ko = k & 1;
            v = (ro == ko) ? gij.x : (ro ? -gij.y : gij.y);
            if (jj == i && ro != ko) v = 0.0;       /* diagonal of G is real */
        }
        factor[(k >> 3) * (N2 * 8) + nrow * 8 + (k & 7)] = __double2bfloat16(v * rs);
    }
    if (tid == 0 && status) *status = bad;
}

/* The generator's table (me_k4_device.cuh): BF16 bits of Phi^-1(1/2 + (i + 1/2) / 8192), i < 4096, by bisection on erfc
 * (monotone, no series to trust), rounded to nearest even.  Host copy + one device copy per device for the process. */
const unsigned short *k4_host_ztab() {
    static unsigned short tab[k4::ZTAB_ENTRIES];
    static std::once_flag once;
    std::call_once(once, [] {
        for (int i = 0; i < k4::ZTAB_ENTRIES; i++) {
            const double pr = 0.5 + ((double)i + 0.5) / (2.0 * k4::ZTAB_ENTRIES);
            double lo = 0.0, hi = 8.0;
            for (int it = 0; it < 200; it++) {
                const double mid = 0.5 * (lo + hi);
                if (mid == lo || mid == hi) break;
                if (0.5 * erfc(-mid * 0.70710678118654752440) < pr) lo = mid; else hi = mid;
            }
            const float f = (float)(0.5 * (lo + hi));
            unsigned int b;
            memcpy(&b, &f, 4);
            b += 0x7fffu + ((b >> 16) & 1u);
            tab[i] = (unsigned short)(b >> 16);
        }
    });
    return tab;
}
const unsigned short *k4_device_ztab(int device) {
    static std::mutex mu;
    static std::map<int, unsigned short *> tabs;
    std::lock_guard<std::mutex> lock(mu);
    auto it = tabs.find(device);
    if (it != tabs.end()) return it->second;
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(device);
    unsigned short *dev = nullptr;
    const size_t bytes = sizeof(unsigned short) * k4::ZTAB_ENTRIES;
    if (cudaMalloc((void **)&dev, bytes) != cudaSuccess ||
        cudaMemcpy(dev, k4_host_ztab(), bytes, cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaGetLastError();
        dev = nullptr;
    }
    if (prev >= 0) cudaSetDevice(prev);
    if (dev) tabs[device] = dev;
    return dev;
}

/* ahead-of-time step kernels for the built-in functor */
/* steps_xp: the instantiation that parks the proposed state in TMEM (me_k4_device.cuh) — launches without a measure tail
   and CTAs of a single tile */
struct AotEntry { int nc; const void *steps, *steps_xp; int smem; };
template <int NC> AotEntry aot_entry() {
    return AotEntry{NC, (const void *)&k4_steps<NC, k4::EnergyCylinder, false>,
                    (const void *)&k4_steps<NC, k4::EnergyCylinder, true>, (int)sizeof(k4::Smem<NC>)};
}

}  // namespace

/* ============================================================================================ C ABI */
struct me_k4 {
    me_k4_config cfg;
    int nc = 64;
    double consts[ME_MAX_CONSTS];
    int use_reject = 0;
    double *state = nullptr;
    const void *factor = nullptr;
    const unsigned short *ztab = nullptr;   /* generator table on cfg.device (owned by the library) */
    unsigned char *last_accept = nullptr;
    long long n_measure = 1;
    unsigned long long step = 0;
    int n_sm = 148;
    int reserved_sms = 0;          /* SMs the step kernel leaves free (for a concurrent factor refresh) */
    bool no_tma = false;           /* the driver has no cuTensorMapEncodeTiled */
    /* step / init kernels: ahead-of-time (built-in functor) or runtime-compiled (user functor) */
    const void *steps_rt = nullptr, *steps_xp_rt = nullptr, *init_rt = nullptr;
    CUfunction steps_drv = nullptr, init_drv = nullptr;
    int steps_smem = 0;
    std::string err;
};

static std::string g_k4_create_error;
static int k4_fail(me_k4 *e, int code, const std::string &msg) {
    if (e) e->err = msg; else g_k4_create_error = msg;
    return code;
}

static void k4_base(me_k4 *e, StepParams &p) {
    memset(&p, 0, sizeof(p));
    p.state = e->state;
    p.ld = e->cfg.n_chains;
    p.n_chains = e->cfg.n_chains;
    p.chain_offset = (unsigned long long)e->cfg.chain_offset;
    for (int r = 0; r < 10; r++) {
        p.rk[2 * r] = (unsigned)e->cfg.seed + (unsigned)r * 0x9E3779B9u;
        p.rk[2 * r + 1] = (unsigned)(e->cfg.seed >> 32) + (unsigned)r * 0xBB67AE85u;
    }
    p.step0 = e->step;
    p.n_meas = e->n_measure;
    p.temp = e->cfg.temp;
    p.inv_temp = e->cfg.temp != 0 ? 1.0 / e->cfg.temp : 0.0;
    p.target = e->cfg.target_acceptance;
    p.ratio = e->cfg.ratio;
    p.m = 1 + e->nc;
    p.n_c = e->nc;
    memcpy(p.consts, e->consts, sizeof(p.consts));
    p.use_wall = e->use_reject;
    p.factor = e->factor;
    p.ztab = e->ztab;
    p.last_accept = e->last_accept;
}

static bool k4_valid_nc(int nc) { return nc == 8 || nc == 16 || nc == 32 || nc == 64; }

static int k4_bind_builtin(me_k4 *e) {
    AotEntry t;
    switch (e->nc) {
    case 8: t = aot_entry<8>(); break;
    case 16: t = aot_entry<16>(); break;
    case 32: t = aot_entry<32>(); break;
    default: t = aot_entry<64>(); break;
    }
    e->steps_rt = t.steps; e->steps_xp_rt = t.steps_xp; e->steps_smem = t.smem; e->steps_drv = nullptr;
    e->init_rt = (const void *)&k4_init<k4::EnergyCylinder>; e->init_drv = nullptr;
    return ME_OK;
}

extern "C" {

int me_k4_layout_for(int32_t nc, me_k4_layout *o) {
    if (!o || !k4_valid_nc(nc)) return ME_ERR_INVALID;
    const Layout L(nc);
    o->X = L.X; o->E = L.E; o->SIG = L.SIG; o->MEAN = L.MEAN; o->OBSM = L.OBSM; o->NACC = L.NACC;
    o->STATUS = L.STATUS; o->WORDS = L.WORDS; o->D = L.D; o->TS_COLS = L.D + 2; o->N_COMPLEX = nc;
    o->TILE = k4::TILE; o->FACTOR_BYTES = 4 * nc * nc * 2; o->MOM_WORDS = momw(nc);
    o->MOM_SCRATCH_PER_SM = partw(nc);
    o->SUM_GROUPS = k4::EPI_GROUPS;
    return ME_OK;
}
int me_k4_layout_get(me_k4_layout *o) { return me_k4_layout_for(64, o); }

int me_k4_create(const me_k4_config *cfg, me_k4 **out) {
    if (!cfg || !out) return k4_fail(nullptr, ME_ERR_INVALID, "null argument");
    if (cfg->n_real != 1 || !k4_valid_nc(cfg->n_complex))
        return k4_fail(nullptr, ME_ERR_UNSUPPORTED, "the shared-covariance tensor-core path serves 1 real + 8 / 16 / 32 / 64 "
                                                    "complex parameters");
    if (cfg->n_chains <= 0 || cfg->n_chains % k4::TILE != 0)
        return k4_fail(nullptr, ME_ERR_INVALID, "n_chains must be a positive multiple of 128 (one MMA tile = 128 chains)");
    if (!(cfg->temp >= 0)) return k4_fail(nullptr, ME_ERR_INVALID, "temp must be >= 0 (reference: assert, ME:92)");
    me_k4 *e = new me_k4();
    e->cfg = *cfg;
    e->nc = cfg->n_complex;
    memset(e->consts, 0, sizeof(e->consts));
    for (int i = 0; i < 4; i++) e->consts[i] = cfg->consts[i];
    e->use_reject = cfg->use_reject;
    int n_sm = 0;
    if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, cfg->device) == cudaSuccess && n_sm > 0) e->n_sm = n_sm;
    else cudaGetLastError();
    k4_bind_builtin(e);
    *out = e;
    return ME_OK;
}

int me_k4_destroy(me_k4 *e) { delete e; return ME_OK; }

/* User energy functor for the shared-covariance path (the plugin surface, ME:20, 110-120): CUDA text defining
 *   __device__ void   me_k4_mode(double q, double re, double im, const double *k, double &s0, double &s1);
 *   __device__ double me_k4_total(double a, double s0, double s1, const double *k, int n_c);
 *   __device__ bool   me_k4_reject(double a, const double *k);          (only when use_reject != 0)
 * compiled for sm_100a with NVRTC into the same warp-specialised step kernel. */
int me_k4_set_energy_source(me_k4 *e, const char *src, const double *consts, int32_t n_consts, int32_t use_reject) {
    if (!e || !src) return ME_ERR_INVALID;
    if (n_consts < 0 || n_consts > ME_MAX_CONSTS) return k4_fail(e, ME_ERR_INVALID, "at most 16 functor constants");
    std::string text = "#include \"me_k4_device.cuh\"\n#line 1 \"user_k4_energy.cu\"\n";
    text += src;
    text += "\nstruct K4UserEnergy {\n"
            "  __device__ __forceinline__ static void mode(double q, double re, double im, const double *k, double &s0, double &s1) {\n"
            "    me_k4_mode(q, re, im, k, s0, s1); }\n"
            "  __device__ __forceinline__ static double total(double a, double s0, double s1, const double *k, int nc) {\n"
            "    return me_k4_total(a, s0, s1, k, nc); }\n"
            "  __device__ __forceinline__ static bool reject(double a, const double *k) {\n";
    text += use_reject ? "    return me_k4_reject(a, k); }\n" : "    return false; }\n";
    text += "};\n"
            "extern \"C\" __global__ void __launch_bounds__(k4::THREADS, 1) me_k4_steps(const __grid_constant__ k4::StepParams p,\n"
            "    const __grid_constant__ k4::TensorMap bmap) { k4::steps_body<ME_K4_NC, K4UserEnergy>(p, &bmap); }\n"
            "extern \"C\" __global__ void me_k4_init(const __grid_constant__ k4::StepParams p, const double *x0, int broadcast,\n"
            "    double sigma0) { k4::init_body<K4UserEnergy>(p, x0, broadcast, sigma0); }\n";
    std::vector<std::string> opts = {"-DME_K4_NC=" + std::to_string(e->nc)};
    std::vector<char> cubin;
    std::string log;
    int rc = me_rt_compile(text, "me_k4_user.cu", opts, cubin, log);
    if (rc != ME_OK) return k4_fail(e, rc, log);
    const char *names[2] = {"me_k4_steps", "me_k4_init"};
    CUfunction fn[2] = {nullptr, nullptr};
    rc = me_rt_load(e->cfg.device, cubin, names, 2, fn, log);
    if (rc != ME_OK) return k4_fail(e, rc, log);
    size_t smem = 0;
    switch (e->nc) {
    case 8: smem = sizeof(k4::Smem<8>); break;
    case 16: smem = sizeof(k4::Smem<16>); break;
    case 32: smem = sizeof(k4::Smem<32>); break;
    default: smem = sizeof(k4::Smem<64>); break;
    }
    rc = me_rt_set_dynamic_smem(fn[0], (int)smem, log);
    if (rc != ME_OK) return k4_fail(e, rc, log);
    e->steps_drv = fn[0]; e->init_drv = fn[1]; e->steps_rt = e->steps_xp_rt = e->init_rt = nullptr; e->steps_smem = (int)smem;
    memset(e->consts, 0, sizeof(e->consts));
    for (int i = 0; i < n_consts; i++) e->consts[i] = consts[i];
    e->use_reject = use_reject ? 1 : 0;
    return ME_OK;
}

/* compile-only check of a shared-covariance functor (works without a GPU) */
int me_k4_check_energy_source(const char *src, int32_t nc, int32_t use_reject, char *log, int64_t cap) {
    if (!src || !k4_valid_nc(nc)) return ME_ERR_INVALID;
    std::string text = "#include \"me_k4_device.cuh\"\n#line 1 \"user_k4_energy.cu\"\n";
    text += src;
    text += "\nstruct K4UserEnergy {\n"
            "  __device__ __forceinline__ static void mode(double q, double re, double im, const double *k, double &s0, double &s1) {\n"
            "    me_k4_mode(q, re, im, k, s0, s1); }\n"
            "  __device__ __forceinline__ static double total(double a, double s0, double s1, const double *k, int nc) {\n"
            "    return me_k4_total(a, s0, s1, k, nc); }\n"
            "  __device__ __forceinline__ static bool reject(double a, const double *k) {\n";
    text += use_reject ? "    return me_k4_reject(a, k); }\n" : "    return false; }\n";
    text += "};\n"
            "extern \"C\" __global__ void __launch_bounds__(k4::THREADS, 1) me_k4_steps(const __grid_constant__ k4::StepParams p,\n"
            "    const __grid_constant__ k4::TensorMap bmap) { k4::steps_body<ME_K4_NC, K4UserEnergy>(p, &bmap); }\n";
    std::vector<std::string> opts = {"-DME_K4_NC=" + std::to_string(nc)};
    std::vector<char> cubin;
    std::string l;
    const int rc = me_rt_compile(text, "me_k4_user.cu", opts, cubin, l);
    if (log && cap > 0) {
        strncpy(log, l.c_str(), (size_t)cap - 1);
        log[cap - 1] = 0;
    }
    return rc;
}

int me_k4_bind(me_k4 *e, double *state, const void *factor_bf16, unsigned char *last_accept) {
    if (!e || !state || !factor_bf16) return ME_ERR_INVALID;
    e->state = state; e->factor = factor_bf16; e->last_accept = last_accept;
    if (!e->ztab) {
        e->ztab = k4_device_ztab(e->cfg.device);
        if (!e->ztab) return k4_fail(e, ME_ERR_CUDA, "allocating the generator table failed");
    }
    return ME_OK;
}

int me_k4_set_factor(me_k4 *e, const void *factor_bf16) {
    if (!e || !factor_bf16) return ME_ERR_INVALID;
    e->factor = factor_bf16;
    return ME_OK;
}

int me_k4_set_reserved_sms(me_k4 *e, int32_t n) {
    if (!e || n < 0) return ME_ERR_INVALID;
    e->reserved_sms = n;
    return ME_OK;
}

int me_k4_init(me_k4 *e, const double *x0, int32_t broadcast, double sigma0, void *stream) {
    if (!e || !e->state || !x0) return ME_ERR_INVALID;
    StepParams p;
    k4_base(e, p);
    int prev = -1; cudaGetDevice(&prev); cudaSetDevice(e->cfg.device);
    const int block = 128, grid = (int)((e->cfg.n_chains + block - 1) / block);
    int rc = ME_OK;
    std::string err;
    int bc = broadcast;
    void *args[] = {&p, (void *)&x0, &bc, &sigma0};
    if (e->init_drv) {
        rc = me_rt_launch(e->init_drv, grid, block, 0, stream, args, err);
    } else {
        cudaError_t ce = cudaLaunchKernel(e->init_rt, dim3(grid), dim3(block), args, 0, (cudaStream_t)stream);
        if (ce != cudaSuccess) { rc = ME_ERR_CUDA; err = cudaGetErrorString(ce); }
    }
    cudaSetDevice(prev);
    e->n_measure = 1; e->step = 0;
    if (rc != ME_OK) return k4_fail(e, rc, "k4_init: " + err);
    return ME_OK;
}

/* one launch of the step kernel; `tail` != nullptr adds the fused measure (see StepParams) */
struct K4Tail { double *ts; long long ts_row; const double *shift; double *mom_part; };
static int k4_launch_steps(me_k4 *e, int64_t n_steps, const double *s_a, float *dbg_z, float *dbg_delta, double *dbg_scal,
                           const K4Tail *tail, int *grid_out, void *stream) {
    const int avail = e->n_sm - e->reserved_sms > 0 ? e->n_sm - e->reserved_sms : 1;
    int rc = ME_OK;
    std::string err;
    StepParams p;
    k4_base(e, p);
    p.n_steps = n_steps; p.s_a = s_a; p.dbg_z = dbg_z; p.dbg_delta = dbg_delta; p.dbg_scal = dbg_scal;
    if (tail) {
        p.do_measure = 1; p.record = tail->ts != nullptr; p.n_meas_after = e->n_measure + 1;
        p.ts = tail->ts; p.ts_row = tail->ts_row; p.shift = tail->shift; p.mom_part = tail->mom_part;
    }
    long long per = (e->cfg.n_chains + avail - 1) / avail;
    per = (per + 31) / 32 * 32;
    /* (whole tiles per CTA — 32,768 chains as 128 CTAs x 2 full tiles, leaving 20 SMs to the side stream — were measured:
       88.4 us per 10 steps against 85.9 us for 147 CTAs x (128 + 96): a partly filled tile is faster than a full one) */
    p.chains_per_cta = per;
    const int grid = (int)((e->cfg.n_chains + per - 1) / per);
    if (grid_out) *grid_out = grid;
    /* tensor map of the factor: rows of 16 bytes, [K/8 chunks x N rows][8 bf16] */
    k4::TensorMap bmap;
    memset(&bmap, 0, sizeof(bmap));
    p.use_tma = 0;
    if (!e->no_tma) {
        const int N = 2 * e->nc, rows = (N / 8) * N;
        if (me_rt_tensor_map_2d_bf16(&bmap, e->factor, 8, rows, 8, rows < 256 ? rows : 256) == ME_OK) p.use_tma = 1;
        else e->no_tma = true;                 /* driver without tensor maps: plain staging from now on */
    }
    void *args[] = {&p, &bmap};
    if (e->steps_drv) {
        rc = me_rt_launch(e->steps_drv, grid, k4::THREADS, e->steps_smem, stream, args, err);
    } else {
        /* the attribute is per device: set it before every launch (a host-side table write, no device work) */
        /* ME_K4_XP=0 / 1 forces one instantiation (tests, probes) */
        const char *force = getenv("ME_K4_XP");
        const bool xp = e->steps_xp_rt != nullptr && (force ? force[0] == '1' : (tail == nullptr || per <= k4::TILE));
        const void *kern = xp ? e->steps_xp_rt : e->steps_rt;
        cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, e->steps_smem);
        if (ce == cudaSuccess)
            ce = cudaLaunchKernel(kern, dim3(grid), dim3(k4::THREADS), args, (size_t)e->steps_smem, (cudaStream_t)stream);
        if (ce != cudaSuccess) { rc = ME_ERR_CUDA; err = cudaGetErrorString(ce); }
    }
    if (rc != ME_OK) return k4_fail(e, rc, "k4_steps: " + err);
    return ME_OK;
}

int me_k4_step(me_k4 *e, int64_t n_steps, const double *s_a, float *dbg_z, float *dbg_delta, double *dbg_scal, void *stream) {
    if (!e || !e->state || !s_a) return ME_ERR_INVALID;
    if (n_steps <= 0) return ME_OK;
    if (e->step + (unsigned long long)n_steps >= 0xffffffffull) return k4_fail(e, ME_ERR_INVALID, "step counter overflow");
    int prev = -1; cudaGetDevice(&prev); cudaSetDevice(e->cfg.device);
    const int rc = k4_launch_steps(e, n_steps, s_a, dbg_z, dbg_delta, dbg_scal, nullptr, nullptr, stream);
    cudaSetDevice(prev);
    if (rc != ME_OK) return rc;
    e->step += (unsigned long long)n_steps;
    return ME_OK;
}

static void k4_moments_finish(me_k4 *e, double *scratch, int n_parts, double *inc, double *mom_accum, double *snapshot,
                              void *stream) {
    const int nc = e->nc, pw = partw(nc), mw = momw(nc);
    double *total = scratch + (long long)n_parts * pw;
    k4_moments_stage2a<<<(pw + 127) / 128, 128, 0, (cudaStream_t)stream>>>(scratch, n_parts, total, nc);
    k4_moments_stage2b<<<(mw + 127) / 128, 128, 0, (cudaStream_t)stream>>>(total, reinterpret_cast<double2 *>(inc),
                                                                       reinterpret_cast<double2 *>(mom_accum),
                                                                       reinterpret_cast<double2 *>(snapshot), nc);
}

/* multi-GPU: after the all-reduce of `inc` (me_comm_allreduce) the running moments advance and the snapshot for the
 * factor refresh is written — what stage 2b does by itself on one GPU */
__global__ void k4_moments_accumulate(const double2 *inc, double2 *mom, double2 *snap, int mw) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= mw) return;
    const double2 v = inc[w];
    double2 m = mom[w];
    if (w != 1) { m.x += v.x; m.y += v.y; mom[w] = m; }
    snap[w] = m;
    if (w < 2) snap[mw + w] = v;
}

/* n_steps x step_all() + measure() in ONE launch of the step kernel, then the two small reduction kernels of the pooled
 * moments: the block a sampling loop repeats (ME README loop: step_all x k, measure).  The per-chain measurement is the
 * one of me_k4_measure bit for bit; the second moments S = sum Y Y^T are formed on the tensor cores from Y split into two
 * BF16 words (relative error of a product ~2^-16, FP32 accumulation per CTA, FP64 across CTAs), the first moments and the
 * scalar sums in FP64.  me_k4_measure + me_k4_moments remain the all-FP64 route. */
int me_k4_step_measure(me_k4 *e, int64_t n_steps, const double *s_a, double *ts, int64_t ts_row, const double *shift,
                       double *scratch, int64_t scratch_doubles, double *inc, double *mom_accum, double *snapshot,
                       void *stream) {
    if (!e || !e->state || !s_a || !shift || !scratch || !inc) return ME_ERR_INVALID;
    if (n_steps <= 0) return k4_fail(e, ME_ERR_INVALID, "me_k4_step_measure needs at least one step");
    if (e->step + (unsigned long long)n_steps >= 0xffffffffull) return k4_fail(e, ME_ERR_INVALID, "step counter overflow");
    const int max_parts = e->n_sm < 1 ? 1 : e->n_sm;
    if (scratch_doubles < (int64_t)(max_parts + 1) * partw(e->nc)) return k4_fail(e, ME_ERR_INVALID, "moments scratch too small");
    int prev = -1; cudaGetDevice(&prev); cudaSetDevice(e->cfg.device);
    K4Tail tail{ts, (long long)ts_row, shift, scratch};
    int grid = 0;
    int rc = k4_launch_steps(e, n_steps, s_a, nullptr, nullptr, nullptr, &tail, &grid, stream);
    if (rc == ME_OK) {
        k4_moments_finish(e, scratch, grid, inc, mom_accum, snapshot, stream);
        cudaError_t ce = cudaGetLastError();
        if (ce != cudaSuccess) rc = k4_fail(e, ME_ERR_CUDA, std::string("k4_moments: ") + cudaGetErrorString(ce));
    }
    cudaSetDevice(prev);
    if (rc != ME_OK) return rc;
    e->step += (unsigned long long)n_steps;
    e->n_measure += 1;
    return ME_OK;
}

int me_k4_measure(me_k4 *e, double *ts, int64_t ts_row, void *stream) {
    if (!e || !e->state) return ME_ERR_INVALID;
    e->n_measure += 1;
    MeasureParams p;
    p.state = e->state; p.ld = e->cfg.n_chains; p.n_chains = e->cfg.n_chains; p.n_meas = e->n_measure; p.n_c = e->nc;
    p.ts = ts; p.ts_row = ts_row; p.record = ts != nullptr;
    int prev = -1; cudaGetDevice(&prev); cudaSetDevice(e->cfg.device);
    const int block = 256;
    const dim3 grid((unsigned)((e->cfg.n_chains + block - 1) / block), e->nc + 1);
    k4_measure<<<grid, block, 0, (cudaStream_t)stream>>>(p);
    cudaError_t ce = cudaGetLastError();
    cudaSetDevice(prev);
    if (ce != cudaSuccess) return k4_fail(e, ME_ERR_CUDA, std::string("k4_measure: ") + cudaGetErrorString(ce));
    return ME_OK;
}

int me_k4_moments(me_k4 *e, const double *shift, double *scratch, int64_t scratch_doubles, double *inc, double *mom_accum,
                  double *snapshot, void *stream) {
    if (!e || !e->state || !shift || !scratch || !inc) return ME_ERR_INVALID;
    const int n_parts = e->n_sm < 1 ? 1 : e->n_sm;
    const int nc = e->nc, pw = partw(nc), mw = momw(nc);
    if (scratch_doubles < (int64_t)(n_parts + 1) * pw) return k4_fail(e, ME_ERR_INVALID, "moments scratch too small");
    const long long per = (e->cfg.n_chains + n_parts - 1) / n_parts;
    int prev = -1; cudaGetDevice(&prev); cudaSetDevice(e->cfg.device);
    k4_moments_stage1<<<n_parts, 256, 0, (cudaStream_t)stream>>>(e->state, e->cfg.n_chains, e->cfg.n_chains, nc, shift,
                                                                 scratch, per);
    k4_moments_finish(e, scratch, n_parts, inc, mom_accum, snapshot, stream);
    cudaError_t ce = cudaGetLastError();
    cudaSetDevice(prev);
    if (ce != cudaSuccess) return k4_fail(e, ME_ERR_CUDA, std::string("k4_moments: ") + cudaGetErrorString(ce));
    return ME_OK;
}

int me_k4_accumulate_moments(me_k4 *e, const double *inc, double *mom_accum, double *snapshot, void *stream) {
    if (!e || !inc || !mom_accum || !snapshot) return ME_ERR_INVALID;
    const int mw = momw(e->nc);
    int prev = -1; cudaGetDevice(&prev); cudaSetDevice(e->cfg.device);
    k4_moments_accumulate<<<(mw + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const double2 *>(inc), reinterpret_cast<double2 *>(mom_accum), reinterpret_cast<double2 *>(snapshot), mw);
    const cudaError_t ce = cudaGetLastError();
    cudaSetDevice(prev);
    if (ce != cudaSuccess) return k4_fail(e, ME_ERR_CUDA, std::string("k4_moments_accumulate: ") + cudaGetErrorString(ce));
    return ME_OK;
}

int me_k4_refactor(me_k4 *e, const double *mom, const double *inc, int64_t n_measure, double *cov_c, double *cov_a,
                   void *factor_bf16, double *s_a, int32_t *status, void *stream) {
    if (!e || !mom || !inc || !cov_c || !cov_a || !factor_bf16 || !s_a) return ME_ERR_INVALID;
    if (n_measure <= 0) n_measure = e->n_measure;
    int prev = -1; cudaGetDevice(&prev); cudaSetDevice(e->cfg.device);
    const int nc = e->nc;
    const int smem = nc * (nc + 1) * (int)sizeof(double2);
    cudaError_t ce = cudaFuncSetAttribute(k4_refactor, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (ce == cudaSuccess) {
        k4_refactor<<<1, 256, smem, (cudaStream_t)stream>>>(reinterpret_cast<const double2 *>(mom),
                                                            reinterpret_cast<const double2 *>(inc), n_measure, nc,
                                                            reinterpret_cast<double2 *>(cov_c), cov_a,
                                                            reinterpret_cast<__nv_bfloat16 *>(factor_bf16), s_a, status);
        ce = cudaGetLastError();
    }
    cudaSetDevice(prev);
    if (ce != cudaSuccess) return k4_fail(e, ME_ERR_CUDA, std::string("k4_refactor: ") + cudaGetErrorString(ce));
    return ME_OK;
}

/* the generator's table (host copy): 4096 BF16 bit patterns, Phi^-1(1/2 + (i + 1/2) / 8192) */
int me_k4_normal_table(uint16_t *out, int32_t n) {
    if (!out || n != k4::ZTAB_ENTRIES) return ME_ERR_INVALID;
    memcpy(out, k4_host_ztab(), sizeof(uint16_t) * k4::ZTAB_ENTRIES);
    return ME_OK;
}

int me_k4_get_counters(me_k4 *e, int64_t *n_measure, uint64_t *step) {
    if (!e) return ME_ERR_INVALID;
    if (n_measure) *n_measure = e->n_measure;
    if (step) *step = e->step;
    return ME_OK;
}

const char *me_k4_last_error(me_k4 *e) { return e ? e->err.c_str() : g_k4_create_error.c_str(); }

}  // extern "C"
