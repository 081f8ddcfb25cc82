/* me_api.cu — host side of libme_b200.so: the C ABI declared in include/me_b200.h.
 *
 * Responsibilities: pick the kernel set for (shape, energy functor, strict) from the ahead-of-time tables or
 * compile it with NVRTC; keep the two counters the reference keeps on the host (measure_step_counter ME:73 and
 * a global step index for the Philox counter); fill MeParams and launch on the caller's stream.
 * No device memory is owned here except nothing: every buffer is borrowed from the caller.
 */
#include <cuda_runtime.h>
#include <cuda.h>
#include <dlfcn.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/me_b200.h"
#include "me_kernels.cuh"
#include "me_rt.h"
#include "me_embedded.inc"   /* generated: the kernel headers as string constants for NVRTC */

extern "C" const MeAotEntry *me_aot_fast_table(int *n);
extern "C" const MeAotEntry *me_aot_strict_table(int *n);
extern "C" void me_generic_kernels(const void **run_measure, const void **init, const void **propose,
                                   const void **accept, const void **energy);

/* shapes with D = n_r + 2 n_c above this use the runtime-shape kernels of me_generic.cu (state in global memory) */
#define ME_FUSED_MAX_D 32

namespace {

std::string g_create_error;

/* ----------------------------------------------------------------------------------------- kernel handles */
struct KernelRef {
    const void *rt = nullptr;   /* runtime-API function pointer (ahead-of-time kernels) */
    CUfunction drv = nullptr;   /* driver-API function (NVRTC kernels) */
    bool valid() const { return rt != nullptr || drv != nullptr; }
};
struct KernelSet {
    KernelRef run, init, propose, accept, energy, run_mp, run_pt, run_hx, mbar, mbar_hist, mbar_cov;
    bool valid() const { return run.valid(); }
};

/* ----------------------------------------------------------------------------------------- driver + NVRTC, loaded lazily */
typedef CUresult (*cuModuleLoadData_t)(CUmodule *, const void *);
typedef CUresult (*cuModuleGetFunction_t)(CUfunction *, CUmodule, const char *);
typedef CUresult (*cuLaunchKernel_t)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned,
                                     CUstream, void **, void **);
typedef CUresult (*cuGetErrorString_t)(CUresult, const char **);
typedef CUresult (*cuOccupancy_t)(int *, CUfunction, int, size_t);
typedef CUresult (*cuFuncSetAttribute_t)(CUfunction, CUfunction_attribute, int);
typedef CUresult (*cuTensorMapEncodeTiled_t)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                             const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                             CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct Driver {
    cuModuleLoadData_t moduleLoadData = nullptr;
    cuModuleGetFunction_t moduleGetFunction = nullptr;
    cuLaunchKernel_t launchKernel = nullptr;
    cuGetErrorString_t getErrorString = nullptr;
    cuOccupancy_t occupancy = nullptr;          /* optional: only the launch balancing of runtime-compiled kernels needs it */
    cuFuncSetAttribute_t funcSetAttribute = nullptr;        /* optional: > 48 KB dynamic shared memory of runtime-compiled kernels */
    cuTensorMapEncodeTiled_t tensorMapEncodeTiled = nullptr; /* optional: TMA tensor maps */
    bool ok = false;
    std::string err;
};

Driver &driver() {
    static Driver d;
    static std::once_flag once;
    std::call_once(once, [] {
        auto get = [&](const char *name, void **fn) {
            cudaDriverEntryPointQueryResult q;
            cudaError_t e = cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &q);
            if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || *fn == nullptr) {
                d.err = std::string("driver entry point not available: ") + name;
                cudaGetLastError();
                return false;
            }
            return true;
        };
        d.ok = get("cuModuleLoadData", (void **)&d.moduleLoadData) &&
               get("cuModuleGetFunction", (void **)&d.moduleGetFunction) &&
               get("cuLaunchKernel", (void **)&d.launchKernel) && get("cuGetErrorString", (void **)&d.getErrorString);
        if (d.ok) {
            const std::string keep = d.err;
            if (!get("cuOccupancyMaxActiveBlocksPerMultiprocessor", (void **)&d.occupancy)) { d.occupancy = nullptr; d.err = keep; }
            if (!get("cuFuncSetAttribute", (void **)&d.funcSetAttribute)) { d.funcSetAttribute = nullptr; d.err = keep; }
            if (!get("cuTensorMapEncodeTiled", (void **)&d.tensorMapEncodeTiled)) { d.tensorMapEncodeTiled = nullptr; d.err = keep; }
        }
    });
    return d;
}

typedef struct _nvrtcProgram *nvrtcProgram;
struct Nvrtc {
    int (*createProgram)(nvrtcProgram *, const char *, const char *, int, const char *const *, const char *const *) = nullptr;
    int (*compileProgram)(nvrtcProgram, int, const char *const *) = nullptr;
    int (*getCUBINSize)(nvrtcProgram, size_t *) = nullptr;
    int (*getCUBIN)(nvrtcProgram, char *) = nullptr;
    int (*getProgramLogSize)(nvrtcProgram, size_t *) = nullptr;
    int (*getProgramLog)(nvrtcProgram, char *) = nullptr;
    int (*destroyProgram)(nvrtcProgram *) = nullptr;
    const char *(*getErrorString)(int) = nullptr;
    bool ok = false;
    std::string err;
};

Nvrtc &nvrtc() {
    static Nvrtc n;
    static std::once_flag once;
    std::call_once(once, [] {
        std::vector<std::string> names;
        if (const char *env = getenv("ME_NVRTC_PATH")) names.push_back(env);
        names.push_back("libnvrtc.so.12");
        names.push_back("/usr/local/cuda/lib64/libnvrtc.so.12");
        names.push_back("libnvrtc.so");
        void *h = nullptr;
        for (auto &nm : names) {
            h = dlopen(nm.c_str(), RTLD_NOW | RTLD_GLOBAL);
            if (h) break;
        }
        if (!h) { n.err = "libnvrtc.so.12 not found (set ME_NVRTC_PATH)"; return; }
        bool all = true;
        auto sym = [&](const char *s, void **fn) { *fn = dlsym(h, s); if (!*fn) all = false; };
        sym("nvrtcCreateProgram", (void **)&n.createProgram);
        sym("nvrtcCompileProgram", (void **)&n.compileProgram);
        sym("nvrtcGetCUBINSize", (void **)&n.getCUBINSize);
        sym("nvrtcGetCUBIN", (void **)&n.getCUBIN);
        sym("nvrtcGetProgramLogSize", (void **)&n.getProgramLogSize);
        sym("nvrtcGetProgramLog", (void **)&n.getProgramLog);
        sym("nvrtcDestroyProgram", (void **)&n.destroyProgram);
        sym("nvrtcGetErrorString", (void **)&n.getErrorString);
        n.ok = all;
        if (!all) n.err = "libnvrtc is missing required symbols";
    });
    return n;
}

const char *builtin_template(int energy_id) {
    switch (energy_id) {
    case ME_ENERGY_X2: return "me::EnergyX2";
    case ME_ENERGY_XY_WELL: return "me::EnergyXYWell";
    case ME_ENERGY_MIXED_WELL: return "me::EnergyMixedWell";
    case ME_ENERGY_CYLINDER: return "me::EnergyCylinder";
    case ME_ENERGY_EXTERNAL: return "me::EnergyNone";
    case ME_ENERGY_USER: return "me::EnergyUser";
    default: return nullptr;
    }
}

/* Runtime compilation of the kernel set for one (shape, functor, strict).  Returns the CUBIN. */
int nvrtc_compile(int n_real, int n_complex, int energy_id, const std::string &user_src, int use_reject, int strict,
                  std::vector<char> &cubin, std::string &log) {
    Nvrtc &n = nvrtc();
    if (!n.ok) { log = n.err; return ME_ERR_UNSUPPORTED; }
    const char *tmpl = builtin_template(energy_id);
    if (!tmpl) { log = "unknown energy id"; return ME_ERR_INVALID; }
    std::string src = "#include \"me_kernels.cuh\"\n";
    if (energy_id == ME_ENERGY_USER) {
        src += "#line 1 \"user_energy.cu\"\n";
        src += user_src;
        src += "\nnamespace me {\n"
               "template <int NR, int NC> struct EnergyUser {\n"
               "  __device__ static __forceinline__ double eval(const double* x, const double* cr, const double* ci, const double* k) {\n"
               "    return me_user_energy(x, cr, ci, k); }\n"
               "  __device__ static __forceinline__ bool reject(const double* x, const double* cr, const double* ci, const double* k) {\n";
        src += use_reject ? "    return me_user_reject(x, cr, ci, k); }\n" : "    return false; }\n";
        src += "};\n}\n";
    }
    src += std::string("typedef me::Cfg<ME_NR, ME_NC, ") + tmpl + ", (ME_STRICT != 0)> UserCfg;\n";
    /* same register policy as the ahead-of-time kernels (me_kernels.cuh): small shapes at most ME_SMALL_MAXNREG registers */
    src += "#if ME_NR + 2 * ME_NC <= 4\n"
           "extern \"C\" __global__ void __maxnreg__(ME_SMALL_MAXNREG) me_k_run(const __grid_constant__ MeParams p) { me::run_body<UserCfg>(p); }\n"
           "#else\n"
           "extern \"C\" __global__ void __launch_bounds__(ME_MAX_BLOCK) me_k_run(const __grid_constant__ MeParams p) { me::run_body<UserCfg>(p); }\n"
           "#endif\n"
           "#if ME_NR + 2 * ME_NC <= 4\n"
           "extern \"C\" __global__ void __maxnreg__(ME_SMALL_MAXNREG) me_k_run_pt(const __grid_constant__ MeParams p) { me::run_body<UserCfg, false, me::LADDER_TEMP>(p); }\n"
           "#else\n"
           "extern \"C\" __global__ void __launch_bounds__(ME_MAX_BLOCK) me_k_run_pt(const __grid_constant__ MeParams p) { me::run_body<UserCfg, false, me::LADDER_TEMP>(p); }\n"
           "#endif\n"
           "#if ME_NR + 2 * ME_NC <= 4\n"
           "extern \"C\" __global__ void __maxnreg__(ME_SMALL_MAXNREG) me_k_run_hx(const __grid_constant__ MeParams p) { me::run_body<UserCfg, false, me::LADDER_HAM>(p); }\n"
           "#else\n"
           "extern \"C\" __global__ void __launch_bounds__(ME_MAX_BLOCK) me_k_run_hx(const __grid_constant__ MeParams p) { me::run_body<UserCfg, false, me::LADDER_HAM>(p); }\n"
           "#endif\n"
           "#if ME_NC > 0\n"
           "extern \"C\" __global__ void __launch_bounds__(ME_MAX_BLOCK) me_k_run_mp(const __grid_constant__ MeParams p) { me::run_body<UserCfg, true>(p); }\n"
           "#endif\n"
           "extern \"C\" __global__ void __launch_bounds__(ME_MAX_BLOCK) me_k_init(const __grid_constant__ MeParams p) { me::init_body<UserCfg>(p); }\n"
           "extern \"C\" __global__ void __launch_bounds__(ME_MAX_BLOCK) me_k_propose(const __grid_constant__ MeParams p) { me::propose_body<UserCfg>(p); }\n"
           "extern \"C\" __global__ void __launch_bounds__(ME_MAX_BLOCK) me_k_accept(const __grid_constant__ MeParams p) { me::accept_body<UserCfg>(p); }\n"
           "extern \"C\" __global__ void __launch_bounds__(ME_MAX_BLOCK) me_k_energy(const __grid_constant__ MeParams p) { me::energy_body<UserCfg>(p); }\n"
           "extern \"C\" __global__ void __launch_bounds__(32 * ME_MBAR_MAX_WARPS, 1) me_k_mbar(const __grid_constant__ MeMbarParams q) { me::mbar_pass_body<UserCfg>(q); }\n"
           "extern \"C\" __global__ void __launch_bounds__(32 * ME_MBAR_MAX_WARPS, 1) me_k_mbar_hist(const __grid_constant__ MeMbarParams q) { me::mbar_hist_body<UserCfg>(q); }\n"
           "extern \"C\" __global__ void __launch_bounds__(32 * ME_MBAR_MAX_WARPS, 1) me_k_mbar_cov(const __grid_constant__ MeMbarParams q) { me::mbar_cov_body<UserCfg>(q); }\n";
    const char *hdr_names[] = {"me_params.h", "me_math.cuh", "me_device.cuh", "me_energies.cuh", "me_kernels.cuh",
                               "me_mbar.cuh"};
    const char *hdr_src[] = {me_src_params_h, me_src_math_cuh, me_src_device_cuh, me_src_energies_cuh,
                             me_src_kernels_cuh, me_src_mbar_cuh};
    nvrtcProgram prog = nullptr;
    int rc = n.createProgram(&prog, src.c_str(), "me_user_kernels.cu", 6, hdr_src, hdr_names);
    if (rc != 0) { log = std::string("nvrtcCreateProgram: ") + n.getErrorString(rc); return ME_ERR_COMPILE; }
    std::string d_nr = "-DME_NR=" + std::to_string(n_real), d_nc = "-DME_NC=" + std::to_string(n_complex);
    std::string d_st = std::string("-DME_STRICT=") + (strict ? "1" : "0");
    std::vector<const char *> opts = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo", "-DME_NVRTC=1",
                                      d_nr.c_str(), d_nc.c_str(), d_st.c_str()};
    if (strict) opts.push_back("--fmad=false");
    rc = n.compileProgram(prog, (int)opts.size(), opts.data());
    size_t lsz = 0;
    n.getProgramLogSize(prog, &lsz);
    if (lsz > 1) { log.resize(lsz); n.getProgramLog(prog, &log[0]); }
    if (rc != 0) {
        log = std::string("NVRTC: ") + n.getErrorString(rc) + "\n" + log;
        n.destroyProgram(&prog);
        return ME_ERR_COMPILE;
    }
    size_t csz = 0;
    n.getCUBINSize(prog, &csz);
    cubin.resize(csz);
    n.getCUBIN(prog, cubin.data());
    n.destroyProgram(&prog);
    return ME_OK;
}

}  // namespace

/* ----------------------------------------------------------------------------------------- me_rt.h */
int me_rt_compile(const std::string &src, const char *name, const std::vector<std::string> &extra, std::vector<char> &cubin,
                  std::string &log) {
    Nvrtc &n = nvrtc();
    if (!n.ok) { log = n.err; return ME_ERR_UNSUPPORTED; }
    const char *hdr_names[] = {"me_params.h", "me_math.cuh", "me_device.cuh", "me_energies.cuh", "me_kernels.cuh",
                               "me_k4_device.cuh", "me_generic.cuh", "me_mbar.cuh"};
    const char *hdr_src[] = {me_src_params_h, me_src_math_cuh, me_src_device_cuh, me_src_energies_cuh, me_src_kernels_cuh,
                             me_src_k4_device_cuh, me_src_generic_cuh, me_src_mbar_cuh};
    nvrtcProgram prog = nullptr;
    int rc = n.createProgram(&prog, src.c_str(), name, 8, hdr_src, hdr_names);
    if (rc != 0) { log = std::string("nvrtcCreateProgram: ") + n.getErrorString(rc); return ME_ERR_COMPILE; }
    std::vector<const char *> opts = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo", "-DME_NVRTC=1"};
    for (auto &o : extra) opts.push_back(o.c_str());
    rc = n.compileProgram(prog, (int)opts.size(), opts.data());
    size_t lsz = 0;
    n.getProgramLogSize(prog, &lsz);
    if (lsz > 1) { log.resize(lsz); n.getProgramLog(prog, &log[0]); }
    if (rc != 0) {
        log = std::string("NVRTC: ") + n.getErrorString(rc) + "\n" + log;
        n.destroyProgram(&prog);
        return ME_ERR_COMPILE;
    }
    size_t csz = 0;
    n.getCUBINSize(prog, &csz);
    cubin.resize(csz);
    n.getCUBIN(prog, cubin.data());
    n.destroyProgram(&prog);
    return ME_OK;
}

int me_rt_load(int device, const std::vector<char> &cubin, const char *const *names, int cnt, CUfunction *out, std::string &err) {
    Driver &d = driver();
    if (!d.ok) { err = d.err; return ME_ERR_UNSUPPORTED; }
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(device);
    cudaFree(0);   /* make sure the primary context exists and is current */
    CUmodule mod = nullptr;
    CUresult r = d.moduleLoadData(&mod, cubin.data());
    int rc = ME_OK;
    if (r != CUDA_SUCCESS) {
        const char *s = nullptr;
        d.getErrorString(r, &s);
        err = std::string("cuModuleLoadData: ") + (s ? s : "?");
        rc = ME_ERR_CUDA;
    }
    for (int i = 0; rc == ME_OK && i < cnt; i++)
        if (d.moduleGetFunction(&out[i], mod, names[i]) != CUDA_SUCCESS) {
            err = std::string("cuModuleGetFunction: ") + names[i];
            rc = ME_ERR_CUDA;
        }
    if (prev >= 0) cudaSetDevice(prev);
    return rc;
}

int me_rt_launch(CUfunction f, unsigned grid, unsigned block, unsigned smem, void *stream, void **args, std::string &err) {
    Driver &d = driver();
    if (!d.ok) { err = d.err; return ME_ERR_UNSUPPORTED; }
    CUresult r = d.launchKernel(f, grid, 1, 1, block, 1, 1, smem, (CUstream)stream, args, nullptr);
    if (r != CUDA_SUCCESS) {
        const char *s = nullptr;
        d.getErrorString(r, &s);
        err = std::string("cuLaunchKernel: ") + (s ? s : "?");
        return ME_ERR_CUDA;
    }
    return ME_OK;
}

int me_rt_set_dynamic_smem(CUfunction f, int bytes, std::string &err) {
    Driver &d = driver();
    if (!d.ok || !d.funcSetAttribute) { err = "cuFuncSetAttribute not available"; return ME_ERR_UNSUPPORTED; }
    if (d.funcSetAttribute(f, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, bytes) != CUDA_SUCCESS) {
        err = "cuFuncSetAttribute(MAX_DYNAMIC_SHARED_SIZE_BYTES) failed";
        return ME_ERR_CUDA;
    }
    return ME_OK;
}

int me_rt_tensor_map_2d_bf16(void *map_out, const void *gaddr, unsigned long long inner, unsigned long long rows,
                             unsigned box_inner, unsigned box_rows) {
    Driver &d = driver();
    if (!d.ok || !d.tensorMapEncodeTiled) return ME_ERR_UNSUPPORTED;
    const cuuint64_t dims[2] = {inner, rows};
    const cuuint64_t strides[1] = {inner * 2};            /* bytes between rows */
    const cuuint32_t box[2] = {box_inner, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = d.tensorMapEncodeTiled(reinterpret_cast<CUtensorMap *>(map_out), CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2,
                                        const_cast<void *>(gaddr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                        CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? ME_OK : ME_ERR_CUDA;
}

namespace {

/* process-wide cache of loaded runtime-compiled kernel sets */
std::mutex g_cache_mu;
std::map<std::string, KernelSet> g_cache;

}  // namespace

/* ----------------------------------------------------------------------------------------- the handle */
struct me_engine {
    me_config cfg;
    me_layout lay;
    KernelSet ks;
    int energy_id = -1;
    int use_reject = 0;
    double consts[ME_MAX_CONSTS];
    int n_consts = 0;
    me_buffers buf;
    bool bound = false;
    long long n_measure = 1;           /* ME:73 */
    unsigned long long step = 0;       /* global step index (Philox counter word 2) */
    int block = 128, grid = 1;
    int n_sm = 148;
    bool generic = false;              /* large shape: runtime-shape kernels, unfused step */
    int group = 0;                     /* 0 step_all, 1 real group, 2 complex group (mixed engines) */
    /* time segmentation of fused launches (me_device.cuh, run_body) */
    unsigned long long *seg_flags = nullptr;   /* work queue (tickets, pushes, ring) followed by its initial image; device
                                                  memory owned by the handle */
    unsigned long long seg_base = 0;           /* ring capacity */
    int run_slots = -1;                        /* CTAs of the fused kernel resident on the device at once (-1: unknown) */
    const void *run_slots_of = nullptr;        /* the kernel run_slots was measured for (run and run_mp have different register caps) */
    const double *logtab = nullptr;            /* me_math.cuh log table on this engine's device */
    double *pool_partial = nullptr;            /* first-stage rows of the pooled-moment reduction (large ensembles) */
    unsigned long long *ctr_dev = nullptr;     /* device copy of (step, n_measure) for CUDA-graph replay of the unfused step */
    bool use_ctr = false;
    /* temperature ladder (me_set_ladder): n_rungs > 1 runs the PT instantiation of the fused kernel */
    int n_rungs = 1;
    long long swap_every = 0;
    void *ladder_dev = nullptr;                /* rung temperatures [R] (double), then the FP32 windows [R][2] */
    int *walker = nullptr;
    unsigned *swap_acc = nullptr;
    int pool_rungs = 1;                        /* rows of POOL_WORDS per CTA in the pool buffer: R for a ladder that pools */
    /* Hamiltonian ladder (me_set_hamiltonian_ladder): rung_k > 0 runs the HX instantiation */
    double *rung_consts = nullptr;             /* [R][rung_k] functor constants of each rung, device memory */
    int rung_k = 0;
    std::vector<double> rung_temps_host, rung_consts_host;   /* host copies: the states of an MBAR pass (me_mbar_pass) */
    double *mbar_buf = nullptr;                /* MBAR pass: per-CTA partial rows, then the reduced row */
    size_t mbar_cap = 0;                       /* doubles */
    std::string err;
};

namespace {

int fail(me_engine *e, int code, const std::string &msg) {
    if (e) e->err = msg; else g_create_error = msg;
    return code;
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int launch(me_engine *e, const KernelRef &k, MeParams &p, void *stream, int grid_mult = 1, int grid_override = 0) {
    if (!k.valid()) return fail(e, ME_ERR_STATE, "no energy functor registered (call me_set_energy_* first)");
    DeviceGuard g(e->cfg.device);
    void *args[] = {&p};
    const unsigned grid = grid_override > 0 ? (unsigned)grid_override : (unsigned)e->grid * (unsigned)grid_mult;
    if (k.rt) {
        cudaError_t ce = cudaLaunchKernel(k.rt, dim3(grid), dim3(e->block), args, 0, (cudaStream_t)stream);
        if (ce != cudaSuccess) return fail(e, ME_ERR_CUDA, std::string("cudaLaunchKernel: ") + cudaGetErrorString(ce));
    } else {
        Driver &d = driver();
        CUresult r = d.launchKernel(k.drv, grid, 1, 1, e->block, 1, 1, 0, (CUstream)stream, args, nullptr);
        if (r != CUDA_SUCCESS) {
            const char *s = nullptr;
            d.getErrorString(r, &s);
            return fail(e, ME_ERR_CUDA, std::string("cuLaunchKernel: ") + (s ? s : "?"));
        }
    }
    return ME_OK;
}

/* The log table of me_math.cuh: computed once per device in long double and kept for the life of the process. */
const double *log_table(int device) {
    static std::mutex mu;
    static std::map<int, double *> tabs;
    std::lock_guard<std::mutex> lock(mu);
    auto it = tabs.find(device);
    if (it != tabs.end()) return it->second;
    std::vector<double> host(2 * (ME_LOGTAB_ENTRIES + ME_SINTAB_ENTRIES));
    const int fold = (int)(0.4142135623730951 * ME_LOGTAB_ENTRIES);          /* first interval whose upper edge exceeds sqrt 2 */
    for (int i = 0; i < ME_LOGTAB_ENTRIES; i++) {
        const double c = 1.0 + (double)(i + 1) / (double)ME_LOGTAB_ENTRIES;
        const double rc = (double)(float)(1.0 / c);
        host[2 * i] = rc;
        host[2 * i + 1] = (double)(2.0L * logl(i >= fold ? (long double)rc * 2.0L : (long double)rc));
    }
    /* sin/cos of the interval midpoints (me_math.cuh, sincospi_tab); the second half of the circle is the exact negative
       of the first, so that opposite angle words give exactly opposite normals */
    double *sc = host.data() + 2 * ME_LOGTAB_ENTRIES;
    const long double two_pi = 6.283185307179586476925286766559L;
    for (int i = 0; i < ME_SINTAB_ENTRIES / 2; i++) {
        const long double a = ((long double)i + 0.5L) * two_pi / (long double)ME_SINTAB_ENTRIES;
        sc[2 * i] = (double)sinl(a);
        sc[2 * i + 1] = (double)cosl(a);
        sc[2 * (i + ME_SINTAB_ENTRIES / 2)] = -sc[2 * i];
        sc[2 * (i + ME_SINTAB_ENTRIES / 2) + 1] = -sc[2 * i + 1];
    }
    DeviceGuard g(device);
    double *dev = nullptr;
    if (cudaMalloc((void **)&dev, host.size() * sizeof(double)) != cudaSuccess ||
        cudaMemcpy(dev, host.data(), host.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    tabs[device] = dev;
    return dev;
}

/* FP32 window of the throughput build's Metropolis test (me_device.cuh, Rng::accept_window).  Its error budget is
   relative to T and holds while T ln2 and 4e-5 T are normal floats far from overflow, i.e. for 1e-30 <= T <= 1e30.
   T = 0: the half-width is the smallest denormal, so that the window is [-2^-149, 2^-149] and a dE that rounds to
   +-0 in FP32 takes the exact test.  Any other T: an infinite half-width sends every decision to the exact test. */
void accept_window_consts(double t, float &t_ln2, float &t_band) {
    if (t == 0) {
        t_ln2 = 0.0f;
        t_band = 0x1p-149f;
    } else if (t >= 1e-30 && t <= 1e30) {
        t_ln2 = (float)(t * 0.69314718055994531);
        t_band = (float)(t * 4e-5);
    } else {
        t_ln2 = 0.0f;
        t_band = HUGE_VALF;
    }
}

int pool_words(const me_engine *e) { return e->lay.POOL_WORDS * e->pool_rungs; }

void base_params(me_engine *e, MeParams &p) {
    memset(&p, 0, sizeof(p));
    p.logtab = e->logtab;
    p.ctr_dev = e->use_ctr ? e->ctr_dev : nullptr;
    p.state = e->buf.state;
    p.ld = e->cfg.n_chains;
    p.n_chains = e->cfg.n_chains;
    p.chain_offset = (unsigned long long)e->cfg.chain_offset;
    p.seed = e->cfg.seed;
    for (int r = 0; r < 10; r++) {
        p.rk[2 * r] = (unsigned)e->cfg.seed + (unsigned)r * 0x9E3779B9u;
        p.rk[2 * r + 1] = (unsigned)(e->cfg.seed >> 32) + (unsigned)r * 0xBB67AE85u;
    }
    p.step0 = e->step;
    p.n_meas0 = e->n_measure;
    p.use_reject = e->use_reject;
    p.m = e->cfg.n_real + e->cfg.n_complex;
    p.temp = e->cfg.temp;
    p.inv_temp = e->cfg.temp != 0 ? 1.0 / e->cfg.temp : 0.0;
    accept_window_consts(e->cfg.temp, p.t_ln2, p.t_band);
    p.target = e->cfg.target_acceptance;
    p.ratio = e->cfg.ratio;
    memcpy(p.consts, e->consts, sizeof(p.consts));
    p.last_accept = e->buf.last_accept;
    p.pool = e->lay.POOL_WORDS > 0 ? e->buf.pool : nullptr;
    p.shift = e->buf.shift;
    p.n_real = e->cfg.n_real;
    p.n_complex = e->cfg.n_complex;
    p.energy_id = e->energy_id;
    p.scratch = e->buf.scratch;
    p.prop = e->buf.prop;
    p.group = e->group;
    if (e->n_rungs > 1) {
        p.n_rungs = e->n_rungs;
        p.swap_every = e->swap_every;
        p.rung_temp = static_cast<const double *>(e->ladder_dev);
        p.rung_window = reinterpret_cast<const float *>(p.rung_temp + e->n_rungs);
        p.walker = e->walker;
        p.swap_acc = e->swap_acc;
        p.rung_consts = e->rung_consts;
        p.n_consts = e->rung_k;
        if (e->pool_rungs != e->n_rungs) p.pool = nullptr;      /* a ladder that does not fit a warp pools nothing */
    }
}

/* Time segmentation of a fused launch (me_device.cuh, run_body): when the whole grid is resident in one wave the
 * launch is cut into time segments per chain group and the CTAs become workers on a FIFO of ready segments, which
 * balances the SM sub-partitions (65,536 chains are 3 or 4 warps per sub-partition, and a sub-partition saturates at
 * 2-3).  Returns the segment count (1 = off), -1 on a CUDA error.  ME_SEGMENTS=<n> overrides (0 / 1 = off). */
#define ME_MAX_SEGMENTS 64      /* the last, partly filled round of items costs ~1/(2 x rounds) of the launch */
int plan_segments(me_engine *e, const KernelRef &k, long long n_blocks, long long spm, bool injected, void *stream) {
    if (injected || e->generic || e->cfg.strict || !k.valid()) return 1;
    if (e->lay.D > ME_SEG_MAX_D) return 1;                               /* compiled out for larger shapes (me_device.cuh) */
    int want = -1;
    if (const char *env = getenv("ME_SEGMENTS")) want = atoi(env);
    if (want == 0 || want == 1) return 1;
    DeviceGuard g(e->cfg.device);
    const void *kid = k.rt ? k.rt : (const void *)k.drv;
    if (e->run_slots < 0 || e->run_slots_of != kid) {
        e->run_slots_of = kid;
        int per_sm = 0;
        if (k.rt) {
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k.rt, e->block, 0) != cudaSuccess) { cudaGetLastError(); per_sm = 0; }
        } else {                                  /* runtime-compiled (NVRTC) kernel: driver API */
            Driver &d = driver();
            if (!d.ok || !d.occupancy || d.occupancy(&per_sm, k.drv, e->block, 0) != CUDA_SUCCESS) per_sm = 0;
        }
        e->run_slots = per_sm * e->n_sm;
    }
    if (e->run_slots <= 0) return 1;
    /* segmentation pays when the groups do not fill an integer number of waves and there are only a few waves */
    if (e->grid % e->run_slots == 0 || e->grid > 4LL * e->run_slots) return 1;
    const long long steps = n_blocks * (spm > 0 ? spm : 1);
    const long long min_steps = 1500;                                    /* per segment: hand-over cost stays < 1 % */
    long long segs = want > 1 ? want : steps / min_steps;
    if (segs > ME_MAX_SEGMENTS) segs = ME_MAX_SEGMENTS;
    if (segs > n_blocks) segs = n_blocks;
    if (segs < 2) return 1;
    if (!e->seg_flags) {
        unsigned long long cap = 2;
        /* one ring slot per item of the largest launch: every CTA takes its ticket as soon as it starts, long before the
           matching push, so a slot must never be shared by two tickets of one launch */
        while (cap < (unsigned long long)ME_MAX_SEGMENTS * (unsigned long long)e->grid) cap <<= 1;
        const size_t words = (size_t)(cap + 2);
        if (cudaMallocAsync((void **)&e->seg_flags, sizeof(unsigned long long) * 2 * words, (cudaStream_t)stream) != cudaSuccess) {
            fail(e, ME_ERR_CUDA, "allocating the segment queue failed");
            return -1;
        }
        /* initial image behind the live queue: no ticket handed out, segment 0 of every group pushed */
        std::vector<unsigned long long> img(words, 0ull);
        img[1] = (unsigned long long)e->grid;
        for (long long gidx = 0; gidx < e->grid; gidx++) img[2 + gidx] = (unsigned long long)gidx + 1ull;
        if (cudaMemcpyAsync(e->seg_flags + words, img.data(), sizeof(unsigned long long) * words, cudaMemcpyHostToDevice,
                            (cudaStream_t)stream) != cudaSuccess ||
            cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) {     /* img is a stack-lifetime host buffer */
            fail(e, ME_ERR_CUDA, "initialising the segment queue failed");
            return -1;
        }
        e->seg_base = cap;
    }
    if (getenv("ME_DEBUG"))
        fprintf(stderr, "[me_b200] segmented launch: %lld groups x %lld segments (%d resident slots)\n",
                (long long)e->grid, segs, e->run_slots);
    const size_t words = (size_t)(e->seg_base + 2);
    if (cudaMemcpyAsync(e->seg_flags, e->seg_flags + words, sizeof(unsigned long long) * words, cudaMemcpyDeviceToDevice,
                        (cudaStream_t)stream) != cudaSuccess) {
        fail(e, ME_ERR_CUDA, "resetting the segment queue failed");
        return -1;
    }
    return (int)segs;
}

/* Launch geometry.  One thread per chain, so the CTA size only trades scheduling granularity against the
 * per-CTA pooled reduction: when the whole ensemble fits in one wave use 32-thread CTAs (finest balance over
 * the 148 SMs), otherwise 128. */
void choose_dims(me_engine *e) {
    const long long n = e->cfg.n_chains;
    int block = 128;
    if (n <= (long long)e->n_sm * 32 * 16) block = 32;          /* up to four warps per sub-partition: finest balance; beyond
                                                                   that 64-thread CTAs halve the per-CTA fixed cost, which
                                                                   short launches feel (tests/scripts/c5_launch_probe.py:
                                                                   131,072 chains x 100 steps, 106.6 -> 100.8 us) */
    else if (n <= (long long)e->n_sm * 32 * 64) block = 64;
    {   /* shapes whose pooled moments run on the FP64 tensor cores stage them per warp in static shared memory sized for
           me_pool_mma_max_block(D) threads (run_body in me_device.cuh: POOL_MMA) */
        const int d = e->cfg.n_real + 2 * e->cfg.n_complex;
        const int poolw = d + d * (d + 1) / 2 + 2 * e->cfg.n_real + e->cfg.n_complex;
        if (me::me_pool_mma_shape(d, poolw) && poolw <= ME_MAX_POOLW && block > me::me_pool_mma_max_block(d))
            block = me::me_pool_mma_max_block(d);
    }
    e->block = block;
    e->grid = (int)((n + block - 1) / block);
}

/* Runtime compilation of the runtime-shape kernel set (D > 32) around a user functor: same contract as the fused kernels'
 * (me_user_energy / me_user_reject over x[ME_NR], c_re[ME_NC], c_im[ME_NC]); -fmad=false like the ahead-of-time build. */
int nvrtc_compile_generic(int n_real, int n_complex, const std::string &user_src, int use_reject, std::vector<char> &cubin,
                          std::string &log) {
    std::string src = "#define ME_GENERIC_USER 1\n";
    if (use_reject) src += "#define ME_GENERIC_USER_REJECT 1\n";
    src += "#include \"me_kernels.cuh\"\n#line 1 \"user_energy.cu\"\n";
    src += user_src;
    src += "\n#include \"me_generic.cuh\"\n";
    std::vector<std::string> extra = {"-DME_NR=" + std::to_string(n_real), "-DME_NC=" + std::to_string(n_complex),
                                      "-DME_STRICT=1", "--fmad=false"};
    return me_rt_compile(src, "me_user_generic_kernels.cu", extra, cubin, log);
}

int resolve_kernels(me_engine *e, int energy_id, const std::string &user_src) {
    const int nr = e->cfg.n_real, nc = e->cfg.n_complex, strict = e->cfg.strict ? 1 : 0;
    if (e->generic && energy_id == ME_ENERGY_USER) {
        /* runtime shape with a user functor: the runtime-shape kernels (me_generic.cuh) compiled around the functor */
        std::string key = "generic," + std::to_string(nr) + "," + std::to_string(nc) + "," + std::to_string(e->use_reject) +
                          "," + std::to_string(e->cfg.device) + "|" + user_src;
        std::lock_guard<std::mutex> lk(g_cache_mu);
        auto it = g_cache.find(key);
        if (it != g_cache.end()) { e->ks = it->second; return ME_OK; }
        std::vector<char> cubin;
        std::string log;
        int rc = nvrtc_compile_generic(nr, nc, user_src, e->use_reject, cubin, log);
        if (rc != ME_OK) return fail(e, rc, log);
        static const char *names[5] = {"me_gk_run", "me_gk_init", "me_gk_propose", "me_gk_accept", "me_gk_energy"};
        CUfunction fn[5];
        std::string err;
        rc = me_rt_load(e->cfg.device, cubin, names, 5, fn, err);
        if (rc != ME_OK) return fail(e, rc, err);
        KernelSet ks;
        ks.run.drv = fn[0]; ks.init.drv = fn[1]; ks.propose.drv = fn[2]; ks.accept.drv = fn[3]; ks.energy.drv = fn[4];
        g_cache[key] = ks;
        e->ks = ks;
        return ME_OK;
    }
    if (e->generic) {
        const void *m, *i, *pr, *ac, *en;
        me_generic_kernels(&m, &i, &pr, &ac, &en);
        e->ks.run.rt = m; e->ks.init.rt = i; e->ks.propose.rt = pr; e->ks.accept.rt = ac; e->ks.energy.rt = en;
        return ME_OK;
    }
    if (energy_id != ME_ENERGY_USER) {
        int n = 0;
        const MeAotEntry *t = strict ? me_aot_strict_table(&n) : me_aot_fast_table(&n);
        for (int i = 0; i < n; i++)
            if (t[i].n_real == nr && t[i].n_complex == nc && t[i].energy_id == energy_id) {
                e->ks.run.rt = t[i].run; e->ks.init.rt = t[i].init; e->ks.run_mp.rt = t[i].run_mp;
                e->ks.propose.rt = t[i].propose; e->ks.accept.rt = t[i].accept; e->ks.energy.rt = t[i].energy;
                e->ks.run_pt.rt = t[i].run_pt; e->ks.run_hx.rt = t[i].run_hx; e->ks.mbar.rt = t[i].mbar;
                e->ks.mbar_hist.rt = t[i].mbar_hist; e->ks.mbar_cov.rt = t[i].mbar_cov;
                return ME_OK;
            }
    }
    /* not instantiated ahead of time: NVRTC */
    std::string key = std::to_string(nr) + "," + std::to_string(nc) + "," + std::to_string(energy_id) + "," +
                      std::to_string(strict) + "," + std::to_string(e->use_reject) + "," +
                      std::to_string(e->cfg.device) + "|" + user_src;
    std::lock_guard<std::mutex> lk(g_cache_mu);
    auto it = g_cache.find(key);
    if (it != g_cache.end()) { e->ks = it->second; return ME_OK; }
    std::vector<char> cubin;
    std::string log;
    int rc = nvrtc_compile(nr, nc, energy_id, user_src, e->use_reject, strict, cubin, log);
    if (rc != ME_OK) return fail(e, rc, log);
    Driver &d = driver();
    if (!d.ok) return fail(e, ME_ERR_UNSUPPORTED, d.err);
    DeviceGuard g(e->cfg.device);
    cudaFree(0);   /* make sure the primary context exists and is current */
    CUmodule mod = nullptr;
    CUresult r = d.moduleLoadData(&mod, cubin.data());
    if (r != CUDA_SUCCESS) {
        const char *s = nullptr;
        d.getErrorString(r, &s);
        return fail(e, ME_ERR_CUDA, std::string("cuModuleLoadData: ") + (s ? s : "?"));
    }
    KernelSet ks;
    if (d.moduleGetFunction(&ks.run.drv, mod, "me_k_run") != CUDA_SUCCESS ||
        d.moduleGetFunction(&ks.init.drv, mod, "me_k_init") != CUDA_SUCCESS ||
        d.moduleGetFunction(&ks.propose.drv, mod, "me_k_propose") != CUDA_SUCCESS ||
        d.moduleGetFunction(&ks.accept.drv, mod, "me_k_accept") != CUDA_SUCCESS ||
        d.moduleGetFunction(&ks.energy.drv, mod, "me_k_energy") != CUDA_SUCCESS ||
        d.moduleGetFunction(&ks.run_pt.drv, mod, "me_k_run_pt") != CUDA_SUCCESS ||
        d.moduleGetFunction(&ks.run_hx.drv, mod, "me_k_run_hx") != CUDA_SUCCESS ||
        d.moduleGetFunction(&ks.mbar.drv, mod, "me_k_mbar") != CUDA_SUCCESS ||
        d.moduleGetFunction(&ks.mbar_hist.drv, mod, "me_k_mbar_hist") != CUDA_SUCCESS ||
        d.moduleGetFunction(&ks.mbar_cov.drv, mod, "me_k_mbar_cov") != CUDA_SUCCESS ||
        (e->cfg.n_complex > 0 && d.moduleGetFunction(&ks.run_mp.drv, mod, "me_k_run_mp") != CUDA_SUCCESS))
        return fail(e, ME_ERR_CUDA, "cuModuleGetFunction failed on the runtime-compiled module");
    g_cache[key] = ks;
    e->ks = ks;
    return ME_OK;
}

/* out[w] = sum over the per-CTA slots pool[b][w] in a fixed order (deterministic): one CTA per word, thread t sums the
 * slots t, t + 256, ... and a shared-memory tree combines the 256 partial sums.  (One thread per word walking all slots
 * serially cost 0.5 ms per call at 2048 slots — pure L2 latency.) */
__global__ void __launch_bounds__(256) k_pool_reduce(double *pool, double *out, int grid, int words, int reset,
                                                     int has_extra = 0, double extra = 0.0) {
    __shared__ double part[256];
    const int w = blockIdx.x, t = threadIdx.x;
    if (w == words) {                           /* me_allreduce_stats: the sample count travels with the moments */
        if (has_extra && t == 0) out[words] = extra;
        return;
    }
    double acc = 0.0;
    for (int b = t; b < grid; b += 256) {
        acc += pool[(long long)b * words + w];
        if (reset) pool[(long long)b * words + w] = 0.0;
    }
    part[t] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (t < o) part[t] += part[t + o];
        __syncthreads();
    }
    if (t == 0) out[w] = part[0];
}

/* First stage for very large ensembles (10^7-10^8 chains: millions of per-CTA moment rows).  The pool is read as the
 * flat array it is: thread t of a CTA owns word (t % words) of row offset (t / words) inside a slab of `rpb` rows, so
 * consecutive threads read consecutive doubles; the slabs of one CTA are `gridDim.x` slabs apart.  The per-thread sums
 * are folded over the row offsets in fixed order, so the result depends on (grid, words, gridDim.x) only. */
#define ME_POOL_STAGE_CTAS 592
__global__ void __launch_bounds__(256) k_pool_partial(double *pool, double *partial, long long grid, int words, int reset) {
    __shared__ double part[256];
    const int rpb = 256 / words, t = threadIdx.x;
    const int ro = t / words, w = t - ro * words;
    double acc = 0.0;
    if (ro < rpb) {
        for (long long r = (long long)blockIdx.x * rpb + ro; r < grid; r += (long long)gridDim.x * rpb) {
            acc += pool[r * words + w];
            if (reset) pool[r * words + w] = 0.0;
        }
    }
    part[t] = acc;
    __syncthreads();
    if (t < words) {
        double a = part[t];
        for (int k = 1; k < rpb; k++) a += part[k * words + t];
        partial[(long long)blockIdx.x * words + t] = a;
    }
}

/* device copy of the step / measure counters (see MeParams::ctr_dev) */
__global__ void k_ctr_set(unsigned long long *ctr, unsigned long long step, unsigned long long n_meas) {
    ctr[0] = step; ctr[1] = n_meas;
}
__global__ void k_ctr_advance(unsigned long long *ctr, unsigned long long dstep) { ctr[0] += dstep; }
__global__ void k_ctr_advance2(unsigned long long *ctr, unsigned long long dstep, unsigned long long dmeas) {
    ctr[0] += dstep; ctr[1] += dmeas;
}
/* totals[w] += inc[w]: the device-resident running moments of me_allreduce_stats */
__global__ void k_accumulate(double *totals, const double *inc, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) totals[i] += inc[i];
}

/* FP64 FMA throughput probe: 8 independent dependent-FMA streams per thread.  The roofline denominator of the
 * step kernels (MEASURED_PEAKS.json carries HBM and bf16 figures only). */
__global__ void __launch_bounds__(256) k_probe_fp64(double *out, long long iters) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 0.99999988, c = 1.25e-7;
    for (long long i = 0; i < iters; i++) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    out[(long long)blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

/* Statistical inefficiency g = 1 + 2 sum_t (1 - t/N) rho_t, truncated at the first non-positive rho_t, of one
 * time-series column per chain (one thread per chain; consecutive threads read consecutive chains, so every row
 * access is coalesced).  This is the quantity the reference obtains from pymbar for its equilibrium statistics
 * (statistics.py:36-38,46; used at metropolis_engine.py:490) and the denominator of ESS/sec. */
__global__ void k_stat_ineff(const double *ts, long long rows, long long row0, int cols, long long ld, int col,
                             long long chain0, long long n_sel, long long max_lag, double *g_out) {
    const long long t_id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t_id >= n_sel) return;
    const double *x = ts + (long long)col * ld + chain0 + t_id;
    const long long stride = (long long)cols * ld;
    const long long N = rows - row0;
    double mean = 0.0;
    for (long long i = 0; i < N; i++) mean += x[(row0 + i) * stride];
    mean /= (double)N;
    double var = 0.0;
    for (long long i = 0; i < N; i++) { const double d = x[(row0 + i) * stride] - mean; var += d * d; }
    var /= (double)N;
    double g = 1.0;
    if (var > 0.0 && N >= 4) {
        const long long tmax = max_lag < N - 1 ? max_lag : N - 2;
        for (long long t = 1; t <= tmax; t++) {
            double c = 0.0;
            for (long long i = 0; i + t < N; i++) c += (x[(row0 + i) * stride] - mean) * (x[(row0 + i + t) * stride] - mean);
            const double rho = c / ((double)(N - t) * var);
            if (!(rho > 0.0)) break;
            g += 2.0 * rho * (1.0 - (double)t / (double)N);
        }
    }
    g_out[t_id] = g > 1.0 ? g : 1.0;
}

/* Equilibration detection (SURVEY §8 row f3): the reference's save_equilibrium_stats (metropolis_engine.py:481-504)
 * -> statistics.get_equilibration_points (statistics.py:25-48) -> pymbar.timeseries.detectEquilibration, restated in
 * the oracle (detect_equilibration).  For every candidate start t0 = cand * nskip the statistical inefficiency
 * g(t0) of rows [t0, T) is computed with pymbar's estimator (C(t) from the mean-removed series, stop at the first
 * non-positive C(t) beyond `mintime`, optional growing lag increments `fast`), and Neff(t0) = (T - t0 + 1) / g(t0).
 * One thread per (chain, candidate); consecutive threads are consecutive chains, so every row access is coalesced. */
__global__ void k_equil_scan(const double *ts, long long rows, int cols, long long ld, int col, long long chain0,
                             long long n_sel, long long nskip, long long n_cand, int fast, int mintime, double *g_t,
                             double *neff_t) {
    const long long t_id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t_id >= n_sel) return;
    const double *x = ts + (long long)col * ld + chain0 + t_id;
    const long long stride = (long long)cols * ld;
    for (long long cand = blockIdx.y; cand < n_cand; cand += gridDim.y) {
        const long long t0 = cand * nskip;
        const long long N = rows - t0;
        double mean = 0.0;
        for (long long i = 0; i < N; i++) mean += x[(t0 + i) * stride];
        mean /= (double)N;
        double var = 0.0;
        for (long long i = 0; i < N; i++) { const double d = x[(t0 + i) * stride] - mean; var += d * d; }
        var /= (double)N;
        double g;
        if (!(var > 0.0)) {
            g = (double)(rows - t0 + 1);                 /* pymbar: ParameterError -> g = T - t + 1 */
        } else {
            g = 1.0;
            long long t = 1, inc = 1;
            while (t < N - 1) {
                double c = 0.0;
                for (long long i = 0; i + t < N; i++) c += (x[(t0 + i) * stride] - mean) * (x[(t0 + i + t) * stride] - mean);
                c /= (double)(N - t) * var;
                if (c <= 0.0 && t > mintime) break;
                g += 2.0 * c * (1.0 - (double)t / (double)N) * (double)inc;
                t += inc;
                if (fast) inc += 1;
            }
            if (g < 1.0) g = 1.0;
        }
        g_t[cand * n_sel + t_id] = g;
        /* a series that is constant from its first row is reported as (0, 1, 1) by detectEquilibration: sentinel */
        neff_t[cand * n_sel + t_id] = (cand == 0 && !(var > 0.0)) ? -1.0 : (double)(rows - t0 + 1) / g;
    }
}

__global__ void k_equil_pick(const double *g_t, const double *neff_t, long long n_cand, long long n_sel, long long nskip,
                             double *t_out, double *g_out, double *neff_out) {
    const long long t_id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t_id >= n_sel) return;
    if (neff_t[t_id] < 0.0) { t_out[t_id] = 0.0; g_out[t_id] = 1.0; neff_out[t_id] = 1.0; return; }
    long long best = 0;
    double bn = neff_t[t_id];
    for (long long cand = 1; cand < n_cand; cand++) {
        const double v = neff_t[cand * n_sel + t_id];
        if (v > bn) { bn = v; best = cand; }              /* first maximum, as numpy.argmax */
    }
    t_out[t_id] = (double)(best * nskip);
    g_out[t_id] = g_t[best * n_sel + t_id];
    neff_out[t_id] = bn;
}

/* Geometry of an MBAR pass (me_mbar.cuh): the 8-row blocks of the staged rows, the tile list in the order k_mbar_unpack
 * reads it — [s: (W_i, ONE)] [G: (W_i, W_j), j <= i] and with observables [(WE_i, ONE)] [(WE2_i, ONE)] [(W_i, XX_j)] —
 * and the length of the documented sums vector (me_b200.h, me_mbar_pass). */
struct MbarLayout {
    int S, nb, nx, n_tiles, z_rows, rw;
    long long words;
    unsigned char ta[ME_MBAR_MAX_TILES], tb[ME_MBAR_MAX_TILES];
};
void mbar_layout(int d, int n_states, int obs, MbarLayout &m) {
    m.S = n_states;
    m.nb = (n_states + 7) / 8;
    m.nx = obs ? (2 * d + 7) / 8 : 0;
    const int nb = m.nb;
    int t = 0;
    auto add = [&](int a, int b) { m.ta[t] = (unsigned char)a; m.tb[t] = (unsigned char)b; t++; };
    for (int i = 0; i < nb; i++) add(i, nb);
    for (int i = 0; i < nb; i++)
        for (int j = 0; j <= i; j++) add(i, j);
    if (obs) {
        for (int i = 0; i < nb; i++) add(nb + 1 + i, nb);
        for (int i = 0; i < nb; i++) add(2 * nb + 1 + i, nb);
        for (int i = 0; i < nb; i++)
            for (int j = 0; j < m.nx; j++) add(i, 3 * nb + 1 + j);
    }
    m.n_tiles = t;
    m.z_rows = 8 * (obs ? 3 * nb + 1 + m.nx : 2 * nb + 1);
    m.rw = 3 + 64 * t;
    m.words = 3 + n_states + (long long)n_states * (n_states + 1) / 2 + (obs ? (long long)n_states * (2 * d + 2) : 0);
}

/* reduced partial row [sum L, n_nan, n_overflow, tiles[n_tiles][8][8]] -> the sums vector of me_mbar_pass
   (sums = that, or sums += that) */
__global__ void k_mbar_unpack(const double *raw, double *sums, int S, int nb, int nx, int d, long long words, int accumulate) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= words) return;
    const double *tile = raw + 3;
    const int we0 = nb + nb * (nb + 1) / 2, we20 = we0 + nb, xx0 = we20 + nb;
    long long o = w - 3;
    double v;
    if (w < 3) {
        v = raw[w];
    } else if (o < S) {
        v = tile[(o / 8) * 64 + (o % 8) * 8];
    } else if ((o -= S) < (long long)S * (S + 1) / 2) {
        int s = 0;
        while ((long long)(s + 1) * (s + 2) / 2 <= o) s++;
        const int t = (int)(o - (long long)s * (s + 1) / 2), i = s / 8, j = t / 8;
        v = tile[(nb + i * (i + 1) / 2 + j) * 64 + (s % 8) * 8 + t % 8];
    } else {
        o -= (long long)S * (S + 1) / 2;
        const int s = (int)(o / (2 * d + 2)), a = (int)(o % (2 * d + 2));
        if (a < 2 * d) v = tile[(xx0 + (s / 8) * nx + a / 8) * 64 + (s % 8) * 8 + a % 8];
        else v = tile[((a == 2 * d ? we0 : we20) + s / 8) * 64 + (s % 8) * 8];
    }
    sums[w] = accumulate ? sums[w] + v : v;
}

/* the checks me_mbar_words and me_mbar_pass share: shape, functor, mode and state count */
int mbar_check(me_engine *e, int n_target) {
    if (e->generic) return fail(e, ME_ERR_UNSUPPORTED, "MBAR passes need a fused shape (n_real + 2 n_complex <= 32)");
    if (e->energy_id == ME_ENERGY_EXTERNAL)
        return fail(e, ME_ERR_UNSUPPORTED, "MBAR passes re-evaluate a device energy functor; this handle's energies are "
                                           "evaluated by the caller");
    if (e->group != 0)
        return fail(e, ME_ERR_UNSUPPORTED, "MBAR passes serve handles that step all parameters (group 0), not group-wise or "
                                           "magnitude-phase modes");
    if (e->energy_id < 0) return fail(e, ME_ERR_STATE, "no energy functor registered (call me_set_energy_* first)");
    if (e->n_rungs > ME_MBAR_MAX_STATES) return fail(e, ME_ERR_INVALID, "MBAR passes take at most 32 rungs");
    if (n_target < 0 || e->n_rungs + n_target > ME_MBAR_MAX_STATES)
        return fail(e, ME_ERR_INVALID, "MBAR passes take at most 32 states (rungs + targets) and n_target >= 0");
    return ME_OK;
}

/* 1 / T and the functor constants [ME_MAX_CONSTS] of one MBAR state: rung r >= 0 (its temperature, and its constants on
   a Hamiltonian ladder), or, r < 0, a target at temperature t with constants tk[K] (NULL: the handle's constants) */
int mbar_state(me_engine *e, int r, double t, const double *tk, double &inv_temp, double *consts) {
    const int R = e->n_rungs;
    const bool ham = e->rung_k > 0;
    const int K = ham ? e->rung_k : e->n_consts;
    if (r >= 0) t = R > 1 ? e->rung_temps_host[r] : e->cfg.temp;
    if (!std::isfinite(t) || !(t > 0))
        return fail(e, ME_ERR_INVALID, std::string(r >= 0 ? "every rung temperature" : "every target temperature") +
                                           " must be finite and > 0 for MBAR");
    inv_temp = 1.0 / t;
    for (int i = 0; i < ME_MAX_CONSTS; i++) {
        double k = e->consts[i];
        if (r >= 0 && ham) k = i < K ? e->rung_consts_host[(size_t)r * K + i] : 0.0;
        if (r < 0 && tk) k = i < K ? tk[i] : 0.0;
        if (!std::isfinite(k)) return fail(e, ME_ERR_INVALID, "MBAR state constants must be finite");
        consts[i] = k;
    }
    return ME_OK;
}

/* Launch one MBAR-type pass kernel over q.n_samples samples and reduce its per-CTA rows of q.rw words in fixed order
   into raw[q.rw] (device, inside the handle's buffer).  CTAs of up to 4 warps inside the default 48 KB of shared
   memory; shapes whose one warp needs more (per_warp bytes) opt in.  At most 8 CTAs per SM; resident_only: no more than fit
   the SMs' shared memory at once, so that wide partial rows (histograms) stay as few as can run together. */
int mbar_launch(me_engine *e, const KernelRef &k, MeMbarParams &q, int per_warp, bool resident_only, cudaStream_t st,
                double *&raw) {
    const int head = ME_MBAR_HEAD * 8;
    int nw = (48 * 1024 - head) / per_warp;
    nw = nw < 1 ? 1 : (nw > ME_MBAR_MAX_WARPS ? ME_MBAR_MAX_WARPS : nw);
    const int smem = head + nw * per_warp;
    const long long want = (q.n_samples + 32LL * nw - 1) / (32LL * nw);
    long long per_sm = 8;
    if (resident_only && 233472 / (smem + 1024) < per_sm) per_sm = std::max(1, 233472 / (smem + 1024));
    const long long cap = per_sm * e->n_sm;
    const int grid = (int)(want < cap ? want : cap);
    DeviceGuard g(e->cfg.device);
    const size_t need = (size_t)(grid + 1) * q.rw;
    if (need > e->mbar_cap) {
        if (e->mbar_buf) cudaFree(e->mbar_buf);
        e->mbar_buf = nullptr;
        e->mbar_cap = 0;
        if (cudaMalloc((void **)&e->mbar_buf, need * sizeof(double)) != cudaSuccess) {
            cudaGetLastError();
            return fail(e, ME_ERR_CUDA, "allocating the MBAR partial rows failed");
        }
        e->mbar_cap = need;
    }
    q.partial = e->mbar_buf;
    raw = e->mbar_buf + (size_t)grid * q.rw;
    void *args[] = {&q};
    if (k.rt) {
        if (smem > 48 * 1024 &&
            cudaFuncSetAttribute(k.rt, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) {
            cudaGetLastError();
            return fail(e, ME_ERR_CUDA, "MBAR pass: cannot raise the kernel's shared-memory limit");
        }
        cudaError_t ce = cudaLaunchKernel(k.rt, dim3(grid), dim3(32 * nw), args, (size_t)smem, st);
        if (ce != cudaSuccess) return fail(e, ME_ERR_CUDA, std::string("cudaLaunchKernel: ") + cudaGetErrorString(ce));
    } else {
        Driver &d = driver();
        if (smem > 48 * 1024 &&
            (!d.funcSetAttribute ||
             d.funcSetAttribute(k.drv, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, smem) != CUDA_SUCCESS))
            return fail(e, ME_ERR_CUDA, "MBAR pass: cannot raise the kernel's shared-memory limit");
        CUresult r = d.launchKernel(k.drv, grid, 1, 1, 32 * nw, 1, 1, smem, (CUstream)st, args, nullptr);
        if (r != CUDA_SUCCESS) {
            const char *s = nullptr;
            d.getErrorString(r, &s);
            return fail(e, ME_ERR_CUDA, std::string("cuLaunchKernel: ") + (s ? s : "?"));
        }
    }
    k_pool_reduce<<<q.rw, 256, 0, st>>>(q.partial, raw, grid, q.rw, 0);
    return ME_OK;
}

/* histogram pass: the reduced row already has the layout of the sums vector (me_mbar_hist_pass) */
__global__ void k_mbar_hist_unpack(const double *raw, double *sums, long long words, int accumulate) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w < words) sums[w] = accumulate ? sums[w] + raw[w] : raw[w];
}

/* bins of a histogram pass: B = prod n_bins over 1 or 2 axes, with B (R + 2) <= ME_MBAR_HIST_MAX_WORDS */
int mbar_hist_bins(me_engine *e, int n_axes, const int32_t *n_bins, long long &B) {
    if (n_axes != 1 && n_axes != 2) return fail(e, ME_ERR_INVALID, "n_axes must be 1 or 2");
    if (!n_bins) return fail(e, ME_ERR_INVALID, "n_bins is required");
    B = 1;
    for (int a = 0; a < n_axes; a++) {
        if (n_bins[a] < 1) return fail(e, ME_ERR_INVALID, "n_bins must be >= 1 on every axis");
        B *= n_bins[a];
        if (B * (e->n_rungs + 2) > ME_MBAR_HIST_MAX_WORDS)
            return fail(e, ME_ERR_INVALID, "histogram too large: bins x (rungs + 2) must not exceed 24576 doubles");
    }
    return ME_OK;
}

/* the samples of an MBAR-type pass (rows [row0, rows) of one storage chunk, every stride-th row, every local chain) and
   the fields every pass shares: q.n_rungs and the sample range (row0 / stride / n_per_state checks) */
int mbar_samples(me_engine *e, const double *ts, int64_t rows, int64_t row0, int64_t stride, const double *f,
                 int64_t n_per_state, MeMbarParams &q) {
    if (rows < 1 || row0 < 0 || row0 >= rows) return fail(e, ME_ERR_INVALID, "row0 must lie in [0, rows)");
    if (stride < 1) return fail(e, ME_ERR_INVALID, "stride must be >= 1");
    if (n_per_state < 1) return fail(e, ME_ERR_INVALID, "n_per_state must be >= 1");
    const long long ld = e->cfg.n_chains, n_rows = (rows - row0 + stride - 1) / stride;
    q.ts = ts; q.ld = ld; q.row0 = row0; q.stride = stride; q.n_samples = n_rows * ld;
    q.ts_cols = e->lay.TS_COLS;
    q.n_rungs = e->n_rungs; q.use_reject = e->use_reject;
    q.n_per_state = (double)n_per_state; q.log_n = std::log((double)n_per_state);
    q.f = f;
    return ME_OK;
}

/* the state table of me_mbar_pass and me_mbar_cov_pass: the R rungs, then n_target targets (target_temps[t],
   target_consts[t][K] or the handle's constants); sets q.n_states = R + n_target */
int mbar_states(me_engine *e, int n_target, const double *target_temps, const double *target_consts, MeMbarParams &q) {
    if (n_target > 0 && !target_temps) return fail(e, ME_ERR_INVALID, "target_temps is required when n_target > 0");
    const int R = e->n_rungs, S = R + n_target;
    const bool ham = e->rung_k > 0;
    const int K = ham ? e->rung_k : e->n_consts;
    if (n_target > 0 && ham && !target_consts)
        return fail(e, ME_ERR_INVALID, "targets of a Hamiltonian ladder need their constants (target_consts)");
    for (int s = 0; s < S; s++) {
        const double *tk = target_consts && s >= R ? target_consts + (size_t)(s - R) * K : nullptr;
        const int rc = s < R ? mbar_state(e, s, 0.0, nullptr, q.inv_temp[s], q.consts[s])
                             : mbar_state(e, -1, target_temps[s - R], tk, q.inv_temp[s], q.consts[s]);
        if (rc != ME_OK) return rc;
    }
    q.n_states = S;
    return ME_OK;
}

/* Geometry of a covariance pass (me_mbar.cuh, mbar_cov_body) over the covered states [first, first + count) of S
 * states: nb 8-row blocks of weights, mb blocks per covered state's m = 2D + 2 observables, and per covered state c the
 * tile list [(V_ci, ONE), (V_ci, W_j) j < nb] for i < mb, then [(V_ci, V_cj), j <= i], which k_mbar_cov_unpack reads.
 * fits: the tiles fit the list and one warp's accumulators and staging fit the 227 KB shared-memory opt-in. */
struct MbarCovLayout {
    int nb, mb, m, n_tiles, z_rows, rw, per_warp;
    long long words;
    bool fits;
    unsigned char ta[ME_MBAR_COV_MAX_TILES], tb[ME_MBAR_COV_MAX_TILES];
};
void mbar_cov_layout(int d, int n_states, int n_rungs, int count, MbarCovLayout &m) {
    m.nb = (n_states + 7) / 8;
    m.m = 2 * d + 2;
    m.mb = (m.m + 7) / 8;
    const int nb = m.nb, mb = m.mb, per = mb * (nb + 1) + mb * (mb + 1) / 2;
    m.n_tiles = count * per;
    m.z_rows = 8 * (2 * nb + 1 + count * mb);
    m.rw = 2 + 64 * m.n_tiles;
    m.per_warp = (m.n_tiles * 64 + m.z_rows * ME_MBAR_LD) * 8;
    m.words = 2 + (long long)count * (m.m + (long long)m.m * (n_rungs + 1) + (long long)m.m * (m.m + 1) / 2);
    m.fits = m.n_tiles <= ME_MBAR_COV_MAX_TILES && ME_MBAR_HEAD * 8 + m.per_warp <= ME_MBAR_SMEM_OPTIN;
    if (!m.fits) return;
    int t = 0;
    for (int c = 0; c < count; c++) {
        const int v0 = 2 * nb + 1 + c * mb;
        for (int i = 0; i < mb; i++) {
            m.ta[t] = (unsigned char)(v0 + i); m.tb[t++] = (unsigned char)nb;
            for (int j = 0; j < nb; j++) { m.ta[t] = (unsigned char)(v0 + i); m.tb[t++] = (unsigned char)j; }
        }
        for (int i = 0; i < mb; i++)
            for (int j = 0; j <= i; j++) { m.ta[t] = (unsigned char)(v0 + i); m.tb[t++] = (unsigned char)(v0 + j); }
    }
}

/* reduced partial row [n_nan, n_overflow, tiles[n_tiles][8][8]] -> the sums vector of me_mbar_cov_pass: per covered
   state o[m], C[m][R + 1] (the last column is C_a*), Q[m (m + 1) / 2] (sums = that, or sums += that) */
__global__ void k_mbar_cov_unpack(const double *raw, double *sums, int R, int nb, int mb, int m, int first, long long words,
                                  int accumulate) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= words) return;
    const double *tile = raw + 2;
    const long long per = m + (long long)m * (R + 1) + (long long)m * (m + 1) / 2;
    const long long tc = mb * (nb + 1) + mb * (mb + 1) / 2;
    double v;
    if (w < 2) {
        v = raw[w];
    } else {
        const long long c = (w - 2) / per;
        long long r = (w - 2) % per;
        const double *tt = tile + c * tc * 64;
        if (r < m) {
            v = tt[(r / 8) * (nb + 1) * 64 + (r % 8) * 8];
        } else if ((r -= m) < (long long)m * (R + 1)) {
            const int a = (int)(r / (R + 1)), k = (int)(r % (R + 1)), col = k < R ? k : first + (int)c;
            v = tt[((a / 8) * (nb + 1) + 1 + col / 8) * 64 + (a % 8) * 8 + col % 8];
        } else {
            r -= (long long)m * (R + 1);
            int a = 0;
            while ((long long)(a + 1) * (a + 2) / 2 <= r) a++;
            const int b = (int)(r - (long long)a * (a + 1) / 2), i = a / 8, j = b / 8;
            v = tt[(mb * (nb + 1) + i * (i + 1) / 2 + j) * 64 + (a % 8) * 8 + b % 8];
        }
    }
    sums[w] = accumulate ? sums[w] + v : v;
}

/* the checks me_mbar_cov_words and me_mbar_cov_pass share: those of me_mbar_pass, the covered range and the fit */
int mbar_cov_check(me_engine *e, int n_target, int cov_first, int cov_count, MbarCovLayout &m) {
    const int rc = mbar_check(e, n_target);
    if (rc != ME_OK) return rc;
    const int S = e->n_rungs + n_target;
    if (cov_count < 1 || cov_first < 0 || cov_first > S - cov_count)
        return fail(e, ME_ERR_INVALID, "the covered states [cov_first, cov_first + cov_count) must be a non-empty range "
                                       "inside [0, rungs + targets)");
    mbar_cov_layout(e->lay.D, S, e->n_rungs, cov_count, m);
    if (!m.fits)
        return fail(e, ME_ERR_INVALID, "too many covered states for one pass: one warp's tiles and staging exceed the "
                                       "227 KB of shared memory (cover fewer states per pass)");
    return ME_OK;
}

}  // namespace

/* ========================================================================================= C ABI */
extern "C" {

int me_abi_version(void) { return ME_ABI_VERSION; }

int me_state_layout(int32_t nr, int32_t nc, me_layout *o) {
    if (!o || nr < 0 || nc < 0 || nr + nc == 0) return ME_ERR_INVALID;
    const int d = nr + 2 * nc;
    int w = 0;
    o->X = w; w += d;
    o->E = w; w += 1;
    o->SIG = w; w += 2;
    o->MEAN = w; w += d;
    o->COVR = w; w += nr * (nr + 1) / 2;
    o->COVC = w; w += nc * nc;
    o->OBSM = w; w += 2 * nr + nc;
    o->FACR = w; w += nr * (nr + 1) / 2;
    o->FACC = w; w += nc * nc;
    o->NACC = w; w += 1;
    o->STATUS = w; w += 1;
    o->WORDS = w;
    o->D = d;
    o->TS_COLS = d + ((nr > 0 && nc > 0) ? 3 : 2);
    const long long pw = (long long)d + (long long)d * (d + 1) / 2 + 2 * nr + nc;
    o->POOL_WORDS = pw <= ME_MAX_POOLW ? (int)pw : 0;
    return ME_OK;
}

int me_create(const me_config *cfg, me_engine **out) {
    if (!cfg || !out) return fail(nullptr, ME_ERR_INVALID, "null argument");
    if (cfg->n_real < 0 || cfg->n_complex < 0 || cfg->n_real + cfg->n_complex == 0)
        return fail(nullptr, ME_ERR_INVALID, "need at least one real or complex parameter (reference: ValueError, ME:37-39)");
    if (cfg->n_chains <= 0) return fail(nullptr, ME_ERR_INVALID, "n_chains must be positive");
    if (!(cfg->temp >= 0)) return fail(nullptr, ME_ERR_INVALID, "temp must be >= 0 (reference: assert, ME:92)");
    me_engine *e = new me_engine();
    e->cfg = *cfg;
    me_state_layout(cfg->n_real, cfg->n_complex, &e->lay);
    memset(e->consts, 0, sizeof(e->consts));
    memset(&e->buf, 0, sizeof(e->buf));
    int n_sm = 0;
    if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, cfg->device) == cudaSuccess && n_sm > 0)
        e->n_sm = n_sm;
    else
        cudaGetLastError();
    choose_dims(e);
    e->generic = e->lay.D > ME_FUSED_MAX_D;
    if (e->generic) { e->block = 128; e->grid = (int)((cfg->n_chains + 127) / 128); }
    *out = e;
    return ME_OK;
}

int me_destroy(me_engine *e) {
    if (e && (e->seg_flags || e->ctr_dev || e->pool_partial || e->ladder_dev || e->rung_consts || e->mbar_buf)) {
        DeviceGuard g(e->cfg.device);
        if (e->mbar_buf) cudaFree(e->mbar_buf);
        if (e->ladder_dev) cudaFree(e->ladder_dev);
        if (e->rung_consts) cudaFree(e->rung_consts);
        if (e->seg_flags) cudaFree(e->seg_flags);
        if (e->ctr_dev) cudaFree(e->ctr_dev);
        if (e->pool_partial) cudaFree(e->pool_partial);
    }
    delete e;
    return ME_OK;
}

static int set_energy(me_engine *e, int id, const char *src, const double *consts, int n_consts, int use_reject) {
    if (!e) return ME_ERR_INVALID;
    if (n_consts < 0 || n_consts > ME_MAX_CONSTS) return fail(e, ME_ERR_INVALID, "at most 16 functor constants");
    if (!builtin_template(id)) return fail(e, ME_ERR_INVALID, "unknown energy id");
    if (e->rung_k > 0 && n_consts != e->rung_k)
        return fail(e, ME_ERR_INVALID, "the handle's Hamiltonian ladder has " + std::to_string(e->rung_k) +
                                           " constants per rung; the functor must take as many");
    memset(e->consts, 0, sizeof(e->consts));
    for (int i = 0; i < n_consts; i++) e->consts[i] = consts[i];
    e->n_consts = n_consts;
    e->use_reject = use_reject ? 1 : 0;
    e->ks = KernelSet();
    e->run_slots = -1;
    const int prev_id = e->energy_id;
    e->energy_id = id;
    int rc = resolve_kernels(e, id, src ? std::string(src) : std::string());
    if (rc != ME_OK) e->energy_id = prev_id;
    return rc;
}

int me_set_energy_builtin(me_engine *e, int32_t id, const double *consts, int32_t n_consts, int32_t use_reject) {
    if (id == ME_ENERGY_USER) return fail(e, ME_ERR_INVALID, "use me_set_energy_source for user functors");
    return set_energy(e, id, nullptr, consts, n_consts, use_reject);
}

int me_set_energy_source(me_engine *e, const char *src, const double *consts, int32_t n_consts, int32_t use_reject) {
    if (!src) return fail(e, ME_ERR_INVALID, "null source");
    return set_energy(e, ME_ENERGY_USER, src, consts, n_consts, use_reject);
}

int me_set_energy_external(me_engine *e) { return set_energy(e, ME_ENERGY_EXTERNAL, nullptr, nullptr, 0, 0); }

int me_check_energy_source(const char *src, int32_t nr, int32_t nc, int32_t use_reject, int32_t strict, char *log,
                           int64_t cap) {
    std::vector<char> cubin;
    std::string l;
    int rc = (src && nr + 2 * nc > ME_FUSED_MAX_D)
                 ? nvrtc_compile_generic(nr, nc, src, use_reject, cubin, l)
                 : nvrtc_compile(nr, nc, src ? ME_ENERGY_USER : ME_ENERGY_EXTERNAL, src ? src : "", use_reject, strict, cubin, l);
    if (log && cap > 0) {
        strncpy(log, l.c_str(), (size_t)cap - 1);
        log[cap - 1] = 0;
    }
    return rc;
}

int me_set_group(me_engine *e, int32_t group) {
    if (!e) return ME_ERR_INVALID;
    if (group < 0 || group > 4)
        return fail(e, ME_ERR_INVALID, "group must be 0 (all), 1 (real), 2 (complex), 3 (complex magnitudes) or 4 (complex phases)");
    if (group == 1 && e->cfg.n_real == 0) return fail(e, ME_ERR_INVALID, "engine has no real parameters");
    if (group >= 2 && e->cfg.n_complex == 0) return fail(e, ME_ERR_INVALID, "engine has no complex parameters");
    e->group = group;
    return ME_OK;
}

/* me_set_ladder is the Hamiltonian ladder without a rung table (consts = NULL): the same checks, upload and geometry */
int me_set_ladder(me_engine *e, const double *temps, int32_t n_rungs, int64_t swap_every, int32_t *walker,
                  uint32_t *swap_acc) {
    return me_set_hamiltonian_ladder(e, temps, nullptr, 0, n_rungs, swap_every, walker, swap_acc);
}

int me_set_hamiltonian_ladder(me_engine *e, const double *temps, const double *consts, int32_t n_consts, int32_t n_rungs,
                              int64_t swap_every, int32_t *walker, uint32_t *swap_acc) {
    if (!e) return ME_ERR_INVALID;
    const bool ham = consts != nullptr;
    if (e->bound) return fail(e, ME_ERR_STATE, "a ladder is set before me_bind (it sets the launch geometry)");
    if (e->generic) return fail(e, ME_ERR_UNSUPPORTED, "ladders need a fused shape (n_real + 2 n_complex <= 32)");
    if (!temps || !walker || !swap_acc) return fail(e, ME_ERR_INVALID, "temps, walker and swap_acc are required");
    if (n_rungs < 2) return fail(e, ME_ERR_INVALID, "a ladder has at least 2 rungs");
    if (swap_every < 0) return fail(e, ME_ERR_INVALID, "swap_every must be >= 0");
    const long long R = n_rungs;
    if (e->cfg.chain_offset % R != 0 || e->cfg.n_chains % R != 0)
        return fail(e, ME_ERR_INVALID, "the chains of a handle must be whole ladders: chain_offset and n_chains multiples of " +
                                           std::to_string(R));
    const bool pow2 = n_rungs <= 32 && (n_rungs & (n_rungs - 1)) == 0;
    if (swap_every > 0 && !pow2) return fail(e, ME_ERR_INVALID, "replica exchange needs 2, 4, 8, 16 or 32 rungs");
    for (int r = 0; r < n_rungs; r++) {
        if (!std::isfinite(temps[r]) || temps[r] < 0)
            return fail(e, ME_ERR_INVALID, "ladder temperatures must be finite and >= 0");
        if (swap_every > 0 && !(temps[r] > 0))
            return fail(e, ME_ERR_INVALID, "replica exchange needs temperatures > 0");
        if (!ham && swap_every > 0 && r > 0 && !(temps[r] > temps[r - 1]))
            return fail(e, ME_ERR_INVALID, "replica exchange needs strictly increasing temperatures");
    }
    if (ham) {
        if (n_consts < 1 || n_consts > ME_MAX_CONSTS)
            return fail(e, ME_ERR_INVALID, "a Hamiltonian ladder has 1 to 16 constants per rung");
        for (long long i = 0; i < R * n_consts; i++)
            if (!std::isfinite(consts[i])) return fail(e, ME_ERR_INVALID, "rung constants must be finite");
        if (e->energy_id >= 0 && e->n_consts != n_consts)
            return fail(e, ME_ERR_INVALID, "the handle's functor takes " + std::to_string(e->n_consts) +
                                               " constants; the rung table must have as many per rung");
    }
    std::vector<char> host(sizeof(double) * R + sizeof(float) * 2 * R);
    double *t = reinterpret_cast<double *>(host.data());
    float *win = reinterpret_cast<float *>(t + R);
    for (int r = 0; r < n_rungs; r++) {
        t[r] = temps[r];
        accept_window_consts(temps[r], win[2 * r], win[2 * r + 1]);
    }
    DeviceGuard g(e->cfg.device);
    if (e->ladder_dev) { cudaFree(e->ladder_dev); e->ladder_dev = nullptr; }
    if (e->rung_consts) { cudaFree(e->rung_consts); e->rung_consts = nullptr; }
    e->rung_k = 0;
    const size_t kbytes = ham ? sizeof(double) * (size_t)(R * n_consts) : 0;
    if (cudaMalloc(&e->ladder_dev, host.size()) != cudaSuccess ||
        cudaMemcpy(e->ladder_dev, host.data(), host.size(), cudaMemcpyHostToDevice) != cudaSuccess ||
        (ham && (cudaMalloc((void **)&e->rung_consts, kbytes) != cudaSuccess ||
                 cudaMemcpy(e->rung_consts, consts, kbytes, cudaMemcpyHostToDevice) != cudaSuccess))) {
        cudaGetLastError();
        if (e->ladder_dev) cudaFree(e->ladder_dev);
        if (e->rung_consts) cudaFree(e->rung_consts);
        e->ladder_dev = nullptr;
        e->rung_consts = nullptr;
        return fail(e, ME_ERR_CUDA, "allocating the ladder failed");
    }
    e->rung_k = ham ? n_consts : 0;
    e->rung_temps_host.assign(temps, temps + n_rungs);
    e->rung_consts_host.assign(consts ? consts : temps, consts ? consts + R * n_consts : temps);
    e->n_rungs = n_rungs;
    e->swap_every = swap_every;
    e->walker = walker;
    e->swap_acc = reinterpret_cast<unsigned *>(swap_acc);
    /* pooled moments per rung need the ladder inside a warp (me_device.cuh, run_body PT); shapes that do not pool in
       registers add the rung sums of every measure straight into their CTA's rows, so their CTAs are one warp */
    e->pool_rungs = pow2 ? n_rungs : 0;
    if (pow2 && e->lay.POOL_WORDS > ME_POOL_REG_MAX) {
        e->block = 32;
        e->grid = (int)((e->cfg.n_chains + 31) / 32);
    }
    e->run_slots = -1;
    return ME_OK;
}

int me_launch_dims(me_engine *e, int32_t *grid, int32_t *block) {
    if (!e) return ME_ERR_INVALID;
    if (grid) *grid = e->grid;
    if (block) *block = e->block;
    return ME_OK;
}

int me_bind(me_engine *e, const me_buffers *b) {
    if (!e || !b) return ME_ERR_INVALID;
    if (!b->state) return fail(e, ME_ERR_INVALID, "state buffer is required");
    if (b->pool && !b->shift) return fail(e, ME_ERR_INVALID, "pool needs a shift vector");
    if (e->generic && !b->scratch) return fail(e, ME_ERR_INVALID, "large parameter spaces need the scratch buffer");
    e->buf = *b;
    e->bound = true;
    if (!e->logtab) {
        e->logtab = log_table(e->cfg.device);
        if (!e->logtab) return fail(e, ME_ERR_CUDA, "allocating the log table failed");
    }
    return ME_OK;
}

int me_init(me_engine *e, const double *x0, int32_t bc, double sigma0, const double *cov_r, const double *cov_c_re,
            const double *cov_c_im, const double *e0, void *stream) {
    if (!e) return ME_ERR_INVALID;
    if (!e->bound) return fail(e, ME_ERR_STATE, "me_bind first");
    if (!x0) return fail(e, ME_ERR_INVALID, "x0 is required");
    if (e->energy_id == ME_ENERGY_EXTERNAL && !e0) return fail(e, ME_ERR_INVALID, "external energies need e0");
    MeParams p;
    base_params(e, p);
    p.x0 = x0; p.x0_broadcast = bc; p.sigma0 = sigma0;
    p.cov_r0 = cov_r; p.cov_c0_re = cov_c_re; p.cov_c0_im = cov_c_im;
    p.e_new = e0; p.have_e0 = e0 != nullptr;
    e->n_measure = 1;
    e->step = 0;
    return launch(e, e->ks.init, p, stream);
}

static int run_common(me_engine *e, int64_t n_blocks, int64_t spm, int do_measure, const double *delta, const double *u,
                      double *ts, int64_t ts_row0, void *stream) {
    if (!e) return ME_ERR_INVALID;
    if (!e->bound) return fail(e, ME_ERR_STATE, "me_bind first");
    if (n_blocks < 0 || spm < 0) return fail(e, ME_ERR_INVALID, "negative schedule");
    if (n_blocks == 0 || (spm == 0 && !do_measure)) return ME_OK;
    if (spm > 0 && e->energy_id == ME_ENERGY_EXTERNAL)
        return fail(e, ME_ERR_STATE, "external energies step through me_propose / me_accept");
    if (e->generic && spm > 0 &&
        (delta != nullptr || e->energy_id < 0 || e->energy_id == ME_ENERGY_EXTERNAL || !e->buf.prop || e->group >= 3))
        return fail(e, ME_ERR_STATE, "large parameter spaces run whole schedules in one launch only with a device functor "
                                     "(and me_buffers.prop bound); otherwise step through me_propose / me_energy_builtin / "
                                     "me_accept and let me_run measure");
    if (e->step + (unsigned long long)(n_blocks * spm) >= 0xffffffffull)
        return fail(e, ME_ERR_INVALID, "step index exceeds the 32-bit Philox counter word");
    MeParams p;
    base_params(e, p);
    p.n_blocks = n_blocks; p.spm = spm; p.do_measure = do_measure ? 1 : 0;
    p.ts = ts; p.ts_row0 = ts_row0; p.record = (ts != nullptr && do_measure) ? 1 : 0;
    p.inj_delta = delta; p.inj_u = u;
    if (e->group >= 3 && !e->ks.run_mp.valid())
        return fail(e, ME_ERR_STATE, "no magnitude-phase kernel for this engine");
    if (e->n_rungs > 1 && (e->group != 0 || delta != nullptr))
        return fail(e, ME_ERR_UNSUPPORTED, "temperature ladders step all parameters with Philox draws only");
    const KernelRef &ladder = e->rung_k > 0 ? e->ks.run_hx : e->ks.run_pt;
    if (e->n_rungs > 1 && !ladder.valid())
        return fail(e, ME_ERR_STATE, "no ladder kernel for this engine (device functors only)");
    const KernelRef &kr = e->n_rungs > 1 ? ladder : (e->group >= 3 ? e->ks.run_mp : e->ks.run);
    const int segs = plan_segments(e, kr, n_blocks, spm, delta != nullptr, stream);
    if (segs < 0) return ME_ERR_CUDA;
    if (segs > 1) {
        p.seg_count = segs; p.seg_groups = e->grid; p.seg_base = e->seg_base; p.seg_flags = e->seg_flags;
    }
    int rc = launch(e, kr, p, stream, segs > 1 ? segs : 1);
    if (rc != ME_OK) return rc;
    e->step += (unsigned long long)(n_blocks * spm);
    if (do_measure) e->n_measure += n_blocks;
    if (e->use_ctr) {            /* the device copy follows, also when this launch is replayed from a CUDA graph */
        DeviceGuard g(e->cfg.device);
        k_ctr_advance2<<<1, 1, 0, (cudaStream_t)stream>>>(e->ctr_dev, (unsigned long long)(n_blocks * spm),
                                                         do_measure ? (unsigned long long)n_blocks : 0ull);
        if (cudaGetLastError() != cudaSuccess) return fail(e, ME_ERR_CUDA, "advancing the device counters failed");
    }
    return ME_OK;
}

int me_run(me_engine *e, int64_t n_blocks, int64_t spm, int32_t do_measure, double *ts, int64_t ts_row0, void *stream) {
    return run_common(e, n_blocks, spm, do_measure, nullptr, nullptr, ts, ts_row0, stream);
}

int me_run_injected(me_engine *e, int64_t n_blocks, int64_t spm, int32_t do_measure, const double *delta,
                    const double *u, double *ts, int64_t ts_row0, void *stream) {
    if (!e) return ME_ERR_INVALID;
    if (!e->cfg.strict) return fail(e, ME_ERR_STATE, "draw injection needs a strict handle (cfg.strict = 1)");
    if (!delta || !u) return fail(e, ME_ERR_INVALID, "delta and u are required");
    return run_common(e, n_blocks, spm, do_measure, delta, u, ts, ts_row0, stream);
}

int me_propose(me_engine *e, double *prop, const double *inj_delta, void *stream) {
    if (!e) return ME_ERR_INVALID;
    if (!e->bound) return fail(e, ME_ERR_STATE, "me_bind first");
    if (!prop) return fail(e, ME_ERR_INVALID, "prop is required");
    if (inj_delta && !e->cfg.strict) return fail(e, ME_ERR_STATE, "draw injection needs a strict handle");
    if (e->n_rungs > 1) return fail(e, ME_ERR_UNSUPPORTED, "temperature ladders step fused only (me_run)");
    MeParams p;
    base_params(e, p);
    p.prop = prop; p.inj_delta = inj_delta;
    return launch(e, e->ks.propose, p, stream);
}

int me_accept(me_engine *e, const double *prop, const double *e_new, const unsigned char *rej, const double *inj_u,
              void *stream) {
    if (!e) return ME_ERR_INVALID;
    if (!e->bound) return fail(e, ME_ERR_STATE, "me_bind first");
    if (!prop || !e_new) return fail(e, ME_ERR_INVALID, "prop and e_new are required");
    if (inj_u && !e->cfg.strict) return fail(e, ME_ERR_STATE, "draw injection needs a strict handle");
    if (e->n_rungs > 1) return fail(e, ME_ERR_UNSUPPORTED, "temperature ladders step fused only (me_run)");
    if (e->step + 1ull >= 0xffffffffull) return fail(e, ME_ERR_INVALID, "step index exceeds the 32-bit Philox counter word");
    MeParams p;
    base_params(e, p);
    p.prop = const_cast<double *>(prop); p.e_new = e_new; p.rej = rej; p.inj_u = inj_u;
    int rc = launch(e, e->ks.accept, p, stream);
    if (rc == ME_OK) {
        e->step += 1;
        if (e->use_ctr) {           /* keeps the device counter in step, also when this call is replayed from a graph */
            DeviceGuard g(e->cfg.device);
            k_ctr_advance<<<1, 1, 0, (cudaStream_t)stream>>>(e->ctr_dev, 1ull);
            if (cudaGetLastError() != cudaSuccess) return fail(e, ME_ERR_CUDA, "advancing the device counters failed");
        }
    }
    return rc;
}

int me_device_counters(me_engine *e, int32_t enable, void *stream) {
    if (!e) return ME_ERR_INVALID;
    if (e->generic) return fail(e, ME_ERR_UNSUPPORTED, "device counters serve the fused-shape unfused path (D <= 32)");
    DeviceGuard g(e->cfg.device);
    if (enable) {
        if (!e->ctr_dev &&
            cudaMallocAsync((void **)&e->ctr_dev, 2 * sizeof(unsigned long long), (cudaStream_t)stream) != cudaSuccess)
            return fail(e, ME_ERR_CUDA, "allocating the device counters failed");
        k_ctr_set<<<1, 1, 0, (cudaStream_t)stream>>>(e->ctr_dev, e->step, (unsigned long long)e->n_measure);
        if (cudaGetLastError() != cudaSuccess) return fail(e, ME_ERR_CUDA, "setting the device counters failed");
    }
    e->use_ctr = enable != 0;
    return ME_OK;
}

int me_energy_builtin(me_engine *e, const double *prop, double *e_out, unsigned char *rej_out, void *stream) {
    if (!e) return ME_ERR_INVALID;
    if (!e->bound) return fail(e, ME_ERR_STATE, "me_bind first");
    if (!prop || !e_out) return fail(e, ME_ERR_INVALID, "prop and e_out are required");
    if (e->energy_id < 0 || e->energy_id == ME_ENERGY_EXTERNAL) return fail(e, ME_ERR_STATE, "no device functor registered");
    if (e->rung_k > 0)
        return fail(e, ME_ERR_UNSUPPORTED, "a Hamiltonian ladder has no single constant vector to evaluate proposals with");
    MeParams p;
    base_params(e, p);
    p.prop = const_cast<double *>(prop); p.e_out = e_out; p.rej_out = rej_out;
    return launch(e, e->ks.energy, p, stream);
}

int me_pool_reduce(me_engine *e, double *out, int32_t reset, void *stream) {
    if (!e || !out) return ME_ERR_INVALID;
    if (!e->bound || !e->buf.pool || pool_words(e) == 0) return fail(e, ME_ERR_STATE, "no pool buffer bound");
    DeviceGuard g(e->cfg.device);
    const int words = pool_words(e);
    if (e->grid > 4096 && words <= 256) {
        /* millions of rows: coalesced first stage into ME_POOL_STAGE_CTAS partial rows, then the fixed-order tree */
        if (!e->pool_partial &&
            cudaMalloc(&e->pool_partial, sizeof(double) * ME_POOL_STAGE_CTAS * words) != cudaSuccess) {
            cudaGetLastError();
            return fail(e, ME_ERR_CUDA, "pool reduce: cannot allocate the partial-sum rows");
        }
        k_pool_partial<<<ME_POOL_STAGE_CTAS, 256, 0, (cudaStream_t)stream>>>(e->buf.pool, e->pool_partial, e->grid, words,
                                                                           reset);
        k_pool_reduce<<<words, 256, 0, (cudaStream_t)stream>>>(e->pool_partial, out, ME_POOL_STAGE_CTAS, words, 0);
    } else {
        k_pool_reduce<<<words, 256, 0, (cudaStream_t)stream>>>(e->buf.pool, out, e->grid, words, reset);
    }
    cudaError_t ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail(e, ME_ERR_CUDA, std::string("pool reduce: ") + cudaGetErrorString(ce));
    return ME_OK;
}

}  // extern "C"

/* ----------------------------------------------------------------------------------------- NCCL, loaded lazily
 * The library does not link NCCL: the Python host already carries torch's copy, a C host names one with
 * me_comm_set_library() or ME_NCCL_PATH. */
namespace {
struct NcclId { char internal[128]; };
struct NcclApi {
    int (*getUniqueId)(NcclId *) = nullptr;
    int (*commInitRank)(void **, int, NcclId, int) = nullptr;
    int (*commInitRankConfig)(void **, int, NcclId, int, void *) = nullptr;      /* optional (NCCL >= 2.17) */
    int (*commDestroy)(void *) = nullptr;
    int (*allReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    const char *(*getErrorString)(int) = nullptr;
    bool ok = false;
    std::string err, path;
};
std::string g_nccl_path;
NcclApi &nccl_api() {
    static NcclApi n;
    static std::once_flag once;
    std::call_once(once, [] {
        std::vector<std::string> names;
        if (!g_nccl_path.empty()) names.push_back(g_nccl_path);
        if (const char *env = getenv("ME_NCCL_PATH")) names.push_back(env);
        names.push_back("libnccl.so.2");
        names.push_back("libnccl.so");
        void *h = nullptr;
        for (auto &nm : names) {
            h = dlopen(nm.c_str(), RTLD_NOW | RTLD_NOLOAD);          /* the copy the host process already loaded */
            if (!h) h = dlopen(nm.c_str(), RTLD_NOW | RTLD_GLOBAL);
            if (h) { n.path = nm; break; }
        }
        if (!h) { n.err = "libnccl.so.2 not found (me_comm_set_library / ME_NCCL_PATH)"; return; }
        bool all = true;
        auto sym = [&](const char *sname, void **fn) { *fn = dlsym(h, sname); if (!*fn) all = false; };
        sym("ncclGetUniqueId", (void **)&n.getUniqueId);
        sym("ncclCommInitRank", (void **)&n.commInitRank);
        sym("ncclCommDestroy", (void **)&n.commDestroy);
        sym("ncclAllReduce", (void **)&n.allReduce);
        sym("ncclGetErrorString", (void **)&n.getErrorString);
        n.commInitRankConfig = (int (*)(void **, int, NcclId, int, void *))dlsym(h, "ncclCommInitRankConfig");
        n.ok = all;
        if (!all) n.err = "libnccl is missing required symbols";
    });
    return n;
}
std::string g_comm_error;
}  // namespace

/* One-shot all-reduce over NVLink peer memory (SURVEY §5 / §8e: the pooled-moment vectors are a few hundred bytes to 130 KB,
 * i.e. latency-bound).  Every rank owns one window  [flags | 2 slots of max_doubles]  in its own HBM, opened by the other
 * ranks of the box through CUDA IPC.  A collective is ONE kernel per rank of up to four CTAs, which walk the chunks of 1,024 doubles (each
 * chunk with its own flags and epoch): publish the chunk in the slot of this epoch's parity, release the epoch number into the own
 * flag (system scope), wait until every peer's flag shows the epoch (acquire loads over NVLink), then sum the W slots in
 * RANK ORDER — so every rank holds bitwise the same result, whatever
 * the arrival order — and write it back in place.  Two slots suffice: a rank can publish epoch e + 2 only after it has
 * seen every peer's flag for e + 1, which a peer raises after it has finished reading epoch e.  The epoch counter lives on
 * the device and is advanced by the kernel, so the collective replays inside CUDA graphs.  Waits are bounded (trap). */
struct PeerWindow {
    char *local = nullptr;              /* this rank's window (cudaMalloc) */
    char **peers_dev = nullptr;         /* device array [world] of window base pointers (own entry = local) */
    unsigned long long *epoch_dev = nullptr;
    std::vector<void *> opened;         /* cudaIpcOpenMemHandle results, to close */
    long long max_doubles = 0;
    bool connected = false, enabled = false;
};
#define ME_PEER_CHUNK 1024              /* doubles per chunk of the collective: each chunk has its own flags and epoch */
#define ME_PEER_MAX_CHUNKS 32
#define ME_PEER_HEADER (2 * ME_PEER_MAX_CHUNKS * 8)     /* bytes in front of the slots: flag[2][ME_PEER_MAX_CHUNKS] (u64) */
#define ME_PEER_THREADS 256
#define ME_PEER_MAX_CTAS 4              /* the CTAs of one collective fit one SM together (the shared-covariance step kernel
                                           leaves few SMs free): a CTA takes the chunks b, b + grid, ... in order, the same
                                           order on every rank, so resident CTAs never wait for chunks of non-resident ones */

struct me_comm {
    void *nccl = nullptr;      /* ncclComm_t */
    int world = 1, rank = 0, device = 0;
    bool owned = false;
    PeerWindow peer;
};

/* the chunks of ME_PEER_CHUNK doubles are independent collectives (own flag, own epoch counter) */
__global__ void __launch_bounds__(ME_PEER_THREADS) k_peer_allreduce(double *buf, long long n, char *const *peers, int world,
                                                                    int rank, unsigned long long *epoch_ctr,
                                                                    long long max_doubles) {
    __shared__ unsigned long long ep;
    const int n_chunks = (int)((n + ME_PEER_CHUNK - 1) / ME_PEER_CHUNK);
    for (int chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x) {
        __syncthreads();
        if (threadIdx.x == 0) ep = epoch_ctr[chunk] + 1ull;
        __syncthreads();
        const unsigned long long e = ep;
        const int par = (int)(e & 1ull);
        const long long lo = (long long)chunk * ME_PEER_CHUNK;
        const long long hi = lo + ME_PEER_CHUNK < n ? lo + ME_PEER_CHUNK : n;
        const long long slot_off = (long long)par * max_doubles;
        double *mine = reinterpret_cast<double *>(peers[rank] + ME_PEER_HEADER) + slot_off;
        for (long long i = lo + threadIdx.x; i < hi; i += ME_PEER_THREADS) mine[i] = buf[i];
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned long long *flag = reinterpret_cast<unsigned long long *>(peers[rank]) + par * ME_PEER_MAX_CHUNKS + chunk;
            asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(e) : "memory");
            epoch_ctr[chunk] = e;
        }
        if ((int)threadIdx.x < world && (int)threadIdx.x != rank) {
            const unsigned long long *flag =
                reinterpret_cast<const unsigned long long *>(peers[threadIdx.x]) + par * ME_PEER_MAX_CHUNKS + chunk;
            unsigned long long seen = 0;
            unsigned spin = 0;
            for (;;) {
                asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(flag) : "memory");
                if (seen >= e) break;
                __nanosleep(spin < 1024u ? 50u : 1000u);
                if (++spin > (1u << 25)) __trap();         /* > 30 s: a peer never arrived; do not hang the GPU for good */
            }
        }
        __syncthreads();
        /* four elements per thread; ranks in order (the sum is the same bits
           on every rank); cache-volatile loads: the slots are rewritten every other epoch */
        constexpr int EPT = ME_PEER_CHUNK / ME_PEER_THREADS;
        double sum[EPT];
#pragma unroll
        for (int k = 0; k < EPT; k++) sum[k] = 0.0;
        for (int r0 = 0; r0 < world; r0 += 4) {            /* the loads from four ranks in flight together */
            double v[4][EPT];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int r = r0 + q < world ? r0 + q : rank;
                const double *slot = reinterpret_cast<const double *>(peers[r] + ME_PEER_HEADER) + slot_off;
#pragma unroll
                for (int k = 0; k < EPT; k++) {
                    const long long i = lo + threadIdx.x + (long long)k * ME_PEER_THREADS;
                    v[q][k] = (i < hi && r0 + q < world) ? __ldcv(slot + i) : 0.0;
                }
            }
#pragma unroll
            for (int q = 0; q < 4; q++)
#pragma unroll
                for (int k = 0; k < EPT; k++)
                    if (r0 + q < world) sum[k] += v[q][k];
        }
#pragma unroll
        for (int k = 0; k < EPT; k++) {
            const long long i = lo + threadIdx.x + (long long)k * ME_PEER_THREADS;
            if (i < hi) buf[i] = sum[k];
        }
    }
}

/* sum all-reduce of buf[0..n) over the ranks of `c`, in place, stream-ordered: peer windows when connected, else NCCL */
static int comm_allreduce(me_comm *c, double *buf, long long n, cudaStream_t st, std::string &err) {
    if (!c || c->world <= 1 || n <= 0) return ME_OK;
    if (c->peer.enabled && n <= c->peer.max_doubles) {
        const int chunks = (int)((n + ME_PEER_CHUNK - 1) / ME_PEER_CHUNK);
        k_peer_allreduce<<<chunks < ME_PEER_MAX_CTAS ? chunks : ME_PEER_MAX_CTAS, ME_PEER_THREADS, 0, st>>>(buf, n, c->peer.peers_dev, c->world, c->rank,
                                                             c->peer.epoch_dev, c->peer.max_doubles);
        cudaError_t ce = cudaGetLastError();
        if (ce != cudaSuccess) { err = std::string("k_peer_allreduce: ") + cudaGetErrorString(ce); return ME_ERR_CUDA; }
        return ME_OK;
    }
    if (!c->nccl) { err = "no NCCL communicator and no peer windows"; return ME_ERR_STATE; }
    NcclApi &nc = nccl_api();
    const int rc = nc.allReduce(buf, buf, (size_t)n, 8 /* ncclDouble */, 0 /* ncclSum */, c->nccl, st);
    if (rc != 0) { err = std::string("ncclAllReduce: ") + nc.getErrorString(rc); return ME_ERR_CUDA; }
    return ME_OK;
}

extern "C" {

int me_comm_set_library(const char *path) {
    if (!path) return ME_ERR_INVALID;
    g_nccl_path = path;
    return ME_OK;
}

int me_comm_unique_id(unsigned char *id128) {
    if (!id128) return ME_ERR_INVALID;
    NcclApi &n = nccl_api();
    if (!n.ok) { g_comm_error = n.err; return ME_ERR_UNSUPPORTED; }
    NcclId id;
    const int rc = n.getUniqueId(&id);
    if (rc != 0) { g_comm_error = std::string("ncclGetUniqueId: ") + n.getErrorString(rc); return ME_ERR_CUDA; }
    memcpy(id128, id.internal, 128);
    return ME_OK;
}

int me_comm_create(const unsigned char *id128, int32_t world, int32_t rank, int32_t device, me_comm **out) {
    if (!id128 || !out || world < 1 || rank < 0 || rank >= world) return ME_ERR_INVALID;
    NcclApi &n = nccl_api();
    if (!n.ok) { g_comm_error = n.err; return ME_ERR_UNSUPPORTED; }
    NcclId id;
    memcpy(id.internal, id128, 128);
    DeviceGuard g(device);
    void *comm = nullptr;
    int rc;
    if (n.commInitRankConfig) {
        /* The collectives of this communicator are latency-bound vectors of at most 130 KB, and they run on a side stream
           beside kernels that fill the GPU (the shared-covariance step kernel leaves ONE SM free): a multi-CTA all-reduce
           then waits for the step kernel's CTAs to retire before its own CTAs can all become resident.  Measured at 4
           ranks (bench c4): 21.8 ms per pass with NCCL's default CTA count, 15.1 ms with one CTA.  The prefix of
           ncclConfig_t that NCCL 2.17 introduced (later versions fill in defaults for the fields this version lacks). */
        struct { size_t size; unsigned magic, version; int blocking, cgaClusterSize, minCTAs, maxCTAs; const char *netName; } cfg;
        int max_ctas = 1;
        if (const char *env = getenv("ME_NCCL_MAX_CTAS")) max_ctas = atoi(env) > 0 ? atoi(env) : 1;
        cfg.size = sizeof(cfg); cfg.magic = 0xcafebeefu; cfg.version = 21700;
        cfg.blocking = cfg.cgaClusterSize = (int)0x80000000;                      /* NCCL_CONFIG_UNDEF_INT */
        cfg.minCTAs = 1; cfg.maxCTAs = max_ctas; cfg.netName = nullptr;
        rc = n.commInitRankConfig(&comm, world, id, rank, &cfg);
        if (rc != 0) { comm = nullptr; rc = n.commInitRank(&comm, world, id, rank); }      /* older NCCL: plain communicator */
    } else {
        rc = n.commInitRank(&comm, world, id, rank);
    }
    if (rc != 0) { g_comm_error = std::string("ncclCommInitRank: ") + n.getErrorString(rc); return ME_ERR_CUDA; }
    me_comm *c = new me_comm();
    c->nccl = comm; c->world = world; c->rank = rank; c->device = device; c->owned = true;
    *out = c;
    return ME_OK;
}

int me_comm_adopt(void *nccl_comm, int32_t world, int32_t rank, int32_t device, me_comm **out) {
    if (!nccl_comm || !out || world < 1 || rank < 0 || rank >= world) return ME_ERR_INVALID;
    NcclApi &n = nccl_api();
    if (!n.ok) { g_comm_error = n.err; return ME_ERR_UNSUPPORTED; }
    me_comm *c = new me_comm();
    c->nccl = nccl_comm; c->world = world; c->rank = rank; c->device = device; c->owned = false;
    *out = c;
    return ME_OK;
}

int me_comm_destroy(me_comm *c) {
    if (!c) return ME_OK;
    if (c->peer.local) {
        DeviceGuard g(c->device);
        for (void *q : c->peer.opened) cudaIpcCloseMemHandle(q);
        if (c->peer.peers_dev) cudaFree(c->peer.peers_dev);
        if (c->peer.epoch_dev) cudaFree(c->peer.epoch_dev);
        cudaFree(c->peer.local);
        cudaGetLastError();
    }
    if (c->owned && c->nccl) nccl_api().commDestroy(c->nccl);
    delete c;
    return ME_OK;
}

/* Peer windows, step 1: allocate this rank's window for vectors of up to max_doubles and export its CUDA IPC handle
   (64 bytes) — the host carries the handles of all ranks to every rank (any transport). */
int me_comm_peer_init(me_comm *c, int64_t max_doubles, unsigned char *handle64) {
    if (!c || !handle64 || max_doubles <= 0 || max_doubles > (int64_t)ME_PEER_CHUNK * ME_PEER_MAX_CHUNKS) return ME_ERR_INVALID;
    if (c->peer.local) { g_comm_error = "peer window already initialised"; return ME_ERR_STATE; }
    DeviceGuard g(c->device);
    const size_t bytes = ME_PEER_HEADER + sizeof(double) * 2 * (size_t)max_doubles;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
    cudaIpcMemHandle_t h;
    if (cudaMalloc((void **)&c->peer.local, bytes) != cudaSuccess || cudaMemset(c->peer.local, 0, bytes) != cudaSuccess ||
        cudaMalloc((void **)&c->peer.epoch_dev, sizeof(unsigned long long) * ME_PEER_MAX_CHUNKS) != cudaSuccess ||
        cudaMemset(c->peer.epoch_dev, 0, sizeof(unsigned long long) * ME_PEER_MAX_CHUNKS) != cudaSuccess ||
        cudaDeviceSynchronize() != cudaSuccess || cudaIpcGetMemHandle(&h, c->peer.local) != cudaSuccess) {
        g_comm_error = std::string("me_comm_peer_init: ") + cudaGetErrorString(cudaGetLastError());
        if (c->peer.local) cudaFree(c->peer.local);
        if (c->peer.epoch_dev) cudaFree(c->peer.epoch_dev);
        c->peer.local = nullptr; c->peer.epoch_dev = nullptr;
        cudaGetLastError();
        return ME_ERR_CUDA;
    }
    c->peer.max_doubles = max_doubles;
    memcpy(handle64, &h, 64);
    return ME_OK;
}

/* step 2: open the windows of all ranks (handles[world][64], own entry ignored).  Collective in spirit: every rank must
   succeed before any rank enables the windows (step 3), so the host agrees on the outcome in between. */
int me_comm_peer_connect(me_comm *c, const unsigned char *handles) {
    if (!c || !handles || !c->peer.local) return ME_ERR_INVALID;
    DeviceGuard g(c->device);
    std::vector<char *> ptrs((size_t)c->world, nullptr);
    for (int r = 0; r < c->world; r++) {
        if (r == c->rank) { ptrs[r] = c->peer.local; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, handles + 64 * (size_t)r, 64);
        void *q = nullptr;
        if (cudaIpcOpenMemHandle(&q, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            g_comm_error = std::string("cudaIpcOpenMemHandle (rank ") + std::to_string(r) + "): " +
                           cudaGetErrorString(cudaGetLastError());
            return ME_ERR_CUDA;
        }
        c->peer.opened.push_back(q);
        ptrs[r] = (char *)q;
    }
    if (cudaMalloc((void **)&c->peer.peers_dev, sizeof(char *) * (size_t)c->world) != cudaSuccess ||
        cudaMemcpy(c->peer.peers_dev, ptrs.data(), sizeof(char *) * (size_t)c->world, cudaMemcpyHostToDevice) != cudaSuccess) {
        g_comm_error = std::string("me_comm_peer_connect: ") + cudaGetErrorString(cudaGetLastError());
        return ME_ERR_CUDA;
    }
    c->peer.connected = true;
    return ME_OK;
}

/* step 3: route the collectives of this communicator through the peer windows (enable != 0) or through NCCL */
int me_comm_peer_enable(me_comm *c, int32_t enable) {
    if (!c) return ME_ERR_INVALID;
    if (enable && !c->peer.connected) { g_comm_error = "peer windows are not connected"; return ME_ERR_STATE; }
    c->peer.enabled = enable != 0;
    return ME_OK;
}

/* sum all-reduce of buf[0..n) doubles over the ranks, in place, stream-ordered (peer windows when enabled and n fits, else
   NCCL); what me_allreduce_stats / me_accumulate_stats use, exported for the shared-covariance path's moment vector */
int me_comm_allreduce(me_comm *c, double *buf, int64_t n, void *stream) {
    if (!c || !buf || n < 0) return ME_ERR_INVALID;
    DeviceGuard g(c->device);
    std::string err;
    const int rc = comm_allreduce(c, buf, n, (cudaStream_t)stream, err);
    if (rc != ME_OK) g_comm_error = err;
    return rc;
}

const char *me_comm_last_error(void) { return g_comm_error.c_str(); }

/* first half of me_allreduce_stats: inc = fixed-order sum of the per-CTA accumulators (which are reset) | n_samples */
int me_reduce_stats(me_engine *e, double *inc, int64_t n_samples, void *stream) {
    if (!e || !inc || n_samples < 0) return ME_ERR_INVALID;
    if (!e->bound || !e->buf.pool || pool_words(e) == 0) return fail(e, ME_ERR_STATE, "no pool buffer bound");
    DeviceGuard g(e->cfg.device);
    const int words = pool_words(e);
    cudaStream_t st = (cudaStream_t)stream;
    if (e->grid > 4096 && words <= 256) {
        if (!e->pool_partial &&
            cudaMalloc(&e->pool_partial, sizeof(double) * ME_POOL_STAGE_CTAS * words) != cudaSuccess) {
            cudaGetLastError();
            return fail(e, ME_ERR_CUDA, "pool reduce: cannot allocate the partial-sum rows");
        }
        k_pool_partial<<<ME_POOL_STAGE_CTAS, 256, 0, st>>>(e->buf.pool, e->pool_partial, e->grid, words, 1);
        k_pool_reduce<<<words + 1, 256, 0, st>>>(e->pool_partial, inc, ME_POOL_STAGE_CTAS, words, 0, 1, (double)n_samples);
    } else {
        k_pool_reduce<<<words + 1, 256, 0, st>>>(e->buf.pool, inc, e->grid, words, 1, 1, (double)n_samples);
    }
    cudaError_t ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail(e, ME_ERR_CUDA, std::string("me_reduce_stats: ") + cudaGetErrorString(ce));
    return ME_OK;
}

/* second half: inc summed over the ranks of `comm` in place, totals += inc.  May run on another stream than the stepping
   launches (ordered after me_reduce_stats by an event), so that the collective overlaps the next launch. */
int me_accumulate_stats(me_engine *e, me_comm *comm, double *inc, double *totals, void *stream) {
    if (!e || !inc || !totals) return ME_ERR_INVALID;
    if (pool_words(e) == 0) return fail(e, ME_ERR_STATE, "no pooled moments for this shape");
    DeviceGuard g(e->cfg.device);
    const int words = pool_words(e);
    cudaStream_t st = (cudaStream_t)stream;
    if (comm && comm->world > 1) {
        std::string err;
        const int rc = comm_allreduce(comm, inc, words + 1, st, err);
        if (rc != ME_OK) return fail(e, rc, err);
    }
    k_accumulate<<<(words + 1 + 127) / 128, 128, 0, st>>>(totals, inc, words + 1);
    cudaError_t ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail(e, ME_ERR_CUDA, std::string("me_accumulate_stats: ") + cudaGetErrorString(ce));
    return ME_OK;
}

int me_allreduce_stats(me_engine *e, me_comm *comm, double *inc, double *totals, int64_t n_samples, void *stream) {
    if (!e || !inc || !totals || n_samples < 0) return ME_ERR_INVALID;
    const int rc = me_reduce_stats(e, inc, n_samples, stream);
    if (rc != ME_OK) return rc;
    return me_accumulate_stats(e, comm, inc, totals, stream);
}

int me_get_counters(me_engine *e, int64_t *n_measure, uint64_t *step) {
    if (!e) return ME_ERR_INVALID;
    if (n_measure) *n_measure = e->n_measure;
    if (step) *step = e->step;
    return ME_OK;
}

int me_set_counters(me_engine *e, int64_t n_measure, uint64_t step) {
    if (!e || n_measure < 1) return ME_ERR_INVALID;
    e->n_measure = n_measure;
    e->step = step;
    return ME_OK;
}

int me_probe_fp64(int32_t device, int64_t iters, double *out, int64_t out_len, void *stream, int64_t *flops) {
    if (!out || iters <= 0) return ME_ERR_INVALID;
    int n_sm = 0;
    if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) {
        cudaGetLastError();
        return ME_ERR_CUDA;
    }
    const int block = 256, grid = n_sm * 8;
    if (out_len < (int64_t)grid * block) return ME_ERR_INVALID;
    DeviceGuard g(device);
    k_probe_fp64<<<grid, block, 0, (cudaStream_t)stream>>>(out, iters);
    if (cudaGetLastError() != cudaSuccess) return ME_ERR_CUDA;
    if (flops) *flops = (int64_t)grid * block * iters * 8 * 2;
    return ME_OK;
}

int me_statistical_inefficiency(const double *ts, int64_t rows, int64_t row0, int32_t cols, int64_t ld, int32_t col,
                                int64_t chain0, int64_t n_sel, int64_t max_lag, double *g_out, void *stream) {
    if (!ts || !g_out || rows <= 0 || row0 < 0 || row0 >= rows || col < 0 || col >= cols || n_sel <= 0 ||
        chain0 < 0 || chain0 + n_sel > ld)
        return ME_ERR_INVALID;
    const int block = 128;
    k_stat_ineff<<<(unsigned)((n_sel + block - 1) / block), block, 0, (cudaStream_t)stream>>>(
        ts, rows, row0, cols, ld, col, chain0, n_sel, max_lag > 0 ? max_lag : rows, g_out);
    if (cudaGetLastError() != cudaSuccess) return ME_ERR_CUDA;
    return ME_OK;
}

int me_detect_equilibration(const double *ts, int64_t rows, int32_t cols, int64_t ld, int32_t col, int64_t chain0,
                            int64_t n_sel, int64_t nskip, int32_t fast, double *scratch, int64_t scratch_doubles,
                            double *t_out, double *g_out, double *neff_out, void *stream) {
    if (!ts || !scratch || !t_out || !g_out || !neff_out || rows < 3 || cols <= 0 || col < 0 || col >= cols ||
        n_sel <= 0 || chain0 < 0 || chain0 + n_sel > ld || nskip <= 0)
        return ME_ERR_INVALID;
    const long long n_cand = (rows - 1 + nskip - 1) / nskip;        /* t0 in range(0, T - 1, nskip) */
    if (scratch_doubles < 2 * n_cand * n_sel) return ME_ERR_INVALID;
    const int block = 128;
    const unsigned gx = (unsigned)((n_sel + block - 1) / block);
    const dim3 grid(gx, (unsigned)(n_cand < 65535 ? n_cand : 65535));
    double *g_t = scratch, *neff_t = scratch + n_cand * n_sel;
    k_equil_scan<<<grid, block, 0, (cudaStream_t)stream>>>(ts, rows, cols, ld, col, chain0, n_sel, nskip, n_cand, fast ? 1 : 0, 3,
                                                          g_t, neff_t);
    k_equil_pick<<<gx, block, 0, (cudaStream_t)stream>>>(g_t, neff_t, n_cand, n_sel, nskip, t_out, g_out, neff_out);
    if (cudaGetLastError() != cudaSuccess) return ME_ERR_CUDA;
    return ME_OK;
}

int me_mbar_words(me_engine *e, int32_t n_target, int32_t with_obs, int64_t *words) {
    if (!e || !words) return ME_ERR_INVALID;
    const int rc = mbar_check(e, n_target);
    if (rc != ME_OK) return rc;
    MbarLayout m;
    mbar_layout(e->lay.D, e->n_rungs + n_target, with_obs ? 1 : 0, m);
    *words = m.words;
    return ME_OK;
}

int me_mbar_pass(me_engine *e, const double *ts, int64_t rows, int64_t row0, int64_t stride, const double *f,
                 int64_t n_per_state, int32_t n_target, const double *target_temps, const double *target_consts,
                 int32_t with_obs, double *sums, int32_t accumulate, void *stream) {
    if (!e) return ME_ERR_INVALID;
    int rc = mbar_check(e, n_target);
    if (rc != ME_OK) return rc;
    if (!ts || !f || !sums) return fail(e, ME_ERR_INVALID, "ts, f and sums are required");
    MeMbarParams q;
    memset(&q, 0, sizeof(q));
    rc = mbar_samples(e, ts, rows, row0, stride, f, n_per_state, q);
    if (rc != ME_OK) return rc;
    rc = mbar_states(e, n_target, target_temps, target_consts, q);
    if (rc != ME_OK) return rc;
    if (!e->ks.mbar.valid()) return fail(e, ME_ERR_STATE, "no MBAR kernel for this engine (device functors only)");
    const int S = q.n_states;
    MbarLayout m;
    mbar_layout(e->lay.D, S, with_obs ? 1 : 0, m);
    q.nb = m.nb; q.nx = m.nx; q.n_tiles = m.n_tiles; q.z_rows = m.z_rows; q.rw = m.rw;
    memcpy(q.tile_a, m.ta, sizeof(m.ta));
    memcpy(q.tile_b, m.tb, sizeof(m.tb));
    double *raw = nullptr;
    rc = mbar_launch(e, e->ks.mbar, q, (m.n_tiles * 64 + m.z_rows * ME_MBAR_LD) * 8, false, (cudaStream_t)stream,
                     raw);
    if (rc != ME_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    k_mbar_unpack<<<(unsigned)((m.words + 127) / 128), 128, 0, st>>>(raw, sums, S, m.nb, m.nx, e->lay.D, m.words,
                                                                    accumulate ? 1 : 0);
    cudaError_t ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail(e, ME_ERR_CUDA, std::string("MBAR pass: ") + cudaGetErrorString(ce));
    return ME_OK;
}

int me_mbar_hist_words(me_engine *e, int32_t n_axes, const int32_t *n_bins, int64_t *words) {
    if (!e || !words) return ME_ERR_INVALID;
    int rc = mbar_check(e, 0);
    if (rc != ME_OK) return rc;
    long long B = 0;
    rc = mbar_hist_bins(e, n_axes, n_bins, B);
    if (rc != ME_OK) return rc;
    *words = 4 + B * (e->n_rungs + 2);
    return ME_OK;
}

int me_mbar_hist_pass(me_engine *e, const double *ts, int64_t rows, int64_t row0, int64_t stride, const double *f,
                      int64_t n_per_state, double target_temp, const double *target_consts, int32_t n_axes,
                      const int32_t *coord_kind, const int32_t *coord_index, const double *lo, const double *hi,
                      const int32_t *n_bins, double *sums, int32_t accumulate, void *stream) {
    if (!e) return ME_ERR_INVALID;
    int rc = mbar_check(e, 0);
    if (rc != ME_OK) return rc;
    if (!ts || !f || !sums) return fail(e, ME_ERR_INVALID, "ts, f and sums are required");
    if (!coord_kind || !coord_index || !lo || !hi)
        return fail(e, ME_ERR_INVALID, "coord_kind, coord_index, lo and hi are required");
    long long B = 0;
    rc = mbar_hist_bins(e, n_axes, n_bins, B);
    if (rc != ME_OK) return rc;
    MeMbarParams q;
    memset(&q, 0, sizeof(q));
    for (int a = 0; a < n_axes; a++) {
        if (coord_kind[a] == 0) {
            if (coord_index[a] < 0 || coord_index[a] >= e->lay.D)
                return fail(e, ME_ERR_INVALID, "a column coordinate must lie in [0, D)");
        } else if (coord_kind[a] == 1) {
            if (coord_index[a] < 0 || coord_index[a] >= e->cfg.n_complex)
                return fail(e, ME_ERR_INVALID, "a modulus coordinate must name a complex parameter in [0, n_complex)");
        } else {
            return fail(e, ME_ERR_INVALID, "coord_kind must be 0 (column) or 1 (modulus of a complex parameter)");
        }
        if (!std::isfinite(lo[a]) || !std::isfinite(hi[a]) || !(hi[a] > lo[a]))
            return fail(e, ME_ERR_INVALID, "every axis needs finite lo and hi with hi > lo");
        q.axis_kind[a] = coord_kind[a];
        q.axis_index[a] = coord_index[a];
        q.axis_lo[a] = lo[a];
        q.axis_hi[a] = hi[a];
        q.axis_inv_w[a] = (double)n_bins[a] / (hi[a] - lo[a]);
        q.n_bins[a] = n_bins[a];
    }
    rc = mbar_samples(e, ts, rows, row0, stride, f, n_per_state, q);
    if (rc != ME_OK) return rc;
    const int R = e->n_rungs;
    if (e->rung_k > 0 && !target_consts)
        return fail(e, ME_ERR_INVALID, "the target of a Hamiltonian ladder needs its constants (target_consts)");
    rc = mbar_states(e, 0, nullptr, nullptr, q);
    if (rc != ME_OK) return rc;
    rc = mbar_state(e, -1, target_temp, target_consts, q.t_inv_temp, q.t_consts);
    if (rc != ME_OK) return rc;
    if (!e->ks.mbar_hist.valid()) return fail(e, ME_ERR_STATE, "no MBAR kernel for this engine (device functors only)");
    q.n_states = R + 1;
    q.n_axes = n_axes;
    q.hw = (int)(B * (R + 2));
    q.z_rows = 2 * (R + 1);
    q.rw = 4 + q.hw;
    double *raw = nullptr;
    rc = mbar_launch(e, e->ks.mbar_hist, q, (q.hw + q.z_rows * ME_MBAR_LD) * 8, true, (cudaStream_t)stream, raw);
    if (rc != ME_OK) return rc;
    k_mbar_hist_unpack<<<(unsigned)((q.rw + 127) / 128), 128, 0, (cudaStream_t)stream>>>(raw, sums, q.rw,
                                                                                         accumulate ? 1 : 0);
    cudaError_t ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail(e, ME_ERR_CUDA, std::string("MBAR histogram pass: ") + cudaGetErrorString(ce));
    return ME_OK;
}

int me_mbar_cov_words(me_engine *e, int32_t n_target, int32_t cov_first, int32_t cov_count, int64_t *words) {
    if (!e || !words) return ME_ERR_INVALID;
    MbarCovLayout m;
    const int rc = mbar_cov_check(e, n_target, cov_first, cov_count, m);
    if (rc != ME_OK) return rc;
    *words = m.words;
    return ME_OK;
}

int me_mbar_cov_pass(me_engine *e, const double *ts, int64_t rows, int64_t row0, int64_t stride, const double *f,
                     int64_t n_per_state, int32_t n_target, const double *target_temps, const double *target_consts,
                     int32_t cov_first, int32_t cov_count, const double *centers, double *sums, int32_t accumulate,
                     void *stream) {
    if (!e) return ME_ERR_INVALID;
    MbarCovLayout m;
    int rc = mbar_cov_check(e, n_target, cov_first, cov_count, m);
    if (rc != ME_OK) return rc;
    if (!ts || !f || !sums) return fail(e, ME_ERR_INVALID, "ts, f and sums are required");
    if (!centers) return fail(e, ME_ERR_INVALID, "centers is required");
    MeMbarParams q;
    memset(&q, 0, sizeof(q));
    rc = mbar_samples(e, ts, rows, row0, stride, f, n_per_state, q);
    if (rc != ME_OK) return rc;
    rc = mbar_states(e, n_target, target_temps, target_consts, q);
    if (rc != ME_OK) return rc;
    if (!e->ks.mbar_cov.valid()) return fail(e, ME_ERR_STATE, "no MBAR kernel for this engine (device functors only)");
    q.nb = m.nb; q.n_tiles = m.n_tiles; q.z_rows = m.z_rows; q.rw = m.rw;
    q.centers = centers; q.cov_first = cov_first; q.n_cov = cov_count; q.cov_mb = m.mb;
    memcpy(q.cov_tile_a, m.ta, sizeof(m.ta));
    memcpy(q.cov_tile_b, m.tb, sizeof(m.tb));
    double *raw = nullptr;
    rc = mbar_launch(e, e->ks.mbar_cov, q, m.per_warp, false, (cudaStream_t)stream, raw);
    if (rc != ME_OK) return rc;
    k_mbar_cov_unpack<<<(unsigned)((m.words + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
        raw, sums, e->n_rungs, m.nb, m.mb, m.m, cov_first, m.words, accumulate ? 1 : 0);
    cudaError_t ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail(e, ME_ERR_CUDA, std::string("MBAR covariance pass: ") + cudaGetErrorString(ce));
    return ME_OK;
}

const char *me_last_error(me_engine *e) { return e ? e->err.c_str() : g_create_error.c_str(); }

}  // extern "C"
