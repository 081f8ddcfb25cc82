/* me_kernels.cuh — __global__ entry points around the device bodies of me_device.cuh, and the table type the
 * host library uses to find ahead-of-time instantiations. */
#ifndef ME_KERNELS_CUH
#define ME_KERNELS_CUH

#include "me_device.cuh"
#include "me_energies.cuh"

namespace me {

template <int NR_, int NC_, template <int, int> class EnergyT, bool STRICT_>
struct Cfg {
    static constexpr int NR = NR_, NC = NC_;
    static constexpr bool STRICT = STRICT_;
    using Energy = EnergyT<NR_, NC_>;
};

/* Small problems (D <= 4) are capped at 160 registers.  The register file holds one-warp CTAs in steps: 16 per SM up to
 * 128 registers per thread, 12 from 129 to 160, 10 beyond; three warps per SM sub-partition (12 per SM) already saturate
 * its pipes, and below ~140 registers ptxas starts to re-materialise loop invariants (Philox counter words, polynomial
 * constants) inside the step loop.  Ensembles that do not fill whole waves of those 12 x 148 slots are balanced by the
 * work-queue time segmentation of run_body. */
template <class C, bool SMALL = (C::NR + 2 * C::NC <= 4)>
struct RunKernel;
#ifndef ME_SMALL_MAXNREG
#define ME_SMALL_MAXNREG 160     /* build-time experiment knob (make SMALL_NREG=...): see tests/scripts/nreg_probe.py */
#endif
template <class C>
__global__ void __maxnreg__(ME_SMALL_MAXNREG) k_run_small(const __grid_constant__ MeParams p) {
    run_body<C>(p);
}
#ifdef ME_BIG_MAXNREG
template <class C>
__global__ void __maxnreg__(ME_BIG_MAXNREG) k_run(const __grid_constant__ MeParams p) {
    run_body<C>(p);
}
#else
template <class C>
__global__ void __launch_bounds__(ME_MAX_BLOCK, 1) k_run(const __grid_constant__ MeParams p) {
    run_body<C>(p);
}
#endif
#ifndef ME_NVRTC   /* host-side selection; the run-time compiled kernels (me_api.cu) name their entry points directly */
template <class C>
struct RunKernel<C, true> { static const void *get() { return (const void *)&k_run_small<C>; } };
template <class C>
struct RunKernel<C, false> { static const void *get() { return (const void *)&k_run<C>; } };
#endif
/* temperature ladders (me_set_ladder): the same register policy as k_run_small / k_run */
template <class C>
__global__ void __maxnreg__(ME_SMALL_MAXNREG) k_run_pt_small(const __grid_constant__ MeParams p) {
    run_body<C, false, LADDER_TEMP>(p);
}
#ifdef ME_BIG_MAXNREG
template <class C>
__global__ void __maxnreg__(ME_BIG_MAXNREG) k_run_pt(const __grid_constant__ MeParams p) {
    run_body<C, false, LADDER_TEMP>(p);
}
#else
template <class C>
__global__ void __launch_bounds__(ME_MAX_BLOCK, 1) k_run_pt(const __grid_constant__ MeParams p) {
    run_body<C, false, LADDER_TEMP>(p);
}
#endif
/* Hamiltonian ladders (me_set_hamiltonian_ladder): the same register policy */
template <class C>
__global__ void __maxnreg__(ME_SMALL_MAXNREG) k_run_hx_small(const __grid_constant__ MeParams p) {
    run_body<C, false, LADDER_HAM>(p);
}
#ifdef ME_BIG_MAXNREG
template <class C>
__global__ void __maxnreg__(ME_BIG_MAXNREG) k_run_hx(const __grid_constant__ MeParams p) {
    run_body<C, false, LADDER_HAM>(p);
}
#else
template <class C>
__global__ void __launch_bounds__(ME_MAX_BLOCK, 1) k_run_hx(const __grid_constant__ MeParams p) {
    run_body<C, false, LADDER_HAM>(p);
}
#endif
#ifndef ME_NVRTC
/* caller-evaluated energies never run fused, so they get no ladder kernel */
template <class C> struct IsExternal { static constexpr bool value = false; };
template <int NR, int NC, bool S> struct IsExternal<Cfg<NR, NC, EnergyNone, S>> { static constexpr bool value = true; };
template <class C, bool SMALL = (C::NR + 2 * C::NC <= 4), bool EXT = IsExternal<C>::value>
struct RunPtKernel { static const void *get() { return (const void *)&k_run_pt_small<C>; } };
template <class C>
struct RunPtKernel<C, false, false> { static const void *get() { return (const void *)&k_run_pt<C>; } };
template <class C, bool SMALL>
struct RunPtKernel<C, SMALL, true> { static const void *get() { return nullptr; } };
template <class C, bool SMALL = (C::NR + 2 * C::NC <= 4), bool EXT = IsExternal<C>::value>
struct RunHxKernel { static const void *get() { return (const void *)&k_run_hx_small<C>; } };
template <class C>
struct RunHxKernel<C, false, false> { static const void *get() { return (const void *)&k_run_hx<C>; } };
template <class C, bool SMALL>
struct RunHxKernel<C, SMALL, true> { static const void *get() { return nullptr; } };
#endif
/* the instantiation that also performs the magnitude / phase complex moves (me_set_group 3, 4; SURVEY §8 row f4) */
template <class C>
__global__ void __launch_bounds__(ME_MAX_BLOCK, 1) k_run_mp(const __grid_constant__ MeParams p) {
    run_body<C, true>(p);
}
#ifndef ME_NVRTC
template <class C, bool HAS_COMPLEX = (C::NC > 0)>
struct RunMpKernel { static const void *get() { return (const void *)&k_run_mp<C>; } };
template <class C>
struct RunMpKernel<C, false> { static const void *get() { return nullptr; } };
#endif
template <class C>
__global__ void __launch_bounds__(ME_MAX_BLOCK) k_init(const __grid_constant__ MeParams p) { init_body<C>(p); }
template <class C>
__global__ void __launch_bounds__(ME_MAX_BLOCK) k_propose(const __grid_constant__ MeParams p) { propose_body<C>(p); }
template <class C>
__global__ void __launch_bounds__(ME_MAX_BLOCK) k_accept(const __grid_constant__ MeParams p) { accept_body<C>(p); }
template <class C>
__global__ void __launch_bounds__(ME_MAX_BLOCK) k_energy(const __grid_constant__ MeParams p) { energy_body<C>(p); }

}  // namespace me

/* one ahead-of-time instantiation */
struct MeAotEntry {
    int n_real, n_complex, energy_id, strict;
    const void *run, *init, *propose, *accept, *run_mp, *energy, *run_pt, *run_hx;
};

#define ME_AOT_ENTRY(NR, NC, ETMPL, EID, STRICT)                                                        \
    { NR, NC, EID, STRICT, me::RunKernel<me::Cfg<NR, NC, ETMPL, STRICT>>::get(),                          \
      (const void *)&me::k_init<me::Cfg<NR, NC, ETMPL, STRICT>>,                                          \
      (const void *)&me::k_propose<me::Cfg<NR, NC, ETMPL, STRICT>>,                                       \
      (const void *)&me::k_accept<me::Cfg<NR, NC, ETMPL, STRICT>>,                                        \
      me::RunMpKernel<me::Cfg<NR, NC, ETMPL, STRICT>>::get(),                                             \
      (const void *)&me::k_energy<me::Cfg<NR, NC, ETMPL, STRICT>>,                                        \
      me::RunPtKernel<me::Cfg<NR, NC, ETMPL, STRICT>>::get(),                                             \
      me::RunHxKernel<me::Cfg<NR, NC, ETMPL, STRICT>>::get() }

/* the shapes of BASELINE.json's configs plus the shapes of the golden fixtures */
#define ME_AOT_TABLE(STRICT)                                                      \
    ME_AOT_ENTRY(1, 0, me::EnergyX2, 0, STRICT),        /* C1 README            */ \
    ME_AOT_ENTRY(2, 0, me::EnergyXYWell, 1, STRICT),    /* C2 xy-well           */ \
    ME_AOT_ENTRY(2, 1, me::EnergyMixedWell, 2, STRICT), /* demo 2r+1c           */ \
    ME_AOT_ENTRY(3, 4, me::EnergyMixedWell, 2, STRICT), /* C3 mixed 3r+4c       */ \
    ME_AOT_ENTRY(1, 8, me::EnergyCylinder, 3, STRICT),  /* cylinder-shaped 1r+8c */ \
    ME_AOT_ENTRY(1, 0, me::EnergyNone, 99, STRICT),     /* caller-evaluated energies */ \
    ME_AOT_ENTRY(2, 0, me::EnergyNone, 99, STRICT),                                  \
    ME_AOT_ENTRY(2, 1, me::EnergyNone, 99, STRICT)

#endif
