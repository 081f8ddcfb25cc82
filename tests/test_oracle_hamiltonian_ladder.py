"""Hamiltonian ladders without a GPU: the C oracle's ``meo_run_hladder`` (oracle/me_oracle_hladder.c) against its
temperature ladder and against the exact Gaussian ladder, and the argument checks of ``me_set_hamiltonian_ladder`` that
run before any device allocation."""
import ctypes

import numpy as np
import pytest


def test_equal_constants_reproduce_the_temperature_ladder():
    """With the same constants on every rung, D = (1/T_a - 1/T_b)(E_b - E_a): the swaps, states, walkers and counts of
    the temperature ladder (decisions exact, states to the last bits of the reordered D)."""
    from oracle import hladder_oracle as ho
    from oracle import ladder_oracle as co
    temps = np.geomspace(0.1, 2.0, 8)
    for chain0 in (0, 8, 40):
        a = co.CLadder(2, 1, "mixed_well", temps, swap_every=1, x0=[0.3, 0.3, 0.2, -0.1], chain0=chain0,
                       consts=[1.0, -1.0, 0.5])
        b = ho.CHLadder(2, 1, "mixed_well", temps, np.tile([1.0, -1.0, 0.5], (8, 1)), swap_every=1,
                        x0=[0.3, 0.3, 0.2, -0.1], chain0=chain0)
        a.run(40, 5, seed=7)
        b.run(40, 5, seed=7)
        assert np.array_equal(a.walker, b.walker)
        assert np.array_equal(a.swap_acc, b.swap_acc) and np.array_equal(a.swap_att, b.swap_att)
        assert a.swap_acc.sum() > 0
        assert np.allclose(a.states, b.states, rtol=1e-13, atol=1e-15)


def _exp_ladder_acceptance(ka, kb):
    """E_r = k_r (x^2 + y^2) at one T: r = |x|^2 is exponential with mean T / k, so D = (k_a - k_b)(e_b / k_b - e_a / k_a)
    with e_a, e_b ~ Exp(1); the swap acceptance is E[min(1, exp(-D))]."""
    from scipy.integrate import dblquad

    def f(ea, eb):
        d = (ka - kb) * (eb / kb - ea / ka)
        return min(1.0, np.exp(-d)) * np.exp(-ea - eb)
    return dblquad(f, 0, 60, 0, 60, epsabs=1e-10)[0]


def test_gaussian_ladder_variance_and_swap_acceptance():
    """xy-well rungs k = (1, 0.3) at T = 0.5: each coordinate has variance T / (2 k_r), and the swap acceptance is the
    exact Gaussians' E[min(1, exp(-D))]."""
    from oracle import hladder_oracle as ho
    ks, T, n_lad = np.array([1.0, 0.3]), 0.5, 192
    x2 = np.zeros((n_lad, 2))
    acc = np.zeros(n_lad)
    att = 0
    for i in range(n_lad):
        lad = ho.CHLadder(2, 0, "xy_well", [T, T], ks[:, None], swap_every=1, x0=np.zeros(2), chain0=2 * i,
                          sampling_width=0.5)
        lad.run(200, 5, seed=3)                                       # burn-in
        lad.swap_acc[:] = 0
        lad.swap_att[:] = 0
        s = np.zeros(2)
        for j in range(10):
            lad.run(100, 5, seed=3, step0=1000 + 500 * j)
            s += (lad.x ** 2).mean(axis=1)
        x2[i] = s / 10
        acc[i] = lad.swap_acc[0] / lad.swap_att[0]
        att = lad.swap_att[0]
    assert att > 0
    for r in range(2):
        se = x2[:, r].std() / np.sqrt(n_lad)
        assert abs(x2[:, r].mean() - T / (2 * ks[r])) < 5 * se, (r, x2[:, r].mean(), T / (2 * ks[r]), se)
    want = _exp_ladder_acceptance(ks[0], ks[1])
    se = acc.std() / np.sqrt(n_lad)
    assert abs(acc.mean() - want) < 5 * se, (acc.mean(), want, se)


# ---------------------------------------------------------------- C ABI argument checks (no device needed)
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__  # noqa: F401  (puts the repository on sys.path)
    from metropolisengine_b200 import _lib
    try:
        _lib.load()
    except ImportError as e:
        pytest.skip(str(e))
    return _lib


def _handle(lib, n_chains=64, chain_offset=0):
    h = ctypes.c_void_p()
    cfg = lib.MeConfig(2, 0, n_chains, chain_offset, 0.5, 0.3, 3.49, 0, 0, 0)
    assert lib.load().me_create(ctypes.byref(cfg), ctypes.byref(h)) == lib.ME_OK
    return h


def _set(lib, h, temps, consts, K, every=1):
    R = len(temps)
    t = (ctypes.c_double * R)(*temps)
    k = (ctypes.c_double * max(len(consts), 1))(*consts)
    walker = (ctypes.c_int32 * 64)()
    sacc = (ctypes.c_uint32 * 64)()
    return lib.load().me_set_hamiltonian_ladder(h, t, k, K, R, every, ctypes.cast(walker, ctypes.c_void_p),
                                                ctypes.cast(sacc, ctypes.c_void_p))


def test_set_hamiltonian_ladder_validates_before_allocating(lib):
    L = lib.load()
    cases = [
        ([0.5, 0.5], [1.0, np.nan], 1, 1, "finite"),                      # non-finite constant
        ([0.5, 0.5], [1.0, np.inf], 1, 0, "finite"),
        ([0.5, 0.5], [], 0, 1, "1 to 16"),                                # K outside [1, 16]
        ([0.5, 0.5], [1.0] * 34, 17, 1, "1 to 16"),
        ([0.0, 0.5], [1.0, 2.0], 1, 1, "> 0"),                            # T = 0 with swaps
        ([-0.5, 0.5], [1.0, 2.0], 1, 0, ">= 0"),                          # T < 0 without
        ([0.5] * 3, [1.0, 2.0, 3.0], 1, 1, "2, 4, 8, 16 or 32"),          # R not a power of two with swaps
        ([0.5] * 64, [1.0] * 64, 1, 1, "2, 4, 8, 16 or 32"),              # R > 32 with swaps
    ]
    for temps, consts, K, every, msg in cases:
        h = _handle(lib, 192)                                             # whole ladders of 2, 3 and 64 rungs
        assert _set(lib, h, temps, consts, K, every) == lib.ME_ERR_INVALID, (temps, consts, K)
        assert msg in L.me_last_error(h).decode(), (msg, L.me_last_error(h))
        L.me_destroy(h)
    for n_chains, off in ((63, 0), (64, 2)):                              # chains that are not whole ladders of 4
        h = _handle(lib, n_chains, off)
        assert _set(lib, h, [0.5] * 4, [1.0, 2.0, 3.0, 4.0], 1) == lib.ME_ERR_INVALID
        assert "whole ladders" in L.me_last_error(h).decode()
        L.me_destroy(h)
    h = _handle(lib)                                                       # decreasing temperatures are fine here
    k1 = (ctypes.c_double * 1)(1.0)
    assert L.me_set_energy_builtin(h, lib.ENERGY_IDS["xy_well"], k1, 1, 0) == lib.ME_OK
    assert _set(lib, h, [0.5, 0.4], [1.0, 2.0, 3.0, 4.0], 2) == lib.ME_ERR_INVALID      # K = 2, functor has 1
    assert "constants" in L.me_last_error(h).decode()
    L.me_destroy(h)
