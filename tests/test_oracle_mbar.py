"""MBAR without a GPU: the numpy oracle (oracle/mbar_oracle.py) pinned on routes independent of it — a generic
minimiser of the MBAR objective, Bennett's acceptance ratio, targets equal to rungs, the exact Gaussian ladder and the
calibration of its error bars — and the argument checks of ``me_mbar_pass`` that run before any device work."""
import ctypes

import numpy as np
import pytest
from scipy.optimize import brentq, minimize

from oracle import mbar_oracle as mo


def _gaussian_ladder(temps, k, n, rng):
    """iid samples of E = k (x^2 + y^2) at every T: x, y ~ N(0, T / (2k)); Z(T) = pi T / k."""
    x = np.concatenate([rng.normal(0.0, np.sqrt(t / (2 * k)), size=(n, 2)) for t in temps])
    E = np.stack([mo.energy("xy_well", x, [k]) for _ in temps])
    return x, E


def test_newton_matches_a_generic_minimiser():
    rng = np.random.default_rng(1)
    temps = np.array([0.5, 0.8, 1.3, 2.0])
    x, E = _gaussian_ladder(temps, 1.0, 400, rng)
    u = mo.reduced(E, np.zeros(E.shape, dtype=bool), temps)
    f, it, conv = mo.solve(u, 400)
    assert conv and f[0] == 0.0
    def fun(g):                           # F and its gradient N (s - 1) over f_1..f_3
        fg = np.concatenate([[0.0], g])
        p = mo.pass_sums(u, fg, 400, 4)
        return p["sum_l"] - 400 * fg.sum(), 400 * (p["s"][1:] - 1.0)
    res = minimize(fun, np.zeros(3), jac=True, method="BFGS", options=dict(gtol=1e-9))
    assert np.allclose(f[1:], res.x, rtol=0, atol=1e-8), (f, res.x)


def test_two_states_are_bennetts_acceptance_ratio():
    rng = np.random.default_rng(2)
    temps = np.array([0.7, 1.1])
    n = 3000
    x, E = _gaussian_ladder(temps, 1.5, n, rng)
    u = mo.reduced(E, np.zeros(E.shape, dtype=bool), temps)
    f, _, conv = mo.solve(u, n)
    assert conv
    w_f = u[1, :n] - u[0, :n]                   # forward work on samples of state 0
    w_r = u[0, n:] - u[1, n:]                   # reverse work on samples of state 1

    def bar(df):
        return np.sum(1.0 / (1.0 + np.exp(w_f - df))) - np.sum(1.0 / (1.0 + np.exp(w_r + df)))
    want = brentq(bar, -20, 20, xtol=1e-14)
    assert abs(f[1] - want) < 1e-10, (f[1], want)


def test_target_equal_to_a_rung_reproduces_it():
    rng = np.random.default_rng(3)
    temps = np.array([0.6, 1.0, 1.7])
    x, E = _gaussian_ladder(temps, 2.0, 500, rng)
    u = mo.reduced(E, np.zeros(E.shape, dtype=bool), temps)
    f, _, _ = mo.solve(u, 500)
    for r in range(3):
        tE = np.concatenate([E, E[r:r + 1]])
        tu = np.concatenate([u, u[r:r + 1]])
        ev = mo.evaluate(tu, tE, x, f, 500, 3)
        assert abs(ev["f"][3] - f[r]) <= 1e-12 * max(1.0, abs(f[r]))
        assert np.allclose(ev["mean"][3], ev["mean"][r], rtol=1e-12, atol=0)


def test_gaussian_ladder_free_energies_and_error_calibration():
    """f_k - f_0 = -ln(T_k / T_0) within 4 df; the z-scores over 200 seeded repeats have standard deviation in
    [0.85, 1.15], which pins the svd-ew covariance."""
    temps = np.array([0.5, 0.75, 1.1, 1.6])
    z = []
    for rep in range(200):
        rng = np.random.default_rng(100 + rep)
        x, E = _gaussian_ladder(temps, 1.0, 300, rng)
        u = mo.reduced(E, np.zeros(E.shape, dtype=bool), temps)
        f, _, conv = mo.solve(u, 300)
        assert conv
        th = mo.theta(mo.pass_sums(u, f, 300, 4)["G"], np.full(4, 300.0))
        for k in range(1, 4):
            exact = -np.log(temps[k] / temps[0])
            d = mo.df(th, 0, k)
            if rep == 0:
                assert abs(f[k] - exact) < 4 * d, (k, f[k], exact, d)
            z.append((f[k] - exact) / d)
    z = np.array(z)
    assert np.mean(np.abs(z) > 4) < 0.01
    assert 0.85 <= z.std() <= 1.15, z.std()


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


def _handle(lib, nr=2, nc=0, temp=0.5, energy="xy_well", consts=(1.0,)):
    h = ctypes.c_void_p()
    cfg = lib.MeConfig(nr, nc, 64, 0, temp, 0.3, 3.49, 0, 0, 0)
    assert lib.load().me_create(ctypes.byref(cfg), ctypes.byref(h)) == lib.ME_OK
    if energy is not None:
        k = (ctypes.c_double * len(consts))(*consts)
        assert lib.load().me_set_energy_builtin(h, lib.ENERGY_IDS[energy], k, len(consts), 0) == lib.ME_OK
    return h


_FAKE = ctypes.c_void_p(0x1000)        # never dereferenced: every case fails its checks before device work


def _pass(lib, h, rows=10, row0=0, stride=1, n_per=64, temps=(), consts=None, ts=_FAKE, f=_FAKE, sums=_FAKE):
    tt = (ctypes.c_double * max(len(temps), 1))(*temps)
    kk = None if consts is None else ctypes.cast((ctypes.c_double * len(consts))(*consts), ctypes.c_void_p)
    return lib.load().me_mbar_pass(h, ts, rows, row0, stride, f, n_per, len(temps), ctypes.cast(tt, ctypes.c_void_p),
                                   kk, 1, sums, 0, None)


def test_mbar_pass_validates_before_device_work(lib):
    L = lib.load()
    cases = [
        (dict(temp=0.0), {}, lib.ME_ERR_INVALID, "rung temperature"),          # a T = 0 rung
        ({}, dict(temps=[0.0]), lib.ME_ERR_INVALID, "target temperature"),
        ({}, dict(temps=[np.nan]), lib.ME_ERR_INVALID, "target temperature"),
        ({}, dict(temps=[np.inf]), lib.ME_ERR_INVALID, "target temperature"),
        ({}, dict(temps=[1.0], consts=[np.nan]), lib.ME_ERR_INVALID, "finite"),
        ({}, dict(temps=[1.0] * 32), lib.ME_ERR_INVALID, "32 states"),          # S = 33
        ({}, dict(row0=10), lib.ME_ERR_INVALID, "row0"),
        ({}, dict(row0=-1), lib.ME_ERR_INVALID, "row0"),
        ({}, dict(stride=0), lib.ME_ERR_INVALID, "stride"),
        ({}, dict(n_per=0), lib.ME_ERR_INVALID, "n_per_state"),
        ({}, dict(ts=None), lib.ME_ERR_INVALID, "required"),
        ({}, dict(f=None), lib.ME_ERR_INVALID, "required"),
        ({}, dict(sums=None), lib.ME_ERR_INVALID, "required"),
        (dict(energy=None), {}, lib.ME_ERR_STATE, "energy functor"),
        (dict(nr=33), {}, lib.ME_ERR_UNSUPPORTED, "fused shape"),              # D > 32
    ]
    for hk, pk, code, msg in cases:
        h = _handle(lib, **hk)
        assert _pass(lib, h, **pk) == code, (hk, pk)
        assert msg in L.me_last_error(h).decode(), (msg, L.me_last_error(h))
        L.me_destroy(h)
    h = _handle(lib, energy=None)                                             # caller-evaluated energies
    assert L.me_set_energy_external(h) == lib.ME_OK
    assert _pass(lib, h) == lib.ME_ERR_UNSUPPORTED
    L.me_destroy(h)
    h = _handle(lib)                                                          # group-wise stepping
    assert L.me_set_group(h, 1) == lib.ME_OK
    assert _pass(lib, h) == lib.ME_ERR_UNSUPPORTED
    assert "group" in L.me_last_error(h).decode()
    L.me_destroy(h)


def test_mbar_words_is_the_documented_length(lib):
    L = lib.load()
    h = _handle(lib)
    w = ctypes.c_int64()
    for n_t, obs in ((0, 0), (2, 0), (2, 1), (31, 1)):
        assert L.me_mbar_words(h, n_t, obs, ctypes.byref(w)) == lib.ME_OK
        S, D = 1 + n_t, 2
        assert w.value == 3 + S + S * (S + 1) // 2 + (S * (2 * D + 2) if obs else 0)
    assert L.me_mbar_words(h, 32, 0, ctypes.byref(w)) == lib.ME_ERR_INVALID
    L.me_destroy(h)
