"""Uncertainties of reweighted expectations without a GPU: the host algebra (metropolisengine_b200/mbar.py,
``expectation_covariance``) on the oracle's covariance sums (oracle/expectation_oracle.py) pinned against pymbar's
explicit-weight-matrix route, the invariance to the centres, the exact single-state identity, a target at a rung, the
calibration of the error bars on the exact Gaussian ladder, and the argument checks of ``me_mbar_cov_pass`` and
``me_mbar_cov_words`` that run before any device work."""
import ctypes

import numpy as np
import pytest

from metropolisengine_b200 import mbar as mb
from oracle import expectation_oracle as xo
from oracle import mbar_oracle as mo


def _ladder(temps, n, rng, k=1.0):
    return np.concatenate([rng.normal(0.0, np.sqrt(t / (2 * k)), size=(n, 2)) for t in temps])


def _states(x, temps, targets, k=1.0):
    """u [S, n] and the observables [S, n, 6] of the xy well over the rungs, then the targets."""
    allt = np.concatenate([temps, targets])
    E = np.stack([mo.energy("xy_well", x, [k])] * allt.size)
    return E / allt[:, None], mo.observables(x, E)


def _host_cov(u, obs, f, n, R, first, count, centers):
    """obs_cov of the states [first, first + count) by the host algebra on the oracle's sums."""
    p = mo.pass_sums(u, f, n, R)
    o, C, Q = xo.cov_sums(u, f, n, R, obs, first, count, centers)
    return np.stack([mb.expectation_covariance(p["G"], p["s"], first + c, o[c], C[c], Q[c], n) for c in range(count)])


def _means(u, obs, f, n, R):
    p = mo.pass_sums(u, f, n, R, obs)
    return p["obs"] / p["s"][:, None]


def _rel(a, b):
    return np.max(np.abs(a - b)) / np.max(np.abs(b))


def _gauss_case(seed=7, n=700):
    rng = np.random.default_rng(seed)
    temps = np.array([0.5, 0.75, 1.1, 1.6])
    targets = np.array([0.6, 0.9, 1.35])
    x = _ladder(temps, n, rng)
    u, obs = _states(x, temps, targets)
    f, _, conv = mo.solve(u[:4], n)
    assert conv
    return u, obs, f, n


def test_host_algebra_matches_pymbars_weight_matrix_route():
    u, obs, f, n = _gauss_case()
    R, S = 4, 7
    mean = _means(u, obs, f, n, R)
    for first, count in ((0, R), (R, S - R)):                          # the rungs, then the targets
        got = _host_cov(u, obs, f, n, R, first, count, mean[first:first + count])
        want_mean, want = xo.pymbar_expectations(u, f, n, R, obs, range(first, first + count))
        assert np.allclose(want_mean, mean[first:first + count], rtol=1e-12, atol=1e-14)
        for c in range(count):
            scale = np.abs(want[c])
            assert np.all(np.abs(got[c] - want[c]) <= 1e-8 * np.maximum(scale, 1e-3 * np.max(scale))), \
                (first + c, _rel(got[c], want[c]))
        assert _rel(got, want) < 1e-8


def test_centre_invariance():
    u, obs, f, n = _gauss_case(seed=11)
    R = 4
    mean = _means(u, obs, f, n, R)
    sd = np.sqrt(np.maximum(_means(u, obs * obs, f, n, R) - mean * mean, 0.0))
    ref = _host_cov(u, obs, f, n, R, 2, 4, mean[2:6])
    for cen in (np.zeros((4, 6)), mean[2:6] + 3 * sd[2:6]):
        got = _host_cov(u, obs, f, n, R, 2, 4, cen)
        assert _rel(got, ref) < 1e-10, _rel(got, ref)


def test_single_state_is_the_plain_standard_error():
    rng = np.random.default_rng(3)
    n = 4000
    x = rng.normal(0.0, 0.6, size=(n, 2))
    u, obs = _states(x, np.array([0.72]), np.zeros(0))
    got = _host_cov(u, obs, np.zeros(1), n, 1, 0, 1, obs[0].mean(axis=0)[None])[0]
    want = np.cov(obs[0].T, bias=True) / n
    assert _rel(got, want) < 1e-10, _rel(got, want)


def test_target_at_a_rung_reproduces_the_rung():
    rng = np.random.default_rng(5)
    temps = np.array([0.5, 0.8, 1.3])
    n = 900
    x = _ladder(temps, n, rng)
    u, obs = _states(x, temps, np.array([temps[1]]))
    f, _, _ = mo.solve(u[:3], n)
    mean = _means(u, obs, f, n, 3)
    rung = _host_cov(u, obs, f, n, 3, 1, 1, mean[1:2])[0]
    tgt = _host_cov(u, obs, f, n, 3, 3, 1, mean[3:4])[0]
    assert _rel(tgt, rung) < 1e-10, _rel(tgt, rung)


def test_exact_gaussian_ladder_calibration():
    """iid samples of the xy well k = 1: <E> = T, <x_0^2> = T / 2 and C = 1 at every temperature.  The z-scores of the
    reweighted means and of the heat capacity at targets between the rungs must have unit spread."""
    temps = np.array([0.4, 0.7, 1.2])
    targets = np.array([0.5, 0.9])
    zE, zx, zc = [], [], []
    for rep in range(200):
        rng = np.random.default_rng(1000 + rep)
        n = 600
        x = _ladder(temps, n, rng)
        u, obs = _states(x, temps, targets)
        f, _, conv = mo.solve(u[:3], n)
        assert conv
        mean = _means(u, obs, f, n, 3)
        cov = _host_cov(u, obs, f, n, 3, 3, 2, mean[3:])
        se = np.sqrt(np.diagonal(cov, axis1=1, axis2=2))
        zE.extend((mean[3:, 4] - targets) / se[:, 4])
        zx.extend((mean[3:, 2] - targets / 2) / se[:, 2])
        c, dc = mb.heat_capacity(mean[3:, 4], mean[3:, 5], cov[:, 4:, 4:], targets)
        zc.extend((c - 1.0) / dc)
    for z in (zE, zx, zc):
        z = np.array(z)
        assert np.mean(np.abs(z) > 4) < 0.01
        assert 0.85 <= z.std() <= 1.15, z.std()


def test_heat_capacity_delta_method_matches_the_oracle():
    u, obs, f, n = _gauss_case(seed=13)
    mean = _means(u, obs, f, n, 4)
    cov = _host_cov(u, obs, f, n, 4, 4, 3, mean[4:])
    T = np.array([0.6, 0.9, 1.35])
    c, dc = mb.heat_capacity(mean[4:, 4], mean[4:, 5], cov[:, 4:, 4:], T)
    for i in range(3):
        wc, wdc = xo.heat_capacity(mean[4 + i, 4], mean[4 + i, 5], cov[i, 4:, 4:], T[i])
        assert abs(c[i] - wc) <= 1e-14 * abs(wc) and abs(dc[i] - wdc) <= 1e-12 * wdc


def test_unpack_cov_layout():
    R, m, n = 3, 4, 2
    per = m + m * (R + 1) + m * (m + 1) // 2
    sums = np.concatenate([[0.0, 0.0], np.arange(n * per, dtype=np.float64)])
    out = mb.unpack_cov(sums, n, m, R)
    assert out["o"][1].tolist() == list(range(per, per + m))
    assert out["C"][0, 1, 2] == m + 1 * (R + 1) + 2
    q0 = m + m * (R + 1)
    assert out["Q"][1, 2, 1] == out["Q"][1, 1, 2] == per + q0 + 2 * 3 // 2 + 1


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


_WIDE = dict(nr=1, nc=8, energy="cylinder", consts=(1.0, 0.5, 0.1, 0.2))   # the widest shape built ahead of time
_FAKE = ctypes.c_void_p(0x1000)        # never dereferenced: every case fails its checks before device work


def _arr(t, v):
    return None if v is None else ctypes.cast((t * max(len(v), 1))(*v), ctypes.c_void_p)


def _pass(lib, h, rows=10, row0=0, stride=1, n_per=64, n_target=1, temps=(0.7,), consts=None, first=0, count=1,
          centers=_FAKE, ts=_FAKE, f=_FAKE, sums=_FAKE):
    f64 = ctypes.c_double
    return lib.load().me_mbar_cov_pass(h, ts, rows, row0, stride, f, n_per, n_target, _arr(f64, temps),
                                       _arr(f64, consts), first, count, centers, sums, 0, None)


def test_mbar_cov_pass_validates_before_device_work(lib):
    L = lib.load()
    inv, nan = lib.ME_ERR_INVALID, float("nan")
    cases = [
        ({}, dict(count=0), inv, "cov_first"),
        ({}, dict(count=-1), inv, "cov_first"),
        ({}, dict(first=-1), inv, "cov_first"),
        ({}, dict(first=2, count=1), inv, "cov_first"),
        ({}, dict(first=0, count=3), inv, "cov_first"),
        ({}, dict(centers=None), inv, "centers"),
        ({}, dict(n_target=32, temps=[0.7] * 32), inv, "32 states"),
        ({}, dict(n_target=-1), inv, "32 states"),
        ({}, dict(temps=None), inv, "target_temps"),
        ({}, dict(temps=(0.0,)), inv, "target temperature"),
        ({}, dict(temps=(nan,)), inv, "target temperature"),
        ({}, dict(consts=[nan]), inv, "finite"),
        (dict(temp=0.0), {}, inv, "rung temperature"),
        ({}, dict(row0=10), inv, "row0"),
        ({}, dict(stride=0), inv, "stride"),
        ({}, dict(n_per=0), inv, "n_per_state"),
        ({}, dict(ts=None), inv, "required"),
        ({}, dict(f=None), inv, "required"),
        ({}, dict(sums=None), inv, "required"),
        (_WIDE, dict(n_target=31, temps=[0.7] * 31, count=32), inv, "227 KB"),         # D = 17, S = 32
        (dict(energy=None), {}, lib.ME_ERR_STATE, "energy functor"),
        (dict(nr=33), {}, lib.ME_ERR_UNSUPPORTED, "fused shape"),             # D > 32
    ]
    for hk, pk, code, msg in cases:
        h = _handle(lib, **hk)
        assert _pass(lib, h, **pk) == code, (hk, pk, L.me_last_error(h))
        assert msg in L.me_last_error(h).decode(), (msg, L.me_last_error(h))
        L.me_destroy(h)
    h = _handle(lib, energy=None)                                             # caller-evaluated energies
    assert L.me_set_energy_external(h) == lib.ME_OK
    assert _pass(lib, h) == lib.ME_ERR_UNSUPPORTED
    L.me_destroy(h)
    h = _handle(lib)                                                          # group-wise stepping
    assert L.me_set_group(h, 1) == lib.ME_OK
    assert _pass(lib, h) == lib.ME_ERR_UNSUPPORTED
    L.me_destroy(h)


def _words(L, h, n_target, first, count):
    w = ctypes.c_int64()
    rc = L.me_mbar_cov_words(h, n_target, first, count, ctypes.byref(w))
    return rc, w.value


def test_mbar_cov_words_is_the_documented_length_and_fit(lib):
    L = lib.load()
    for nr, n_target, first, count in ((2, 0, 0, 1), (2, 5, 0, 6), (2, 20, 1, 20), (1, 3, 2, 1)):
        h = _handle(lib, nr=nr, energy="x2" if nr == 1 else "xy_well")
        m, R = 2 * nr + 2, 1
        rc, w = _words(L, h, n_target, first, count)
        assert rc == lib.ME_OK, L.me_last_error(h)
        assert w == 2 + count * (m + m * (R + 1) + m * (m + 1) // 2)
        L.me_destroy(h)
    h = _handle(lib, **_WIDE)                                                # D = 17, S = 32
    assert _words(L, h, 31, 0, 1)[0] == lib.ME_OK                             # one covered state always fits
    assert _words(L, h, 31, 31, 1)[0] == lib.ME_OK
    rc, _ = _words(L, h, 31, 0, 32)
    assert rc == lib.ME_ERR_INVALID and "227 KB" in L.me_last_error(h).decode()
    ok = [c for c in range(1, 33) if _words(L, h, 31, 0, c)[0] == lib.ME_OK]
    assert ok == list(range(1, len(ok) + 1)) and 1 < len(ok) < 32             # the fit is monotone in the count
    assert _words(L, h, 31, 0, 0)[0] == lib.ME_ERR_INVALID
    assert _words(L, h, 32, 0, 1)[0] == lib.ME_ERR_INVALID                    # S = 33
    L.me_destroy(h)
