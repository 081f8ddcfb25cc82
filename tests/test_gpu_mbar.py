"""MBAR over recorded ladder rows on the GPU (csrc/me_mbar.cuh, me_mbar_pass; metropolisengine_b200/mbar.py): the pass
sums against the numpy oracle (oracle/mbar_oracle.py) on the engine's own recorded rows, the solve against the oracle's
solve, analytic ladders sampled by real Metropolis chains, the invariances and the refusals."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

WALL_SRC = """
__device__ double me_user_energy(const double* x, const double* cr, const double* ci, const double* k) {
    return k[0] * (x[0] * x[0] + x[1] * x[1]);
}
__device__ bool me_user_reject(const double* x, const double* cr, const double* ci, const double* k) {
    return x[0] >= k[1];
}
"""
NAN_SRC = """
__device__ double me_user_energy(const double* x, const double* cr, const double* ci, const double* k) {
    return k[0] < 0.0 ? sqrt(k[0]) : k[0] * (x[0] * x[0] + x[1] * x[1]);
}
"""


def _me():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import metropolisengine_b200 as me
    return me


def _case(me, name, R, strict=False, n_per_rung=64, **kw):
    """(engine, numpy energy function, reject function, rung temperatures, rung constants [R, 16])."""
    from oracle import mbar_oracle as mo
    n = R * n_per_rung
    common = dict(n_chains=n, seed=11, strict=strict, device="cuda:0", **kw)
    if name == "scalar":
        eng = me.MetropolisEngine(("xy_well", 1.3), initial_real_params=np.array([0.1, -0.2]), temp=0.6, **common)
        return eng, lambda x, k: mo.energy("xy_well", x, k), None, np.array([0.6]), _pad([[1.3]])
    if name == "xy_temp":
        temps = np.geomspace(0.2, 2.0, R)
        eng = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.array([0.1, -0.2]), temp=list(temps),
                                  replica_exchange=1, **common)
        return eng, lambda x, k: mo.energy("xy_well", x, k), None, temps, _pad(np.ones((R, 1)))
    if name == "xy_ham":
        kr = np.geomspace(0.3, 3.0, R)[:, None]
        eng = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.array([0.1, -0.2]), temp=0.5,
                                  rung_consts=kr, replica_exchange=1, **common)
        return eng, lambda x, k: mo.energy("xy_well", x, k), None, np.full(R, 0.5), _pad(kr)
    if name == "mixed_ham":
        kr = np.stack([np.linspace(0.5, 1.5, R), np.linspace(-1.0, -0.2, R), np.linspace(0.3, 0.8, R),
                       np.ones(R)], axis=1)
        eng = me.MetropolisEngine(me.BuiltinEnergy("mixed_well", *kr[0]), initial_real_params=np.array([0.3, 0.3]),
                                  initial_complex_params=np.array([0.2 - 0.1j]), temp=0.4, rung_consts=kr,
                                  replica_exchange=1, **common)
        return eng, mo.mixed_well(2, 1), None, np.full(R, 0.4), _pad(kr)
    if name == "wall":
        kr = np.stack([np.linspace(0.5, 1.5, R), np.linspace(0.3, 1.2, R)], axis=1)
        eng = me.MetropolisEngine(me.CudaEnergy(WALL_SRC, consts=list(kr[0]), has_reject=True),
                                  initial_real_params=np.array([0.0, 0.0]), temp=0.7, rung_consts=kr,
                                  replica_exchange=1, **common)
        return (eng, lambda x, k: k[0] * (x[:, 0] ** 2 + x[:, 1] ** 2), lambda x, k: x[:, 0] >= k[1],
                np.full(R, 0.7), _pad(kr))
    raise ValueError(name)


def _pad(k):
    k = np.atleast_2d(np.asarray(k, dtype=np.float64))
    return np.concatenate([k, np.zeros((k.shape[0], 16 - k.shape[1]))], axis=1)


def _targets(name, temps, consts):
    """Two target states between the rungs."""
    if name in ("xy_temp", "scalar"):
        return np.array([temps[0] * 1.05, temps[-1] * 0.97]), None
    kt = 0.5 * (consts[:2, :] + consts[1:3, :]) if len(consts) > 2 else consts[:1] * np.array([[1.1] + [1.0] * 15])
    K = {"xy_ham": 1, "mixed_ham": 4, "wall": 2}[name]
    return np.full(kt.shape[0], temps[0]), kt[:, :K]


def _samples(eng, row0, stride):
    ts = eng.time_series().cpu().numpy()[row0::stride]
    d = eng._d
    return ts[:, :d, :].transpose(0, 2, 1).reshape(-1, d)          # sample n = (row, chain), chain fastest


def _oracle(eng, efn, rej, temps, consts, f, tt, kt, row0, stride):
    from oracle import mbar_oracle as mo
    R = temps.size
    x = _samples(eng, row0, stride)
    allk = consts if kt is None and tt.size == 0 else np.concatenate(
        [consts, np.repeat(consts[:1], tt.size, axis=0) if kt is None else _pad(kt)])
    allt = np.concatenate([temps, tt])
    E, walled = mo.energies(efn, x, allk, rej)
    u = mo.reduced(E, walled, allt)
    n_per = x.shape[0] // R
    return mo.pass_sums(u, f, n_per, R, mo.observables(x, E)), walled, u, n_per


def _close(a, b, rel):
    a, b = np.asarray(a), np.asarray(b)
    scale = max(np.max(np.abs(b)), 1e-300)
    assert np.all(np.abs(a - b) <= rel * scale), (np.max(np.abs(a - b)) / scale, a, b)


CASES = [("xy_temp", 2, False), ("xy_temp", 8, False), ("xy_temp", 32, False), ("xy_temp", 8, True),
         ("xy_ham", 8, False), ("xy_ham", 8, True), ("mixed_ham", 4, False), ("wall", 4, False), ("wall", 4, True),
         ("scalar", 1, False), ("scalar", 1, True)]


@pytest.mark.parametrize("name,R,strict", CASES)
@pytest.mark.parametrize("targets", [False, True])
def test_pass_sums_match_the_oracle(name, R, strict, targets):
    me = _me()
    eng, efn, rej, temps, consts = _case(me, name, R, strict)
    eng.run(30, 4)
    rng = np.random.default_rng(R)
    f = np.concatenate([[0.0], rng.normal(0.0, 0.5, R - 1)])
    tt, kt = _targets(name, temps, consts) if targets else (np.zeros(0), None)
    row0, stride = 5, 2
    if R + tt.size > 32:                                               # S = 34: refused before any device work
        with pytest.raises(ValueError, match="32 states"):
            eng._mbar_sums(f, tt, kt, True, row0, stride)
        return
    got = eng._mbar_sums(f, tt, kt, True, row0, stride)
    want, walled, _, _ = _oracle(eng, efn, rej, temps, consts, f, tt, kt, row0, stride)
    assert got["n_nan"] == 0 and got["n_overflow"] == 0
    assert abs(got["sum_l"] - want["sum_l"]) <= 1e-12 * abs(want["sum_l"]) + 1e-12
    _close(got["s"], want["s"], 1e-12)
    _close(got["G"], want["G"], 1e-12)
    for c in range(want["obs"].shape[1]):
        _close(got["obs"][:, c], want["obs"][:, c], 1e-12)
    if name == "wall":
        assert walled[:R].any(), "the case must wall some samples in some rungs"
        W = want["W"]
        assert np.all(W[walled.T] == 0.0)                              # walled cross-states carry no weight


def test_solved_free_energies_match_the_oracle_solve():
    from oracle import mbar_oracle as mo
    me = _me()
    eng, efn, rej, temps, consts = _case(me, "xy_temp", 8, n_per_rung=256)
    eng.run(50, 5)
    res = eng.mbar(burn_in=0.2, stride=1)
    assert res.converged and res.free_energies[0] == 0.0
    row0 = int(eng._ts_rows * 0.2)
    _, _, u, n_per = _oracle(eng, efn, rej, temps, consts, np.zeros(8), np.zeros(0), None, row0, 1)
    f, _, conv = mo.solve(u, n_per)
    assert conv
    assert np.allclose(res.free_energies, f, rtol=0, atol=1e-9), (res.free_energies, f)


def _stride(eng):
    g = eng.statistical_inefficiency(column=eng._d, n_chains=2048, burn_in=0.5)
    return int(math.ceil(float(g.max().item())))


def test_temperature_ladder_is_analytic():
    """xy well k = 1: Z(T) = pi T, so f_k - f_0 = -ln(T_k / T_0); at targets between the rungs <E> = T and
    <x_0^2> = T / 2."""
    me = _me()
    temps = np.geomspace(0.5, 2.0, 8)
    eng = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.array([0.0, 0.0]), temp=list(temps),
                              replica_exchange=1, n_chains=8 * 4096, seed=3, sampling_width=0.5, device="cuda:0")
    eng.run(1000, 10)
    res = eng.mbar(burn_in=0.5, stride=_stride(eng))
    assert res.converged
    exact = -np.log(temps / temps[0])
    err = res.free_energy_errors[0]
    assert np.all(np.abs(res.free_energies - exact) <= 4 * err + 1e-3 * np.abs(exact)), (res.free_energies, exact, err)
    tt = np.geomspace(0.55, 1.9, 20)
    ev = res.evaluate(temp=tt)
    assert np.all(np.abs(ev["f"] + np.log(tt / temps[0])) <= 4 * ev["df"] + 1e-3 * np.abs(np.log(tt / temps[0])))
    n_eff = res._n
    se = tt / np.sqrt(n_eff)                                         # Var(E) = T^2 at every state
    assert np.all(np.abs(ev["E_mean"] - tt) <= 4 * 2 * se + 1e-3 * tt), (ev["E_mean"], tt)
    assert np.all(np.abs(ev["x2_mean"][:, 0] - tt / 2) <= 4 * 2 * se / 2 + 1e-3 * tt / 2)


def test_hamiltonian_ladder_is_analytic():
    """xy well at one T with rung constants k_r: Z_r = pi T / k_r, so f_r - f_0 = ln(k_r / k_0)."""
    me = _me()
    kr = np.geomspace(0.5, 2.0, 4)[:, None]
    eng = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.array([0.0, 0.0]), temp=0.5, rung_consts=kr,
                              replica_exchange=1, n_chains=4 * 8192, seed=5, sampling_width=0.5, device="cuda:0")
    eng.run(1000, 10)
    res = eng.mbar(burn_in=0.5, stride=_stride(eng))
    exact = np.log(kr[:, 0] / kr[0, 0])
    err = res.free_energy_errors[0]
    assert res.converged
    assert np.all(np.abs(res.free_energies - exact) <= 4 * err + 1e-3 * np.abs(exact)), (res.free_energies, exact, err)


def test_scalar_engine_reweights_to_another_temperature():
    me = _me()
    eng = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.array([0.0, 0.0]), temp=0.8, n_chains=16384,
                              seed=9, sampling_width=0.5, device="cuda:0")
    eng.run(1000, 10)
    res = eng.mbar(burn_in=0.5, stride=_stride(eng))
    assert res.converged and res.free_energies.shape == (1,)
    ev = res.evaluate(temp=0.88)
    exact = -np.log(1.1)
    assert abs(ev["f"][0] - exact) <= 4 * ev["df"][0] + 1e-3 * abs(exact), (ev["f"], exact, ev["df"])
    rung = res.evaluate()
    assert abs(rung["E_mean"][0] - 0.8) < 0.02


def test_invariances():
    me = _me()
    temps = list(np.geomspace(0.3, 1.5, 4))
    kw = dict(initial_real_params=np.array([0.1, 0.0]), temp=temps, replica_exchange=1, seed=21, device="cuda:0")
    a = me.MetropolisEngine(("xy_well", 1.0), n_chains=1024, **kw)
    a.run(40, 5)
    r1, r2 = a.mbar(burn_in=0.1), a.mbar(burn_in=0.1)
    assert np.array_equal(r1.free_energies, r2.free_energies)                     # bit-identical from run to run
    b = me.MetropolisEngine(("xy_well", 1.0), n_chains=1024, ts_chunk_bytes=7 * 3 * 1024 * 8, **kw)   # several chunks
    b.run(40, 5)
    assert len([c for c in b._ts_chunks if c[1]]) > 3
    rb = b.mbar(burn_in=0.1)
    assert np.allclose(rb.free_energies, r1.free_energies, rtol=0, atol=1e-12)
    f = r1.free_energies
    full = a._mbar_sums(f, np.array([0.7]), None, True, 4, 3)
    halves = []
    for lo, hi in ((0, 512), (512, 1024)):
        e = me.MetropolisEngine(("xy_well", 1.0), n_chains=1024, _shard=(lo, hi), **kw)
        e.run(40, 5)
        halves.append(e._mbar_sums(f, np.array([0.7]), None, True, 4, 3))
    for key in ("s", "G", "obs"):
        _close(halves[0][key] + halves[1][key], full[key], 1e-13)
    assert abs(halves[0]["sum_l"] + halves[1]["sum_l"] - full["sum_l"]) <= 1e-13 * abs(full["sum_l"])


def test_refusals():
    me = _me()
    x0 = np.array([0.1, 0.0])
    e = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=0.5, n_chains=64, record=False,
                            device="cuda:0")
    e.run(5, 2)
    with pytest.raises(RuntimeError):
        e.mbar()
    e = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=0.5, n_chains=64, device="cuda:0")
    with pytest.raises(RuntimeError):
        e.mbar()                                                    # no rows recorded
    e.run(10, 2)
    with pytest.raises(ValueError):
        e.mbar(stride=0)
    res = e.mbar()
    with pytest.raises(ValueError):
        res.evaluate(temp=0.0)
    with pytest.raises(ValueError):
        res.evaluate(temp=float("nan"))
    with pytest.raises(ValueError):
        res.evaluate(temp=[1.0] * 32)                               # S = 33
    with pytest.raises(ValueError):
        res.evaluate(temp=1.0, consts=[[1.0, 2.0]])                 # K = 2, functor has 1
    with pytest.raises(ValueError):
        res.evaluate(temp=1.0, consts=[[float("inf")]])
    n = me.MetropolisEngine(me.CudaEnergy(NAN_SRC, consts=[1.0]), initial_real_params=x0, temp=0.5, n_chains=64,
                            device="cuda:0")
    n.run(10, 2)
    with pytest.raises(RuntimeError, match="ME_STATUS_ENERGY_NAN"):
        n.mbar().evaluate(temp=0.5, consts=[[-1.0]])
    sweep = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=[0.0, 0.5], n_chains=64,
                                device="cuda:0")
    sweep.run(10, 2)
    with pytest.raises(ValueError, match="rung temperature"):
        sweep.mbar()
    big = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=list(np.linspace(0.5, 1.0, 64)),
                              n_chains=128, device="cuda:0")
    big.run(4, 2)
    with pytest.raises(ValueError, match="32 rungs"):
        big.mbar()
    ham = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=0.5, rung_consts=[[1.0], [2.0]],
                              n_chains=64, device="cuda:0")
    ham.run(10, 2)
    with pytest.raises(ValueError, match="target_consts"):
        ham.mbar().evaluate(temp=0.5)
    wide = me.MetropolisEngine(("x2",), initial_real_params=np.zeros(33), temp=0.5, n_chains=32, device="cuda:0")
    with pytest.raises(NotImplementedError):
        wide.mbar()
    import torch
    cal = me.MetropolisEngine(lambda r, c: (r * r).sum(dim=1), initial_real_params=x0, temp=0.5, n_chains=64,
                              device="cuda:0")
    with pytest.raises(NotImplementedError):
        cal.mbar()
    sc = me.SharedCovarianceEngine(energy_consts=(10.0, -1.0, 0.05, 1.0), temp=.1, n_chains=128, seed=3, record=False,
                                   initial_real_params=np.array([0.1]), initial_complex_params=0.05 * np.ones(16),
                                   sampling_width=0.02, device="cuda:0")
    with pytest.raises(NotImplementedError):
        sc.mbar()
    del torch
