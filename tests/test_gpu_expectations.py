"""Uncertainties of reweighted expectations on the GPU (csrc/me_mbar.cuh, k_mbar_cov / me_mbar_cov_pass;
metropolisengine_b200/mbar.py, ``evaluate(uncertainty=True)``): the covariance sums against the numpy oracle
(oracle/expectation_oracle.py) on the engine's own recorded rows, the full result against pymbar's explicit route,
analytic ladders sampled by real chains, the split into several passes, the invariances and the refusals."""
import numpy as np
import pytest

from tests.test_gpu_mbar import NAN_SRC, _case, _close, _me, _oracle, _pad, _samples, _stride, _targets

pytestmark = pytest.mark.gpu


def _ranges(R, n_t):
    """(first, count) of the covered ranges: all rungs, all targets, one state."""
    out = [(0, R), (R + n_t - 1, 1)]
    if n_t:
        out.append((R, n_t))
    return out


CASES = [("scalar", 1, False), ("scalar", 1, True), ("xy_temp", 2, False), ("xy_temp", 8, False),
         ("xy_temp", 8, True), ("xy_temp", 32, False), ("xy_ham", 8, False), ("xy_ham", 8, True),
         ("mixed_ham", 4, False), ("wall", 4, False), ("wall", 4, True)]


@pytest.mark.parametrize("name,R,strict", CASES)
def test_cov_sums_match_the_oracle(name, R, strict):
    from oracle import expectation_oracle as xo
    from oracle import mbar_oracle as mo
    me = _me()
    eng, efn, rej, temps, consts = _case(me, name, R, strict)
    eng.run(30, 4)
    rng = np.random.default_rng(R)
    f = np.concatenate([[0.0], rng.normal(0.0, 0.5, R - 1)])
    tt, kt = _targets(name, temps, consts) if R + 2 <= 32 else (np.zeros(0), None)
    row0, stride = 5, 2
    want, _, u, n_per = _oracle(eng, efn, rej, temps, consts, f, tt, kt, row0, stride)
    x = _samples(eng, row0, stride)
    allk = np.concatenate([consts, np.repeat(consts[:1], tt.size, axis=0) if kt is None else _pad(kt)]) \
        if tt.size else consts
    E, _ = mo.energies(efn, x, allk, rej)
    obs = mo.observables(x, E)
    mean = want["obs"] / want["s"][:, None]
    for first, count in _ranges(R, tt.size):
        cen = mean[first:first + count] + 0.1 * rng.normal(size=(count, mean.shape[1]))
        got = eng._mbar_cov_sums(f, tt, kt, first, count, cen, row0, stride)
        o, C, Q = xo.cov_sums(u, f, n_per, R, obs, first, count, cen)
        for c in range(count):
            _close(got["o"][c], o[c], 1e-12)
            _close(got["C"][c], C[c], 1e-12)
            _close(got["Q"][c], Q[c], 1e-12)


def _pymbar_check(eng, efn, rej, temps, consts, res, tt, kt):
    from oracle import expectation_oracle as xo
    from oracle import mbar_oracle as mo
    R, d = temps.size, eng._d
    row0, stride = res._sample
    _, _, u, n_per = _oracle(eng, efn, rej, temps, consts, res.free_energies, tt, kt, row0, stride)
    x = _samples(eng, row0, stride)
    allk = np.concatenate([consts, np.repeat(consts[:1], tt.size, axis=0) if kt is None else _pad(kt)]) \
        if tt.size else consts
    E, _ = mo.energies(efn, x, allk, rej)
    obs = mo.observables(x, E)
    states = range(R, R + tt.size) if tt.size else range(R)
    mean, cov = xo.pymbar_expectations(u, res.free_energies, n_per, R, obs, states)
    plain = res.evaluate(temp=tt if tt.size else None, consts=kt)
    ev = res.evaluate(temp=tt if tt.size else None, consts=kt, uncertainty=True)
    for k, v in plain.items():
        assert np.array_equal(ev[k], v), k                                    # the same bits as the default call
    for i in range(len(states)):
        _close(ev["obs_cov"][i], cov[i], 1e-9)
    se = np.sqrt(np.diagonal(cov, axis1=1, axis2=2))
    for key, want in (("dx_mean", se[:, :d]), ("dx2_mean", se[:, d:2 * d]), ("dE_mean", se[:, 2 * d]),
                      ("dE2_mean", se[:, 2 * d + 1])):
        _close(ev[key], want, 1e-9)
    ts = tt if tt.size else np.broadcast_to(temps, (R,))
    for i in range(len(states)):
        c, dc = xo.heat_capacity(mean[i, 2 * d], mean[i, 2 * d + 1], cov[i, 2 * d:, 2 * d:], ts[i])
        assert abs(ev["heat_capacity"][i] - c) <= 1e-9 * abs(c) + 1e-12
        assert abs(ev["dheat_capacity"][i] - dc) <= 1e-9 * dc
    return ev


@pytest.mark.parametrize("name,R", [("xy_temp", 8), ("mixed_ham", 4), ("wall", 4), ("scalar", 1)])
def test_evaluate_matches_pymbars_route(name, R):
    me = _me()
    eng, efn, rej, temps, consts = _case(me, name, R, n_per_rung=256)
    eng.run(40, 4)
    res = eng.mbar(burn_in=0.2)
    tt, kt = _targets(name, temps, consts)
    _pymbar_check(eng, efn, rej, temps, consts, res, tt, kt)
    _pymbar_check(eng, efn, rej, temps, consts, res, np.zeros(0), None)     # the rungs


# The adaptive chains carry a systematic bias of their own, about 2e-3 of <E> on these ladders (the MBAR analytic tests
# allow 1e-3 beside twice the naive error); the checks below allow it beside 4 returned standard errors.
BIAS = 3e-3


def _within(got, exact, err, rel):
    assert np.all(np.abs(got - exact) <= 4 * err + rel * np.abs(exact)), ((got - exact) / err, (got - exact) / exact)


def test_temperature_ladder_is_analytic():
    """xy well k = 1 (two degrees of freedom): <E> = T, <x_0^2> = T / 2 and C = 1 at every temperature."""
    me = _me()
    temps = np.geomspace(0.5, 2.0, 8)
    eng = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.array([0.0, 0.0]), temp=list(temps),
                              replica_exchange=1, n_chains=8 * 4096, seed=3, sampling_width=0.5, device="cuda:0")
    eng.run(1000, 10)
    res = eng.mbar(burn_in=0.5, stride=_stride(eng))
    tt = np.geomspace(0.55, 1.9, 20)
    ev = res.evaluate(temp=tt, uncertainty=True)
    _within(ev["E_mean"], tt, ev["dE_mean"], BIAS)
    _within(ev["x2_mean"][:, 0], tt / 2, ev["dx2_mean"][:, 0], BIAS)
    _within(ev["heat_capacity"], np.ones(20), ev["dheat_capacity"], 2 * BIAS)
    assert np.all(ev["dheat_capacity"] < 0.05)


def test_hamiltonian_ladder_is_analytic():
    """xy well at one T with constants k: <E> = T and C = 1 whatever k, at the rungs and at targets between them."""
    me = _me()
    kr = np.geomspace(0.5, 2.0, 4)[:, None]
    T = 0.5
    eng = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.array([0.0, 0.0]), temp=T, rung_consts=kr,
                              replica_exchange=1, n_chains=4 * 8192, seed=5, sampling_width=0.5, device="cuda:0")
    eng.run(1000, 10)
    res = eng.mbar(burn_in=0.5, stride=_stride(eng))
    kt = np.geomspace(0.6, 1.8, 6)[:, None]
    for ev in (res.evaluate(uncertainty=True), res.evaluate(temp=T, consts=kt, uncertainty=True)):
        n = ev["E_mean"].size
        _within(ev["E_mean"], np.full(n, T), ev["dE_mean"], BIAS)
        _within(ev["heat_capacity"], np.ones(n), ev["dheat_capacity"], 2 * BIAS)


def _wide(me, **kw):
    """Mixed well 3r + 4c (D = 11) on a 4-rung Hamiltonian ladder."""
    kr = np.stack([np.linspace(0.5, 1.5, 4), np.linspace(-1.0, -0.2, 4), np.linspace(0.3, 0.8, 4), np.ones(4)], axis=1)
    eng = me.MetropolisEngine(me.BuiltinEnergy("mixed_well", *kr[0]), initial_real_params=np.array([0.3, 0.3, 0.1]),
                              initial_complex_params=0.2 * np.exp(1j * np.arange(4)), temp=0.4, rung_consts=kr,
                              replica_exchange=1, seed=13, device="cuda:0", **kw)
    return eng, kr


def test_several_passes_equal_single_state_passes():
    me = _me()
    eng, kr = _wide(me, n_chains=4 * 256)
    eng.run(30, 4)
    res = eng.mbar(burn_in=0.2)
    a = np.linspace(0.0, 1.0, 28)[:, None]
    kt = (1 - a) * kr[0] + a * kr[-1]
    tt = np.full(28, 0.4)
    m = 2 * eng._d + 2
    cen = np.random.default_rng(1).normal(size=(28, m))
    full = eng._mbar_cov_sums(res.free_energies, tt, kt, 4, 28, cen, *res._sample)
    assert len(full["passes"]) > 1, full["passes"]
    for i in range(28):
        one = eng._mbar_cov_sums(res.free_energies, tt, kt, 4 + i, 1, cen[i:i + 1], *res._sample)
        assert one["passes"] == [(4 + i, 1)]
        for key in ("o", "C", "Q"):
            _close(full[key][i], one[key][0], 1e-13)
    ev = res.evaluate(temp=tt, consts=kt, uncertainty=True)
    assert ev["obs_cov"].shape == (28, m, m) and np.all(np.isfinite(ev["obs_cov"]))


def test_widest_shape_covers_one_state_per_pass_at_least():
    """D = 32 with S = 32: a single covered state fits the shared-memory bound, and a wide range is split."""
    me = _me()
    eng = me.MetropolisEngine(("x2",), initial_real_params=np.zeros(32), temp=0.5, n_chains=256, seed=2,
                              device="cuda:0")
    eng.run(20, 4)
    res = eng.mbar(burn_in=0.2)
    tt = np.linspace(0.45, 0.55, 31)
    cen = np.zeros((31, 66))
    out = eng._mbar_cov_sums(res.free_energies, tt, None, 1, 31, cen, *res._sample)
    assert 1 < len(out["passes"]) < 31
    one = eng._mbar_cov_sums(res.free_energies, tt, None, 31, 1, cen[-1:], *res._sample)
    _close(out["Q"][-1], one["Q"][0], 1e-13)


def test_invariances():
    me = _me()
    temps = list(np.geomspace(0.3, 1.5, 4))
    kw = dict(initial_real_params=np.array([0.1, 0.0]), temp=temps, replica_exchange=1, seed=21, device="cuda:0")
    a = me.MetropolisEngine(("xy_well", 1.0), n_chains=1024, **kw)
    a.run(40, 5)
    res = a.mbar(burn_in=0.1)
    e1 = res.evaluate(temp=[0.5, 0.9], uncertainty=True)
    e2 = res.evaluate(temp=[0.5, 0.9], uncertainty=True)
    for k in e1:
        assert np.array_equal(e1[k], e2[k]), k                              # bit-identical from run to run
    f, tt = res.free_energies, np.array([0.7, 1.1])
    cen = np.random.default_rng(4).normal(size=(6, 6))
    full = a._mbar_cov_sums(f, tt, None, 0, 6, cen, 4, 3)
    b = me.MetropolisEngine(("xy_well", 1.0), n_chains=1024, ts_chunk_bytes=7 * 3 * 1024 * 8, **kw)   # several chunks
    b.run(40, 5)
    assert len([c for c in b._ts_chunks if c[1]]) > 3
    chunked = b._mbar_cov_sums(f, tt, None, 0, 6, cen, 4, 3)
    halves = []
    for lo, hi in ((0, 512), (512, 1024)):
        e = me.MetropolisEngine(("xy_well", 1.0), n_chains=1024, _shard=(lo, hi), **kw)
        e.run(40, 5)
        halves.append(e._mbar_cov_sums(f, tt, None, 0, 6, cen, 4, 3))
    for key in ("o", "C", "Q"):
        _close(chunked[key], full[key], 1e-13)
        _close(halves[0][key] + halves[1][key], full[key], 1e-13)


def test_refusals():
    me = _me()
    x0 = np.array([0.1, 0.0])
    e = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=0.5, n_chains=64, device="cuda:0")
    e.run(10, 2)
    res = e.mbar()
    with pytest.raises(ValueError, match="32 states"):
        res.evaluate(temp=[1.0] * 32, uncertainty=True)                     # S = 33
    with pytest.raises(ValueError, match="32 states"):
        e._mbar_cov_sums(res.free_energies, np.ones(32), None, 0, 1, np.zeros((1, 6)), *res._sample)
    n = me.MetropolisEngine(me.CudaEnergy(NAN_SRC, consts=[1.0]), initial_real_params=x0, temp=0.5, n_chains=64,
                            device="cuda:0")
    n.run(10, 2)
    rn = n.mbar()
    with pytest.raises(RuntimeError, match="ME_STATUS_ENERGY_NAN"):
        n._mbar_cov_sums(rn.free_energies, np.array([0.5]), np.array([[-1.0]]), 1, 1, np.zeros((1, 6)), *rn._sample)
    with pytest.raises(RuntimeError, match="ME_STATUS_ENERGY_NAN"):
        rn.evaluate(temp=0.5, consts=[[-1.0]], uncertainty=True)
    wide = me.MetropolisEngine(("x2",), initial_real_params=np.zeros(33), temp=0.5, n_chains=32, device="cuda:0")
    with pytest.raises(NotImplementedError):
        wide.mbar()
    cal = me.MetropolisEngine(lambda r, c: (r * r).sum(dim=1), initial_real_params=x0, temp=0.5, n_chains=64,
                              device="cuda:0")
    with pytest.raises(NotImplementedError):
        cal.mbar()
    sc = me.SharedCovarianceEngine(energy_consts=(10.0, -1.0, 0.05, 1.0), temp=.1, n_chains=128, seed=3, record=False,
                                   initial_real_params=np.array([0.1]), initial_complex_params=0.05 * np.ones(16),
                                   sampling_width=0.02, device="cuda:0")
    with pytest.raises(NotImplementedError):
        sc.mbar()
