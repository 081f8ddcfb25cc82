"""Temperature ladders and replica exchange in the fused step kernel (me_device.cuh, run_body's PT instantiation) on the
GPU: chain by chain against the C oracle's ladders (oracle/me_oracle_ladder.c, meo_run_ladder), the per-chain temperature
against the scalar kernel, what the swaps are for (crossing a barrier at low T), the invariances of the swap schedule,
and the combinations a ladder engine refuses."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

USER_SRC = """
__device__ double me_user_energy(const double* x, const double* cr, const double* ci, const double* k) {
    return k[0] * x[0] * x[0] + x[1] * x[1] * x[1] * x[1];
}
"""
WELL_SRC = """
__device__ double me_user_energy(const double* x, const double* cr, const double* ci, const double* k) {
    const double a = x[0] * x[0] - 1.0;
    return k[0] * a * a;
}
"""

SHAPES = {   # name -> (engine energy, n_real, n_complex, oracle energy, oracle consts)
    "x2": (("x2",), 1, 0, "x2", []),
    "xy_well": (("xy_well", 1.0), 2, 0, "xy_well", [1.0]),
    "2r1c": (("mixed_well", 1.0, -1.0, 0.5), 2, 1, "mixed_well", [1.0, -1.0, 0.5]),
    "user": (None, 2, 0, lambda x: 0.7 * x[0] * x[0] + x[1] ** 4, []),
}


def _energy(me, name):
    spec = SHAPES[name][0]
    return me.CudaEnergy(USER_SRC, consts=[0.7]) if spec is None else me.BuiltinEnergy(*spec)


def _engine(me, name, temps, n, every=1, **kw):
    _, nr, nc, _, _ = SHAPES[name]
    x0r = np.full(nr, 0.3)
    x0c = np.full(nc, 0.2 - 0.1j) if nc else None
    return me.MetropolisEngine(_energy(me, name), initial_real_params=x0r, initial_complex_params=x0c, temp=list(temps),
                               replica_exchange=every, n_chains=n, **kw)


@pytest.mark.parametrize("strict", [False, True])
@pytest.mark.parametrize("R", [2, 8, 32])
@pytest.mark.parametrize("name", ["x2", "xy_well", "2r1c", "user"])
def test_ladder_matches_oracle_chain_by_chain(name, R, strict):
    import metropolisengine_b200 as me
    from oracle import ladder_oracle as co
    n, M, K, seed = 2048, 20, 5, 31
    temps = np.geomspace(0.05, 2.0, R)
    eng = _engine(me, name, temps, n, seed=seed, strict=strict)
    eng.run(M, K)
    eng.check_status()
    st = eng.state.cpu().numpy()
    walker = eng.walker_per_chain.cpu().numpy()
    sacc = eng._swap_acc.cpu().numpy().astype(np.uint32)
    _, nr, nc, oen, oconsts = SHAPES[name]
    x0 = np.concatenate([np.full(nr, 0.3), np.full(nc, 0.2), np.full(nc, -0.1)])
    lay = eng._lay
    tol = 2e-10 if strict else 2e-9
    for lad in range(n // R):
        o = co.CLadder(nr, nc, oen, temps, swap_every=1, x0=x0, chain0=lad * R, consts=oconsts)
        o.run(M, K, seed=seed)
        cols = slice(lad * R, (lad + 1) * R)
        assert np.array_equal(st[lay.NACC, cols], o.states[:, o.off.NACC]), lad
        assert np.array_equal(walker[cols], o.walker), lad
        assert np.array_equal(sacc[cols], o.swap_acc), lad
        got = st[lay.X:lay.X + lay.D, cols].T
        assert np.allclose(got, o.x, rtol=tol, atol=tol), (lad, got, o.x)
        assert np.allclose(st[lay.SIG, cols], o.states[:, o.off.SIG], rtol=tol, atol=0), lad


@pytest.mark.parametrize("name", ["xy_well", "x2", "user"])
def test_sweep_step_equals_scalar_step(name):
    """temp=[T]*R without swaps runs every chain at T: bit-identical to the scalar engine."""
    import metropolisengine_b200 as me
    n, T = 1024, 0.37
    a = _engine(me, name, [T] * 4, n, every=0, seed=9)
    _, nr, nc, _, _ = SHAPES[name]
    b = me.MetropolisEngine(_energy(me, name), initial_real_params=np.full(nr, 0.3), temp=T, n_chains=n, seed=9)
    for e in (a, b):
        e.run(30, 7)
        e.step(5)
        e.measure()
    assert np.array_equal(a.state.cpu().numpy(), b.state.cpu().numpy())
    assert np.array_equal(a.time_series().cpu().numpy(), b.time_series().cpu().numpy())


def _double_well_fraction(swaps):
    # the default initial width (0.05) keeps the cold rungs from jumping the barrier in one proposal before their
    # widths adapt to the well (about 0.1 at T = 0.25); only swaps bring the other well to them
    import metropolisengine_b200 as me
    from scipy.integrate import quad
    h, R, n = 5.0, 8, 8 * 2048
    temps = np.geomspace(0.25, 8.0, R)
    eng = me.MetropolisEngine(me.CudaEnergy(WELL_SRC, consts=[h]), initial_real_params=np.array([1.0]), temp=list(temps),
                              replica_exchange=1 if swaps else 0, n_chains=n, seed=4)
    eng.run(2000, 10)
    ts = eng.time_series().cpu().numpy()[500:, 0, :]          # [rows, chains], burn-in dropped
    x0 = ts[:, ::R]                                            # rung 0 of every ladder
    neg = (x0 < 0).mean(axis=0)                                # per ladder
    x2 = (x0 ** 2).mean(axis=0)
    z = quad(lambda x: np.exp(-h * (x * x - 1) ** 2 / temps[0]), -4, 4)[0]
    want_x2 = quad(lambda x: x * x * np.exp(-h * (x * x - 1) ** 2 / temps[0]), -4, 4)[0] / z
    return eng, neg, x2, want_x2


def test_swaps_cross_the_barrier():
    eng, neg, x2, want_x2 = _double_well_fraction(True)
    se = neg.std() / np.sqrt(neg.size)
    assert abs(neg.mean() - 0.5) < 5 * se, (neg.mean(), se)
    se2 = x2.std() / np.sqrt(x2.size)
    assert abs(x2.mean() - want_x2) < 5 * se2, (x2.mean(), want_x2, se2)
    rate = eng.swap_acceptance_rate
    assert rate.shape == (7,) and np.all(rate > 0.05) and np.all(rate <= 1), rate
    assert eng.real_mean.shape == (8, 1)


def test_without_swaps_the_cold_rung_stays_in_its_well():
    """Without swaps rung 0 is the scalar engine at T = 0.25 (bit for bit, test_sweep_step_equals_scalar_step): its
    adapted random walk still jumps the barrier in one proposal now and then (about 1e-7 per step here: 5 of the 2,048
    cold chains over 20,000 steps, 0.0016 of the samples on the left), so the bound is 1 % — two orders of
    magnitude below the 0.5 that the swaps reach on the same schedule."""
    _, neg, _, _ = _double_well_fraction(False)
    assert neg.mean() < 1e-2, neg.mean()


def _ladder_state(eng):
    return (eng.state.cpu().numpy(), eng.walker_per_chain.cpu().numpy(), eng._swap_acc.cpu().numpy())


def _same(a, b):
    for u, v in zip(a, b):
        assert np.array_equal(u, v)


def test_run_equals_step_measure_loop_and_segments():
    import metropolisengine_b200 as me
    temps, n = np.geomspace(0.1, 3.0, 8), 8 * 1024
    a = _engine(me, "xy_well", temps, n, every=2, seed=3)
    a.run(40, 6)
    b = _engine(me, "xy_well", temps, n, every=2, seed=3)
    for _ in range(40):
        b.step(6)
        b.measure()
    _same(_ladder_state(a), _ladder_state(b))
    assert np.array_equal(a.time_series().cpu().numpy(), b.time_series().cpu().numpy())
    old = os.environ.get("ME_SEGMENTS")
    os.environ["ME_SEGMENTS"] = "5"
    try:
        c = _engine(me, "xy_well", temps, n, every=2, seed=3)
        c.run(40, 6)
    finally:
        if old is None:
            del os.environ["ME_SEGMENTS"]
        else:
            os.environ["ME_SEGMENTS"] = old
    _same(_ladder_state(a), _ladder_state(c))
    pa, pc = a.pooled_statistics(), c.pooled_statistics()
    assert pa["mean_real"].shape == (8, 2)
    assert np.allclose(pa["mean_real"], pc["mean_real"], rtol=1e-12, atol=1e-14)


def test_graph_replay_checkpoint_and_shards():
    import metropolisengine_b200 as me
    temps, n = np.geomspace(0.1, 3.0, 4), 4 * 2048
    ref = _engine(me, "x2", temps, n, every=1, seed=8, record=False)
    for _ in range(4):
        ref.run(10, 5)
    g = _engine(me, "x2", temps, n, every=1, seed=8, record=False)
    for _ in range(4):
        g.run_graphed(10, 5)
    _same(_ladder_state(ref), _ladder_state(g))
    c = _engine(me, "x2", temps, n, every=1, seed=8, record=False)
    c.run(20, 5)
    sd = c.state_dict()
    d = _engine(me, "x2", temps, n, every=1, seed=8, record=False)
    d.load_state_dict(sd)
    d.run(20, 5)
    _same(_ladder_state(ref), _ladder_state(d))
    halves = [_engine(me, "x2", temps, n, every=1, seed=8, record=False, _shard=(lo, hi))
              for lo, hi in ((0, n // 2), (n // 2, n))]
    for h in halves:
        for _ in range(4):
            h.run(10, 5)
    full = _ladder_state(ref)
    for k, h in enumerate(halves):
        part = _ladder_state(h)
        cols = slice(k * n // 2, (k + 1) * n // 2)
        assert np.array_equal(part[0], full[0][:, cols])
        assert np.array_equal(part[1], full[1][cols]) and np.array_equal(part[2], full[2][cols])


def test_rejections():
    import torch
    import metropolisengine_b200 as me
    x0 = np.zeros(1)
    ok = dict(initial_real_params=x0, n_chains=64)
    with pytest.raises(NotImplementedError):
        me.MetropolisEngine("x2", temp=[0.5, 1.0], adapt="pooled", **ok)
    with pytest.raises(NotImplementedError):
        me.MetropolisEngine(lambda r, c: (r ** 2).sum(-1), temp=[0.5, 1.0], **ok)
    with pytest.raises(NotImplementedError):
        me.MetropolisEngine("x2", reject_condition=lambda r, c: torch.zeros(64, dtype=torch.bool), temp=[0.5, 1.0], **ok)
    with pytest.raises(NotImplementedError):
        me.MetropolisEngine(("cylinder", 1, 1, 1, 1), initial_real_params=x0, initial_complex_params=np.zeros(16),
                            temp=[0.5, 1.0], n_chains=64)
    eng = me.MetropolisEngine("x2", temp=[0.5, 1.0], replica_exchange=1, **ok)
    with pytest.raises(NotImplementedError):
        eng.run_injected(np.zeros((1, 1)), np.zeros(1), 1, 1)
    mixed = me.MetropolisEngine(("mixed_well", 1.0, -1.0, 0.5), initial_real_params=np.zeros(2),
                                initial_complex_params=np.zeros(1), temp=[0.5, 1.0], n_chains=64)
    with pytest.raises(NotImplementedError):
        mixed.step_real_group()
    with pytest.raises(NotImplementedError):
        me.MetropolisEngine(("mixed_well", 1.0, -1.0, 0.5), initial_real_params=np.zeros(2),
                            initial_complex_params=np.zeros(1), temp=[0.5, 1.0], n_chains=64,
                            complex_sample_method="magnitude-phase")
    bad = [dict(temp=[0.5, 1.0], n_chains=63),                                # not whole ladders
           dict(temp=[1.0, 0.5], replica_exchange=1, n_chains=64),            # not increasing
           dict(temp=[0.0, 0.5], replica_exchange=1, n_chains=64),            # T = 0 with swaps
           dict(temp=[0.5, np.inf], n_chains=64),                             # not finite
           dict(temp=[0.5, 1.0, 2.0], replica_exchange=1, n_chains=63),       # 3 rungs with swaps
           dict(temp=[-0.5, 1.0], n_chains=64),                               # negative
           dict(temp=[0.5, 1.0], replica_exchange=-1, n_chains=64),
           dict(temp=0.5, replica_exchange=1, n_chains=64),                   # swaps need a ladder
           dict(temp=[0.5, 1.0], n_chains=64, _shard=(1, 33))]                # shard not ladder-aligned
    for kw in bad:
        with pytest.raises((ValueError, AssertionError)):
            me.MetropolisEngine("x2", initial_real_params=x0, **kw)
    sweep = me.MetropolisEngine("x2", temp=[0.5, 1.0, 2.0], initial_real_params=x0, n_chains=63)   # sweep: any R
    sweep.run(3, 2)
    assert sweep.real_mean.shape == (3, 1)
    with pytest.raises(NotImplementedError):
        sweep.pooled_statistics()
