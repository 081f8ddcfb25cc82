"""Hamiltonian ladders in the fused step kernel (me_device.cuh, run_body's HX instantiation) on the GPU: chain by chain
against the C oracle (oracle/me_oracle_hladder.c, meo_run_hladder), the per-rung constants against the scalar kernel, the
energy a chain holds after a swap, walls per rung, the link to temperature ladders, what the swaps are for (a barrier
ladder at one temperature), the exact Gaussian ladder, the invariances of the swap schedule, and the refusals."""
import ctypes
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

WALL_SRC = """
__device__ double me_user_energy(const double* x, const double* cr, const double* ci, const double* k) {
    return k[0] * x[0] * x[0] + x[1] * x[1] * x[1] * x[1];
}
__device__ bool me_user_reject(const double* x, const double* cr, const double* ci, const double* k) {
    return fabs(x[0]) >= k[1];
}
"""
WELL_SRC = """
__device__ double me_user_energy(const double* x, const double* cr, const double* ci, const double* k) {
    const double a = x[0] * x[0] - 1.0;
    return k[0] * a * a;
}
"""
GAUSS_SRC = """
__device__ double me_user_energy(const double* x, const double* cr, const double* ci, const double* k) {
    return k[0] * x[0] * x[0];
}
"""


def _rung_consts(name, R):
    if name == "xy_well":
        return np.geomspace(0.2, 5.0, R)[:, None]
    if name == "2r1c":
        return np.stack([np.linspace(0.5, 1.5, R), np.linspace(-1.0, -0.2, R), np.linspace(0.3, 0.8, R)], axis=1)
    return np.stack([np.linspace(0.5, 1.5, R), np.linspace(0.8, 2.0, R)], axis=1)          # "wall": k[1] is the wall


SHAPES = {"xy_well": (2, 0), "2r1c": (2, 1), "wall": (2, 0)}


def _energy(me, name, consts):
    if name == "xy_well":
        return me.BuiltinEnergy("xy_well", *consts)
    if name == "2r1c":
        return me.BuiltinEnergy("mixed_well", *consts)
    return me.CudaEnergy(WALL_SRC, consts=list(consts), has_reject=True)


def _x0(name):
    nr, nc = SHAPES[name]
    return np.full(nr, 0.3), (np.full(nc, 0.2 - 0.1j) if nc else None)


def _engine(me, name, kr, temp, n, every=1, **kw):
    xr, xc = _x0(name)
    return me.MetropolisEngine(_energy(me, name, kr[0]), initial_real_params=xr, initial_complex_params=xc,
                               temp=temp, rung_consts=kr, replica_exchange=every, n_chains=n, **kw)


def _oracle_ladder(co, name, kr, temps, chain0):
    nr, nc = SHAPES[name]
    x0 = np.concatenate([np.full(nr, 0.3), np.full(nc, 0.2), np.full(nc, -0.1)])
    if name == "wall":
        en = [lambda x, k=k: k[0] * x[0] * x[0] + x[1] * x[1] * x[1] * x[1] for k in kr]
        rej = [lambda x, k=k: abs(x[0]) >= k[1] for k in kr]
        return co.CHLadder(nr, nc, en, temps, kr, swap_every=1, x0=x0, chain0=chain0, reject=rej)
    return co.CHLadder(nr, nc, "xy_well" if name == "xy_well" else "mixed_well", temps, kr, swap_every=1, x0=x0,
                       chain0=chain0)


@pytest.mark.parametrize("strict", [False, True])
@pytest.mark.parametrize("ladder_t", [False, True])
@pytest.mark.parametrize("R", [2, 8, 32])
@pytest.mark.parametrize("name", ["xy_well", "2r1c", "wall"])
def test_hamiltonian_ladder_matches_oracle_chain_by_chain(name, R, ladder_t, strict):
    import metropolisengine_b200 as me
    from oracle import hladder_oracle as co
    n, M, K, seed = 1024, 20, 5, 31
    kr = _rung_consts(name, R)
    temps = np.geomspace(0.05, 2.0, R) if ladder_t else np.full(R, 0.5)
    eng = _engine(me, name, kr, list(temps) if ladder_t else 0.5, n, seed=seed, strict=strict)
    eng.run(M, K)
    eng.check_status()
    st = eng.state.cpu().numpy()
    walker = eng.walker_per_chain.cpu().numpy()
    sacc = eng._swap_acc.cpu().numpy().astype(np.uint32)
    lay = eng._lay
    tol = 2e-10 if strict else 2e-9
    swaps = 0
    for lad in range(n // R):
        o = _oracle_ladder(co, name, kr, temps, lad * R)
        o.run(M, K, seed=seed)
        cols = slice(lad * R, (lad + 1) * R)
        assert np.array_equal(st[lay.NACC, cols], o.states[:, o.off.NACC]), lad
        assert np.array_equal(walker[cols], o.walker), lad
        assert np.array_equal(sacc[cols], o.swap_acc), lad
        got = st[lay.X:lay.X + lay.D, cols].T
        assert np.allclose(got, o.x, rtol=tol, atol=tol), (lad, got, o.x)
        assert np.allclose(st[lay.SIG, cols], o.states[:, o.off.SIG], rtol=tol, atol=0), lad
        assert np.allclose(st[lay.E, cols], o.states[:, o.off.E], rtol=tol, atol=tol), lad
        swaps += int(o.swap_acc.sum())
    assert swaps > 0


@pytest.mark.parametrize("strict", [False, True])
@pytest.mark.parametrize("name", ["xy_well", "2r1c", "wall"])
def test_sweep_columns_equal_scalar_engines(name, strict):
    """Without swaps, rung r's columns are the scalar engine with (k_r, T_r) and the same seed, bit for bit."""
    import metropolisengine_b200 as me
    R, n = 4, 1024
    kr, temps = _rung_consts(name, R), [0.3, 0.7, 0.5, 1.1]
    a = _engine(me, name, kr, temps, n, every=0, seed=9, strict=strict)
    a.run(30, 7)
    a.step(5)
    a.measure()
    sa, ta = a.state.cpu().numpy(), a.time_series().cpu().numpy()
    xr, xc = _x0(name)
    for r in range(R):
        b = me.MetropolisEngine(_energy(me, name, kr[r]), initial_real_params=xr, initial_complex_params=xc,
                                temp=temps[r], n_chains=n, seed=9, strict=strict)
        b.run(30, 7)
        b.step(5)
        b.measure()
        assert np.array_equal(sa[:, r::R], b.state.cpu().numpy()[:, r::R]), r
        assert np.array_equal(ta[..., r::R], b.time_series().cpu().numpy()[..., r::R]), r


def _host_energy(name, x, k):
    """The built-in functors in their device operation order (me_energies.cuh), one chain per column."""
    if name == "xy_well":
        return k[0] * (x[0] * x[0] + x[1] * x[1])
    area = np.zeros(x.shape[1])
    for i in range(2):
        e = 1.0 - x[i]
        area = area + k[0] * (e * e)
    a = x[2] * x[2] + x[3] * x[3]
    s = np.zeros(x.shape[1]) + (k[1] * a + k[2] * (a * a))
    return area + (x[0] * x[1]) * (s / 1.0)


@pytest.mark.parametrize("strict", [False, True])
@pytest.mark.parametrize("name", ["xy_well", "2r1c"])
def test_energy_is_the_own_rungs_energy(name, strict):
    import metropolisengine_b200 as me
    R, n = 8, 8 * 512
    kr = _rung_consts(name, R)
    eng = _engine(me, name, kr, 0.5, n, seed=12, strict=strict)
    eng.run(50, 4)
    assert eng._swap_acc.sum().item() > 0
    st = eng.state.cpu().numpy()
    lay = eng._lay
    for r in range(R):
        cols = slice(r, None, R)
        want = _host_energy(name, st[lay.X:lay.X + lay.D, cols], kr[r])
        got = st[lay.E, cols]
        if strict:
            assert np.array_equal(got, want), r
        else:
            # FMA contraction rounds the terms, not the sum: the scale is that of the largest energy on the rung
            assert np.allclose(got, want, rtol=1e-12, atol=1e-12 * np.abs(want).max()), r


def test_walls_hold_per_rung():
    import metropolisengine_b200 as me
    R, n = 8, 8 * 256
    kr = _rung_consts("wall", R)
    eng = _engine(me, "wall", kr, list(np.geomspace(0.2, 3.0, R)), n, seed=5)
    eng.run(200, 5)
    assert eng._swap_acc.sum().item() > 0
    x0 = eng.time_series().cpu().numpy()[:, 0, :]                 # [rows, chains]
    for r in range(R):
        assert np.all(np.abs(x0[:, r::R]) < kr[r, 1]), r
    assert np.any(np.abs(x0[:, ::R]) > 0.6 * kr[0, 1])          # rung 0 does reach towards its wall


@pytest.mark.parametrize("strict", [False, True])
def test_equal_constants_are_the_temperature_ladder(strict):
    import metropolisengine_b200 as me
    R, n = 8, 8 * 512
    temps = list(np.geomspace(0.05, 2.0, R))
    h = _engine(me, "xy_well", np.ones((R, 1)), temps, n, seed=21, strict=strict)
    t = me.MetropolisEngine(me.BuiltinEnergy("xy_well", 1.0), initial_real_params=np.full(2, 0.3), temp=temps,
                            replica_exchange=1, n_chains=n, seed=21, strict=strict)
    for e in (h, t):
        e.run(40, 5)
    assert t._swap_acc.sum().item() > 0
    assert np.array_equal(h.walker_per_chain.cpu().numpy(), t.walker_per_chain.cpu().numpy())
    assert np.array_equal(h._swap_acc.cpu().numpy(), t._swap_acc.cpu().numpy())
    if strict:
        assert np.array_equal(h.state.cpu().numpy(), t.state.cpu().numpy())


def _barrier_ladder(swaps):
    import metropolisengine_b200 as me
    from scipy.integrate import quad
    T, R, n = 0.25, 8, 8 * 4096
    h = np.geomspace(5.0, 0.05, R)
    eng = me.MetropolisEngine(me.CudaEnergy(WELL_SRC, consts=[5.0]), initial_real_params=np.array([1.0]), temp=T,
                              rung_consts=h[:, None], replica_exchange=1 if swaps else 0, n_chains=n, seed=4)
    eng.run(2000, 10)
    ts = eng.time_series().cpu().numpy()[500:, 0, :]
    x0 = ts[:, ::R]                                             # rung 0 (the physical barrier) of every ladder
    neg = (x0 < 0).mean(axis=0)
    x2 = (x0 ** 2).mean(axis=0)
    z = quad(lambda x: np.exp(-h[0] * (x * x - 1) ** 2 / T), -4, 4)[0]
    want_x2 = quad(lambda x: x * x * np.exp(-h[0] * (x * x - 1) ** 2 / T), -4, 4)[0] / z
    return eng, neg, x2, want_x2


def test_barrier_ladder_carries_walkers_across():
    eng, neg, x2, want_x2 = _barrier_ladder(True)
    se = neg.std() / np.sqrt(neg.size)
    assert abs(neg.mean() - 0.5) < 5 * se, (neg.mean(), se)
    se2 = x2.std() / np.sqrt(x2.size)
    assert abs(x2.mean() - want_x2) < 5 * se2, (x2.mean(), want_x2, se2)
    rate = eng.swap_acceptance_rate
    assert rate.shape == (7,) and np.all(rate > 0.05) and np.all(rate <= 1), rate
    assert eng.rung_consts.shape == (8, 1) and np.array_equal(eng.temperatures, np.full(8, 0.25))


def test_without_swaps_the_physical_rung_stays_in_its_well():
    _, neg, _, _ = _barrier_ladder(False)
    assert neg.mean() < 1e-2, neg.mean()


def _gauss_acceptance(ka, kb):
    """E_r = k_r x^2 at one T: x_r = sqrt(T / (2 k_r)) z_r, so D = (k_a - k_b)(z_b^2 / k_b - z_a^2 / k_a) / 2."""
    from scipy.integrate import dblquad
    c = 1.0 / (2 * np.pi)

    def f(za, zb):
        d = 0.5 * (ka - kb) * (zb * zb / kb - za * za / ka)
        return min(1.0, np.exp(-d)) * c * np.exp(-0.5 * (za * za + zb * zb))
    return dblquad(f, -9, 9, -9, 9, epsabs=1e-9)[0]


def test_gaussian_ladder_variance_and_swap_acceptance():
    import metropolisengine_b200 as me
    T, R, n = 0.5, 8, 8 * 4096
    k = np.geomspace(0.25, 4.0, R)
    eng = me.MetropolisEngine(me.CudaEnergy(GAUSS_SRC, consts=[1.0]), initial_real_params=np.zeros(1), temp=T,
                              rung_consts=k[:, None], replica_exchange=1, n_chains=n, seed=17)
    eng.run(200, 5)                                              # burn-in
    eng.reset_pooled_statistics()
    eng.clear_time_series()
    acc0, att0 = eng._swap_acc.to(dtype=eng.state.dtype).cpu().numpy(), eng._swap_attempts()
    eng.run(1000, 5)
    var = eng.pooled_statistics()["cov_real"][:, 0, 0]
    x2 = (eng.time_series().cpu().numpy()[:, 0, :] ** 2).mean(axis=0).reshape(n // R, R)      # per ladder and rung
    for r in range(R):
        se = x2[:, r].std() / np.sqrt(n // R)
        assert abs(var[r] - T / (2 * k[r])) < 5 * se, (r, var[r], T / (2 * k[r]), se)
    acc = (eng._swap_acc.to(dtype=eng.state.dtype).cpu().numpy() - acc0).reshape(n // R, R)
    att = eng._swap_attempts() - att0
    for r in range(R - 1):
        per = acc[:, r] / att[r]
        se = per.std() / np.sqrt(per.size)
        want = _gauss_acceptance(k[r], k[r + 1])
        assert abs(per.mean() - want) < 5 * se, (r, per.mean(), want, se)


def _state(eng):
    return (eng.state.cpu().numpy(), eng.walker_per_chain.cpu().numpy(), eng._swap_acc.cpu().numpy())


def _same(a, b):
    for u, v in zip(a, b):
        assert np.array_equal(u, v)


def test_invariances():
    """run = the step / measure loop = ME_SEGMENTS=5 = run_graphed = checkpoint and resume = two shards."""
    import metropolisengine_b200 as me
    R, n = 8, 8 * 1024
    kr, temps = _rung_consts("xy_well", R), list(np.geomspace(0.1, 3.0, R))
    a = _engine(me, "xy_well", kr, temps, n, every=2, seed=3)
    a.run(40, 6)
    b = _engine(me, "xy_well", kr, temps, n, every=2, seed=3)
    for _ in range(40):
        b.step(6)
        b.measure()
    _same(_state(a), _state(b))
    assert np.array_equal(a.time_series().cpu().numpy(), b.time_series().cpu().numpy())
    old = os.environ.get("ME_SEGMENTS")
    os.environ["ME_SEGMENTS"] = "5"
    try:
        c = _engine(me, "xy_well", kr, temps, n, every=2, seed=3)
        c.run(40, 6)
    finally:
        if old is None:
            del os.environ["ME_SEGMENTS"]
        else:
            os.environ["ME_SEGMENTS"] = old
    _same(_state(a), _state(c))
    pa, pc = a.pooled_statistics(), c.pooled_statistics()
    assert pa["mean_real"].shape == (R, 2)
    assert np.allclose(pa["mean_real"], pc["mean_real"], rtol=1e-12, atol=1e-14)

    ref = _engine(me, "xy_well", kr, temps, n, every=1, seed=8, record=False)
    for _ in range(4):
        ref.run(10, 5)
    g = _engine(me, "xy_well", kr, temps, n, every=1, seed=8, record=False)
    for _ in range(4):
        g.run_graphed(10, 5)
    _same(_state(ref), _state(g))
    d0 = _engine(me, "xy_well", kr, temps, n, every=1, seed=8, record=False)
    d0.run(20, 5)
    sd = d0.state_dict()
    d = _engine(me, "xy_well", kr, temps, n, every=1, seed=8, record=False)
    d.load_state_dict(sd)
    d.run(20, 5)
    _same(_state(ref), _state(d))
    halves = [_engine(me, "xy_well", kr, temps, n, every=1, seed=8, record=False, _shard=(lo, hi))
              for lo, hi in ((0, n // 2), (n // 2, n))]
    for h in halves:
        for _ in range(4):
            h.run(10, 5)
    full = _state(ref)
    for i, h in enumerate(halves):
        part = _state(h)
        cols = slice(i * n // 2, (i + 1) * n // 2)
        assert np.array_equal(part[0], full[0][:, cols])
        assert np.array_equal(part[1], full[1][cols]) and np.array_equal(part[2], full[2][cols])


def test_rejections():
    import torch
    import metropolisengine_b200 as me
    from metropolisengine_b200 import _lib
    x0 = np.zeros(2)
    kr = np.array([[1.0], [2.0]])
    ok = dict(initial_real_params=x0, n_chains=64, rung_consts=kr)
    with pytest.raises(NotImplementedError):
        me.MetropolisEngine(("xy_well", 1.0), temp=0.5, adapt="pooled", **ok)
    with pytest.raises(NotImplementedError):
        me.MetropolisEngine(lambda r, c: (r ** 2).sum(-1), temp=0.5, **ok)
    with pytest.raises(NotImplementedError):
        me.MetropolisEngine(("xy_well", 1.0), reject_condition=lambda r, c: torch.zeros(64, dtype=torch.bool), temp=0.5,
                            **ok)
    with pytest.raises(NotImplementedError):
        me.MetropolisEngine(("cylinder", 1, 1, 1, 1), initial_real_params=np.zeros(1), initial_complex_params=np.zeros(16),
                            temp=0.5, n_chains=64, rung_consts=np.ones((2, 4)))
    with pytest.raises(NotImplementedError):
        me.MetropolisEngine(("mixed_well", 1.0, -1.0, 0.5), initial_real_params=np.zeros(2),
                            initial_complex_params=np.zeros(1), temp=0.5, n_chains=64, rung_consts=np.ones((2, 3)),
                            complex_sample_method="magnitude-phase")
    eng = me.MetropolisEngine(("xy_well", 1.0), temp=0.5, replica_exchange=1, **ok)
    with pytest.raises(NotImplementedError):
        eng.run_injected(np.zeros((1, 2)), np.zeros(1), 1, 1)
    with pytest.raises(NotImplementedError):
        eng.set_energy_function(("xy_well", 2.0))
    mixed = me.MetropolisEngine(("mixed_well", 1.0, -1.0, 0.5), initial_real_params=np.zeros(2),
                                initial_complex_params=np.zeros(1), temp=0.5, n_chains=64, rung_consts=np.ones((2, 3)))
    with pytest.raises(NotImplementedError):
        mixed.step_real_group()
    # the library refuses to evaluate proposals with one constant vector on a Hamiltonian ladder
    prop = torch.zeros((2, 64), dtype=torch.float64, device=eng.device)
    out = torch.zeros(64, dtype=torch.float64, device=eng.device)
    rc = eng._lib.me_energy_builtin(eng._h, ctypes.c_void_p(prop.data_ptr()), ctypes.c_void_p(out.data_ptr()), None,
                                    eng._stream())
    assert rc == _lib.ME_ERR_UNSUPPORTED
    bad = [dict(energy="x2", rung_consts=kr),                                       # the energy takes no constants
           dict(rung_consts=np.ones((2, 2))),                                       # K mismatch
           dict(rung_consts=kr, temp=[0.5, 1.0, 2.0]),                              # R != len(temp)
           dict(rung_consts=np.array([[1.0], [np.nan]])),                           # non-finite constants
           dict(rung_consts=np.array([[1.0], [np.inf]]), replica_exchange=0),
           dict(rung_consts=kr, temp=[0.0, 0.5], replica_exchange=1),              # T = 0 with swaps
           dict(rung_consts=kr, temp=0.0, replica_exchange=1),
           dict(rung_consts=np.ones(2)),                                            # not [R, K]
           dict(rung_consts=np.ones((1, 1))),                                       # one rung
           dict(rung_consts=np.ones((3, 1)), replica_exchange=1, n_chains=63),     # 3 rungs with swaps
           dict(rung_consts=kr, n_chains=63),                                       # not whole ladders
           dict(rung_consts=kr, _shard=(1, 33))]                                    # shard not ladder-aligned
    for kw in bad:
        args = dict(energy=("xy_well", 1.0), temp=0.5, n_chains=64)
        args.update(kw)
        energy = args.pop("energy")
        with pytest.raises((ValueError, AssertionError)):
            me.MetropolisEngine(energy, initial_real_params=x0, **args)
    down = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=[1.0, 0.5], rung_consts=kr,
                               replica_exchange=1, n_chains=64)        # any temperature order on a Hamiltonian ladder
    down.run(3, 2)
    sweep = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=0.5, rung_consts=np.ones((3, 1)),
                                n_chains=63)                              # sweep: any R
    sweep.run(3, 2)
    assert sweep.real_mean.shape == (3, 2)
