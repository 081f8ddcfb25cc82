"""MBAR free-energy profiles on the GPU (k_mbar_hist, me_mbar_hist_pass; MBARResult.pmf): the histogram sums against
the numpy oracle (oracle/pmf_oracle.py) on the engine's own rows, the full profile against the oracle's, analytic
profiles from real Metropolis chains, the invariances and the refusals."""
import math

import numpy as np
import pytest
from scipy.integrate import quad
from scipy.special import erf

pytestmark = pytest.mark.gpu

WALL_SRC = """
__device__ double me_user_energy(const double* x, const double* cr, const double* ci, const double* k) {
    return k[0] * (x[0] * x[0] + x[1] * x[1]);
}
__device__ bool me_user_reject(const double* x, const double* cr, const double* ci, const double* k) {
    return x[0] >= k[1];
}
"""
WELL_SRC = """
__device__ double me_user_energy(const double* x, const double* cr, const double* ci, const double* k) {
    const double a = x[0] * x[0] - 1.0; return k[0] * a * a; }"""


def _me():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import metropolisengine_b200 as me
    return me


def _pad(k):
    k = np.atleast_2d(np.asarray(k, dtype=np.float64))
    return np.concatenate([k, np.zeros((k.shape[0], 16 - k.shape[1]))], axis=1)


def _case(me, name, R, strict=False, n_per_rung=64):
    """(engine, numpy energy, reject, rung temperatures, rung constants [R, 16], (n_real, n_complex), K)."""
    from oracle import mbar_oracle as mo
    common = dict(n_chains=R * n_per_rung, seed=13, strict=strict, device="cuda:0")
    xy = lambda x, k: mo.energy("xy_well", x, k)  # noqa: E731
    if name == "xy_temp":
        temps = np.geomspace(0.2, 2.0, R)
        eng = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.array([0.1, -0.2]),
                                  temp=list(temps) if R > 1 else float(temps[0]), replica_exchange=1 if R > 1 else 0,
                                  **common)
        return eng, xy, None, temps, _pad(np.ones((R, 1))), (2, 0), 1
    if name == "xy_ham":
        kr = np.geomspace(0.3, 3.0, R)[:, None]
        eng = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.array([0.1, -0.2]), temp=0.5,
                                  rung_consts=kr, replica_exchange=1, **common)
        return eng, xy, None, np.full(R, 0.5), _pad(kr), (2, 0), 1
    if name == "mixed_ham":
        kr = np.stack([np.linspace(0.5, 1.5, R), np.linspace(-1.0, -0.2, R), np.linspace(0.3, 0.8, R),
                       np.ones(R)], axis=1)
        eng = me.MetropolisEngine(me.BuiltinEnergy("mixed_well", *kr[0]), initial_real_params=np.array([0.3, 0.3]),
                                  initial_complex_params=np.array([0.2 - 0.1j]), temp=0.4, rung_consts=kr,
                                  replica_exchange=1, **common)
        return eng, mo.mixed_well(2, 1), None, np.full(R, 0.4), _pad(kr), (2, 1), 4
    if name == "wall":
        kr = np.stack([np.linspace(0.5, 1.5, R), np.linspace(0.3, 1.2, R)], axis=1)
        eng = me.MetropolisEngine(me.CudaEnergy(WALL_SRC, consts=list(kr[0]), has_reject=True),
                                  initial_real_params=np.array([0.0, 0.0]), temp=0.7, rung_consts=kr,
                                  replica_exchange=1, **common)
        return (eng, lambda x, k: k[0] * (x[:, 0] ** 2 + x[:, 1] ** 2), lambda x, k: x[:, 0] >= k[1],
                np.full(R, 0.7), _pad(kr), (2, 0), 2)
    raise ValueError(name)


def _samples(eng, row0, stride):
    ts = eng.time_series().cpu().numpy()[row0::stride]
    d = eng._d
    return ts[:, :d, :].transpose(0, 2, 1).reshape(-1, d)          # sample n = (row, chain), chain fastest


def _oracle_sums(eng, efn, rej, temps, consts, f, tt, kt, axes, lo, hi, nb, shape, row0, stride):
    from oracle import mbar_oracle as mo
    from oracle import pmf_oracle as po
    R = temps.size
    x = _samples(eng, row0, stride)
    allk = np.concatenate([consts, _pad(kt) if kt is not None else consts[:1]])
    E, walled = mo.energies(efn, x, allk, rej)
    u = mo.reduced(E, walled, np.concatenate([temps, [tt]]))
    n_per = x.shape[0] // R
    coords = [po.coordinate(x, k, j, *shape) for k, j in axes]
    return po.hist_sums(u, f, n_per, R, coords, lo, hi, nb), mo.pass_sums(u[:R], f, n_per, R)["G"], n_per


def _close(a, b, rel):
    a, b = np.asarray(a), np.asarray(b)
    scale = max(np.max(np.abs(b)), 1e-300)
    assert np.all(np.abs(a - b) <= rel * scale), (np.max(np.abs(a - b)) / scale, a, b)


CASES = [("xy_temp", 1, False), ("xy_temp", 2, False), ("xy_temp", 8, False), ("xy_temp", 32, False),
         ("xy_temp", 8, True), ("xy_ham", 8, False), ("xy_ham", 8, True), ("mixed_ham", 4, False),
         ("mixed_ham", 4, True), ("wall", 4, False), ("wall", 4, True)]


@pytest.mark.parametrize("name,R,strict", CASES)
@pytest.mark.parametrize("between", [False, True])
@pytest.mark.parametrize("two_d", [False, True])
def test_hist_sums_match_the_oracle(name, R, strict, between, two_d):
    me = _me()
    eng, efn, rej, temps, consts, shape, K = _case(me, name, R, strict)
    eng.run(30, 4)
    rng = np.random.default_rng(R + 100 * between)
    f = np.concatenate([[0.0], rng.normal(0.0, 0.5, R - 1)])
    if between:
        tt = float(temps[0] * 1.07)
        kt = None if name == "xy_temp" else 0.5 * (consts[0, :K] + consts[min(1, R - 1), :K])
    else:
        tt, kt = float(temps[0]), (None if name == "xy_temp" else consts[0, :K])
    if name == "mixed_ham":
        axes = [(1, 0), (0, 0)] if two_d else [(1, 0)]                  # |c_0|, then x_0
        lo, hi, nb = [0.05, -0.5][:len(axes)], [0.6, 1.0][:len(axes)], [13, 9][:len(axes)]
    else:
        axes = [(0, 0), (0, 1)] if two_d else [(0, 0)]
        lo, hi, nb = [-0.5, -0.45][:len(axes)], [0.4, 0.6][:len(axes)], [17, 11][:len(axes)]
    row0, stride = 5, 2
    got = eng._mbar_hist_sums(f, tt, kt, [a[0] for a in axes], [a[1] for a in axes], lo, hi, nb, row0, stride)
    want, _, _ = _oracle_sums(eng, efn, rej, temps, consts, f, tt, kt, axes, lo, hi, nb, shape, row0, stride)
    assert got["n_nan"] == 0 and got["n_overflow"] == 0
    assert got["n_out"] == want["n_out"]
    assert np.count_nonzero(want["h"]) > 3                                 # several bins fill
    # every sample in the same bin: each bin's own sum agrees to rounding (a moved sample changes it by its weight)
    hb, wb = got["h"], want["h"]
    assert np.array_equal(hb > 0, wb > 0)
    assert np.all(np.abs(hb - wb) <= 1e-12 * wb), np.max(np.abs(hb - wb) / np.maximum(wb, 1e-300))
    _close(got["q"], want["q"], 1e-12)
    _close(got["c"], want["c"], 1e-12)
    assert abs(got["w_out"] - want["w_out"]) <= 1e-12 * max(want["w_out"], 1e-300)


def test_pmf_matches_the_oracle_pmf():
    from oracle import pmf_oracle as po
    me = _me()
    eng, efn, rej, temps, consts, shape, _ = _case(me, "xy_temp", 8, n_per_rung=256)
    eng.run(50, 5)
    res = eng.mbar(burn_in=0.2, stride=1)
    row0 = int(eng._ts_rows * 0.2)
    for axes, bins, rng_ in ((0, 15, (-1.0, 1.0)), ((0, 1), (9, 7), ((-1.0, 1.0), (-0.8, 0.8)))):
        got = res.pmf(axes, bins, rng_, temp=0.5)
        ax = [(0, a) for a in np.atleast_1d(axes)]
        nb = list(np.atleast_1d(bins))
        rg = np.atleast_2d(rng_)
        want, G, n_per = _oracle_sums(eng, efn, rej, temps, consts, res.free_energies, 0.5, None, ax, rg[:, 0],
                                      rg[:, 1], nb, shape, row0, 1)
        f, df, p = po.pmf(want["h"], want["q"], want["c"], want["w_out"], G, n_per)
        full = want["h"] > 0
        assert np.allclose(got["f"].ravel()[full], f[full], rtol=0, atol=1e-9)
        assert np.allclose(got["df"].ravel()[full], df[full], rtol=1e-7, atol=1e-12)
        assert np.allclose(got["p"].ravel(), p, rtol=1e-10, atol=1e-15)
        assert got["f"].shape == tuple(nb) and len(got["edges"]) == len(nb)


def _stride(eng):
    g = eng.statistical_inefficiency(column=eng._d, n_chains=2048, burn_in=0.5)
    return int(math.ceil(float(g.max().item())))


def test_double_well_hremd_profile_is_analytic():
    """README's H-REMD double well: rung 0 (barrier 5 at T = 0.25) along x against -ln int_bin exp(-k (x^2 - 1)^2 / T)."""
    me = _me()
    h = np.geomspace(5.0, 0.05, 8)
    eng = me.MetropolisEngine(me.CudaEnergy(WELL_SRC, consts=[5.0]), initial_real_params=np.array([1.0]), temp=0.25,
                              rung_consts=h[:, None], replica_exchange=1, n_chains=8 * 4096, seed=17, device="cuda:0",
                              ts_chunk_bytes=4 << 30)                  # one chunk: statistical_inefficiency reads it
    eng.run(2000, 10)
    res = eng.mbar(burn_in=0.5, stride=_stride(eng))
    nb, lo, hi = 24, -1.6, 1.6
    out = res.pmf(0, nb, (lo, hi), reference=6)
    e = out["edges"][0]
    Z = np.array([quad(lambda x: np.exp(-5.0 * (x * x - 1) ** 2 / 0.25), e[i], e[i + 1])[0] for i in range(nb)])
    exact = -np.log(Z / Z[6])
    keep = np.isfinite(out["f"]) & (np.arange(nb) != 6)
    assert keep.sum() >= nb - 2
    z = (out["f"] - exact)[keep] / out["df"][keep]
    assert np.mean(np.abs(z) > 4) <= 0.1, z
    mid = nb // 2                                                        # the barrier bins hold weight at rung 0
    assert np.isfinite(out["f"][mid]) and out["f"][mid] > 10


def test_xy_temperature_ladder_2d_profile_is_analytic():
    me = _me()
    temps = np.geomspace(0.5, 2.0, 8)
    eng = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=np.array([0.0, 0.0]), temp=list(temps),
                              replica_exchange=1, n_chains=8 * 4096, seed=3, sampling_width=0.5, device="cuda:0")
    eng.run(1000, 10)
    res = eng.mbar(burn_in=0.5, stride=_stride(eng))
    tt, nb, lo, hi = 0.8, 8, -1.2, 1.2
    ref = (3, 4)
    out = res.pmf((0, 1), (nb, nb), ((lo, hi), (lo, hi)), temp=tt, reference=ref)
    e = out["edges"][0]
    s = np.sqrt(tt / 2) * np.sqrt(2)
    P1 = 0.5 * (erf(e[1:] / s) - erf(e[:-1] / s))
    P = np.outer(P1, P1)
    exact = -np.log(P / P[ref])
    keep = np.ones((nb, nb), dtype=bool)
    keep[ref] = False
    z = (out["f"] - exact)[keep] / out["df"][keep]
    assert np.mean(np.abs(z) > 4) <= 0.05, z
    assert abs(out["weight_outside"] - (1 - P.sum())) <= 0.02


def test_invariances():
    me = _me()
    temps = list(np.geomspace(0.3, 1.5, 4))
    kw = dict(initial_real_params=np.array([0.1, 0.0]), temp=temps, replica_exchange=1, seed=21, device="cuda:0")
    a = me.MetropolisEngine(("xy_well", 1.0), n_chains=1024, **kw)
    a.run(40, 5)
    f = a.mbar(burn_in=0.1).free_energies
    args = (f, 0.7, None, [0, 0], [0, 1], [-1.0, -1.0], [1.0, 1.0], [12, 10], 4, 3)
    s1, s2 = a._mbar_hist_sums(*args), a._mbar_hist_sums(*args)
    for k in ("h", "q", "c"):
        assert np.array_equal(s1[k], s2[k])                                       # bit-identical from run to run
    assert s1["w_out"] == s2["w_out"]
    b = me.MetropolisEngine(("xy_well", 1.0), n_chains=1024, ts_chunk_bytes=7 * 3 * 1024 * 8, **kw)   # several chunks
    b.run(40, 5)
    assert len([c for c in b._ts_chunks if c[1]]) > 3
    sb = b._mbar_hist_sums(*args)
    for k in ("h", "q", "c"):
        _close(sb[k], s1[k], 1e-13)
    halves = []
    for lo, hi in ((0, 512), (512, 1024)):
        e = me.MetropolisEngine(("xy_well", 1.0), n_chains=1024, _shard=(lo, hi), **kw)
        e.run(40, 5)
        halves.append(e._mbar_hist_sums(*args))
    for k in ("h", "q", "c"):
        _close(halves[0][k] + halves[1][k], s1[k], 1e-13)
    assert halves[0]["n_out"] + halves[1]["n_out"] == s1["n_out"]


def test_shard_ranges_hold_whole_ladders():
    from metropolisengine_b200 import parallel
    me = _me()
    R = 4
    kw = dict(initial_real_params=np.array([0.1, 0.0]), temp=list(np.geomspace(0.3, 1.5, R)), replica_exchange=1,
              seed=23, device="cuda:0")
    full = me.MetropolisEngine(("xy_well", 1.0), n_chains=R * 300, **kw)
    full.run(20, 5)
    f = full.mbar(burn_in=0.1).free_energies
    args = (f, 0.9, None, [0], [0], [-1.0], [1.0], [20], 2, 2)
    want = full._mbar_hist_sums(*args)
    got = None
    for rank in range(3):
        lo, hi = parallel.shard_range(R * 300, rank, 3, granule=R)
        e = me.MetropolisEngine(("xy_well", 1.0), n_chains=R * 300, _shard=(lo, hi), **kw)
        e.run(20, 5)
        s = e._mbar_hist_sums(*args)
        got = s if got is None else {k: got[k] + s[k] for k in ("h", "q", "c", "w_out", "n_out")}
    for k in ("h", "q", "c"):
        _close(got[k], want[k], 1e-13)


def test_refusals():
    me = _me()
    x0 = np.array([0.1, 0.0])
    e = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=0.5, n_chains=64, seed=2, device="cuda:0")
    e.run(10, 2)
    res = e.mbar()
    for bad in (dict(coords=2), dict(coords=("abs", 0)), dict(coords=-1), dict(coords=(0, 1, 0)),
                dict(coords="x"), dict(bins=0), dict(bins=(4, 4)), dict(bins=2.5), dict(range=(1.0, 1.0)),
                dict(range=(0.0, float("inf"))), dict(range=(1.0, -1.0)), dict(bins=30000),
                dict(temp=0.0), dict(temp=[0.5, 0.6]), dict(consts=[1.0, 2.0]), dict(consts=[float("nan")]),
                dict(reference=50), dict(reference="highest")):
        kw = dict(coords=0, bins=10, range=(-1.0, 1.0))
        kw.update(bad)
        with pytest.raises(ValueError):
            res.pmf(**kw)
    with pytest.raises(ValueError, match="reference bin is empty"):
        res.pmf(0, 10, (-50.0, 50.0), reference=0)
    ham = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=0.5, rung_consts=[[1.0], [2.0]],
                              n_chains=64, device="cuda:0")
    ham.run(10, 2)
    hres = ham.mbar()
    with pytest.raises(ValueError, match="target_consts"):
        hres.pmf(0, 10, (-1.0, 1.0), temp=0.5)
    assert np.isfinite(hres.pmf(0, 10, (-1.0, 1.0))["f"]).any()             # default target: rung 0 and its consts
    lad = me.MetropolisEngine(("xy_well", 1.0), initial_real_params=x0, temp=[0.5, 0.7], n_chains=64, device="cuda:0")
    lad.run(10, 2)
    with pytest.raises(ValueError, match="temp"):
        lad.mbar().pmf(0, 10, (-1.0, 1.0), consts=[1.0])
    wide = me.MetropolisEngine(("x2",), initial_real_params=np.zeros(33), temp=0.5, n_chains=32, device="cuda:0")
    with pytest.raises(NotImplementedError):
        wide.mbar()
    cal = me.MetropolisEngine(lambda r, c: (r * r).sum(dim=1), initial_real_params=x0, temp=0.5, n_chains=64,
                              device="cuda:0")
    with pytest.raises(NotImplementedError):
        cal.mbar()
