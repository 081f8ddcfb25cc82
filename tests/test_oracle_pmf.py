"""Free-energy profiles without a GPU: the numpy oracle (oracle/pmf_oracle.py) and the host algebra
(metropolisengine_b200/mbar.py, ``profile``) pinned on routes independent of them — pymbar's SVD of the explicit weight
matrix, a single rung's plain histogram, exact Gaussian bin integrals with the calibration of the error bars, the target
sum of ``pass_sums`` — and the argument checks of ``me_mbar_hist_pass`` that run before any device work."""
import ctypes

import numpy as np
import pytest
from scipy.special import erf

from metropolisengine_b200 import mbar as mb
from oracle import mbar_oracle as mo
from oracle import pmf_oracle as po


def _ladder(temps, n, rng, k=1.0):
    x = np.concatenate([rng.normal(0.0, np.sqrt(t / (2 * k)), size=(n, 2)) for t in temps])
    return x


def _u(x, temps, t_target, k=1.0):
    E = mo.energy("xy_well", x, [k])
    return np.stack([E / t for t in temps] + [E / t_target])


def _svd_route(W, n):
    """pymbar's svd-ew on the explicit weight matrix W [N, S]: W = U Sigma V^T,
    Theta = V Sigma (I - Sigma V^T diag(n) V Sigma)^+ Sigma V^T."""
    _, sig, vt = np.linalg.svd(W, full_matrices=False)
    V = vt.T
    inner = np.eye(sig.size) - np.diag(sig) @ V.T @ np.diag(n) @ V @ np.diag(sig)
    return V @ np.diag(sig) @ np.linalg.pinv(inner, rcond=1e-10) @ np.diag(sig) @ V.T


def test_oracle_matches_pymbars_weight_matrix_route():
    rng = np.random.default_rng(7)
    temps = np.array([0.5, 0.8, 1.3])
    n = 800
    x = _ladder(temps, n, rng)
    u = _u(x, temps, 0.65)
    f, _, conv = mo.solve(u[:3], n)
    assert conv
    lo, hi, nb = -1.2, 1.2, 12
    hs = po.hist_sums(u, f, n, 3, [x[:, 0]], [lo], [hi], [nb])
    G = mo.pass_sums(u[:3], f, n, 3)["G"]
    got_f, got_df, _ = po.pmf(hs["h"], hs["q"], hs["c"], hs["w_out"], G, n)
    host_f, host_df, _ = mb.profile(hs["h"], hs["q"], hs["c"], hs["w_out"], G, n)
    W = mo.pass_sums(u, f, n, 3)["W"]
    b = hs["bins"]
    full = np.flatnonzero(hs["h"] > 0)
    Wb = np.stack([np.where(b == k, W[:, 3], 0.0) / hs["h"][k] for k in full], axis=1)
    th = _svd_route(np.concatenate([W[:, :3], Wb], axis=1), np.concatenate([np.full(3, float(n)), np.zeros(full.size)]))
    fb = -np.log(hs["h"][full])
    r = int(np.argmin(fb))
    want_f = fb - fb[r]
    want_df = np.sqrt(np.clip(np.diag(th)[3:] + th[3 + r, 3 + r] - 2 * th[3:, 3 + r], 0, None))
    for ff, dd in ((got_f, got_df), (host_f, host_df)):
        assert np.allclose(ff[full], want_f, rtol=0, atol=1e-10)
        assert np.allclose(dd[full], want_df, rtol=0, atol=1e-10), (dd[full], want_df)


def test_single_rung_is_the_plain_histogram():
    rng = np.random.default_rng(8)
    x = rng.normal(0.0, 0.5, size=(5000, 2))
    u = _u(x, [0.5], 0.5)
    hs = po.hist_sums(u, np.zeros(1), 5000, 1, [x[:, 1]], [-1.0], [1.0], [16])
    counts, _ = np.histogram(x[:, 1], bins=16, range=(-1.0, 1.0))
    for fn in (po.pmf, mb.profile):
        f, _, p = fn(hs["h"], hs["q"], hs["c"], hs["w_out"], np.array([[1.0 / 5000]]), 5000, reference=8)
        assert np.allclose(f, -np.log(counts / counts[8]), rtol=0, atol=1e-12)
        assert np.allclose(p, counts / 5000.0, rtol=0, atol=1e-14)


def test_exact_gaussian_profile_and_error_calibration():
    """x ~ N(0, T / 2) at a target T between the rungs: f_b - f_r = -ln(P_b / P_r) with P_b the exact bin integral.
    The reference bin is fixed (the argmin of "lowest" would bias the z-scores)."""
    temps = np.array([0.4, 0.7, 1.2])
    tt, lo, hi, nb, ref = 0.55, -1.0, 1.0, 8, 3
    edges = np.linspace(lo, hi, nb + 1)
    s = np.sqrt(tt / 2)
    P = 0.5 * (erf(edges[1:] / (s * np.sqrt(2))) - erf(edges[:-1] / (s * np.sqrt(2))))
    exact = -np.log(P / P[ref])
    z = []
    for rep in range(200):
        rng = np.random.default_rng(500 + rep)
        n = 600
        x = _ladder(temps, n, rng)
        u = _u(x, temps, tt)
        f, _, conv = mo.solve(u[:3], n)
        assert conv
        hs = po.hist_sums(u, f, n, 3, [x[:, 0]], [lo], [hi], [nb])
        G = mo.pass_sums(u[:3], f, n, 3)["G"]
        fb, dfb, _ = mb.profile(hs["h"], hs["q"], hs["c"], hs["w_out"], G, n, reference=ref)
        keep = np.arange(nb) != ref
        z.extend(((fb - exact) / dfb)[keep])
    z = np.array(z)
    assert np.mean(np.abs(z) > 4) < 0.01
    assert 0.85 <= z.std() <= 1.15, z.std()


def test_bin_weights_and_outside_weight_sum_to_the_target_sum():
    rng = np.random.default_rng(9)
    temps = np.array([0.5, 1.0])
    x = _ladder(temps, 1000, rng)
    u = _u(x, temps, 0.7)
    f, _, _ = mo.solve(u[:2], 1000)
    hs = po.hist_sums(u, f, 1000, 2, [x[:, 0], x[:, 1]], [-0.8, -0.5], [0.8, 0.9], [7, 5])
    s_t = mo.pass_sums(u, f, 1000, 2)["s"][2]
    assert abs(hs["h"].sum() + hs["w_out"] - s_t) <= 1e-12 * s_t
    assert hs["n_out"] > 0 and hs["h"].shape == (35,)


def test_bin_rule_edges():
    c = np.array([-1.0, -0.5, 0.0, 1.0 - 1e-16, 1.0, np.nan, -1.0000000001, 0.25])
    assert po.bin_index(c, -1.0, 1.0, 4).tolist() == [0, 1, 2, 3, -1, -1, -1, 2]
    # (hi - eps - lo) * inv_w can round to n: that sample stays in the last bin
    lo, hi, n = 0.1, 0.7, 3
    top = np.nextafter(hi, 0.0)
    assert po.bin_index(np.array([top]), lo, hi, n)[0] == n - 1


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


def _arr(t, v):
    return None if v is None else ctypes.cast((t * max(len(v), 1))(*v), ctypes.c_void_p)


def _pass(lib, h, rows=10, row0=0, stride=1, n_per=64, temp=0.7, consts=None, n_axes=1, kind=(0,), index=(0,),
          lo=(-1.0,), hi=(1.0,), bins=(10,), ts=_FAKE, f=_FAKE, sums=_FAKE):
    i32, f64 = ctypes.c_int32, ctypes.c_double
    return lib.load().me_mbar_hist_pass(h, ts, rows, row0, stride, f, n_per, temp, _arr(f64, consts), n_axes,
                                        _arr(i32, kind), _arr(i32, index), _arr(f64, lo), _arr(f64, hi),
                                        _arr(i32, bins), sums, 0, None)


def test_mbar_hist_pass_validates_before_device_work(lib):
    L = lib.load()
    inv, nan, inf = lib.ME_ERR_INVALID, float("nan"), float("inf")
    cases = [
        ({}, dict(n_axes=0), inv, "n_axes"),
        ({}, dict(n_axes=3), inv, "n_axes"),
        ({}, dict(kind=(2,)), inv, "coord_kind"),
        ({}, dict(index=(2,)), inv, "[0, D)"),
        ({}, dict(index=(-1,)), inv, "[0, D)"),
        ({}, dict(kind=(1,)), inv, "n_complex"),                               # no complex parameter
        (dict(nr=2, nc=1, energy="mixed_well", consts=(1.0, -1.0, 0.5, 1.0)), dict(kind=(1,), index=(1,)), inv,
         "n_complex"),
        ({}, dict(lo=(nan,)), inv, "finite lo and hi"),
        ({}, dict(hi=(inf,)), inv, "finite lo and hi"),
        ({}, dict(lo=(1.0,), hi=(1.0,)), inv, "hi > lo"),
        ({}, dict(bins=(0,)), inv, "n_bins"),
        ({}, dict(n_axes=2, kind=(0, 0), index=(0, 1), lo=(0, 0), hi=(1, 1), bins=(4, -1)), inv, "n_bins"),
        ({}, dict(bins=(8193,)), inv, "24576"),                                # 8193 x (1 + 2) > 24576
        ({}, dict(n_axes=2, kind=(0, 0), index=(0, 1), lo=(0, 0), hi=(1, 1), bins=(100, 100)), inv, "24576"),
        ({}, dict(temp=0.0), inv, "target temperature"),
        ({}, dict(temp=nan), inv, "target temperature"),
        ({}, dict(temp=inf), inv, "target temperature"),
        ({}, dict(consts=[nan]), inv, "finite"),
        (dict(temp=0.0), {}, inv, "rung temperature"),
        ({}, dict(row0=10), inv, "row0"),
        ({}, dict(row0=-1), inv, "row0"),
        ({}, dict(stride=0), inv, "stride"),
        ({}, dict(n_per=0), inv, "n_per_state"),
        ({}, dict(ts=None), inv, "required"),
        ({}, dict(f=None), inv, "required"),
        ({}, dict(sums=None), inv, "required"),
        ({}, dict(kind=None), inv, "required"),
        ({}, dict(index=None), inv, "required"),
        ({}, dict(lo=None), inv, "required"),
        ({}, dict(hi=None), inv, "required"),
        ({}, dict(bins=None), inv, "required"),
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
    assert "group" in L.me_last_error(h).decode()
    L.me_destroy(h)


def test_mbar_hist_words_is_the_documented_length(lib):
    L = lib.load()
    h = _handle(lib)
    w = ctypes.c_int64()
    for bins in ((1,), (100,), (40, 40), (3, 7)):
        nb = (ctypes.c_int32 * len(bins))(*bins)
        assert L.me_mbar_hist_words(h, len(bins), ctypes.cast(nb, ctypes.c_void_p), ctypes.byref(w)) == lib.ME_OK
        assert w.value == 4 + int(np.prod(bins)) * (1 + 2)
    nb = (ctypes.c_int32 * 1)(8193)
    assert L.me_mbar_hist_words(h, 1, ctypes.cast(nb, ctypes.c_void_p), ctypes.byref(w)) == lib.ME_ERR_INVALID
    L.me_destroy(h)
