"""Host restatement of the MBAR contract (DESIGN §3 "MBAR over recorded ladder rows") on numpy arrays of samples.

Checker code only: the product computes the same quantities with the device pass (csrc/me_mbar.cuh) and
``metropolisengine_b200/mbar.py``.  Everything is written from the contract, not from those files:

    u_s(x) = E(x; k_s) / T_s (+inf where the wall rejects x under k_s)
    L_n = ln sum_k N_k exp(f_k - u_k(x_n)),  w_ns = exp(f_s - u_s(x_n) - L_n)   (f = 0 for target states)
    sum L, s_s = sum_n w_ns, G_st = sum_n w_ns w_nt, sum_n w_ns a_s(x_n), a_s = [x, x^2, E_s, E_s^2]
    F(f) = sum L - sum_k N_k f_k, gradient N_i (s_i - 1), Hessian diag(N s) - N N^T * G; Newton with f_0 = 0
    Theta = V Sigma (I - Sigma V^T diag(N) V Sigma)^+ Sigma V^T from G = V Sigma^2 V^T
"""
import numpy as np
from scipy.special import logsumexp


# ---------------------------------------------------------------------------------------- energies on [n, D] samples
def energy(name, x, k):
    """The built-in functors of csrc/me_energies.cuh, vectorised over samples x [n, D] (real, Re c, Im c)."""
    x = np.asarray(x, dtype=np.float64)
    if name == "x2":
        return x[:, 0] * x[:, 0]
    if name == "xy_well":
        return k[0] * (x[:, 0] * x[:, 0] + x[:, 1] * x[:, 1])
    raise ValueError(name)


def mixed_well(nr, nc):
    def e(x, k):
        area = sum(k[0] * (1.0 - x[:, i]) ** 2 for i in range(nr))
        s = 0.0
        for j in range(nc):
            a = x[:, nr + j] ** 2 + x[:, nr + nc + j] ** 2
            s = s + (k[1] * a + k[2] * a * a)
        w = x[:, 0] * x[:, 1]
        return area + (np.abs(w) if k[3] != 0 else w) * (s / nc)
    return e


def energies(efn, x, consts, reject=None):
    """E [S, n] of samples x [n, D] under every constant vector of consts [S, K]; walled[S, n] from reject(x, k)."""
    E = np.stack([efn(x, k) for k in consts])
    walled = np.zeros(E.shape, dtype=bool) if reject is None else np.stack([reject(x, k) for k in consts])
    return np.where(walled, 0.0, E), walled


def reduced(E, walled, temps):
    return np.where(walled, np.inf, E / np.asarray(temps, dtype=np.float64)[:, None])


# ---------------------------------------------------------------------------------------- one pass
def pass_sums(u, f, n_per, n_rungs, obs=None):
    """u [S, n] reduced potentials (rungs first), f [R].  obs: [S, n, m] per-state observables a_s(x_n).
    Returns sum_l, s [S], G [S, S], W [n, S] and, with obs, sum_n w_ns a_s [S, m]."""
    R = n_rungs
    with np.errstate(invalid="ignore"):
        a = np.log(float(n_per)) + np.asarray(f, dtype=np.float64)[:, None] - u[:R]
    L = logsumexp(a, axis=0)
    fs = np.concatenate([np.asarray(f, dtype=np.float64), np.zeros(u.shape[0] - R)])
    W = np.exp(fs[:, None] - u - L[None, :]).T
    out = dict(sum_l=float(L.sum()), s=W.sum(axis=0), G=W.T @ W, W=W)
    if obs is not None:
        out["obs"] = np.einsum("ns,snm->sm", W, obs)
    return out


def objective(f, u_rungs, n_per):
    return pass_sums(u_rungs, f, n_per, u_rungs.shape[0])["sum_l"] - n_per * np.sum(f)


def solve(u_rungs, n_per, tol=1e-10, max_iter=100):
    """Newton on F with f_0 = 0, Armijo backtracking, self-consistent step when the reduced Hessian is indefinite."""
    R, N = u_rungs.shape[0], float(n_per)
    f = np.zeros(R)
    for it in range(max_iter + 1):
        p = pass_sums(u_rungs, f, N, R)
        if np.max(np.abs(p["s"] - 1.0)) < tol or it == max_iter:
            return f, it, bool(np.max(np.abs(p["s"] - 1.0)) < tol)
        g = N * (p["s"] - 1.0)
        H = np.diag(N * p["s"]) - N * N * p["G"]
        try:
            np.linalg.cholesky(H[1:, 1:])
        except np.linalg.LinAlgError:
            f = f - np.log(p["s"])
            f -= f[0]
            continue
        d = np.zeros(R)
        d[1:] = -np.linalg.solve(H[1:, 1:], g[1:])
        F0, t = p["sum_l"] - N * f.sum(), 1.0
        while t > 1e-8 and objective(f + t * d, u_rungs, N) > F0 + 1e-4 * t * (g @ d) + 1e-12 * max(abs(F0), 1.0):
            t *= 0.5
        f = f + t * d


def theta(G, n):
    lam, V = np.linalg.eigh(G)
    sig = np.sqrt(np.clip(lam, 0.0, None))
    M = np.eye(G.shape[0]) - np.diag(sig) @ V.T @ np.diag(np.asarray(n, dtype=np.float64)) @ V @ np.diag(sig)
    return V @ np.diag(sig) @ np.linalg.pinv(M, rcond=1e-10) @ np.diag(sig) @ V.T


def df(th, i, j):
    return float(np.sqrt(max(th[i, i] + th[j, j] - 2.0 * th[i, j], 0.0)))


def observables(x, E):
    """a_s(x_n) = [x, x^2, E_s, E_s^2] for every state: [S, n, 2D + 2] from x [n, D] and E [S, n]."""
    S = E.shape[0]
    xx = np.concatenate([x, x * x], axis=1)
    return np.concatenate([np.broadcast_to(xx, (S,) + xx.shape), E[:, :, None], (E * E)[:, :, None]], axis=2)


def evaluate(u, E, x, f, n_per, n_rungs):
    """Targets (the states after the rungs in u / E): f_t = -ln s_t, <a>_t, df against rung 0; for every state."""
    R, S = n_rungs, u.shape[0]
    p = pass_sums(u, f, n_per, R, observables(x, E))
    fa = np.concatenate([np.asarray(f, dtype=np.float64), -np.log(p["s"][R:])])
    th = theta(p["G"], np.concatenate([np.full(R, float(n_per)), np.zeros(S - R)]))
    mean = p["obs"] / p["s"][:, None]
    return dict(f=fa, df=np.array([df(th, 0, s) for s in range(S)]), mean=mean, sums=p)
