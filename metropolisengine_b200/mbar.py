"""MBAR over the recorded rows of a ladder: free energies between rungs, reweighted expectations and their asymptotic
uncertainties (Shirts & Chodera, J. Chem. Phys. 129, 124105, 2008; pymbar's ``MBAR``).

The device pass (``me_mbar_pass``, csrc/me_mbar.cuh) reduces every sample to a few FP64 sums for a given vector of rung
free energies f; everything here is S x S algebra on those sums (S <= 32 states):

* the Newton solve of the convex objective F(f) = sum_n L_n - N sum_k f_k in the gauge f_0 = 0, with a backtracking
  line search on F (one pass per trial point) and the self-consistent step f_i <- f_i - ln s_i when the reduced Hessian
  is not positive definite;
* pymbar's ``svd-ew`` asymptotic covariance Theta from the Gram matrix G of the weights;
* target states: f_t = -ln s_t and <a>_t = sum_n w_nt a_t / s_t.

The covariance assumes uncorrelated samples: pass ``stride`` of about the statistical inefficiency g of the energy
column (``MetropolisEngine.statistical_inefficiency``).
"""
import numpy as np


def unpack(sums, n_states, d, with_obs):
    """The sums vector of ``me_mbar_pass`` as a dict: ``sum_l``, ``n_nan``, ``n_overflow``, ``s`` [S], ``G`` [S, S]
    (symmetric) and, with observables, ``obs`` [S, 2D + 2] (sum_n w_ns [x, x^2, E_s, E_s^2])."""
    S = n_states
    sums = np.asarray(sums, dtype=np.float64)
    out = dict(sum_l=float(sums[0]), n_nan=int(sums[1]), n_overflow=int(sums[2]), s=sums[3:3 + S].copy())
    G = np.zeros((S, S))
    G[np.tril_indices(S)] = sums[3 + S:3 + S + S * (S + 1) // 2]
    out["G"] = G + np.tril(G, -1).T
    if with_obs:
        o = 3 + S + S * (S + 1) // 2
        out["obs"] = sums[o:o + S * (2 * d + 2)].reshape(S, 2 * d + 2).copy()
    return out


def theta(G, n):
    """pymbar's ``svd-ew`` covariance of the states' reduced free energies from the Gram matrix G = W^T W of the
    weights: with G = V Sigma^2 V^T, Theta = V Sigma (I - Sigma V^T diag(n) V Sigma)^+ Sigma V^T (n = 0 for targets)."""
    lam, V = np.linalg.eigh(G)
    A = V * np.sqrt(np.clip(lam, 0.0, None))
    inner = np.eye(G.shape[0]) - A.T @ (np.asarray(n, dtype=np.float64)[:, None] * A)
    return A @ np.linalg.pinv(inner, rcond=1e-10) @ A.T


def differences(th):
    """d(f_j - f_i) = sqrt(Theta_ii + Theta_jj - 2 Theta_ij), [S, S]."""
    dg = np.diag(th)
    return np.sqrt(np.clip(dg[:, None] + dg[None, :] - 2.0 * th, 0.0, None))


def solve(pass_fn, n_rungs, n_per_state, tol=1e-10, max_iter=100):
    """Newton on F(f) = sum L - N sum_k f_k with f_0 = 0.  ``pass_fn(f)`` returns the unpacked sums of one pass at f.
    Returns (f, sums at f, iterations, converged)."""
    R, N = n_rungs, float(n_per_state)
    f = np.zeros(R)
    p = pass_fn(f)
    F = p["sum_l"] - N * f.sum()
    it = 0
    converged = bool(np.max(np.abs(p["s"][:R] - 1.0)) < tol)
    while not converged and it < max_iter:
        it += 1
        s, G = p["s"][:R], p["G"][:R, :R]
        g = N * (s - 1.0)
        H = np.diag(N * s) - N * N * G
        try:
            np.linalg.cholesky(H[1:, 1:])
            newton = True
        except np.linalg.LinAlgError:
            newton = False
        if newton:
            step = np.zeros(R)
            step[1:] = -np.linalg.solve(H[1:, 1:], g[1:])
            gd = float(g[1:] @ step[1:])
            t = 1.0
            while True:                  # Armijo; the slack absorbs the rounding of sum L near the optimum
                ft = f + t * step
                pt = pass_fn(ft)
                Ft = pt["sum_l"] - N * ft.sum()
                if Ft <= F + 1e-4 * t * gd + 1e-12 * max(abs(F), 1.0) or t < 1e-8:
                    break
                t *= 0.5
            f, p, F = ft, pt, Ft
        else:
            f = f - np.log(s)
            f -= f[0]
            p = pass_fn(f)
            F = p["sum_l"] - N * f.sum()
        converged = bool(np.max(np.abs(p["s"][:R] - 1.0)) < tol)
    return f, p, it, converged


class MBARResult:
    """Result of ``MetropolisEngine.mbar()``.

    free_energies       [R] reduced free energies f_r = -ln Z_r of the rungs, f_0 = 0
    free_energy_errors  [R, R] asymptotic standard errors of f_j - f_i (``svd-ew``; uncorrelated samples assumed)
    n_iterations        Newton iterations
    converged           max_r |s_r - 1| < tol was reached
    """

    def __init__(self, engine, f, sums, n_iterations, converged, n_per_state, sample):
        self._engine = engine
        self._sample = sample                 # (burn-in row, stride) of the solve
        self._n = float(n_per_state)
        R = f.size
        self.free_energies = f.copy()
        self.free_energy_errors = differences(theta(sums["G"][:R, :R], np.full(R, self._n)))
        self.n_iterations = int(n_iterations)
        self.converged = bool(converged)

    def evaluate(self, temp=None, consts=None):
        """Free energies and expectations at target states, or at the rungs when both arguments are None.

        temp    one temperature or a sequence (one per target); None: the rungs' own temperatures when consts names
                the targets (temperature ladders and scalar engines use the engine's temperature)
        consts  [K] (every target) or [n_target, K] functor constants; None: the engine's constants (not allowed on a
                Hamiltonian ladder, whose targets must name theirs)

        Returns a dict of numpy arrays over the requested states (Q of them): ``f`` [Q] (reduced, same gauge as
        ``free_energies``), ``df`` [Q] (standard error of f - f_0), ``x_mean`` [Q, D], ``x2_mean`` [Q, D] (parameters
        in the order real, Re c, Im c), ``E_mean`` [Q], ``E2_mean`` [Q] (the energy with the state's constants)."""
        eng = self._engine
        R = self.free_energies.size
        if temp is None and consts is None:
            temps, kt = np.zeros(0), None
        else:
            kt = None if consts is None else np.atleast_2d(np.asarray(consts, dtype=np.float64))
            nt = max(np.size(temp) if temp is not None else 1, 1 if kt is None else kt.shape[0])
            if temp is None:
                if eng.rung_consts is None and np.unique(eng.temperatures).size != 1:
                    raise ValueError("give temp for targets of a temperature ladder")
                temp = eng.temperatures[0]
            temps = np.broadcast_to(np.asarray(temp, dtype=np.float64).ravel(), (nt,)).copy() if np.size(temp) in (1, nt) \
                else None
            if temps is None:
                raise ValueError("temp and consts name different numbers of target states")
            if kt is not None:
                if kt.shape[0] == 1 and nt > 1:
                    kt = np.repeat(kt, nt, axis=0)
                if kt.shape[0] != nt:
                    raise ValueError("temp and consts name different numbers of target states")
        n_t = temps.size
        sums = eng._mbar_sums(self.free_energies, temps, kt, True, *self._sample)
        S, d = R + n_t, eng._d
        s = sums["s"]
        if np.any(~(s > 0)):
            raise RuntimeError("a requested state has no weight on the recorded samples (no overlap)")
        f_all = np.concatenate([self.free_energies, -np.log(s[R:])])
        th = theta(sums["G"], np.concatenate([np.full(R, self._n), np.zeros(n_t)]))
        df_all = differences(th)[0]
        ob = sums["obs"] / s[:, None]
        sel = slice(R, S) if n_t else slice(0, R)
        return dict(f=f_all[sel].copy(), df=df_all[sel].copy(), x_mean=ob[sel, :d].copy(), x2_mean=ob[sel, d:2 * d].copy(),
                    E_mean=ob[sel, 2 * d].copy(), E2_mean=ob[sel, 2 * d + 1].copy())
