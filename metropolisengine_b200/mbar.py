"""MBAR over the recorded rows of a ladder: free energies between rungs, reweighted expectations and their asymptotic
uncertainties (Shirts & Chodera, J. Chem. Phys. 129, 124105, 2008; pymbar's ``MBAR``).

The device pass (``me_mbar_pass``, csrc/me_mbar.cuh) reduces every sample to a few FP64 sums for a given vector of rung
free energies f; everything here is S x S algebra on those sums (S <= 32 states):

* the Newton solve of the convex objective F(f) = sum_n L_n - N sum_k f_k in the gauge f_0 = 0, with a backtracking
  line search on F (one pass per trial point) and the self-consistent step f_i <- f_i - ln s_i when the reduced Hessian
  is not positive definite;
* pymbar's ``svd-ew`` asymptotic covariance Theta from the Gram matrix G of the weights;
* target states: f_t = -ln s_t and <a>_t = sum_n w_nt a_t / s_t;
* free-energy profiles (pymbar's histogram FES): the histogram pass (``me_mbar_hist_pass``) sums a target's weights per
  bin of one or two coordinates, and ``profile`` turns them into f_b, p_b and their errors by Theta over the rungs plus
  one state per non-empty bin;
* uncertainties of expectations (pymbar's ``compute_expectations`` covariance): the covariance pass
  (``me_mbar_cov_pass``) sums products of the centred observables with the weights, and ``expectation_covariance``
  turns them into the covariance of a state's means by Theta over the rungs plus one centred column per observable.

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


def unpack_hist(sums, n_rungs, n_bins):
    """The sums vector of ``me_mbar_hist_pass`` as a dict: ``n_nan``, ``n_overflow``, ``w_out``, ``n_out``, and per flat
    bin ``h`` [B], ``q`` [B] and ``c`` [B, R]."""
    R, B = n_rungs, int(np.prod(n_bins))
    sums = np.asarray(sums, dtype=np.float64)
    body = sums[4:4 + B * (R + 2)].reshape(B, R + 2)
    return dict(n_nan=int(sums[0]), n_overflow=int(sums[1]), w_out=float(sums[2]), n_out=int(sums[3]),
                h=body[:, 0].copy(), q=body[:, 1].copy(), c=body[:, 2:].copy())


def profile(h, q, c, w_out, G, n_per_state, reference="lowest"):
    """pymbar's histogram free-energy surface from the per-bin sums of one target (flat bins).

    f_b = -ln h_b, reported as f_b - f_ref; p_b = h_b / (sum h + w_out).  Errors: Theta of the augmented Gram matrix
    over the R rungs (G, the rung Gram matrix at the MBAR solution) and the non-empty bins, G_bk = c_bk / h_b,
    G_bb = q_b / h_b^2, G_bb' = 0, with N = 0 for the bins; df_b = sqrt(Theta_bb + Theta_rr - 2 Theta_br).  reference:
    "lowest" (the bin of smallest f) or a flat bin index.  Empty bins: f = +inf, df = NaN.  Returns (f, df, p)."""
    h, q, c = np.asarray(h, dtype=np.float64), np.asarray(q, dtype=np.float64), np.asarray(c, dtype=np.float64)
    R, B = G.shape[0], h.size
    full = np.flatnonzero(h > 0)
    f = np.full(B, np.inf)
    f[full] = -np.log(h[full])
    p = h / (h.sum() + w_out)
    if isinstance(reference, str):
        if reference != "lowest":
            raise ValueError('reference is "lowest" or a bin index')
        if full.size == 0:
            raise ValueError("every bin is empty: the range holds none of the target's weight")
        ref = int(full[np.argmin(f[full])])
    else:
        ref = int(reference)
        if not 0 <= ref < B:
            raise ValueError("the reference bin lies outside the bins")
        if not h[ref] > 0:
            raise ValueError("the reference bin is empty")
    nb = full.size
    Ga = np.zeros((R + nb, R + nb))
    Ga[:R, :R] = G
    gbk = c[full] / h[full, None]
    Ga[R:, :R] = gbk
    Ga[:R, R:] = gbk.T
    Ga[np.arange(R, R + nb), np.arange(R, R + nb)] = q[full] / (h[full] * h[full])
    th = theta(Ga, np.concatenate([np.full(R, float(n_per_state)), np.zeros(nb)]))
    j = R + int(np.searchsorted(full, ref))
    df = np.full(B, np.nan)
    df[full] = np.sqrt(np.clip(np.diag(th)[R:] + th[j, j] - 2.0 * th[R:, j], 0.0, None))
    return f - f[ref], df, p


def unpack_cov(sums, n_cov, m, n_rungs):
    """The sums vector of ``me_mbar_cov_pass`` as a dict: ``n_nan``, ``n_overflow``, and per covered state ``o`` [n, m]
    (sum w a~), ``C`` [n, m, R + 1] (sum w a~ w_k, then the self column sum w^2 a~) and ``Q`` [n, m, m] (sum w^2 a~ a~,
    symmetric)."""
    sums = np.asarray(sums, dtype=np.float64)
    R, p = n_rungs, m * (m + 1) // 2
    body = sums[2:2 + n_cov * (m + m * (R + 1) + p)].reshape(n_cov, -1)
    Q = np.zeros((n_cov, m, m))
    Q[:, np.tril_indices(m)[0], np.tril_indices(m)[1]] = body[:, m + m * (R + 1):]
    Q = Q + np.tril(Q, -1).transpose(0, 2, 1)
    return dict(n_nan=int(sums[0]), n_overflow=int(sums[1]), o=body[:, :m].copy(),
                C=body[:, m:m + m * (R + 1)].reshape(n_cov, m, R + 1), Q=Q)


def expectation_covariance(G, s, state, o, C, Q, n_per_state):
    """Covariance [m, m] of the means <a>_s of one state from its covariance sums (o [m], C [m, R + 1], Q [m, m], about
    any centres) and the plain pass's s [S] and G [S, S] (R = C.shape[1] - 1 rungs first) at the same f.

    delta = o / s_s; the centred column v_a = w_s (a - <a>_s) / s_s has G(v_a, k) = (C_ak - delta_a G_sk) / s_s and
    G(v_a, v_b) = (Q_ab - delta_a C_b* - delta_b C_a* + delta_a delta_b G_ss) / s_s^2; Theta over [rungs, v] with
    N = [N .. N, 0 .. 0] gives Cov(<a>_s, <b>_s) = Theta(v_a, v_b).  This is pymbar's compute_expectations covariance
    A_i A_j (Theta_AiAj - Theta_Ai,s - Theta_s,Aj + Theta_ss) with its shifted, normalised columns A: Theta is bilinear
    in the columns."""
    R, m = C.shape[1] - 1, o.size
    ss = s[state]
    d = o / ss
    gvk = (C[:, :R] - d[:, None] * G[state, :R][None, :]) / ss
    cs = C[:, R]
    gvv = (Q - np.outer(d, cs) - np.outer(cs, d) + np.outer(d, d) * G[state, state]) / (ss * ss)
    Ga = np.block([[G[:R, :R], gvk.T], [gvk, gvv]])
    th = theta(Ga, np.concatenate([np.full(R, float(n_per_state)), np.zeros(m)]))
    return th[R:, R:]


def heat_capacity(E, E2, cov, T):
    """C = (<E^2> - <E>^2) / T^2 (k_B = 1) and its standard error by the delta method over the (E, E^2) block cov
    [..., 2, 2] of the means, gradient [-2 <E>, 1] / T^2."""
    E, E2, T = np.asarray(E, dtype=np.float64), np.asarray(E2, dtype=np.float64), np.asarray(T, dtype=np.float64)
    g = np.stack([-2.0 * E, np.ones_like(E)], axis=-1) / (T * T)[..., None]
    var = np.einsum("...i,...ij,...j->...", g, cov, g)
    return (E2 - E * E) / (T * T), np.sqrt(np.clip(var, 0.0, None))


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
        self._G = sums["G"][:R, :R].copy()    # rung Gram matrix at the solution (profile errors)
        self.free_energies = f.copy()
        self.free_energy_errors = differences(theta(sums["G"][:R, :R], np.full(R, self._n)))
        self.n_iterations = int(n_iterations)
        self.converged = bool(converged)

    def evaluate(self, temp=None, consts=None, uncertainty=False):
        """Free energies and expectations at target states, or at the rungs when both arguments are None.

        temp    one temperature or a sequence (one per target); None: the rungs' own temperatures when consts names
                the targets (temperature ladders and scalar engines use the engine's temperature)
        consts  [K] (every target) or [n_target, K] functor constants; None: the engine's constants (not allowed on a
                Hamiltonian ladder, whose targets must name theirs)

        Returns a dict of numpy arrays over the requested states (Q of them): ``f`` [Q] (reduced, same gauge as
        ``free_energies``), ``df`` [Q] (standard error of f - f_0), ``x_mean`` [Q, D], ``x2_mean`` [Q, D] (parameters
        in the order real, Re c, Im c), ``E_mean`` [Q], ``E2_mean`` [Q] (the energy with the state's constants).

        uncertainty=True adds the errors of the means (pymbar's compute_expectations covariance) from device covariance
        passes over the same rows, as many as the shared-memory bound needs; the keys above are the same bits as
        without it.  Added: ``dx_mean`` [Q, D], ``dx2_mean`` [Q, D], ``dE_mean`` [Q], ``dE2_mean`` [Q] (standard
        errors), ``obs_cov`` [Q, m, m] (covariance of the m = 2D + 2 means in the order x, x^2, E, E^2), and
        ``heat_capacity`` [Q] = (<E^2> - <E>^2) / T^2 (k_B = 1, the functor's energy units) with ``dheat_capacity``
        [Q] (delta method).  Like ``df`` these errors assume uncorrelated samples: they are only as good as the
        ``stride`` of ``MetropolisEngine.mbar`` (about the statistical inefficiency of the energy column)."""
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
        out = dict(f=f_all[sel].copy(), df=df_all[sel].copy(), x_mean=ob[sel, :d].copy(), x2_mean=ob[sel, d:2 * d].copy(),
                   E_mean=ob[sel, 2 * d].copy(), E2_mean=ob[sel, 2 * d + 1].copy())
        if not uncertainty:
            return out
        first, q = (R, n_t) if n_t else (0, R)
        cs = eng._mbar_cov_sums(self.free_energies, temps, kt, first, q, ob[sel], *self._sample)
        cov = np.stack([expectation_covariance(sums["G"], s, first + i, cs["o"][i], cs["C"][i], cs["Q"][i], self._n)
                        for i in range(q)])
        se = np.sqrt(np.clip(np.diagonal(cov, axis1=1, axis2=2), 0.0, None))
        t_states = temps if n_t else np.broadcast_to(np.asarray(eng.temperatures, dtype=np.float64), (R,))
        c, dc = heat_capacity(out["E_mean"], out["E2_mean"], cov[:, 2 * d:, 2 * d:], t_states)
        out.update(dx_mean=se[:, :d].copy(), dx2_mean=se[:, d:2 * d].copy(), dE_mean=se[:, 2 * d].copy(),
                   dE2_mean=se[:, 2 * d + 1].copy(), obs_cov=cov, heat_capacity=c, dheat_capacity=dc)
        return out

    def pmf(self, coords, bins, range, temp=None, consts=None, reference="lowest"):
        """Free-energy profile of one target state along one or two coordinates (pymbar's histogram FES), from a device
        histogram pass over the rows of the solve.

        coords     an int (stored parameter column, order real, Re c, Im c), ("abs", j) (the modulus of complex
                   parameter j), or a pair of those for a 2-D profile
        bins       an int, or a pair (one per axis)
        range      (lo, hi), or a pair of those; a sample counts iff lo <= c < hi on every axis
        temp, consts  the target state, with the rules of ``evaluate``: consts is one [K] vector; both None: rung 0 (its
                   temperature, and its constants on a Hamiltonian ladder)
        reference  "lowest" (the bin of smallest f, pymbar's from-lowest) or a bin index (a pair in 2-D)

        Returns a dict of numpy arrays: ``f`` and ``df`` shaped [n] or [n_x, n_y] (reduced free energy against the
        reference bin and its standard error; empty bins: f = +inf, df = NaN), ``p`` (bin probabilities), ``edges``
        (one array per axis) and ``weight_outside`` (the target's probability outside the range)."""
        eng = self._engine
        one = isinstance(coords, (int, np.integer)) or (isinstance(coords, (tuple, list)) and len(coords) == 2
                                                        and isinstance(coords[0], str))
        axes = [coords] if one else list(coords)
        if not 1 <= len(axes) <= 2:
            raise ValueError("coords names one or two axes")
        n_ax = len(axes)
        kinds, idx = [], []
        for a in axes:
            if isinstance(a, (int, np.integer)) and not isinstance(a, bool):
                kinds.append(0)
                idx.append(int(a))
            elif isinstance(a, (tuple, list)) and len(a) == 2 and a[0] == "abs" and isinstance(a[1], (int, np.integer)):
                kinds.append(1)
                idx.append(int(a[1]))
            else:
                raise ValueError('a coordinate is a column index or ("abs", j), got %r' % (a,))
        nb = [bins] if n_ax == 1 and np.ndim(bins) == 0 else list(np.ravel(bins))
        rg = np.asarray(range, dtype=np.float64)
        rg = rg.reshape(1, -1) if n_ax == 1 and rg.ndim == 1 else rg
        if len(nb) != n_ax or rg.shape != (n_ax, 2):
            raise ValueError("bins and range need one entry per axis")
        if any(not isinstance(n, (int, np.integer)) or isinstance(n, bool) for n in nb):
            raise ValueError("bins are integers")
        nb = [int(n) for n in nb]
        if temp is None and consts is None:
            temp = eng.temperatures[0]
            kt = None if eng.rung_consts is None else eng.rung_consts[0]
        else:
            if temp is None:
                if eng.rung_consts is None and np.unique(eng.temperatures).size != 1:
                    raise ValueError("give temp for the target of a temperature ladder")
                temp = eng.temperatures[0]
            kt = None if consts is None else np.asarray(consts, dtype=np.float64)
        if np.size(temp) != 1 or (kt is not None and kt.ndim != 1):
            raise ValueError("pmf takes one target state: a scalar temp and one [K] constant vector")
        sums = eng._mbar_hist_sums(self.free_energies, float(np.asarray(temp).ravel()[0]), kt, kinds, idx, rg[:, 0],
                                   rg[:, 1], nb, *self._sample)
        if isinstance(reference, str):
            ref = reference
        else:
            r = np.ravel(reference)
            if r.size != n_ax or np.any(r < 0) or np.any(r >= np.array(nb)):
                raise ValueError("the reference bin lies outside the bins")
            ref = int(np.ravel_multi_index(tuple(int(v) for v in r), nb))
        f, df, p = profile(sums["h"], sums["q"], sums["c"], sums["w_out"], self._G, self._n, ref)
        shape = tuple(nb)
        return dict(f=f.reshape(shape), df=df.reshape(shape), p=p.reshape(shape),
                    edges=[np.linspace(rg[a, 0], rg[a, 1], nb[a] + 1) for a in np.arange(n_ax)],
                    weight_outside=sums["w_out"] / (sums["h"].sum() + sums["w_out"]))
