"""Host restatement of the expectation-uncertainty contract (DESIGN §3 "Uncertainties of reweighted expectations") on
numpy arrays of samples, beside oracle/mbar_oracle.py (whose pass it uses).

Checker code only: the product computes the same quantities with the covariance pass (csrc/me_mbar.cuh, k_mbar_cov) and
``metropolisengine_b200/mbar.py``.  Written from the contract and from pymbar's compute_expectations:

    a~ = a_s - c_s,  o_a = sum w_ns a~_a,  C_ak = sum w_ns a~_a w_nk (k < R),  C_a* = sum w_ns^2 a~_a,
    Q_ab = sum w_ns^2 a~_a a~_b
    pymbar: one column per observable, A shifted by (min - 1) so that it is positive, weights w_ns A_n normalised to sum
    1; Theta by the SVD of the explicit weight matrix; Cov(A_i, A_j) = <A_i> <A_j> (Theta_ij - Theta_is - Theta_sj
    + Theta_ss)
"""
import numpy as np

from oracle.mbar_oracle import pass_sums


def cov_sums(u, f, n_per, n_rungs, obs, first, count, centers):
    """u [S, n] reduced potentials (rungs first), obs [S, n, m] per-state observables, centres [count, m] of the states
    [first, first + count).  Returns o [count, m], C [count, m, R + 1], Q [count, m, m]."""
    R = n_rungs
    W = pass_sums(u, f, n_per, R)["W"]
    o, C, Q = [], [], []
    for c in range(count):
        s = first + c
        at = obs[s] - np.asarray(centers[c], dtype=np.float64)[None, :]
        wa = W[:, s:s + 1] * at
        o.append(wa.sum(axis=0))
        C.append(np.concatenate([wa.T @ W[:, :R], (wa.T @ W[:, s])[:, None]], axis=1))
        Q.append(wa.T @ wa)
    return np.array(o), np.array(C), np.array(Q)


def _svd_theta(W, n):
    """pymbar's svd-ew on the explicit weight matrix W [N, K]: W = U Sigma V^T,
    Theta = V Sigma (I - Sigma V^T diag(n) V Sigma)^+ Sigma V^T."""
    _, sig, vt = np.linalg.svd(W, full_matrices=False)
    V = vt.T
    inner = np.eye(sig.size) - np.diag(sig) @ V.T @ np.diag(n) @ V @ np.diag(sig)
    return V @ np.diag(sig) @ np.linalg.pinv(inner, rcond=1e-10) @ np.diag(sig) @ V.T


def pymbar_expectations(u, f, n_per, n_rungs, obs, states):
    """pymbar's compute_expectations route for every state in ``states``: the explicit N x (S + m) weight matrix of
    log-weights [rungs, the other states normalised, one normalised column per shifted observable of the state], Theta
    by SVD, and covA.  Returns means [Q, m] and covariances [Q, m, m]."""
    R = n_rungs
    W = pass_sums(u, f, n_per, R)["W"]
    with np.errstate(divide="ignore"):
        logW = np.log(W)
    means, covs = [], []
    for s in states:
        A = obs[s]
        m = A.shape[1]
        shift = A.min(axis=0) - 1.0
        As = A - shift[None, :]
        logs = logW[:, s] - np.log(np.exp(logW[:, s]).sum())          # the state's column, normalised
        cols = [logW[:, k] for k in range(R)] + [logs]
        for a in range(m):
            la = logs + np.log(As[:, a])
            cols.append(la - np.log(np.exp(la).sum()))
        Wx = np.exp(np.stack(cols, axis=1))
        th = _svd_theta(Wx, np.concatenate([np.full(R, float(n_per)), np.zeros(1 + m)]))
        mA = np.exp(logs) @ As                                          # shifted means
        i0 = R + 1
        cov = np.empty((m, m))
        for i in range(m):
            for j in range(m):
                cov[i, j] = mA[i] * mA[j] * (th[i0 + i, i0 + j] - th[i0 + i, R] - th[R, i0 + j] + th[R, R])
        means.append(mA + shift)
        covs.append(cov)
    return np.array(means), np.array(covs)


def heat_capacity(E, E2, cov_ee, T):
    """C = (<E^2> - <E>^2) / T^2 and its delta-method error from the (E, E^2) covariance block."""
    g = np.array([-2.0 * E, 1.0]) / T ** 2
    return (E2 - E * E) / T ** 2, float(np.sqrt(max(g @ cov_ee @ g, 0.0)))
