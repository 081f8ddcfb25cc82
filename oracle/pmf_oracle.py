"""Host restatement of the free-energy profile contract (DESIGN §3 "MBAR free-energy profiles") on numpy arrays of
samples, beside oracle/mbar_oracle.py (whose pass and Theta it uses).

Checker code only: the product computes the same quantities with the histogram pass (csrc/me_mbar.cuh, k_mbar_hist) and
``metropolisengine_b200/mbar.py``.  Written from the contract:

    w_nt = exp(-u_t(x_n) - L_n), w_nk = exp(f_k - u_k(x_n) - L_n)
    bin i = floor((c - lo) * inv_w), inv_w = n / (hi - lo), in range iff lo <= c < hi, i = n -> n - 1; b = i_0 n_1 + i_1
    h_b = sum w_nt, q_b = sum w_nt^2, c_bk = sum w_nt w_nk over the samples of bin b; w_out over the samples outside
    f_b = -ln h_b - f_ref; df_b from Theta over [rungs, non-empty bins]: G_bk = c_bk / h_b, G_bb = q_b / h_b^2, N_b = 0
"""
import numpy as np

from oracle.mbar_oracle import df, pass_sums, theta

# ---------------------------------------------------------------------------------------- free-energy profiles
def coordinate(x, kind, j, nr, nc):
    """Axis value of samples x [n, D]: stored column j (kind 0) or |c_j| = sqrt(Re c_j^2 + Im c_j^2) (kind 1), each
    product and the sum rounded once, as IEEE FP64 without contraction."""
    x = np.asarray(x, dtype=np.float64)
    if kind == 0:
        return x[:, j].copy()
    re, im = x[:, nr + j], x[:, nr + nc + j]
    return np.sqrt(re * re + im * im)


def bin_index(c, lo, hi, n):
    """i = floor((c - lo) * inv_w) with inv_w = n / (hi - lo); -1 outside [lo, hi) (NaN too); i = n becomes n - 1."""
    inv_w = n / (hi - lo)
    with np.errstate(invalid="ignore"):
        inside = (c >= lo) & (c < hi)
        i = np.floor((c - lo) * inv_w)
    return np.where(inside, np.minimum(np.where(inside, i, 0), n - 1), -1).astype(np.int64)


def hist_sums(u, f, n_per, n_rungs, coords, lo, hi, n_bins):
    """u [R + 1, n] reduced potentials (rungs, then the target), coords: one array [n] per axis.  Returns w_out, n_out
    and per flat bin b = i_0 n_1 + i_1: h [B] = sum w_nt, q [B] = sum w_nt^2, c [B, R] = sum w_nt w_nk."""
    R = n_rungs
    W = pass_sums(u, f, n_per, R)["W"]
    wt = W[:, R]
    b = np.zeros(wt.size, dtype=np.int64)
    out = np.zeros(wt.size, dtype=bool)
    for c, a, z, n in zip(coords, lo, hi, n_bins):
        i = bin_index(c, a, z, n)
        out |= i < 0
        b = b * n + np.maximum(i, 0)
    B = int(np.prod(n_bins))
    inb = ~out
    h = np.bincount(b[inb], weights=wt[inb], minlength=B)
    q = np.bincount(b[inb], weights=wt[inb] ** 2, minlength=B)
    cc = np.stack([np.bincount(b[inb], weights=wt[inb] * W[inb, k], minlength=B) for k in range(R)], axis=1)
    return dict(w_out=float(wt[out].sum()), n_out=int(out.sum()), h=h, q=q, c=cc, bins=np.where(out, -1, b))


def pmf(h, q, c, w_out, G, n_per, reference="lowest"):
    """Histogram FES: f_b = -ln h_b - f_ref; p_b = h_b / (sum h + w_out); df_b from Theta over [rungs, non-empty bins]
    with G_bk = c_bk / h_b, G_bb = q_b / h_b^2, N = [N_k, 0].  Returns f, df, p (empty bins: inf, nan)."""
    R = G.shape[0]
    idx = np.flatnonzero(h > 0)
    f = np.full(h.size, np.inf)
    f[idx] = -np.log(h[idx])
    ref = idx[np.argmin(f[idx])] if reference == "lowest" else int(reference)
    if h[ref] <= 0:
        raise ValueError("empty reference bin")
    m = idx.size
    Ga = np.block([[G, (c[idx] / h[idx, None]).T], [c[idx] / h[idx, None], np.diag(q[idx] / h[idx] ** 2)]])
    th = theta(Ga, np.concatenate([np.full(R, float(n_per)), np.zeros(m)]))
    r = R + int(np.flatnonzero(idx == ref)[0])
    df_ = np.full(h.size, np.nan)
    for k, b in enumerate(idx):
        df_[b] = df(th, R + k, r)
    return f - f[ref], df_, h / (h.sum() + w_out)
