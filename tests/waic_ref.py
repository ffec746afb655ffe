"""float64 numpy reference of bmm_mcmc_b200.waic(), written from the definitions (Watanabe 2010; Vehtari, Gelman &
Gabry 2017, as R's loo::waic).  For draw (c, s) of C chains x S draws and observation i:

    l[c,s,i] = log sum_k pi_k prod_d theta_kd^x_id (1 - theta_kd)^(1 - x_id)

loglik[c, s] = sum_i l; lppd_i = log mean exp l over the D = C S draws; p_waic_i = var(l, ddof=1) over the draws; the
per-chain totals use chain c's S draws alone."""
import numpy as np
from scipy.special import logsumexp


def loglik_matrix(theta, pi, X):
    """l[g, i] for draws g of theta (K x P x S) and pi (S x K): an S x N matrix."""
    X = np.asarray(X, dtype=np.float64)
    th = np.asarray(theta, dtype=np.float64).transpose(2, 0, 1)          # S x K x P
    with np.errstate(divide="ignore", invalid="ignore"):
        l1, l0 = np.log(th), np.log1p(-th)
        lp = np.log(np.asarray(pi, dtype=np.float64))                    # S x K
    # x log theta + (1 - x) log(1 - theta), with 0 * (-inf) read as 0 (the term is absent for that x)
    a = np.einsum("ip,skp->sik", X, np.where(np.isfinite(l1), l1, 0.0))
    a += np.einsum("ip,skp->sik", 1.0 - X, np.where(np.isfinite(l0), l0, 0.0))
    bad1 = np.einsum("ip,skp->sik", X, ~np.isfinite(l1)) > 0
    bad0 = np.einsum("ip,skp->sik", 1.0 - X, ~np.isfinite(l0)) > 0
    a = np.where(bad1 | bad0, -np.inf, a) + lp[:, None, :]
    return logsumexp(a, axis=2)                                           # S x N


def waic_ref(fit, X):
    th, pi = np.asarray(fit["theta"], dtype=np.float64), np.asarray(fit["pi"], dtype=np.float64)
    chains = th.ndim == 4
    if not chains:
        th, pi = th[None], pi[None]
    Cn, K, P, S = th.shape
    L = np.stack([loglik_matrix(th[c], pi[c], X) for c in range(Cn)])    # C x S x N
    D = Cn * S
    flat = L.reshape(D, -1)
    with np.errstate(invalid="ignore"):
        lppd = logsumexp(flat, axis=0) - np.log(D)
        pw = np.var(flat, axis=0, ddof=1)
        clppd = (logsumexp(L, axis=1) - np.log(S)).sum(axis=1)
        cpw = np.var(L, axis=1, ddof=1).sum(axis=1) if S > 1 else np.full(Cn, np.nan)
    elpd = lppd - pw
    N = flat.shape[1]
    out = {"pointwise_lppd": lppd, "pointwise_p_waic": pw, "pointwise_elpd_waic": elpd, "pointwise_waic": -2 * elpd}
    for name in ("lppd", "p_waic", "elpd_waic", "waic"):
        v = out["pointwise_" + name]
        out[name] = v.sum()
        out["se_" + name] = np.sqrt(N * np.var(v, ddof=1)) if N > 1 else np.nan
    out["loglik"] = L.sum(axis=2) if chains else L.sum(axis=2)[0]
    if chains:
        out["chain_elpd_waic"] = clppd - cpw
        out["chain_waic"] = -2 * (clppd - cpw)
        out["chain_p_waic"] = cpw
    return out
