"""float64 numpy reference of bmm_mcmc_b200.loo(): Pareto-smoothed importance-sampling leave-one-out cross-validation
(Vehtari, Gelman & Gabry 2017; Vehtari, Simpson, Gelman, Yao & Gabry 2024), transcribed from R's loo package
(R/psis.R, R/gpdfit.R, R/loo.R) with its function names, so each can be checked against the R source line by line.

For observation i with log-likelihood values l_g over the D = C S pooled draws, the raw log importance ratios are
r_g = -l_g.  PSIS smooths the largest M = n_pareto_tail(D, r_eff) of them with a generalized Pareto fit (Zhang &
Stephens 2009), truncates at the largest raw ratio and normalises; elpd_loo_i = logsumexp(w~ + l)."""
import numpy as np
from scipy.special import logsumexp

from waic_ref import loglik_matrix

DOUBLE_EPS = np.finfo(np.float64).eps        # R's .Machine$double.eps


def n_pareto_tail(S, r_eff):
    """psis.R: min(ceiling(0.2 * S), ceiling(3 * sqrt(S / r_eff)))."""
    return int(min(np.ceil(0.2 * S), np.ceil(3 * np.sqrt(S / r_eff))))


def enough_tail_samples(tail_len, min_len=5):
    return tail_len >= min_len


def qgpd(p, k, sigma):
    """gpdfit.R: quantile function of the generalized Pareto distribution (location 0)."""
    if np.isnan(sigma) or sigma <= 0:
        return np.full(np.shape(p), np.nan)
    return sigma * np.expm1(-k * np.log1p(-p)) / k


def lx(a, x):
    """gpdfit.R: profile log-likelihood per observation at theta = a (a vector)."""
    a = -a
    k = np.array([np.mean(np.log1p(ai * x)) for ai in a])
    return np.log(a / k) - k - 1


def adjust_k_wip(k, n):
    a = 10
    n_plus_a = n + a
    return k * n / n_plus_a + a * 0.5 / n_plus_a


def gpdfit(x, wip=True, min_grid_pts=30, sort_x=True):
    """gpdfit.R (section 4 of Zhang & Stephens 2009): returns (k, sigma)."""
    x = np.asarray(x, dtype=np.float64)
    if sort_x:
        x = np.sort(x)
    N = len(x)
    prior = 3
    M = min_grid_pts + int(np.floor(np.sqrt(N)))
    jj = np.arange(1, M + 1, dtype=np.float64)
    xstar = x[int(np.floor(N / 4 + 0.5)) - 1]                  # first quartile of the sample (R is 1-based)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        theta = 1 / x[N - 1] + (1 - np.sqrt(M / (jj - 0.5))) / prior / xstar
        l_theta = N * lx(theta, x)
        w_theta = np.exp(l_theta - logsumexp(l_theta))
        theta_hat = np.sum(theta * w_theta)
        k = np.mean(np.log1p(-theta_hat * x))
        sigma = -k / theta_hat
    if wip:
        k = adjust_k_wip(k, n=N)
    if np.isnan(k):
        k = np.inf
    return k, sigma


def psis_smooth_tail(x, cutoff):
    """psis.R: x is the sorted tail of the log weights, cutoff the value just below it."""
    length = len(x)
    with np.errstate(over="ignore", invalid="ignore"):
        exp_cutoff = np.exp(cutoff)
        k, sigma = gpdfit(np.exp(x) - exp_cutoff, sort_x=False)
        if np.isfinite(k):
            p = (np.arange(1, length + 1) - 0.5) / length
            qq = qgpd(p, k, sigma) + exp_cutoff
            tail = np.log(qq)
        else:
            tail = x
    return tail, k


def do_psis_i(log_ratios_i, tail_len_i):
    """psis.R: the PSIS log weights (unnormalised) and Pareto k of one observation."""
    S = len(log_ratios_i)
    with np.errstate(invalid="ignore"):
        lw_i = log_ratios_i - np.max(log_ratios_i)
    khat = np.inf
    if enough_tail_samples(tail_len_i):
        ix = np.argsort(lw_i, kind="stable")
        xs = lw_i[ix]
        tail_ids = np.arange(S - tail_len_i, S)
        lw_tail = xs[tail_ids]
        with np.errstate(invalid="ignore"):
            flat = abs(np.max(lw_tail) - np.min(lw_tail)) < DOUBLE_EPS / 100
        if not flat:
            cutoff = xs[tail_ids[0] - 1]                       # largest value smaller than the tail values
            smoothed, khat = psis_smooth_tail(lw_tail, cutoff)
            lw_i = lw_i.copy()
            lw_i[ix[tail_ids]] = smoothed
    with np.errstate(invalid="ignore"):
        lw_i = np.where(lw_i > 0, 0.0, lw_i)                   # lw_i[lw_i > 0] <- 0 (NaN stays NaN)
        lw_i = lw_i + np.max(log_ratios_i)
    return lw_i, khat


def pointwise_loo_calcs(ll_i, lw_i, r_eff_i):
    """loo.R: elpd_loo, lpd, p_loo, looic of one observation, with lw_i normalised; and psis_n_eff."""
    with np.errstate(invalid="ignore"):
        lw_i = lw_i - logsumexp(lw_i)
        elpd_loo = logsumexp(ll_i + lw_i)
        lpd = logsumexp(ll_i) - np.log(len(ll_i))
        n_eff = r_eff_i / np.sum(np.exp(2 * lw_i))
    return elpd_loo, lpd, lpd - elpd_loo, -2 * elpd_loo, n_eff


def ps_khat_threshold(S):
    return min(1 - 1 / np.log10(S), 0.7)


def loo_matrix(L, r_eff=1.0):
    """PSIS-LOO of a D x N log-likelihood matrix; r_eff a scalar or N values."""
    L = np.asarray(L, dtype=np.float64)
    D, N = L.shape
    r_eff = np.broadcast_to(np.asarray(r_eff, dtype=np.float64), (N,))
    cols = {n: np.zeros(N) for n in ("elpd_loo", "lpd", "p_loo", "looic", "n_eff", "pareto_k")}
    for i in range(N):
        with np.errstate(invalid="ignore"):
            lw_i, k = do_psis_i(-L[:, i], n_pareto_tail(D, r_eff[i]))
        e, lpd, p, ic, ne = pointwise_loo_calcs(L[:, i], lw_i, r_eff[i])
        for n, v in zip(("elpd_loo", "lpd", "p_loo", "looic", "n_eff", "pareto_k"), (e, lpd, p, ic, ne, k)):
            cols[n][i] = v
    out = {"pointwise_" + n: cols[n] for n in ("elpd_loo", "lpd", "p_loo", "looic")}
    for n in ("elpd_loo", "lpd", "p_loo", "looic"):
        v = cols[n]
        out[n] = v.sum()
        out["se_" + n] = np.sqrt(N * np.var(v, ddof=1)) if N > 1 else np.nan
    out["pareto_k"], out["n_eff"] = cols["pareto_k"], cols["n_eff"]
    thr = ps_khat_threshold(D)
    k = cols["pareto_k"]
    out["k_threshold"] = thr
    out["n_k_good"] = int(np.sum(k <= thr))
    out["n_k_bad"] = int(np.sum((k > thr) & (k <= 1)))
    out["n_k_very_bad"] = int(np.sum(k > 1))
    return out


def loglik_draws(fit, X):
    """The D x N matrix l[g, i] of a fit with or without a chain axis, draws g = c S + s."""
    th, pi = np.asarray(fit["theta"], dtype=np.float64), np.asarray(fit["pi"], dtype=np.float64)
    if th.ndim == 3:
        th, pi = th[None], pi[None]
    return np.concatenate([loglik_matrix(th[c], pi[c], X) for c in range(th.shape[0])], axis=0)


def loo_ref(fit, X, r_eff=1.0):
    return loo_matrix(loglik_draws(fit, X), r_eff)
