"""The float64 PSIS-LOO reference (tests/loo_ref.py) against scipy, hand-worked cases and an exact leave-one-out
predictive, and loo() / loglik_matrix()'s host-side checks.  No GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats
from scipy.special import logsumexp

import bmm_mcmc_b200 as B
from bmm_mcmc_b200 import _lib
from conftest import ROOT, gpu_available
from loo_ref import gpdfit, loo_matrix, loo_ref, n_pareto_tail, qgpd

LOO_KEYS = ("pointwise_elpd_loo", "pointwise_lpd", "pointwise_p_loo", "pointwise_looic", "pareto_k", "n_eff")


def build_rhost_loo(out_dir):
    """r-package/src/host.cpp + tests/rhost/loo_driver.cpp against the Rcpp stand-in, linked with libbmm_b200.so."""
    _lib.lib()      # libbmm_b200.so must exist
    so = os.path.join(str(out_dir), "librhost_loo.so")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", os.path.join(ROOT, "oracle", "shim"),
                           "-I", os.path.join(ROOT, "oracle"), "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "rhost", "loo_driver.cpp"), "-o", so,
                           "-L", os.path.join(ROOT, "bmm_mcmc_b200"), "-l:libbmm_b200.so",
                           "-Wl,-rpath," + os.path.join(ROOT, "bmm_mcmc_b200")])
    L = C.CDLL(so)
    L.rhost_loo_last_error.restype = C.c_char_p
    L.rhost_loo.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 7
    L.rhost_loglik.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 3
    return L


def _fit(rng, K, P, S, chains=None):
    shp = (K, P, S) if chains is None else (chains, K, P, S)
    return {"theta": rng.uniform(0.05, 0.95, shp), "pi": rng.dirichlet(np.ones(K), S if chains is None else (chains, S))}


def test_qgpd_is_scipy_genpareto_ppf():
    p = (np.arange(1, 101) - 0.5) / 100
    for k, sigma in [(-0.4, 0.7), (0.1, 2.0), (0.5, 1.3), (0.9, 0.05), (1e-6, 1.0)]:
        np.testing.assert_allclose(qgpd(p, k, sigma), stats.genpareto.ppf(p, c=k, scale=sigma), rtol=1e-12, atol=0)
    assert np.isnan(qgpd(p, 0.3, 0.0)).all() and np.isnan(qgpd(p, 0.3, -1.0)).all() and np.isnan(qgpd(p, 0.3, np.nan)).all()


@pytest.mark.parametrize("k", [-0.2, 0.1, 0.5, 0.9])
def test_gpdfit_recovers_the_shape(k):
    x = stats.genpareto.rvs(c=k, scale=1.5, size=100_000, random_state=np.random.default_rng(int(100 * (k + 1))))
    khat, sigma = gpdfit(x)
    assert abs(khat - k) < 0.02, (k, khat)
    assert sigma == pytest.approx(1.5, rel=0.05)


def test_n_pareto_tail():
    assert n_pareto_tail(100, 1.0) == 20 and n_pareto_tail(800, 1.0) == 85 and n_pareto_tail(1_843_200, 1.0) == 4073
    assert n_pareto_tail(20, 1.0) == 4 and n_pareto_tail(21, 1.0) == 5 and n_pareto_tail(1000, 0.25) == 190


def test_no_smoothing_below_21_draws_by_hand():
    rng = np.random.default_rng(0)
    L = np.log(rng.uniform(0.05, 0.9, (20, 7)))
    r = loo_matrix(L)
    assert np.all(np.isinf(r["pareto_k"]))
    np.testing.assert_allclose(r["pointwise_elpd_loo"], -np.log(np.mean(np.exp(-L), axis=0)), rtol=1e-14)
    np.testing.assert_allclose(r["pointwise_lpd"], np.log(np.mean(np.exp(L), axis=0)), rtol=1e-14)
    w = np.exp(-L) / np.exp(-L).sum(0)
    np.testing.assert_allclose(r["n_eff"], 1 / (w ** 2).sum(0), rtol=1e-12)
    assert r["n_k_very_bad"] == 7 and r["n_k_good"] == 0


def test_identical_draws():
    L = np.tile(np.log(np.random.default_rng(1).uniform(0.1, 0.9, 6)), (400, 1))
    r = loo_matrix(L)
    assert np.all(np.isinf(r["pareto_k"]))
    np.testing.assert_allclose(r["pointwise_p_loo"], 0.0, atol=1e-13)
    np.testing.assert_allclose(r["pointwise_elpd_loo"], r["pointwise_lpd"], rtol=1e-13)
    np.testing.assert_allclose(r["n_eff"], 400, rtol=1e-12)


def test_permutation_and_ties_at_the_cutoff_change_nothing():
    rng = np.random.default_rng(2)
    D = 500                                             # M = 67 at r_eff = 1
    L = np.log(rng.uniform(0.02, 0.9, (D, 5)))
    order = np.argsort(-L[:, 1])                        # column 1: ties straddling the cutoff
    L[order[60:75], 1] = L[order[67], 1]
    L[order[:10], 2] = L[order[0], 2]                   # column 2: ties at the top of the tail
    base = loo_matrix(L, r_eff=1.0)
    for seed in range(3):
        p = np.random.default_rng(seed).permutation(D)
        r = loo_matrix(L[p], r_eff=1.0)
        for k in LOO_KEYS:
            np.testing.assert_allclose(r[k], base[k], rtol=1e-13, atol=0, err_msg=k)
    assert np.isfinite(base["pareto_k"]).all()


def test_beta_bernoulli_exact_leave_one_out():
    # K = 1, P independent Bernoulli(theta_d), theta_d ~ Beta(1, 1): exact posterior draws; p(x_i | x_-i) is analytic
    rng = np.random.default_rng(3)
    N, P, S = 40, 3, 4000
    X = (rng.uniform(size=(N, P)) < [0.3, 0.6, 0.8]).astype(np.int32)
    n1 = X.sum(0)
    th = rng.beta(1 + n1, 1 + N - n1, size=(S, P)).T[None]           # 1 x P x S
    fit = {"theta": th, "pi": np.ones((S, 1))}
    r = loo_ref(fit, X)
    exact = np.log(np.where(X == 1, n1, N - n1) / (N + 1)).sum(1)
    # MC standard error of the self-normalised importance-sampling estimate of p(x_i | x_-i)
    from waic_ref import loglik_matrix
    L = loglik_matrix(th, np.ones((S, 1)), X)
    w = np.exp(-L - logsumexp(-L, axis=0))
    pr = np.exp(L)
    phat = (w * pr).sum(0)
    se = np.sqrt((w ** 2 * (pr - phat) ** 2).sum(0)) / phat
    assert np.all(np.abs(r["pointwise_elpd_loo"] - exact) < 4 * se), np.abs(r["pointwise_elpd_loo"] - exact) / se
    assert np.all(r["pareto_k"] < 0.5), r["pareto_k"].max()
    assert r["n_k_good"] == N and r["k_threshold"] == 0.7


def test_loo_rejects_bad_input_before_the_library():
    rng = np.random.default_rng(4)
    X = rng.integers(0, 2, (20, 5))
    f = _fit(rng, 2, 5, 30)
    for call in (B.loo, B.loglik_matrix):
        with pytest.raises(ValueError, match="pi"):
            call({"theta": f["theta"]}, X)
        with pytest.raises(ValueError):
            call(f, X[:, :4])
        with pytest.raises(ValueError):
            call({"theta": f["theta"], "pi": f["pi"][:3]}, X)
        with pytest.raises(ValueError, match="2 draws"):
            call({"theta": f["theta"][:, :, :1], "pi": f["pi"][:1]}, X)
    for bad in (np.ones(19), np.ones((20, 1)), 0.0, -1.0, np.nan, np.inf, np.r_[np.ones(19), 0.0]):
        with pytest.raises(ValueError, match="r_eff"):
            B.loo(f, X, r_eff=bad)


def test_bmm_loo_is_exported_and_needs_a_device():
    L = _lib.lib()
    for name in ("bmm_loo", "bmm_loo_kernel_ms", "bmm_loglik_matrix"):
        assert name in _lib.EXPORTS and hasattr(L, name)
    if gpu_available():
        pytest.skip("only meaningful on a box without a GPU")
    rng = np.random.default_rng(5)
    X = rng.integers(0, 2, (10, 3))
    f = _fit(rng, 2, 3, 30)
    with pytest.raises(_lib.BmmError, match="CUDA"):
        B.loo(f, X)
    with pytest.raises(_lib.BmmError, match="CUDA"):
        B.loglik_matrix(f, X)
    # argument errors are reported before the device check
    Xc = np.asfortranarray(X, dtype=np.int32)
    th, pi, out = np.full(2 * 3 * 30, 0.5), np.full(30 * 2, 0.5), np.zeros(10)
    d = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    args = lambda S, re: (C.c_void_p(Xc.ctypes.data), 10, 3, 2, S, 1, d(th), d(pi), re, 0, 0, d(out), None, None, None)
    assert L.bmm_loo(*args(30, None)) == -2 and b"CUDA" in L.bmm_last_error()
    assert L.bmm_loo(*args(1, None)) == -1
    assert L.bmm_loo(*args(30, d(np.r_[np.ones(9), -1.0]))) == -1 and b"r_eff" in L.bmm_last_error()
    # a Pareto tail longer than the fit kernel's shared memory holds is refused, not computed some other way
    big = (C.c_void_p(Xc.ctypes.data), 10, 3, 2, 1, 30_000_000, d(th), d(pi), None, 0, 0, d(out), None, None, None)
    assert L.bmm_loo(*big) == -1 and b"at most 16384" in L.bmm_last_error()


def test_rcpp_host_loo_builds_and_reports_the_missing_device(tmp_path):
    L = build_rhost_loo(tmp_path)
    if gpu_available():
        pytest.skip("only meaningful on a box without a GPU")
    X = np.asfortranarray(np.random.default_rng(6).integers(0, 2, (10, 3)), dtype=np.int32)
    th, pi = np.full(2 * 3 * 30, 0.5), np.full(30 * 2, 0.5)
    re, est, pw, k, ne, ll = np.ones(10), np.zeros(6), np.zeros(40), np.zeros(10), np.zeros(10), np.zeros(300)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert L.rhost_loo(p(X), 10, 3, 2, 30, p(th), p(pi), p(re), p(est), p(pw), p(k), p(ne)) == -1
    assert b"CUDA" in L.rhost_loo_last_error()
    assert L.rhost_loglik(p(X), 10, 3, 2, 30, p(th), p(pi), p(ll)) == -1
    assert b"CUDA" in L.rhost_loo_last_error()
