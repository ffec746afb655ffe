"""The float64 WAIC reference (tests/waic_ref.py) against hand-worked cases, and waic()'s host-side checks.  No GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.special import logsumexp

import bmm_mcmc_b200 as B
from bmm_mcmc_b200 import _lib
from conftest import ROOT, gpu_available
from waic_ref import loglik_matrix, waic_ref


def build_rhost_waic(out_dir):
    """r-package/src/host.cpp + tests/rhost/waic_driver.cpp against the Rcpp stand-in, linked with libbmm_b200.so."""
    _lib.lib()      # libbmm_b200.so must exist
    so = os.path.join(str(out_dir), "librhost_waic.so")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", os.path.join(ROOT, "oracle", "shim"),
                           "-I", os.path.join(ROOT, "oracle"), "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "rhost", "waic_driver.cpp"), "-o", so,
                           "-L", os.path.join(ROOT, "bmm_mcmc_b200"), "-l:libbmm_b200.so",
                           "-Wl,-rpath," + os.path.join(ROOT, "bmm_mcmc_b200")])
    L = C.CDLL(so)
    L.rhost_waic_last_error.restype = C.c_char_p
    L.rhost_waic.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 5
    return L


def _fit(rng, K, P, S, chains=None):
    shp = (K, P, S) if chains is None else (chains, K, P, S)
    th = rng.uniform(0.05, 0.95, shp)
    pi = rng.dirichlet(np.ones(K), S if chains is None else (chains, S))
    return {"theta": th, "pi": pi}


def test_identical_draws_have_no_effective_parameters():
    rng = np.random.default_rng(0)
    f = _fit(rng, 3, 6, 1)
    f = {"theta": np.repeat(f["theta"], 5, axis=2), "pi": np.repeat(f["pi"], 5, axis=0)}
    X = rng.integers(0, 2, (40, 6))
    r = waic_ref(f, X)
    assert np.all(np.abs(r["pointwise_p_waic"]) < 1e-24)
    assert r["p_waic"] == pytest.approx(0.0, abs=1e-20)
    np.testing.assert_allclose(r["elpd_waic"], r["lppd"], rtol=1e-15)
    np.testing.assert_allclose(r["loglik"], r["lppd"], rtol=1e-13)


def test_one_cluster_is_the_bernoulli_likelihood():
    rng = np.random.default_rng(1)
    P, S = 4, 3
    th = rng.uniform(0.1, 0.9, (1, P, S))
    X = rng.integers(0, 2, (25, P))
    want = np.array([(X * np.log(th[0, :, s]) + (1 - X) * np.log(1 - th[0, :, s])).sum(1) for s in range(S)])
    np.testing.assert_allclose(loglik_matrix(th, np.ones((S, 1)), X), want, rtol=1e-14)
    r = waic_ref({"theta": th, "pi": np.ones((S, 1))}, X)
    np.testing.assert_allclose(r["loglik"], want.sum(1), rtol=1e-14)
    np.testing.assert_allclose(r["pointwise_p_waic"], want.var(0, ddof=1), rtol=1e-12)


def test_two_draws_by_hand():
    # one observation x = (1, 0); draw 1: pi = (0.5, 0.5), theta = (0.8, 0.3 | 0.2, 0.6); draw 2: one cluster of mass 1
    th = np.zeros((2, 2, 2))
    th[:, :, 0] = [[0.8, 0.3], [0.2, 0.6]]
    th[:, :, 1] = [[0.5, 0.5], [0.9, 0.1]]
    pi = np.array([[0.5, 0.5], [1.0, 0.0]])
    p1 = 0.5 * 0.8 * 0.7 + 0.5 * 0.2 * 0.4
    p2 = 0.5 * 0.5
    l = np.log([p1, p2])
    r = waic_ref({"theta": th, "pi": pi}, np.array([[1, 0]]))
    np.testing.assert_allclose(r["loglik"], l, rtol=1e-14)
    assert r["lppd"] == pytest.approx(np.log((p1 + p2) / 2), rel=1e-14)
    assert r["p_waic"] == pytest.approx((l[0] - l[1]) ** 2 / 2, rel=1e-13)
    assert r["waic"] == pytest.approx(-2 * (np.log((p1 + p2) / 2) - (l[0] - l[1]) ** 2 / 2), rel=1e-13)


def test_chain_axis_and_per_chain_totals():
    rng = np.random.default_rng(2)
    f = _fit(rng, 2, 5, 4, chains=3)
    X = rng.integers(0, 2, (30, 5))
    r = waic_ref(f, X)
    assert r["loglik"].shape == (3, 4)
    for c in range(3):
        rc = waic_ref({"theta": f["theta"][c], "pi": f["pi"][c]}, X)
        assert r["chain_p_waic"][c] == pytest.approx(rc["p_waic"], rel=1e-12)
        assert r["chain_waic"][c] == pytest.approx(rc["waic"], rel=1e-12)


def test_theta_zero_gives_minus_inf_and_nan():
    th = np.full((1, 2, 3), 0.5)
    th[0, 0, 1] = 0.0
    r = waic_ref({"theta": th, "pi": np.ones((3, 1))}, np.array([[1, 0], [0, 0]]))
    L = loglik_matrix(th, np.ones((3, 1)), np.array([[1, 0], [0, 0]]))
    assert L[1, 0] == -np.inf and np.isfinite(L[1, 1])
    assert np.isfinite(r["pointwise_lppd"]).all()
    assert np.isnan(r["pointwise_p_waic"][0]) and np.isfinite(r["pointwise_p_waic"][1])
    assert np.isnan(r["p_waic"]) and np.isnan(r["waic"])


def test_waic_rejects_bad_input_before_the_library():
    rng = np.random.default_rng(3)
    X = rng.integers(0, 2, (20, 5))
    f = _fit(rng, 2, 5, 4)
    with pytest.raises(ValueError, match="pi"):
        B.waic({"theta": f["theta"]}, X)                       # collapsed / DP fits return no pi
    with pytest.raises(ValueError):
        B.waic(f, X[:, :4])                                     # P mismatch
    with pytest.raises(ValueError):
        B.waic({"theta": f["theta"], "pi": f["pi"][:3]}, X)     # S mismatch
    with pytest.raises(ValueError, match="2 draws"):
        B.waic({"theta": f["theta"][:, :, :1], "pi": f["pi"][:1]}, X)
    with pytest.raises(ValueError, match="2 draws"):
        B.waic({"theta": f["theta"][None, :, :, :1], "pi": f["pi"][None, :1]}, X)


def test_bmm_waic_is_exported_and_needs_a_device():
    L = _lib.lib()
    assert "bmm_waic" in _lib.EXPORTS and hasattr(L, "bmm_waic")
    if gpu_available():
        pytest.skip("only meaningful on a box without a GPU")
    rng = np.random.default_rng(4)
    X = np.asfortranarray(rng.integers(0, 2, (10, 3)), dtype=np.int32)
    th = np.full(2 * 3 * 4, 0.5)
    pi = np.full(4 * 2, 0.5)
    d = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    lp = np.zeros(10)
    rc = L.bmm_waic(C.c_void_p(X.ctypes.data), 10, 3, 2, 4, 1, d(th), d(pi), 0, 0, None, d(lp), None, None, None)
    assert rc == -2 and b"CUDA" in L.bmm_last_error()
    # argument errors are reported before the device check
    assert L.bmm_waic(C.c_void_p(X.ctypes.data), 10, 3, 2, 1, 1, d(th), d(pi), 0, 0, None, d(lp), None, None, None) == -1
    assert L.bmm_waic(C.c_void_p(X.ctypes.data), 10, 3, 256, 4, 1, d(th), d(pi), 0, 0, None, d(lp), None, None, None) == -1


def test_rcpp_host_waic_builds_and_reports_the_missing_device(tmp_path):
    L = build_rhost_waic(tmp_path)
    if gpu_available():
        pytest.skip("only meaningful on a box without a GPU")
    X = np.asfortranarray(np.random.default_rng(5).integers(0, 2, (10, 3)), dtype=np.int32)
    th, pi = np.full(2 * 3 * 4, 0.5), np.full(4 * 2, 0.5)
    est, pw, ll = np.zeros(6), np.zeros(30), np.zeros(4)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert L.rhost_waic(p(X), 10, 3, 2, 4, p(th), p(pi), p(est), p(pw), p(ll)) == -1
    assert b"CUDA" in L.rhost_waic_last_error()
