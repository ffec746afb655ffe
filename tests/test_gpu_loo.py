"""PSIS-LOO and the log-likelihood matrix on the device (bmm_loo, bmm_loglik_matrix) against the float64 reference of
tests/loo_ref.py, the invariances the definitions imply, the tcgen05 matrix against the fp64 one, model choice, and the
Rcpp host."""
import ctypes as C

import numpy as np
import pytest

import bmm_mcmc_b200 as B
from bmm_mcmc_b200 import _lib
from conftest import gpu_available
from loo_ref import loo_ref
from waic_ref import loglik_matrix as ref_loglik

pytestmark = pytest.mark.gpu

POINTWISE = ("pointwise_elpd_loo", "pointwise_lpd", "pointwise_p_loo", "pointwise_looic", "n_eff")
TOTALS = ("elpd_loo", "lpd", "p_loo", "looic", "se_elpd_loo", "se_lpd", "se_p_loo", "se_looic")
COUNTS = ("k_threshold", "n_k_good", "n_k_bad", "n_k_very_bad")
ALL = POINTWISE + TOTALS + ("pareto_k",) + COUNTS


@pytest.fixture(autouse=True)
def _need_gpu():
    if not gpu_available():
        pytest.skip("needs a GPU")


def _last_path():
    ms, t = C.c_float(), C.c_int32()
    _lib.check(_lib.lib().bmm_loo_kernel_ms(C.byref(ms), C.byref(t)))
    return "tensor" if t.value else "fp64"


def _close(got, want, rtol=1e-10, katol=1e-9):
    for k in POINTWISE + TOTALS:
        np.testing.assert_allclose(got[k], want[k], rtol=rtol, atol=0, err_msg=k)
    np.testing.assert_allclose(got["pareto_k"], want["pareto_k"], rtol=0, atol=katol, err_msg="pareto_k")
    for k in COUNTS:
        assert got[k] == want[k], k


def _same_bits(a, b):
    for k in ALL:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize("name,K", [("K2_N100_P5", 2), ("K2_N1000_P5", 2), ("K3_N1000_P5", 3)])
@pytest.mark.parametrize("chains", [1, 8])
def test_fp64_equals_reference_gibbs_full(datasets, name, K, chains):
    # D = 100 (M = 20, one thread per row) and D = 800 (M = 85, the radix-select path)
    X = datasets[name]
    fit = B.gibbs_full(X, 120, K, burnin=20, seed=11, chains=chains)
    got = B.loo(fit, X, no_tensor=True)
    assert _last_path() == "fp64"
    _close(got, loo_ref(fit, X))


def test_fp64_equals_reference_stickbreaking_p70_thin_short_and_long(datasets):
    rng = np.random.default_rng(5)
    X = (rng.uniform(size=(400, 70)) < np.where(rng.integers(0, 2, (400, 1)) == 1, 0.8, 0.2)).astype(np.int32)
    fit = B.gibbs_stickbreaking(X, 80, 6, burnin=20, seed=2, chains=8)
    _close(B.loo(fit, X, no_tensor=True), loo_ref(fit, X))
    X3 = datasets["K3_N1000_P5"]
    fit = B.gibbs_full(X3, 151, 3, burnin=31, seed=4, thin=3)
    assert fit["theta"].shape[2] == 40
    _close(B.loo(fit, X3), loo_ref(fit, X3))
    # D = 15 <= 20: no smoothing, k = inf everywhere
    fit = B.gibbs_full(X3, 25, 3, burnin=10, seed=6)
    got = B.loo(fit, X3)
    assert np.isinf(got["pareto_k"]).all()
    _close(got, loo_ref(fit, X3))
    # D = 20000: M = 425, several CTAs per row
    X2 = datasets["K2_N100_P5"]
    fit = B.gibbs_full(X2, 20050, 2, burnin=50, seed=8)
    _close(B.loo(fit, X2), loo_ref(fit, X2))


def test_vector_r_eff_on_identical_rows(datasets):
    X = datasets["K2_N100_P5"]                                  # 100 rows of 5 bits: many identical rows
    fit = B.gibbs_full(X, 600, 2, burnin=100, seed=12, chains=2)
    re = np.random.default_rng(7).uniform(0.05, 3.0, len(X))   # M from 200 down to 55: both paths
    got = B.loo(fit, X, r_eff=re)
    _close(got, loo_ref(fit, X, re))
    assert len(np.unique(got["pareto_k"])) > len(np.unique(X, axis=0))


def test_lpd_and_matrix_cross_checks(datasets):
    X = datasets["K3_N1000_P5"]
    fit = B.gibbs_full(X, 200, 3, burnin=50, seed=7, chains=4)
    w = B.waic(fit, X)
    np.testing.assert_allclose(B.loo(fit, X)["pointwise_lpd"], w["pointwise_lppd"], rtol=1e-12, atol=0)
    L = B.loglik_matrix(fit, X)
    assert L.shape == (4, 150, len(X))
    want = np.stack([ref_loglik(fit["theta"][c], fit["pi"][c], X) for c in range(4)])
    np.testing.assert_allclose(L, want, rtol=1e-12, atol=0)
    np.testing.assert_allclose(L.sum(axis=2), w["loglik"], rtol=1e-12, atol=0)
    f1 = {"theta": fit["theta"][0], "pi": fit["pi"][0]}
    assert np.array_equal(B.loglik_matrix(f1, X), L[0])


def test_invariances(datasets, monkeypatch):
    X = datasets["K3_N1000_P5"]
    fit = B.gibbs_full(X, 150, 3, burnin=50, seed=9, chains=3)       # D = 300: M = 52, one thread per row
    base = B.loo(fit, X)
    perm = [2, 0, 1]
    _close(B.loo({"theta": fit["theta"][:, perm], "pi": fit["pi"][:, :, perm]}, X), base, 1e-12, 1e-12)
    rng = np.random.default_rng(1)
    idx = rng.permutation(np.concatenate([np.arange(len(X)), rng.integers(0, len(X), 500)]))
    r = B.loo(fit, X[idx])
    for k in POINTWISE + ("pareto_k",):
        np.testing.assert_allclose(r[k], base[k][idx], rtol=1e-12, atol=0, err_msg=k)
    for again in (B.loo(fit, B.PackedX.pack(X)), B.loo(fit, X)):
        _same_bits(again, base)
    monkeypatch.setenv("BMM_LOO_CHUNK_ROWS", "5")
    _same_bits(B.loo(fit, X), base)
    # long rows (D = 1200, M = 104) in small chunks, and a second call
    monkeypatch.delenv("BMM_LOO_CHUNK_ROWS")
    fit = B.gibbs_full(X, 450, 3, burnin=50, seed=10, chains=3)
    base = B.loo(fit, X)
    _same_bits(B.loo(fit, X), base)
    monkeypatch.setenv("BMM_LOO_CHUNK_ROWS", "3")
    _same_bits(B.loo(fit, X), base)
    L3 = B.loglik_matrix(fit, X)
    monkeypatch.delenv("BMM_LOO_CHUNK_ROWS")
    assert np.array_equal(L3, B.loglik_matrix(fit, X))


def test_theta_zero_one_nan_pattern(datasets):
    X = datasets["K2_N100_P5"]
    fit = B.gibbs_full(X, 60, 2, burnin=10, seed=1)
    th = fit["theta"].copy()
    th[:, 0, 3] = 0.0          # every row with x_0 = 1 has no mass under draw 3: l = -inf, elpd_loo = nan
    th[1, 2, 5] = 1.0
    f2 = {"theta": th, "pi": fit["pi"].copy()}
    f2["pi"][7] = [1.0, 0.0]
    got, want = B.loo(f2, X, no_tensor=True), loo_ref(f2, X)
    for k in POINTWISE + ("pareto_k",):
        assert np.array_equal(np.isnan(got[k]), np.isnan(want[k])), k
        assert np.array_equal(np.isinf(got[k]), np.isinf(want[k])), k
        fin = np.isfinite(want[k])
        np.testing.assert_allclose(got[k][fin], want[k][fin], rtol=1e-10, err_msg=k)
    assert np.isnan(got["pointwise_elpd_loo"]).any() and np.isfinite(got["pointwise_elpd_loo"]).any()
    assert np.isfinite(got["pointwise_lpd"]).all()


def _tc_case(K, P, source, N=20011, S=40):
    rng = np.random.default_rng(K * 1000 + P)
    centres = rng.uniform(0.1, 0.9, (max(K, 2), P))
    z = rng.integers(0, max(K, 2), N)
    X = (rng.uniform(size=(N, P)) < centres[z]).astype(np.int32)
    if source == "fit":
        fit = B.gibbs_full(B.PackedX.pack(X), 10 + S, K, burnin=10, seed=3, grid_path=True, no_z_history=True)
        fit = {"theta": fit["theta"], "pi": fit["pi"]}
    else:
        fit = {"theta": rng.uniform(1e-3, 1 - 1e-3, (K, P, S)), "pi": rng.dirichlet(np.ones(K), S)}
    return X, fit


@pytest.mark.parametrize("K,P", [(32, 64), (5, 20), (32, 112), (1, 7)])
@pytest.mark.parametrize("source", ["fit", "uniform"])
def test_tensor_matrix_against_fp64(K, P, source, monkeypatch):
    X, fit = _tc_case(K, P, source)
    want = B.loo(fit, X, no_tensor=True)
    monkeypatch.setenv("BMM_WAIC_TENSOR", "1")
    got = B.loo(fit, X)
    assert _last_path() == "tensor"
    Lt = B.loglik_matrix(fit, X)
    monkeypatch.setenv("BMM_GRID_MAX_CTAS", "3")
    _same_bits(B.loo(fit, X), got)
    assert np.array_equal(B.loglik_matrix(fit, X), Lt)
    d_el = np.abs(got["pointwise_elpd_loo"] - want["pointwise_elpd_loo"]).max()
    d_p = np.abs(got["pointwise_p_loo"] - want["pointwise_p_loo"]).max()
    fin = np.isfinite(want["pareto_k"])
    d_k = np.abs(got["pareto_k"][fin] - want["pareto_k"][fin]).max() if fin.any() else 0.0
    print("tc-vs-fp64 K=%d P=%d %s: |d elpd_loo_i| %.3g |d p_loo_i| %.3g |d k_i| %.3g elpd_loo rel %.3g" % (
        K, P, source, d_el, d_p, d_k, abs(got["elpd_loo"] / want["elpd_loo"] - 1)))
    assert np.array_equal(np.isfinite(got["pareto_k"]), fin)
    # observed maxima on a B200 over these cases: 1.07e-3 (elpd_loo_i, p_loo_i), 0.031 (k, fitted to 8 tail draws at
    # D = 40) and 6.4e-9 (elpd_loo total, relative) (DESIGN.md section 4)
    assert d_el <= 5e-3 and d_p <= 5e-3 and d_k <= 0.15
    assert got["elpd_loo"] == pytest.approx(want["elpd_loo"], rel=1e-7)


def test_loo_picks_the_true_number_of_clusters():
    rng = np.random.default_rng(2024)
    centres = np.where(rng.integers(0, 2, (3, 20)) == 1, 0.9, 0.1)
    centres[1] = 1 - centres[0]
    X = (rng.uniform(size=(3000, 20)) < centres[rng.integers(0, 3, 3000)]).astype(np.int32)
    r = [B.loo(B.gibbs_full(X, 300, K, burnin=100, seed=5), X) for K in (1, 2, 3)]
    ic = [x["looic"] for x in r]
    assert ic[2] + 100 < ic[1] and ic[1] + 100 < ic[0], ic
    assert r[2]["n_k_very_bad"] == 0


def test_rcpp_host_loo_equals_ctypes(datasets, tmp_path):
    from test_loo_ref import build_rhost_loo
    L = build_rhost_loo(tmp_path)
    X = np.asfortranarray(datasets["K3_N1000_P5"], dtype=np.int32)
    fit = B.gibbs_full(X, 520, 3, burnin=20, seed=3)          # D = 500: M = 68, the radix-select path
    K, P, S = fit["theta"].shape
    N = len(X)
    th = np.ascontiguousarray(fit["theta"].transpose(2, 1, 0))
    pi = np.ascontiguousarray(fit["pi"].T)
    re = np.random.default_rng(3).uniform(0.3, 1.2, N)
    est, pw, k, ne = np.zeros(6), np.zeros(N * 4), np.zeros(N), np.zeros(N)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert L.rhost_loo(p(X), N, P, K, S, p(th), p(pi), p(re), p(est), p(pw), p(k), p(ne)) == 0, L.rhost_loo_last_error()
    want = B.loo(fit, X, r_eff=re)
    est, pw = est.reshape(2, 3).T, pw.reshape(4, N).T
    for j, name in enumerate(("elpd_loo", "p_loo", "looic")):
        assert np.array_equal(pw[:, j], want["pointwise_" + name])
        np.testing.assert_allclose(est[j], [want[name], want["se_" + name]], rtol=1e-12)
    assert np.array_equal(pw[:, 3], want["pareto_k"]) and np.array_equal(k, want["pareto_k"])
    assert np.array_equal(ne, want["n_eff"])
    ll = np.zeros(S * N)
    assert L.rhost_loglik(p(X), N, P, K, S, p(th), p(pi), p(ll)) == 0, L.rhost_loo_last_error()
    assert np.array_equal(ll.reshape(N, S).T, B.loglik_matrix(fit, X))
