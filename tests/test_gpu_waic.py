"""WAIC and the log-likelihood trace on the device (bmm_waic) against the float64 reference of tests/waic_ref.py, the
invariances the definitions imply, the tcgen05 kernel against the fp64 kernel, model choice, and the Rcpp host."""
import ctypes as C
import os

import numpy as np
import pytest

import bmm_mcmc_b200 as B
from bmm_mcmc_b200 import _lib
from conftest import gpu_available
from waic_ref import waic_ref

pytestmark = pytest.mark.gpu

OUTS = ("pointwise_lppd", "pointwise_p_waic", "pointwise_elpd_waic", "pointwise_waic", "lppd", "p_waic", "elpd_waic",
        "waic", "se_lppd", "se_p_waic", "se_elpd_waic", "se_waic", "loglik")
CHAIN_OUTS = ("chain_elpd_waic", "chain_waic", "chain_p_waic")


@pytest.fixture(autouse=True)
def _need_gpu():
    if not gpu_available():
        pytest.skip("needs a GPU")


def _last_path():
    ms, t = C.c_float(), C.c_int32()
    _lib.check(_lib.lib().bmm_waic_kernel_ms(C.byref(ms), C.byref(t)))
    return "tensor" if t.value else "fp64"


def _close(got, want, rtol, chains=False):
    for k in OUTS + (CHAIN_OUTS if chains else ()):
        np.testing.assert_allclose(got[k], want[k], rtol=rtol, atol=0, err_msg=k)


@pytest.mark.parametrize("name,K", [("K2_N100_P5", 2), ("K2_N1000_P5", 2), ("K3_N1000_P5", 3)])
@pytest.mark.parametrize("chains", [1, 8])
def test_fp64_equals_reference_gibbs_full(datasets, name, K, chains):
    X = datasets[name]
    fit = B.gibbs_full(X, 120, K, burnin=20, seed=11, chains=chains)
    got = B.waic(fit, X, no_tensor=True)
    assert _last_path() == "fp64"
    _close(got, waic_ref(fit, X), 1e-10, chains > 1)
    assert got["loglik"].shape == ((chains, 100) if chains > 1 else (100,))


def test_fp64_equals_reference_stickbreaking_p70_and_thin(datasets):
    rng = np.random.default_rng(5)
    X = (rng.uniform(size=(400, 70)) < np.where(rng.integers(0, 2, (400, 1)) == 1, 0.8, 0.2)).astype(np.int32)
    fit = B.gibbs_stickbreaking(X, 80, 6, burnin=20, seed=2, chains=8)
    _close(B.waic(fit, X, no_tensor=True), waic_ref(fit, X), 1e-10, True)
    fit = B.gibbs_full(datasets["K3_N1000_P5"], 151, 3, burnin=31, seed=4, thin=3)
    assert fit["theta"].shape[2] == 40
    _close(B.waic(fit, datasets["K3_N1000_P5"]), waic_ref(fit, datasets["K3_N1000_P5"]), 1e-10)


def test_pooled_lppd_is_predictive_log_pred(datasets):
    X = datasets["K3_N1000_P5"]
    fit = B.gibbs_full(X, 200, 3, burnin=50, seed=7, chains=4)
    np.testing.assert_allclose(B.waic(fit, X)["pointwise_lppd"], B.predictive(fit, X, membership=False)["log_pred"],
                               rtol=1e-12, atol=0)


def test_invariances(datasets):
    X = datasets["K3_N1000_P5"]
    fit = B.gibbs_full(X, 150, 3, burnin=50, seed=9, chains=3)
    base = B.waic(fit, X)
    # relabelling the clusters
    perm = [2, 0, 1]
    pf = {"theta": fit["theta"][:, perm], "pi": fit["pi"][:, :, perm]}
    _close(B.waic(pf, X), base, 1e-12, True)
    # duplicated and shuffled rows: pointwise values move with the rows
    rng = np.random.default_rng(1)
    idx = rng.permutation(np.concatenate([np.arange(len(X)), rng.integers(0, len(X), 500)]))
    r = B.waic(fit, X[idx])
    for k in ("pointwise_lppd", "pointwise_p_waic"):
        np.testing.assert_allclose(r[k], base[k][idx], rtol=1e-12, atol=0)
    want = waic_ref(fit, X[idx])
    for k in ("lppd", "p_waic", "waic", "loglik", "chain_waic", "chain_p_waic"):
        np.testing.assert_allclose(r[k], want[k], rtol=1e-12, atol=0, err_msg=k)
    # bit-packed input and a second call: the same bits
    for again in (B.waic(fit, B.PackedX.pack(X)), B.waic(fit, X)):
        for k in OUTS + CHAIN_OUTS:
            assert np.array_equal(again[k], base[k]), k


def test_theta_zero_one_minus_inf_nan_pattern(datasets):
    X = datasets["K2_N100_P5"]
    fit = B.gibbs_full(X, 40, 2, burnin=10, seed=1)
    th = fit["theta"].copy()
    th[:, 0, 3] = 0.0          # every row with x_0 = 1 has no mass under draw 3: l = -inf, p_waic = nan
    th[1, 2, 5] = 1.0          # cluster 1 of draw 5 gives no mass to rows with x_2 = 0, cluster 0 still does
    f2 = {"theta": th, "pi": fit["pi"].copy()}
    f2["pi"][7] = [1.0, 0.0]
    got, want = B.waic(f2, X, no_tensor=True), waic_ref(f2, X)
    for k in ("pointwise_lppd", "pointwise_p_waic", "loglik"):
        assert np.array_equal(np.isnan(got[k]), np.isnan(want[k])), k
        assert np.array_equal(np.isneginf(got[k]), np.isneginf(want[k])), k
        fin = np.isfinite(want[k])
        np.testing.assert_allclose(got[k][fin], want[k][fin], rtol=1e-10)
    assert np.isnan(want["p_waic"]) and np.isnan(got["p_waic"]) and np.isnan(got["waic"])
    assert np.isfinite(got["pointwise_lppd"]).all()


def test_non_binary_data_is_rejected(datasets):
    X = datasets["K2_N100_P5"].copy()
    fit = B.gibbs_full(X, 30, 2, burnin=10, seed=1)
    X[3, 2] = 2
    with pytest.raises(_lib.BmmError, match="NOT_BINARY"):
        B.waic(fit, X)


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
def test_tensor_kernel_against_fp64(K, P, source, monkeypatch):
    X, fit = _tc_case(K, P, source)
    want = B.waic(fit, X, no_tensor=True)
    monkeypatch.setenv("BMM_WAIC_TENSOR", "1")
    got = B.waic(fit, X)
    assert _last_path() == "tensor"
    monkeypatch.setenv("BMM_GRID_MAX_CTAS", "3")
    got3 = B.waic(fit, X)
    for k in OUTS:
        assert np.array_equal(got3[k], got[k]), k
    d_lppd = np.abs(got["pointwise_lppd"] - want["pointwise_lppd"]).max()
    d_pw = np.abs(got["pointwise_p_waic"] - want["pointwise_p_waic"]).max()
    r_ll = np.abs(got["loglik"] / want["loglik"] - 1).max()
    print("tc-vs-fp64 K=%d P=%d %s: |d lppd_i| %.3g |d p_waic_i| %.3g loglik rel %.3g lppd rel %.3g p_waic rel %.3g" % (
        K, P, source, d_lppd, d_pw, r_ll, abs(got["lppd"] / want["lppd"] - 1), abs(got["p_waic"] / want["p_waic"] - 1)))
    # observed maxima on a B200 over these cases: 1.3e-5, 2.3e-5, 6.4e-8, 6.2e-9, 1.5e-7 (DESIGN.md section 4)
    assert d_lppd <= 1e-4 and d_pw <= 1e-4
    assert r_ll <= 1e-6
    assert got["lppd"] == pytest.approx(want["lppd"], rel=1e-7)
    assert got["p_waic"] == pytest.approx(want["p_waic"], rel=1e-5)


def test_waic_picks_the_true_number_of_clusters():
    rng = np.random.default_rng(2024)
    centres = np.where(rng.integers(0, 2, (3, 20)) == 1, 0.9, 0.1)
    centres[1] = 1 - centres[0]
    X = (rng.uniform(size=(3000, 20)) < centres[rng.integers(0, 3, 3000)]).astype(np.int32)
    w = [B.waic(B.gibbs_full(X, 300, K, burnin=100, seed=5), X)["waic"] for K in (1, 2, 3)]
    assert w[2] + 100 < w[1] and w[1] + 100 < w[0], w


def test_rcpp_host_waic_equals_ctypes(datasets, tmp_path):
    from test_waic_ref import build_rhost_waic
    L = build_rhost_waic(tmp_path)
    X = np.asfortranarray(datasets["K3_N1000_P5"], dtype=np.int32)
    fit = B.gibbs_full(X, 120, 3, burnin=20, seed=3)
    K, P, S = fit["theta"].shape
    th = np.ascontiguousarray(fit["theta"].transpose(2, 1, 0))
    pi = np.ascontiguousarray(fit["pi"].T)
    est, pw, ll = np.zeros(6), np.zeros(len(X) * 3), np.zeros(S)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert L.rhost_waic(p(X), len(X), P, K, S, p(th), p(pi), p(est), p(pw), p(ll)) == 0, L.rhost_waic_last_error()
    want = B.waic(fit, X)
    est = est.reshape(2, 3).T
    pw = pw.reshape(3, len(X)).T
    assert np.array_equal(ll, want["loglik"])
    for j, k in enumerate(("elpd_waic", "p_waic", "waic")):
        assert np.array_equal(pw[:, j], want["pointwise_" + k])
        np.testing.assert_allclose(est[j], [want[k], want["se_" + k]], rtol=1e-12)
