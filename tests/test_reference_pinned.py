"""Pins oracle/oracle.cpp (the restatement every GPU parity test compares with) against the REFERENCE'S OWN
SOURCE, compiled here unmodified: /root/reference/src/{full_gibbs,stickbreaking,collapsed_gibbs,
collapsed_gibbs_dp,stephens,utils,my_lpsolve,RcppExports}.cpp -> oracle/_ref/libbmm_ref.so
(oracle/build_ref.sh, header shim oracle/shim/).  Calls go through the seven registered `.Call` symbols
(src/RcppExports.cpp:137-146) with the argument order of R/RcppExports.R.

Bar: every element of the returned R list (z, z_original, permutations, theta, theta_original, pi, alpha)
bit for bit equal to the oracle's, on the three bundled fixtures, all four samplers, relabel off / on,
fixed and sampled alpha, three seeds.  Both sides draw from the same R-compatible generator (oracle/rrng.h):
unif_rand / rbinom are pinned by the fixture known-answer test; rgamma / rbeta are exact samplers of the same
laws but not nmath's algorithms ("modulo nmath generators", DESIGN.md section 2).
"""
import hashlib
import json
import os

import numpy as np
import pytest

from bmm_mcmc_b200.rcompat import RRng
from conftest import ROOT
from oracle import pyref

# Without the compiled reference, each comparison is made against digests of what the reference returned for the same
# call (tests/golden/reference_pinned.json, tools/make_reference_golden.py).  They hold the outputs that do not depend on
# the assignment solver: the whole list with relabel off; with relabel on the sampled chain (z_original,
# theta_original, pi, alpha) -- relabelling is applied to the outputs and never feeds back into the chain.  The
# relabelled z, theta and permutations also depend on how lp_solve breaks ties, so only the live comparison checks them.
HAVE_REF = pyref.available()
GOLDEN_PATH = os.path.join(ROOT, "tests", "golden", "reference_pinned.json")
SOLVER_FREE = {False: ("alpha", "pi", "z", "theta"), True: ("alpha", "pi", "z_original", "theta_original")}


def digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()[:24]


def golden_entry(ref_list, relabel):
    return {"keys": sorted(ref_list), **{k: digest(ref_list[k]) for k in SOLVER_FREE[relabel] if k in ref_list}}


def _golden():
    with open(GOLDEN_PATH) as f:
        return json.load(f)


def needs_reference(fn):
    return pytest.mark.skipif(not HAVE_REF, reason="needs the compiled reference (oracle/_ref/libbmm_ref.so)")(fn)


SEEDS = (1, 7, 20191)
FIXTURES = ("K2_N100_P5", "K2_N1000_P5", "K3_N1000_P5")


def _init_full(K, P, seed):
    # R/utils.R:68-74: initial_pi = softmax(runif(K)); initial_theta = matrix(runif(K*P), nrow=K)
    rng = RRng(seed)
    ip = np.exp(rng.runif(K))
    ip /= ip.sum()
    return ip, rng.runif(K * P).reshape(P, K).T


def _same(ref_list, oracle_result, relabel, what):
    t = oracle_result.tail()
    keys = set(ref_list)
    expect = {"alpha", "permutations", "z", "theta"} | ({"pi"} if "pi" in t else set())
    if relabel:
        expect |= {"z_original", "theta_original"}
    assert keys == expect, (what, keys)
    for k in sorted(keys):
        if k == "permutations" and not relabel:
            continue  # uninitialised memory in the reference (SURVEY App. D quirk 14)
        a, b = np.asarray(t[k]), ref_list[k]
        assert a.shape == b.shape, (what, k, a.shape, b.shape)
        assert np.array_equal(a, b, equal_nan=True), "%s: %s differs from the reference (max |d| = %s)" % (
            what, k, np.nanmax(np.abs(a.astype(float) - b.astype(float))))


def _same_golden(g, oracle_result, relabel, what):
    t = oracle_result.tail()
    expect = {"alpha", "permutations", "z", "theta"} | ({"pi"} if "pi" in t else set())
    if relabel:
        expect |= {"z_original", "theta_original"}
    assert set(g["keys"]) == expect, (what, g["keys"])
    for k in SOLVER_FREE[relabel]:
        if k in g:
            assert digest(t[k]) == g[k], "%s: %s differs from the reference's recorded output" % (what, k)


def check(what, ref_call, oracle_result, relabel):
    """The oracle's returned list against the reference's for the same call: live when the compiled reference is
    present, else against the recorded digests."""
    if HAVE_REF:
        _same(ref_call(), oracle_result, relabel, what)
    else:
        _same_golden(_golden()["%s relabel=%s" % (what, relabel)], oracle_result, relabel, what)


def check_array(what, ref_call, value):
    if HAVE_REF:
        assert np.array_equal(ref_call(), value), what
    else:
        assert digest(value) == _golden()[what], "%s differs from the reference's recorded output" % what


@needs_reference
def test_registered_symbols_are_the_reference_boundary():
    # src/RcppExports.cpp:137-146
    assert pyref.registered() == {
        "_bmmmcmc_collapsed_gibbs_cpp": 13, "_bmmmcmc_collapsed_gibbs_dp_cpp": 12, "_bmmmcmc_rdirichlet_cpp": 1,
        "_bmmmcmc_gibbs_cpp": 14, "_bmmmcmc_my_lpsolve": 1, "_bmmmcmc_my_stephens_batch": 2,
        "_bmmmcmc_gibbs_stickbreaking_cpp": 14}
    with pytest.raises(RuntimeError, match="Incorrect number of arguments"):
        pyref.dotcall("_bmmmcmc_my_lpsolve", np.eye(2), 1)


@pytest.mark.parametrize("name", FIXTURES)
@pytest.mark.parametrize("relabel", [False, True])
def test_gibbs_full_equals_reference(oracle, datasets, name, relabel):
    X = datasets[name]
    K = 3 if name.startswith("K3") else 2
    ns, burnin, br = (60, 20, 6) if X.shape[0] > 100 else (120, 40, 10)
    for seed in SEEDS:
        for alpha in (0.0, 2.5):
            ip, ith = _init_full(K, X.shape[1], seed + 100)
            o = oracle.gibbs_full(X, ip, ith, ns, K, alpha=alpha, burnin=burnin, relabel=relabel, burnrelabel=br, seed=seed)
            check("gibbs_cpp %s seed %d alpha %g" % (name, seed, alpha),
                  lambda: pyref.gibbs_cpp(X, ip, ith, ns, K, alpha, 0.5, 0.5, 1.0, 1.0, burnin, relabel, br, seed=seed),
                  o, relabel)


@pytest.mark.parametrize("name", FIXTURES)
@pytest.mark.parametrize("relabel", [False, True])
def test_gibbs_stickbreaking_equals_reference(oracle, datasets, name, relabel):
    X = datasets[name]
    maxK = 6
    ns, burnin, br = (50, 20, 5) if X.shape[0] > 100 else (100, 40, 8)
    for seed in SEEDS:
        for alpha in (0.0, 1.0):
            ip, ith = _init_full(maxK, X.shape[1], seed + 200)
            o = oracle.gibbs_stickbreaking(X, ip, ith, ns, maxK, alpha=alpha, burnin=burnin, relabel=relabel,
                                           burnrelabel=br, seed=seed)
            check("gibbs_stickbreaking_cpp %s seed %d alpha %g" % (name, seed, alpha),
                  lambda: pyref.gibbs_stickbreaking_cpp(X, ip, ith, ns, maxK, alpha, 0.5, 0.5, 1.0, 1.0, burnin, relabel, br,
                                                        seed=seed),
                  o, relabel)


def test_gibbs_stickbreaking_burnrelabel_above_burnin_equals_reference(oracle, datasets):
    # R/utils.R:95-107 has no burnrelabel clamp for this sampler: the leading probs_out slices stay zero and
    # become 1e-6 in my_stephens_batch (stephens.cpp:30-31)
    X = datasets["K2_N100_P5"]
    ip, ith = _init_full(4, X.shape[1], 5)
    o = oracle.gibbs_stickbreaking(X, ip, ith, 60, 4, burnin=6, relabel=True, burnrelabel=50, seed=3)
    check("stick-breaking burnrelabel > burnin",
          lambda: pyref.gibbs_stickbreaking_cpp(X, ip, ith, 60, 4, 0.0, 0.5, 0.5, 1.0, 1.0, 6, True, 50, seed=3), o, True)


@pytest.mark.parametrize("name", FIXTURES)
@pytest.mark.parametrize("relabel", [False, True])
def test_gibbs_collapsed_equals_reference(oracle, datasets, name, relabel):
    X = datasets[name]
    K = 3 if name.startswith("K3") else 2
    ns, burnin, br = (24, 10, 4) if X.shape[0] > 100 else (150, 50, 10)
    for seed in SEEDS:
        for alpha in (0.0, 1.5):
            iz = RRng(seed + 300).sample_int(K, X.shape[0])  # R/utils.R:42
            o = oracle.gibbs_collapsed(X, iz, ns, K, alpha=alpha, burnin=burnin, relabel=relabel, burnrelabel=br, seed=seed)
            check("collapsed_gibbs_cpp %s seed %d alpha %g" % (name, seed, alpha),
                  lambda: pyref.collapsed_gibbs_cpp(X, iz, ns, K, alpha, 0.5, 0.5, 1.0, 1.0, burnin, relabel, br, seed=seed),
                  o, relabel)


def test_gibbs_collapsed_empty_cluster_equals_reference(oracle, datasets):
    # quirks 7 and 8: a cluster that starts empty stays empty and its theta is NaN (collapsed_gibbs.cpp:104,214)
    X = datasets["K2_N100_P5"]
    iz = np.where(np.arange(100) % 2 == 0, 1, 3).astype(np.int32)
    o = oracle.gibbs_collapsed(X, iz, 40, 3, burnin=10, relabel=True, burnrelabel=5, seed=11)
    check("collapsed with an empty cluster",
          lambda: pyref.collapsed_gibbs_cpp(X, iz, 40, 3, 0.0, 0.5, 0.5, 1.0, 1.0, 10, True, 5, seed=11), o, True)
    assert np.isnan(o.tail()["theta_original"][1]).all()


@pytest.mark.parametrize("name", FIXTURES)
@pytest.mark.parametrize("relabel", [False, True])
def test_gibbs_dp_equals_reference(oracle, datasets, name, relabel):
    X = datasets[name]
    ns, burnin, br = (16, 8, 3) if X.shape[0] > 100 else (120, 40, 8)
    for seed in SEEDS:
        # with relabelling every sweep solves a maxK x maxK assignment in lp_solve (5 ms at 30, 34 ms at 64) and the
        # batch step 100 x burnrelabel of them: keep maxK small there
        for alpha, maxK in (((0.0, 12), (1.0, 14)) if relabel else ((0.0, 30), (1.0, 64))):
            o = oracle.gibbs_dp(X, ns, alpha=alpha, burnin=burnin, relabel=relabel, burnrelabel=br, maxK=maxK, seed=seed)
            check("collapsed_gibbs_dp_cpp %s seed %d alpha %g" % (name, seed, alpha),
                  lambda: pyref.collapsed_gibbs_dp_cpp(X, ns, alpha, 0.5, 0.5, 1.0, 1.0, burnin, relabel, br, maxK, seed=seed),
                  o, relabel)


def test_gibbs_dp_truncation_equals_reference(oracle, datasets):
    # quirk 9 (collapsed_gibbs_dp.cpp:213-231): at the cap the draw falls back to an index into used_clusters
    X = datasets["K2_N100_P5"]
    hit = 0
    for seed in range(1, 9):
        try:
            o = oracle.gibbs_dp(X, 30, alpha=8.0, burnin=10, relabel=False, maxK=5, seed=seed)
        except RuntimeError:
            continue  # the reference's own state went inconsistent (undefined behaviour there): not comparable
        check("DP at the truncation cap, seed %d" % seed,
              lambda: pyref.collapsed_gibbs_dp_cpp(X, 30, 8.0, 0.5, 0.5, 1.0, 1.0, 10, False, 50, 5, seed=seed), o, False)
        hit += 1
    assert hit >= 1


@needs_reference
def test_gibbs_dp_requires_symmetric_prior_like_reference(datasets):
    with pytest.raises(RuntimeError, match="non-symmetric priors"):
        pyref.collapsed_gibbs_dp_cpp(datasets["K2_N100_P5"], 10, 1.0, 0.5, 0.6, 1.0, 1.0, 2, False, 1, 10)


@needs_reference
def test_stephens_batch_and_online_equal_reference(oracle):
    rng = np.random.default_rng(5)
    for N, K, M in ((100, 2, 6), (250, 3, 5), (60, 5, 4), (40, 8, 3)):
        p = rng.dirichlet(np.ones(K) * 0.7, size=(M, N)).transpose(1, 2, 0).copy()
        p[rng.random(p.shape) < 0.02] = 0.0  # exercises p.replace(0, 1e-6) (stephens.cpp:30-31)
        q_o, _ = oracle.stephens_batch(p)
        q_r = pyref.my_stephens_batch(p)
        assert np.array_equal(q_o, q_r)
        ps = rng.dirichlet(np.ones(K), size=N)
        for j in (5, 77):
            perm_o, qn_o, _ = oracle.stephens_online(q_o, ps, j)
            perm_r, qn_r = pyref.my_stephens_online(q_r, ps, j)
            assert np.array_equal(perm_o, perm_r) and np.array_equal(qn_o, qn_r)


def test_my_lpsolve_equals_reference(oracle):
    rng = np.random.default_rng(9)
    for K in (2, 3, 5, 8, 16):
        for _ in range(4):
            c = rng.uniform(0, 50, (K, K))
            # random costs: the optimum is unique, so the exact solver the oracle falls back to gives lp_solve's answer
            check_array("my_lpsolve K=%d #%d" % (K, _), lambda: pyref.my_lpsolve(c), oracle.assign(c, True if HAVE_REF else None))
    if HAVE_REF:   # a tie: lp_solve's own tie-break, which only lp_solve itself reproduces
        assert np.array_equal(pyref.my_lpsolve(np.zeros((3, 3))), np.eye(3, dtype=np.int32)[::-1])  # SURVEY 8a11


def test_rdirichlet_and_update_alpha_equal_reference(oracle):
    for seed in SEEDS:
        am = np.array([0.3, 2.0, 11.5, 1.0])
        check_array("rdirichlet_cpp seed %d" % seed, lambda: pyref.rdirichlet_cpp(am, seed=seed), oracle.rdirichlet(seed, am))
    if not HAVE_REF:
        return
    # update_alpha (utils.cpp:6-14): the oracle's copy is only reachable through a sampler; one sweep of the
    # collapsed sampler with alpha sampled exposes it (alpha[1] = update_alpha(1, a, b, N, K) after N rmultinom draws)
    a1 = pyref.update_alpha(1.0, 1.0, 1.0, 100, 2, seed=4)
    assert np.isfinite(a1) and a1 > 0


@needs_reference
def test_reference_consumes_the_uniforms_the_oracle_records(oracle, datasets):
    """The per-draw uniforms the oracle logs (what the GPU replays) are, in order, a subsequence of the stream
    the compiled reference consumed: the z-draw uniforms of sweep j, then that sweep's parameter draws."""
    import ctypes as C
    X = datasets["K2_N100_P5"]
    iz = RRng(2).sample_int(2, 100)
    L = pyref.lib()
    buf = np.zeros(200000)
    L.ref_set_seed(C.c_uint(13))
    L.ref_record_uniforms(buf.ctypes.data_as(C.POINTER(C.c_double)), buf.size)
    pyref.collapsed_gibbs_cpp(X, iz, 12, 2, 1.0, 0.5, 0.5, 1.0, 1.0, 4, False, 1, seed=None)
    n = L.ref_recorded()
    L.ref_record_uniforms(None, 0)
    o = oracle.gibbs_collapsed(X, iz, 12, 2, alpha=1.0, burnin=4, seed=13)
    u = o["u_rec"][1:].ravel()
    u = u[u >= 0]
    # alpha fixed => no parameter draws at all: the streams are identical
    assert n == u.size and np.array_equal(buf[:n], u)
