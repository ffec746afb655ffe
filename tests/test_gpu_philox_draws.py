"""Every Philox-mode draw of a run against the float64 transcription of its stream (tests/philox_ref.py).

Runs keep every sweep (thin = 1) from burnin = 0 (burnin = 2 where relabelling needs a window before it), so the
returned histories hold the state every checked sweep started from.  For each sweep the tests check
  - allocations: each z is the inverse-CDF category of the float64 conditional at the transcribed uniform; a draw is
    exempt only when u lies within DELTA of an interior CDF boundary (fewer than max(3, 5 x expected) of them), and a
    drawn category of float64 probability < 1e-12 is never exempt;
  - parameters: theta, pi (sticks), alpha equal the transcribed draws from the counts of the returned z to 1e-12
    (skipped only where a rejection decision or the 0.01 K_viable threshold fell within 1e-10 of its boundary);
    collapsed theta is S_kd / N_k exactly, NaN for an empty cluster.
The replay-mode tests feed the oracle's uniforms and parameters in; these check the branches users run.
"""
import numpy as np
import pytest

import bmm_mcmc_b200 as B
import philox_ref as R
from bmm_mcmc_b200 import _lib
from conftest import gpu_available

pytestmark = pytest.mark.gpu

DELTA64 = 1e-12     # fp64 paths
DELTA32 = 2e-4      # fp32 tensor-core and CUDA-core grid paths (1e-4 relative on the probabilities)
DELTA_C32 = 1e-5    # collapsed product form in fp32
SEED_HI = (0x2B << 32) | 977      # non-zero high 32 bits: the stream word carries seed_hi << 8


def _need_gpu():
    assert gpu_available(), "CUDA library/device unavailable: " + repr(_lib.LIB_PATH)


def _synthetic(N, P, K, seed):
    rng = np.random.default_rng(seed)
    th = rng.uniform(0.1, 0.9, (K, P))
    return (rng.random((N, P)) < th[rng.integers(0, K, N)]).astype(np.int32)


def _init(chains, K, P, seed, zero_last=False):
    rng = np.random.default_rng(seed)
    pi = rng.uniform(0.5, 1.5, (chains, K))
    if zero_last:
        pi[:, K - 1] = 0.0
    pi /= pi.sum(1, keepdims=True)
    return pi, rng.uniform(0.2, 0.8, (chains, K, P))


def _chain(res, c):
    return {k: v[c] for k, v in res.items()}


class Tally:
    def __init__(self):
        self.exempt, self.expected, self.near, self.sweeps = 0, 0.0, 0, 0

    def finish(self, label):
        print("%s: %d sweeps, %d allocation exemptions (expected %.2f), %d parameter draws near a boundary"
              % (label, self.sweeps, self.exempt, self.expected, self.near))
        assert self.exempt <= max(3, 5 * self.expected), "%d exemptions, %.2f expected" % (self.exempt, self.expected)


def _check_z(prob, u, z, delta, tally, where):
    bad, ex, tiny = R.icdf_check(prob, u, z, delta)
    ref = np.minimum((u[:, None] >= np.cumsum(prob, 1)[:, :-1] / prob.sum(1)[:, None]).sum(1), prob.shape[1] - 1)
    assert len(tiny) == 0, "%s: rows %s drew categories of probability %s" % (where, tiny[:5], prob[tiny[:5], z[tiny[:5]]])
    assert len(bad) == 0, "%s: %d allocations differ, rows %s: z %s, reference %s, u %s" % (
        where, len(bad), bad[:5], z[bad[:5]], ref[bad[:5]], u[bad[:5]])
    tally.exempt += len(ex)
    tally.expected += R.expected_exempt(prob, delta)


def check_uncollapsed(res, X, K, *, seed, chain, stickbreaking, alpha0, delta, float_u=False, relabel=False,
                      params=True, tally=None, burnin=0, beta=0.5, gamma=0.5, a=1.0, b=1.0):
    """One chain of gibbs_full / gibbs_stickbreaking (kern_full.cu, kern_big*.cu).  Row r of the histories is
    sweep burnin + r; rows r >= 1 are checked."""
    zk, tk = ("z_original", "theta_original") if relabel else ("z", "theta")
    Z, TH, PI, AL = res[zk], res[tk], res["pi"], res["alpha"][:, 0]
    S, N = Z.shape
    t = tally or Tally()
    for r in range(1, S):
        j = burnin + r
        w = R.z_words_rows(seed, chain, j, np.arange(N))
        u = R.u32_unit_f(w).astype(np.float64) if float_u else R.u32_unit(w)
        z = Z[r].astype(np.int64) - 1
        _check_z(R.uncollapsed_probs(X, TH[:, :, r - 1], PI[r - 1]), u, z, delta, t, "chain %d sweep %d" % (chain, j))
        t.sweeps += 1
        if not params:
            continue
        th, pi, al, _, near = R.uncollapsed_params(seed, chain, j, z, X, K, AL[r - 1], alpha0, beta, gamma, a, b, stickbreaking)
        if near:
            t.near += 1
            continue
        np.testing.assert_allclose(TH[:, :, r], th, rtol=1e-12, atol=0, err_msg="theta, chain %d sweep %d" % (chain, j))
        np.testing.assert_allclose(PI[r], pi, rtol=1e-12, atol=0, err_msg="pi, chain %d sweep %d" % (chain, j))
        np.testing.assert_allclose(AL[r], al, rtol=1e-12, atol=0, err_msg="alpha, chain %d sweep %d" % (chain, j))
    if tally is None:
        t.finish("chain %d" % chain)
    return t


def check_collapsed(res, X, K, z0, *, seed, chain, alpha0, delta, fp32=False, relabel=False, tally=None, burnin=0,
                    beta=0.5, gamma=0.5, a=1.0, b=1.0):
    """One chain of gibbs_collapsed (kern_collapsed.cu): sequential conditionals, S / N theta, sequential alpha.
    Row r is sweep burnin + r; sweep 1 starts from the initial labels z0."""
    zk, tk = ("z_original", "theta_original") if relabel else ("z", "theta")
    Z, TH, AL = res[zk], res[tk], res["alpha"][:, 0]
    S, N = Z.shape
    X64 = np.asarray(X, dtype=np.int64)
    t = tally or Tally()
    z_prev = (np.asarray(z0) if burnin == 0 else Z[0]).astype(np.int64) - 1
    for r in range(1, S):
        j = burnin + r
        z = Z[r].astype(np.int64) - 1
        u = R.z_uniforms_collapsed(seed, chain, j, N)
        if fp32:
            u = np.minimum(u.astype(np.float32), R.UF_MAX).astype(np.float64)
        prob = R.collapsed_probs_sweep(X, z_prev, z, K, AL[r - 1], beta, gamma)
        _check_z(prob, u, z, delta, t, "chain %d sweep %d" % (chain, j))
        t.sweeps += 1
        Nk = np.bincount(z, minlength=K)
        Skd = np.zeros((K, X.shape[1]), dtype=np.int64)
        np.add.at(Skd, z, X64)
        with np.errstate(invalid="ignore", divide="ignore"):
            th = Skd / Nk[:, None].astype(np.float64)
        assert np.array_equal(TH[:, :, r], th, equal_nan=True), "collapsed theta, chain %d sweep %d" % (chain, j)
        st = R.Stream(seed, chain, j, R.ST_ALPHA, 0)
        al = AL[r - 1] if alpha0 != 0 else R.update_alpha_seq(st, AL[r - 1], a, b, N, K)
        if st.near:
            t.near += 1
        else:
            np.testing.assert_allclose(AL[r], al, rtol=1e-12, atol=0, err_msg="alpha, chain %d sweep %d" % (chain, j))
        z_prev = z
    if tally is None:
        t.finish("chain %d" % chain)
    return t


# ---------------------------------------------------------------------------------------------------------------
# chain path (kern_full.cu): one chain per block
# ---------------------------------------------------------------------------------------------------------------
CHAIN_RUNS = {
    # id: (threads, stickbreaking, relabel, alpha, K, data, seed, chain_offset)
    "t32_full": (32, False, False, None, 3, "K3_N1000_P5", SEED_HI, 5),
    "t64_full_relabel": (64, False, True, None, 3, "K3_N1000_P5", 7, 0),
    "t128_full": (128, False, False, None, 3, "K3_N1000_P5", 12, 3),
    "t32_sb": (32, True, False, None, 5, "K2_N1000_P5", 21, 1),
    "t64_sb_relabel_fixed_alpha": (64, True, True, 1.0, 4, "K2_N1000_P5", SEED_HI, 9),
    "t128_sb": (128, True, False, None, 6, "K3_N1000_P5", (1 << 40) | 3, 2),
    "t128_K1": (128, False, False, 0.7, 1, "K2_N100_P5", 4, 0),
    "t64_no_hist_P20": (64, False, False, None, 4, ("syn", 1000, 20), SEED_HI, 6),
    "t128_no_hist_P20_sb": (128, True, False, None, 4, ("syn", 1000, 20), 8, 0),
    "t32_P33": (32, False, False, None, 3, ("syn", 500, 33), 13, 11),
    "t64_P33_sb": (64, True, False, 2.0, 3, ("syn", 500, 33), SEED_HI, 0),
}


@pytest.mark.parametrize("run", list(CHAIN_RUNS))
def test_chain_path_draws(datasets, monkeypatch, run):
    """BMM_FULL_THREADS = 32 / 64 / 128 (the 64-thread entry point relabels on warp 1 beside the draws of warp 0),
    alpha sampled and fixed, K = 1, the non-histogram branch (U K > 3072) and P = 33 (two bit words per row)."""
    _need_gpu()
    threads, sb, relabel, alpha, K, data, seed, off = CHAIN_RUNS[run]
    X = datasets[data] if isinstance(data, str) else _synthetic(data[1], data[2], 4, 17)
    N, P = X.shape
    chains, ns = 2, 6
    monkeypatch.setenv("BMM_FULL_THREADS", str(threads))
    ip, th = _init(chains, K, P, seed & 0xFFFF)
    fn = B.gibbs_stickbreaking if sb else B.gibbs_full
    burnin = 2 if relabel else 0       # relabelling needs a burn-in window of >= 1 sweep before it
    res = fn(X, ns, K, alpha=alpha, burnin=burnin, relabel=relabel, burnrelabel=1, chains=chains, seed=seed,
             chain_offset=off, initial_pi=ip, initial_theta=th)
    t = Tally()
    for c in range(chains):
        check_uncollapsed(_chain(res, c), X, K, seed=seed, chain=off + c, stickbreaking=sb, alpha0=alpha or 0.0,
                          delta=DELTA64, relabel=relabel, tally=t, burnin=burnin)
    t.finish(run)


def test_chain_path_1024_chains(datasets, monkeypatch):
    """The C2 configuration: 1024 chains of gibbs_full on K3_N1000_P5, where the library picks the 64-thread entry
    point capped at 144 registers.  Every chain's allocations; parameters of 16 chains, the first and the last included."""
    _need_gpu()
    monkeypatch.delenv("BMM_FULL_THREADS", raising=False)
    X = datasets["K3_N1000_P5"]
    N, P = X.shape
    K, chains, ns, seed = 3, 1024, 4, 2025
    ip, th = _init(chains, K, P, 99)
    res = B.gibbs_full(X, ns, K, burnin=0, chains=chains, seed=seed, initial_pi=ip, initial_theta=th)
    with_params = set(np.linspace(0, chains - 1, 16).astype(int).tolist())
    assert {0, chains - 1} <= with_params
    t = Tally()
    for c in range(chains):
        check_uncollapsed(_chain(res, c), X, K, seed=seed, chain=c, stickbreaking=False, alpha0=0.0, delta=DELTA64,
                          params=c in with_params, tally=t)
    t.finish("1024 chains")


# ---------------------------------------------------------------------------------------------------------------
# grid paths (kern_big.cu, kern_big_ws.cu, kern_big_lp.cu): one chain over the whole GPU
# ---------------------------------------------------------------------------------------------------------------
GRID_RUNS = {
    # id: (N, P, K, stickbreaking, precision, no_tensor, max_ctas, seed, chain_offset, alpha)
    "fp64_full": (3001, 20, 5, False, "fp64", False, None, SEED_HI, 3, None),
    "fp64_sb": (2003, 9, 6, True, "fp64", False, None, 5, 0, None),
    "fp32_cudacore_full": (3001, 20, 5, False, "fp32", True, None, 6, 1, None),
    "fp32_cudacore_sb_P33": (2003, 33, 6, True, "fp32", True, None, SEED_HI, 0, 1.5),
    "ws_sb_20077_64_32": (20077, 64, 32, True, "fp32", False, None, SEED_HI, 2, None),
    "ws_full_12003_20_7": (12003, 20, 7, False, "fp32", False, None, 14, 0, None),
    "ws_full_12003_20_7_3ctas": (12003, 20, 7, False, "fp32", False, 3, 14, 0, None),
    "lp_3077_512_100": (3077, 512, 100, False, "fp32", False, None, SEED_HI, 1, None),
    "lp_900_33_128": (900, 33, 128, False, "fp32", False, None, 15, 0, None),
}


@pytest.mark.parametrize("run", list(GRID_RUNS))
def test_grid_path_draws(monkeypatch, run):
    """fp64 and fp32 CUDA-core grid kernels, the tcgen05 z-sweep (also with many tiles per CTA) and the large-P / K
    tcgen05 sweep: allocations at the transcribed uniforms and every parameter draw of the update kernel."""
    _need_gpu()
    N, P, K, sb, prec, no_tensor, ctas, seed, off, alpha = GRID_RUNS[run]
    if ctas:
        monkeypatch.setenv("BMM_GRID_MAX_CTAS", str(ctas))
    X = _synthetic(N, P, min(K, 12), 31)
    ns = 3 if P * K > 10000 else 5
    ip, th = _init(1, K, P, 32)
    fn = B.gibbs_stickbreaking if sb else B.gibbs_full
    res = fn(X, ns, K, alpha=alpha, burnin=0, seed=seed, chain_offset=off, initial_pi=ip[0], initial_theta=th[0],
             grid_path=True, precision=prec, no_tensor=no_tensor)
    tensor = prec == "fp32" and not no_tensor
    check_uncollapsed(res, X, K, seed=seed, chain=off, stickbreaking=sb, alpha0=alpha or 0.0,
                      delta=DELTA64 if prec == "fp64" else DELTA32, float_u=tensor).finish(run)


# ---------------------------------------------------------------------------------------------------------------
# collapsed samplers (kern_collapsed.cu)
# ---------------------------------------------------------------------------------------------------------------
COLLAPSED_RUNS = {
    # id: (BMM_COLLAPSED_KERNEL, precision, K, data, relabel, alpha, seed)
    "generic": ("generic", "fp64", 3, "K3_N1000_P5", False, None, SEED_HI),
    "generic_relabel": ("generic", "fp64", 4, "K3_N1000_P5", True, None, 3),
    "log": ("log", "fp64", 3, "K3_N1000_P5", False, None, 4),
    "prod_fp64": (None, "fp64", 3, "K3_N1000_P5", False, None, SEED_HI),
    "prod_fp64_K12": (None, "fp64", 12, "K2_N1000_P5", False, 2.0, 5),
    "prod_fp32": (None, "fp32", 3, "K3_N1000_P5", False, None, 6),
    "prod_fp32_K12": (None, "fp32", 12, "K3_N1000_P5", False, None, SEED_HI),
    "K72": (None, "fp64", 72, "K3_N1000_P5", False, None, 7),
}


@pytest.mark.parametrize("run", list(COLLAPSED_RUNS))
def test_collapsed_draws(datasets, monkeypatch, run):
    """Generic, log-form and product-form (fp64, fp32) kernels and K = 72 (two labels per lane)."""
    _need_gpu()
    kern, prec, K, data, relabel, alpha, seed = COLLAPSED_RUNS[run]
    if kern:
        monkeypatch.setenv("BMM_COLLAPSED_KERNEL", kern)
    else:
        monkeypatch.delenv("BMM_COLLAPSED_KERNEL", raising=False)
    X = datasets[data]
    N = X.shape[0]
    chains, ns, off = 2, 5, 4
    z0 = np.random.default_rng(seed & 0xFFFF).integers(1, K + 1, (chains, N)).astype(np.int32)
    burnin = 2 if relabel else 0
    res = B.gibbs_collapsed(X, ns + burnin, K, alpha=alpha, burnin=burnin, relabel=relabel, burnrelabel=1, chains=chains,
                            seed=seed, chain_offset=off, initial_K=z0, precision=prec)
    t = Tally()
    for c in range(chains):
        check_collapsed(_chain(res, c), X, K, z0[c], seed=seed, chain=off + c, alpha0=alpha or 0.0, burnin=burnin,
                        delta=DELTA_C32 if prec == "fp32" else DELTA64, fp32=prec == "fp32", relabel=relabel, tally=t)
    t.finish(run)


DP_RUNS = {
    # id: (BMM_DP_LOGFORM, maxK, data, alpha, seed)
    "product": (None, 30, "K3_N1000_P5", None, SEED_HI),
    "product_fixed_alpha": (None, 30, "K2_N100_P5", 1.5, 8),
    "logform": ("1", 30, "K3_N1000_P5", None, 9),
}


@pytest.mark.parametrize("run", list(DP_RUNS))
def test_dp_draws(datasets, monkeypatch, run):
    """DP / CRP sampler, product and log form: every update drawn from the float64 conditional over the used-list
    order plus the new cluster (smallest free label), theta = S / N for the used labels, alpha with K = used clusters."""
    _need_gpu()
    logform, maxK, data, alpha, seed = DP_RUNS[run]
    if logform:
        monkeypatch.setenv("BMM_DP_LOGFORM", logform)
    else:
        monkeypatch.delenv("BMM_DP_LOGFORM", raising=False)
    X = datasets[data]
    N, P = X.shape
    chains, ns, off = 2, 5, 6
    res = B.gibbs_dp(X, ns, alpha=alpha, burnin=0, maxK=maxK, chains=chains, seed=seed, chain_offset=off)
    t = Tally()
    for c in range(chains):
        r, chain = _chain(res, c), off + c
        Z, TH, AL = r["z"], r["theta"], r["alpha"][:, 0]
        st = R.DPState(X, maxK)
        for j in range(1, ns):
            z = Z[j].astype(np.int64) - 1
            prob, pos = st.sweep(j, z, AL[j - 1], 0.5, 0.5)
            miss = np.nonzero(pos < 0)[0]
            assert len(miss) == 0, "chain %d sweep %d: row %d drew label %d, not in the used list nor the new one" % (
                chain, j, miss[0], z[miss[0]])
            _check_z(prob, R.z_uniforms_collapsed(seed, chain, j, N), pos, DELTA64, t, "chain %d sweep %d" % (chain, j))
            t.sweeps += 1
            used = np.array(sorted(st.used))
            assert np.array_equal(TH[used, :, j], st.S[used] / st.Nk[used, None].astype(np.float64))
            s_a = R.Stream(seed, chain, j, R.ST_ALPHA, 0)
            al = AL[j - 1] if alpha else R.update_alpha_seq(s_a, AL[j - 1], 1.0, 1.0, N, len(st.used))
            if s_a.near:
                t.near += 1
            else:
                np.testing.assert_allclose(AL[j], al, rtol=1e-12, atol=0, err_msg="alpha, chain %d sweep %d" % (chain, j))
    t.finish(run)


# ---------------------------------------------------------------------------------------------------------------
# the top of the uniform range: a cluster of weight 0 must never be drawn
# ---------------------------------------------------------------------------------------------------------------
TOP_SEED, TOP_N, TOP_SWEEPS = 9, 20077, 8
# chain offsets whose sweeps 1..7 draw words >= 0xFFFFFF00 (333, 919 at sweep 1) and >= 0xFFFFFFF0 (1839, 5050, 5320)
# for seed 9 and 20 077 rows; found by scanning the transcribed streams, checked again by the test
TOP_OFFSETS = (333, 919, 1839, 5050, 5320)
TOP_PATHS = {"ws": (64, 32, False), "lp": (130, 40, False), "cudacore": (64, 32, True)}


@pytest.mark.parametrize("path", list(TOP_PATHS))
def test_grid_top_of_range_never_draws_empty_cluster(path):
    """pi_K = 0 (kept at 0 by alpha = 1e-300: its Gamma(alpha / K) draw underflows), rows whose uniform is within 2^-24
    of 1 (and, for the float CUDA-core kernel, within 4e-9, where its float prefix sum can fall short of u): no row
    may draw cluster K.  A float uniform of exactly 1, or a draw that runs past the last cluster with weight, put
    every such row on cluster K."""
    _need_gpu()
    P, K, no_tensor = TOP_PATHS[path]
    X = _synthetic(TOP_N, P, 8, 41)
    ip, th = _init(1, K, P, 42, zero_last=True)
    n8 = n4 = 0
    for off in TOP_OFFSETS:
        w = np.stack([R.z_words_rows(TOP_SEED, off, j, np.arange(TOP_N)) for j in range(1, TOP_SWEEPS)])
        n8 += int((w >= 0xFFFFFF00).sum())
        n4 += int((w >= 0xFFFFFFF0).sum())
        res = B.gibbs_full(X, TOP_SWEEPS, K, alpha=1e-300, burnin=0, seed=TOP_SEED, chain_offset=off, initial_pi=ip[0],
                           initial_theta=th[0], grid_path=True, precision="fp32", no_tensor=no_tensor)
        z = res["z"][1:]
        top = np.nonzero(w >= 0xFFFFFF00)
        assert not (z == K).any(), "chain offset %d: %d rows drew the empty cluster K (rows with top words: %s, their z: %s)" % (
            off, int((z == K).sum()), list(zip(*top)), z[top].tolist())
        assert (res["pi"][:, K - 1] == 0).all()
    print("%s: %d rows with words >= 0xFFFFFF00, %d >= 0xFFFFFFF0" % (path, n8, n4))
    assert n8 >= 2 and (n4 >= 2 or not no_tensor)


# chains whose sweeps 1..10 hold an update with w0 >= 0xFFFFFF80 (u53 >= 1 - 2^-25: 1.0 once cast to float) for
# seed 31 and N = 1000: chain 9598 at sweep 6, 15800 and 36060 at sweep 1
TOP_C_SEED, TOP_C_CHAINS, TOP_C_SWEEPS = 31, (9598, 15800, 36060), 11


@pytest.mark.parametrize("kern,prec,K", [(None, "fp32", 3), (None, "fp32", 6), (None, "fp64", 3), ("log", "fp64", 3),
                                         ("generic", "fp64", 3), ("generic", "fp64", 6)])
def test_collapsed_top_of_range_never_revives_empty_cluster(datasets, monkeypatch, kern, prec, K):
    """initial_K without label K, and an update at the top of the uniform range in every run: an empty cluster has
    probability exactly 0 (collapsed_gibbs.cpp:104,131-133), so label K must never appear."""
    _need_gpu()
    if kern:
        monkeypatch.setenv("BMM_COLLAPSED_KERNEL", kern)
    else:
        monkeypatch.delenv("BMM_COLLAPSED_KERNEL", raising=False)
    X = datasets["K3_N1000_P5"]
    N = X.shape[0]
    z0 = np.random.default_rng(K).integers(1, K, N).astype(np.int32)      # labels 1 .. K-1
    for ch in TOP_C_CHAINS:
        hits = 0
        for j in range(1, TOP_C_SWEEPS):
            r = R.philox(np.arange(N // 2), 0, 0, j, TOP_C_SEED, ch)
            hits += int((r[:, 0] >= 0xFFFFFF80).sum() + (r[:, 2] >= 0xFFFFFF80).sum())
        assert hits >= 1
        res = B.gibbs_collapsed(X, TOP_C_SWEEPS, K, burnin=0, seed=TOP_C_SEED, chain_offset=ch, initial_K=z0[None],
                                precision=prec)
        assert not (res["z"][1:] == K).any(), "chain %d: label %d revived in sweeps %s" % (
            ch, K, np.nonzero((res["z"][1:] == K).any(1))[0] + 1)
