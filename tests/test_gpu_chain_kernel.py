"""chain_sweep_kernel (the specialised Philox-mode sweep of kern_full.cu) against full_chain_kernel, bit for bit.

Each test runs one plan twice, once with BMM_CHAIN_KERNEL=generic (full_chain_kernel) and once with the library's own
choice, and asserts that every returned array -- z, z_original, theta, theta_original, pi, alpha, permutations, status
-- is identical.  The Philox draw tests check full_chain_kernel against the float64 transcription of its streams; this
file carries that check over to the specialised kernel.
"""
import ctypes as C

import numpy as np
import pytest

import bmm_mcmc_b200 as B
from bmm_mcmc_b200 import _lib
from conftest import gpu_available
from test_gpu_philox_draws import CHAIN_RUNS, _init, _synthetic

pytestmark = pytest.mark.gpu

GENERIC, SWEEP = 1, 2


def _need_gpu():
    assert gpu_available(), "CUDA library/device unavailable: " + repr(_lib.LIB_PATH)


def _kernel():
    return _lib.lib().bmm_debug_chain_kernel()


def _both(monkeypatch, fn, *args, **kw):
    """(generic result, default result, kernel the default run picked)"""
    monkeypatch.setenv("BMM_CHAIN_KERNEL", "generic")
    ref = fn(*args, **kw)
    assert _kernel() == GENERIC
    monkeypatch.delenv("BMM_CHAIN_KERNEL")
    got = fn(*args, **kw)
    return ref, got, _kernel()


def _assert_same(ref, got, where):
    assert sorted(ref) == sorted(got)
    for k in ref:
        a, b = np.asarray(ref[k]), np.asarray(got[k])
        assert a.dtype == b.dtype and a.shape == b.shape, "%s: %s shape/dtype" % (where, k)
        if a.dtype.kind == "f":   # bitwise: the same NaN and the same sign of zero as well
            a, b = np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8)
        if not np.array_equal(a, b):
            bad = np.argwhere(a != b)
            pytest.fail("%s: %s differs at %d entries, first %s" % (where, k, len(bad), bad[:3].tolist()))


@pytest.fixture(scope="module")
def data():
    return {name: B.load_dataset(name) for name in ("K2_N100_P5", "K2_N1000_P5", "K3_N1000_P5")}


@pytest.mark.parametrize("threads", [32, 64, 128])
@pytest.mark.parametrize("run", list(CHAIN_RUNS))
def test_sweep_kernel_matches_generic(data, monkeypatch, run, threads):
    """Every chain configuration of the Philox draw tests at each block size: full and stick-breaking, relabelling,
    alpha fixed and sampled, K = 1, P = 33; the non-histogram configurations (U K > 3072) keep the generic kernel."""
    _need_gpu()
    _, sb, relabel, alpha, K, d, seed, off = CHAIN_RUNS[run]
    X = data[d] if isinstance(d, str) else _synthetic(d[1], d[2], 4, 17)
    N, P = X.shape
    chains, ns = 3, 14
    monkeypatch.setenv("BMM_FULL_THREADS", str(threads))
    ip, th = _init(chains, K, P, seed & 0xFFFF)
    fn = B.gibbs_stickbreaking if sb else B.gibbs_full
    burnin = 5 if relabel else 0
    ref, got, kern = _both(monkeypatch, fn, X, ns, K, alpha=alpha, burnin=burnin, relabel=relabel, burnrelabel=3,
                           chains=chains, seed=seed, chain_offset=off, initial_pi=ip, initial_theta=th)
    assert kern == (GENERIC if "no_hist" in run else SWEEP)
    _assert_same(ref, got, "%s, %d threads" % (run, threads))


@pytest.mark.parametrize("sb", [False, True])
@pytest.mark.parametrize("threads", [32, 64, 128])
def test_sweep_kernel_fixed_stephens_odd_n(monkeypatch, threads, sb):
    """BMM_FLAG_STEPHENS_FIXED, P = 33 (two words per row), N % 4 != 0 (byte-wise label stores), more than 256 distinct
    rows (16-bit row ids), stable softmax."""
    _need_gpu()
    X = _synthetic(1003, 33, 4, 5)
    N, P = X.shape
    K, chains = 3, 3
    monkeypatch.setenv("BMM_FULL_THREADS", str(threads))
    ip, th = _init(chains, K, P, 77)
    fn = B.gibbs_stickbreaking if sb else B.gibbs_full
    ref, got, kern = _both(monkeypatch, fn, X, 16, K, burnin=6, relabel=True, burnrelabel=4, chains=chains, seed=1234,
                           chain_offset=2, initial_pi=ip, initial_theta=th, stephens_fixed=True, stable_softmax=True)
    assert kern == SWEEP
    _assert_same(ref, got, "fixed Stephens, %d threads, stick-breaking %s" % (threads, sb))


def test_sweep_kernel_c2(data, monkeypatch):
    """The benchmark's configuration: 1024 chains of gibbs_full on K3_N1000_P5, K = 3, relabelling with burnin 200 and
    burnrelabel 50, 400 kept sweeps in three download segments; the library picks the specialised kernel."""
    _need_gpu()
    monkeypatch.delenv("BMM_FULL_THREADS", raising=False)
    monkeypatch.setenv("BMM_FETCH_SEGMENTS", "3")
    X = data["K3_N1000_P5"]
    ref, got, kern = _both(monkeypatch, B.gibbs_full, X, 600, 3, burnin=200, relabel=True, burnrelabel=50, chains=1024,
                           seed=2025)
    assert kern == SWEEP
    _assert_same(ref, got, "C2")


def test_chain_kernel_switch_and_phase_query():
    """bmm_debug_chain_phases needs a -DBMM_CHAIN_PHASE_CLOCKS build; the default build reports BMM_ERR_UNSUPPORTED."""
    _need_gpu()
    buf = (C.c_uint64 * 8)()
    assert _lib.lib().bmm_debug_chain_phases(buf, 8) == -8
