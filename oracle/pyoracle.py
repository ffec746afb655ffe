"""ctypes binding of the CPU oracle (oracle/liboracle.so).

TEST INFRASTRUCTURE: import only from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package (bmm_mcmc_b200) never imports this.

All arrays follow R's column-major layout; histories are returned at full length (nsamples)
plus `tail()` helpers that apply the reference's return-block slicing
(full_gibbs.cpp:233-248 etc.).
"""
import ctypes as C
import os
import subprocess
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class OracleOut(C.Structure):
    _fields_ = [
        ("pi", C.POINTER(C.c_double)), ("alpha", C.POINTER(C.c_double)),
        ("permutations", C.POINTER(C.c_int)), ("z", C.POINTER(C.c_int)), ("z_rel", C.POINTER(C.c_int)),
        ("theta", C.POINTER(C.c_double)), ("theta_rel", C.POINTER(C.c_double)),
        ("u_rec", C.POINTER(C.c_double)), ("u_slots", C.c_int),
        ("probs", C.POINTER(C.c_double)), ("loglik", C.POINTER(C.c_double)),
        ("Q_final", C.POINTER(C.c_double)), ("Kactive", C.POINTER(C.c_int)),
    ]


def build(force=False):
    so = os.path.join(_HERE, "liboracle.so")
    src = [os.path.join(_HERE, f) for f in ("oracle.cpp", "rrng.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["make", "-C", _HERE, "liboracle.so"], stdout=subprocess.DEVNULL)
    opt = os.path.join(_HERE, "libopt_cpu.so")
    if force or not os.path.exists(opt) or os.path.getmtime(os.path.join(_HERE, "opt_cpu.cpp")) > os.path.getmtime(opt):
        subprocess.check_call(["make", "-C", _HERE, "libopt_cpu.so"], stdout=subprocess.DEVNULL)
    ref_out = [os.path.join(_HERE, "_ref", f) for f in ("liblpsolve_ref.so", "libbmm_ref.so")]
    ref_src = [os.path.join(_HERE, "build_ref.sh"), os.path.join(_HERE, "rrng.h")] + \
        [os.path.join(_HERE, "shim", f) for f in ("RcppArmadillo.h", "ref_capi.cpp", "RcppArmadilloExtensions/sample.h")]
    if os.path.isdir("/root/reference/src") and (
            force or not all(os.path.exists(f) for f in ref_out)
            or any(os.path.getmtime(s) > min(os.path.getmtime(f) for f in ref_out) for s in ref_src)):
        subprocess.check_call(["sh", os.path.join(_HERE, "build_ref.sh")], stdout=subprocess.DEVNULL)
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.oracle_has_lpsolve_ref.restype = C.c_int
    return _LIB


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int)) if a is not None else None


def has_ref():
    return bool(lib().oracle_has_lpsolve_ref())


def _use_ref(use_ref):
    """use_ref=None: the reference's lp_solve when oracle/_ref is built, else the exact Hungarian solver.  Both return
    the unique optimum of a cost matrix without ties; only True insists on lp_solve (and its tie-break)."""
    return int(has_ref() if use_ref is None else bool(use_ref))


def assign(cost, use_ref=None):
    """my_lpsolve: K x K cost -> K x K 0/1 solution."""
    cost = np.asfortranarray(cost, dtype=np.float64)
    K = cost.shape[0]
    sol = np.zeros((K, K), dtype=np.int32, order="F")
    rc = lib().oracle_assign(K, _dp(cost), _ip(sol), _use_ref(use_ref))
    if rc:
        raise RuntimeError("oracle_assign rc=%d" % rc)
    return sol


def set_stephens_fixed(on):
    """Correctness-fixed Stephens mode (SURVEY 8f-3): real threshold, inverse permutation for the column
    re-ordering, log p in the online cost, running-mean Q.  Process-wide switch; the default (off) is the
    reference's behaviour."""
    lib().oracle_set_stephens_fixed(int(bool(on)))


def set_sample_stable(on):
    """DP sampler: tie order of sample()'s descending sort.  Off (default) = std::sort like the reference build
    (stable up to 16 candidates); on = stable for every candidate count.  Process-wide switch."""
    lib().oracle_set_sample_stable(int(bool(on)))


def stephens_batch(p, use_ref=None):
    p = np.asfortranarray(p, dtype=np.float64)
    N, K, M = p.shape
    q = np.zeros((N, K), order="F")
    perm = np.zeros((M, K), dtype=np.int32, order="F")
    rc = lib().oracle_stephens_batch(N, K, M, _dp(p), _dp(q), _use_ref(use_ref), _ip(perm))
    if rc:
        raise RuntimeError("oracle_stephens_batch rc=%d" % rc)
    return q, perm


def stephens_online(q, p, sample_num, use_ref=None):
    q = np.asfortranarray(q, dtype=np.float64)
    p = np.asfortranarray(p, dtype=np.float64)
    N, K = p.shape
    perm = np.zeros(K, dtype=np.int32)
    qn = np.zeros((N, K), order="F")
    cost = np.zeros((K, K), order="F")
    rc = lib().oracle_stephens_online(N, K, _dp(q), _dp(p), int(sample_num), _ip(perm), _dp(qn), _use_ref(use_ref), _dp(cost))
    if rc:
        raise RuntimeError("oracle_stephens_online rc=%d" % rc)
    return perm, qn, cost


def unif_rand(seed, n):
    out = np.zeros(n)
    lib().oracle_unif_rand(C.c_uint(seed), n, _dp(out))
    return out


def rbinom1_blocks(seed, counts, ps):
    counts = np.asarray(counts, dtype=np.int32)
    ps = np.asarray(ps, dtype=np.float64)
    out = np.zeros(int(counts.sum()), dtype=np.int32)
    lib().oracle_rbinom1(C.c_uint(seed), len(counts), _ip(counts), _dp(ps), _ip(out))
    return out


def rmultinom1(seed, prob):
    prob = np.asarray(prob, dtype=np.float64)
    K = len(prob)
    rN = np.zeros(K, dtype=np.int32)
    u = np.full(K, -1.0)
    n = C.c_int(0)
    rc = lib().oracle_rmultinom1_seeded(C.c_uint(seed), _dp(prob), K, _ip(rN), _dp(u), C.byref(n))
    return rc, rN, u[:n.value]


def rdirichlet(seed, alpha_m):
    alpha_m = np.asarray(alpha_m, dtype=np.float64)
    out = np.zeros(len(alpha_m))
    lib().oracle_rdirichlet(C.c_uint(seed), len(alpha_m), _dp(alpha_m), _dp(out))
    return out


def rgamma(seed, n, shape, scale=1.0):
    out = np.zeros(n)
    lib().oracle_rgamma(C.c_uint(seed), n, C.c_double(shape), C.c_double(scale), _dp(out))
    return out


def rbeta(seed, n, a, b):
    out = np.zeros(n)
    lib().oracle_rbeta(C.c_uint(seed), n, C.c_double(a), C.c_double(b), _dp(out))
    return out


class Result(dict):
    """Full-length histories (R layout).  `tail()` gives the reference's returned list."""

    def tail(self):
        ns, burnin, relabel = self["nsamples"], self["burnin"], self["relabel"]
        out = {}
        if "pi" in self:
            out["pi"] = self["pi"][burnin:, :]
        out["alpha"] = self["alpha"][burnin:].reshape(-1, 1)
        out["permutations"] = self["permutations"]
        th = self["theta"][:, :, burnin:]
        if relabel:
            out["z"] = self["z_rel"][burnin:, :]
            out["theta"] = self["theta_rel"][:, :, burnin:]
            out["z_original"] = self["z"][burnin:, :]
            out["theta_original"] = th
        else:
            out["z"] = self["z"][burnin:, :]
            out["theta"] = th
        return out


def _alloc(N, P, K, nsamples, burnin, slots, want_pi, probes):
    r = Result()
    r["alpha"] = np.zeros(nsamples)
    r["permutations"] = np.zeros((max(nsamples - burnin, 0), K), dtype=np.int32, order="F")
    r["z"] = np.zeros((nsamples, N), dtype=np.int32, order="F")
    r["z_rel"] = np.zeros((nsamples, N), dtype=np.int32, order="F")
    r["theta"] = np.zeros((K, P, nsamples), order="F")
    r["theta_rel"] = np.zeros((K, P, nsamples), order="F")
    r["u_rec"] = np.full((nsamples, N, max(slots, 1)), -1.0)  # C order: slot fastest
    r["Q_final"] = np.zeros((N, K), order="F")
    if want_pi:
        r["pi"] = np.zeros((nsamples, K), order="F")
    if probes:
        r["probs"] = np.zeros((nsamples, N, K)).transpose(0, 1, 2)  # [j] blocks of N x K col-major, see below
        r["probs"] = np.zeros((nsamples, K, N)).transpose(0, 2, 1)  # shape (ns, N, K); element (j,i,k) at j*N*K + i + N*k
        r["loglik"] = np.zeros((nsamples, K, N)).transpose(0, 2, 1)
    o = OracleOut()
    o.pi = _dp(r.get("pi"))
    o.alpha = _dp(r["alpha"])
    o.permutations = _ip(r["permutations"])
    o.z = _ip(r["z"])
    o.z_rel = _ip(r["z_rel"])
    o.theta = _dp(r["theta"])
    o.theta_rel = _dp(r["theta_rel"])
    o.u_rec = _dp(r["u_rec"])
    o.u_slots = max(slots, 1)
    if probes:
        o.probs = C.cast(r["probs"].base.ctypes.data, C.POINTER(C.c_double))
        o.loglik = C.cast(r["loglik"].base.ctypes.data, C.POINTER(C.c_double))
    o.Q_final = _dp(r["Q_final"])
    return r, o


def _df(X):
    return np.asfortranarray(X, dtype=np.int32)


def gibbs_full(X, initial_pi, initial_theta, nsamples, K, alpha=0.0, beta=0.5, gamma=0.5, a=1.0, b=1.0,
               burnin=None, relabel=False, burnrelabel=50, seed=1, use_ref=None, probes=True, stabilise=False,
               stickbreaking=False):
    X = _df(X)
    N, P = X.shape
    if burnin is None:
        burnin = int(round(0.1 * nsamples))
    r, o = _alloc(N, P, K, nsamples, burnin, K - 1, True, probes)
    ipi = np.asarray(initial_pi, dtype=np.float64)
    ith = np.asfortranarray(initial_theta, dtype=np.float64)
    fn = lib().oracle_gibbs_stickbreaking if stickbreaking else lib().oracle_gibbs_full
    rc = fn(_ip(X), N, P, _dp(ipi), _dp(ith), nsamples, K, C.c_double(alpha), C.c_double(beta), C.c_double(gamma),
            C.c_double(a), C.c_double(b), burnin, int(relabel), burnrelabel, C.c_uint(seed), _use_ref(use_ref),
            int(stabilise), C.byref(o))
    if rc:
        raise RuntimeError("oracle sampler rc=%d" % rc)
    r.update(nsamples=nsamples, burnin=burnin, relabel=relabel)
    return r


def gibbs_stickbreaking(X, initial_pi, initial_theta, nsamples, maxK, **kw):
    return gibbs_full(X, initial_pi, initial_theta, nsamples, maxK, stickbreaking=True, **kw)


def gibbs_collapsed(X, initial_K, nsamples, K, alpha=0.0, beta=0.5, gamma=0.5, a=1.0, b=1.0, burnin=None,
                    relabel=False, burnrelabel=50, seed=1, use_ref=None, probes=True):
    X = _df(X)
    N, P = X.shape
    if burnin is None:
        burnin = int(round(0.1 * nsamples))
    r, o = _alloc(N, P, K, nsamples, burnin, K - 1, False, probes)
    iz = np.asarray(initial_K, dtype=np.int32)
    rc = lib().oracle_gibbs_collapsed(_ip(X), N, P, _ip(iz), nsamples, K, C.c_double(alpha), C.c_double(beta),
                                      C.c_double(gamma), C.c_double(a), C.c_double(b), burnin, int(relabel),
                                      burnrelabel, C.c_uint(seed), _use_ref(use_ref), C.byref(o))
    if rc:
        raise RuntimeError("oracle sampler rc=%d" % rc)
    r.update(nsamples=nsamples, burnin=burnin, relabel=relabel)
    return r


def gibbs_dp(X, nsamples, alpha=0.0, beta=0.5, gamma=0.5, a=1.0, b=1.0, burnin=None, relabel=False,
             burnrelabel=50, maxK=30, seed=1, use_ref=None, probes=True):
    X = _df(X)
    N, P = X.shape
    if burnin is None:
        burnin = int(round(0.1 * nsamples))
    r, o = _alloc(N, P, maxK, nsamples, burnin, 1, False, probes)
    r["Kactive"] = np.zeros(nsamples, dtype=np.int32)
    o.Kactive = _ip(r["Kactive"])
    rc = lib().oracle_gibbs_dp(_ip(X), N, P, nsamples, C.c_double(alpha), C.c_double(beta), C.c_double(gamma),
                               C.c_double(a), C.c_double(b), burnin, int(relabel), burnrelabel, maxK,
                               C.c_uint(seed), _use_ref(use_ref), C.byref(o))
    if rc:
        raise RuntimeError("oracle sampler rc=%d" % rc)
    r.update(nsamples=nsamples, burnin=burnin, relabel=relabel)
    return r


def opt_cpu_full_gibbs(X, K, nsamples, burnin, chains, threads):
    """Bench baseline (oracle/opt_cpu.cpp): `chains` chains of the count-maintaining, row-deduplicated CPU sampler with
    online relabelling on `threads` host threads; returns wall seconds."""
    import ctypes as C
    build()
    L = C.CDLL(os.path.join(_HERE, "libopt_cpu.so"))
    L.opt_cpu_full_gibbs.restype = C.c_double
    L.opt_cpu_full_gibbs.argtypes = [C.c_void_p] + [C.c_int] * 7
    Xf = np.asfortranarray(X, dtype=np.int32)
    s = L.opt_cpu_full_gibbs(Xf.ctypes.data, Xf.shape[0], Xf.shape[1], int(K), int(nsamples), int(burnin), int(chains), int(threads))
    if s < 0:
        raise RuntimeError("opt_cpu_full_gibbs: unsupported shape")
    return s


def opt_cpu_collapsed_gibbs(X, K, nsamples, chains, threads):
    """Bench baseline (oracle/opt_cpu.cpp): count-maintaining collapsed sampler in product form; returns wall seconds."""
    import ctypes as C
    build()
    L = C.CDLL(os.path.join(_HERE, "libopt_cpu.so"))
    L.opt_cpu_collapsed_gibbs.restype = C.c_double
    L.opt_cpu_collapsed_gibbs.argtypes = [C.c_void_p] + [C.c_int] * 6
    Xf = np.asfortranarray(X, dtype=np.int32)
    s = L.opt_cpu_collapsed_gibbs(Xf.ctypes.data, Xf.shape[0], Xf.shape[1], int(K), int(nsamples), int(chains), int(threads))
    if s < 0:
        raise RuntimeError("opt_cpu_collapsed_gibbs: unsupported shape")
    return s
