"""Host-side mirror of the reference's R user API (R/utils.R:23-107) over the C ABI.

Same function names, argument names, defaults and returned list layout as the R package:
`gibbs_full`, `gibbs_collapsed`, `gibbs_dp`, `gibbs_stickbreaking`.  The returned dict has the
R list's names and shapes (`pi` S x K, `alpha` S x 1, `permutations` S x K, `z` S x N,
`theta` K x P x S, and with `relabel=True` also `z_original`, `theta_original`); labels in `z`
are 1-based like R's.  Extra keyword-only arguments (`chains`, `seed`, `device`, ...) default to the
reference's behaviour; with `chains > 1` every array gains a leading chain axis.

The initial state is drawn on the host like the R wrappers do (R/utils.R:42,68-74,98-103), with an
R-compatible Mersenne-Twister (`rcompat.RRng`) so `seed=s` plays the role of `set.seed(s)`.
All sampling runs in the CUDA library; there is no CPU fallback.
"""
import ctypes as C
import numpy as np

from . import _lib
from .rcompat import RRng

__all__ = ["gibbs_full", "gibbs_collapsed", "gibbs_dp", "gibbs_stickbreaking", "predictive", "waic", "loo", "loglik_matrix", "Plan",
           "PackedX"]


def _r_round(x):
    return int(round(x))  # R's round() and Python's are both half-to-even


class PackedX:
    """Bit-packed observations for the grid path (BMM_FLAG_X_PACKED): uint32 [N][ceil(P/32)], bit d%32
    of word d//32 of row i is x_id.  `PackedX.pack(X)` packs a 0/1 matrix."""

    def __init__(self, bits, P):
        self.bits = np.ascontiguousarray(bits, dtype=np.uint32)
        assert self.bits.ndim == 2 and self.bits.shape[1] == (P + 31) // 32
        self.shape = (self.bits.shape[0], int(P))
        self.nbytes = self.bits.nbytes
        self.ctypes = self.bits.ctypes

    @classmethod
    def pack(cls, X):
        X = np.asarray(X)
        N, P = X.shape
        W = (P + 31) // 32
        b = np.zeros((N, W * 32), dtype=np.uint8)
        b[:, :P] = X != 0
        return cls(np.packbits(b, axis=1, bitorder="little").view("<u4").reshape(N, W), P)

    def rows(self, lo, hi):
        return PackedX(self.bits[lo:hi], self.shape[1])


def _as_X(data):
    if isinstance(data, PackedX):
        return data
    X = np.asarray(data)
    if X.ndim != 2:
        raise ValueError("data must be a 2-d matrix (observations x binary variables)")
    if not np.issubdtype(X.dtype, np.integer):
        Xi = X.astype(np.int32)
        if not np.array_equal(Xi, X):
            raise ValueError("data must be integer 0/1")
        X = Xi
    return np.asfortranarray(X, dtype=np.int32)


def _p(arr, typ):
    return arr.ctypes.data_as(C.POINTER(typ)) if arr is not None else None


class _Pinned:
    """numpy arrays over cudaHostAlloc'ed memory (freed when the owner array is collected)."""

    def __init__(self, nbytes):
        self.ptr = C.c_void_p()
        _lib.check(_lib.lib().bmm_host_alloc(int(nbytes), C.byref(self.ptr)))
        self.nbytes = int(nbytes)

    def __del__(self):
        try:
            if self.ptr:
                _lib.lib().bmm_host_free(self.ptr)
        except Exception:
            pass


def _empty(shape, dtype, pinned):
    if not pinned:
        return np.zeros(shape, dtype=dtype)
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    owner = _Pinned(max(n, 1))
    buf = (C.c_char * max(n, 1)).from_address(owner.ptr.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _KEEP[id(buf)] = owner
    import weakref
    weakref.finalize(buf, _KEEP.pop, id(buf), None)
    return arr


_KEEP = {}


def _chain_cm(C_, shape, dtype, pinned=False):
    """Array of shape (C_, *shape) whose per-chain blocks are column-major (R layout)."""
    rev = tuple(reversed(shape))
    base = _empty((C_,) + rev, dtype, pinned)
    axes = (0,) + tuple(range(len(shape), 0, -1))
    return base.transpose(axes)


def _build_args(sampler, X, nsamples, K, alpha, beta, gamma, a, b, burnin, relabel, burnrelabel, debug,
                chains, seed, device, precision, init_pi=None, init_theta=None, init_z=None, replay=None,
                compact_z=False, stable_softmax=False, chain_offset=0, grid_path=False, no_z_history=False,
                n_global=0, row_offset=0, no_tensor=False, stephens_fixed=False, thin=1):
    """ctypes bmm_args / bmm_init for one call; returns (args, init, keepalive)."""
    N, P = X.shape
    args = _lib.Args()
    args.X = _p(X, C.c_int32)
    args.N, args.P, args.nsamples, args.K = N, P, int(nsamples), int(K)
    args.alpha, args.beta, args.gamma, args.a, args.b = float(alpha), float(beta), float(gamma), float(a), float(b)
    args.burnin, args.relabel, args.burnrelabel, args.debug = int(burnin), int(bool(relabel)), int(burnrelabel), int(bool(debug))
    args.n_chains, args.chain_offset, args.seed = int(chains), int(chain_offset), int(seed) & 0xFFFFFFFFFFFFFFFF
    args.precision = {"fp64": _lib.BMM_FP64, "fp32": _lib.BMM_FP32}[precision]
    args.device = int(device)
    args.thin = int(thin)
    args.flags = ((_lib.FLAG_COMPACT_Z if compact_z else 0) | (_lib.FLAG_STABLE_SOFTMAX if stable_softmax else 0) |
                  (_lib.FLAG_GRID_PATH if grid_path else 0) | (_lib.FLAG_NO_Z_HISTORY if no_z_history else 0) |
                  (_lib.FLAG_NO_TENSOR if no_tensor else 0) | (_lib.FLAG_STEPHENS_FIXED if stephens_fixed else 0))
    if isinstance(X, PackedX):
        args.flags |= _lib.FLAG_X_PACKED
    args.n_global, args.row_offset = int(n_global), int(row_offset)
    keep = [X, init_pi, init_theta, init_z]
    if replay is not None:
        rp = _lib.Replay()
        u = np.ascontiguousarray(replay["u"], dtype=np.float64)
        rp.u = _p(u, C.c_double)
        rp.u_slots = int(u.shape[-1])
        keep.append(u)
        for name in ("pi", "theta", "alpha"):
            if replay.get(name) is not None:
                arr = replay[name]
                keep.append(arr)
                setattr(rp, name, _p(arr, C.c_double))
        keep.append(rp)
        args.replay = C.pointer(rp)
    init = _lib.Init()
    if init_pi is not None:
        init.pi = _p(init_pi, C.c_double)
        init.theta = _p(init_theta, C.c_double)
    if init_z is not None:
        init.z = _p(init_z, C.c_int32)
    return args, init, keep


def kept_sweeps(nsamples, burnin, thin=1):
    """Rows of the returned histories: every thin-th post-burn-in sweep (thin = 1: all of them, as the reference)."""
    S = nsamples - burnin
    return (S + thin - 1) // thin if thin > 1 else S


def _alloc_out(sampler, Cn, N, P, K, nsamples, burnin, relabel, compact_z, probes, pinned, no_z=False, thin=1):
    """Caller-side output buffers in the reference's returned-list layout; returns (dict, bmm_out, status)."""
    S = kept_sweeps(nsamples, burnin, thin)
    zt = np.uint8 if compact_z else np.int32
    res = {}
    out = _lib.Out()
    if sampler in (_lib.SAMPLER_FULL, _lib.SAMPLER_STICKBREAKING):
        res["pi"] = _chain_cm(Cn, (S, K), np.float64, pinned)
        out.pi = _p(res["pi"], C.c_double)
    res["alpha"] = _chain_cm(Cn, (S, 1), np.float64, pinned)
    out.alpha = _p(res["alpha"], C.c_double)
    res["permutations"] = _chain_cm(Cn, (S, K), np.int32, pinned)
    out.permutations = _p(res["permutations"], C.c_int32)
    if not no_z:
        res["z"] = _chain_cm(Cn, (S, N), zt, pinned)
        out.z = C.cast(res["z"].ctypes.data, C.POINTER(C.c_int32))
    res["theta"] = _chain_cm(Cn, (K, P, S), np.float64, pinned)
    out.theta = _p(res["theta"], C.c_double)
    if relabel:
        if not no_z:
            res["z_original"] = _chain_cm(Cn, (S, N), zt, pinned)
            out.z_original = C.cast(res["z_original"].ctypes.data, C.POINTER(C.c_int32))
        res["theta_original"] = _chain_cm(Cn, (K, P, S), np.float64, pinned)
        out.theta_original = _p(res["theta_original"], C.c_double)
    if "probs" in probes:
        res["probs"] = np.zeros((Cn, nsamples, K, N)).transpose(0, 1, 3, 2)  # [c][j] blocks of N x K cm
        out.probs = C.cast(res["probs"].ctypes.data, C.POINTER(C.c_double))
    if "loglik" in probes:
        res["loglik"] = np.zeros((Cn, nsamples, K, N)).transpose(0, 1, 3, 2)
        out.loglik = C.cast(res["loglik"].ctypes.data, C.POINTER(C.c_double))
    if "Q_final" in probes and relabel:
        res["Q_final"] = _chain_cm(Cn, (N, K), np.float64)
        out.Q_final = _p(res["Q_final"], C.c_double)
    if "counts" in probes:
        res["counts"] = np.zeros((Cn, nsamples, K + K * P), dtype=np.int32)
        out.counts = _p(res["counts"], C.c_int32)
    if "z_freq" in probes:       # grid path posterior summaries (usable with no_z_history)
        res["z_freq"] = _chain_cm(Cn, (N, K), np.uint32)
        out.z_freq = _p(res["z_freq"], C.c_uint32)
    if "z_last" in probes:
        res["z_last"] = np.zeros((Cn, N), dtype=np.int32)
        out.z_last = _p(res["z_last"], C.c_int32)
    status = np.zeros(Cn, dtype=np.int32)
    out.status = _p(status, C.c_int32)
    return res, out, status


def out_nbytes(res):
    return int(sum(v.nbytes for v in res.values()))


class Plan:
    """Device-resident run (bmm_plan_*): upload once, `run()` any number of times, `fetch()` the lists.

    The one-shot `gibbs_*` functions are create + run + fetch + destroy of exactly this."""

    def __init__(self, sampler, X, nsamples, K, alpha, beta, gamma, a, b, burnin, relabel, burnrelabel,
                 chains=1, seed=0, device=0, precision="fp64", init_pi=None, init_theta=None, init_z=None,
                 compact_z=False, chain_offset=0, probes=(), stable_softmax=False, grid_path=False,
                 no_z_history=False, n_global=0, row_offset=0, no_tensor=False, stephens_fixed=False, thin=1):
        self.L = _lib.lib()
        self.X = _as_X(X)
        self.meta = dict(sampler=sampler, Cn=int(chains), N=self.X.shape[0], P=self.X.shape[1], K=int(K),
                         nsamples=int(nsamples), burnin=int(burnin), relabel=bool(relabel), compact_z=compact_z,
                         probes=probes, no_z=bool(no_z_history), thin=int(thin))
        args, init, self._keep = _build_args(sampler, self.X, nsamples, K, alpha, beta, gamma, a, b, burnin, relabel,
                                             burnrelabel, False, chains, seed, device, precision, init_pi, init_theta,
                                             init_z, None, compact_z, stable_softmax, chain_offset, grid_path,
                                             no_z_history, n_global, row_offset, no_tensor, stephens_fixed, thin)
        if "probs" in probes:
            args.flags |= 0x100
        if "loglik" in probes:
            args.flags |= 0x200
        if "counts" in probes:
            args.flags |= 0x400
        if "z_freq" in probes:
            args.flags |= 0x1000
        self.h = C.c_void_p()
        _lib.check(self.L.bmm_plan_create(sampler, C.byref(args), C.byref(init), C.byref(self.h)))

    def run(self):
        _lib.check(self.L.bmm_plan_run(self.h))

    def sync(self):
        _lib.check(self.L.bmm_plan_sync(self.h))

    def check(self):
        """Raise if any chain of the last run stopped with an error status (fetch with no output buffers)."""
        out = _lib.Out()
        _lib.check(self.L.bmm_plan_fetch(self.h, C.byref(out)))

    def elapsed_ms(self):
        a, b = C.c_float(), C.c_float()
        _lib.check(self.L.bmm_plan_elapsed_ms(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def kernel_ms(self):
        ms = (C.c_float * 4)()
        _lib.check(self.L.bmm_plan_kernel_ms(self.h, ms))
        return list(ms)

    def alloc_out(self, pinned=False):
        m = self.meta
        return _alloc_out(m["sampler"], m["Cn"], m["N"], m["P"], m["K"], m["nsamples"], m["burnin"], m["relabel"],
                          m["compact_z"], m["probes"], pinned, no_z=m["no_z"], thin=m["thin"])

    def fetch(self, bufs=None, pinned=False):
        res, out, status = bufs if bufs is not None else self.alloc_out(pinned)
        _lib.check(self.L.bmm_plan_fetch(self.h, C.byref(out)))
        return res

    def close(self):
        if self.h:
            self.L.bmm_plan_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _run(sampler, X, nsamples, K, alpha, beta, gamma, a, b, burnin, relabel, burnrelabel, debug,
         chains, seed, device, precision, init_pi=None, init_theta=None, init_z=None, replay=None,
         compact_z=False, stable_softmax=False, probes=(), chain_offset=0, pinned=False, out_bufs=None,
         grid_path=False, no_z_history=False, n_global=0, row_offset=0, no_tensor=False, stephens_fixed=False, thin=1):
    L = _lib.lib()
    N, P = X.shape
    Cn = int(chains)
    args, init, keep = _build_args(sampler, X, nsamples, K, alpha, beta, gamma, a, b, burnin, relabel, burnrelabel,
                                   debug, chains, seed, device, precision, init_pi, init_theta, init_z, replay,
                                   compact_z, stable_softmax, chain_offset, grid_path, no_z_history, n_global,
                                   row_offset, no_tensor, stephens_fixed, thin)
    res, out, status = out_bufs if out_bufs is not None else _alloc_out(
        sampler, Cn, N, P, K, nsamples, burnin, relabel, compact_z, probes, pinned, no_z=no_z_history, thin=thin)
    if sampler == _lib.SAMPLER_DP:
        rc = L.bmm_gibbs_dp(C.byref(args), C.byref(out))
    else:
        fn = {_lib.SAMPLER_FULL: L.bmm_gibbs_full, _lib.SAMPLER_STICKBREAKING: L.bmm_gibbs_stickbreaking,
              _lib.SAMPLER_COLLAPSED: L.bmm_gibbs_collapsed}[sampler]
        rc = fn(C.byref(args), C.byref(init), C.byref(out))
    _lib.check(rc)
    if Cn == 1 and chains == 1:
        res = {k: v[0] for k, v in res.items()}
    return res


def _defaults(nsamples, burnin, burnrelabel, alpha, clamp=True):
    if burnin is None:
        burnin = _r_round(0.1 * nsamples)
    if clamp and burnrelabel > burnin:
        burnrelabel = _r_round(0.1 * burnin)
    if alpha is None:
        alpha = 0
    return burnin, burnrelabel, alpha


def gibbs_full(data, nsamples, K, alpha=None, beta=0.5, gamma=0.5, a=1, b=1, burnin=None, relabel=False,
               burnrelabel=50, debug=False, *, chains=1, seed=0, device=0, precision="fp64", rng=None,
               initial_pi=None, initial_theta=None, replay=None, compact_z=False, stable_softmax=False,
               probes=(), chain_offset=0, pinned=False, out_bufs=None, grid_path=False, no_z_history=False,
               n_global=0, row_offset=0, no_tensor=False, stephens_fixed=False, thin=1, _sampler=None):
    """Full Gibbs sampler for a finite Bernoulli mixture model (R/utils.R:64-78 -> full_gibbs.cpp:32).

    `stephens_fixed=True` (BMM_FLAG_STEPHENS_FIXED, not the reference's behaviour) relabels with the corrected
    Stephens steps: inverse permutation for the column re-ordering, log p in the online cost, running-mean Q.

    `thin=k` keeps every k-th post-burn-in sweep in all returned histories (the reference keeps every sweep,
    full_gibbs.cpp:52-57); `probes=("z_freq", "z_last")` adds the posterior summaries a large run keeps instead."""
    X = _as_X(data)
    N, P = X.shape
    burnin, burnrelabel, alpha = _defaults(nsamples, burnin, burnrelabel, alpha, clamp=_sampler is None)
    rng = rng or RRng(seed)
    if initial_pi is None:
        initial_pi = np.empty((chains, K))
        initial_theta = np.empty((chains, P, K))
        for c in range(chains):
            ip = np.exp(rng.runif(K))                       # R/utils.R:68-70
            initial_pi[c] = ip / ip.sum()
            initial_theta[c] = rng.runif(K * P).reshape(P, K)  # matrix(runif(K*P), nrow=K): column-major
    else:
        initial_pi = np.ascontiguousarray(np.asarray(initial_pi, dtype=np.float64).reshape(chains, K))
        th = np.asarray(initial_theta, dtype=np.float64).reshape(chains, K, P)
        initial_theta = np.ascontiguousarray(th.transpose(0, 2, 1))
    sampler = _lib.SAMPLER_FULL if _sampler is None else _sampler
    return _run(sampler, X, nsamples, K, alpha, beta, gamma, a, b, burnin, relabel, burnrelabel, debug, chains, seed,
                device, precision, init_pi=np.ascontiguousarray(initial_pi), init_theta=np.ascontiguousarray(initial_theta),
                replay=replay, compact_z=compact_z, stable_softmax=stable_softmax, probes=probes, chain_offset=chain_offset,
                pinned=pinned, out_bufs=out_bufs, grid_path=grid_path, no_z_history=no_z_history, n_global=n_global,
                row_offset=row_offset, no_tensor=no_tensor, stephens_fixed=stephens_fixed, thin=thin)


def gibbs_stickbreaking(data, nsamples, maxK, alpha=None, beta=0.5, gamma=0.5, a=1, b=1, burnin=None,
                        relabel=False, burnrelabel=50, debug=False, **kw):
    """Stick-breaking blocked Gibbs sampler (R/utils.R:95-107 -> stickbreaking.cpp:10).

    Like the reference wrapper it does NOT clamp burnrelabel to burnin (R/utils.R:97-101)."""
    return gibbs_full(data, nsamples, maxK, alpha, beta, gamma, a, b, burnin, relabel, burnrelabel, debug,
                      _sampler=_lib.SAMPLER_STICKBREAKING, **kw)


def gibbs_collapsed(data, nsamples, K, alpha=None, beta=0.5, gamma=0.5, a=1, b=1, burnin=None, relabel=False,
                    burnrelabel=50, debug=False, *, chains=1, seed=0, device=0, precision="fp64", rng=None,
                    initial_K=None, replay=None, compact_z=False, probes=(), chain_offset=0, pinned=False, out_bufs=None,
                    stephens_fixed=False, thin=1):
    """Collapsed Gibbs sampler for a finite mixture (R/utils.R:37-47 -> collapsed_gibbs.cpp:24)."""
    X = _as_X(data)
    N, P = X.shape
    burnin, burnrelabel, alpha = _defaults(nsamples, burnin, burnrelabel, alpha)
    rng = rng or RRng(seed)
    if initial_K is None:
        initial_K = np.stack([rng.sample_int(K, N) for _ in range(chains)])   # sample(1:K, N, replace=T)
    initial_K = np.ascontiguousarray(np.asarray(initial_K, dtype=np.int32).reshape(chains, N))
    return _run(_lib.SAMPLER_COLLAPSED, X, nsamples, K, alpha, beta, gamma, a, b, burnin, relabel, burnrelabel, debug,
                chains, seed, device, precision, init_z=initial_K, replay=replay, compact_z=compact_z, probes=probes,
                chain_offset=chain_offset, pinned=pinned, out_bufs=out_bufs, stephens_fixed=stephens_fixed, thin=thin)


def gibbs_dp(data, nsamples, alpha=None, a=1, b=1, beta=0.5, gamma=0.5, burnin=None, relabel=False,
             burnrelabel=50, maxK=30, debug=False, *, chains=1, seed=0, device=0, precision="fp64", replay=None,
             compact_z=False, probes=(), chain_offset=0, pinned=False, out_bufs=None, stephens_fixed=False, thin=1):
    """Collapsed Gibbs sampler for the DP (CRP) infinite mixture (R/utils.R:23-30 -> collapsed_gibbs_dp.cpp:27)."""
    X = _as_X(data)
    burnin, burnrelabel, alpha = _defaults(nsamples, burnin, burnrelabel, alpha)
    return _run(_lib.SAMPLER_DP, X, nsamples, maxK, alpha, beta, gamma, a, b, burnin, relabel, burnrelabel, debug,
                chains, seed, device, precision, replay=replay, compact_z=compact_z, probes=probes,
                chain_offset=chain_offset, pinned=pinned, out_bufs=out_bufs, stephens_fixed=stephens_fixed, thin=thin)


def predictive(fit, newdata, membership=True):
    """Posterior predictive distribution of new 0/1 rows under a fitted `gibbs_full` / `gibbs_stickbreaking` model -- the
    reference's TODO list names it ("Implement predictive distribution", /root/reference/TODO:6), it has no reference code.

    `fit` is the list a sampler returned (`theta` K x P x S, `pi` S x K; with `chains > 1` the chains' draws are pooled).
    Returns `log_pred[m] = log 1/S sum_s sum_k pi_k prod_d theta_kd^x (1 - theta_kd)^(1 - x)` and, with `membership`,
    the M x K responsibilities averaged over the draws (relabelled draws give label-consistent columns)."""
    X = np.asfortranarray(np.asarray(newdata, dtype=np.int32))
    if X.ndim != 2:
        raise ValueError("newdata must be an M x P matrix")
    if "pi" not in fit:
        raise ValueError("predictive() needs the pi history of an uncollapsed sampler (gibbs_full / gibbs_stickbreaking)")
    th, pi = np.asarray(fit["theta"], dtype=np.float64), np.asarray(fit["pi"], dtype=np.float64)
    if th.ndim == 4:        # chains x K x P x S -> K x P x (chains * S)
        th = np.concatenate(list(th), axis=2)
        pi = np.concatenate(list(pi), axis=0)
    K, P, S = th.shape
    M = X.shape[0]
    if X.shape[1] != P or pi.shape != (S, K):
        raise ValueError("newdata / theta / pi shapes do not match")
    th_cm = np.ascontiguousarray(th.transpose(2, 1, 0))      # memory order k + K d + K P s
    pi_cm = np.ascontiguousarray(pi.T)                        # S x K column-major
    lp = np.zeros(M)
    mem = np.zeros((K, M)) if membership else None
    L = _lib.lib()
    _lib.check(L.bmm_predictive(_p(X, C.c_int32), M, P, K, S, _p(th_cm, C.c_double), _p(pi_cm, C.c_double),
                                _p(lp, C.c_double), _p(mem, C.c_double) if membership else None))
    out = {"log_pred": lp}
    if membership:
        out["membership"] = np.ascontiguousarray(mem.T)
    return out


def _waic_draws(fit):
    """theta [C][K x P x S] and pi [C][S x K] in the C ABI's memory order, from a fit with or without a chain axis."""
    if "pi" not in fit:
        raise ValueError("waic() needs the pi history of an uncollapsed sampler (gibbs_full / gibbs_stickbreaking)")
    th, pi = np.asarray(fit["theta"], dtype=np.float64), np.asarray(fit["pi"], dtype=np.float64)
    chains = th.ndim == 4
    if not chains:
        th, pi = th[None], pi[None]
    if th.ndim != 4 or pi.ndim != 3:
        raise ValueError("theta must be K x P x S (C x K x P x S) and pi S x K (C x S x K)")
    Cn, K, P, S = th.shape
    if pi.shape != (Cn, S, K):
        raise ValueError("theta / pi shapes do not match")
    return (np.ascontiguousarray(th.transpose(0, 3, 2, 1)), np.ascontiguousarray(pi.transpose(0, 2, 1)),
            Cn, K, P, S, chains)


def _loglik_inputs(fit, data, no_tensor, what):
    """The C ABI's arguments shared by waic(), loo() and loglik_matrix(), checked on the host.  X is returned with its
    address: the caller keeps it alive across the library call."""
    th, pi, Cn, K, P, S, chains = _waic_draws(fit)
    X = _as_X(data)
    if X.shape[1] != P:
        raise ValueError("data has %d columns, theta has %d variables" % (X.shape[1], P))
    if Cn * S < 2:
        raise ValueError("%s needs at least 2 draws" % what)
    flags = (_lib.FLAG_X_PACKED if isinstance(X, PackedX) else 0) | (_lib.FLAG_NO_TENSOR if no_tensor else 0)
    xp = X.bits.ctypes.data if isinstance(X, PackedX) else X.ctypes.data
    return th, pi, Cn, K, P, S, chains, X, flags, C.c_void_p(xp)


def waic(fit, data, *, no_tensor=False, device=0):
    """WAIC of a fitted `gibbs_full` / `gibbs_stickbreaking` model and the log-likelihood trace of its draws, computed on the
    device (Watanabe 2010; Vehtari, Gelman & Gabry 2017, the layout of R's `loo::waic`).

    `data` is the N x P 0/1 matrix the model was fitted to, or a `PackedX`.  With a chain axis the C chains' S draws are
    pooled (D = C S >= 2).  With l[c,s,i] = log p(x_i | draw (c, s)): `pointwise_lppd` = log mean exp l, `pointwise_p_waic`
    = the sample variance of l over the draws, `pointwise_elpd_waic` = their difference, `pointwise_waic` = -2 times it;
    the totals are sums over i and `se_*` = sqrt(N var_i(pointwise)).  `loglik[c, s]` = sum_i l[c,s,i], the trace.  With a
    chain axis `chain_elpd_waic`, `chain_waic` and `chain_p_waic` are the same totals from each chain's draws alone.

    K <= 32 and P <= 112 fits with many distinct rows run on the tcgen05 kernel (fp16 hi|lo operands, fp32 log-sum-exp,
    fp64 moments); `no_tensor=True` forces the fp64 kernel."""
    th, pi, Cn, K, P, S, chains, X, flags, xp = _loglik_inputs(fit, data, no_tensor, "waic")
    N = X.shape[0]
    ll = np.zeros((Cn, S))
    lppd, pw = np.zeros(N), np.zeros(N)
    clp, cpw = np.zeros(Cn), np.zeros(Cn)
    _lib.check(_lib.lib().bmm_waic(xp, N, P, K, S, Cn, _p(th, C.c_double), _p(pi, C.c_double), flags,
                                   int(device), _p(ll, C.c_double), _p(lppd, C.c_double), _p(pw, C.c_double),
                                   _p(clp, C.c_double), _p(cpw, C.c_double)))
    elpd = lppd - pw
    out = {"pointwise_lppd": lppd, "pointwise_p_waic": pw, "pointwise_elpd_waic": elpd, "pointwise_waic": -2.0 * elpd}
    for name in ("lppd", "p_waic", "elpd_waic", "waic"):
        v = out["pointwise_" + name]
        out[name] = float(v.sum())
        out["se_" + name] = float(np.sqrt(N * np.var(v, ddof=1))) if N > 1 else float("nan")
    out["loglik"] = ll if chains else ll[0]
    if chains:
        out["chain_elpd_waic"] = clp - cpw
        out["chain_waic"] = -2.0 * (clp - cpw)
        out["chain_p_waic"] = cpw
    return out


def loo(fit, data, *, r_eff=1.0, no_tensor=False, device=0):
    """PSIS-LOO of a fitted `gibbs_full` / `gibbs_stickbreaking` model, computed on the device (Vehtari, Gelman & Gabry
    2017; the algorithm and the layout of R's `loo::loo`, without `mcse_elpd_loo`).

    `data` is the N x P 0/1 matrix the model was fitted to, or a `PackedX`; with a chain axis the C chains' S draws are
    pooled (D = C S >= 2).  `r_eff` (a scalar or N values, finite and > 0) is the relative efficiency of each observation's
    draws: it sets the Pareto tail length min(ceil(0.2 D), ceil(3 sqrt(D / r_eff))) and scales `n_eff`; computing it
    from the chains (`loo::relative_eff`) is left to the caller.  Returns the pointwise arrays `pointwise_elpd_loo`,
    `pointwise_lpd` (= waic()'s lppd), `pointwise_p_loo` = lpd - elpd_loo and `pointwise_looic` = -2 elpd_loo; their
    totals and `se_*` = sqrt(N var_i(pointwise)); `pareto_k` (inf where the tail has fewer than 5 draws or is flat) and
    `n_eff` per observation; `k_threshold` = min(1 - 1 / log10(D), 0.7) and the counts of observations with k at most
    the threshold (`n_k_good`), in (threshold, 1] (`n_k_bad`) and above 1 (`n_k_very_bad`, where the estimate cannot
    be trusted).

    The log-likelihood matrix comes from the tcgen05 kernel for K <= 32, P <= 112 fits with many distinct rows (as in
    waic()); `no_tensor=True` forces the fp64 kernel.  The smoothing and the sums run in fp64."""
    th, pi, Cn, K, P, S, chains, X, flags, xp = _loglik_inputs(fit, data, no_tensor, "loo")
    N = X.shape[0]
    re = np.asarray(r_eff, dtype=np.float64)
    if re.ndim == 0:
        re = np.full(N, float(re))
    if re.shape != (N,):
        raise ValueError("r_eff must be a scalar or have one value per observation (%d)" % N)
    if not (np.isfinite(re).all() and (re > 0).all()):
        raise ValueError("r_eff must be finite and > 0")
    re = np.ascontiguousarray(re)
    elpd, lpd, k, neff = np.zeros(N), np.zeros(N), np.zeros(N), np.zeros(N)
    _lib.check(_lib.lib().bmm_loo(xp, N, P, K, S, Cn, _p(th, C.c_double), _p(pi, C.c_double), _p(re, C.c_double), flags,
                                  int(device), _p(elpd, C.c_double), _p(lpd, C.c_double), _p(k, C.c_double),
                                  _p(neff, C.c_double)))
    out = {"pointwise_elpd_loo": elpd, "pointwise_lpd": lpd, "pointwise_p_loo": lpd - elpd, "pointwise_looic": -2.0 * elpd}
    for name in ("elpd_loo", "lpd", "p_loo", "looic"):
        v = out["pointwise_" + name]
        out[name] = float(v.sum())
        out["se_" + name] = float(np.sqrt(N * np.var(v, ddof=1))) if N > 1 else float("nan")
    out["pareto_k"], out["n_eff"] = k, neff
    D = Cn * S
    thr = min(1.0 - 1.0 / np.log10(D), 0.7)
    out["k_threshold"] = thr
    out["n_k_good"] = int(np.sum(k <= thr))
    out["n_k_bad"] = int(np.sum((k > thr) & (k <= 1)))
    out["n_k_very_bad"] = int(np.sum(k > 1))
    return out


def loglik_matrix(fit, data, *, no_tensor=False, device=0):
    """l[g, i] = log p(x_i | draw g) of a fitted `gibbs_full` / `gibbs_stickbreaking` model, computed on the device: a
    D x N array over the S kept draws, or C x S x N when the fit has a chain axis (the matrix / array `loo::loo()` takes).
    The kernels and `no_tensor` are those of loo()."""
    th, pi, Cn, K, P, S, chains, X, flags, xp = _loglik_inputs(fit, data, no_tensor, "loglik_matrix")
    N = X.shape[0]
    out = np.zeros((N, Cn * S))
    _lib.check(_lib.lib().bmm_loglik_matrix(xp, N, P, K, S, Cn, _p(th, C.c_double), _p(pi, C.c_double), flags, int(device),
                                            _p(out, C.c_double)))
    return out.T.reshape(Cn, S, N) if chains else out.T
