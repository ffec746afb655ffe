"""Host transcription of the Philox-mode draws of the samplers, in numpy (test infrastructure).

Every Philox-mode draw of the library is a pure function of (seed, chain, sweep, stream, index) and the
previous state, and the returned histories (burnin = 0, thin = 1) hold that state.  This module rebuilds
the uniforms each kernel consumes and the float64 conditionals it draws from, so that a test can check
each allocation and each parameter draw of a run:

  - the RNG primitives of csrc/common.cuh (Philox4x32-10, u53, u32_unit, u32_unit_f) bit for bit;
  - `Stream`, the sequential parameter stream (uniform, normal, Gamma, Beta) to ~1 ulp of libm;
  - both alpha updates (four substreams for the uncollapsed samplers, sequential for the collapsed ones);
  - the z-uniform layout of each kernel family and the float64 conditionals the allocations are drawn from.

Device lines are cited as file:line of bmm_mcmc_b200/csrc.
"""
import math

import numpy as np

ST_Z, ST_PI, ST_THETA, ST_ALPHA, ST_STICK, ST_MISC = 0, 1, 2, 3, 4, 5   # common.cuh:11

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_MASK = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)

U53_MAX = float.fromhex("0x1.fffffffffffffp-1")   # largest double below 1
UF_MAX = np.float32(float.fromhex("0x1.fffffep-1"))  # largest float below 1


# ---- RNG primitives (common.cuh:13-44) ------------------------------------------------------------
def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (common.cuh:13-28), vectorised over broadcastable counters and keys.
    Returns a uint32 array of shape (..., 4)."""
    c0, c1, c2, c3, k0, k1 = np.broadcast_arrays(*[np.asarray(v, dtype=np.uint64) & _MASK for v in (c0, c1, c2, c3, k0, k1)])
    c0, c1, c2, c3, k0, k1 = (v.copy() for v in (c0, c1, c2, c3, k0, k1))
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = ((p1 >> _S32) ^ c1 ^ k0), (p1 & _MASK), ((p0 >> _S32) ^ c3 ^ k1), (p0 & _MASK)
        k0 = (k0 + np.uint64(_W0)) & _MASK
        k1 = (k1 + np.uint64(_W1)) & _MASK
    return np.stack([c0, c1, c2, c3], -1).astype(np.uint32)


def philox_int(c, k):
    """Scalar Philox4x32-10 on Python ints (the per-draw path of `Stream`; same function as `philox`)."""
    c0, c1, c2, c3 = c
    k0, k1 = k
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
        c0, c1, c2, c3 = (p1 >> 32) ^ c1 ^ k0, p1 & 0xFFFFFFFF, (p0 >> 32) ^ c3 ^ k1, p0 & 0xFFFFFFFF
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


def _u53_int(a, b):
    return min((float((a << 21) ^ (b >> 11)) + 0.5) * (1.0 / 9007199254740992.0), U53_MAX)


def u53(a, b):
    """53-bit uniform from two words (common.cuh:31-35), strictly inside (0, 1)."""
    v = (np.asarray(a, dtype=np.uint64) << np.uint64(21)) ^ (np.asarray(b, dtype=np.uint64) >> np.uint64(11))
    return np.minimum((v.astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0), U53_MAX)


def u32_unit(w):
    """32-bit uniform (common.cuh:43): (w + 0.5) / 2^32 in double."""
    return (np.asarray(w, dtype=np.uint32).astype(np.float64) + 0.5) * (1.0 / 4294967296.0)


def u32_unit_f(w):
    """24-bit float uniform of the tensor-core sweeps (common.cuh:44), emulated in float32, strictly below 1."""
    hi = (np.asarray(w, dtype=np.uint32) >> np.uint32(8)).astype(np.float32)
    u = (hi + np.float32(0.5)) * np.float32(5.9604644775390625e-08)
    return np.minimum(u, UF_MAX)


# ---- sequential parameter stream (common.cuh:48-98) ------------------------------------------------
class Stream:
    """The device `Stream`: key (seed_lo, chain), counter (attempt, index, stream ^ seed_hi << 8, sweep).

    `near` is set when a rejection decision fell within `tol` (relative) of its boundary: libm and CUDA's
    fp64 log / exp differ in the last ulp, so such a draw may legitimately go the other way on the device."""

    def __init__(self, seed, chain, sweep, stream, index, tol=1e-10):
        seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.key = (seed & 0xFFFFFFFF, int(chain) & 0xFFFFFFFF)
        self.ctr = [0, int(index) & 0xFFFFFFFF, (int(stream) ^ ((seed >> 32) << 8)) & 0xFFFFFFFF, int(sweep) & 0xFFFFFFFF]
        self.buf = None
        self.n = 0
        self.tol = tol
        self.near = False

    def uniform(self):
        if self.n % 2 == 0:
            self.buf = philox_int(self.ctr, self.key)
            self.ctr[0] += 1
        w = self.buf
        u = _u53_int(w[2], w[3]) if self.n % 2 else _u53_int(w[0], w[1])
        self.n += 1
        return u

    def normal(self):
        u1, u2 = self.uniform(), self.uniform()
        return math.sqrt(-2.0 * math.log(u1)) * math.cos(2.0 * math.pi * u2)   # cospi(2 u2)

    def _close(self, x, y, scale):
        if abs(x - y) <= self.tol * max(scale, 1e-300):
            self.near = True

    def gamma(self, shape):
        """Marsaglia-Tsang with the shape < 1 boost and the 256-attempt cap (common.cuh:69-82)."""
        if not shape > 0.0:
            return 0.0
        boost = 1.0
        if shape < 1.0:
            boost = math.exp(math.log(self.uniform()) / shape)
            shape += 1.0
        d = shape - 1.0 / 3.0
        c = 1.0 / math.sqrt(9.0 * d)
        for _ in range(256):
            x = self.normal()
            v = 1.0 + c * x
            self._close(v, 0.0, 1.0)
            if v <= 0.0:
                continue
            v = v * v * v
            u = self.uniform()
            lhs, rhs = math.log(u), 0.5 * x * x + d - d * v + d * math.log(v)
            self._close(lhs, rhs, max(abs(lhs), abs(rhs), d * abs(math.log(v)) + d * v + d))
            if lhs < rhs:
                return boost * d * v
        return boost * d

    def beta(self, a, b):
        x = self.gamma(a)
        y = self.gamma(b)
        s = x + y
        return x / s if s > 0.0 else 0.5


def alpha_gamma_shape(q, alpha_old, a, N, K):
    """common.cuh:116-118"""
    return (alpha_old + 1.0, float(N), a + K, a + K - 1)[q]


def alpha_combine(g, a, b, N, K):
    """common.cuh:119-124"""
    sb = g[0] + g[1]
    bt = g[0] / sb if sb > 0.0 else 0.5
    b_eps = b - math.log(bt)
    pi1, pi2 = a + K - 1, N * b_eps
    pi = pi1 / (pi1 + pi2)
    return pi * (g[2] / b_eps) + (1 - pi) * (g[3] / b_eps)


def alpha_update_substreams(seed, chain, j, alpha_old, a, b, N, K):
    """Uncollapsed alpha update: Gamma q on substream q of ST_ALPHA (kern_full.cu:222-226,257-266,
    kern_big.cu:303-333).  Stick-breaking passes K_viable as K.  Returns (alpha, near)."""
    g, near = [], False
    for q in range(4):
        st = Stream(seed, chain, j, ST_ALPHA, q)
        g.append(st.gamma(alpha_gamma_shape(q, alpha_old, a, N, K)))
        near |= st.near
    return alpha_combine(g, a, b, N, K), near


def update_alpha_seq(st, alpha_old, a, b, N, K):
    """Collapsed alpha update on one stream (common.cuh:101-108, kern_collapsed.cu:102-103)."""
    b_eps = b - math.log(st.beta(alpha_old + 1.0, float(N)))
    pi1, pi2 = a + K - 1, N * b_eps
    pi = pi1 / (pi1 + pi2)
    g1 = st.gamma(a + K) / b_eps
    g2 = st.gamma(a + K - 1) / b_eps
    return pi * g1 + (1 - pi) * g2


# ---- z-uniform layouts -------------------------------------------------------------------------------
def _sid(seed, stream=ST_Z):
    return (stream ^ ((int(seed) >> 32) << 8)) & 0xFFFFFFFF


def z_words_rows(seed, chain, j, gi):
    """Allocation word of global row gi at sweep j: word gi & 3 of Philox((gi >> 2, gi >> 34, sid, j), (seed_lo, chain)).
    Chain path (kern_full.cu:142-150, chain = chain_offset + c) and grid paths (kern_big.cu:120-121,
    kern_big_ws.cu:274-289, kern_big_lp.cu:174-176, chain = chain_offset)."""
    gi = np.asarray(gi, dtype=np.uint64)
    r = philox(gi >> np.uint64(2), gi >> np.uint64(34), _sid(seed), j, int(seed) & 0xFFFFFFFF, chain)
    return np.take_along_axis(r, (gi & np.uint64(3)).astype(np.int64)[..., None], -1)[..., 0]


def z_uniforms_collapsed(seed, chain, j, N):
    """Uniform of update i in sweep j of the collapsed kernels: counter (i >> 1, 0, sid, j), words (x, y) for
    even i and (z, w) for odd i, through u53 (kern_collapsed.cu:150-151,202-205,439-448)."""
    i = np.arange(N)
    r = philox(i >> 1, 0, _sid(seed), j, int(seed) & 0xFFFFFFFF, chain)
    odd = (i & 1).astype(bool)
    w0 = np.where(odd, r[:, 2], r[:, 0])
    w1 = np.where(odd, r[:, 3], r[:, 1])
    return u53(w0, w1)


# ---- float64 conditionals and the inverse-CDF check ------------------------------------------------------
def uncollapsed_probs(X, theta, pi):
    """Conditional allocation probabilities (full_gibbs.cpp:92-122) in float64 with the maximum subtracted.
    X: N x P 0/1, theta: K x P, pi: K.  Returns N x K."""
    X = np.asarray(X, dtype=np.float64)
    with np.errstate(divide="ignore"):
        l1, l0, lpi = np.log(theta), np.log1p(-theta), np.log(pi)
    ll = X @ l1.T + (1.0 - X) @ l0.T + lpi[None, :]
    ll -= ll.max(1, keepdims=True)
    p = np.exp(ll)
    return p / p.sum(1, keepdims=True)


def icdf_check(prob, u, z, delta, pmin=1e-12):
    """Check allocations z (0-based) against the inverse-CDF category of `prob` (rows) at uniforms u.

    A row is exempt when u lies within `delta` of an interior CDF boundary.  Returns
    (bad rows, exempt rows, rows whose drawn category has probability < pmin); the last are never exempt."""
    prob = np.asarray(prob, dtype=np.float64)
    u = np.asarray(u, dtype=np.float64)
    cdf = np.cumsum(prob, 1)
    cdf /= cdf[:, -1:]
    K = prob.shape[1]
    ref = np.minimum((u[:, None] >= cdf[:, :-1]).sum(1), K - 1)
    # a boundary at u beyond the last category with mass is where float draws used to land on a zero-weight tail
    near = (np.abs(u[:, None] - cdf[:, :-1]) < delta).any(1)
    drawn_p = prob[np.arange(len(z)), z]
    tiny = np.nonzero(drawn_p < pmin)[0]
    bad = np.nonzero((ref != z) & ~near)[0]
    exempt = np.nonzero((ref != z) & near)[0]
    return bad, exempt, tiny


def expected_exempt(prob, delta):
    """Expected number of rows within delta of an interior boundary: 2 delta (K - 1) per row at most."""
    return 2.0 * delta * (prob.shape[1] - 1) * prob.shape[0]


def collapsed_probs_sweep(X, z_prev, z_cur, K, alpha, beta, gamma):
    """Conditionals of every update of one finite-K collapsed sweep (collapsed_gibbs.cpp:98-140) in float64.

    The state seen by update i is z_cur[:i] and z_prev[i:] (labels 0-based); observation i itself is removed
    from its cluster; an empty cluster has probability exactly 0.  Product form (kern_collapsed.cu:376-386):
    (N_k + a/K) prod_d (beta + S_kd | gamma + N_k - S_kd) / (beta + gamma + N_k)^P, in logs."""
    X = np.asarray(X, dtype=np.int64)
    N, P = X.shape
    z = np.array(z_prev, dtype=np.int64)
    Nk = np.bincount(z, minlength=K).astype(np.int64)
    S = np.zeros((K, P), dtype=np.int64)
    np.add.at(S, z, X)
    out = np.zeros((N, K))
    for i in range(N):
        x = X[i]
        a = z[i]
        Nk[a] -= 1
        S[a] -= x
        with np.errstate(divide="ignore", invalid="ignore"):
            lw = (np.log(Nk + alpha / K) + np.where(x[None, :] == 1, np.log(beta + S), np.log(gamma + Nk[:, None] - S)).sum(1)
                  - P * np.log(beta + gamma + Nk))
        lw = np.where(Nk > 0, lw, -np.inf)
        w = np.exp(lw - lw.max())
        out[i] = w / w.sum()
        b = z_cur[i]
        z[i] = b
        Nk[b] += 1
        S[b] += x
    return out


# ---- parameter draws ---------------------------------------------------------------------------------------
def uncollapsed_params(seed, chain, j, z, X, K, alpha_prev, alpha0, beta, gamma, a, b, stickbreaking):
    """theta (K x P), pi (K), alpha and K_viable of sweep j from the allocations z (0-based) of that sweep
    (kern_full.cu:198-267, kern_big.cu:227-335).  Returns (theta, pi, alpha, K_viable, near)."""
    X = np.asarray(X, dtype=np.int64)
    N, P = X.shape
    ck = np.bincount(z, minlength=K)
    V = np.zeros((K, P), dtype=np.int64)
    np.add.at(V, z, X)
    near = False
    theta = np.empty((K, P))
    for k in range(K):
        for d in range(P):
            st = Stream(seed, chain, j, ST_THETA, k * P + d)
            theta[k, d] = st.beta(beta + V[k, d], gamma + ck[k] - V[k, d])
            near |= st.near
    g = np.empty(K)
    kv = None
    if not stickbreaking:
        for k in range(K):
            st = Stream(seed, chain, j, ST_PI, k)
            g[k] = st.gamma(alpha_prev / K + ck[k])
            near |= st.near
        pi = g / g.sum()
        K_alpha = K
    else:
        later = np.concatenate([np.cumsum(ck[::-1])[::-1][1:], [0]])
        for k in range(K):
            st = Stream(seed, chain, j, ST_STICK, k)
            g[k] = st.beta(1.0 + ck[k], alpha_prev + later[k])
            near |= st.near
        g[K - 1] = 1.0
        pi = np.empty(K)
        cum = 1.0
        for k in range(K):
            pi[k] = g[0] if k == 0 else cum * g[k]
            cum *= 1 - g[k]
        kv = int((pi > 0.01).sum())
        near |= bool((np.abs(pi - 0.01) < 1e-10).any())
        K_alpha = kv
    alpha = alpha_prev
    if alpha0 == 0.0:
        alpha, nr = alpha_update_substreams(seed, chain, j, alpha_prev, a, b, N, K_alpha)
        near |= nr
    return theta, pi, alpha, kv, near


class DPState:
    """Label bookkeeping of dp_kernel (kern_collapsed.cu:564-825, collapsed_gibbs_dp.cpp:108-242): the used-label list
    in its order (erase keeps the order of the rest), the free-label multiset (a new cluster takes the smallest free
    label), integer counts.  Every observation starts unassigned; sweep 1 removes nothing."""

    def __init__(self, X, maxK):
        self.X = np.asarray(X, dtype=np.int64)
        self.N, self.P = self.X.shape
        self.maxK = maxK
        self.used = []
        self.free = np.ones(maxK, dtype=np.int64)
        self.Nk = np.zeros(maxK, dtype=np.int64)
        self.S = np.zeros((maxK, self.P), dtype=np.int64)
        self.z = np.full(self.N, -1, dtype=np.int64)

    def sweep(self, j, z_drawn, alpha, beta, gamma):
        """Conditionals of every update of sweep j over the positions (used list + the new cluster) in float64, and the
        position of each drawn label; the state follows the drawn labels z_drawn (0-based).  Returns (probs, pos),
        probs padded with zeros to maxK + 1 columns, pos = -1 where the drawn label is not a possible outcome."""
        X, P, maxK = self.X, self.P, self.maxK
        probs = np.zeros((self.N, maxK + 1))
        pos = np.full(self.N, -1, dtype=np.int64)
        with np.errstate(divide="ignore"):
            lnew = math.log(alpha) + P * (math.log(beta) - math.log(beta + gamma))
        for i in range(self.N):
            x = X[i]
            if j > 1:                                   # drop i from its cluster (:112-131)
                a = self.z[i]
                self.Nk[a] -= 1
                self.S[a] -= x
                if self.Nk[a] == 0:
                    self.used.remove(a)
                    self.free[a] += 1
            new = int(np.argmax(self.free > 0))
            assert self.free[new] > 0 and len(self.used) < maxK - 1, "truncation state: not transcribed"
            u = np.array(self.used, dtype=np.int64)
            nk, S = self.Nk[u], self.S[u]
            lw = (np.log(nk) + np.where(x[None, :] == 1, np.log(beta + S), np.log(gamma + nk[:, None] - S)).sum(1)
                  - P * np.log(beta + gamma + nk))
            lw = np.concatenate([lw, [lnew]])
            w = np.exp(lw - lw.max())
            probs[i, :len(w)] = w / w.sum()
            b = int(z_drawn[i])
            if b in self.used:
                pos[i] = self.used.index(b)
            elif b == new:
                pos[i] = len(self.used)
                self.free[new] -= 1
                self.used.append(new)
            else:
                return probs, pos                       # the caller reports row i
            self.z[i] = b
            self.Nk[b] += 1
            self.S[b] += x
        return probs, pos
