// Device building blocks shared by the sampler kernels (sm_100a).
//   Philox4x32-10 counter RNG, uniform/normal/gamma/beta draws, the two categorical draw rules
//   (rmultinom replay rule and single-uniform inverse CDF), warp helpers.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace bmm {

// RNG stream ids (Philox counter word 2)
enum : uint32_t { ST_Z = 0, ST_PI = 1, ST_THETA = 2, ST_ALPHA = 3, ST_STICK = 4, ST_MISC = 5 };

__host__ __device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
#ifdef __CUDA_ARCH__
        uint32_t hi0 = __umulhi(M0, c.x), hi1 = __umulhi(M1, c.z);
#else
        uint32_t hi0 = (uint32_t)(((uint64_t)M0 * c.x) >> 32), hi1 = (uint32_t)(((uint64_t)M1 * c.z) >> 32);
#endif
        uint32_t lo0 = M0 * c.x, lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += W0;
        k.y += W1;
    }
    return c;
}

// 53-bit uniform in (0,1) from two 32-bit words.  (2^53 - 0.5) / 2^53 rounds to 1.0, so the top value is clamped to
// the largest double below 1: an inverse-CDF draw at u = 1 would run past every category with mass.
__host__ __device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
    uint64_t v = ((uint64_t)a << 21) ^ (uint64_t)(b >> 11);
    return fmin(((double)v + 0.5) * (1.0 / 9007199254740992.0), 0x1.fffffffffffffp-1);
}
// A u53 uniform cast to float: every u53 >= 1 - 2^-25 rounds to 1.0f, so it is clamped to the largest float below 1.
__host__ __device__ __forceinline__ float unit_f(double u) { return fminf((float)u, 0x1.fffffep-1f); }

// Allocation draws of the uncollapsed samplers: observation gi of sweep j uses word gi & 3 of
// Philox(counter = (gi >> 2, gi >> 34, stream, j)), i.e. one Philox evaluation serves four consecutive
// observations (the chain-per-block kernel draws them in one lane).  32 bits per uniform: categories
// below 2^-32 are never drawn, far under any Monte Carlo resolution.
__host__ __device__ __forceinline__ uint32_t philox_word(const uint4 &r, int h) {
    return h == 0 ? r.x : (h == 1 ? r.y : (h == 2 ? r.z : r.w));
}
__host__ __device__ __forceinline__ double u32_unit(uint32_t w) { return ((double)w + 0.5) * (1.0 / 4294967296.0); }
// 24-bit float uniform: 16777215.5 rounds to 2^24 in float, so every w >= 0xFFFFFF00 would give exactly 1.0f; those are
// clamped to the largest float below 1 (all other words keep their value).
__host__ __device__ __forceinline__ float u32_unit_f(uint32_t w) {
    return fminf(((float)(w >> 8) + 0.5f) * 5.9604644775390625e-08f, 0x1.fffffep-1f);
}

// Sequential stream for the (rare, rejection-based) parameter draws.
// key = (seed_lo, chain); counter = (attempt, index, stream, sweep ^ seed_hi-mix)
struct Stream {
    uint2 key;
    uint4 ctr;
    uint4 buf;
    int n;
    __device__ Stream(uint64_t seed, uint32_t chain, uint32_t sweep, uint32_t stream, uint32_t index) {
        key = make_uint2((uint32_t)seed, chain);
        ctr = make_uint4(0u, index, stream ^ ((uint32_t)(seed >> 32) << 8), sweep);
        n = 0;
    }
    __device__ double uniform() {
        if ((n & 1) == 0) { buf = philox4x32_10(ctr, key); ctr.x++; }
        double u = (n & 1) ? u53(buf.z, buf.w) : u53(buf.x, buf.y);
        n++;
        return u;
    }
    __device__ double normal() {
        double u1 = uniform(), u2 = uniform();
        return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
    }
    // Gamma(shape, 1): Marsaglia-Tsang (shape < 1 boosted).  Same law as R::rgamma(shape, 1).
    __device__ __forceinline__ double gamma(double shape) {
        if (!(shape > 0.0)) return 0.0;
        double boost = 1.0;
        if (shape < 1.0) { boost = exp(log(uniform()) / shape); shape += 1.0; }
        double d = shape - 1.0 / 3.0, c = rsqrt(9.0 * d);
        for (int it = 0; it < 256; ++it) {
            double x = normal(), v = 1.0 + c * x;
            if (v <= 0.0) continue;
            v = v * v * v;
            double u = uniform();
            if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) return boost * d * v;
        }
        return boost * d;
    }
    __device__ double beta(double a, double b) {
        double x = gamma(a), y = gamma(b);
        double s = x + y;
        return s > 0.0 ? x / s : 0.5;
    }
    // Out-of-line copy: ~300 fp64-heavy instructions per inlined call.  Measured per kernel (ncu showed
    // instruction-fetch stalls in the chain kernels): sharing one copy makes dp_kernel 30 % faster
    // (8.7e8 -> 1.13e9 updates/s), does nothing for full_chain_kernel and halves collapsed_kernel, so
    // only the DP path uses it.
    __device__ __noinline__ double gamma_shared(double shape) { return gamma(shape); }
    __device__ double beta_shared(double a, double b) {
        double x = gamma_shared(a), y = gamma_shared(b);
        double s = x + y;
        return s > 0.0 ? x / s : 0.5;
    }
};

// update_alpha (utils.cpp:6-14): alpha' = pi*G(a+K, 1/b_eps) + (1-pi)*G(a+K-1, 1/b_eps)
template <bool SHARED = false>
__device__ __forceinline__ double update_alpha_dev(Stream &s, double alpha_old, double a, double b, int N, int K) {
    double b_eps = b - log(SHARED ? s.beta_shared(alpha_old + 1.0, (double)N) : s.beta(alpha_old + 1.0, (double)N));
    double pi1 = a + K - 1, pi2 = N * b_eps, pi = pi1 / (pi1 + pi2);
    double g1 = (SHARED ? s.gamma_shared(a + K) : s.gamma(a + K)) / b_eps;
    double g2 = (SHARED ? s.gamma_shared(a + K - 1) : s.gamma(a + K - 1)) / b_eps;
    return pi * g1 + (1 - pi) * g2;
}

// The same update with its four Gamma draws on independent substreams (index q of ST_ALPHA), used by the
// uncollapsed samplers: the chain kernel draws them on four lanes next to the theta / pi draws instead of one
// lane drawing them in turn after everybody else (that serial tail was a third of a C2 sweep), the grid
// kernel draws the same four substreams so both paths keep producing the same chain.
//   q = 0, 1: x ~ G(alpha + 1), y ~ G(N)   -> rbeta(alpha + 1, N) = x / (x + y)   (utils.cpp:8)
//   q = 2, 3: G(a + K), G(a + K - 1)                                               (utils.cpp:12)
__device__ __forceinline__ double alpha_gamma_shape(int q, double alpha_old, double a, int N, int K) {
    return q == 0 ? alpha_old + 1.0 : (q == 1 ? (double)N : (q == 2 ? a + K : a + K - 1));
}
__device__ __forceinline__ double alpha_combine(const double *g, double a, double b, int N, int K) {
    const double sb = g[0] + g[1], bt = sb > 0.0 ? g[0] / sb : 0.5;
    const double b_eps = b - log(bt);
    const double pi1 = a + K - 1, pi2 = N * b_eps, pi = pi1 / (pi1 + pi2);
    return pi * (g[2] / b_eps) + (1 - pi) * (g[3] / b_eps);
}

// rmultinom(1, prob, K) replay rule (R nmath rmultinom.c / rbinom.c inversion branch, SURVEY App. A
// items 3-4): sequential conditional binomials; one recorded uniform per non-zero category visited.
// `getp(k)` returns prob[k]; u points at this draw's recorded uniforms.  Returns the 0-based label.
// The reference keeps the running total p_tot in `long double` (x87, 64-bit significand).  A plain double
// total goes wrong exactly where it matters: when the categories left have equal probabilities (clusters
// with identical sufficient statistics) pp = p_k / p_tot sits on the 0.5 switch of the rbinom inversion
// rule, and which side it lands on must not be decided by cancellation noise of the subtractions.  The
// total is therefore carried as an unevaluated double-double sum (error-free additions, >= 106 bits),
// which reproduces the extended-precision result whenever that result is itself above its own noise.
struct DD { double hi, lo; };
__device__ __forceinline__ DD dd_add(DD x, double y) {
    const double s = __dadd_rn(x.hi, y), bb = __dadd_rn(s, -x.hi);
    double e = __dadd_rn(__dadd_rn(x.hi, -__dadd_rn(s, -bb)), __dadd_rn(y, -bb));
    e = __dadd_rn(e, x.lo);
    const double hi = __dadd_rn(s, e);
    return DD{hi, __dadd_rn(e, -__dadd_rn(hi, -s))};
}
__device__ __forceinline__ double dd_div_into(double a, DD t) {   // (double)(a / t)
    const double q1 = a / t.hi;
    const double r = __dadd_rn(__fma_rn(-q1, t.hi, a), -__dmul_rn(q1, t.lo));
    return __dadd_rn(q1, r / t.hi);
}

template <typename GetP>
__device__ __forceinline__ int rmultinom1_replay(int K, GetP getp, const double *__restrict__ u) {
    DD p_tot{0.0, 0.0};
    for (int k = 0; k < K; ++k) p_tot = dd_add(p_tot, getp(k));
    int slot = 0;
    for (int k = 0; k < K - 1; ++k) {
        double pk = getp(k);
        if (pk != 0.0) {
            double pp = dd_div_into(pk, p_tot);
            int got;
            if (pp < 1.0) {
                double p = fmin(pp, 1.0 - pp), q = 1.0 - p;
                double uu = u[slot++];
                int ix = (uu < q) ? 0 : 1;
                got = (pp > 0.5) ? 1 - ix : ix;
            } else {
                got = 1;
            }
            if (got) return k;
        }
        p_tot = dd_add(p_tot, -pk);
    }
    return K - 1;
}

// Single-uniform inverse-CDF categorical draw over normalised probabilities (Philox mode).
template <typename GetP>
__device__ __forceinline__ int categorical_icdf(int K, GetP getp, double u) {
    double cum = 0.0;
    for (int k = 0; k < K - 1; ++k) {
        cum += getp(k);
        if (u < cum) return k;
    }
    return K - 1;
}

__device__ __forceinline__ double warp_sum_xor(double v, int width) {
    for (int off = 1; off < width; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

template <typename T>
__device__ __forceinline__ T ld_any(const T *p) { return *p; }

}  // namespace bmm
