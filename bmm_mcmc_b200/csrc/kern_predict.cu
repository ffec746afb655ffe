// Posterior predictive distribution of a fitted Bernoulli mixture (the reference's TODO list, /root/reference/TODO:6,
// "Implement predictive distribution"; SURVEY 8f-4).  From the S kept draws (theta^(s), pi^(s)) an uncollapsed sampler
// returns (full_gibbs.cpp:233-248):
//     p(x* | data) ~= 1/S sum_s sum_k pi_k^(s) prod_d theta_kd^(s)^x*_d (1 - theta_kd^(s))^(1 - x*_d)
// and the averaged responsibilities r_k(x*) = 1/S sum_s pi_k L_k / sum_l pi_l L_l.  New rows are bit-packed like the data;
// one thread per new row walks the draws with a running log-sum-exp in fp64; the per-draw log tables are built once.
//
// WAIC (Watanabe 2010; Vehtari, Gelman & Gabry 2017) reuses the tables: l[g,i] = log p(x_i | draw g) for the D = C S pooled
// draws, lppd_i = log 1/D sum_g exp l[g,i], p_waic_i = var_g l[g,i] (denominator D - 1), and the trace sum_i l[g,i].
// waic_fp64_kernel runs one warp per (tile of 32 distinct rows, slice of draws inside one chain), lane = row, and leaves
// mergeable partials per (slice, row): Welford (n, mean, M2) and a running log-sum-exp (max, sum); per (tile, draw) it
// leaves the multiplicity-weighted sum of l.  waic_merge_kernel combines slices into chains and chains into the pooled
// figure in a fixed order (Chan et al.'s variance merge), waic_sum_kernel sums partials in a fixed order: no atomics, so
// two calls return the same bits.  The tcgen05 kernel (kern_waic_tc.cu) leaves the same partials, one slice per chain.
// loglik_fp64_kernel stores the same l[g,u] of a chunk of distinct rows instead, the matrix PSIS-LOO reads (kern_loo.cu).
#include "kernels.h"

namespace bmm {
namespace {

// tab[s][k][0..P) = log theta_kd, [P..2P) = log(1 - theta_kd), [2P] = log pi_k   (theta: K x P x S, k + K d + K P s; pi: S x K cm)
__global__ void predict_tables_kernel(int K, int P, int S, const double *__restrict__ theta, const double *__restrict__ pi,
                                      double *__restrict__ tab) {
    const size_t n = (size_t)S * K * (2 * P + 1), row = 2 * P + 1;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
        const size_t sk = e / row;
        const int c = (int)(e % row), s = (int)(sk / K), k = (int)(sk % K);
        double v;
        if (c == 2 * P) v = log(pi[s + (size_t)S * k]);
        else {
            const int d = c < P ? c : c - P;
            const double th = theta[k + (size_t)K * d + (size_t)K * P * s];
            v = c < P ? log(th) : log(1.0 - th);
        }
        tab[e] = v;
    }
}

__global__ void __launch_bounds__(128) predict_kernel(int M, int P, int W, int K, int S, const uint32_t *__restrict__ xbits,
                                                      const double *__restrict__ tab, double *__restrict__ logpred,
                                                      double *__restrict__ member) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    const uint32_t *xb = xbits + (size_t)m * W;
    const size_t row = 2 * P + 1;
    double mx = -INFINITY, acc = 0.0;     // running log-sum-exp over (s, k)
    for (int s = 0; s < S; ++s) {
        double lmx = -INFINITY, lsum = 0.0;
        for (int pass = 0; pass < (member ? 2 : 1); ++pass) {
            for (int k = 0; k < K; ++k) {
                const double *t = tab + ((size_t)s * K + k) * row;
                double ll = t[2 * P];
                for (int d = 0; d < P; ++d) ll += ((xb[d >> 5] >> (d & 31)) & 1u) ? t[d] : t[P + d];
                if (pass == 0) {
                    if (ll > lmx) { lsum = lsum * exp(lmx - ll) + 1.0; lmx = ll; }
                    else if (ll > -INFINITY) lsum += exp(ll - lmx);
                } else if (lsum > 0.0) {
                    member[m + (size_t)M * k] += exp(ll - lmx) / lsum / S;     // responsibility of cluster k under draw s
                }
            }
        }
        if (lsum > 0.0) {
            const double lse = lmx + log(lsum);                              // log p(x* | draw s)
            if (lse > mx) { acc = acc * exp(mx - lse) + 1.0; mx = lse; }
            else acc += exp(lse - mx);
        }
    }
    logpred[m] = acc > 0.0 ? mx + log(acc) - log((double)S) : -INFINITY;
}

// l = log sum_k exp(tab[g][k][2P] + sum_d tab[g][k][d or P + d]) of one packed row under draw g
__device__ __forceinline__ double draw_loglik(const uint32_t *xb, const double *tab, size_t g, int K, int P) {
    const size_t row = 2 * P + 1;
    double lmx = -INFINITY, lsum = 0.0;
    for (int k = 0; k < K; ++k) {
        const double *t = tab + (g * K + k) * row;
        double ll = t[2 * P];
        for (int d = 0; d < P; ++d) ll += ((xb[d >> 5] >> (d & 31)) & 1u) ? t[d] : t[P + d];
        if (ll > lmx) { lsum = lsum * exp(lmx - ll) + 1.0; lmx = ll; }
        else if (ll > -INFINITY) lsum += exp(ll - lmx);
    }
    return lsum > 0.0 ? lmx + log(lsum) : -INFINITY;
}

__global__ void __launch_bounds__(128) waic_fp64_kernel(int U, int P, int W, int K, int S, int CQ, int Q, int SL, int ntiles,
                                                        const uint32_t *__restrict__ rowbits, const int *__restrict__ wt,
                                                        const double *__restrict__ tab, double *__restrict__ stat,
                                                        double *__restrict__ tpart) {
    const int lane = threadIdx.x & 31, tile = blockIdx.x % ntiles;
    const int q = (blockIdx.x / ntiles) * 4 + (threadIdx.x >> 5);     // slice: chain q / Q, draws [s0, s1) of it
    if (q >= CQ) return;
    const int c = q / Q, s0 = (q % Q) * SL, s1 = min(S, s0 + SL);
    const int u = tile * 32 + lane;
    const bool valid = u < U;
    const uint32_t *xb = rowbits + (size_t)(valid ? u : 0) * W;
    const double w = valid ? (double)wt[u] : 0.0;
    double st[WAIC_STAT];
    waic_stat_init(st);
    for (int s = s0; s < s1; ++s) {
        const size_t g = (size_t)c * S + s;
        const double l = draw_loglik(xb, tab, g, K, P);
        waic_push(st, l);
        double v = valid ? w * l : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) tpart[g * ntiles + tile] = v;
    }
    if (valid)
        for (int e = 0; e < WAIC_STAT; ++e) stat[((size_t)q * U + u) * WAIC_STAT + e] = st[e];
}

// L[g Uc + u] = l of distinct row u under draw g; one warp per (tile of 32 rows, slice of SL draws), lane = row
__global__ void __launch_bounds__(128) loglik_fp64_kernel(int Uc, int P, int W, int K, long long D, long long SL, int nslices,
                                                          int ntiles, const uint32_t *__restrict__ rowbits,
                                                          const double *__restrict__ tab, double *__restrict__ L) {
    const int lane = threadIdx.x & 31, tile = blockIdx.x % ntiles;
    const int q = (blockIdx.x / ntiles) * 4 + (threadIdx.x >> 5);
    if (q >= nslices) return;
    const int u = tile * 32 + lane;
    const bool valid = u < Uc;
    const uint32_t *xb = rowbits + (size_t)(valid ? u : 0) * W;
    const long long g1 = min(D, (q + 1) * SL);
    for (long long g = q * SL; g < g1; ++g) {
        const double l = draw_loglik(xb, tab, (size_t)g, K, P);
        if (valid) L[(size_t)g * Uc + u] = l;
    }
}

// One thread per distinct row: chain c = merge of its Q slices in order, pooled = merge of the chains in order.
// cv[c U + u] = w_u (lse_c - log S), cv[(C + c) U + u] = w_u M2_c / (S - 1): the rows of the per-chain totals.
__global__ void waic_merge_kernel(int U, int C, int S, int Q, const int *__restrict__ wt, const double *__restrict__ stat,
                                  double *__restrict__ lppd, double *__restrict__ pwaic, double *__restrict__ cv) {
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    const double w = (double)wt[u];
    double pool[WAIC_STAT];
    waic_stat_init(pool);
    for (int c = 0; c < C; ++c) {
        double ch[WAIC_STAT];
        waic_stat_init(ch);
        for (int q = 0; q < Q; ++q) waic_stat_merge(ch, stat + ((size_t)(c * Q + q) * U + u) * WAIC_STAT);
        cv[(size_t)c * U + u] = w * ((ch[4] > 0.0 ? ch[3] + log(ch[4]) : -INFINITY) - log((double)S));
        cv[(size_t)(C + c) * U + u] = w * (ch[2] / (S - 1));
        waic_stat_merge(pool, ch);
    }
    const double D = (double)C * S;
    lppd[u] = (pool[4] > 0.0 ? pool[3] + log(pool[4]) : -INFINITY) - log(D);
    pwaic[u] = pool[2] / (D - 1.0);
}

// out[m] = sum_l in[m L + l], one block per m, in an order fixed by L alone
__global__ void __launch_bounds__(256) waic_sum_kernel(long long L, const double *__restrict__ in, double *__restrict__ out) {
    __shared__ double sh[256];
    const double *r = in + (size_t)blockIdx.x * L;
    double a = 0.0;
    for (long long l = threadIdx.x; l < L; l += 256) a += r[l];
    sh[threadIdx.x] = a;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[blockIdx.x] = sh[0];
}

}  // namespace

cudaError_t launch_predict_tables(int K, int P, int S, const double *theta, const double *pi, double *tab, cudaStream_t st) {
    const size_t n = (size_t)S * K * (2 * P + 1);
    predict_tables_kernel<<<(unsigned)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096), 256, 0, st>>>(K, P, S, theta, pi, tab);
    g_launches++;
    return cudaGetLastError();
}

int waic_fp64_slices(int ntiles, int C, int S) {
    const long long want = 32768 / ((long long)ntiles * C);      // enough warps to fill the GPU several times over
    return (int)(want < 1 ? 1 : (want > S ? S : want));
}

cudaError_t launch_waic_fp64(int U, int P, int W, int K, int S, int C, int Q, const uint32_t *rowbits, const int *wt,
                             const double *tab, double *stat, double *tpart, cudaStream_t st) {
    const int ntiles = (U + 31) / 32, SL = (S + Q - 1) / Q;
    const long long blocks = (long long)ntiles * ((C * Q + 3) / 4);
    if (blocks > 0x7FFFFFFFLL) return cudaErrorInvalidConfiguration;
    waic_fp64_kernel<<<(unsigned)blocks, 128, 0, st>>>(U, P, W, K, S, C * Q, Q, SL, ntiles, rowbits, wt, tab, stat, tpart);
    g_launches++;
    return cudaGetLastError();
}

cudaError_t launch_loglik_fp64(int Uc, int P, int W, int K, long long D, const uint32_t *rowbits, const double *tab,
                               double *L, cudaStream_t st) {
    const int ntiles = (Uc + 31) / 32;
    long long q = 32768 / ntiles;                                 // enough warps to fill the GPU several times over
    q = q < 1 ? 1 : (q > D ? D : q);
    const long long SL = (D + q - 1) / q, nslices = (D + SL - 1) / SL;
    const long long blocks = (long long)ntiles * ((nslices + 3) / 4);
    if (blocks > 0x7FFFFFFFLL) return cudaErrorInvalidConfiguration;
    loglik_fp64_kernel<<<(unsigned)blocks, 128, 0, st>>>(Uc, P, W, K, D, SL, (int)nslices, ntiles, rowbits, tab, L);
    g_launches++;
    return cudaGetLastError();
}

cudaError_t launch_waic_merge(int U, int C, int S, int Q, const int *wt, const double *stat, long long G, const double *tpart,
                              double *lppd, double *pwaic, double *cv, double *loglik, double *chain_tot, cudaStream_t st) {
    waic_merge_kernel<<<(U + 127) / 128, 128, 0, st>>>(U, C, S, Q, wt, stat, lppd, pwaic, cv);
    waic_sum_kernel<<<(unsigned)C * S, 256, 0, st>>>(G, tpart, loglik);
    waic_sum_kernel<<<(unsigned)(2 * C), 256, 0, st>>>(U, cv, chain_tot);
    g_launches += 3;
    return cudaGetLastError();
}

cudaError_t launch_predict(int M, int P, int W, int K, int S, const uint32_t *xbits, const double *theta, const double *pi,
                           double *tab, double *logpred, double *member, cudaStream_t st) {
    if (cudaError_t e = launch_predict_tables(K, P, S, theta, pi, tab, st)) return e;
    predict_kernel<<<(M + 127) / 128, 128, 0, st>>>(M, P, W, K, S, xbits, tab, logpred, member);
    g_launches++;
    return cudaGetLastError();
}

}  // namespace bmm
