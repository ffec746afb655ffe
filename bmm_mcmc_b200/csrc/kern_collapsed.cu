// Collapsed samplers: finite-K (collapsed_gibbs.cpp:84-225) and Dirichlet-process / CRP
// (collapsed_gibbs_dp.cpp:98-283).  The sweep is strictly sequential in i, so one chain is run by
// one 32-thread block (a single warp: lanes = clusters), the whole chain segment in one launch, and
// throughput comes from running thousands of chains concurrently.
//
// Versus the reference's O(N*P) member-list rescans per update (collapsed_gibbs.cpp:101,111-114) the
// kernel keeps integer sufficient statistics S_kd, N_k in shared memory (O(K*P) per update) and reads
// log(beta+n), log(gamma+n), log(beta+gamma+n), log(n) from tables -- the arguments are small
// integers plus constants, so the values are identical to evaluating the logs in place.
// Operation order inside one conditional follows the reference: per cluster a d-ordered sum of
// (selected log - denominator), exp(LHS + logLH), division by the sum.
#include <cstdlib>

#include "kernels.h"
#include "stephens.cuh"

namespace bmm {
namespace {

struct CSmem {
    uint32_t *x;      // [N*W]
    int *cnt;         // [K*(P+1)]
    double *logA;     // [N+1]   log(n + alpha/K)         (finite-K only)
    double *cost;     // [K*K]
    int *perm;        // [K]
    int *used;        // [K]     (dp)
    uint8_t *freec;   // [K]     (dp)
    uint8_t *z;       // [N]
};

__host__ __device__ inline size_t collapsed_layout(const CollapsedParams &p, char *base, CSmem *s) {
    size_t off = 0;
    auto take = [&](size_t bytes) { char *r = base + off; off += (bytes + 7) & ~(size_t)7; return r; };
    double *logA = (double *)take(p.dp ? 0 : (size_t)(p.N + 1) * 8);
    double *cost = (double *)take(p.relabel && p.K * p.K <= COST_SMEM_MAX ? (size_t)p.K * p.K * 8 : 0);
    uint32_t *x = (uint32_t *)take((size_t)p.N * p.W * 4);
    int *cnt = (int *)take((size_t)p.K * (p.P + 1) * 4);
    int *perm = (int *)take((size_t)p.K * 4);
    int *used = (int *)take(p.dp ? (size_t)p.K * 4 : 0);
    uint8_t *freec = (uint8_t *)take(p.dp ? (size_t)p.K : 0);
    uint8_t *z = (uint8_t *)take((size_t)p.N);
    if (s) { s->x = x; s->cnt = cnt; s->logA = logA; s->cost = cost; s->perm = perm; s->used = used; s->freec = freec; s->z = z; }
    return (off + 15) & ~(size_t)15;
}

__device__ __forceinline__ double warp_max_xor(double v) {
    for (int off = 16; off; off >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, off));
    return v;
}
__device__ __forceinline__ double warp_sum_all(double v) {
    for (int off = 1; off < 32; off <<= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}

// Where this sweep's conditional probabilities are stashed for relabelling: the batch cube slice
// during the burn-in window, the persistent probs_sample matrix afterwards, nowhere before
// (collapsed_gibbs.cpp:162-172, collapsed_gibbs_dp.cpp:190-200; probs_sample is never cleared).
__device__ inline double *stash_target(const CollapsedParams &p, int c, int j) {
    if (!p.relabel) return nullptr;
    const size_t NK = (size_t)p.N * p.K;
    if (j < p.burnin && j >= p.burnin - p.burnrelabel)
        return p.cube + ((size_t)c * p.burnrelabel + (j - p.burnin + p.burnrelabel)) * NK;
    if (j >= p.burnin) return p.probs_sample + (size_t)c * NK;
    return nullptr;
}

// Relabelling hooks + theta estimates + alpha + history rows, common to both collapsed samplers.
// Called by the whole (32-thread) block after the i loop of sweep j.
template <bool DP = false>
__device__ inline void collapsed_after_sweep(const CollapsedParams &p, CSmem &s, int c, int j, double *alpha_sh,
                                            int Kalpha, const int *used, int nused) {
    const int lane = threadIdx.x, K = p.K, P = p.P, N = p.N, ns = p.nsamples, S = hist_count(ns, p.burnin, p.thin);
    const size_t NK = (size_t)N * K;
    if (p.relabel) {
        // window sweeps were stashed straight into their cube slice (see stash_target)
        if (j >= p.burnin) {
            stephens_online_block(N, K, nullptr, p.Q + (size_t)c * NK, p.logQ + (size_t)c * NK,
                                  p.probs_sample + (size_t)c * NK, j, p.cost_g ? p.cost_g + (size_t)c * K * K : s.cost, s.perm,
                                  p.assign_ws + (size_t)c * assign_ws_bytes(K), (p.flags & 64u) != 0);  // BMM_FLAG_STEPHENS_FIXED
        }
    }
    const int sidx = hist_slot(j, p.burnin, p.thin);
    if (sidx >= 0) {
        const size_t KP = (size_t)K * P;
        // theta point estimates S_kd / N_k (collapsed_gibbs.cpp:205-219; NaN for empty clusters;
        // dp: only used labels are written, the rest stay 0: collapsed_gibbs_dp.cpp:77,266-281)
        const int nk = p.dp ? nused : K;
        for (int e = lane; e < nk * P; e += 32) {
            const int k = p.dp ? used[e / P] : e / P, d = e % P;
            const double th = (double)s.cnt[k * (P + 1) + d] / (double)s.cnt[k * (P + 1) + P];
            p.theta_out[(size_t)c * KP * S + KP * sidx + k + (size_t)K * d] = th;
            if (p.relabel) p.theta_rel_out[(size_t)c * KP * S + KP * sidx + s.perm[k] + (size_t)K * d] = th;
        }
        if (p.relabel)
            for (int k = lane; k < K; k += 32) p.perm_out[(size_t)c * S * K + sidx + (size_t)S * k] = s.perm[k];
    }
    __syncthreads();
    if (lane == 0) {
        double al = *alpha_sh;
        if (p.ralpha) al = p.ralpha[(size_t)c * ns + j];
        else if (p.alpha0 == 0.0) {
            Stream st(p.seed, (uint32_t)(p.chain_offset + c), (uint32_t)j, ST_ALPHA, 0u);
            al = update_alpha_dev<DP>(st, al, p.a, p.b, N, Kalpha);
        }
        *alpha_sh = al;
        if (sidx >= 0) p.alpha_out[(size_t)c * S + sidx] = al;
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// finite-K collapsed Gibbs.  SLOTS labels per lane (K <= 32*SLOTS).
// ------------------------------------------------------------------------------------------------
template <int SLOTS>
__global__ void __launch_bounds__(32) collapsed_kernel(const CollapsedParams p) {
    extern __shared__ __align__(16) char smem_raw[];
    __shared__ double alpha_sh;
    CSmem s;
    collapsed_layout(p, smem_raw, &s);
    const int c = blockIdx.x, lane = threadIdx.x;
    const int K = p.K, P = p.P, N = p.N, W = p.W, ns = p.nsamples, P1 = P + 1;
    const uint32_t chain = (uint32_t)(p.chain_offset + c);
    const bool replay = p.ru != nullptr;
    const size_t NK = (size_t)N * K;

    for (int e = lane; e < N * W; e += 32) s.x[e] = p.xbits[e];
    for (int e = lane; e < K * P1; e += 32) s.cnt[e] = p.cnt[(size_t)c * K * P1 + e];
    for (int e = lane; e < N; e += 32) s.z[e] = p.z_cur[(size_t)c * N + e];
    for (int k = lane; k < K; k += 32) s.perm[k] = k;
    if (lane == 0) alpha_sh = p.alpha_cur[c];
    __syncthreads();
    if (p.j_begin == 1 && p.burnin == 0 && lane == 0) p.alpha_out[(size_t)c * hist_count(ns, p.burnin, p.thin)] = alpha_sh;
    double alpha_tab = -1.0;
    const uint2 key = make_uint2((uint32_t)p.seed, chain);
    const uint32_t sid = ST_Z ^ ((uint32_t)(p.seed >> 32) << 8);

    for (int j = p.j_begin; j < p.j_end; ++j) {
        const double alpha = replay && p.ralpha ? p.ralpha[(size_t)c * ns + (j - 1)] : alpha_sh;
        if (alpha != alpha_tab) {  // log(N_k + alpha/K) table (collapsed_gibbs.cpp:105)
            for (int n = lane; n <= N; n += 32) s.logA[n] = log(n + (alpha / K));
            alpha_tab = alpha;
            __syncwarp();
        }
        const double left_denom = log(N - 1 + alpha);
        uint8_t *zrow = p.zhist + ((size_t)c * ns + j) * N;
        double *stash_dst = stash_target(p, c, j);
        const bool stash = stash_dst || p.probs_out;
        uint4 rnd = make_uint4(0, 0, 0, 0);
        for (int i = 0; i < N; ++i) {
            if (!replay && (i & 63) == 0)  // 64 updates' uniforms per Philox round: lane l serves i0+2l, i0+2l+1
                rnd = philox4x32_10(make_uint4((uint32_t)((i >> 1) + lane), 0u, sid, (uint32_t)j), key);
            const int a = s.z[i];
            double pr[SLOTS];
            double tot = 0.0;
#pragma unroll
            for (int sl = 0; sl < SLOTS; ++sl) {
                const int k = lane + 32 * sl;
                double v = 0.0;
                if (k < K) {
                    const int own = (k == a);
                    const int Nk = s.cnt[k * P1 + P] - own;
                    if (Nk > 0) {  // empty cluster: probability exactly 0 (collapsed_gibbs.cpp:104,131-133)
                        const double LHS = s.logA[Nk] - left_denom;
                        const double denom = __ldg(&p.logBG[Nk]);
                        double logLH = 0.0;
                        for (int d = 0; d < P; ++d) {
                            const int xd = (s.x[i * W + (d >> 5)] >> (d & 31)) & 1;
                            const int Sd = s.cnt[k * P1 + d] - (own & xd);
                            const double sel = xd ? __ldg(&p.logB[Sd]) : __ldg(&p.logG[Nk - Sd]);
                            logLH += sel - denom;
                        }
                        v = exp(LHS + logLH);
                    }
                }
                pr[sl] = v;
                tot += v;
            }
            tot = warp_sum_all(tot);
#pragma unroll
            for (int sl = 0; sl < SLOTS; ++sl) pr[sl] /= tot;
            if (!(tot > 0.0) || !isfinite(tot)) { if (lane == 0) p.status[c] = -9; }
            if (stash) {
#pragma unroll
                for (int sl = 0; sl < SLOTS; ++sl) {
                    const int k = lane + 32 * sl;
                    if (k < K) {
                        if (stash_dst) stash_dst[i + (size_t)N * k] = pr[sl];
                        if (p.probs_out) p.probs_out[((size_t)c * ns + j) * NK + i + (size_t)N * k] = pr[sl];
                    }
                }
            }
            auto getp = [&](int k) {
                double v = 0.0;
#pragma unroll
                for (int sl = 0; sl < SLOTS; ++sl) { double t = __shfl_sync(0xffffffffu, pr[sl], k & 31); if ((k >> 5) == sl) v = t; }
                return v;
            };
            int z;
            if (replay) {
                z = rmultinom1_replay(K, getp, p.ru + (((size_t)c * ns + j) * N + i) * p.ru_slots);
            } else {
                const int src = (i & 63) >> 1;
                const uint32_t w0 = __shfl_sync(0xffffffffu, (i & 1) ? rnd.z : rnd.x, src);
                const uint32_t w1 = __shfl_sync(0xffffffffu, (i & 1) ? rnd.w : rnd.y, src);
                z = categorical_icdf(K, getp, u53(w0, w1));
            }
            if (z != a) {
                for (int d = lane; d < P; d += 32) {
                    if ((s.x[i * W + (d >> 5)] >> (d & 31)) & 1) { s.cnt[a * P1 + d]--; s.cnt[z * P1 + d]++; }
                }
                if (lane == 0) { s.cnt[a * P1 + P]--; s.cnt[z * P1 + P]++; s.z[i] = (uint8_t)z; }
            }
            if (lane == 0) zrow[i] = (uint8_t)(z + 1);
            __syncwarp();
        }
        collapsed_after_sweep(p, s, c, j, &alpha_sh, K, nullptr, 0);
    }
    for (int e = lane; e < K * P1; e += 32) p.cnt[(size_t)c * K * P1 + e] = s.cnt[e];
    for (int e = lane; e < N; e += 32) p.z_cur[(size_t)c * N + e] = s.z[e];
    if (lane == 0) p.alpha_cur[c] = alpha_sh;
}

// ------------------------------------------------------------------------------------------------
// finite-K collapsed Gibbs, low-latency variant for K <= 32 clusters and P <= 8 variables (all the
// bundled data sets).  The sweep is one long dependent chain, so what matters is the length of that
// chain per update, not throughput: lane k keeps its cluster's sufficient statistics S_kd, N_k in
// REGISTERS, an observation is one byte of bits, the four log tables sit in shared memory, the
// normaliser is a log2(K)-step butterfly, and in Philox mode the draw compares u * total against the
// running sums (no division).  The arithmetic of one conditional -- d-ordered sum of (selected log -
// denominator), exp(LHS + logLH) -- is unchanged (collapsed_gibbs.cpp:105-130), so replay-mode parity
// holds exactly as for the generic kernel.
// ------------------------------------------------------------------------------------------------
struct FastTabs { double *logB, *logG, *logBG, *logA; uint8_t *xs; };

__host__ __device__ inline size_t collapsed_fast_extra(const CollapsedParams &p, char *base, FastTabs *t) {
    // only the alpha-dependent table is per chain; log(beta+n), log(gamma+n), log(beta+gamma+n) are shared
    // by all chains and read through L1 (keeping them here cost 24 KB per chain at N = 1000: 2 waves at C2 size)
    const size_t n1 = (size_t)p.N + 1;
    size_t off = 0;
    double *logB = nullptr, *logG = nullptr, *logBG = nullptr;
    double *logA = (double *)(base + off); off += n1 * 8;
    uint8_t *xs = (uint8_t *)(base + off); off += ((size_t)p.N + 15) & ~(size_t)15;
    if (t) { t->logB = logB; t->logG = logG; t->logBG = logBG; t->logA = logA; t->xs = xs; }
    return off;
}

template <int PM, int WIDTH>
__global__ void __launch_bounds__(32) collapsed_fast_kernel(const CollapsedParams p) {
    extern __shared__ __align__(16) char smem_raw[];
    __shared__ double alpha_sh;
    CSmem s;
    const size_t base_bytes = collapsed_layout(p, smem_raw, &s);
    FastTabs tb;
    collapsed_fast_extra(p, smem_raw + base_bytes, &tb);
    const int c = blockIdx.x, lane = threadIdx.x;
    const int K = p.K, P = p.P, N = p.N, W = p.W, ns = p.nsamples, P1 = P + 1;
    const uint32_t chain = (uint32_t)(p.chain_offset + c);
    const bool replay = p.ru != nullptr;
    const size_t NK = (size_t)N * K;

    for (int e = lane; e < N; e += 32) { tb.xs[e] = (uint8_t)(p.xbits[(size_t)e * W] & 0xFFu); s.z[e] = p.z_cur[(size_t)c * N + e]; }
    for (int k = lane; k < K; k += 32) s.perm[k] = k;
    int S[PM], Nk = 0;
#pragma unroll
    for (int d = 0; d < PM; ++d) S[d] = (lane < K && d < P) ? p.cnt[((size_t)c * K + lane) * P1 + d] : 0;
    if (lane < K) Nk = p.cnt[((size_t)c * K + lane) * P1 + P];
    if (lane == 0) alpha_sh = p.alpha_cur[c];
    __syncthreads();
    if (p.j_begin == 1 && p.burnin == 0 && lane == 0) p.alpha_out[(size_t)c * hist_count(ns, p.burnin, p.thin)] = alpha_sh;
    double alpha_tab = -1.0;
    const uint2 key = make_uint2((uint32_t)p.seed, chain);
    const uint32_t sid = ST_Z ^ ((uint32_t)(p.seed >> 32) << 8);

    for (int j = p.j_begin; j < p.j_end; ++j) {
        const double alpha = replay && p.ralpha ? p.ralpha[(size_t)c * ns + (j - 1)] : alpha_sh;
        if (alpha != alpha_tab) {  // log(N_k + alpha/K) table (collapsed_gibbs.cpp:105)
            for (int n = lane; n <= N; n += 32) tb.logA[n] = log(n + (alpha / K));
            alpha_tab = alpha;
            __syncwarp();
        }
        const double left_denom = log(N - 1 + alpha);
        uint8_t *zrow = p.zhist + ((size_t)c * ns + j) * N;
        double *stash_dst = stash_target(p, c, j);
        const bool need_probs = stash_dst || p.probs_out || replay;
        uint4 rnd = make_uint4(0, 0, 0, 0);
        int a = s.z[0];
        uint32_t xb = tb.xs[0];
        for (int i = 0; i < N; ++i) {
            if (!replay && (i & 63) == 0)
                rnd = philox4x32_10(make_uint4((uint32_t)((i >> 1) + lane), 0u, sid, (uint32_t)j), key);
            // next observation's byte and label are fetched now; they do not depend on this update
            const int inext = i + 1 < N ? i + 1 : i;
            const int a_next = s.z[inext];
            const uint32_t xb_next = tb.xs[inext];
            const int own = (lane == a);
            const int Nk1 = Nk - own;
            double v = 0.0;
            if (lane < K && Nk1 > 0) {  // empty cluster: probability exactly 0 (collapsed_gibbs.cpp:104,131-133)
                const double LHS = tb.logA[Nk1] - left_denom;
                const double denom = __ldg(&p.logBG[Nk1]);
                double sel[PM];
#pragma unroll
                for (int d = 0; d < PM; ++d) {
                    const int xd = (xb >> d) & 1;
                    const int Sd = S[d] - (own & xd);
                    sel[d] = d < P ? (xd ? __ldg(&p.logB[Sd]) : __ldg(&p.logG[Nk1 - Sd])) : 0.0;
                }
                double logLH = 0.0;
#pragma unroll
                for (int d = 0; d < PM; ++d) if (d < P) logLH += sel[d] - denom;
                v = exp(LHS + logLH);
            }
            double tot = v;
#pragma unroll
            for (int off = 1; off < WIDTH; off <<= 1) tot += __shfl_xor_sync(0xffffffffu, tot, off);
            if (!(tot > 0.0) || !isfinite(tot)) { if (lane == 0) p.status[c] = -9; }
            int z;
            if (need_probs) {
                const double pr = v / tot;
                if (lane < K) {
                    if (stash_dst) stash_dst[i + (size_t)N * lane] = pr;
                    if (p.probs_out) p.probs_out[((size_t)c * ns + j) * NK + i + (size_t)N * lane] = pr;
                }
                auto getp = [&](int k) { return __shfl_sync(0xffffffffu, pr, k); };
                if (replay) z = rmultinom1_replay(K, getp, p.ru + (((size_t)c * ns + j) * N + i) * p.ru_slots);
                else {
                    const int src = (i & 63) >> 1;
                    const uint32_t w0 = __shfl_sync(0xffffffffu, (i & 1) ? rnd.z : rnd.x, src);
                    const uint32_t w1 = __shfl_sync(0xffffffffu, (i & 1) ? rnd.w : rnd.y, src);
                    z = categorical_icdf(K, getp, u53(w0, w1));
                }
            } else {
                const int src = (i & 63) >> 1;
                const uint32_t w0 = __shfl_sync(0xffffffffu, (i & 1) ? rnd.z : rnd.x, src);
                const uint32_t w1 = __shfl_sync(0xffffffffu, (i & 1) ? rnd.w : rnd.y, src);
                const double target = u53(w0, w1) * tot;
                double cum = v;                               // inclusive prefix sums over the lanes
#pragma unroll
                for (int off = 1; off < WIDTH; off <<= 1) {
                    const double t = __shfl_up_sync(0xffffffffu, cum, off);
                    if (lane >= off) cum += t;
                }
                const unsigned hit = __ballot_sync(0xffffffffu, lane < K - 1 && target < cum);
                z = hit ? __ffs(hit) - 1 : K - 1;
            }
            if (z != a) {
                const int da = (lane == z) - (lane == a);     // +1 for the new cluster, -1 for the old one
                Nk += da;
#pragma unroll
                for (int d = 0; d < PM; ++d) S[d] += da * (int)((xb >> d) & 1);
                if (lane == 0) s.z[i] = (uint8_t)z;
            }
            if (lane == 0) zrow[i] = (uint8_t)(z + 1);
            a = a_next;
            xb = xb_next;
        }
        // the end-of-sweep code (theta estimates, relabelling) reads the statistics from shared memory
        if (lane < K) {
#pragma unroll
            for (int d = 0; d < PM; ++d) if (d < P) s.cnt[lane * P1 + d] = S[d];
            s.cnt[lane * P1 + P] = Nk;
        }
        __syncwarp();
        collapsed_after_sweep(p, s, c, j, &alpha_sh, K, nullptr, 0);
    }
    if (lane < K) {
#pragma unroll
        for (int d = 0; d < PM; ++d) if (d < P) p.cnt[((size_t)c * K + lane) * P1 + d] = S[d];
        p.cnt[((size_t)c * K + lane) * P1 + P] = Nk;
    }
    for (int e = lane; e < N; e += 32) p.z_cur[(size_t)c * N + e] = s.z[e];
    if (lane == 0) p.alpha_cur[c] = alpha_sh;
}

// ------------------------------------------------------------------------------------------------
// finite-K collapsed Gibbs in PRODUCT form (Philox mode, K <= 32, P <= 8).  The conditional of
// collapsed_gibbs.cpp:105-130 is exp(log(N_k + a/K) - log(N - 1 + a) + sum_d [log(beta + S_kd) or
// log(gamma + N_k - S_kd)] - P log(beta + gamma + N_k)); up to the factor 1 / (N - 1 + a), which is the same
// for every cluster and cancels in the normalisation, that is
//     (N_k + a/K) * prod_d (beta + S_kd  |  gamma + N_k - S_kd) / (beta + gamma + N_k)^P
// -- a handful of multiplications instead of P + 2 table look-ups, P dependent additions and an fp64 exp.
// Lane k keeps beta + S_kd and gamma + N_k - S_kd as reals in registers (they change by exactly +-1) and the
// reciprocal (beta + gamma + n)^-P comes from a table in shared memory.  The draw gathers the K weights into
// every lane when K <= 4 (no dependent shuffle chain), else uses the butterfly sum and scan.
// R = double agrees with the log form to ~1e-15 relative; R = float (precision fp32) to ~5e-7.
// The replay mode keeps the log-form kernels: bit-exact parity is defined on the reference's operation order.
// ------------------------------------------------------------------------------------------------
template <typename R> __device__ __forceinline__ R shfl_r(R v, int src);
template <> __device__ __forceinline__ double shfl_r<double>(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
template <> __device__ __forceinline__ float shfl_r<float>(float v, int src) { return __shfl_sync(0xffffffffu, v, src); }

template <typename R, int PM, int WIDTH>
__global__ void __launch_bounds__(32) collapsed_prod_kernel(const CollapsedParams p) {
    extern __shared__ __align__(16) char smem_raw[];
    __shared__ double alpha_sh;
    CSmem s;
    const size_t base_bytes = collapsed_layout(p, smem_raw, &s);
    FastTabs tb;
    collapsed_fast_extra(p, smem_raw + base_bytes, &tb);
    R *rbgp = (R *)tb.logA;                         // (beta + gamma + n)^-P, n = 0..N (the table area of the log-form kernel)
    const int c = blockIdx.x, lane = threadIdx.x;
    const int K = p.K, P = p.P, N = p.N, W = p.W, ns = p.nsamples, P1 = P + 1;
    const uint32_t chain = (uint32_t)(p.chain_offset + c);
    const size_t NK = (size_t)N * K;

    for (int e = lane; e < N; e += 32) { tb.xs[e] = (uint8_t)(p.xbits[(size_t)e * W] & 0xFFu); s.z[e] = p.z_cur[(size_t)c * N + e]; }
    for (int n = lane; n <= N; n += 32) {
        const double x = p.beta + p.gamma + n;
        double r = 1.0;
        for (int d = 0; d < P; ++d) r *= x;
        rbgp[n] = (R)(1.0 / r);
    }
    for (int k = lane; k < K; k += 32) s.perm[k] = k;
    int S[PM], Nk = 0;
#pragma unroll
    for (int d = 0; d < PM; ++d) S[d] = (lane < K && d < P) ? p.cnt[((size_t)c * K + lane) * P1 + d] : 0;
    if (lane < K) Nk = p.cnt[((size_t)c * K + lane) * P1 + P];
    R SB[PM], G[PM];                                 // beta + S_kd, gamma + N_k - S_kd; 1 for the padding d >= P
#pragma unroll
    for (int d = 0; d < PM; ++d) {
        SB[d] = d < P ? (R)(p.beta + S[d]) : (R)1;
        G[d] = d < P ? (R)(p.gamma + (Nk - S[d])) : (R)1;
    }
    if (lane == 0) alpha_sh = p.alpha_cur[c];
    __syncthreads();
    if (p.j_begin == 1 && p.burnin == 0 && lane == 0) p.alpha_out[(size_t)c * hist_count(ns, p.burnin, p.thin)] = alpha_sh;
    const uint2 key = make_uint2((uint32_t)p.seed, chain);
    const uint32_t sid = ST_Z ^ ((uint32_t)(p.seed >> 32) << 8);

    for (int j = p.j_begin; j < p.j_end; ++j) {
        const R aK = (R)(alpha_sh / K);
        uint8_t *zrow = p.zhist + ((size_t)c * ns + j) * N;
        double *stash_dst = stash_target(p, c, j);
        const bool need_probs = stash_dst || p.probs_out;
        uint4 rnd = make_uint4(0, 0, 0, 0);
        int a = s.z[0];
        uint32_t xb = tb.xs[0];
        for (int i = 0; i < N; ++i) {
            if ((i & 63) == 0)
                rnd = philox4x32_10(make_uint4((uint32_t)((i >> 1) + lane), 0u, sid, (uint32_t)j), key);
            const int inext = i + 1 < N ? i + 1 : i;
            const int a_next = s.z[inext];
            const uint32_t xb_next = tb.xs[inext];
            // this update's uniform does not depend on the weights: fetch it first
            const int src = (i & 63) >> 1;
            const uint32_t w0 = __shfl_sync(0xffffffffu, (i & 1) ? rnd.z : rnd.x, src);
            const uint32_t w1 = __shfl_sync(0xffffffffu, (i & 1) ? rnd.w : rnd.y, src);
            const R u = sizeof(R) == 4 ? (R)unit_f(u53(w0, w1)) : (R)u53(w0, w1);
            const int own = (lane == a);
            const int Nk1 = Nk - own;
            const R ownr = own ? (R)1 : (R)0;
            R v = (R)0;
            {
                R f[PM];
#pragma unroll
                for (int d = 0; d < PM; ++d) f[d] = d < P ? (((xb >> d) & 1u) ? SB[d] : G[d]) - ownr : (R)1;
#pragma unroll
                for (int w = PM / 2; w >= 1; w >>= 1)
#pragma unroll
                    for (int d = 0; d < w; ++d) f[d] *= f[d + w];
                const R head = ((R)Nk1 + aK) * rbgp[Nk1 > 0 ? Nk1 : 0];
                // empty cluster: probability exactly 0 (collapsed_gibbs.cpp:104,131-133)
                v = (lane < K && Nk1 > 0) ? head * f[0] : (R)0;
            }
            R tot;
            int z;
            if (WIDTH <= 4) {
                R g[WIDTH];
#pragma unroll
                for (int k = 0; k < WIDTH; ++k) g[k] = shfl_r<R>(v, k);
                R cum[WIDTH];
                cum[0] = g[0];
#pragma unroll
                for (int k = 1; k < WIDTH; ++k) cum[k] = cum[k - 1] + g[k];
                tot = cum[WIDTH - 1];
                const R target = u * tot;
                z = 0;
                // tot is the last of these serial prefix sums, so every cum from the last cluster with weight on equals tot
                // > u * tot (u < 1, also as a float): an empty cluster after it is never counted
#pragma unroll
                for (int k = 0; k < WIDTH - 1; ++k) z += (k < K - 1 && !(target < cum[k])) ? 1 : 0;
            } else {
                tot = v;
#pragma unroll
                for (int off = 1; off < WIDTH; off <<= 1) tot += shfl_r<R>(tot, lane ^ off);
                const R target = u * tot;
                R cum = v;                                    // inclusive prefix sums over the lanes
#pragma unroll
                for (int off = 1; off < WIDTH; off <<= 1) {
                    const R t = shfl_r<R>(cum, lane >= off ? lane - off : lane);
                    if (lane >= off) cum += t;
                }
                // The total is a butterfly sum and cum a scan: they round differently, so target can pass every cum, and
                // a scan entry of an empty cluster can exceed its predecessor's.  Only clusters with weight are drawn;
                // when no prefix passes the target the draw falls back to the last cluster with weight.
                const unsigned hit = __ballot_sync(0xffffffffu, lane < K - 1 && v > (R)0 && target < cum);
                const unsigned live = __ballot_sync(0xffffffffu, v > (R)0);
                z = hit ? __ffs(hit) - 1 : (live ? 31 - __clz(live) : K - 1);
            }
            if (!(tot > (R)0) || !isfinite(tot)) { if (lane == 0) p.status[c] = -9; }
            if (need_probs && lane < K) {
                const double pr = (double)v / (double)tot;
                if (stash_dst) stash_dst[i + (size_t)N * lane] = pr;
                if (p.probs_out) p.probs_out[((size_t)c * ns + j) * NK + i + (size_t)N * lane] = pr;
            }
            if (z != a) {
                const int da = (lane == z) - (lane == a);     // +1 for the new cluster, -1 for the old one
                const R dr = (R)da;
                Nk += da;
#pragma unroll
                for (int d = 0; d < PM; ++d) {
                    if (d < P) {
                        const int xd = (int)((xb >> d) & 1);
                        S[d] += da * xd;
                        if (xd) SB[d] += dr; else G[d] += dr;
                    }
                }
                if (lane == 0) s.z[i] = (uint8_t)z;
            }
            if (lane == 0) zrow[i] = (uint8_t)(z + 1);
            a = a_next;
            xb = xb_next;
        }
        if (lane < K) {
#pragma unroll
            for (int d = 0; d < PM; ++d) if (d < P) s.cnt[lane * P1 + d] = S[d];
            s.cnt[lane * P1 + P] = Nk;
        }
        __syncwarp();
        collapsed_after_sweep(p, s, c, j, &alpha_sh, K, nullptr, 0);
    }
    if (lane < K) {
#pragma unroll
        for (int d = 0; d < PM; ++d) if (d < P) p.cnt[((size_t)c * K + lane) * P1 + d] = S[d];
        p.cnt[((size_t)c * K + lane) * P1 + P] = Nk;
    }
    for (int e = lane; e < N; e += 32) p.z_cur[(size_t)c * N + e] = s.z[e];
    if (lane == 0) p.alpha_cur[c] = alpha_sh;
}

template <typename R, int WIDTH>
cudaError_t launch_prod_w(const CollapsedParams &p, int n_chains, size_t smem, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(collapsed_prod_kernel<R, 8, WIDTH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    collapsed_prod_kernel<R, 8, WIDTH><<<n_chains, 32, smem, st>>>(p);
    g_launches++;
    return cudaGetLastError();
}
template <typename R>
cudaError_t launch_prod(const CollapsedParams &p, int n_chains, size_t smem, cudaStream_t st) {
    if (p.K <= 2) return launch_prod_w<R, 2>(p, n_chains, smem, st);
    if (p.K <= 4) return launch_prod_w<R, 4>(p, n_chains, smem, st);
    if (p.K <= 8) return launch_prod_w<R, 8>(p, n_chains, smem, st);
    if (p.K <= 16) return launch_prod_w<R, 16>(p, n_chains, smem, st);
    return launch_prod_w<R, 32>(p, n_chains, smem, st);
}

template <int WIDTH>
cudaError_t launch_fast_w(const CollapsedParams &p, int n_chains, size_t smem, cudaStream_t st) {
    cudaError_t e = cudaFuncSetAttribute(collapsed_fast_kernel<8, WIDTH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    collapsed_fast_kernel<8, WIDTH><<<n_chains, 32, smem, st>>>(p);
    g_launches++;
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// DP / CRP collapsed Gibbs (Neal Alg. 3).  Entry `pos` of the used-cluster list is handled by lane
// pos % 32, slot pos / 32; the extra entry at pos == Kvar is the new cluster.
// ------------------------------------------------------------------------------------------------
template <int SLOTS>
__global__ void __launch_bounds__(32) dp_kernel(const CollapsedParams p) {
    extern __shared__ __align__(16) char smem_raw[];
    __shared__ double alpha_sh;
    __shared__ int nused_sh, kvar_sh;
    CSmem s;
    collapsed_layout(p, smem_raw, &s);
    const int c = blockIdx.x, lane = threadIdx.x;
    const int maxK = p.K, P = p.P, N = p.N, W = p.W, ns = p.nsamples, P1 = P + 1;
    const uint32_t chain = (uint32_t)(p.chain_offset + c);
    const bool replay = p.ru != nullptr;
    const size_t NK = (size_t)N * maxK;

    for (int e = lane; e < N * W; e += 32) s.x[e] = p.xbits[e];
    for (int e = lane; e < maxK * P1; e += 32) s.cnt[e] = p.cnt[(size_t)c * maxK * P1 + e];
    for (int e = lane; e < N; e += 32) s.z[e] = p.z_cur[(size_t)c * N + e];
    for (int k = lane; k < maxK; k += 32) {
        s.perm[k] = k;
        s.used[k] = p.dp_used[(size_t)c * (maxK + 2) + k];
        s.freec[k] = p.dp_free[(size_t)c * maxK + k];
    }
    if (lane == 0) {
        alpha_sh = p.alpha_cur[c];
        nused_sh = p.dp_used[(size_t)c * (maxK + 2) + maxK];
        kvar_sh = p.dp_used[(size_t)c * (maxK + 2) + maxK + 1];
    }
    __syncthreads();
    const uint2 key = make_uint2((uint32_t)p.seed, chain);
    const uint32_t sid = ST_Z ^ ((uint32_t)(p.seed >> 32) << 8);
    if (p.j_begin == 1 && p.burnin == 0 && lane == 0) p.alpha_out[(size_t)c * hist_count(ns, p.burnin, p.thin)] = alpha_sh;
    const double RHS_newk = P * (log(p.beta) - log(p.beta + p.gamma));  // (:71)
    // Philox mode, when the products stay inside the double range: the conditional in product form, as in
    // collapsed_prod_kernel -- N_k prod_d (beta + S_kd | gamma + N_k - S_kd) (beta + gamma + N_k)^-P for an existing
    // cluster and alpha (beta / (beta + gamma))^P for a new one (the common 1 / (N - 1 + alpha) cancels).  No table
    // logs, no max pass, no exp; normalised only when the probabilities themselves are stored.
    const bool prod = !replay && p.rBGP != nullptr;
    const double newk_c0 = exp(RHS_newk);
    bool dead = p.status[c] != 0;

    for (int j = p.j_begin; j < p.j_end && !dead; ++j) {
        const double alpha = replay && p.ralpha ? p.ralpha[(size_t)c * ns + (j - 1)] : alpha_sh;
        const double left_denom = log(N - 1 + alpha);                      // (:102)
        const double probs_newk = log(alpha) - left_denom + RHS_newk;      // (:106)
        uint8_t *zrow = p.zhist + ((size_t)c * ns + j) * N;
        double *stash_dst = stash_target(p, c, j);
        const bool stash_rel = stash_dst != nullptr;
        int nused = nused_sh, Kvar = kvar_sh;
        if (Kvar != nused) { dead = true; if (lane == 0) p.status[c] = -6; break; }
        uint4 rnd = make_uint4(0, 0, 0, 0);
        for (int i = 0; i < N; ++i) {
            if (!replay && (i & 63) == 0)
                rnd = philox4x32_10(make_uint4((uint32_t)((i >> 1) + lane), 0u, sid, (uint32_t)j), key);
            if (j > 1) {  // drop i from its cluster (:112-131)
                const int a = s.z[i];
                for (int d = lane; d < P; d += 32)
                    if ((s.x[i * W + (d >> 5)] >> (d & 31)) & 1) s.cnt[a * P1 + d]--;
                __syncwarp();
                int na = s.cnt[a * P1 + P] - 1;
                __syncwarp();
                if (lane == 0) s.cnt[a * P1 + P] = na;
                if (na == 0) {
                    // erase label a from the used list (order preserving), push it on the free heap
                    int pos = -1;
                    for (int q0 = 0; q0 < nused; q0 += 32) {
                        const int q = q0 + lane;
                        unsigned m = __ballot_sync(0xffffffffu, q < nused && s.used[q] == a);
                        if (m) { pos = q0 + __ffs(m) - 1; break; }
                    }
                    if (pos >= 0) {
                        for (int q0 = pos; q0 < nused - 1; q0 += 32) {
                            const int q = q0 + lane;
                            int v = (q < nused - 1) ? s.used[q + 1] : 0;
                            __syncwarp();
                            if (q < nused - 1) s.used[q] = v;
                            __syncwarp();
                        }
                        nused--;
                    }
                    if (lane == 0) s.freec[a]++;
                    Kvar--;
                }
                __syncwarp();
            }
            if (Kvar < 0 || Kvar != nused) { dead = true; if (lane == 0) p.status[c] = -6; break; }
            // new label = smallest free label (:169)
            int new_label = -1;
            for (int k0 = 0; k0 < maxK; k0 += 32) {
                unsigned m = __ballot_sync(0xffffffffu, (k0 + lane) < maxK && s.freec[k0 + lane] > 0);
                if (m) { new_label = k0 + __ffs(m) - 1; break; }
            }
            if (new_label < 0) { dead = true; if (lane == 0) p.status[c] = -5; break; }
            const int n_ent = Kvar + 1;
            double lp[SLOTS];
            int lab[SLOTS];
            double mx = -INFINITY;
            double pn[SLOTS], tot = 0.0;
            if (prod) {
#pragma unroll
                for (int sl = 0; sl < SLOTS; ++sl) {
                    const int pos = lane + 32 * sl;
                    double v = 0.0;
                    int label = -1;
                    if (pos < Kvar) {
                        label = s.used[pos];
                        const int Nk = s.cnt[label * P1 + P];
                        v = (double)Nk * __ldg(&p.rBGP[Nk]);
                        for (int d = 0; d < P; ++d) {
                            const int xd = (s.x[i * W + (d >> 5)] >> (d & 31)) & 1;
                            const int Sd = s.cnt[label * P1 + d];
                            v *= xd ? p.beta + Sd : p.gamma + (Nk - Sd);
                        }
                    } else if (pos == Kvar) {
                        label = new_label;
                        v = alpha * newk_c0;
                    }
                    pn[sl] = v; lab[sl] = label;
                    tot += v;
                }
                tot = warp_sum_all(tot);
                if (!(tot > 0.0) || !isfinite(tot)) { if (lane == 0) p.status[c] = -9; }
                if (stash_rel || p.probs_out) {
#pragma unroll
                    for (int sl = 0; sl < SLOTS; ++sl) pn[sl] /= tot;
                }
            } else {
#pragma unroll
            for (int sl = 0; sl < SLOTS; ++sl) {
                const int pos = lane + 32 * sl;
                double v = -INFINITY;
                int label = -1;
                if (pos < Kvar) {
                    label = s.used[pos];
                    const int Nk = s.cnt[label * P1 + P];
                    const double LHS = __ldg(&p.logN[Nk]) - left_denom;   // log N_k (:145)
                    const double denom = __ldg(&p.logBG[Nk]);
                    double logLH = 0.0;
                    for (int d = 0; d < P; ++d) {
                        const int xd = (s.x[i * W + (d >> 5)] >> (d & 31)) & 1;
                        const int Sd = s.cnt[label * P1 + d];
                        const double sel = xd ? __ldg(&p.logB[Sd]) : __ldg(&p.logG[Nk - Sd]);
                        logLH += sel - denom;
                    }
                    v = LHS + logLH;
                } else if (pos == Kvar) {
                    label = new_label;
                    v = probs_newk;
                }
                lp[sl] = v; lab[sl] = label;
                mx = fmax(mx, v);
            }
            mx = warp_max_xor(mx);
#pragma unroll
            for (int sl = 0; sl < SLOTS; ++sl) { pn[sl] = (lab[sl] >= 0) ? exp(lp[sl] - mx) : 0.0; tot += pn[sl]; }
            tot = warp_sum_all(tot);
#pragma unroll
            for (int sl = 0; sl < SLOTS; ++sl) pn[sl] /= tot;                // exp-normalise (:174-186)
            }
            if (stash_rel || p.probs_out) {                                 // stored by LABEL (:190-200)
#pragma unroll
                for (int sl = 0; sl < SLOTS; ++sl)
                    if (lab[sl] >= 0 && lab[sl] < maxK) {
                        if (stash_rel) stash_dst[i + (size_t)N * lab[sl]] = pn[sl];
                        if (p.probs_out) p.probs_out[((size_t)c * ns + j) * NK + i + (size_t)N * lab[sl]] = pn[sl];
                    }
            }
            unsigned best = 0xffffffffu;  // (rank << 8) | pos of the first entry of the walk with rT <= mass
            if (replay) {
                // RcppArmadillo::sample(choices, 1, false, probs_norm): renormalise, walk in descending
                // order (collapsed_gibbs_dp.cpp:207) -- reproduced exactly so a recorded uniform picks the
                // same label as in the reference
                double tot2 = 0.0;
#pragma unroll
                for (int sl = 0; sl < SLOTS; ++sl) tot2 += pn[sl];
                tot2 = warp_sum_all(tot2);
                double q[SLOTS], mass[SLOTS];
                int rank[SLOTS];
#pragma unroll
                for (int sl = 0; sl < SLOTS; ++sl) { q[sl] = pn[sl] / tot2; mass[sl] = 0.0; rank[sl] = 0; }
                for (int src = 0; src < n_ent; ++src) {
                    double qs = 0.0;
#pragma unroll
                    for (int sl = 0; sl < SLOTS; ++sl) { double t = __shfl_sync(0xffffffffu, q[sl], src & 31); if ((src >> 5) == sl) qs = t; }
#pragma unroll
                    for (int sl = 0; sl < SLOTS; ++sl) {
                        const int pos = lane + 32 * sl;
                        const bool before = (qs > q[sl]) || (qs == q[sl] && src < pos);   // stable descending
                        if (before) rank[sl]++;
                        if (before || src == pos) mass[sl] += qs;
                    }
                }
                const double rT = p.ru[(((size_t)c * ns + j) * N + i) * p.ru_slots];
#pragma unroll
                for (int sl = 0; sl < SLOTS; ++sl) {
                    const int pos = lane + 32 * sl;
                    if (pos < n_ent && (rank[sl] == n_ent - 1 || rT <= mass[sl])) best = min(best, ((unsigned)rank[sl] << 8) | (unsigned)pos);
                }
            } else {
                // Philox: the same categorical law by inverse CDF over the used-list order (the order of the
                // walk does not change the distribution of the draw), one warp scan instead of a sort
                const int usrc = (i & 63) >> 1;
                const uint32_t w0 = __shfl_sync(0xffffffffu, (i & 1) ? rnd.z : rnd.x, usrc);
                const uint32_t w1 = __shfl_sync(0xffffffffu, (i & 1) ? rnd.w : rnd.y, usrc);
                const double rT = u53(w0, w1);
                double cum[SLOTS], base = 0.0;
#pragma unroll
                for (int sl = 0; sl < SLOTS; ++sl) {
                    double v = pn[sl];
#pragma unroll
                    for (int off = 1; off < 32; off <<= 1) {
                        const double t = __shfl_up_sync(0xffffffffu, v, off);
                        if (lane >= off) v += t;
                    }
                    cum[sl] = v + base;
                    base = __shfl_sync(0xffffffffu, cum[sl], 31);
                }
                const double target = rT * base;
#pragma unroll
                for (int sl = 0; sl < SLOTS; ++sl) {
                    const int pos = lane + 32 * sl;
                    if (pos < n_ent && (pos == n_ent - 1 || target <= cum[sl])) best = min(best, ((unsigned)pos << 8) | (unsigned)pos);
                }
            }
            best = __reduce_min_sync(0xffffffffu, best);
            const int wpos = (int)(best & 0xffu);
            int ret = (wpos == Kvar) ? new_label : s.used[wpos];
            if (ret == new_label) {
                if (Kvar < maxK - 1) {                   // create (:213-217)
                    if (lane == 0) { s.freec[new_label]--; s.used[nused] = new_label; }
                    nused++; Kvar++;
                } else {                                 // truncation fallback (:218-230, quirk 9)
                    int smallest = 0, ssize = N + 1;
                    for (int k = 0; k < Kvar; ++k) {
                        const int sz = s.cnt[s.used[k] * P1 + P];
                        if (sz < ssize) { ssize = sz; smallest = k; }
                    }
                    if (Kvar > 0) ret = smallest;        // an index into used_clusters, not a label
                }
            }
            if (ret < 0 || ret >= maxK) { dead = true; if (lane == 0) p.status[c] = -6; break; }
            __syncwarp();
            for (int d = lane; d < P; d += 32)
                if ((s.x[i * W + (d >> 5)] >> (d & 31)) & 1) s.cnt[ret * P1 + d]++;
            if (lane == 0) { s.cnt[ret * P1 + P]++; s.z[i] = (uint8_t)ret; zrow[i] = (uint8_t)(ret + 1); }
            __syncwarp();
        }
        if (dead) break;
        if (lane == 0) { nused_sh = nused; kvar_sh = Kvar; }
        if (p.kactive_out && lane == 0) p.kactive_out[(size_t)c * ns + j] = Kvar;
        __syncthreads();
        collapsed_after_sweep<true>(p, s, c, j, &alpha_sh, Kvar, s.used, nused);
    }
    __syncthreads();
    for (int e = lane; e < maxK * P1; e += 32) p.cnt[(size_t)c * maxK * P1 + e] = s.cnt[e];
    for (int e = lane; e < N; e += 32) p.z_cur[(size_t)c * N + e] = s.z[e];
    for (int k = lane; k < maxK; k += 32) {
        p.dp_used[(size_t)c * (maxK + 2) + k] = s.used[k];
        p.dp_free[(size_t)c * maxK + k] = s.freec[k];
    }
    if (lane == 0) {
        p.alpha_cur[c] = alpha_sh;
        p.dp_used[(size_t)c * (maxK + 2) + maxK] = nused_sh;
        p.dp_used[(size_t)c * (maxK + 2) + maxK + 1] = kvar_sh;
    }
}

template <int SLOTS>
cudaError_t launch_slots(const CollapsedParams &p, int n_chains, size_t smem, cudaStream_t st) {
    cudaError_t e;
    if (p.dp) {
        e = cudaFuncSetAttribute(dp_kernel<SLOTS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        dp_kernel<SLOTS><<<n_chains, 32, smem, st>>>(p);
    } else {
        e = cudaFuncSetAttribute(collapsed_kernel<SLOTS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        collapsed_kernel<SLOTS><<<n_chains, 32, smem, st>>>(p);
    }
    g_launches++;
    return cudaGetLastError();
}

}  // namespace

static bool collapsed_fast_ok(const CollapsedParams &p) {
    return !p.dp && p.K <= 32 && p.P <= 8 &&
           collapsed_layout(p, (char *)0, nullptr) + collapsed_fast_extra(p, (char *)0, nullptr) <= 200 * 1024;
}

size_t collapsed_smem_bytes(const CollapsedParams &p) {
    return collapsed_layout(p, (char *)0, nullptr) + (collapsed_fast_ok(p) ? collapsed_fast_extra(p, (char *)0, nullptr) : 0);
}

cudaError_t launch_collapsed(const CollapsedParams &p, int n_chains, cudaStream_t st) {
    size_t smem = collapsed_layout(p, (char *)0, nullptr);   // the generic kernels: no table area (occupancy!)
    // Measured on B200 (K3_N1000_P5): the register-resident kernel gives 1.07e6 vs 0.88e6 updates/s for one
    // chain and 1.01e9 vs 0.86e9 for 1024 chains, so it is used whenever the shape fits (K <= 32, P <= 8).
    // BMM_COLLAPSED_KERNEL=fast|generic overrides (the parity tests run both).
    const char *force = getenv("BMM_COLLAPSED_KERNEL");
    const bool want_fast = force ? force[0] != 'g' : true;
    if (want_fast && collapsed_fast_ok(p)) {
        smem += collapsed_fast_extra(p, (char *)0, nullptr);
        // Philox mode: the product-form kernel (no exp, no log tables); replay keeps the reference's operation order.
        // BMM_COLLAPSED_KERNEL=log keeps the log form in Philox mode too (A/B).
        if (!p.ru && !(force && force[0] == 'l')) {
            // the chain-parallel fp32 variant is opt-in through precision = fp32
            return p.fp32 ? launch_prod<float>(p, n_chains, smem, st) : launch_prod<double>(p, n_chains, smem, st);
        }
        if (p.K <= 2) return launch_fast_w<2>(p, n_chains, smem, st);
        if (p.K <= 4) return launch_fast_w<4>(p, n_chains, smem, st);
        if (p.K <= 8) return launch_fast_w<8>(p, n_chains, smem, st);
        if (p.K <= 16) return launch_fast_w<16>(p, n_chains, smem, st);
        return launch_fast_w<32>(p, n_chains, smem, st);
    }
    if (p.K <= 32) return launch_slots<1>(p, n_chains, smem, st);
    if (p.K <= 64) return launch_slots<2>(p, n_chains, smem, st);
    if (p.K <= 128) return launch_slots<4>(p, n_chains, smem, st);
    return launch_slots<8>(p, n_chains, smem, st);
}

}  // namespace bmm
