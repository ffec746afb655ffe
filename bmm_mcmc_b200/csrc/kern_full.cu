// Uncollapsed samplers (finite-K full Gibbs and truncated stick-breaking), one chain per thread
// block, whole chain segments in one launch.  Replaces, per sweep,
//   z-sweep              /root/reference/src/full_gibbs.cpp:87-157, stickbreaking.cpp:70-140
//   sufficient statistics full_gibbs.cpp:182-200, stickbreaking.cpp:164-186
//   pi / sticks / theta / alpha draws  full_gibbs.cpp:10-27,202-230, stickbreaking.cpp:187-235,
//                                      utils.cpp:6-14
//   online relabelling   full_gibbs.cpp:162-176 -> stephens.cpp:66-94
//
// Design: given (theta, pi) every observation with the same data row x has the same conditional
// probability vector, so the block first builds a row table prob[U x K] (U unique rows; U = 32 at
// most for the bundled P = 5 datasets), then each observation only draws from its row.  Counts are
// accumulated as a (row, label) histogram in shared memory and folded into c_k / V_kd once per
// sweep.  Stephens' Q lives in the same row space.  All probability arithmetic is fp64 and follows
// the reference's operation order (sum over d, exp(log pi + loglh), running normaliser).
#include "kernels.h"
#include "stephens.cuh"

namespace bmm {

unsigned long long g_launches = 0;

namespace {

constexpr int FULL_SMEM_ROWS_MAX = 3072;  // U*K entries kept in shared memory

struct FullSmem {
    double *theta, *w1, *w0, *pi, *lpi, *gsc, *cost, *scal, *prob, *Q, *logQ;
    int *ck, *Vkd, *perm, *hist;
};

__host__ __device__ inline size_t full_layout(const FullParams &p, char *base, FullSmem *s) {
    const size_t KP = (size_t)p.K * p.P, K = p.K, UK = (size_t)p.U * p.K;
    size_t off = 0;
    auto takeD = [&](size_t n) { double *r = (double *)(base + off); off += n * sizeof(double); return r; };
    auto takeI = [&](size_t n) { int *r = (int *)(base + off); off += n * sizeof(int); return r; };
    double *theta = takeD(KP), *w1 = takeD(KP), *w0 = takeD(KP), *pi = takeD(K), *lpi = takeD(K), *gsc = takeD(K);
    double *cost = takeD(K * K <= (size_t)COST_SMEM_MAX ? K * K : 0), *scal = takeD(8);   // [0] alpha, [4..7] the Gamma draws of its update
    double *prob = nullptr, *Q = nullptr, *logQ = nullptr;
    if (p.use_hist) { prob = takeD(UK); if (p.relabel) { Q = takeD(UK); logQ = takeD(UK); } }
    int *ck = takeI(K), *Vkd = takeI(KP), *perm = takeI(K), *hist = nullptr;
    if (p.use_hist) hist = takeI(UK);
    if (s) { s->theta = theta; s->w1 = w1; s->w0 = w0; s->pi = pi; s->lpi = lpi; s->gsc = gsc; s->cost = cost;
             s->scal = scal; s->prob = prob; s->Q = Q; s->logQ = logQ; s->ck = ck; s->Vkd = Vkd; s->perm = perm; s->hist = hist; }
    return (off + 15) & ~(size_t)15;
}

// Per-phase cycle accounting (compile with -DBMM_CHAIN_PHASE_CLOCKS; tools/chain_phases.py): lane 0 of each of the first
// four warps reads clock64() at the end of every phase of a sweep and adds the cycles since its previous reading to
// // its warp's total in shared memory; the block adds them to g_chain_phase[chain][warp][phase] when it exits.  A phase's
// total includes the wait at the barrier that closes it, except for E and F (relabelling and parameter draws, side by
// side on warps 1 and 0 of a block of two warps or more): their wait is PH_WAIT_EF.  Slot CHAIN_PHASE_SWEEPS counts the
// sweeps.  The default build compiles none of it.
enum { PH_A = 0, PH_B, PH_C, PH_D, PH_E, PH_F, PH_HIST, PH_WAIT_EF, CHAIN_PHASE_SWEEPS, CHAIN_PHASES };
#ifdef BMM_CHAIN_PHASE_CLOCKS
constexpr int CHAIN_PHASE_MAX_CHAINS = 4096;
__device__ unsigned long long g_chain_phase[CHAIN_PHASE_MAX_CHAINS * 4 * CHAIN_PHASES];
__shared__ unsigned long long s_chain_phase[4][CHAIN_PHASES];   // this launch's totals, added to g_chain_phase at exit
#define PHASE_INIT()                                                                                               \
    do {                                                                                                           \
        if (threadIdx.x < 4 * CHAIN_PHASES) s_chain_phase[threadIdx.x / CHAIN_PHASES][threadIdx.x % CHAIN_PHASES] = 0; \
        __syncthreads();                                                                                           \
    } while (0)
#define PHASE_BEGIN() unsigned long long phase_t_ = clock64()
#define PHASE_END(ph)                                                                                              \
    do {                                                                                                           \
        if ((threadIdx.x & 31) == 0 && threadIdx.x < 128) {                                                        \
            const unsigned long long n_ = clock64();                                                               \
            s_chain_phase[threadIdx.x >> 5][(ph)] += n_ - phase_t_;                                                \
            phase_t_ = n_;                                                                                         \
        }                                                                                                          \
    } while (0)
#define PHASE_SWEEP() do { if ((threadIdx.x & 31) == 0 && threadIdx.x < 128) s_chain_phase[threadIdx.x >> 5][CHAIN_PHASE_SWEEPS] += 1; } while (0)
#define PHASE_FLUSH()                                                                                              \
    do {                                                                                                           \
        __syncthreads();                                                                                           \
        if (threadIdx.x < 4 * CHAIN_PHASES && c < CHAIN_PHASE_MAX_CHAINS)                                          \
            g_chain_phase[(size_t)c * 4 * CHAIN_PHASES + threadIdx.x] += s_chain_phase[threadIdx.x / CHAIN_PHASES][threadIdx.x % CHAIN_PHASES]; \
    } while (0)
#else
#define PHASE_INIT() do {} while (0)
#define PHASE_BEGIN() do {} while (0)
#define PHASE_END(ph) do {} while (0)
#define PHASE_SWEEP() do {} while (0)
#define PHASE_FLUSH() do {} while (0)
#endif

__device__ __forceinline__ void full_chain_body(const FullParams &p) {
    extern __shared__ __align__(16) char smem_raw[];
    FullSmem s;
    full_layout(p, smem_raw, &s);
    const int c = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
    const int K = p.K, P = p.P, U = p.U, N = p.N, W = p.W, KP = K * P, ns = p.nsamples;
    const int S = hist_count(ns, p.burnin, p.thin);
    const size_t UK = (size_t)U * K;
    const uint32_t chain = (uint32_t)(p.chain_offset + c);
    const bool replay = p.ru != nullptr;
    PHASE_INIT();
    double *prob = p.use_hist ? s.prob : p.prob_g + (size_t)c * UK;
    double *Q = (p.use_hist && p.relabel) ? s.Q : (p.Q ? p.Q + (size_t)c * UK : nullptr);
    double *logQ = (p.use_hist && p.relabel) ? s.logQ : (p.logQ ? p.logQ + (size_t)c * UK : nullptr);
    int *hist = s.hist;
    char *aws = p.assign_ws + (size_t)c * assign_ws_bytes(K);

    for (int t = tid; t < KP; t += nthr) s.theta[t] = p.theta_cur[(size_t)c * KP + t];
    for (int t = tid; t < K; t += nthr) { s.pi[t] = p.pi_cur[(size_t)c * K + t]; s.perm[t] = t; }
    if (tid == 0) s.scal[0] = p.alpha_cur[c];
    if (p.use_hist && p.relabel)
        for (size_t e = tid; e < UK; e += nthr) { s.Q[e] = p.Q[(size_t)c * UK + e]; s.logQ[e] = p.logQ[(size_t)c * UK + e]; }
    __syncthreads();
    if (p.j_begin == 1 && p.burnin == 0) {  // iteration 0 of the returned histories = initial state
        for (int t = tid; t < KP; t += nthr) p.theta_out[(size_t)c * KP * S + t] = s.theta[t];
        for (int t = tid; t < K; t += nthr) p.pi_out[(size_t)c * S * K + (size_t)S * t] = s.pi[t];
        if (tid == 0) p.alpha_out[(size_t)c * S] = s.scal[0];
    }

    for (int j = p.j_begin; j < p.j_end; ++j) {
        PHASE_BEGIN();
        if (replay) {  // state of sweep j-1 comes from the recorded run
            for (int t = tid; t < KP; t += nthr) s.theta[t] = p.rtheta[(size_t)c * KP * ns + (size_t)KP * (j - 1) + t];
            for (int t = tid; t < K; t += nthr) s.pi[t] = p.rpi[(size_t)c * ns * K + (j - 1) + (size_t)ns * t];
            if (tid == 0) s.scal[0] = p.ralpha[(size_t)c * ns + (j - 1)];
            __syncthreads();
        }
        // ---- A: log tables of theta_{j-1}, pi_{j-1} (hoisted out of the i loop of full_gibbs.cpp:97)
        for (int t = tid; t < KP; t += nthr) {
            double th = s.theta[t];
            s.w1[t] = log(th);
            s.w0[t] = log(1 - th);
            s.Vkd[t] = 0;
        }
        for (int t = tid; t < K; t += nthr) { s.lpi[t] = log(s.pi[t]); s.ck[t] = 0; }
        __syncthreads();
        PHASE_END(PH_A);
        // ---- B: row table prob[u, k] = exp(log pi_k + loglh_k(u)) / sum (full_gibbs.cpp:92-122)
        for (int u = tid; u < U; u += nthr) {
            const uint32_t *xb = p.rowbits + (size_t)u * W;
            double cum = 0.0, mx = 0.0;
            if (p.flags & 1u) {  // BMM_FLAG_STABLE_SOFTMAX
                mx = -INFINITY;
                for (int k = 0; k < K; ++k) {
                    double ll = 0.0;
                    for (int d = 0; d < P; ++d) ll += ((xb[d >> 5] >> (d & 31)) & 1u) ? s.w1[k + K * d] : s.w0[k + K * d];
                    mx = fmax(mx, s.lpi[k] + ll);
                }
            }
            for (int k = 0; k < K; ++k) {
                double ll = 0.0;
                for (int d = 0; d < P; ++d) ll += ((xb[d >> 5] >> (d & 31)) & 1u) ? s.w1[k + K * d] : s.w0[k + K * d];
                if (p.loglik_out) p.ll_g[(size_t)c * UK + u + (size_t)U * k] = ll;
                double sk = exp(s.lpi[k] + ll - mx);
                prob[u + (size_t)U * k] = sk;
                cum += sk;
            }
            if (!(cum > 0.0) || !isfinite(cum)) p.status[c] = -9;  // BMM_ERR_PROB
            for (int k = 0; k < K; ++k) {
                prob[u + (size_t)U * k] /= cum;
                if (hist) hist[u + (size_t)U * k] = 0;
            }
        }
        __syncthreads();
        PHASE_END(PH_B);
        if (p.probs_out) {
            double *po = p.probs_out + ((size_t)c * ns + j) * N * K;
            for (size_t e = tid; e < (size_t)N * K; e += nthr) po[e] = prob[p.rowid[e % N] + (size_t)U * (e / N)];
        }
        if (p.loglik_out) {
            double *lo = p.loglik_out + ((size_t)c * ns + j) * N * K;
            for (size_t e = tid; e < (size_t)N * K; e += nthr) lo[e] = p.ll_g[(size_t)c * UK + p.rowid[e % N] + (size_t)U * (e / N)];
        }
        // ---- C: allocation draws (full_gibbs.cpp:133-142) + fused sufficient statistics
        uint8_t *zrow = p.zhist + ((size_t)c * ns + j) * N;
        if (replay) {
            for (int i = tid; i < N; i += nthr) {
                const int r = p.rowid[i];
                const double *uu = p.ru + (((size_t)c * ns + j) * N + i) * p.ru_slots;
                int z = rmultinom1_replay(K, [&](int k) { return prob[r + (size_t)U * k]; }, uu);
                zrow[i] = (uint8_t)(z + 1);
                if (hist) atomicAdd(&hist[r + (size_t)U * z], 1);
                else {
                    atomicAdd(&s.ck[z], 1);
                    const uint32_t *xb = p.rowbits + (size_t)r * W;
                    for (int d = 0; d < P; ++d) if ((xb[d >> 5] >> (d & 31)) & 1u) atomicAdd(&s.Vkd[z + K * d], 1);
                }
            }
        } else {
            const uint2 key = make_uint2((uint32_t)p.seed, chain);
            const uint32_t sid = ST_Z ^ ((uint32_t)(p.seed >> 32) << 8);
            for (int i4 = tid; 4 * i4 < N; i4 += nthr) {
                const uint4 rnd = philox4x32_10(make_uint4((uint32_t)i4, 0u, sid, (uint32_t)j), key);
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                    const int i = 4 * i4 + h;
                    if (i >= N) break;
                    const double uu = u32_unit(philox_word(rnd, h));
                    const int r = p.rowid[i];
                    int z = categorical_icdf(K, [&](int k) { return prob[r + (size_t)U * k]; }, uu);
                    zrow[i] = (uint8_t)(z + 1);
                    if (hist) atomicAdd(&hist[r + (size_t)U * z], 1);
                    else {
                        atomicAdd(&s.ck[z], 1);
                        const uint32_t *xb = p.rowbits + (size_t)r * W;
                        for (int d = 0; d < P; ++d) if ((xb[d >> 5] >> (d & 31)) & 1u) atomicAdd(&s.Vkd[z + K * d], 1);
                    }
                }
            }
        }
        __syncthreads();
        PHASE_END(PH_C);
        // ---- D: fold the (row, label) histogram into c_k and V_kd (full_gibbs.cpp:182-200)
        if (hist) {
            for (int t = tid; t < KP + K; t += nthr) {
                int acc = 0;
                if (t < KP) {
                    const int k = t % K, d = t / K;
                    for (int u = 0; u < U; ++u)
                        if ((p.rowbits[(size_t)u * W + (d >> 5)] >> (d & 31)) & 1u) acc += hist[u + (size_t)U * k];
                    s.Vkd[t] = acc;
                } else {
                    const int k = t - KP;
                    for (int u = 0; u < U; ++u) acc += hist[u + (size_t)U * k];
                    s.ck[k] = acc;
                }
            }
            __syncthreads();
        }
        PHASE_END(PH_D);
        // ---- E: Stephens relabelling hooks (full_gibbs.cpp:146-176)   F: parameter draws
        // E (reads prob, Q; writes Q, perm) and F (reads the counts; writes theta, pi, alpha) are independent.  Both
        // are narrow -- K*K costs, K + K*P + 4 draws -- so with two or more warps per chain warp 1 relabels
        // while warp 0 draws, each synchronising with __syncwarp; a one-warp block runs them in turn.
        const double alpha_prev = s.scal[0];
        auto phase_e = [&](const int tid, const int nthr, auto sync) {
            if (p.relabel && j >= p.burnin)
                stephens_online_group(U, K, p.wt, Q, logQ, prob, j, p.cost_g ? p.cost_g + (size_t)c * K * K : s.cost, s.perm, aws,
                                      (p.flags & 64u) != 0 /* BMM_FLAG_STEPHENS_FIXED */, tid, nthr, sync);
        };
        auto phase_f = [&](const int tid, const int nthr, auto sync) {
            if (replay) {
                for (int t = tid; t < KP; t += nthr) s.theta[t] = p.rtheta[(size_t)c * KP * ns + (size_t)KP * j + t];
                for (int t = tid; t < K; t += nthr) s.pi[t] = p.rpi[(size_t)c * ns * K + j + (size_t)ns * t];
                if (tid == 0) s.scal[0] = p.ralpha[(size_t)c * ns + j];
                return;
            }
            // alpha update: its Gamma draws ride along on spare lanes (substream q of ST_ALPHA); the two whose
            // shape needs K_viable (stick-breaking) are drawn after the sticks
            const int nalpha = p.alpha0 == 0.0 ? (p.stickbreaking ? 2 : 4) : 0;
            // Every lane describes its draw (substream, shapes) and then all of them run ONE copy of the sampler:
            // with a separate inlined Gamma/Beta call per kind of parameter the diverged lanes executed the
            // rejection sampler four times in turn (pi, theta x, theta y, alpha) instead of twice.
            for (int t = tid; t < K + KP + nalpha; t += nthr) {
                uint32_t sid, idx;
                double sa, sb = 0.0;
                bool is_beta = false;
                double *dst;
                if (t < K) {
                    idx = (uint32_t)t; dst = &s.gsc[t];
                    if (!p.stickbreaking) {  // Dirichlet via K Gamma(alpha/K + c_k, 1) (full_gibbs.cpp:202-210)
                        sid = ST_PI; sa = alpha_prev / K + s.ck[t];
                    } else {                 // v_k ~ Beta(1 + c_k, alpha + sum_{l>k} c_l) (stickbreaking.cpp:187-193)
                        int later = 0;
                        for (int l = t + 1; l < K; ++l) later += s.ck[l];
                        sid = ST_STICK; sa = 1.0 + s.ck[t]; sb = alpha_prev + later; is_beta = true;
                    }
                } else if (t < K + KP) {     // theta_kd ~ Beta(beta + V_kd, gamma + c_k - V_kd) (:213-225)
                    const int e = t - K, k = e % K, d = e / K;
                    sid = ST_THETA; idx = (uint32_t)(k * P + d); dst = &s.theta[e];
                    sa = p.beta + s.Vkd[e]; sb = p.gamma + s.ck[k] - s.Vkd[e]; is_beta = true;
                } else {
                    const int q = t - K - KP;
                    sid = ST_ALPHA; idx = (uint32_t)q; dst = &s.scal[4 + q];
                    sa = alpha_gamma_shape(q, alpha_prev, p.a, N, K);
                }
                Stream st(p.seed, chain, (uint32_t)j, sid, idx);
                double val = st.gamma(sa);
                if (is_beta) {               // Stream::beta: x / (x + y), 0.5 when both vanish
                    const double y = st.gamma(sb), sum = val + y;
                    val = sum > 0.0 ? val / sum : 0.5;
                }
                *dst = val;
            }
            sync();
            if (!p.stickbreaking) {
                for (int t = tid; t < K; t += nthr) {
                    double sum = 0.0;
                    for (int k = 0; k < K; ++k) sum += s.gsc[k];
                    s.pi[t] = s.gsc[t] / sum;
                }
                if (tid == 0 && p.alpha0 == 0.0) s.scal[0] = alpha_combine(s.scal + 4, p.a, p.b, N, K);
            } else {                         // stick-breaking weights (stickbreaking.cpp:195-214)
                if (tid == 0) {
                    s.gsc[K - 1] = 1.0;
                    int K_viable = 0;
                    s.pi[0] = s.gsc[0];
                    if (s.pi[0] > 0.01) K_viable++;
                    double cumprod = 1 - s.gsc[0];
                    for (int k = 1; k < K; ++k) {
                        s.pi[k] = cumprod * s.gsc[k];
                        if (s.pi[k] > 0.01) K_viable++;
                        cumprod *= (1 - s.gsc[k]);
                    }
                    s.scal[1] = (double)K_viable;
                }
                if (p.alpha0 == 0.0) {       // the two draws whose shape is a + K_viable (- 1), side by side
                    sync();
                    const int K_viable = (int)s.scal[1];
                    for (int q = 2 + tid; q < 4; q += nthr) {
                        Stream st(p.seed, chain, (uint32_t)j, ST_ALPHA, (uint32_t)q);
                        s.scal[4 + q] = st.gamma(alpha_gamma_shape(q, alpha_prev, p.a, N, K_viable));
                    }
                    sync();
                    if (tid == 0) s.scal[0] = alpha_combine(s.scal + 4, p.a, p.b, N, K_viable);
                }
            }
        };
        if (p.relabel && j < p.burnin && j >= p.burnin - p.burnrelabel) {
            double *dst = p.cube + ((size_t)c * p.burnrelabel + (j - p.burnin + p.burnrelabel)) * UK;
            for (size_t e = tid; e < UK; e += nthr) dst[e] = prob[e];
        }
        if (nthr >= 64) {
            const int w = tid >> 5, lane = tid & 31;
            if (w == 0) phase_f(lane, 32, [] { __syncwarp(); });
            else if (w == 1) phase_e(lane, 32, [] { __syncwarp(); });
            PHASE_END(w == 1 ? PH_E : PH_F);
        } else {
            phase_e(tid, nthr, [] { __syncthreads(); });
            PHASE_END(PH_E);
            phase_f(tid, nthr, [] { __syncthreads(); });
            PHASE_END(PH_F);
        }
        __syncthreads();
        PHASE_END(PH_WAIT_EF);
        const int sidx = hist_slot(j, p.burnin, p.thin);
        if (sidx >= 0) {
            for (int t = tid; t < KP; t += nthr) {
                p.theta_out[(size_t)c * KP * S + (size_t)KP * sidx + t] = s.theta[t];
                if (p.relabel) {
                    const int k = t % K, d = t / K;
                    p.theta_rel_out[(size_t)c * KP * S + (size_t)KP * sidx + s.perm[k] + K * d] = s.theta[t];
                }
            }
            for (int t = tid; t < K; t += nthr) {
                p.pi_out[(size_t)c * S * K + sidx + (size_t)S * t] = s.pi[t];
                if (p.relabel) p.perm_out[(size_t)c * S * K + sidx + (size_t)S * t] = s.perm[t];
            }
            if (tid == 0) p.alpha_out[(size_t)c * S + sidx] = s.scal[0];
        }
        __syncthreads();
        PHASE_END(PH_HIST);
        PHASE_SWEEP();
    }
    // persist chain state for the next segment
    for (int t = tid; t < KP; t += nthr) p.theta_cur[(size_t)c * KP + t] = s.theta[t];
    for (int t = tid; t < K; t += nthr) p.pi_cur[(size_t)c * K + t] = s.pi[t];
    if (tid == 0) p.alpha_cur[c] = s.scal[0];
    if (p.use_hist && p.relabel)
        for (size_t e = tid; e < UK; e += nthr) { p.Q[(size_t)c * UK + e] = s.Q[e]; p.logQ[(size_t)c * UK + e] = s.logQ[e]; }
    PHASE_FLUSH();
}

// Two entry points over one body: blocks of 64 threads are capped at 144 registers so that seven of them fit
// an SM (1024 chains resident on 148 SMs); the 32- and 128-thread launches use the uncapped one.
__global__ void __launch_bounds__(128) full_chain_kernel(const FullParams p) { full_chain_body(p); }
__global__ void __launch_bounds__(64, 7) full_chain_kernel_64(const FullParams p) { full_chain_body(p); }

// ---- chain_sweep_kernel: the same chain as full_chain_kernel, specialised to the case most runs take ----------------
// Philox mode, the (row, label) histogram in shared memory, no probability / log-likelihood probes.  Every draw, every
// fp64 expression and its evaluation order are those of full_chain_body, so both kernels return the same bits
// (tests/test_gpu_chain_kernel.py); what differs is the code around them:
//   - the per-plan switches (stick-breaking, relabelling and its variant, sampled alpha) are template parameters, and
//     the replay, probe and direct-count paths are absent, so the sweep loop is a fraction of the generic body;
//   - one copy of the Gamma rejection sampler serves both Gammas of a Beta draw (param_draw);
//   - the distinct rows and the observation -> row map live in shared memory (the map as bytes when U <= 256);
//   - with N % 4 == 0 the four labels of one Philox block are stored as one word;
//   - the log tables are rebuilt at the end of the parameter draws, by the lanes that wait while lane 0 updates alpha
//     (no separate pass and barrier per sweep).

// Extra shared memory behind full_layout: rowbits [U][W] and rowid [N] as uint8 (U <= 256) or uint16.
__host__ __device__ inline size_t sweep_extra_bytes(const FullParams &p) {
    return ((size_t)p.U * p.W * 4 + (size_t)p.N * (p.U <= 256 ? 1 : 2) + 15) & ~(size_t)15;
}

// Gamma(sa, 1), or Beta(sa, sb) = x / (x + y) from two Gammas of one stream (Stream::beta's rule), drawn by one
// copy of the rejection sampler.
__device__ __forceinline__ double param_draw(unsigned long long seed, uint32_t chain, uint32_t sweep, uint32_t sid,
                                             uint32_t idx, double sa, double sb, bool is_beta) {
    Stream st(seed, chain, sweep, sid, idx);
    double x = 0.0, shape = sa;
#pragma unroll 1
    for (int h = 0;; ++h) {
        const double g = st.gamma(shape);
        if (h == 0) {
            if (!is_beta) return g;
            x = g; shape = sb;
            continue;
        }
        const double sum = x + g;
        return sum > 0.0 ? x / sum : 0.5;
    }
}

// REL: 0 no relabelling, 1 the reference's online step, 2 BMM_FLAG_STEPHENS_FIXED.  ALPHA: alpha is sampled (alpha0 == 0).
template <bool STICK, int REL, bool ALPHA>
__device__ __forceinline__ void chain_sweep_body(const FullParams &p) {
    extern __shared__ __align__(16) char smem_raw[];
    FullSmem s;
    uint32_t *rowbits = (uint32_t *)(smem_raw + full_layout(p, smem_raw, &s));
    const int c = blockIdx.x, tid = threadIdx.x, nthr = blockDim.x;
    const int K = p.K, P = p.P, U = p.U, N = p.N, W = p.W, KP = K * P, ns = p.nsamples;
    const int S = hist_count(ns, p.burnin, p.thin);
    const size_t UK = (size_t)U * K;
    const uint32_t chain = (uint32_t)(p.chain_offset + c);
    const bool id8 = U <= 256;
    uint8_t *rid8 = (uint8_t *)(rowbits + (size_t)U * W);
    uint16_t *rid16 = (uint16_t *)rid8;
    double *prob = s.prob;
    int *hist = s.hist;
    char *aws = p.assign_ws + (size_t)c * assign_ws_bytes(K);
    PHASE_INIT();

    for (int t = tid; t < KP; t += nthr) s.theta[t] = p.theta_cur[(size_t)c * KP + t];
    for (int t = tid; t < K; t += nthr) { s.pi[t] = p.pi_cur[(size_t)c * K + t]; s.perm[t] = t; }
    if (tid == 0) s.scal[0] = p.alpha_cur[c];
    if (REL)
        for (size_t e = tid; e < UK; e += nthr) { s.Q[e] = p.Q[(size_t)c * UK + e]; s.logQ[e] = p.logQ[(size_t)c * UK + e]; }
    for (int e = tid; e < U * W; e += nthr) rowbits[e] = p.rowbits[e];
    for (int i = tid; i < N; i += nthr) {
        if (id8) rid8[i] = (uint8_t)p.rowid[i];
        else rid16[i] = (uint16_t)p.rowid[i];
    }
    __syncthreads();
    if (p.j_begin == 1 && p.burnin == 0) {  // iteration 0 of the returned histories = initial state
        for (int t = tid; t < KP; t += nthr) p.theta_out[(size_t)c * KP * S + t] = s.theta[t];
        for (int t = tid; t < K; t += nthr) p.pi_out[(size_t)c * S * K + (size_t)S * t] = s.pi[t];
        if (tid == 0) p.alpha_out[(size_t)c * S] = s.scal[0];
    }
    // A: log tables of the starting state; from here on the lanes that draw theta and pi keep them current
    for (int t = tid; t < KP; t += nthr) { const double th = s.theta[t]; s.w1[t] = log(th); s.w0[t] = log(1 - th); }
    for (int t = tid; t < K; t += nthr) s.lpi[t] = log(s.pi[t]);
    __syncthreads();

    for (int j = p.j_begin; j < p.j_end; ++j) {
        PHASE_BEGIN();
        // ---- B: row table prob[u, k] = exp(log pi_k + loglh_k(u)) / sum
        for (int u = tid; u < U; u += nthr) {
            const uint32_t *xb = rowbits + (size_t)u * W;
            double cum = 0.0, mx = 0.0;
            if (p.flags & 1u) {  // BMM_FLAG_STABLE_SOFTMAX
                mx = -INFINITY;
                for (int k = 0; k < K; ++k) {
                    double ll = 0.0;
                    for (int d = 0; d < P; ++d) ll += ((xb[d >> 5] >> (d & 31)) & 1u) ? s.w1[k + K * d] : s.w0[k + K * d];
                    mx = fmax(mx, s.lpi[k] + ll);
                }
            }
            for (int k = 0; k < K; ++k) {
                double ll = 0.0;
                for (int d = 0; d < P; ++d) ll += ((xb[d >> 5] >> (d & 31)) & 1u) ? s.w1[k + K * d] : s.w0[k + K * d];
                double sk = exp(s.lpi[k] + ll - mx);
                prob[u + (size_t)U * k] = sk;
                cum += sk;
            }
            if (!(cum > 0.0) || !isfinite(cum)) p.status[c] = -9;  // BMM_ERR_PROB
            for (int k = 0; k < K; ++k) {
                prob[u + (size_t)U * k] /= cum;
                hist[u + (size_t)U * k] = 0;
            }
        }
        __syncthreads();
        PHASE_END(PH_B);
        // ---- C: allocation draws
        {
            uint8_t *zrow = p.zhist + ((size_t)c * ns + j) * N;
            const uint2 key = make_uint2((uint32_t)p.seed, chain);
            const uint32_t sid = ST_Z ^ ((uint32_t)(p.seed >> 32) << 8);
            const bool word_store = (N & 3) == 0;
            for (int i4 = tid; 4 * i4 < N; i4 += nthr) {
                const uint4 rnd = philox4x32_10(make_uint4((uint32_t)i4, 0u, sid, (uint32_t)j), key);
                uint32_t zw = 0;
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                    const int i = 4 * i4 + h;
                    if (i >= N) break;
                    const double uu = u32_unit(philox_word(rnd, h));
                    const int r = id8 ? rid8[i] : rid16[i];
                    const int z = categorical_icdf(K, [&](int k) { return prob[r + (size_t)U * k]; }, uu);
                    if (word_store) zw |= (uint32_t)(z + 1) << (8 * h);
                    else zrow[i] = (uint8_t)(z + 1);
                    atomicAdd(&hist[r + (size_t)U * z], 1);
                }
                if (word_store) *(uint32_t *)(zrow + 4 * i4) = zw;
            }
        }
        __syncthreads();
        PHASE_END(PH_C);
        // ---- D: fold the (row, label) histogram into c_k and V_kd
        for (int t = tid; t < KP + K; t += nthr) {
            int acc = 0;
            if (t < KP) {
                const int k = t % K, d = t / K;
                for (int u = 0; u < U; ++u)
                    if ((rowbits[(size_t)u * W + (d >> 5)] >> (d & 31)) & 1u) acc += hist[u + (size_t)U * k];
                s.Vkd[t] = acc;
            } else {
                const int k = t - KP;
                for (int u = 0; u < U; ++u) acc += hist[u + (size_t)U * k];
                s.ck[k] = acc;
            }
        }
        __syncthreads();
        PHASE_END(PH_D);
        // ---- E: Stephens relabelling   F: parameter draws (see full_chain_body)
        const double alpha_prev = s.scal[0];
        auto phase_e = [&](const int tid, const int nthr, auto sync) {
            if (REL && j >= p.burnin)
                stephens_online_group(U, K, p.wt, s.Q, s.logQ, prob, j, p.cost_g ? p.cost_g + (size_t)c * K * K : s.cost, s.perm,
                                      aws, REL == 2, tid, nthr, sync);
        };
        auto phase_f = [&](const int tid, const int nthr, auto sync) {
            const int nalpha = ALPHA ? (STICK ? 2 : 4) : 0;
            for (int t = tid; t < K + KP + nalpha; t += nthr) {
                uint32_t sid, idx;
                double sa, sb = 0.0;
                bool is_beta = false;
                double *dst;
                if (t < K) {
                    idx = (uint32_t)t; dst = &s.gsc[t];
                    if (!STICK) {
                        sid = ST_PI; sa = alpha_prev / K + s.ck[t];
                    } else {
                        int later = 0;
                        for (int l = t + 1; l < K; ++l) later += s.ck[l];
                        sid = ST_STICK; sa = 1.0 + s.ck[t]; sb = alpha_prev + later; is_beta = true;
                    }
                } else if (t < K + KP) {
                    const int e = t - K, k = e % K, d = e / K;
                    sid = ST_THETA; idx = (uint32_t)(k * P + d); dst = &s.theta[e];
                    sa = p.beta + s.Vkd[e]; sb = p.gamma + s.ck[k] - s.Vkd[e]; is_beta = true;
                } else {
                    const int q = t - K - KP;
                    sid = ST_ALPHA; idx = (uint32_t)q; dst = &s.scal[4 + q];
                    sa = alpha_gamma_shape(q, alpha_prev, p.a, N, K);
                }
                const double val = param_draw(p.seed, chain, (uint32_t)j, sid, idx, sa, sb, is_beta);
                *dst = val;
            }
            sync();
            // log tables for sweep j + 1 (phase A of full_chain_body): lane t < K normalises pi_t, lane K + e takes
            // theta_e, both beside lane 0's alpha update
            auto log_theta = [&](const int e) { const double th = s.theta[e]; s.w1[e] = log(th); s.w0[e] = log(1 - th); };
            if (!STICK) {
                for (int t = tid; t < K + KP; t += nthr) {
                    if (t >= K) { log_theta(t - K); continue; }
                    double sum = 0.0;
                    for (int k = 0; k < K; ++k) sum += s.gsc[k];
                    s.pi[t] = s.gsc[t] / sum;
                    s.lpi[t] = log(s.pi[t]);
                }
                if (tid == 0 && ALPHA) s.scal[0] = alpha_combine(s.scal + 4, p.a, p.b, N, K);
            } else {
                if (tid == 0) {
                    s.gsc[K - 1] = 1.0;
                    int K_viable = 0;
                    s.pi[0] = s.gsc[0];
                    if (s.pi[0] > 0.01) K_viable++;
                    double cumprod = 1 - s.gsc[0];
                    for (int k = 1; k < K; ++k) {
                        s.pi[k] = cumprod * s.gsc[k];
                        if (s.pi[k] > 0.01) K_viable++;
                        cumprod *= (1 - s.gsc[k]);
                    }
                    s.scal[1] = (double)K_viable;
                }
                sync();
                for (int t = tid; t < K + KP; t += nthr) {
                    if (t >= K) log_theta(t - K);
                    else s.lpi[t] = log(s.pi[t]);
                }
                if (ALPHA) {
                    const int K_viable = (int)s.scal[1];
                    for (int q = 2 + tid; q < 4; q += nthr)
                        s.scal[4 + q] = param_draw(p.seed, chain, (uint32_t)j, ST_ALPHA, (uint32_t)q,
                                                   alpha_gamma_shape(q, alpha_prev, p.a, N, K_viable), 0.0, false);
                    sync();
                    if (tid == 0) s.scal[0] = alpha_combine(s.scal + 4, p.a, p.b, N, K_viable);
                }
            }
        };
        if (REL && j < p.burnin && j >= p.burnin - p.burnrelabel) {
            double *dst = p.cube + ((size_t)c * p.burnrelabel + (j - p.burnin + p.burnrelabel)) * UK;
            for (size_t e = tid; e < UK; e += nthr) dst[e] = prob[e];
        }
        if (nthr >= 64) {
            const int w = tid >> 5, lane = tid & 31;
            if (w == 0) phase_f(lane, 32, [] { __syncwarp(); });
            else if (w == 1) phase_e(lane, 32, [] { __syncwarp(); });
            PHASE_END(w == 1 ? PH_E : PH_F);
        } else {
            phase_e(tid, nthr, [] { __syncthreads(); });
            PHASE_END(PH_E);
            phase_f(tid, nthr, [] { __syncthreads(); });
            PHASE_END(PH_F);
        }
        __syncthreads();
        PHASE_END(PH_WAIT_EF);
        const int sidx = hist_slot(j, p.burnin, p.thin);
        if (sidx >= 0) {
            for (int t = tid; t < KP; t += nthr) {
                p.theta_out[(size_t)c * KP * S + (size_t)KP * sidx + t] = s.theta[t];
                if (REL) {
                    const int k = t % K, d = t / K;
                    p.theta_rel_out[(size_t)c * KP * S + (size_t)KP * sidx + s.perm[k] + K * d] = s.theta[t];
                }
            }
            for (int t = tid; t < K; t += nthr) {
                p.pi_out[(size_t)c * S * K + sidx + (size_t)S * t] = s.pi[t];
                if (REL) p.perm_out[(size_t)c * S * K + sidx + (size_t)S * t] = s.perm[t];
            }
            if (tid == 0) p.alpha_out[(size_t)c * S + sidx] = s.scal[0];
        }
        __syncthreads();
        PHASE_END(PH_HIST);
        PHASE_SWEEP();
    }
    for (int t = tid; t < KP; t += nthr) p.theta_cur[(size_t)c * KP + t] = s.theta[t];
    for (int t = tid; t < K; t += nthr) p.pi_cur[(size_t)c * K + t] = s.pi[t];
    if (tid == 0) p.alpha_cur[c] = s.scal[0];
    if (REL)
        for (size_t e = tid; e < UK; e += nthr) { p.Q[(size_t)c * UK + e] = s.Q[e]; p.logQ[(size_t)c * UK + e] = s.logQ[e]; }
    PHASE_FLUSH();
}

// One entry point for 32, 64 and 128 threads: at most 128 registers, so that eight 64-thread blocks fit an SM.
template <bool STICK, int REL, bool ALPHA>
__global__ void __launch_bounds__(128, 4) chain_sweep_kernel(const FullParams p) { chain_sweep_body<STICK, REL, ALPHA>(p); }

template <bool STICK, int REL, bool ALPHA>
cudaError_t launch_sweep_t(const FullParams &p, int n_chains, int threads, cudaStream_t st) {
    static FuncAttrCache attr;
    const size_t smem = full_layout(p, nullptr, nullptr) + sweep_extra_bytes(p);
    cudaError_t e = attr.ensure_smem(chain_sweep_kernel<STICK, REL, ALPHA>, (int)smem);
    if (e != cudaSuccess) return e;
    chain_sweep_kernel<STICK, REL, ALPHA><<<n_chains, threads, smem, st>>>(p);
    g_launches++;
    return cudaGetLastError();
}

template <bool STICK, int REL>
cudaError_t launch_sweep_a(const FullParams &p, int n_chains, int threads, cudaStream_t st) {
    return p.alpha0 == 0.0 ? launch_sweep_t<STICK, REL, true>(p, n_chains, threads, st)
                           : launch_sweep_t<STICK, REL, false>(p, n_chains, threads, st);
}

template <bool STICK>
cudaError_t launch_sweep_r(const FullParams &p, int n_chains, int threads, cudaStream_t st) {
    if (!p.relabel) return launch_sweep_a<STICK, 0>(p, n_chains, threads, st);
    return (p.flags & 64u) ? launch_sweep_a<STICK, 2>(p, n_chains, threads, st) : launch_sweep_a<STICK, 1>(p, n_chains, threads, st);
}

}  // namespace

size_t full_smem_bytes(const FullParams &p, int) { return full_layout(p, nullptr, nullptr); }

cudaError_t launch_full(const FullParams &p, int n_chains, int threads, cudaStream_t st) {
    size_t smem = full_smem_bytes(p, threads);
    auto kern = threads == 64 ? full_chain_kernel_64 : full_chain_kernel;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<n_chains, threads, smem, st>>>(p);
    g_launches++;
    return cudaGetLastError();
}

bool full_rows_fit_smem(int U, int K) { return (size_t)U * K <= FULL_SMEM_ROWS_MAX; }

// The observation -> row map is kept in shared memory only up to 16 KiB (N = 16384 observations with byte ids), so that
// the seven or eight chains an SM holds at C2's shape are not limited by shared memory; larger N run the generic kernel.
bool chain_sweep_supported(const FullParams &p, int threads) {
    return p.ru == nullptr && p.use_hist && !p.probs_out && !p.loglik_out && p.U <= 65536 &&
           (threads == 32 || threads == 64 || threads == 128) && sweep_extra_bytes(p) <= 16384;
}

cudaError_t launch_chain_sweep(const FullParams &p, int n_chains, int threads, cudaStream_t st) {
    return p.stickbreaking ? launch_sweep_r<true>(p, n_chains, threads, st) : launch_sweep_r<false>(p, n_chains, threads, st);
}

cudaError_t chain_phase_read(unsigned long long *out, size_t n, bool *supported) {
#ifdef BMM_CHAIN_PHASE_CLOCKS
    *supported = true;
    const size_t cap = (size_t)CHAIN_PHASE_MAX_CHAINS * 4 * CHAIN_PHASES;
    cudaError_t e = cudaMemcpyFromSymbol(out, g_chain_phase, (n < cap ? n : cap) * sizeof(unsigned long long));
    if (e != cudaSuccess) return e;
    static const unsigned long long zeros[CHAIN_PHASE_MAX_CHAINS * 4 * CHAIN_PHASES] = {};
    return cudaMemcpyToSymbol(g_chain_phase, zeros, sizeof(zeros));
#else
    (void)out; (void)n;
    *supported = false;
    return cudaSuccess;
#endif
}

}  // namespace bmm
