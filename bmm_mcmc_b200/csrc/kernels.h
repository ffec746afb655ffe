// Host-visible parameter blocks and launchers of the sampler kernels.
#pragma once
#include <cmath>
#include <cstdint>
#include <cuda_runtime.h>

namespace bmm {

// Counter of kernel launches made by this library (bmm_launch_count()).
extern unsigned long long g_launches;

// History thinning (f2): the returned histories keep every thin-th post-burn-in sweep, j = burnin + t * thin
// (the reference keeps them all: full_gibbs.cpp:52-57,233-248).  hist_slot: index of sweep j in the kept histories
// or -1; hist_count: number of kept sweeps.
__host__ __device__ inline int hist_slot(int j, int burnin, int thin) {
    const int r = j - burnin;
    if (r < 0) return -1;
    if (thin <= 1) return r;
    return (r % thin) ? -1 : r / thin;
}
__host__ __device__ inline int hist_count(int nsamples, int burnin, int thin) {
    const int S = nsamples - burnin;
    return thin > 1 ? (S + thin - 1) / thin : S;
}

// cudaFuncSetAttribute is per device: remember, per kernel, the value already set on each device.
struct FuncAttrCache {
    int set[64] = {};
    template <typename F>
    cudaError_t ensure_smem(F *kernel, int bytes) {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        if (dev >= 0 && dev < 64 && set[dev] >= bytes) return cudaSuccess;
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e == cudaSuccess && dev >= 0 && dev < 64) set[dev] = bytes;
        return e;
    }
};

// ---- uncollapsed samplers, one chain per thread block (kern_full.cu) --------------------------
// Data rows are de-duplicated on the host: U unique bit-packed rows, multiplicities wt[U],
// rowid[N] maps each observation to its row.  Every per-row quantity (probabilities, Stephens Q)
// is shared by all observations with the same x.
struct FullParams {
    int N, P, K, U, W;            // W = 32-bit words per row
    int nsamples, burnin, relabel, burnrelabel, stickbreaking;
    int thin;                     // history thinning (hist_slot)
    int j_begin, j_end;           // sweeps [j_begin, j_end)
    double alpha0, beta, gamma, a, b;
    unsigned long long seed;
    int chain_offset;
    unsigned flags;
    int use_hist;                 // 1: (row,label) histogram path; 0: direct count atomics
    // data, shared by all chains
    const uint32_t *rowbits;      // [U][W]
    const int *rowid;             // [N]
    const int *wt;                // [U]
    // chain state in global memory (persists between launches)
    double *theta_cur;            // [c][K*P] cm
    double *pi_cur;               // [c][K]
    double *alpha_cur;            // [c]
    double *Q, *logQ;             // [c][U*K]
    double *cube;                 // [c][burnrelabel][U*K]
    double *prob_g;               // [c][U*K] (used when the row table does not fit shared memory)
    int *hist_g;                  // [c][U*K]
    double *ll_g;                 // [c][U*K] (loglik probe only)
    char *assign_ws;              // [c][assign_ws_bytes(K)]
    double *cost_g;               // [c][K*K] Stephens cost when K*K doubles do not fit shared memory, else nullptr
    int *status;                  // [c]
    // histories
    uint8_t *zhist;               // [c][nsamples][N], labels 1..K
    double *theta_out;            // [c][K*P*S]   original labelling
    double *theta_rel_out;        // [c][K*P*S]   relabelled
    double *pi_out;               // [c][S*K cm]
    double *alpha_out;            // [c][S]
    int *perm_out;                // [c][S*K cm]
    double *probs_out;            // [c][nsamples][N*K] or nullptr
    double *loglik_out;           // [c][nsamples][N*K] or nullptr
    // replay (nullptr = Philox)
    const double *ru; int ru_slots;
    const double *rpi, *rtheta, *ralpha;
};
// K x K cost matrices up to this many entries live in shared memory, larger ones in cost_g
constexpr int COST_SMEM_MAX = 64 * 64;
size_t full_smem_bytes(const FullParams &p, int threads);
cudaError_t launch_full(const FullParams &p, int n_chains, int threads, cudaStream_t st);
// chain_sweep_kernel: the same chain, bit for bit, specialised to Philox mode with the (row, label) histogram and no
// probes, which is what chain_sweep_supported checks; everything else runs full_chain_kernel
bool chain_sweep_supported(const FullParams &p, int threads);
cudaError_t launch_chain_sweep(const FullParams &p, int n_chains, int threads, cudaStream_t st);
// per-phase cycle totals [chain][warp < 4][9] of builds with -DBMM_CHAIN_PHASE_CLOCKS (read and cleared);
// *supported = false in the default build
cudaError_t chain_phase_read(unsigned long long *out, size_t n, bool *supported);

// ---- collapsed finite-K and DP samplers, one chain per warp-sized block (kern_collapsed.cu) ---
struct CollapsedParams {
    int N, P, K, W;               // K = maxK for dp
    int nsamples, burnin, relabel, burnrelabel, dp;
    int j_begin, j_end;
    int fp32;                     // BMM_FP32: single-precision weights in the product-form kernel
    int thin;                     // history thinning (hist_slot)
    double alpha0, beta, gamma, a, b;
    unsigned long long seed;
    int chain_offset;
    unsigned flags;
    const uint32_t *xbits;        // [N][W]
    // tables shared by all chains: log(beta+n), log(gamma+n), log(beta+gamma+n), n = 0..N
    const double *logB, *logG, *logBG;
    const double *logN;           // log(n), n = 0..N (dp: log N_k)
    const double *rBGP;           // dp, Philox mode: (beta + gamma + n)^-P, n = 0..N; nullptr when the products could leave the double range
    // chain state (global, persists between launches)
    uint8_t *z_cur;               // [c][N] labels 0..K-1 (0xFF = unseated, dp sweep 1)
    int *cnt;                     // [c][K*(P+1)]: S_kd at k*(P+1)+d, N_k at k*(P+1)+P
    double *alpha_cur;            // [c]
    int *dp_used;                 // [c][K+2]: used[0..K), then nused, Kvar
    uint8_t *dp_free;             // [c][K] multiplicity of each label in the free heap
    double *Q, *logQ;             // [c][N*K]
    double *probs_sample;         // [c][N*K]
    double *cube;                 // [c][burnrelabel][N*K]
    char *assign_ws;
    double *cost_g;               // [c][K*K] or nullptr (see FullParams)
    int *status;
    // histories
    uint8_t *zhist;               // [c][nsamples][N] labels 1..K
    double *theta_out, *theta_rel_out;   // [c][K*P*S]
    double *alpha_out;            // [c][S]
    int *perm_out;                // [c][S*K cm]
    double *probs_out;            // [c][nsamples][N*K] or nullptr
    int *kactive_out;             // [c][nsamples] or nullptr (dp)
    const double *ru; int ru_slots;
    const double *ralpha;
};
size_t collapsed_smem_bytes(const CollapsedParams &p);
cudaError_t launch_collapsed(const CollapsedParams &p, int n_chains, cudaStream_t st);

// ---- uncollapsed samplers, one chain over the whole GPU / N-sharded over GPUs (kern_big.cu) ----
struct BigParams {
    long long N_global, row_offset;   // this rank holds observations [row_offset, row_offset + N_local)
    int N_local, P, K, W;
    int nsamples, burnin, stickbreaking, precision;
    int thin;                         // history thinning (hist_slot)
    int tables_in_smem;               // K*P log tables + count histogram fit shared memory
    int keep_history;                 // zhist holds every sweep ([nsamples][N_local]) or only the current one
    double alpha0, beta, gamma, a, b;
    unsigned long long seed;
    int chain_offset;
    unsigned flags;
    const uint32_t *xbits;            // [N_local][W]
    double *w1, *w0, *lpi;            // log theta [K*P] (k + K*d), log(1-theta), log pi [K]
    double *theta_cur, *pi_cur, *alpha_cur, *gsc;
    int *counts;                      // 2 x (K + K*P): c_k then V_kd (k + K*d); sweep j uses buffer j & 1
    int *status;
    uint8_t *zhist;
    double *theta_out, *pi_out, *alpha_out;   // [K*P*S], [S*K cm], [S]
    double *probs_out, *loglik_out;   // [nsamples][N_local*K cm] or nullptr
    int *counts_out;                  // [nsamples][K + K*P] probe or nullptr
    float *probs_f32;                 // relabelling: this sweep's probabilities, row-major [N_local][K], or nullptr
    const int *perm_cur;              // relabelling: permutation of the current sweep [K] (device), or nullptr
    double *theta_rel_out;            // [K*P*S] relabelled theta history, or nullptr
    void *lp_table;                   // large-P tensor path: split weight table in operand-image order
    double *lp_bias;                  // [128] uncentred b_k
    int *cnt_ws;                      // scratch of launch_big_counts: 2*(K+1) + N_local ints
    const double *ru; int ru_slots;   // replay
    const double *rpi, *rtheta, *ralpha;
    // tensor path for K <= 32, P <= 112 (kern_big_ws.cu): operand image of the split weight table and
    // s0_k = sum_d log(1 - theta_kd), written by the update kernel so that the sweep's prologue is a copy
    unsigned char *ws_b1;             // [ws_b1_bytes(P)] or nullptr
    double *ws_s0;                    // [32]
    int *ws_rep;                      // [ws_rep_bytes(K, P)] replicas of the count vector (zero between launches)
    // Counts handed from the sweep kernel to the update kernel through an inbox of tagged words: over peer memory on
    // an N-sharded run (dist.cu), through a local inbox (x_world = 1) on one GPU -- the tags make the hand-over
    // self-synchronising, so the update kernel can be launched before the sweep kernel has drained.
    // x_world = 0: the counts in `counts` are complete when the update kernel starts (other sweep kernels, NCCL)
    int x_world, x_rank;
    int x_fused;                      // the sweep kernel's last CTA pushes the counts itself
    unsigned long long x_cap;         // ints per inbox slot
    int2 *const *x_peer;              // [x_world] every rank's inbox block as mapped here
    const int2 *x_local;              // this rank's inbox block
    const int *x_seq;                 // x_seq[0] + j = exchange number of sweep j
    unsigned *x_done;                 // CTA ticket counter of the fused push (zero between launches)
};
// Inbox of the count exchange: [2 parities][world][cap] words of (count, exchange number).  Every word carries
// its own validity tag and is written with one 8-byte store, so neither side needs a fence or a separate flag
// (the "LL" idea of NCCL's low-latency protocol): the consumer re-reads a word until its tag is the number it
// waits for.
__host__ __device__ inline size_t x_slot_off(int s, int world, int rank, size_t cap) { return ((size_t)(s & 1) * world + rank) * cap; }
__device__ __forceinline__ void x_store(int2 *dst, int value, int s) {     // one 64-bit scalar store: single-copy atomic
    const unsigned long long w = (unsigned long long)(unsigned)value | ((unsigned long long)(unsigned)s << 32);
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" :: "l"(dst), "l"(w) : "memory");
}
__device__ __forceinline__ int2 x_load(const int2 *src) {
    unsigned long long w;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(w) : "l"(src) : "memory");
    return make_int2((int)(unsigned)w, (int)(unsigned)(w >> 32));
}
// Programmatic dependent launch: a kernel launched with launch_pdl may start while its predecessor in the stream is
// still running; it must call griddep_wait() before touching anything the predecessor writes (the call returns once
// the predecessor has completed and its writes are visible).  griddep_launch() lets the successor start early.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool pdl_enabled();
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
cudaError_t launch_x_begin_run(int *seq, int n_sweeps, cudaStream_t st);   // seq[0] = seq[1]; seq[1] += n_sweeps

// Single-pass online relabelling of the tensor path (kern_big_ws_relabel.cu): pass j recomputes p_j and p_{j-1} from the
// packed rows, applies the pending Q update, and accumulates G(k,l) = sum_i log q_ik p_il into cost_out.
struct WsRelabelParams {
    long long N_local;
    int P, K, W;
    const uint32_t *xbits;            // [N_local][W]
    const unsigned char *b1_cur;      // operand image of this sweep's table (BigParams::ws_b1)
    const double *lpi, *s0;           // this sweep's log pi and s0 (BigParams::lpi, ws_s0)
    unsigned char *b1_hist;           // [2][ws_b1_bytes(P)] images of past sweeps (kept by CTA 0)
    float *bias_hist;                 // [2][32] their biases
    int hist_prev, hist_next;         // which copy holds the pending update's table; which one receives this sweep's (-1: none)
    const int *perm;                  // [K] column order of the pending update: perm_{j-1} (its inverse in the fixed mode)
    int upd, do_cost;                 // apply the pending update; accumulate the cost matrix
    float cq, cp;                     // Q' = cq * Q + cp * p[:, perm]
    int q_in_rowmajor, q_out_rowmajor;
    int q_direct;                     // diagnostic: read the Q tiles straight from global memory instead of through the bulk-copy ring
    float *Q_rm;                      // row-major [N_local][K] (batch step's output / final result)
    float *Q_tiled;                   // [tiles of 128 rows][8][128][4 floats]
    double *cost_out;                 // [K*K] G at k + K*l (+= ; the s_l block behind it stays zero)
    int *status;
};
size_t wsr_q_tiled_bytes(long long N);
cudaError_t launch_big_relabel_ws(const WsRelabelParams &p, int sm_count, cudaStream_t st);
size_t ws_b1_bytes(int P);
size_t ws_rep_bytes(int K, int P);
cudaError_t ws_trace_read(unsigned long long out[16]);   // phase stamps of the last two tensor-sweep launches (diagnostic)
cudaError_t ws_cta_read(unsigned long long out[320]);
cudaError_t upd_trace_read(unsigned long long out[16]);  // ... and of the last two update launches
cudaError_t launch_ws_table(const BigParams &p, cudaStream_t st);   // operand image from w1 / w0 (initial state)
bool big_tables_fit_smem(int K, int P, int precision);
int big_replay_max_k();
cudaError_t launch_big_init(const BigParams &p, cudaStream_t st);
cudaError_t launch_big_replay_load(const BigParams &p, int j, cudaStream_t st);
cudaError_t launch_big_sweep(const BigParams &p, int j, int sm_count, cudaStream_t st);
cudaError_t launch_big_params(const BigParams &p, int j, cudaStream_t st);
// tcgen05 sweep for K <= 32, P <= 112 (kern_big_ws.cu): log-likelihood and sufficient statistics as tensor-core
// contractions, warp-specialised (producer / MMA / epilogue warps over mbarrier rings)
bool big_tc_supported(const BigParams &p);
cudaError_t launch_big_sweep_ws(const BigParams &p, int j, int sm_count, cudaStream_t st);
// sufficient statistics from the bit-packed rows (kern_big_counts.cu): counting sort by cluster + bit-sliced
// per-variable counters; counts must be zero on entry, ws holds 2*(K+1) + N ints
cudaError_t launch_big_counts(long long N, int K, int P, int W, const uint32_t *xbits, const uint8_t *z, int *counts,
                              int *ws, int sm_count, cudaStream_t st);
// large-P / large-K tcgen05 path (kern_big_lp.cu): pipelined k-loop contraction + counts kernel
bool big_lp_supported(const BigParams &p);
size_t big_lp_table_bytes(int P);
cudaError_t launch_big_sweep_lp(const BigParams &p, int j, int sm_count, cudaStream_t st);

// ---- relabelling on the grid path (kern_big_relabel.cu); P, Q row-major float [N][K] ----------
// acc: K*K + K doubles; tc != 0 allows the tcgen05 kernel (kern_big_cost_tc.cu, 8 <= K <= 128, K % 8 == 0),
// which reports a pipeline timeout through *status
cudaError_t launch_grid_cost(long long N, int K, const float *P, const float *Q, int use_logp, double *acc,
                             int sm_count, cudaStream_t st, int tc = 0, int *status = nullptr);
bool grid_cost_tc_supported(long long N, int K);
cudaError_t launch_grid_cost_tc(long long N, int K, const float *P, const float *Q, int use_logp, double *acc, int *status,
                                int sm_count, cudaStream_t st);
// *changed (device, optional) is set to 1 when the stored permutation differs from the new one
cudaError_t launch_grid_assign(int K, double *acc, char *ws, int *perm_cur, int *perm_dst, int perm_stride, cudaStream_t st,
                               int *changed = nullptr);
cudaError_t launch_grid_qupdate(long long N, int K, float *Q, const float *P, const int *perm, int sample_num,
                                int sm_count, cudaStream_t st, int fixed = 0);
cudaError_t launch_grid_invert_perm(int n, int K, const int *perm, int *inv, cudaStream_t st);
cudaError_t launch_grid_clamp(long long n, float *p, int sm_count, cudaStream_t st);
cudaError_t launch_grid_qmean(long long N, int K, int M, const float *cube, const int *perm, float *Q, int sm_count,
                              cudaStream_t st);
cudaError_t launch_grid_identity_perm(int n, int K, int *perm, cudaStream_t st);
// relabelled theta history from the original one and the permutation history, all kept sweeps in one launch
cudaError_t launch_grid_theta_rel(int K, int P, int S, const double *theta, const int *perm, double *theta_rel, int sm_count, cudaStream_t st);
// posterior summary: zfreq[i + N*perm[z_i - 1]] += 1 over one sweep's allocations (perm may be nullptr)
cudaError_t launch_grid_zfreq(long long N, int K, const uint8_t *z, const int *perm, unsigned *zfreq, int sm_count, cudaStream_t st);

// ---- Stephens batch (kern_stephens.cu) -------------------------------------------------------
cudaError_t launch_stephens_batch(int n_chains, int U, int K, int M, const int *wt, double *cube, double *logp,
                                  double *Q, double *logQ, int *perm, double *cost, char *assign_ws,
                                  cudaStream_t st, int fixed = 0);
cudaError_t launch_stephens_online(int U, int K, double *Q, double *logQ, const double *p, int sample_num,
                                   double *cost, int *perm, char *assign_ws, cudaStream_t st, int fixed = 0);
cudaError_t launch_assign(int K, int batch, const double *cost, int *solution, char *ws, cudaStream_t st);
cudaError_t launch_rdirichlet(int K, const double *alpha_m, unsigned long long seed, double *out, cudaStream_t st);

// ---- posterior predictive distribution from the kept draws (kern_predict.cu) ------------------
// tab: scratch of S * K * (2 P + 1) doubles; member (optional, zeroed by the caller): M x K column-major
cudaError_t launch_predict(int M, int P, int W, int K, int S, const uint32_t *xbits, const double *theta, const double *pi,
                           double *tab, double *logpred, double *member, cudaStream_t st);
// tab[g][k][0..P) = log theta_kd, [P..2P) = log(1 - theta_kd), [2P] = log pi_k of S draws (theta K x P x S, pi S x K cm)
cudaError_t launch_predict_tables(int K, int P, int S, const double *theta, const double *pi, double *tab, cudaStream_t st);

// ---- WAIC and the log-likelihood trace (kern_predict.cu fp64, kern_waic_tc.cu tcgen05) ---------------------------------
// Mergeable partials of one row over a run of draws: n, mean, M2 (Welford) and max, sum (log-sum-exp of l).
constexpr int WAIC_STAT = 5;
__host__ __device__ inline void waic_stat_init(double (&a)[WAIC_STAT]) { a[0] = a[1] = a[2] = a[4] = 0.0; a[3] = -INFINITY; }
__host__ __device__ inline void waic_stat_merge(double (&a)[WAIC_STAT], const double *b) {
    if (b[0] == 0.0) return;
    if (a[0] == 0.0) { for (int e = 0; e < WAIC_STAT; ++e) a[e] = b[e]; return; }
    const double na = a[0], nb = b[0], n = na + nb, delta = b[1] - a[1];   // Chan, Golub & LeVeque (1979)
    a[1] += delta * (nb / n);
    a[2] += b[2] + delta * delta * (na * nb / n);
    a[0] = n;
    if (b[4] > 0.0) {
        if (b[3] > a[3]) { a[4] = a[4] * exp(a[3] - b[3]) + b[4]; a[3] = b[3]; }
        else a[4] += b[4] * exp(b[3] - a[3]);
    }
}
// one more draw's l
__host__ __device__ inline void waic_push(double (&st)[WAIC_STAT], double l) {
    st[0] += 1.0;
    const double delta = l - st[1];
    st[1] += delta / st[0];
    st[2] += delta * (l - st[1]);
    if (l > st[3]) { st[4] = st[4] * exp(st[3] - l) + 1.0; st[3] = l; }
    else if (l > -INFINITY) st[4] += exp(l - st[3]);
}
// slices per chain of the fp64 kernel for ntiles tiles of 32 distinct rows
int waic_fp64_slices(int ntiles, int C, int S);
// stat: [C Q][U][WAIC_STAT]; tpart: [C S][ceil(U / 32)]; tab from launch_predict_tables over the C S draws
cudaError_t launch_waic_fp64(int U, int P, int W, int K, int S, int C, int Q, const uint32_t *rowbits, const int *wt,
                             const double *tab, double *stat, double *tpart, cudaStream_t st);
// pooled pointwise lppd / p_waic [U]; cv scratch [2 C][U]; loglik [C S] = sum of the G trace partials of each draw
// (tpart [C S][G]); chain_tot [2 C] = per-chain lppd, then per-chain p_waic (multiplicity-weighted sums over rows)
cudaError_t launch_waic_merge(int U, int C, int S, int Q, const int *wt, const double *stat, long long G, const double *tpart,
                              double *lppd, double *pwaic, double *cv, double *loglik, double *chain_tot, cudaStream_t st);
// tcgen05 path, K <= 32 and P <= 112: img [C S][ws_nch(P) * WS_B1_ROW] operand images and bias [C S][32] (log2 units),
// built by launch_waic_tc_tables; stat [C][U][WAIC_STAT] (one slice per chain); tpart [C S][4 ceil(U / 128)]
bool waic_tc_supported(int K, int P);
size_t waic_tc_img_bytes(int P);
cudaError_t launch_waic_tc_tables(int K, int P, long long D, const double *theta, const double *pi, unsigned char *img,
                                  float *bias, cudaStream_t st);
cudaError_t launch_waic_tc(int U, int P, int W, int K, int S, int C, const uint32_t *rowbits, const int *wt,
                           const unsigned char *img, const float *bias, double *stat, double *tpart, int *status,
                           int sm_count, cudaStream_t st);

// ---- PSIS-LOO and the log-likelihood matrix (kern_predict.cu / kern_waic_tc.cu producers, kern_loo.cu) ----------------
// L [D][Uc]: l of the Uc distinct rows rowbits [Uc][W] under each of the D pooled draws.  fp64 from launch_predict_tables'
// tables over the D draws; tcgen05 (waic_tc_supported shapes) from launch_waic_tc_tables' images.
cudaError_t launch_loglik_fp64(int Uc, int P, int W, int K, long long D, const uint32_t *rowbits, const double *tab,
                               double *L, cudaStream_t st);
cudaError_t launch_loglik_tc(int Uc, int P, int W, long long D, const uint32_t *rowbits, const unsigned char *img,
                             const float *bias, double *L, int *status, int sm_count, cudaStream_t st);
// Rows whose Pareto tail has at most LOO_SHORT_MAX_M draws take one thread each, longer tails (up to LOO_MAX_TAIL draws,
// sorted in shared memory) a radix select over several CTAs.
constexpr int LOO_SHORT_MAX_M = 64;
constexpr int LOO_MAX_TAIL = 16384;
// radix-select state of one long row: selected key prefix, rank still to find, keys above the prefix, max / min key,
// tail draws gathered
struct LooSel {
    unsigned long long prefix, kmax, kmin;
    unsigned rank, gt, tcount, pad;
};
int loo_long_blocks(long long D);
// Outputs per chunk row (elpd, lpd, khat, neff, each [Uc]); Mrow [Uc] = tail length of each row (rows with
// Mrow > LOO_SHORT_MAX_M are skipped); max_m = the largest Mrow <= LOO_SHORT_MAX_M (sizes shared memory).
cudaError_t launch_loo_short(int Uc, long long D, int max_m, const double *L, const int *Mrow, double *elpd, double *lpd,
                             double *khat, double *neff, cudaStream_t st);
// nlong rows lrow [nlong] of the chunk with tail lengths lM (> LOO_SHORT_MAX_M, <= LOO_MAX_TAIL, max_m the largest) and
// tail storage tail + ltoff[r]; scratch sel [nlong], hist [nlong][256], part [nlong][loo_long_blocks(D)][4]
cudaError_t launch_loo_long(int Uc, long long D, int nlong, int max_m, const double *L, const int *lrow, const int *lM,
                            const long long *ltoff, LooSel *sel, unsigned *hist, double *tail, double *part, double *elpd,
                            double *lpd, double *khat, double *neff, cudaStream_t st);

// ---- history layout conversion (kern_finalize.cu) --------------------------------------------
// zhist [c][nsamples][N] uint8 -> R layout [c][S x N cm]; optional relabelling through perm_out.
// elem_bytes = 4 (int32) or 1 (uint8, BMM_FLAG_COMPACT_Z).
cudaError_t launch_finalize_z(int n_chains, int N, int nsamples, int burnin, int thin, int K, const uint8_t *zhist,
                              const int *perm_out, void *z_orig, void *z_rel, int elem_bytes, cudaStream_t st, int s_lo = 0, int s_hi = -1);
// posterior summary of the chain-parallel paths: zfreq[c][i + N*k] = number of kept sweeps whose (relabelled, when perm is
// given) allocation of observation i is k + 1; reads the raw history [c][nsamples][N]
cudaError_t launch_chain_zfreq(int n_chains, int N, int nsamples, int burnin, int thin, int K, const uint8_t *zhist, const int *perm,
                               unsigned *zfreq, cudaStream_t st);
// expand a per-row matrix [c][U*K] to per-observation [c][N*K]
cudaError_t launch_expand_rows(int n_chains, int N, int U, int K, const int *rowid, const double *src, double *dst,
                               cudaStream_t st);

}  // namespace bmm
