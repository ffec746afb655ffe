/* bmm_capi.h -- C ABI of the B200-native allocation-sampling path of bmm-mcmc.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  Each entry point replaces one `.Call`
 * symbol that the reference registers in /root/reference/src/RcppExports.cpp:137-146; an Rcpp host
 * (r-package/src/host.cpp, see INTEGRATION.md) allocates the R objects, passes their raw pointers
 * here, and turns a non-zero return into Rcpp::stop(bmm_last_error()).
 *
 * Conventions
 *   - plain pointers and sizes only; all HOST pointers unless a name says `dev`;
 *   - every matrix/array uses R's column-major layout, exactly the shapes the reference returns
 *     (full_gibbs.cpp:233-248, stickbreaking.cpp:238-254, collapsed_gibbs.cpp:229-243,
 *     collapsed_gibbs_dp.cpp:285-299); with n_chains > 1 a slowest "chain" dimension is prepended;
 *   - S = nsamples - burnin rows/slices are returned (the reference's tail_rows/tail_slices);
 *   - labels are 1-based in z / z_original, 0-based in permutations, as in the reference;
 *   - return 0 on success, a negative BMM_ERR_* otherwise; bmm_last_error() gives the text;
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     BMM_ERR_CUDA.
 */
#ifndef BMM_CAPI_H
#define BMM_CAPI_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BMM_OK 0
#define BMM_ERR_INVALID (-1)         /* bad argument (shape, NULL, range)                          */
#define BMM_ERR_CUDA (-2)            /* CUDA runtime error / no device                             */
#define BMM_ERR_NOT_BINARY (-3)      /* X holds a value other than 0/1 (SURVEY App. D quirk 18)    */
#define BMM_ERR_BETA_GAMMA (-4)      /* gibbs_dp needs beta == gamma (collapsed_gibbs_dp.cpp:48)   */
#define BMM_ERR_NO_FREE_CLUSTER (-5) /* collapsed_gibbs_dp.cpp:166-168                             */
#define BMM_ERR_DP_STATE (-6)        /* reference state undefined after truncation fallback        */
#define BMM_ERR_NCCL (-7)
#define BMM_ERR_UNSUPPORTED (-8)     /* shape outside what the kernels cover                       */
#define BMM_ERR_PROB (-9)            /* non-finite conditional probabilities (reference: NA draw)  */
#define BMM_ERR_TIMEOUT (-10)        /* a device-side barrier never completed (kernel bug guard)   */

#define BMM_FP64 0
#define BMM_FP32 1

/* flags */
#define BMM_FLAG_STABLE_SOFTMAX 1u   /* subtract the row maximum before exp (NOT the reference:
                                        full_gibbs.cpp:106 underflows to NaN at large P)          */
#define BMM_FLAG_COMPACT_Z 2u        /* out->z / z_original are uint8 buffers (cast pointer), not
                                        int32: 1 B per allocation over PCIe; K must be <= 255     */
#define BMM_FLAG_NO_Z_HISTORY 4u     /* keep only the current allocations on the device; out->z is
                                        not written (large-N runs: S x N would not fit anywhere)   */
#define BMM_FLAG_X_PACKED 16u         /* args->X points at bit-packed rows instead of an IntegerMatrix:
                                        uint32 [N][ceil(P/32)], bit d%32 of word d/32 = x_id (grid
                                        path only; 8 B per row at P = 64 instead of 256 B)         */
#define BMM_FLAG_NO_TENSOR 32u        /* grid path, BMM_FP32: use the CUDA-core float kernel instead of
                                        the tcgen05 contraction (A/B testing); bmm_waic, bmm_loo,
                                        bmm_loglik_matrix: the fp64 kernel                         */
#define BMM_FLAG_STEPHENS_FIXED 64u   /* correctness-fixed relabelling (NOT the reference, SURVEY 8f-3): the batch
                                      * initialisation and the online Q update re-order columns with the
                                      * inverse of index_max(solution.col(.)) -- what the no-op
                                      * `perm <- sort_index(perm)` (stephens.cpp:56,85) was meant to do --,
                                      * the online cost uses log p like the batch cost (:79), and
                                      * Q' = (j Q + p_reordered) / (j + 1) is a running mean (:92).  The
                                      * batch loop's real threshold (1e-6, :24) needs no switch: it stops
                                      * at the same fixed point the 100 iterations reach.                  */
#define BMM_FLAG_GRID_PATH 8u        /* force the one-chain-over-the-whole-GPU kernels (default:
                                        chosen when n_chains <= 1 and N >= 32768, or when K*P is
                                        too large for the chain-per-block kernel)                  */

/* Replay mode: the z draws consume these uniforms instead of Philox, and the parameter draws
 * (pi, theta, alpha) are taken from the recorded histories, so allocations and counts can be
 * compared bit-exactly with a recorded reference/oracle run (BASELINE.json north_star). */
typedef struct bmm_replay {
    const double *u;     /* [chain][nsamples][N][u_slots]: uniforms in consumption order, <0 = none */
    int32_t u_slots;     /* K-1 for rmultinom samplers, 1 for gibbs_dp                             */
    const double *pi;    /* [chain][nsamples x K cm]   (full / stick-breaking)                     */
    const double *theta; /* [chain][K x P x nsamples]  (full / stick-breaking)                     */
    const double *alpha; /* [chain][nsamples]                                                      */
} bmm_replay;

/* Arguments shared by the four samplers.  Field order follows the reference's C++ signatures
 * (full_gibbs.cpp:32-45, stickbreaking.cpp:10-23, collapsed_gibbs.cpp:24-36,
 * collapsed_gibbs_dp.cpp:27-38).  Zero-initialise the extension block for reference behaviour. */
typedef struct bmm_args {
    const int32_t *X;    /* df: N x P IntegerMatrix, column-major, values 0/1                      */
    int32_t N, P;
    int32_t nsamples;
    int32_t K;           /* K (full, collapsed) or maxK (stick-breaking, dp)                       */
    double alpha;        /* 0 = sample alpha ~ Gamma(a,b), starting at 1 (R/utils.R:27,43,71,101)  */
    double beta, gamma, a, b;
    int32_t burnin;
    int32_t relabel;
    int32_t burnrelabel;
    int32_t debug;       /* accepted and ignored (the reference only prints)                       */
    /* ---- extensions ---- */
    int32_t n_chains;    /* 0/1 = a single chain                                                   */
    int32_t chain_offset;/* global index of this call's first chain (chain-split across GPUs)      */
    uint64_t seed;       /* Philox key; chain c draws from (seed, chain_offset + c)                */
    int32_t precision;   /* BMM_FP64 (default) or BMM_FP32 for the probability arithmetic          */
    int32_t device;      /* CUDA device ordinal                                                    */
    uint32_t flags;      /* BMM_FLAG_*                                                             */
    const bmm_replay *replay; /* NULL = Philox                                                     */
    /* N-sharded single chain (full / stick-breaking, n_chains <= 1): X holds this rank's rows
     * [row_offset, row_offset + N) of an n_global-row data set; counts are all-reduced over the
     * ranks of bmm_dist_init each sweep.  0 = not sharded (n_global = N).                         */
    int64_t n_global;
    int64_t row_offset;
    /* History thinning: keep every thin-th post-burn-in sweep (j = burnin + t * thin) in ALL returned histories
     * (pi, alpha, permutations, z, theta, ...), i.e. S = ceil((nsamples - burnin) / thin) everywhere below.
     * 0 / 1 = keep every sweep, the reference's behaviour (full_gibbs.cpp:52-57,233-248).  The sampler and the
     * online relabelling still run every sweep; only the storage is thinned.                              */
    int32_t thin;
    int32_t reserved_;
} bmm_args;

/* Initial state, drawn by the R wrappers before entering C++ (R/utils.R:42,68-74,98-103). */
typedef struct bmm_init {
    const double *pi;     /* initialPi    [chain][K]          full / stick-breaking                */
    const double *theta;  /* initialTheta [chain][K x P cm]   full / stick-breaking                */
    const int32_t *z;     /* initialK     [chain][N], 1-based collapsed                            */
} bmm_init;

/* Caller-allocated outputs.  Any pointer may be NULL to skip that output. */
typedef struct bmm_out {
    double *pi;              /* [chain][S x K cm]      full / stick-breaking                       */
    double *alpha;           /* [chain][S]                                                         */
    int32_t *permutations;   /* [chain][S x K cm]      written only when relabel (the reference
                                returns uninitialised memory otherwise, full_gibbs.cpp:65,237)     */
    int32_t *z;              /* [chain][S x N cm]      relabelled if relabel, else original        */
    double *theta;           /* [chain][K x P x S]     relabelled if relabel, else original        */
    int32_t *z_original;     /* [chain][S x N cm]      relabel only                                */
    double *theta_original;  /* [chain][K x P x S]     relabel only                                */
    /* probes (parity tests) */
    double *probs;           /* [chain][nsamples][N x K cm] conditional probabilities, every sweep */
    double *loglik;          /* [chain][nsamples][N x K cm] Bernoulli log-likelihood (full / SB)   */
    double *Q_final;         /* [chain][N x K cm] running Stephens Q after the last sweep          */
    int32_t *status;         /* [chain] 0 or a BMM_ERR_* raised inside that chain                  */
    int32_t *counts;         /* grid path probe: [nsamples][K + K*P] sufficient statistics of every
                                sweep, c_k then V_kd (k + K*d) (full_gibbs.cpp:182-200)             */
    /* grid path posterior summaries (SURVEY 8f-2): what a large-N caller needs instead of the S x N
     * history, which BMM_FLAG_NO_Z_HISTORY suppresses.                                             */
    uint32_t *z_freq;        /* [N x K cm] number of post-burn-in sweeps observation i spent in label k
                                (relabelled labels when relabel)                                    */
    int32_t *z_last;         /* [N] allocations of the last sweep, 1-based, original labels          */
} bmm_out;

/* ---- samplers: replace the four sampler .Call symbols ---------------------------------------- */
/* _bmmmcmc_gibbs_cpp                 (RcppExports.cpp:67-88;  full_gibbs.cpp:32)                   */
int bmm_gibbs_full(const bmm_args *args, const bmm_init *init, bmm_out *out);
/* _bmmmcmc_gibbs_stickbreaking_cpp   (RcppExports.cpp:114-135; stickbreaking.cpp:10)               */
int bmm_gibbs_stickbreaking(const bmm_args *args, const bmm_init *init, bmm_out *out);
/* _bmmmcmc_collapsed_gibbs_cpp       (RcppExports.cpp:11-31;  collapsed_gibbs.cpp:24)              */
int bmm_gibbs_collapsed(const bmm_args *args, const bmm_init *init, bmm_out *out);
/* _bmmmcmc_collapsed_gibbs_dp_cpp    (RcppExports.cpp:34-53;  collapsed_gibbs_dp.cpp:27)           */
int bmm_gibbs_dp(const bmm_args *args, bmm_out *out);

/* ---- helpers: replace the three helper .Call symbols ----------------------------------------- */
/* _bmmmcmc_my_stephens_batch (stephens.cpp:6-64): p is an N x K x M cube, q is N x K.             */
int bmm_stephens_batch(int32_t N, int32_t K, int32_t M, const double *p, double *q, int32_t *perm_MxK);
/* my_stephens_online (stephens.cpp:66-94): perm[K], q_new N x K, optional cost K x K.             */
int bmm_stephens_online(int32_t N, int32_t K, const double *q, const double *p, int32_t sample_num,
                        int32_t *perm, double *q_new, double *cost);
/* The same two helpers with a flags word: BMM_FLAG_STEPHENS_FIXED selects the corrected variant
 * (batch: perm_MxK then holds the inverse permutations, reference label -> sample column).          */
int bmm_stephens_batch_ex(int32_t N, int32_t K, int32_t M, const double *p, double *q, int32_t *perm_MxK, uint32_t flags);
int bmm_stephens_online_ex(int32_t N, int32_t K, const double *q, const double *p, int32_t sample_num,
                           int32_t *perm, double *q_new, double *cost, uint32_t flags);
/* _bmmmcmc_my_lpsolve (my_lpsolve.cpp:6-31): K x K cost (cm) -> K x K 0/1 solution (cm).
 * `batch` independent problems, consecutive in memory.                                            */
int bmm_assign(int32_t K, int32_t batch, const double *cost, int32_t *solution);
/* Same problem through the solver the grid path uses (warp-parallel Jonker-Volgenant for K > 5):
 * perm[c] = index_max(solution.col(c)) (stephens.cpp:82-84).                                      */
int bmm_assign_warp(int32_t K, const double *cost, int32_t *perm);
/* The K x K cost contraction of the grid path's relabelling (stephens.cpp:45-53,76-84) on host
 * matrices p, q (row-major float N x K): out[k + K*l] = sum_i log q_ik * p_il and
 * out[K*K + l] = sum_i p_il^2 (use_logp: p_il log p_il).  tensor != 0 forces the tcgen05 kernel
 * (8 <= K <= 128, K % 8 == 0), 0 the CUDA-core kernel.  Test entry point.                         */
int bmm_grid_cost(int64_t N, int32_t K, const float *p, const float *q, int32_t use_logp, int32_t tensor, double *out);
/* _bmmmcmc_rdirichlet_cpp (full_gibbs.cpp:10-27) with an explicit Philox seed.                    */
int bmm_rdirichlet(int32_t K, const double *alpha_m, uint64_t seed, double *out);
/* Posterior predictive distribution of a fitted model (no reference counterpart: /root/reference/TODO:6 lists it as
 * "Implement predictive distribution").  Xnew: M x P int32 column-major 0/1 rows; theta: K x P x S and pi: S x K
 * column-major, the kept draws as gibbs_full / gibbs_stickbreaking return them (full_gibbs.cpp:233-248).
 * log_pred[m] = log( 1/S sum_s sum_k pi_k^(s) prod_d theta_kd^(s)^x (1 - theta_kd^(s))^(1 - x) );
 * membership (optional, M x K column-major) = the responsibilities averaged over the draws.             */
int bmm_predictive(const int32_t *Xnew, int32_t M, int32_t P, int32_t K, int32_t S, const double *theta, const double *pi,
                   double *log_pred, double *membership);
/* WAIC (Watanabe 2010; as R's loo::waic) and the observed-data log-likelihood trace of a fitted gibbs_full /
 * gibbs_stickbreaking model (no reference counterpart).  X: N x P int32 column-major 0/1, or with BMM_FLAG_X_PACKED
 * uint32 [N][ceil(P/32)] bit-packed rows.  theta [C][K x P x S] and pi [C][S x K cm]: the kept draws of C chains as the
 * samplers return them.  With l[c,s,i] = log sum_k pi_k prod_d theta_kd^x_id (1 - theta_kd)^(1 - x_id) of draw (c, s):
 *   loglik [C x S]        sum_i l[c,s,i]
 *   lppd [N]              log 1/(C S) sum_{c,s} exp l[c,s,i]
 *   p_waic [N]            variance of l[.,.,i] over the C S draws, denominator C S - 1
 *   chain_lppd [C], chain_p_waic [C]   the totals over i of the same two figures from chain c's S draws alone
 * Any output may be NULL.  C S >= 2.  Computed on the device in a fixed order (two calls return the same bits): the fp64
 * kernel, or for K <= 32, P <= 112 and enough distinct rows a tcgen05 kernel (fp16 hi|lo operands, fp32 log-sum-exp over
 * k, fp64 moments); BMM_FLAG_NO_TENSOR forces the fp64 kernel.  theta exactly 0 or 1 gives l = -inf on the fp64 kernel,
 * and then p_waic = nan, as the float64 definition does.                                                          */
int bmm_waic(const void *X, int32_t N, int32_t P, int32_t K, int32_t S, int32_t C, const double *theta, const double *pi,
             uint32_t flags, int32_t device, double *loglik, double *lppd, double *p_waic, double *chain_lppd,
             double *chain_p_waic);
/* Device time in ms of the last bmm_waic's kernels on this thread, and 1 if it took the tcgen05 kernel.               */
int bmm_waic_kernel_ms(float *ms, int32_t *tensor);
/* PSIS-LOO (Vehtari, Gelman & Gabry 2017; as R's loo::loo, without mcse_elpd_loo) of a fitted gibbs_full /
 * gibbs_stickbreaking model (no reference counterpart).  X, theta, pi, flags and device as bmm_waic; r_eff: NULL (1) or
 * N relative efficiencies > 0, which set each observation's Pareto tail length M = min(ceil(0.2 D), ceil(3 sqrt(D / r_eff)))
 * (D = C S; M <= 16384, so D <= 29826161 at r_eff = 1).  With l[g, i] the log-likelihood of observation i under pooled
 * draw g and w~ the Pareto-smoothed, truncated, normalised log weights of r = -l:
 *   elpd_loo [N]   log sum_g exp(w~_g + l[g, i])
 *   lpd [N]        log 1/D sum_g exp l[g, i] (WAIC's lppd)
 *   pareto_k [N]   the tail's generalized Pareto shape (inf when M < 5 or the tail is flat)
 *   n_eff [N]      r_eff_i / sum_g exp(2 w~_g)
 * Any output may be NULL.  Computed on the device in a fixed order (two calls return the same bits).  theta exactly 0 or 1
 * can give l = -inf; then elpd_loo and n_eff are nan and pareto_k inf, as the float64 definition gives.              */
int bmm_loo(const void *X, int32_t N, int32_t P, int32_t K, int32_t S, int32_t C, const double *theta, const double *pi,
            const double *r_eff, uint32_t flags, int32_t device, double *elpd_loo, double *lpd, double *pareto_k,
            double *n_eff);
/* Device time in ms of the last bmm_loo's kernels on this thread, and 1 if its log-likelihood matrix came from the
 * tcgen05 kernel.                                                                                                       */
int bmm_loo_kernel_ms(float *ms, int32_t *tensor);
/* The log-likelihood matrix out [(C S) x N] column-major, out[g + C S i] = l[g, i] over the chain-major pooled draws
 * g = c S + s: the draws x observations matrix loo::loo() takes.  Inputs as bmm_waic.                                 */
int bmm_loglik_matrix(const void *X, int32_t N, int32_t P, int32_t K, int32_t S, int32_t C, const double *theta,
                      const double *pi, uint32_t flags, int32_t device, double *out);

/* Diagnostic (no reference counterpart): %globaltimer stamps in ns of the last two sweeps of the tensor grid path.
 * out[8 * (j & 1) + s], z-sweep kernel CTA 0: s = 0 entry, 1 pipeline start, 2 first tile drawn, 3 last tile drawn,
 * 4 counts flushed, 5 exit.  out[16 + 8 * (j & 1) + s], update kernel: s = 0 block 0 start, 1 block 0 has its counts,
 * 2 block 0 end, 3 last block start, 4 last block end.                                                               */
int bmm_debug_ws_trace(uint64_t out[32]);
/* ... and per CTA b of the last launch: out[2b] = (entry ns << 10) | SM id, out[2b + 1] = counts-flushed ns.      */
int bmm_debug_ws_cta(uint64_t out[320]);
/* Kernel of the last chain-per-block launch of gibbs_full / gibbs_stickbreaking: 0 none yet, 1 full_chain_kernel (the
 * generic one), 2 chain_sweep_kernel (Philox mode with the row histogram and no probes; BMM_CHAIN_KERNEL=generic
 * forces 1).                                                                                                         */
int bmm_debug_chain_kernel(void);
/* Per-phase cycle totals of the chain kernels, out[(chain * 4 + warp) * 9 + phase] for chains < 4096, phases A log
 * tables, B row table, C allocations, D histogram fold, E relabelling, F parameter draws, history write, the wait
 * after E / F, then the number of sweeps; the totals are cleared by the read.  Only builds with -DBMM_CHAIN_PHASE_CLOCKS (of kern_full.cu)
 * record them; the default build returns BMM_ERR_UNSUPPORTED.                                                         */
int bmm_debug_chain_phases(uint64_t *out, int64_t n);

/* ---- probes --------------------------------------------------------------------------------- */
/* One uncollapsed z-sweep at a given state (full_gibbs.cpp:87-133): log-likelihood and
 * conditional-probability matrices (N x K cm each; either may be NULL).                           */
int bmm_full_condprob(const int32_t *X, int32_t N, int32_t P, int32_t K, const double *theta,
                      const double *pi, int32_t precision, uint32_t flags, double *loglik, double *probs);

/* ---- device-resident plans (what the one-shot calls are built from) --------------------------- */
typedef struct bmm_plan bmm_plan;
#define BMM_SAMPLER_FULL 0
#define BMM_SAMPLER_STICKBREAKING 1
#define BMM_SAMPLER_COLLAPSED 2
#define BMM_SAMPLER_DP 3
/* Upload X / initial state, allocate device histories.  `init` may be NULL for dp. */
int bmm_plan_create(int32_t sampler, const bmm_args *args, const bmm_init *init, bmm_plan **plan);
/* Launch the whole run (all sweeps, relabelling, layout conversion) on the plan's stream. */
int bmm_plan_run(bmm_plan *plan);
int bmm_plan_sync(bmm_plan *plan);
/* Device time of the last bmm_plan_run in ms (CUDA events on the launching stream). */
int bmm_plan_elapsed_ms(bmm_plan *plan, float *total_ms, float *sampler_kernel_ms);
/* Device time of each launch group of the last run, in ms: [0] sampler sweeps 1..burnin-1,
 * [1] Stephens batch, [2] sampler sweeps burnin..nsamples-1 (all sweeps when !relabel),
 * [3] history layout conversion.  CUDA events on the launching stream. */
int bmm_plan_kernel_ms(bmm_plan *plan, float ms_out[4]);
/* Copy the results into caller (host) buffers. */
int bmm_plan_fetch(bmm_plan *plan, bmm_out *out);
int bmm_plan_destroy(bmm_plan *plan);

/* ---- multi-GPU (one process per GPU; the N-sharded uncollapsed samplers all-reduce counts) ---- */
int bmm_dist_unique_id(uint8_t id_out[128]);
int bmm_dist_init(int32_t rank, int32_t world, const uint8_t id[128], int32_t device);
int bmm_dist_finalize(void);
/* Optional one-shot all-reduce over NVLink peer memory for the per-sweep count exchange (replaces the
 * NCCL call, which is latency-bound at a few KB).  After bmm_dist_init every rank calls
 * bmm_dist_p2p_local(cap_ints, handle) -- cap_ints >= K + K*P of the largest run -- ships its 64-byte
 * CUDA IPC handle to all ranks (rank order), and calls bmm_dist_p2p_attach(handles[world][64]).       */
int bmm_dist_p2p_local(uint64_t cap_ints, uint8_t handle_out[64]);
int bmm_dist_p2p_attach(const uint8_t *handles);
int bmm_dist_p2p_detach(void);   /* back to NCCL; call on every rank if any attach failed */

/* ---- misc ----------------------------------------------------------------------------------- */
/* Page-locked host memory for output buffers (cudaHostAlloc): D2H into it runs at PCIe speed.    */
int bmm_host_alloc(uint64_t bytes, void **ptr_out);
int bmm_host_free(void *ptr);
/* Device buffers of finished calls are kept for reuse by the next call of the same shape (cudaMalloc /
 * cudaFree of GB-sized histories cost more than the sampling); this returns them to the driver.      */
int bmm_release_cache(void);
const char *bmm_last_error(void);
int bmm_device_count(void);
uint64_t bmm_launch_count(void);   /* kernels launched by this library so far */
uint64_t bmm_fetch_bytes(void);    /* device-to-host bytes moved by the calling thread's last bmm_plan_fetch (or one-shot gibbs call) */
const char *bmm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BMM_CAPI_H */
