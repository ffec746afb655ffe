// Host side of the C ABI declared in include/bmm_capi.h: argument checks, bit-packing and row
// de-duplication of X, device-resident plans, launches, result download.  No CPU fallback: every
// compute entry point needs a CUDA device and fails with BMM_ERR_CUDA otherwise.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <unistd.h>
#include <unordered_map>
#include <vector>

#include "../../include/bmm_capi.h"
#include "assign.cuh"
#include "kernels.h"
#include "dist.h"

#define BMM_FLAG_PROBE_PROBS 0x100u
#define BMM_FLAG_PROBE_LOGLIK 0x200u
#define BMM_FLAG_PROBE_COUNTS 0x400u
#define BMM_FLAG_PROBE_ZFREQ 0x1000u

namespace bmm {
bool full_rows_fit_smem(int U, int K);
}
extern "C" void bmm_widen_u8_i32(const uint8_t *src, int32_t *dst, size_t n, int threads);  // host_widen.cpp
extern "C" void bmm_widen_runs_u8_i32(const uint8_t *src, size_t x0, size_t n, int L, int S, int s_off, int N, int K,
                                      const int32_t *perm, int32_t *dst_z, int32_t *dst_zo, int threads);

namespace {

thread_local std::string g_err;
thread_local uint64_t g_fetch_bytes = 0;   // device-to-host bytes of this thread's last bmm_plan_fetch

int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(BMM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));         \
    } while (0)

// Device allocations are recycled across calls: cudaMalloc / cudaFree of the multi-GB history buffers
// cost 10-200 ms per call (cudaFree synchronises and unmaps), more than the sampling itself at C2 size.
// Freed blocks go to a per-device free list keyed by size and are handed out again on an exact-size
// match (repeated runs of one configuration, which is what a caller looping over data sets or seeds
// does); bmm_release_cache() returns everything to the driver, and so does an out-of-memory retry.
struct DevCache {
    std::mutex m;
    std::map<std::pair<int, size_t>, std::vector<void *>> free_list;
    size_t cached = 0;
    size_t cap = (size_t)24 << 30;   // bytes kept across calls (all devices), BMM_CACHE_GB overrides
    DevCache() { if (const char *e = getenv("BMM_CACHE_GB")) cap = (size_t)atoll(e) << 30; }
    void *take(int dev, size_t n) {
        std::lock_guard<std::mutex> g(m);
        auto it = free_list.find({dev, n});
        if (it == free_list.end() || it->second.empty()) return nullptr;
        void *p = it->second.back();
        it->second.pop_back();
        cached -= n;
        return p;
    }
    void give(int dev, size_t n, void *p) {
        std::lock_guard<std::mutex> g(m);
        if (cached + n > cap) {      // keep the idle footprint bounded: beyond the cap blocks go back to the driver
            int cur = 0;
            cudaGetDevice(&cur);
            if (cur != dev) cudaSetDevice(dev);
            cudaFree(p);
            if (cur != dev) cudaSetDevice(cur);
            return;
        }
        free_list[{dev, n}].push_back(p);
        cached += n;
    }
    void release() {
        std::lock_guard<std::mutex> g(m);
        int cur = 0;
        cudaGetDevice(&cur);
        for (auto &kv : free_list) {
            cudaSetDevice(kv.first.first);
            for (void *p : kv.second) cudaFree(p);
        }
        free_list.clear();
        cached = 0;
        cudaSetDevice(cur);
    }
} g_cache;

struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
    int dev = 0;
    ~DevBuf() { if (p) g_cache.give(dev, bytes, p); }
    cudaError_t alloc(size_t n, bool zero = true) {
        bytes = n;
        if (n == 0) return cudaSuccess;
        cudaGetDevice(&dev);
        p = g_cache.take(dev, n);
        if (!p) {
            cudaError_t e = cudaMalloc(&p, n);
            if (e == cudaErrorMemoryAllocation) {   // give the cached blocks back and try once more
                cudaGetLastError();
                g_cache.release();
                e = cudaMalloc(&p, n);
            }
            if (e != cudaSuccess) { p = nullptr; return e; }
        }
        return zero ? cudaMemset(p, 0, n) : cudaSuccess;
    }
    template <typename T> T *as() const { return (T *)p; }
};

}  // namespace

struct bmm_plan {
    int sampler = 0;
    bmm_args a{};
    int C = 1, N = 0, P = 0, K = 0, W = 0, U = 0, S = 0, ns = 0, thin = 1;   // S = kept sweeps (hist_count)
    bool relabel = false, replay = false;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr;
    cudaEvent_t evs[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    bmm::FullParams fp{};
    bmm::CollapsedParams cp{};
    bmm::BigParams bp{};
    bool grid_path = false;       // one chain over the whole GPU (kern_big.cu)
    int deb = 4;                  // bytes per allocation of the device-side R-layout z (1: widened on the host)
    bool derive_z = false;        // only z_original crosses PCIe; the host applies `permutations` while widening
    // Download of the chain-parallel paths when the host widens (deb == 1): the allocations travel as bytes, one buffer per
    // sweep segment, so that a segment is copied and widened while the next one is still being sampled.  (Widening a share
    // of the chains on the device and DMA-ing their int32 matrices beside the host workers was measured and lost: the
    // link of the GPU boxes moves ~25 GB/s, the 12 workers write ~130-150 GB/s.)
    std::vector<int> seg_slot;    // nseg + 1 boundaries in kept-history slots
    std::vector<cudaEvent_t> seg_ev;
    cudaStream_t copy_stream = nullptr;
    int sm_count = 148;
    std::vector<cudaEvent_t> sweep_ev;   // start/stop of the timed sweep kernels of the last run (grid path)
    std::vector<cudaEvent_t> relabel_ev; // ... and of the single-pass relabelling kernels, same stride
    int ev_stride = 1;            // every ev_stride-th sweep kernel is bracketed by events (0: none)
    bool sharded = false;         // rows of one chain block-partitioned over the ranks of bmm_dist_init
    bool x_p2p = false;           // counts exchanged over peer memory (else NCCL)
    bool use_graph = true, capturing = false;
    cudaGraphExec_t gexec[2] = {nullptr, nullptr};
    unsigned long long glaunches[2] = {0, 0};
    DevBuf ws_b1, ws_s0, ws_rep, x_done;
    DevBuf x_inbox, x_peer_arr, x_seq;   // single-GPU inbox of the tensor path (x_world = 1)
    DevBuf w1, w0, lpi, gsc, counts, counts_out, lp_table, lp_bias, cnt_ws;
    DevBuf probs_f32, Qf, cube_f, cost_acc, perm_cur;   // grid-path relabelling (float, row-major N x K)
    DevBuf sb_vws;                // warm-start potentials of the batch step's M assignments, (K + 1) doubles each
    bool fused_relabel = false;   // tensor path: online relabelling in one pass over Q per sweep (kern_big_ws_relabel.cu)
    // ... whose assignment solve (one warp, ~0.16 ms at K = 32) runs on a side stream beside the parameter update and the next
    // z-sweep; the sweep then leaves one SM to it (its CTAs take a whole SM's registers)
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool assign_inflight = false;
    DevBuf Qt, b1_hist, bias_hist;
    DevBuf zfreq;                 // grid-path posterior summary [N x K cm] uint32
    // data
    DevBuf rowbits, rowid, wt, xbits, logB, logG, logBG, logN, rBGP;
    // state
    DevBuf theta_cur, pi_cur, alpha_cur, Q, logQ, cube, logp, prob_g, hist_g, ll_g, assign_ws, status, cost_g;
    DevBuf z_cur, cnt, dp_used, dp_free, probs_sample, sb_perm, sb_cost, sb_ws, perm_inv;
    // histories
    DevBuf zhist, theta_out, theta_rel_out, pi_out, alpha_out, perm_out, probs_out, loglik_out, kactive;
    DevBuf z_orig, z_rel, Qexp;
    // replay
    DevBuf ru, rpi, rtheta, ralpha;
    bool ran = false;
    // Chain state as bmm_plan_create left it, restored at the start of every bmm_plan_run so that a plan can be
    // run any number of times (each run is the same chain from the same initial state).
    struct Snap { DevBuf *live; DevBuf copy; };
    std::vector<std::unique_ptr<Snap>> snaps;
    std::vector<DevBuf *> zero_at_run;   // buffers the reference starts from zero (arma::fill::zeros) and only partly writes
    int runs = 0;
    ~bmm_plan() {
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (evk0) cudaEventDestroy(evk0);
        if (evk1) cudaEventDestroy(evk1);
        for (auto &e : evs) if (e) cudaEventDestroy(e);
        for (auto &e : sweep_ev) if (e) cudaEventDestroy(e);
        for (auto &e : relabel_ev) if (e) cudaEventDestroy(e);
        for (auto &e : seg_ev) if (e) cudaEventDestroy(e);
        if (copy_stream) cudaStreamDestroy(copy_stream);
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_join) cudaEventDestroy(ev_join);
        if (side) cudaStreamDestroy(side);
        for (auto &g : gexec) if (g) cudaGraphExecDestroy(g);
        if (stream) cudaStreamDestroy(stream);
    }
};

namespace {

int check_args(int sampler, const bmm_args *a, const bmm_init *init) {
    if (!a) return fail(BMM_ERR_INVALID, "args is NULL");
    if (!a->X || a->N <= 0 || a->P <= 0) return fail(BMM_ERR_INVALID, "X must be a non-empty N x P matrix");
    if (a->nsamples < 2) return fail(BMM_ERR_INVALID, "nsamples must be >= 2");
    if (a->K < 1 || a->K > 255) return fail(BMM_ERR_INVALID, "K / maxK must be in 1..255");
    if (a->burnin < 0 || a->burnin >= a->nsamples) return fail(BMM_ERR_INVALID, "burnin must be in [0, nsamples)");
    if (a->thin < 0) return fail(BMM_ERR_INVALID, "thin must be >= 0 (0 / 1 = keep every sweep)");
    if (a->relabel) {
        // the reference's behaviour is undefined otherwise (SURVEY App. D quirk 15)
        if (a->burnin < 2) return fail(BMM_ERR_INVALID, "relabel needs burnin >= 2 (Q is initialised at sweep burnin-1)");
        // burnrelabel > burnin is legal at this level, as at the reference's .Call level: only the R wrappers clamp
        // it, and gibbs_stickbreaking's does not (R/utils.R:95-107).  The slices of probs_out before sweep 1 stay
        // zero and become 1e-6 in my_stephens_batch (stephens.cpp:30-31).
        if (a->burnrelabel < 1) return fail(BMM_ERR_INVALID, "relabel needs burnrelabel >= 1");
        if (a->burnrelabel > 100000) return fail(BMM_ERR_INVALID, "burnrelabel too large");
    }
    if (!(a->beta > 0) || !(a->gamma > 0)) return fail(BMM_ERR_INVALID, "beta and gamma must be > 0");
    if (a->alpha < 0) return fail(BMM_ERR_INVALID, "alpha must be >= 0 (0 = sample it)");
    if (a->precision != BMM_FP64 && a->precision != BMM_FP32) return fail(BMM_ERR_INVALID, "precision must be BMM_FP64 or BMM_FP32");
    if (sampler == BMM_SAMPLER_DP && a->beta != a->gamma)
        return fail(BMM_ERR_BETA_GAMMA, "Error: sampler currently not implemented for non-symmetric priors on beta and gamma");
    if (sampler == BMM_SAMPLER_FULL || sampler == BMM_SAMPLER_STICKBREAKING) {
        if (!init || !init->pi || !init->theta) return fail(BMM_ERR_INVALID, "initialPi / initialTheta required");
    }
    if (sampler == BMM_SAMPLER_COLLAPSED && (!init || !init->z)) return fail(BMM_ERR_INVALID, "initialK required");
    if (a->replay) {
        const bmm_replay *r = a->replay;
        if (!r->u || r->u_slots < 1) return fail(BMM_ERR_INVALID, "replay needs u and u_slots");
        if ((sampler == BMM_SAMPLER_FULL || sampler == BMM_SAMPLER_STICKBREAKING) && (!r->pi || !r->theta || !r->alpha))
            return fail(BMM_ERR_INVALID, "replay of an uncollapsed sampler needs pi, theta and alpha histories");
    }
    return BMM_OK;
}

// X (N x P int32 cm) -> bit-packed rows [N][W]; rejects non-binary input.
int pack_rows(const int32_t *X, int N, int P, std::vector<uint32_t> &bits, int &W) {
    W = (P + 31) / 32;
    bits.assign((size_t)N * W, 0u);
    for (int d = 0; d < P; ++d) {
        const int32_t *col = X + (size_t)N * d;
        const uint32_t m = 1u << (d & 31);
        const int w = d >> 5;
        for (int i = 0; i < N; ++i) {
            const int32_t v = col[i];
            if (v == 1) bits[(size_t)i * W + w] |= m;
            else if (v != 0) return fail(BMM_ERR_NOT_BINARY, "X must contain only 0/1 (the bit-packed path rejects other integers)");
        }
    }
    return BMM_OK;
}

template <typename T>
int upload(DevBuf &b, const T *src, size_t n) {
    CU(b.alloc(n * sizeof(T), false));
    if (n) CU(cudaMemcpy(b.p, src, n * sizeof(T), cudaMemcpyHostToDevice));
    return BMM_OK;
}

#define TRY(x) do { int rc_ = (x); if (rc_) return rc_; } while (0)

// De-duplicate bit-packed rows [N][W] in first-occurrence order: rowid[i] = index of row i among the U distinct rows,
// wt[u] = multiplicity of distinct row u, rowbits = the distinct rows [U][W].  The hash set keys on row indices and
// reads the words in place, so N = 1e7 rows need no per-row allocation.
void dedup_rows(const uint32_t *bits, int N, int W, std::vector<int> &rowid, std::vector<int> &wt,
                std::vector<uint32_t> &rowbits) {
    auto hash = [&](int i) {
        uint64_t h = 1469598103934665603ull;
        for (int w = 0; w < W; ++w) { h ^= bits[(size_t)i * W + w]; h *= 1099511628211ull; }
        return (size_t)h;
    };
    auto eq = [&](int i, int j) { return std::memcmp(bits + (size_t)i * W, bits + (size_t)j * W, (size_t)W * 4) == 0; };
    std::unordered_map<int, int, decltype(hash), decltype(eq)> seen(std::min(N, 1 << 20), hash, eq);
    rowid.assign(N, 0);
    wt.clear();
    rowbits.clear();
    for (int i = 0; i < N; ++i) {
        auto it = seen.find(i);
        if (it == seen.end()) {
            const int u = (int)wt.size();
            seen.emplace(i, u);
            wt.push_back(1);
            rowbits.insert(rowbits.end(), bits + (size_t)i * W, bits + (size_t)(i + 1) * W);
            rowid[i] = u;
        } else {
            wt[it->second]++;
            rowid[i] = it->second;
        }
    }
}

int create_full(bmm_plan *pl, const bmm_init *init) {
    const bmm_args &a = pl->a;
    const int N = pl->N, P = pl->P, K = pl->K, C = pl->C, ns = pl->ns, S = pl->S;
    std::vector<uint32_t> bits;
    int W;
    TRY(pack_rows(a.X, N, P, bits, W));
    pl->W = W;
    std::vector<int> rowid, wt;
    std::vector<uint32_t> rowbits;
    dedup_rows(bits.data(), N, W, rowid, wt, rowbits);
    const int U = (int)wt.size();
    pl->U = U;
    const size_t UK = (size_t)U * K, KP = (size_t)K * P;
    TRY(upload(pl->rowbits, rowbits.data(), rowbits.size()));
    TRY(upload(pl->rowid, rowid.data(), rowid.size()));
    TRY(upload(pl->wt, wt.data(), wt.size()));
    // initial state
    TRY(upload(pl->theta_cur, init->theta, (size_t)C * KP));
    TRY(upload(pl->pi_cur, init->pi, (size_t)C * K));
    std::vector<double> al(C, a.alpha == 0 ? 1.0 : a.alpha);
    TRY(upload(pl->alpha_cur, al.data(), al.size()));
    const bool use_hist = bmm::full_rows_fit_smem(U, K);
    const bool probes = (a.flags & (BMM_FLAG_PROBE_PROBS | BMM_FLAG_PROBE_LOGLIK)) != 0;
    (void)probes;
    if (pl->relabel) {
        CU(pl->Q.alloc((size_t)C * UK * 8));
        CU(pl->logQ.alloc((size_t)C * UK * 8));
        CU(pl->cube.alloc((size_t)C * a.burnrelabel * UK * 8));
        CU(pl->logp.alloc((size_t)C * a.burnrelabel * UK * 8));
        CU(pl->sb_perm.alloc((size_t)C * a.burnrelabel * K * 4));
        CU(pl->sb_cost.alloc((size_t)C * a.burnrelabel * K * K * 8));
        CU(pl->sb_ws.alloc((size_t)C * a.burnrelabel * bmm::assign_ws_bytes(K)));
        CU(pl->perm_out.alloc((size_t)C * S * K * 4));
        CU(pl->theta_rel_out.alloc((size_t)C * KP * S * 8));
        if (K * K > bmm::COST_SMEM_MAX) CU(pl->cost_g.alloc((size_t)C * K * K * 8));
    }
    if (!use_hist) CU(pl->prob_g.alloc((size_t)C * UK * 8));
    if (a.flags & BMM_FLAG_PROBE_LOGLIK) CU(pl->ll_g.alloc((size_t)C * UK * 8));
    CU(pl->assign_ws.alloc((size_t)C * bmm::assign_ws_bytes(K)));
    CU(pl->status.alloc((size_t)C * 4));
    CU(pl->zhist.alloc((size_t)C * ns * N));
    CU(pl->theta_out.alloc((size_t)C * KP * S * 8));
    CU(pl->pi_out.alloc((size_t)C * S * K * 8));
    CU(pl->alpha_out.alloc((size_t)C * S * 8));
    if (a.flags & BMM_FLAG_PROBE_PROBS) CU(pl->probs_out.alloc((size_t)C * ns * N * K * 8));
    if (a.flags & BMM_FLAG_PROBE_LOGLIK) CU(pl->loglik_out.alloc((size_t)C * ns * N * K * 8));
    if (a.replay) {
        const bmm_replay *r = a.replay;
        TRY(upload(pl->ru, r->u, (size_t)C * ns * N * r->u_slots));
        TRY(upload(pl->rpi, r->pi, (size_t)C * ns * K));
        TRY(upload(pl->rtheta, r->theta, (size_t)C * KP * ns));
        TRY(upload(pl->ralpha, r->alpha, (size_t)C * ns));
    }
    bmm::FullParams &f = pl->fp;
    f.N = N; f.P = P; f.K = K; f.U = U; f.W = W;
    f.nsamples = ns; f.burnin = a.burnin; f.relabel = pl->relabel; f.burnrelabel = a.burnrelabel; f.thin = pl->thin;
    f.stickbreaking = pl->sampler == BMM_SAMPLER_STICKBREAKING;
    f.alpha0 = a.alpha; f.beta = a.beta; f.gamma = a.gamma; f.a = a.a; f.b = a.b;
    f.seed = a.seed; f.chain_offset = a.chain_offset; f.flags = a.flags; f.use_hist = use_hist;
    f.rowbits = pl->rowbits.as<uint32_t>(); f.rowid = pl->rowid.as<int>(); f.wt = pl->wt.as<int>();
    f.theta_cur = pl->theta_cur.as<double>(); f.pi_cur = pl->pi_cur.as<double>(); f.alpha_cur = pl->alpha_cur.as<double>();
    f.Q = pl->Q.as<double>(); f.logQ = pl->logQ.as<double>(); f.cube = pl->cube.as<double>();
    f.prob_g = pl->prob_g.as<double>(); f.hist_g = nullptr; f.ll_g = pl->ll_g.as<double>();
    f.assign_ws = pl->assign_ws.as<char>(); f.status = pl->status.as<int>(); f.cost_g = pl->cost_g.as<double>();
    f.zhist = pl->zhist.as<uint8_t>(); f.theta_out = pl->theta_out.as<double>(); f.theta_rel_out = pl->theta_rel_out.as<double>();
    f.pi_out = pl->pi_out.as<double>(); f.alpha_out = pl->alpha_out.as<double>(); f.perm_out = pl->perm_out.as<int>();
    f.probs_out = pl->probs_out.as<double>(); f.loglik_out = pl->loglik_out.as<double>();
    f.ru = pl->ru.as<double>(); f.ru_slots = a.replay ? a.replay->u_slots : 0;
    f.rpi = pl->rpi.as<double>(); f.rtheta = pl->rtheta.as<double>(); f.ralpha = pl->ralpha.as<double>();
    size_t smem = bmm::full_smem_bytes(f, 128);
    if (smem > 200 * 1024) return fail(BMM_ERR_UNSUPPORTED, "K*P too large for the chain-per-block kernel");
    return BMM_OK;
}

// One chain over the whole GPU (and N-sharded over the ranks of bmm_dist_init): kern_big.cu.
int create_big(bmm_plan *pl, const bmm_init *init) {
    const bmm_args &a = pl->a;
    const int N = pl->N, P = pl->P, K = pl->K, ns = pl->ns, S = pl->S;
    if (pl->C != 1) return fail(BMM_ERR_UNSUPPORTED, "the grid path runs one chain (n_chains <= 1)");
    if (a.replay && K > bmm::big_replay_max_k()) return fail(BMM_ERR_UNSUPPORTED, "grid-path replay needs K <= 64");
    const long long n_global = a.n_global > 0 ? a.n_global : N;
    if (a.row_offset < 0 || a.row_offset + N > n_global) return fail(BMM_ERR_INVALID, "row_offset + N exceeds n_global");
    int W = (P + 31) / 32;
    if (a.flags & BMM_FLAG_X_PACKED) {
        TRY(upload(pl->xbits, (const uint32_t *)a.X, (size_t)N * W));
    } else {
        std::vector<uint32_t> bits;
        TRY(pack_rows(a.X, N, P, bits, W));
        TRY(upload(pl->xbits, bits.data(), bits.size()));
    }
    pl->W = W; pl->U = N;
    const size_t KP = (size_t)K * P;
    TRY(upload(pl->theta_cur, init->theta, KP));
    TRY(upload(pl->pi_cur, init->pi, (size_t)K));
    std::vector<double> al(1, a.alpha == 0 ? 1.0 : a.alpha);
    TRY(upload(pl->alpha_cur, al.data(), 1));
    CU(pl->w1.alloc(KP * 8)); CU(pl->w0.alloc(KP * 8)); CU(pl->lpi.alloc((size_t)K * 8)); CU(pl->gsc.alloc((size_t)K * 8));
    CU(pl->counts.alloc(2 * (K + KP) * 4));
    CU(pl->status.alloc(8));   // [0] chain status, [1] scratch flag of the batch relabelling loop
    const bool keep = !(a.flags & BMM_FLAG_NO_Z_HISTORY);
    CU(pl->zhist.alloc(keep ? (size_t)ns * N : (size_t)N));
    CU(pl->theta_out.alloc(KP * S * 8));
    CU(pl->pi_out.alloc((size_t)S * K * 8));
    CU(pl->alpha_out.alloc((size_t)S * 8));
    if (a.flags & BMM_FLAG_PROBE_PROBS) CU(pl->probs_out.alloc((size_t)ns * N * K * 8));
    if (a.flags & BMM_FLAG_PROBE_LOGLIK) CU(pl->loglik_out.alloc((size_t)ns * N * K * 8));
    if (a.flags & BMM_FLAG_PROBE_COUNTS) CU(pl->counts_out.alloc((size_t)ns * (K + KP) * 4));
    if (a.flags & BMM_FLAG_PROBE_ZFREQ) CU(pl->zfreq.alloc((size_t)N * K * 4));
    if (pl->relabel) {
        const size_t NK = (size_t)N * K;
        size_t free_b = 0, total_b = 0;
        CU(cudaMemGetInfo(&free_b, &total_b));
        if ((2 + (size_t)a.burnrelabel) * NK * 4 > free_b / 2)
            return fail(BMM_ERR_UNSUPPORTED, "relabel on the grid path: burnrelabel x N x K probabilities do not fit the device; lower burnrelabel");
        // shapes of the tensor sweep (big_tc_supported): P is recomputed instead of stored, Q streams once per sweep
        const char *fenv = getenv("BMM_RELABEL_FUSED");
        pl->fused_relabel = a.precision == BMM_FP32 && !(a.flags & (BMM_FLAG_NO_TENSOR | BMM_FLAG_PROBE_LOGLIK)) && !getenv("BMM_NO_TC") &&
                            K <= 32 && P <= 112 && !a.replay && !(fenv && fenv[0] == '0');
        if (pl->fused_relabel) {
            CU(cudaStreamCreateWithFlags(&pl->side, cudaStreamNonBlocking));
            CU(cudaEventCreateWithFlags(&pl->ev_fork, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&pl->ev_join, cudaEventDisableTiming));
            CU(pl->Qt.alloc(bmm::wsr_q_tiled_bytes(N), false));
            CU(pl->b1_hist.alloc(2 * bmm::ws_b1_bytes(P)));
            CU(pl->bias_hist.alloc(2 * 32 * sizeof(float)));
        } else CU(pl->probs_f32.alloc(NK * 4));
        CU(pl->Qf.alloc(NK * 4)); CU(pl->cube_f.alloc((size_t)a.burnrelabel * NK * 4));
        CU(pl->cost_acc.alloc(((size_t)K * K + K) * 8));
        CU(pl->perm_cur.alloc((size_t)K * 4));
        CU(pl->sb_perm.alloc((size_t)a.burnrelabel * K * 4));
        CU(pl->perm_inv.alloc((size_t)(a.burnrelabel > 1 ? a.burnrelabel : 1) * K * 4));   // BMM_FLAG_STEPHENS_FIXED
        CU(pl->perm_out.alloc((size_t)S * K * 4));
        CU(pl->theta_rel_out.alloc(KP * S * 8));
        CU(pl->assign_ws.alloc(bmm::assign_ws_bytes(K)));
        CU(pl->sb_vws.alloc((size_t)a.burnrelabel * (K + 1) * sizeof(double)));
    }
    if (a.replay) {
        const bmm_replay *r = a.replay;
        TRY(upload(pl->ru, r->u, (size_t)ns * N * r->u_slots));
        TRY(upload(pl->rpi, r->pi, (size_t)ns * K));
        TRY(upload(pl->rtheta, r->theta, KP * ns));
        TRY(upload(pl->ralpha, r->alpha, (size_t)ns));
    }
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, a.device));
    pl->sm_count = prop.multiProcessorCount;
    bmm::BigParams &b = pl->bp;
    b.N_global = n_global; b.row_offset = a.row_offset; b.N_local = N; b.P = P; b.K = K; b.W = W;
    b.nsamples = ns; b.burnin = a.burnin; b.stickbreaking = pl->sampler == BMM_SAMPLER_STICKBREAKING; b.thin = pl->thin;
    b.precision = a.precision; b.tables_in_smem = bmm::big_tables_fit_smem(K, P, a.precision); b.keep_history = keep;
    b.alpha0 = a.alpha; b.beta = a.beta; b.gamma = a.gamma; b.a = a.a; b.b = a.b;
    b.seed = a.seed; b.chain_offset = a.chain_offset; b.flags = a.flags;
    b.xbits = pl->xbits.as<uint32_t>();
    b.w1 = pl->w1.as<double>(); b.w0 = pl->w0.as<double>(); b.lpi = pl->lpi.as<double>();
    b.theta_cur = pl->theta_cur.as<double>(); b.pi_cur = pl->pi_cur.as<double>(); b.alpha_cur = pl->alpha_cur.as<double>();
    b.gsc = pl->gsc.as<double>(); b.counts = pl->counts.as<int>(); b.status = pl->status.as<int>();
    b.zhist = pl->zhist.as<uint8_t>();
    b.theta_out = pl->theta_out.as<double>(); b.pi_out = pl->pi_out.as<double>(); b.alpha_out = pl->alpha_out.as<double>();
    b.probs_out = pl->probs_out.as<double>(); b.loglik_out = pl->loglik_out.as<double>();
    b.counts_out = pl->counts_out.as<int>();
    // single-pass relabelling: the relabelled theta history is produced at the end of the run from the permutation history,
    // so the update kernel need not wait for the sweep's assignment
    b.probs_f32 = nullptr; b.perm_cur = pl->perm_cur.as<int>(); b.theta_rel_out = pl->fused_relabel ? nullptr : pl->theta_rel_out.as<double>();
    if (a.precision == BMM_FP32 && !(a.flags & BMM_FLAG_NO_TENSOR) && K <= 128 && (K > 32 || P > 112)) {
        CU(pl->lp_table.alloc(bmm::big_lp_table_bytes(P)));
        CU(pl->lp_bias.alloc(128 * 8));
        CU(pl->cnt_ws.alloc((2 * ((size_t)K + 1) + (size_t)N) * 4, false));
        if (!pl->zhist.p) return fail(BMM_ERR_INVALID, "internal: allocation buffer missing");
    }
    b.lp_table = pl->lp_table.p; b.lp_bias = pl->lp_bias.as<double>(); b.cnt_ws = pl->cnt_ws.as<int>();
    b.ru = pl->ru.as<double>(); b.ru_slots = a.replay ? a.replay->u_slots : 0;
    b.rpi = pl->rpi.as<double>(); b.rtheta = pl->rtheta.as<double>(); b.ralpha = pl->ralpha.as<double>();
    const bool tensor_ws = !(a.flags & BMM_FLAG_NO_TENSOR) && !getenv("BMM_NO_TC") && bmm::big_tc_supported(b);
    if (tensor_ws) {
        CU(pl->ws_b1.alloc(bmm::ws_b1_bytes(P)));     // zero: rows k >= K and columns d >= P stay zero
        CU(pl->ws_s0.alloc(32 * 8));
        CU(pl->ws_rep.alloc(bmm::ws_rep_bytes(K, P)));
        CU(pl->x_done.alloc(sizeof(unsigned)));
        b.ws_b1 = pl->ws_b1.as<unsigned char>(); b.ws_s0 = pl->ws_s0.as<double>(); b.ws_rep = pl->ws_rep.as<int>();
        b.x_done = pl->x_done.as<unsigned>();
    }
    pl->sharded = n_global > N;
    if (pl->sharded) {
        if (bmm::dist_world() < 2) return fail(BMM_ERR_NCCL, "N-sharded run needs bmm_dist_init with world > 1");
        const size_t ncnt = (size_t)K + KP;
        pl->x_p2p = bmm::dist_p2p_ready(ncnt);
        if (pl->x_p2p) {
            const bmm::P2PView v = bmm::dist_p2p_view();
            if (!pl->x_done.p) CU(pl->x_done.alloc(sizeof(unsigned)));
            b.x_world = v.world; b.x_rank = v.rank; b.x_cap = v.cap; b.x_peer = v.peer; b.x_local = v.local; b.x_seq = v.seq;
            b.x_done = pl->x_done.as<unsigned>();
            b.x_fused = tensor_ws ? 1 : 0;
        }
    }
    if (tensor_ws && !pl->sharded) {     // one GPU: the same tagged hand-over through a local inbox
        const size_t ncnt = (size_t)K + KP;
        CU(pl->x_inbox.alloc(2 * ncnt * sizeof(int2), false));
        CU(cudaMemset(pl->x_inbox.p, 0xFF, pl->x_inbox.bytes));
        int2 *self = pl->x_inbox.as<int2>();
        TRY(upload(pl->x_peer_arr, &self, 1));
        const int seq0[2] = {1, 1};
        TRY(upload(pl->x_seq, seq0, 2));
        b.x_world = 1; b.x_rank = 0; b.x_cap = ncnt; b.x_peer = pl->x_peer_arr.as<int2 *>(); b.x_local = self;
        b.x_seq = pl->x_seq.as<int>(); b.x_done = pl->x_done.as<unsigned>(); b.x_fused = 1;
    }
    {   // sweep-kernel timing: every sweep for short runs, every 8th otherwise (BMM_SWEEP_EVENTS = stride, 0 = none)
        const char *e = getenv("BMM_SWEEP_EVENTS");
        pl->ev_stride = e ? atoi(e) : (ns <= 24 ? 1 : 8);
        if (const char *g = getenv("BMM_GRAPH")) pl->use_graph = g[0] != '0';
    }
    return BMM_OK;
}

// ---- the grid path's sweep loop -------------------------------------------------------------------------
// One sweep = front (z-sweep kernel, count exchange) + back (online relabelling, parameter update).  The batch
// initialisation of the relabelling sits between the front and the back of sweep burnin-1 and needs the host
// (its early exit reads a flag), so a run is: segment A = everything up to and including front(burnin-1),
// the batch step, segment B = the rest.  Each segment is captured once into a CUDA graph and replayed by later
// runs: per sweep the host would otherwise issue 3-8 launches, and at 8 GPUs a sweep kernel lasts ~45 us.
int sweep_front(bmm_plan *pl, int j) {
    const bmm::BigParams &b = pl->bp;
    const int burnin = pl->a.burnin, M = pl->a.burnrelabel, K = b.K;
    const size_t NK = (size_t)b.N_local * K, ncnt = (size_t)K + (size_t)K * b.P;
    bmm::BigParams bj = b;
    if (pl->relabel) {   // where this sweep's probabilities go (full_gibbs.cpp:146-156)
        if (j < burnin && j >= burnin - M) bj.probs_f32 = pl->cube_f.as<float>() + (size_t)(j - burnin + M) * NK;
        else if (j >= burnin && !pl->fused_relabel) bj.probs_f32 = pl->probs_f32.as<float>();
    }
    if (b.ru) CU(bmm::launch_big_replay_load(bj, j, pl->stream));
    const bool timed = pl->ev_stride > 0 && (j % pl->ev_stride) == 0;
    if (timed) CU(cudaEventRecordWithFlags(pl->sweep_ev[2 * j], pl->stream, pl->capturing ? cudaEventRecordExternal : 0));
    CU(bmm::launch_big_sweep(bj, j, pl->assign_inflight && pl->sm_count > 8 ? pl->sm_count - 1 : pl->sm_count, pl->stream));
    if (timed) CU(cudaEventRecordWithFlags(pl->sweep_ev[2 * j + 1], pl->stream, pl->capturing ? cudaEventRecordExternal : 0));
    if (pl->sharded) {   // counts of all ranks: pushed over peer memory when attached (consumed by the update kernel), else NCCL
        int *cj = pl->counts.as<int>() + (size_t)(j & 1) * ncnt;
        if (pl->x_p2p) {
            if (!b.x_fused && bmm::dist_p2p_publish(cj, ncnt, j, pl->stream)) return fail(BMM_ERR_NCCL, bmm::dist_error());
        } else if (bmm::dist_allreduce_i32(cj, ncnt, pl->stream)) return fail(BMM_ERR_NCCL, bmm::dist_error());
    }
    return BMM_OK;
}

// One pass of the fused online relabelling: j in [burnin, ns) accumulates sweep j's cost matrix and applies the Q update of
// sweep j - 1; j == ns only applies the last update and returns Q to its row-major form.
int relabel_pass(bmm_plan *pl, int j) {
    const bmm::BigParams &b = pl->bp;
    const int burnin = pl->a.burnin, ns = pl->ns;
    const bool st_fixed = (pl->a.flags & BMM_FLAG_STEPHENS_FIXED) != 0;
    bmm::WsRelabelParams r{};
    r.N_local = b.N_local; r.P = b.P; r.K = b.K; r.W = b.W;
    r.xbits = b.xbits; r.b1_cur = b.ws_b1; r.lpi = b.lpi; r.s0 = b.ws_s0;
    r.b1_hist = pl->b1_hist.as<unsigned char>(); r.bias_hist = pl->bias_hist.as<float>();
    r.hist_prev = (j - 1) & 1; r.hist_next = j < ns ? (j & 1) : -1;
    r.perm = st_fixed ? pl->perm_inv.as<int>() : pl->perm_cur.as<int>();
    r.upd = j > burnin; r.do_cost = j < ns;
    const float sn = (float)(j - 1), inv = 1.f / (float)j;       // the pending update is sweep j - 1's (stephens.cpp:92)
    r.cq = sn * inv; r.cp = st_fixed ? inv : sn * inv;
    r.q_in_rowmajor = j == burnin; r.q_out_rowmajor = j == ns;
    r.q_direct = getenv("BMM_WSR_QDIRECT") != nullptr;
    r.Q_rm = pl->Qf.as<float>(); r.Q_tiled = pl->Qt.as<float>();
    r.cost_out = pl->cost_acc.as<double>(); r.status = pl->status.as<int>();
    if (r.do_cost) CU(cudaMemsetAsync(pl->cost_acc.p, 0, pl->cost_acc.bytes, pl->stream));
    const bool timed = j < ns && pl->ev_stride > 0 && (j % pl->ev_stride) == 0 && pl->relabel_ev.size() >= (size_t)2 * ns;
    if (timed) CU(cudaEventRecordWithFlags(pl->relabel_ev[2 * j], pl->stream, pl->capturing ? cudaEventRecordExternal : 0));
    CU(bmm::launch_big_relabel_ws(r, pl->sm_count, pl->stream));
    if (timed) CU(cudaEventRecordWithFlags(pl->relabel_ev[2 * j + 1], pl->stream, pl->capturing ? cudaEventRecordExternal : 0));
    return BMM_OK;
}

// the side stream's assignment solve must have finished before anything on the main stream reads perm_cur
int join_assign(bmm_plan *pl) {
    if (pl->assign_inflight) {
        CU(cudaStreamWaitEvent(pl->stream, pl->ev_join, 0));
        pl->assign_inflight = false;
    }
    return BMM_OK;
}

int sweep_back(bmm_plan *pl, int j) {
    const bmm::BigParams &b = pl->bp;
    const int burnin = pl->a.burnin, K = b.K;
    const long long N = b.N_local;
    const int st_fixed = (pl->a.flags & BMM_FLAG_STEPHENS_FIXED) ? 1 : 0;
    const int cost_tc = (pl->a.precision == BMM_FP32 && !(pl->a.flags & BMM_FLAG_NO_TENSOR)) ? 1 : 0;
    if (pl->relabel && j >= burnin && pl->fused_relabel) {
        TRY(join_assign(pl));                    // this pass applies the permutation of sweep j - 1
        TRY(relabel_pass(pl, j));
        if (pl->sharded && bmm::dist_allreduce_f64(pl->cost_acc.as<double>(), (size_t)K * K + K, pl->stream))
            return fail(BMM_ERR_NCCL, bmm::dist_error());
        const int slot = bmm::hist_slot(j, burnin, pl->thin);
        static const bool fork = !(getenv("BMM_ASSIGN_FORK") && getenv("BMM_ASSIGN_FORK")[0] == '0');
        cudaStream_t as = fork ? pl->side : pl->stream;
        if (fork) {
            CU(cudaEventRecord(pl->ev_fork, pl->stream));
            CU(cudaStreamWaitEvent(pl->side, pl->ev_fork, 0));
        }
        CU(bmm::launch_grid_assign(K, pl->cost_acc.as<double>(), pl->assign_ws.as<char>(), pl->perm_cur.as<int>(),
                                   slot >= 0 ? pl->perm_out.as<int>() + slot : nullptr, pl->S, as));
        if (st_fixed) CU(bmm::launch_grid_invert_perm(1, K, pl->perm_cur.as<int>(), pl->perm_inv.as<int>(), as));
        if (fork) {
            CU(cudaEventRecord(pl->ev_join, pl->side));
            pl->assign_inflight = true;
        }
        if (pl->zfreq.p) TRY(join_assign(pl));   // the summary below reads perm_cur
    } else if (pl->relabel && j >= burnin) {       // my_stephens_online (full_gibbs.cpp:166-175)
        CU(bmm::launch_grid_cost(N, K, pl->probs_f32.as<float>(), pl->Qf.as<float>(), st_fixed, pl->cost_acc.as<double>(),
                                 pl->sm_count, pl->stream, cost_tc, pl->status.as<int>()));
        if (pl->sharded && bmm::dist_allreduce_f64(pl->cost_acc.as<double>(), (size_t)K * K + K, pl->stream))
            return fail(BMM_ERR_NCCL, bmm::dist_error());
        const int slot = bmm::hist_slot(j, burnin, pl->thin);
        CU(bmm::launch_grid_assign(K, pl->cost_acc.as<double>(), pl->assign_ws.as<char>(), pl->perm_cur.as<int>(),
                                   slot >= 0 ? pl->perm_out.as<int>() + slot : nullptr, pl->S, pl->stream));
        if (st_fixed) CU(bmm::launch_grid_invert_perm(1, K, pl->perm_cur.as<int>(), pl->perm_inv.as<int>(), pl->stream));
        CU(bmm::launch_grid_qupdate(N, K, pl->Qf.as<float>(), pl->probs_f32.as<float>(),
                                    st_fixed ? pl->perm_inv.as<int>() : pl->perm_cur.as<int>(), j, pl->sm_count, pl->stream, st_fixed));
    }
    if (pl->zfreq.p && j >= burnin)
        CU(bmm::launch_grid_zfreq(N, K, pl->zhist.as<uint8_t>() + (size_t)(b.keep_history ? j : 0) * N,
                                  pl->relabel ? pl->perm_cur.as<int>() : nullptr, pl->zfreq.as<unsigned>(), pl->sm_count, pl->stream));
    CU(bmm::launch_big_params(b, j, pl->stream));
    return BMM_OK;
}

// my_stephens_batch on the grid path (full_gibbs.cpp:163-165), after front(burnin - 1); host-synchronised
int batch_relabel_big(bmm_plan *pl) {
    const bmm::BigParams &b = pl->bp;
    const int M = pl->a.burnrelabel, K = b.K;
    const long long N = b.N_local;
    const size_t NK = (size_t)N * K;
    const int st_fixed = (pl->a.flags & BMM_FLAG_STEPHENS_FIXED) ? 1 : 0;
    const int cost_tc = (pl->a.precision == BMM_FP32 && !(pl->a.flags & BMM_FLAG_NO_TENSOR)) ? 1 : 0;
    float *cube = pl->cube_f.as<float>();
    int *sbp = pl->sb_perm.as<int>();
    CU(bmm::launch_grid_clamp((long long)M * (long long)NK, cube, pl->sm_count, pl->stream));
    CU(bmm::launch_grid_identity_perm(M * K, K, sbp, pl->stream));
    // The reference always runs 100 iterations (threshold 10^(-6) == -16, quirk 1).  Once an iteration
    // leaves every permutation unchanged the following ones recompute the same Q, costs and
    // assignments, so stopping there returns exactly what the 100th iteration would.
    int *flag = pl->status.as<int>() + 1;
    for (int iter = 0; iter < 100; ++iter) {
        if (st_fixed) CU(bmm::launch_grid_invert_perm(M, K, sbp, pl->perm_inv.as<int>(), pl->stream));
        CU(bmm::launch_grid_qmean(N, K, M, cube, st_fixed ? pl->perm_inv.as<int>() : sbp, pl->Qf.as<float>(), pl->sm_count,
                                  pl->stream));
        CU(cudaMemsetAsync(flag, 0, sizeof(int), pl->stream));
        for (int t = 0; t < M; ++t) {
            CU(bmm::launch_grid_cost(N, K, cube + (size_t)t * NK, pl->Qf.as<float>(), 1, pl->cost_acc.as<double>(),
                                     pl->sm_count, pl->stream, cost_tc, pl->status.as<int>()));
            if (pl->sharded && bmm::dist_allreduce_f64(pl->cost_acc.as<double>(), (size_t)K * K + K, pl->stream))
                return fail(BMM_ERR_NCCL, bmm::dist_error());
            CU(bmm::launch_grid_assign(K, pl->cost_acc.as<double>(), pl->sb_vws.as<char>() + (size_t)t * (K + 1) * sizeof(double), nullptr,
                                       sbp + (size_t)t * K, 1, pl->stream, flag));
        }
        int changed = 1;   // every rank sees the same all-reduced costs, hence the same flag
        CU(cudaMemcpyAsync(&changed, flag, sizeof(int), cudaMemcpyDeviceToHost, pl->stream));
        CU(cudaStreamSynchronize(pl->stream));
        if (!changed) break;
    }
    return BMM_OK;
}

// Segment 0: run prologue, sweeps [1, jsplit) in full, front(jsplit).  Segment 1: back(jsplit), sweeps (jsplit, ns).
// Without relabelling there is only segment 0 with jsplit = ns (no trailing front).
int enqueue_segment(bmm_plan *pl, int seg, int jsplit) {
    const bmm::BigParams &b = pl->bp;
    const int ns = pl->ns;
    if (seg == 0) {
        CU(cudaMemsetAsync(pl->counts.p, 0, pl->counts.bytes, pl->stream));
        if (pl->zfreq.p) CU(cudaMemsetAsync(pl->zfreq.p, 0, pl->zfreq.bytes, pl->stream));
        if (pl->x_done.p) CU(cudaMemsetAsync(pl->x_done.p, 0, pl->x_done.bytes, pl->stream));
        if (pl->ws_rep.p) CU(cudaMemsetAsync(pl->ws_rep.p, 0, pl->ws_rep.bytes, pl->stream));
        if (pl->x_p2p && bmm::dist_p2p_begin_run(ns, pl->stream)) return fail(BMM_ERR_NCCL, bmm::dist_error());
        if (pl->x_seq.p) CU(bmm::launch_x_begin_run(pl->x_seq.as<int>(), ns, pl->stream));
        CU(bmm::launch_big_init(b, pl->stream));
        CU(bmm::launch_ws_table(b, pl->stream));
        if (pl->relabel) CU(bmm::launch_grid_identity_perm(b.K, b.K, pl->perm_cur.as<int>(), pl->stream));
        for (int j = 1; j < jsplit; ++j) { TRY(sweep_front(pl, j)); TRY(sweep_back(pl, j)); }
        if (jsplit < ns) TRY(sweep_front(pl, jsplit));
    } else {
        TRY(sweep_back(pl, jsplit));
        for (int j = jsplit + 1; j < ns; ++j) { TRY(sweep_front(pl, j)); TRY(sweep_back(pl, j)); }
        if (pl->fused_relabel) {
            TRY(join_assign(pl));
            TRY(relabel_pass(pl, ns));      // the last sweep's Q update, Q back in row-major form
            CU(bmm::launch_grid_theta_rel(b.K, b.P, pl->S, pl->theta_out.as<double>(), pl->perm_out.as<int>(),
                                          pl->theta_rel_out.as<double>(), pl->sm_count, pl->stream));
        }
    }
    return BMM_OK;
}

// Run one segment through its CUDA graph (captured on first use).  Falls back to plain launches if the capture
// or the instantiation is refused.
int run_segment_big(bmm_plan *pl, int seg, int jsplit) {
    if (pl->use_graph && !pl->gexec[seg]) {
        const unsigned long long l0 = bmm::g_launches;
        cudaError_t e = cudaStreamBeginCapture(pl->stream, cudaStreamCaptureModeRelaxed);
        if (e == cudaSuccess) {
            pl->capturing = true;
            const int rc = enqueue_segment(pl, seg, jsplit);
            pl->capturing = false;
            cudaGraph_t g = nullptr;
            e = cudaStreamEndCapture(pl->stream, &g);
            if (rc == BMM_OK && e == cudaSuccess && g) e = cudaGraphInstantiate(&pl->gexec[seg], g, 0);
            else if (e == cudaSuccess) e = cudaErrorUnknown;
            if (g) cudaGraphDestroy(g);
            if (rc != BMM_OK && rc != BMM_ERR_CUDA) return rc;     // a real (non-capture) error: report it
        }
        if (e != cudaSuccess || !pl->gexec[seg]) {
            cudaGetLastError();
            pl->gexec[seg] = nullptr;
            pl->use_graph = false;
            bmm::g_launches = l0;
        } else {
            pl->glaunches[seg] = bmm::g_launches - l0;
            bmm::g_launches = l0;
        }
    }
    if (pl->use_graph && pl->gexec[seg]) {
        CU(cudaGraphLaunch(pl->gexec[seg], pl->stream));
        bmm::g_launches += pl->glaunches[seg];
        return BMM_OK;
    }
    return enqueue_segment(pl, seg, jsplit);
}

// All sweeps of the grid path on the plan's stream.
int run_big(bmm_plan *pl) {
    const int ns = pl->ns, burnin = pl->a.burnin;
    if (pl->sharded && bmm::dist_world() < 2) return fail(BMM_ERR_NCCL, "N-sharded run needs bmm_dist_init with world > 1");
    while (pl->sweep_ev.size() < (size_t)2 * ns) {
        cudaEvent_t e;
        CU(cudaEventCreate(&e));
        pl->sweep_ev.push_back(e);
    }
    while (pl->fused_relabel && pl->relabel_ev.size() < (size_t)2 * ns) {
        cudaEvent_t e;
        CU(cudaEventCreate(&e));
        pl->relabel_ev.push_back(e);
    }
    if (!pl->relabel) return run_segment_big(pl, 0, ns);
    TRY(run_segment_big(pl, 0, burnin - 1));
    TRY(batch_relabel_big(pl));
    return run_segment_big(pl, 1, burnin - 1);
}

int create_collapsed(bmm_plan *pl, const bmm_init *init) {
    const bmm_args &a = pl->a;
    const int N = pl->N, P = pl->P, K = pl->K, C = pl->C, ns = pl->ns, S = pl->S;
    const bool dp = pl->sampler == BMM_SAMPLER_DP;
    std::vector<uint32_t> bits;
    int W;
    TRY(pack_rows(a.X, N, P, bits, W));
    pl->W = W; pl->U = N;
    TRY(upload(pl->xbits, bits.data(), bits.size()));
    std::vector<double> lB(N + 1), lG(N + 1), lBG(N + 1), lN(N + 1);
    for (int n = 0; n <= N; ++n) {
        lB[n] = std::log(a.beta + n); lG[n] = std::log(a.gamma + n); lBG[n] = std::log(a.beta + a.gamma + n);
        lN[n] = std::log((double)n);
    }
    TRY(upload(pl->logN, lN.data(), lN.size()));
    TRY(upload(pl->logB, lB.data(), lB.size()));
    TRY(upload(pl->logG, lG.data(), lG.size()));
    TRY(upload(pl->logBG, lBG.data(), lBG.size()));
    // product form of the DP conditional (kern_collapsed.cu): the factors reach (beta or gamma + N)^P and (beta + gamma)^-P ... (.. + N)^-P
    const bool prod_ok = dp && !a.replay && !getenv("BMM_DP_LOGFORM") &&
                         P * std::fabs(std::log10(a.beta + a.gamma + N)) < 250.0 && P * std::fabs(std::log10(a.beta + a.gamma)) < 250.0;
    if (prod_ok) {
        std::vector<double> r(N + 1);
        for (int n = 0; n <= N; ++n) r[n] = std::pow(a.beta + a.gamma + n, -(double)P);
        TRY(upload(pl->rBGP, r.data(), r.size()));
    }
    const size_t P1 = P + 1, NK = (size_t)N * K, KP = (size_t)K * P;
    std::vector<uint8_t> zc((size_t)C * N, 0xFF);
    std::vector<int> cnt((size_t)C * K * P1, 0);
    CU(pl->zhist.alloc((size_t)C * ns * N));
    if (!dp) {
        std::vector<uint8_t> row0((size_t)N);
        for (int c = 0; c < C; ++c) {
            for (int i = 0; i < N; ++i) {
                int z = init->z[(size_t)c * N + i];
                if (z < 1 || z > K) return fail(BMM_ERR_INVALID, "initialK must be in 1..K");
                zc[(size_t)c * N + i] = (uint8_t)(z - 1);
                row0[i] = (uint8_t)z;
                int *cc = &cnt[((size_t)c * K + (z - 1)) * P1];
                cc[P]++;
                for (int d = 0; d < P; ++d) cc[d] += (bits[(size_t)i * W + (d >> 5)] >> (d & 31)) & 1;
            }
            // z_out.row(0) = initialK (collapsed_gibbs.cpp:46)
            CU(cudaMemcpy(pl->zhist.as<uint8_t>() + (size_t)c * ns * N, row0.data(), N, cudaMemcpyHostToDevice));
        }
    } else {
        std::vector<int> used((size_t)C * (K + 2), 0);
        std::vector<uint8_t> fr((size_t)C * K, 1);
        TRY(upload(pl->dp_used, used.data(), used.size()));
        TRY(upload(pl->dp_free, fr.data(), fr.size()));
        if (a.flags & BMM_FLAG_PROBE_PROBS) CU(pl->kactive.alloc((size_t)C * ns * 4));
    }
    TRY(upload(pl->z_cur, zc.data(), zc.size()));
    TRY(upload(pl->cnt, cnt.data(), cnt.size()));
    std::vector<double> al(C, a.alpha == 0 ? 1.0 : a.alpha);
    TRY(upload(pl->alpha_cur, al.data(), al.size()));
    if (pl->relabel) {
        CU(pl->Q.alloc((size_t)C * NK * 8));
        CU(pl->logQ.alloc((size_t)C * NK * 8));
        CU(pl->probs_sample.alloc((size_t)C * NK * 8));
        CU(pl->cube.alloc((size_t)C * a.burnrelabel * NK * 8));
        CU(pl->logp.alloc((size_t)C * a.burnrelabel * NK * 8));
        CU(pl->sb_perm.alloc((size_t)C * a.burnrelabel * K * 4));
        CU(pl->sb_cost.alloc((size_t)C * a.burnrelabel * K * K * 8));
        CU(pl->sb_ws.alloc((size_t)C * a.burnrelabel * bmm::assign_ws_bytes(K)));
        CU(pl->perm_out.alloc((size_t)C * S * K * 4));
        CU(pl->theta_rel_out.alloc((size_t)C * KP * S * 8));
        if (K * K > bmm::COST_SMEM_MAX) CU(pl->cost_g.alloc((size_t)C * K * K * 8));
    }
    CU(pl->assign_ws.alloc((size_t)C * bmm::assign_ws_bytes(K)));
    CU(pl->status.alloc((size_t)C * 4));
    CU(pl->theta_out.alloc((size_t)C * KP * S * 8));
    CU(pl->alpha_out.alloc((size_t)C * S * 8));
    if (a.flags & BMM_FLAG_PROBE_PROBS) CU(pl->probs_out.alloc((size_t)C * ns * NK * 8));
    if (a.replay) {
        const bmm_replay *r = a.replay;
        TRY(upload(pl->ru, r->u, (size_t)C * ns * N * r->u_slots));
        if (r->alpha) TRY(upload(pl->ralpha, r->alpha, (size_t)C * ns));
    }
    bmm::CollapsedParams &q = pl->cp;
    q.N = N; q.P = P; q.K = K; q.W = W;
    q.nsamples = ns; q.burnin = a.burnin; q.relabel = pl->relabel; q.burnrelabel = a.burnrelabel; q.dp = dp;
    q.fp32 = a.precision == BMM_FP32; q.thin = pl->thin;
    q.alpha0 = a.alpha; q.beta = a.beta; q.gamma = a.gamma; q.a = a.a; q.b = a.b;
    q.seed = a.seed; q.chain_offset = a.chain_offset; q.flags = a.flags;
    q.xbits = pl->xbits.as<uint32_t>();
    q.logB = pl->logB.as<double>(); q.logG = pl->logG.as<double>(); q.logBG = pl->logBG.as<double>();
    q.logN = pl->logN.as<double>(); q.rBGP = pl->rBGP.as<double>();
    q.z_cur = pl->z_cur.as<uint8_t>(); q.cnt = pl->cnt.as<int>(); q.alpha_cur = pl->alpha_cur.as<double>();
    q.dp_used = pl->dp_used.as<int>(); q.dp_free = pl->dp_free.as<uint8_t>();
    q.Q = pl->Q.as<double>(); q.logQ = pl->logQ.as<double>(); q.probs_sample = pl->probs_sample.as<double>();
    q.cube = pl->cube.as<double>(); q.assign_ws = pl->assign_ws.as<char>(); q.status = pl->status.as<int>();
    q.cost_g = pl->cost_g.as<double>();
    q.zhist = pl->zhist.as<uint8_t>(); q.theta_out = pl->theta_out.as<double>(); q.theta_rel_out = pl->theta_rel_out.as<double>();
    q.alpha_out = pl->alpha_out.as<double>(); q.perm_out = pl->perm_out.as<int>();
    q.probs_out = pl->probs_out.as<double>(); q.kactive_out = pl->kactive.as<int>();
    q.ru = pl->ru.as<double>(); q.ru_slots = a.replay ? a.replay->u_slots : 0; q.ralpha = pl->ralpha.as<double>();
    if (bmm::collapsed_smem_bytes(q) > 200 * 1024)
        return fail(BMM_ERR_UNSUPPORTED, "N*P (bit-packed data + allocations) too large for the shared memory of the chain-per-warp collapsed kernel");
    return BMM_OK;
}

// Threads per chain block of the uncollapsed chain-per-block kernel.  The per-sweep work of one chain is
// narrow (32 unique rows, 18 parameters), so the block size is about latency hiding: two warps let the
// relabelling step run beside the parameter draws, and the 64-thread entry point is capped at 144
// registers so that seven blocks (1024 chains on 148 SMs) stay resident.  Measured on C2 per step:
// 32 threads 28.0 ms, 64 threads 23.3 ms (before the two-warp split: 9.5 / 9.9 / 14.4 ms per 300 sweeps for
// 32 / 64 / 128).  BMM_FULL_THREADS overrides (tuning).
int full_threads(int n_chains) {
    if (const char *e = getenv("BMM_FULL_THREADS")) {
        int t = atoi(e);
        if (t == 32 || t == 64 || t == 128) return t;
    }
    return n_chains >= 512 ? 64 : 128;
}

// Kernel of the last chain-per-block launch of the uncollapsed samplers (bmm_debug_chain_kernel): 1 full_chain_kernel,
// 2 chain_sweep_kernel.
int g_chain_kernel = 0;

int run_segment(bmm_plan *pl, int j0, int j1) {
    if (j1 <= j0) return BMM_OK;
    if (pl->sampler == BMM_SAMPLER_FULL || pl->sampler == BMM_SAMPLER_STICKBREAKING) {
        pl->fp.j_begin = j0; pl->fp.j_end = j1;
        const int threads = full_threads(pl->C);
        // the specialised sweep kernel where it applies; BMM_CHAIN_KERNEL=generic keeps full_chain_kernel (tests, A/B)
        const char *force = getenv("BMM_CHAIN_KERNEL");
        const bool sweep = !(force && !strcmp(force, "generic")) && bmm::chain_sweep_supported(pl->fp, threads);
        g_chain_kernel = sweep ? 2 : 1;
        if (sweep) CU(bmm::launch_chain_sweep(pl->fp, pl->C, threads, pl->stream));
        else CU(bmm::launch_full(pl->fp, pl->C, threads, pl->stream));
    } else {
        pl->cp.j_begin = j0; pl->cp.j_end = j1;
        CU(bmm::launch_collapsed(pl->cp, pl->C, pl->stream));
    }
    return BMM_OK;
}

// Pinned staging for the byte-wide allocation history: two buffers, so the DMA of chunk c+1 overlaps
// the host-side widening of chunk c.
struct Staging {
    uint8_t *buf[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    size_t bytes = 0;
};
std::mutex g_stage_m;                 // one download at a time per process: the staging buffers are shared
std::map<int, Staging> g_stages;      // per device (events belong to the device they were created on)

// Bytes [0, n) of `src` -- one sweep segment (L of the S kept sweeps, starting at s_off) of `rows` (chain, observation)
// pairs -- through the pinned staging buffers into the int32 matrices.  perm == NULL: dst_zo receives the widened bytes.
// perm != NULL: the bytes are z_original; dst_zo receives them and dst_z the relabelled allocations (either may be NULL).
// The copies run on `cs`, which the caller has ordered after the kernels that produce `src`.
int fetch_widen(bmm_plan *pl, cudaStream_t cs, const uint8_t *src, size_t n, int L, int s_off, const int32_t *perm,
                int32_t *dst_z, int32_t *dst_zo) {
    if ((!dst_z && !dst_zo) || !src || n == 0) return BMM_OK;
    const size_t CH = (size_t)32 << 20;
    std::lock_guard<std::mutex> lock(g_stage_m);
    Staging &g_stage = g_stages[pl->a.device];
    if (!g_stage.buf[0]) {
        for (int b = 0; b < 2; ++b) {
            CU(cudaHostAlloc((void **)&g_stage.buf[b], CH, cudaHostAllocDefault));
            CU(cudaEventCreateWithFlags(&g_stage.ev[b], cudaEventDisableTiming));
        }
        g_stage.bytes = CH;
    }
    static const int threads = [] {
        const char *e = getenv("BMM_FETCH_THREADS");
        // three quarters of the online CPUs, at most 12: measured on the 16-vCPU GPU boxes (C2, 7.4 GB of int32
        // output per step) 4 / 8 / 12 / 16 workers take 87 / 61 / 52 / 57 ms; 16 oversubscribe the cores the DMA
        // completion path needs.  With one process per GPU (torchrun sets LOCAL_WORLD_SIZE) the cores are
        // shared between the ranks.
        int ranks = 1;
        if (const char *lw = getenv("LOCAL_WORLD_SIZE")) ranks = atoi(lw) > 0 ? atoi(lw) : 1;
        long hw = sysconf(_SC_NPROCESSORS_ONLN);
        if ((long)std::thread::hardware_concurrency() > hw) hw = (long)std::thread::hardware_concurrency();
        int t = e ? atoi(e) : (int)(hw * 3 / (4 * ranks));
        return t < 1 ? 1 : (t > 12 && !e ? 12 : (t > 32 ? 32 : t));
    }();
    const size_t nch = (n + CH - 1) / CH;
    auto issue = [&](size_t c) -> cudaError_t {
        const size_t lo = c * CH, cnt = lo + CH <= n ? CH : n - lo;
        cudaError_t e = cudaMemcpyAsync(g_stage.buf[c & 1], src + lo, cnt, cudaMemcpyDeviceToHost, cs);
        g_fetch_bytes += cnt;
        return e != cudaSuccess ? e : cudaEventRecord(g_stage.ev[c & 1], cs);
    };
    CU(issue(0));
    for (size_t c = 0; c < nch; ++c) {
        if (c + 1 < nch) CU(issue(c + 1));
        CU(cudaEventSynchronize(g_stage.ev[c & 1]));
        const size_t lo = c * CH, cnt = lo + CH <= n ? CH : n - lo;
        if (L == pl->S && !perm) bmm_widen_u8_i32(g_stage.buf[c & 1], dst_zo + lo, cnt, threads);
        else bmm_widen_runs_u8_i32(g_stage.buf[c & 1], lo, cnt, L, pl->S, s_off, pl->N, pl->K, perm, dst_z, dst_zo, threads);
    }
    return BMM_OK;
}

// Record the initial chain state (called once, at the end of bmm_plan_create).
int snapshot_state(bmm_plan *pl) {
    std::vector<DevBuf *> live;
    if (pl->grid_path) live = {&pl->theta_cur, &pl->pi_cur, &pl->alpha_cur};
    else if (pl->sampler == BMM_SAMPLER_FULL || pl->sampler == BMM_SAMPLER_STICKBREAKING)
        live = {&pl->theta_cur, &pl->pi_cur, &pl->alpha_cur};
    else live = {&pl->z_cur, &pl->cnt, &pl->alpha_cur, &pl->dp_used, &pl->dp_free};
    for (DevBuf *b : live) {
        if (!b->p || !b->bytes) continue;
        std::unique_ptr<bmm_plan::Snap> sn(new bmm_plan::Snap());
        sn->live = b;
        CU(sn->copy.alloc(b->bytes, false));
        CU(cudaMemcpy(sn->copy.p, b->p, b->bytes, cudaMemcpyDeviceToDevice));
        pl->snaps.push_back(std::move(sn));
    }
    // zero-initialised in the reference and not fully overwritten by a run: the relabelling stores (slices before
    // sweep 1 when burnrelabel > burnin; the DP sampler writes only the columns of live labels and never clears
    // probs_sample, collapsed_gibbs_dp.cpp:91-92,195-199), the DP theta histories (:77-78), the status words
    pl->zero_at_run = {&pl->status, &pl->cube, &pl->cube_f, &pl->probs_sample, &pl->Q, &pl->logQ};
    if (pl->grid_path) {          // warm-start state of the assignment solver: every run starts cold, like the first
        pl->zero_at_run.push_back(&pl->assign_ws);
        pl->zero_at_run.push_back(&pl->sb_vws);
    }
    if (pl->sampler == BMM_SAMPLER_DP) {
        pl->zero_at_run.push_back(&pl->theta_out);
        pl->zero_at_run.push_back(&pl->theta_rel_out);
        pl->zero_at_run.push_back(&pl->kactive);
    }
    return BMM_OK;
}

int restore_state(bmm_plan *pl) {
    for (auto &sn : pl->snaps)
        CU(cudaMemcpyAsync(sn->live->p, sn->copy.p, sn->copy.bytes, cudaMemcpyDeviceToDevice, pl->stream));
    for (DevBuf *b : pl->zero_at_run)
        if (b->p && b->bytes) CU(cudaMemsetAsync(b->p, 0, b->bytes, pl->stream));
    return BMM_OK;
}

int first_status(bmm_plan *pl, std::vector<int> &st) {
    st.assign(pl->C, 0);
    CU(cudaMemcpy(st.data(), pl->status.p, (size_t)pl->C * 4, cudaMemcpyDeviceToHost));
    return BMM_OK;
}

}  // namespace

namespace bmm {
void set_last_error(const char *msg) { g_err = msg ? msg : ""; }
}

#pragma GCC visibility push(default)
extern "C" {

const char *bmm_last_error(void) { return g_err.c_str(); }
const char *bmm_version(void) { return "bmm-mcmc_b200 0.1 (sm_100a)"; }
uint64_t bmm_launch_count(void) { return bmm::g_launches; }
uint64_t bmm_fetch_bytes(void) { return g_fetch_bytes; }

int bmm_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int bmm_plan_create(int32_t sampler, const bmm_args *args, const bmm_init *init, bmm_plan **plan) {
    if (!plan) return fail(BMM_ERR_INVALID, "plan is NULL");
    *plan = nullptr;
    if (sampler < 0 || sampler > 3) return fail(BMM_ERR_INVALID, "unknown sampler");
    TRY(check_args(sampler, args, init));
    if (bmm_device_count() <= args->device) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    CU(cudaSetDevice(args->device));
    bmm_plan *pl = new bmm_plan();
    pl->sampler = sampler; pl->a = *args;
    pl->C = args->n_chains < 1 ? 1 : args->n_chains;
    pl->N = args->N; pl->P = args->P; pl->K = args->K; pl->ns = args->nsamples;
    pl->thin = args->thin > 1 ? args->thin : 1;
    pl->S = bmm::hist_count(args->nsamples, args->burnin, pl->thin);
    pl->relabel = args->relabel != 0; pl->replay = args->replay != nullptr;
    int rc = BMM_OK;
    cudaError_t e = cudaStreamCreateWithFlags(&pl->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&pl->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&pl->ev1);
    if (e == cudaSuccess) e = cudaEventCreate(&pl->evk0);
    if (e == cudaSuccess) e = cudaEventCreate(&pl->evk1);
    for (auto &ev : pl->evs) if (e == cudaSuccess) e = cudaEventCreate(&ev);
    if (e != cudaSuccess) rc = fail(BMM_ERR_CUDA, cudaGetErrorString(e));
    const bool uncollapsed = sampler == BMM_SAMPLER_FULL || sampler == BMM_SAMPLER_STICKBREAKING;
    if (uncollapsed)
        pl->grid_path = (args->flags & (BMM_FLAG_GRID_PATH | BMM_FLAG_X_PACKED)) || args->n_global > args->N ||
                        (pl->C == 1 && (args->N >= 32768 || (size_t)args->K * args->P > 4096));
    if (!rc) rc = pl->grid_path ? create_big(pl, init) : (uncollapsed ? create_full(pl, init) : create_collapsed(pl, init));
    if (!rc) {
        // R-layout allocation histories are produced on the device by the finalize kernel
        // int32 output larger than a few MB: keep bytes on the device and widen on the host (fetch_z)
        const size_t zelems = (size_t)pl->C * pl->S * pl->N;
        // Widening on the host moves an eighth (a quarter without relabelling) of the bytes over PCIe; the int32 matrices are
        // then written by the host cores.  With several ranks per host the ranks share those cores (fetch_widen divides the
        // workers by LOCAL_WORLD_SIZE) and, above all, the host's memory: measured on the 8-GPU box (C2, 14.7 GB of int32 per
        // rank and step, 118 GB per step over all ranks) the call takes 899 ms with host widening on 3 or 4 workers per rank
        // against 1356 ms with device widening and int32 DMA -- either way ~100-140 GB/s into host memory is the limit, and
        // the device-side widening costs 6 ms of the 37 ms run as well.  (Round 1 measured the opposite with 12 workers per
        // rank oversubscribing the 32 cores.)  BMM_FETCH_WIDEN=0 keeps the int32 DMA path.
        const char *wenv = getenv("BMM_FETCH_WIDEN");
        const bool widen_dflt = wenv ? wenv[0] != '0' : true;
        const bool widen = !(args->flags & BMM_FLAG_COMPACT_Z) && zelems >= ((size_t)8 << 20) && widen_dflt;
        pl->deb = ((args->flags & BMM_FLAG_COMPACT_Z) || widen) ? 1 : 4;
        // z = perm[z_original] (full_gibbs.cpp:171-174): with host widening the relabelled matrix is derived on the host from
        // the original one and the permutations instead of crossing PCIe as well (BMM_FETCH_DERIVE=0 ships both)
        const char *denv = getenv("BMM_FETCH_DERIVE");
        pl->derive_z = widen && pl->relabel && !pl->grid_path && pl->K <= 16 && !(denv && denv[0] == '0');
        const size_t eb = (size_t)pl->deb;
        const bool no_z = pl->grid_path && (args->flags & BMM_FLAG_NO_Z_HISTORY);
        cudaError_t e2 = cudaSuccess;
        pl->seg_slot = {0, pl->S};
        if (widen && !pl->grid_path) {
            // Sweep segments, on 64-slot boundaries, at least 256 slots each.  Measured on C2 (S = 1800, run 37 ms) in one
            // session: 1 / 2 / 3 segments 159-170 / 155-159 / 144-146 ms per call; a boundary that does not fall on a cache
            // line of the output (S * 4 bytes per run need not be a multiple of 64) costs two partial-line streaming stores
            // per (chain, observation) run, which is what limits the count.
            const char *senv = getenv("BMM_FETCH_SEGMENTS");
            int nseg = senv ? atoi(senv) : (pl->S >= 1024 ? 4 : pl->S / 256);
            if (pl->thin != 1 || nseg < 1) nseg = 1;
            pl->seg_slot.assign(1, 0);
            // a short first segment (half a share) lets the host start while as much of the run as possible is still ahead
            for (int g = 1; g < nseg; ++g) {
                const long long num = 2LL * g - 1, den = 2LL * nseg - 1;
                const int b = (int)((((long long)pl->S * num) / den) & ~63LL);
                if (b > pl->seg_slot.back() && b < pl->S) pl->seg_slot.push_back(b);
            }
            pl->seg_slot.push_back(pl->S);
            if (e2 == cudaSuccess) e2 = cudaStreamCreateWithFlags(&pl->copy_stream, cudaStreamNonBlocking);
            for (size_t g = 0; g + 1 < pl->seg_slot.size() && e2 == cudaSuccess; ++g) {
                cudaEvent_t ev;
                e2 = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
                if (e2 == cudaSuccess) pl->seg_ev.push_back(ev);
            }
        }
        if (e2 == cudaSuccess && !no_z) e2 = pl->z_orig.alloc(zelems * eb, false);
        if (e2 == cudaSuccess && pl->relabel && !pl->derive_z) e2 = pl->z_rel.alloc(zelems * eb, false);
        if (e2 != cudaSuccess) rc = fail(BMM_ERR_CUDA, std::string("history allocation: ") + cudaGetErrorString(e2));
    }
    if (!rc) rc = snapshot_state(pl);
    if (!rc) { cudaError_t e3 = cudaDeviceSynchronize(); if (e3 != cudaSuccess) rc = fail(BMM_ERR_CUDA, cudaGetErrorString(e3)); }
    if (rc) { cudaDeviceSynchronize(); delete pl; return rc; }
    *plan = pl;
    return BMM_OK;
}

int bmm_plan_run(bmm_plan *pl) {
    if (!pl) return fail(BMM_ERR_INVALID, "plan is NULL");
    CU(cudaSetDevice(pl->a.device));
    const int ns = pl->ns, burnin = pl->a.burnin;
    if (pl->runs++ > 0) TRY(restore_state(pl));   // the first run starts from the freshly created state
    CU(cudaEventRecord(pl->ev0, pl->stream));
    CU(cudaEventRecord(pl->evk0, pl->stream));
    CU(cudaEventRecord(pl->evs[0], pl->stream));
    if (pl->grid_path) {
        TRY(run_big(pl));
        CU(cudaEventRecord(pl->evs[1], pl->stream));
        CU(cudaEventRecord(pl->evs[2], pl->stream));
    } else {
        if (pl->relabel) {
            TRY(run_segment(pl, 1, burnin));
            CU(cudaEventRecord(pl->evs[1], pl->stream));
            const bool full = pl->sampler == BMM_SAMPLER_FULL || pl->sampler == BMM_SAMPLER_STICKBREAKING;
            CU(bmm::launch_stephens_batch(pl->C, pl->U, pl->K, pl->a.burnrelabel, full ? pl->wt.as<int>() : nullptr,
                                          pl->cube.as<double>(), pl->logp.as<double>(), pl->Q.as<double>(),
                                          pl->logQ.as<double>(), pl->sb_perm.as<int>(), pl->sb_cost.as<double>(),
                                          pl->sb_ws.as<char>(), pl->stream, (pl->a.flags & BMM_FLAG_STEPHENS_FIXED) ? 1 : 0));
            CU(cudaEventRecord(pl->evs[2], pl->stream));
        } else {
            CU(cudaEventRecord(pl->evs[1], pl->stream));
            CU(cudaEventRecord(pl->evs[2], pl->stream));
        }
        // the kept sweeps, one launch per download segment (a single one unless the host widens, see bmm_plan_create);
        // a finished segment of the host-widened chains is laid out at once so that its download can start
        const size_t nseg = pl->seg_slot.size() - 1;
        int j0 = pl->relabel ? burnin : 1;
        for (size_t g = 0; g < nseg; ++g) {
            const int j1 = g + 1 == nseg ? ns : burnin + pl->seg_slot[g + 1];      // segments exist only with thin == 1
            TRY(run_segment(pl, j0, j1));
            j0 = j1 > j0 ? j1 : j0;
            if (nseg > 1) {
                if (pl->z_orig.p) {
                    const size_t off = (size_t)pl->C * pl->N * pl->seg_slot[g];
                    CU(bmm::launch_finalize_z(pl->C, pl->N, ns, burnin, pl->thin, pl->K, pl->zhist.as<uint8_t>(),
                                              pl->relabel ? pl->perm_out.as<int>() : nullptr, pl->z_orig.as<uint8_t>() + off,
                                              pl->z_rel.p ? pl->z_rel.as<uint8_t>() + off : nullptr, 1, pl->stream,
                                              pl->seg_slot[g], pl->seg_slot[g + 1]));
                }
                CU(cudaEventRecord(pl->seg_ev[g], pl->stream));
            }
        }
    }
    CU(cudaEventRecord(pl->evs[3], pl->stream));
    CU(cudaEventRecord(pl->evk1, pl->stream));
    const int eb = pl->deb;
    const bool split = !pl->grid_path && pl->seg_slot.size() > 2;
    if (pl->z_orig.p && !split)
        CU(bmm::launch_finalize_z(pl->C, pl->N, ns, burnin, pl->thin, pl->K, pl->zhist.as<uint8_t>(),
                                  pl->relabel ? pl->perm_out.as<int>() : nullptr, pl->z_orig.p,
                                  pl->relabel && !pl->derive_z ? pl->z_rel.p : nullptr, eb, pl->stream));
    CU(cudaEventRecord(pl->evs[4], pl->stream));
    CU(cudaEventRecord(pl->ev1, pl->stream));
    pl->ran = true;
    return BMM_OK;
}

int bmm_plan_sync(bmm_plan *pl) {
    if (!pl) return fail(BMM_ERR_INVALID, "plan is NULL");
    CU(cudaStreamSynchronize(pl->stream));
    return BMM_OK;
}

int bmm_plan_elapsed_ms(bmm_plan *pl, float *total_ms, float *sampler_kernel_ms) {
    if (!pl || !pl->ran) return fail(BMM_ERR_INVALID, "plan has not run");
    CU(cudaEventSynchronize(pl->ev1));
    if (total_ms) CU(cudaEventElapsedTime(total_ms, pl->ev0, pl->ev1));
    if (sampler_kernel_ms) CU(cudaEventElapsedTime(sampler_kernel_ms, pl->evk0, pl->evk1));
    return BMM_OK;
}

int bmm_plan_kernel_ms(bmm_plan *pl, float ms_out[4]) {
    if (!pl || !pl->ran || !ms_out) return fail(BMM_ERR_INVALID, "plan has not run");
    CU(cudaEventSynchronize(pl->evs[4]));
    for (int i = 0; i < 4; ++i) CU(cudaEventElapsedTime(&ms_out[i], pl->evs[i], pl->evs[i + 1]));
    if (pl->grid_path) {
        // [0] sum of the sweep kernels, [1] everything else in the sweep loop (parameter kernels,
        // all-reduce), [2] 0, [3] history layout conversion
        // (the sweep kernels bracketed by events -- every ev_stride-th -- scaled to all ns - 1 of them)
        float sweeps = 0.f, total = ms_out[0];
        int timed = 0;
        for (int j = 1; j < pl->ns; ++j) {
            if (pl->ev_stride <= 0 || (j % pl->ev_stride) != 0) continue;
            float t = 0.f;
            CU(cudaEventElapsedTime(&t, pl->sweep_ev[2 * j], pl->sweep_ev[2 * j + 1]));
            sweeps += t;
            ++timed;
        }
        sweeps = timed ? sweeps * (float)(pl->ns - 1) / (float)timed : 0.f;
        // [2]: the single-pass relabelling kernels of sweeps burnin .. ns - 1 (same scaling)
        float rel = 0.f;
        int rtimed = 0;
        const int nrel = pl->ns - pl->a.burnin;
        if (pl->fused_relabel && pl->relabel_ev.size() >= (size_t)2 * pl->ns)
            for (int j = pl->a.burnin; j < pl->ns; ++j) {
                if (pl->ev_stride <= 0 || (j % pl->ev_stride) != 0) continue;
                float t = 0.f;
                CU(cudaEventElapsedTime(&t, pl->relabel_ev[2 * j], pl->relabel_ev[2 * j + 1]));
                rel += t;
                ++rtimed;
            }
        rel = rtimed ? rel * (float)nrel / (float)rtimed : 0.f;
        ms_out[0] = sweeps; ms_out[1] = total - sweeps - rel; ms_out[2] = rel;
    }
    return BMM_OK;
}

int bmm_host_alloc(uint64_t bytes, void **ptr_out) {
    if (!ptr_out) return fail(BMM_ERR_INVALID, "ptr_out is NULL");
    *ptr_out = nullptr;
    if (bmm_device_count() < 1) return fail(BMM_ERR_CUDA, "no CUDA device");
    CU(cudaHostAlloc(ptr_out, bytes ? bytes : 1, cudaHostAllocDefault));
    return BMM_OK;
}

int bmm_release_cache(void) {
    g_cache.release();
    return BMM_OK;
}

int bmm_host_free(void *ptr) {
    if (ptr) CU(cudaFreeHost(ptr));
    return BMM_OK;
}

int bmm_plan_fetch(bmm_plan *pl, bmm_out *out) {
    if (!pl || !out) return fail(BMM_ERR_INVALID, "plan/out is NULL");
    if (!pl->ran) return fail(BMM_ERR_INVALID, "plan has not run");
    CU(cudaSetDevice(pl->a.device));
    g_fetch_bytes = 0;
    const size_t C = pl->C, S = pl->S, N = pl->N, K = pl->K, P = pl->P, ns = pl->ns;
    const size_t eb = (pl->a.flags & BMM_FLAG_COMPACT_Z) ? 1 : 4;
    if (pl->deb == 1 && eb == 4 && !pl->grid_path) {
        // Host-widened chain paths: the allocation matrices are downloaded segment by segment while the later sweeps are
        // still running on the plan's stream.
        const size_t nseg = pl->seg_slot.size() - 1;
        std::vector<int32_t> perm_host;
        int32_t *perm = nullptr;
        if (pl->derive_z) {
            perm = out->permutations;
            if (!perm) { perm_host.resize(C * S * K); perm = perm_host.data(); }
        }
        int32_t *dz = pl->relabel ? out->z : nullptr, *dzo = pl->relabel ? out->z_original : out->z;
        for (size_t g = 0; g < nseg; ++g) {
            const int s0 = pl->seg_slot[g], L = pl->seg_slot[g + 1] - s0;
            CU(cudaStreamWaitEvent(pl->copy_stream, nseg > 1 ? pl->seg_ev[g] : pl->ev1, 0));
            if (perm) {   // this segment's permutations: columns [s0, s0 + L) of every (chain, label) row of S entries
                CU(cudaMemcpy2DAsync(perm + s0, S * 4, pl->perm_out.as<int>() + s0, S * 4, (size_t)L * 4, C * K, cudaMemcpyDeviceToHost,
                                     pl->copy_stream));
                g_fetch_bytes += C * K * (size_t)L * 4;
                CU(cudaStreamSynchronize(pl->copy_stream));
            }
            const size_t off = C * N * (size_t)s0, n = C * N * (size_t)L;
            if (pl->derive_z) TRY(fetch_widen(pl, pl->copy_stream, pl->z_orig.as<uint8_t>() + off, n, L, s0, perm, dz, dzo));
            else {
                if (pl->relabel) TRY(fetch_widen(pl, pl->copy_stream, pl->z_rel.as<uint8_t>() + off, n, L, s0, nullptr, nullptr, dz));
                TRY(fetch_widen(pl, pl->copy_stream, pl->z_orig.as<uint8_t>() + off, n, L, s0, nullptr, nullptr, dzo));
            }
        }
    }
    CU(cudaStreamSynchronize(pl->stream));
    auto d2h = [&](void *dst, const DevBuf &src, size_t bytes) -> cudaError_t {
        if (!dst || !src.p || bytes == 0) return cudaSuccess;
        g_fetch_bytes += bytes;
        return cudaMemcpyAsync(dst, src.p, bytes, cudaMemcpyDeviceToHost, pl->stream);
    };
    CU(d2h(out->pi, pl->pi_out, C * S * K * 8));
    CU(d2h(out->alpha, pl->alpha_out, C * S * 8));
    const bool widen = pl->deb == 1 && eb == 4;
    if (pl->relabel) {
        CU(d2h(out->permutations, pl->perm_out, C * S * K * 4));
        if (!widen) CU(d2h(out->z, pl->z_rel, C * S * N * eb));
        CU(d2h(out->theta, pl->theta_rel_out, C * K * P * S * 8));
        if (!widen) CU(d2h(out->z_original, pl->z_orig, C * S * N * eb));
        CU(d2h(out->theta_original, pl->theta_out, C * K * P * S * 8));
    } else {
        if (!widen) CU(d2h(out->z, pl->z_orig, C * S * N * eb));
        CU(d2h(out->theta, pl->theta_out, C * K * P * S * 8));
    }
    if (widen && pl->grid_path) {     // one chain over the whole GPU: a single segment, after the run
        if (pl->relabel) {
            TRY(fetch_widen(pl, pl->stream, pl->z_rel.as<uint8_t>(), C * S * N, (int)S, 0, nullptr, nullptr, out->z));
            TRY(fetch_widen(pl, pl->stream, pl->z_orig.as<uint8_t>(), C * S * N, (int)S, 0, nullptr, nullptr, out->z_original));
        } else {
            TRY(fetch_widen(pl, pl->stream, pl->z_orig.as<uint8_t>(), C * S * N, (int)S, 0, nullptr, nullptr, out->z));
        }
    }
    CU(d2h(out->probs, pl->probs_out, C * ns * N * K * 8));
    CU(d2h(out->loglik, pl->loglik_out, C * ns * N * K * 8));
    std::vector<float> qf_host;
    std::vector<uint8_t> zlast_host;
    if (out->Q_final && pl->relabel && pl->grid_path) {
        qf_host.resize(N * K);
        CU(cudaMemcpyAsync(qf_host.data(), pl->Qf.p, N * K * 4, cudaMemcpyDeviceToHost, pl->stream));
    } else if (out->Q_final && pl->relabel) {
        if (pl->U == pl->N && pl->sampler >= BMM_SAMPLER_COLLAPSED) {
            CU(d2h(out->Q_final, pl->Q, C * N * K * 8));
        } else {
            if (!pl->Qexp.p) CU(pl->Qexp.alloc(C * N * K * 8, false));
            CU(bmm::launch_expand_rows((int)C, (int)N, pl->U, (int)K, pl->rowid.as<int>(), pl->Q.as<double>(),
                                       pl->Qexp.as<double>(), pl->stream));
            CU(d2h(out->Q_final, pl->Qexp, C * N * K * 8));
        }
    }
    CU(d2h(out->counts, pl->counts_out, ns * (K + K * P) * 4));
    std::vector<uint8_t> zlast_chain;
    if (!pl->grid_path) {
        // posterior summaries of the chain-parallel paths (f2): allocation counts over the kept sweeps (relabelled when
        // relabel), last sweep's allocations -- what a caller keeps instead of the S x N histories
        if (out->z_freq) {
            if (!pl->zhist.p) return fail(BMM_ERR_INVALID, "z_freq needs the allocation history on the device");
            if (!pl->zfreq.p) CU(pl->zfreq.alloc(C * N * K * 4, false));
            CU(bmm::launch_chain_zfreq((int)C, (int)N, (int)ns, pl->a.burnin, pl->thin, (int)K, pl->zhist.as<uint8_t>(),
                                       pl->relabel ? pl->perm_out.as<int>() : nullptr, pl->zfreq.as<unsigned>(), pl->stream));
            CU(d2h(out->z_freq, pl->zfreq, C * N * K * 4));
        }
        if (out->z_last && pl->zhist.p) {
            zlast_chain.resize(C * N);
            CU(cudaMemcpy2DAsync(zlast_chain.data(), N, pl->zhist.as<uint8_t>() + (ns - 1) * N, ns * N, N, C,
                                 cudaMemcpyDeviceToHost, pl->stream));
        }
    }
    if (pl->grid_path) {
        CU(d2h(out->z_freq, pl->zfreq, N * K * 4));
        if (out->z_last && pl->zhist.p) {   // bytes -> int32 through a small staging vector
            zlast_host.resize(N);
            const uint8_t *src = pl->zhist.as<uint8_t>() + (pl->bp.keep_history ? (ns - 1) * N : 0);
            CU(cudaMemcpyAsync(zlast_host.data(), src, N, cudaMemcpyDeviceToHost, pl->stream));
        }
    }
    CU(d2h(out->status, pl->status, C * 4));
    CU(cudaStreamSynchronize(pl->stream));
    for (size_t i = 0; i < zlast_host.size(); ++i) out->z_last[i] = (int32_t)zlast_host[i];
    for (size_t i = 0; i < zlast_chain.size(); ++i) out->z_last[i] = (int32_t)zlast_chain[i];
    if (!qf_host.empty())   // grid path keeps Q as row-major float; the ABI returns N x K column-major double
        for (size_t i = 0; i < N; ++i)
            for (size_t k = 0; k < K; ++k) out->Q_final[i + N * k] = (double)qf_host[i * K + k];
    std::vector<int> st;
    TRY(first_status(pl, st));
    for (size_t c = 0; c < C; ++c)
        if (st[c]) {
            char buf[160];
            snprintf(buf, sizeof buf, "chain %zu stopped with status %d%s", c, st[c],
                     st[c] == BMM_ERR_NO_FREE_CLUSTER ? " (Error: have no free clusters, need to create one.)" : "");
            return fail(st[c], buf);
        }
    return BMM_OK;
}

int bmm_plan_destroy(bmm_plan *pl) {
    if (pl) {
        // the blocks go back to the free list on delete: nothing of this plan may still be running on them
        cudaSetDevice(pl->a.device);
        if (pl->stream) cudaStreamSynchronize(pl->stream);
        if (pl->copy_stream) cudaStreamSynchronize(pl->copy_stream);
        delete pl;
    }
    return BMM_OK;
}

static int run_once(int sampler, const bmm_args *args, const bmm_init *init, bmm_out *out) {
    if (!out) return fail(BMM_ERR_INVALID, "out is NULL");
    if (!args) return fail(BMM_ERR_INVALID, "args is NULL");
    bmm_args a = *args;
    if (out->probs) a.flags |= BMM_FLAG_PROBE_PROBS;
    if (out->loglik) a.flags |= BMM_FLAG_PROBE_LOGLIK;
    if (out->counts) a.flags |= BMM_FLAG_PROBE_COUNTS;
    if (out->z_freq) a.flags |= BMM_FLAG_PROBE_ZFREQ;
    bmm_plan *pl = nullptr;
    static const bool trace = getenv("BMM_TRACE") != nullptr;   // wall-clock phases of the one-shot call on stderr
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = now();
    int rc = bmm_plan_create(sampler, &a, init, &pl);
    if (rc) return rc;
    const double t1 = now();
    rc = bmm_plan_run(pl);
    if (!rc && trace) rc = bmm_plan_sync(pl);
    const double t2 = now();
    if (!rc) rc = bmm_plan_fetch(pl, out);
    const double t3 = now();
    bmm_plan_destroy(pl);
    if (trace) fprintf(stderr, "bmm trace: create %.1f ms, run %.1f ms, fetch %.1f ms, destroy %.1f ms\n", t1 - t0, t2 - t1, t3 - t2, now() - t3);
    return rc;
}

int bmm_gibbs_full(const bmm_args *args, const bmm_init *init, bmm_out *out) { return run_once(BMM_SAMPLER_FULL, args, init, out); }
int bmm_gibbs_stickbreaking(const bmm_args *args, const bmm_init *init, bmm_out *out) { return run_once(BMM_SAMPLER_STICKBREAKING, args, init, out); }
int bmm_gibbs_collapsed(const bmm_args *args, const bmm_init *init, bmm_out *out) { return run_once(BMM_SAMPLER_COLLAPSED, args, init, out); }
int bmm_gibbs_dp(const bmm_args *args, bmm_out *out) { return run_once(BMM_SAMPLER_DP, args, nullptr, out); }

// ---- helpers --------------------------------------------------------------------------------------
int bmm_stephens_batch(int32_t N, int32_t K, int32_t M, const double *p, double *q, int32_t *perm_MxK) {
    return bmm_stephens_batch_ex(N, K, M, p, q, perm_MxK, 0);
}

int bmm_stephens_batch_ex(int32_t N, int32_t K, int32_t M, const double *p, double *q, int32_t *perm_MxK, uint32_t flags) {
    if (!p || !q || N < 1 || K < 1 || K > 255 || M < 1) return fail(BMM_ERR_INVALID, "bad stephens_batch arguments");
    if (bmm_device_count() < 1) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    const size_t NK = (size_t)N * K;
    DevBuf cube, logp, Q, logQ, perm, cost, ws;
    TRY(upload(cube, p, NK * M));
    CU(logp.alloc(NK * M * 8)); CU(Q.alloc(NK * 8)); CU(logQ.alloc(NK * 8));
    CU(perm.alloc((size_t)M * K * 4)); CU(cost.alloc((size_t)M * K * K * 8)); CU(ws.alloc((size_t)M * bmm::assign_ws_bytes(K)));
    CU(bmm::launch_stephens_batch(1, N, K, M, nullptr, cube.as<double>(), logp.as<double>(), Q.as<double>(),
                                  logQ.as<double>(), perm.as<int>(), cost.as<double>(), ws.as<char>(), 0,
                                  (flags & BMM_FLAG_STEPHENS_FIXED) ? 1 : 0));
    CU(cudaMemcpy(q, Q.p, NK * 8, cudaMemcpyDeviceToHost));
    if (perm_MxK) CU(cudaMemcpy(perm_MxK, perm.p, (size_t)M * K * 4, cudaMemcpyDeviceToHost));
    return BMM_OK;
}

int bmm_stephens_online(int32_t N, int32_t K, const double *q, const double *p, int32_t sample_num,
                        int32_t *perm, double *q_new, double *cost) {
    return bmm_stephens_online_ex(N, K, q, p, sample_num, perm, q_new, cost, 0);
}

int bmm_stephens_online_ex(int32_t N, int32_t K, const double *q, const double *p, int32_t sample_num,
                           int32_t *perm, double *q_new, double *cost, uint32_t flags) {
    if (!p || !q || !perm || !q_new || N < 1 || K < 1 || K > 255) return fail(BMM_ERR_INVALID, "bad stephens_online arguments");
    if (bmm_device_count() < 1) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    const size_t NK = (size_t)N * K;
    DevBuf Q, logQ, pd, cd, pm, ws;
    TRY(upload(Q, q, NK)); TRY(upload(pd, p, NK));
    CU(logQ.alloc(NK * 8)); CU(cd.alloc((size_t)K * K * 8)); CU(pm.alloc((size_t)K * 4)); CU(ws.alloc(bmm::assign_ws_bytes(K)));
    CU(bmm::launch_stephens_online(N, K, Q.as<double>(), logQ.as<double>(), pd.as<double>(), sample_num,
                                   cd.as<double>(), pm.as<int>(), ws.as<char>(), 0, (flags & BMM_FLAG_STEPHENS_FIXED) ? 1 : 0));
    CU(cudaMemcpy(q_new, Q.p, NK * 8, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(perm, pm.p, (size_t)K * 4, cudaMemcpyDeviceToHost));
    if (cost) CU(cudaMemcpy(cost, cd.p, (size_t)K * K * 8, cudaMemcpyDeviceToHost));
    return BMM_OK;
}

int bmm_assign(int32_t K, int32_t batch, const double *cost, int32_t *solution) {
    if (!cost || !solution || K < 1 || K > 255 || batch < 1) return fail(BMM_ERR_INVALID, "bad assign arguments");
    if (bmm_device_count() < 1) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    DevBuf cd, sd, ws;
    TRY(upload(cd, cost, (size_t)batch * K * K));
    CU(sd.alloc((size_t)batch * K * K * 4)); CU(ws.alloc((size_t)batch * bmm::assign_ws_bytes(K)));
    CU(bmm::launch_assign(K, batch, cd.as<double>(), sd.as<int>(), ws.as<char>(), 0));
    CU(cudaMemcpy(solution, sd.p, (size_t)batch * K * K * 4, cudaMemcpyDeviceToHost));
    return BMM_OK;
}

// Assignment with the grid path's solver (enumeration for K <= 5, warp-parallel Jonker-Volgenant above):
// cost is K x K column-major (rows = reference labels), perm[c] = row assigned to column c.
int bmm_assign_warp(int32_t K, const double *cost, int32_t *perm) {
    if (!cost || !perm || K < 1 || K > 255) return fail(BMM_ERR_INVALID, "bad assign arguments");
    if (bmm_device_count() < 1) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    // the kernel computes s_l - G(k,l): feed G = -cost, s = 0
    std::vector<double> acc((size_t)K * K + K, 0.0);
    for (size_t e = 0; e < (size_t)K * K; ++e) acc[e] = -cost[e];
    DevBuf ad, pd, ws;
    TRY(upload(ad, acc.data(), acc.size()));
    CU(pd.alloc((size_t)K * 4)); CU(ws.alloc(bmm::assign_ws_bytes(K)));
    CU(bmm::launch_grid_assign(K, ad.as<double>(), ws.as<char>(), pd.as<int>(), nullptr, 1, 0));
    CU(cudaMemcpy(perm, pd.p, (size_t)K * 4, cudaMemcpyDeviceToHost));
    return BMM_OK;
}

// Cost contraction of the grid path's relabelling on host matrices (row-major float N x K):
// out[k + K*l] = sum_i log q_ik * p_il, out[K*K + l] = sum_i p_il^2 (or p log p when use_logp).
int bmm_grid_cost(int64_t N, int32_t K, const float *p, const float *q, int32_t use_logp, int32_t tensor, double *out) {
    if (!p || !q || !out || N < 1 || K < 1 || K > 128) return fail(BMM_ERR_INVALID, "bad grid_cost arguments");
    if (bmm_device_count() < 1) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    if (tensor && !bmm::grid_cost_tc_supported(N, K)) return fail(BMM_ERR_INVALID, "tensor cost kernel needs 8 <= K <= 128, K % 8 == 0");
    DevBuf pd, qd, od, sd;
    TRY(upload(pd, p, (size_t)N * K));
    TRY(upload(qd, q, (size_t)N * K));
    CU(od.alloc(((size_t)K * K + K) * 8)); CU(sd.alloc(16));
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    CU(bmm::launch_grid_cost(N, K, pd.as<float>(), qd.as<float>(), use_logp, od.as<double>(), sms, 0, tensor, sd.as<int>()));
    int st[2] = {0, 0};
    CU(cudaMemcpy(st, sd.p, 8, cudaMemcpyDeviceToHost));
    if (st[0]) return fail(st[0], "grid cost kernel failed");
    CU(cudaMemcpy(out, od.p, ((size_t)K * K + K) * 8, cudaMemcpyDeviceToHost));
    return BMM_OK;
}

/* diagnostic: %globaltimer stamps (ns) of CTA 0 of the last tensor-sweep launch, see kern_big_ws.cu */
int bmm_debug_ws_trace(uint64_t out[32]) {
    if (!out) return fail(BMM_ERR_INVALID, "out is NULL");
    CU(cudaDeviceSynchronize());
    unsigned long long t[32];
    CU(bmm::ws_trace_read(t));
    CU(bmm::upd_trace_read(t + 16));
    for (int i = 0; i < 32; ++i) out[i] = t[i];
    return BMM_OK;
}

int bmm_debug_chain_kernel(void) { return g_chain_kernel; }

int bmm_debug_chain_phases(uint64_t *out, int64_t n) {
    if (!out || n < 0) return fail(BMM_ERR_INVALID, "out is NULL or n < 0");
    CU(cudaDeviceSynchronize());
    bool supported = false;
    CU(bmm::chain_phase_read((unsigned long long *)out, (size_t)n, &supported));
    if (!supported) return fail(BMM_ERR_UNSUPPORTED, "built without BMM_CHAIN_PHASE_CLOCKS");
    return BMM_OK;
}

/* diagnostic: per CTA of the last tensor-sweep launch, out[2b] = (entry ns << 10) | SM id, out[2b + 1] = counts flushed ns */
int bmm_debug_ws_cta(uint64_t out[320]) {
    if (!out) return fail(BMM_ERR_INVALID, "out is NULL");
    CU(cudaDeviceSynchronize());
    unsigned long long t[320];
    CU(bmm::ws_cta_read(t));
    for (int i = 0; i < 320; ++i) out[i] = t[i];
    return BMM_OK;
}

int bmm_rdirichlet(int32_t K, const double *alpha_m, uint64_t seed, double *out) {
    if (!alpha_m || !out || K < 1 || K > 4096) return fail(BMM_ERR_INVALID, "bad rdirichlet arguments");
    if (bmm_device_count() < 1) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    DevBuf ad, od;
    TRY(upload(ad, alpha_m, (size_t)K));
    CU(od.alloc((size_t)K * 8));
    CU(bmm::launch_rdirichlet(K, ad.as<double>(), seed, od.as<double>(), 0));
    CU(cudaMemcpy(out, od.p, (size_t)K * 8, cudaMemcpyDeviceToHost));
    return BMM_OK;
}

int bmm_predictive(const int32_t *Xnew, int32_t M, int32_t P, int32_t K, int32_t S, const double *theta, const double *pi,
                   double *log_pred, double *membership) {
    if (!Xnew || !theta || !pi || !log_pred || M < 1 || P < 1 || K < 1 || K > 255 || S < 1)
        return fail(BMM_ERR_INVALID, "bad predictive arguments");
    if (bmm_device_count() < 1) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    std::vector<uint32_t> bits;
    int W;
    TRY(pack_rows(Xnew, M, P, bits, W));
    DevBuf xb, th, pd, tab, lp, mem;
    TRY(upload(xb, bits.data(), bits.size()));
    TRY(upload(th, theta, (size_t)K * P * S));
    TRY(upload(pd, pi, (size_t)S * K));
    CU(tab.alloc((size_t)S * K * (2 * P + 1) * 8, false));
    CU(lp.alloc((size_t)M * 8, false));
    if (membership) CU(mem.alloc((size_t)M * K * 8));
    CU(bmm::launch_predict(M, P, W, K, S, xb.as<uint32_t>(), th.as<double>(), pd.as<double>(), tab.as<double>(), lp.as<double>(),
                           membership ? mem.as<double>() : nullptr, 0));
    CU(cudaMemcpy(log_pred, lp.p, (size_t)M * 8, cudaMemcpyDeviceToHost));
    if (membership) CU(cudaMemcpy(membership, mem.p, (size_t)M * K * 8, cudaMemcpyDeviceToHost));
    return BMM_OK;
}

// WAIC and the log-likelihood trace of C chains x S kept draws (kern_predict.cu, kern_waic_tc.cu).  The rows are
// de-duplicated first; the tcgen05 kernel takes shapes it covers once there are enough distinct rows to give every SM
// tiles of its own (below that the fp64 kernel's split of the draws over warps is the faster, DESIGN.md section 4).
static thread_local float g_waic_ms = 0.f;
static thread_local int32_t g_waic_tensor = 0;
static constexpr int WAIC_TC_MIN_TILES_PER_SM = 1;

// X as bit-packed rows [N][W]: packs an int32 N x P column-major 0/1 matrix, or copies BMM_FLAG_X_PACKED rows with the
// bits beyond P cleared (they are not part of the row)
static int input_rows(const void *X, int N, int P, uint32_t flags, std::vector<uint32_t> &bits, int &W) {
    W = (P + 31) / 32;
    if (flags & BMM_FLAG_X_PACKED) {
        const uint32_t *xb = (const uint32_t *)X, tail = (P & 31) ? (1u << (P & 31)) - 1u : ~0u;
        bits.assign(xb, xb + (size_t)N * W);
        for (int i = 0; i < N; ++i) bits[(size_t)i * W + W - 1] &= tail;
        return BMM_OK;
    }
    return pack_rows((const int32_t *)X, N, P, bits, W);
}

// pi [C][S x K cm] -> D x K cm over the chain-major draws g = c S + s (theta [C][K x P x S] already is K x P x D)
static std::vector<double> pooled_pi(const double *pi, int C, int S, int K) {
    const size_t D = (size_t)C * S;
    std::vector<double> pid(D * K);
    for (int c = 0; c < C; ++c)
        for (int k = 0; k < K; ++k)
            for (int s = 0; s < S; ++s) pid[(size_t)c * S + s + D * k] = pi[(size_t)c * S * K + s + (size_t)S * k];
    return pid;
}

// the tcgen05 kernels take the shapes they cover once there are U distinct rows enough to give every SM a 128-row tile
static bool waic_tensor_path(uint32_t flags, int K, int P, int U, int sms) {
    const char *force = getenv("BMM_WAIC_TENSOR");   // tests: the tcgen05 kernel at any number of distinct rows
    return !(flags & BMM_FLAG_NO_TENSOR) && bmm::waic_tc_supported(K, P) &&
           ((force && force[0] == '1') || (long long)(U + 127) / 128 >= (long long)WAIC_TC_MIN_TILES_PER_SM * sms);
}

int bmm_waic(const void *X, int32_t N, int32_t P, int32_t K, int32_t S, int32_t C, const double *theta, const double *pi,
             uint32_t flags, int32_t device, double *loglik, double *lppd, double *p_waic, double *chain_lppd,
             double *chain_p_waic) {
    if (!X || !theta || !pi || N < 1 || P < 1 || K < 1 || K > 255 || S < 1 || C < 1)
        return fail(BMM_ERR_INVALID, "bad waic arguments");
    const long long D = (long long)C * S;
    if (D < 2) return fail(BMM_ERR_INVALID, "waic needs at least 2 draws (C * S >= 2)");
    if (D > 0x7FFFFFFFLL) return fail(BMM_ERR_INVALID, "waic: C * S too large");
    if (device < 0 || bmm_device_count() <= device) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    std::vector<uint32_t> bits;
    int W;
    TRY(input_rows(X, N, P, flags, bits, W));
    std::vector<int> rowid, wt;
    std::vector<uint32_t> rowbits;
    dedup_rows(bits.data(), N, W, rowid, wt, rowbits);
    std::vector<uint32_t>().swap(bits);
    const int U = (int)wt.size();
    const std::vector<double> pid = pooled_pi(pi, C, S, K);
    CU(cudaSetDevice(device));
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    const int ntc = (U + 127) / 128;
    const bool tensor = waic_tensor_path(flags, K, P, U, sms);
    DevBuf rb, wd, th, pd, tab, img, bias, stat, tpart, lp, pw, cv, ll, ct, sd;
    TRY(upload(rb, rowbits.data(), rowbits.size()));
    TRY(upload(wd, wt.data(), wt.size()));
    TRY(upload(th, theta, (size_t)D * K * P));
    TRY(upload(pd, pid.data(), pid.size()));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    struct EvPair { cudaEvent_t a, b; ~EvPair() { cudaEventDestroy(a); cudaEventDestroy(b); } } evs{e0, e1};
    int Q;
    long long G;
    CU(cudaEventRecord(e0, 0));
    if (tensor) {
        Q = 1;
        G = 4LL * ntc;
        CU(img.alloc((size_t)D * bmm::waic_tc_img_bytes(P), false));
        CU(bias.alloc((size_t)D * 32 * 4, false));
        CU(sd.alloc(4));
        CU(stat.alloc((size_t)C * U * bmm::WAIC_STAT * 8, false));
        CU(tpart.alloc((size_t)D * G * 8, false));
        CU(bmm::launch_waic_tc_tables(K, P, D, th.as<double>(), pd.as<double>(), img.as<unsigned char>(), bias.as<float>(), 0));
        CU(bmm::launch_waic_tc(U, P, W, K, S, C, rb.as<uint32_t>(), wd.as<int>(), img.as<unsigned char>(), bias.as<float>(),
                               stat.as<double>(), tpart.as<double>(), sd.as<int>(), sms, 0));
    } else {
        const int nt = (U + 31) / 32;
        const int q0 = bmm::waic_fp64_slices(nt, C, S), SL = (S + q0 - 1) / q0;
        Q = (S + SL - 1) / SL;                               // slices of SL = ceil(S / Q) draws, none empty
        G = nt;
        CU(tab.alloc((size_t)D * K * (2 * P + 1) * 8, false));
        CU(stat.alloc((size_t)C * Q * U * bmm::WAIC_STAT * 8, false));
        CU(tpart.alloc((size_t)D * G * 8, false));
        CU(bmm::launch_predict_tables(K, P, (int)D, th.as<double>(), pd.as<double>(), tab.as<double>(), 0));
        CU(bmm::launch_waic_fp64(U, P, W, K, S, C, Q, rb.as<uint32_t>(), wd.as<int>(), tab.as<double>(), stat.as<double>(),
                                 tpart.as<double>(), 0));
    }
    CU(lp.alloc((size_t)U * 8, false));
    CU(pw.alloc((size_t)U * 8, false));
    CU(cv.alloc((size_t)2 * C * U * 8, false));
    CU(ll.alloc((size_t)D * 8, false));
    CU(ct.alloc((size_t)2 * C * 8, false));
    CU(bmm::launch_waic_merge(U, C, S, Q, wd.as<int>(), stat.as<double>(), G, tpart.as<double>(), lp.as<double>(),
                              pw.as<double>(), cv.as<double>(), ll.as<double>(), ct.as<double>(), 0));
    CU(cudaEventRecord(e1, 0));
    CU(cudaEventSynchronize(e1));
    CU(cudaEventElapsedTime(&g_waic_ms, e0, e1));
    g_waic_tensor = tensor;
    if (tensor) {
        int st = 0;
        CU(cudaMemcpy(&st, sd.p, 4, cudaMemcpyDeviceToHost));
        if (st) return fail(st, "waic tensor kernel: an mbarrier wait timed out");
    }
    if (loglik) CU(cudaMemcpy(loglik, ll.p, (size_t)D * 8, cudaMemcpyDeviceToHost));
    if (chain_lppd) CU(cudaMemcpy(chain_lppd, ct.p, (size_t)C * 8, cudaMemcpyDeviceToHost));
    if (chain_p_waic) CU(cudaMemcpy(chain_p_waic, ct.as<double>() + C, (size_t)C * 8, cudaMemcpyDeviceToHost));
    if (lppd || p_waic) {
        std::vector<double> ul(U), up(U);
        CU(cudaMemcpy(ul.data(), lp.p, (size_t)U * 8, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(up.data(), pw.p, (size_t)U * 8, cudaMemcpyDeviceToHost));
        for (int i = 0; i < N; ++i) {
            if (lppd) lppd[i] = ul[rowid[i]];
            if (p_waic) p_waic[i] = up[rowid[i]];
        }
    }
    return BMM_OK;
}

int bmm_waic_kernel_ms(float *ms, int32_t *tensor) {
    if (!ms || !tensor) return fail(BMM_ERR_INVALID, "ms / tensor is NULL");
    *ms = g_waic_ms;
    *tensor = g_waic_tensor;
    return BMM_OK;
}

// PSIS-LOO and the log-likelihood matrix (kern_loo.cu).  Both read l[g, u] of the distinct rows from one device buffer
// that holds a chunk of rows at a time: the smaller of LOGLIK_CHUNK_CAP bytes and a quarter of the free device memory
// (the whole C4 matrix would take 7.2 GB).  BMM_LOO_CHUNK_ROWS caps the rows of a chunk (tests: many chunks).
static thread_local float g_loo_ms = 0.f;
static thread_local int32_t g_loo_tensor = 0;
static constexpr size_t LOGLIK_CHUNK_CAP = (size_t)2 << 30;

// The draws' tables and the matrix producer: L [D][uc] <- l of distinct rows [u0, u0 + uc), fp64 or tcgen05 kernel
struct LoglikMat {
    long long D = 0;
    int U = 0, W = 0, P = 0, K = 0, sms = 0, rows = 0;   // rows: the chunk size
    bool tensor = false;
    DevBuf rb, th, pd, tab, img, bias, sd, L;

    int init(const std::vector<uint32_t> &rowbits, int U_, int W_, int P_, int K_, int S, int C, const double *theta,
             const double *pi, uint32_t flags, int device) {
        U = U_; W = W_; P = P_; K = K_;
        D = (long long)C * S;
        CU(cudaSetDevice(device));
        CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
        tensor = waic_tensor_path(flags, K, P, U, sms);
        const std::vector<double> pid = pooled_pi(pi, C, S, K);
        TRY(upload(rb, rowbits.data(), rowbits.size()));
        TRY(upload(th, theta, (size_t)D * K * P));
        TRY(upload(pd, pid.data(), pid.size()));
        size_t fre = 0, tot = 0;
        CU(cudaMemGetInfo(&fre, &tot));
        long long r = (long long)(std::min(LOGLIK_CHUNK_CAP, fre / 4) / ((size_t)D * 8));
        if (const char *e = getenv("BMM_LOO_CHUNK_ROWS")) { const long long c = atoll(e); if (c > 0 && r > c) r = c; }
        rows = (int)std::max(1LL, std::min(r, (long long)U));
        CU(L.alloc((size_t)rows * D * 8, false));
        if (tensor) {
            CU(img.alloc((size_t)D * bmm::waic_tc_img_bytes(P), false));
            CU(bias.alloc((size_t)D * 32 * 4, false));
            CU(sd.alloc(4));
        } else {
            CU(tab.alloc((size_t)D * K * (2 * P + 1) * 8, false));
        }
        return BMM_OK;
    }
    int tables() {
        if (tensor)
            CU(bmm::launch_waic_tc_tables(K, P, D, th.as<double>(), pd.as<double>(), img.as<unsigned char>(), bias.as<float>(), 0));
        else
            CU(bmm::launch_predict_tables(K, P, (int)D, th.as<double>(), pd.as<double>(), tab.as<double>(), 0));
        return BMM_OK;
    }
    int produce(int u0, int n) {
        const uint32_t *xb = rb.as<uint32_t>() + (size_t)u0 * W;
        if (tensor)
            CU(bmm::launch_loglik_tc(n, P, W, D, xb, img.as<unsigned char>(), bias.as<float>(), L.as<double>(), sd.as<int>(), sms, 0));
        else
            CU(bmm::launch_loglik_fp64(n, P, W, K, D, xb, tab.as<double>(), L.as<double>(), 0));
        return BMM_OK;
    }
    int status() {
        if (!tensor) return BMM_OK;
        int st = 0;
        CU(cudaMemcpy(&st, sd.p, 4, cudaMemcpyDeviceToHost));
        return st ? fail(st, "log-likelihood tensor kernel: an mbarrier wait timed out") : BMM_OK;
    }
};

static int loglik_args(const void *X, int N, int P, int K, int S, int C, const double *theta, const double *pi,
                       const char *what) {
    if (!X || !theta || !pi || N < 1 || P < 1 || K < 1 || K > 255 || S < 1 || C < 1)
        return fail(BMM_ERR_INVALID, std::string("bad ") + what + " arguments");
    const long long D = (long long)C * S;
    if (D < 2) return fail(BMM_ERR_INVALID, std::string(what) + " needs at least 2 draws (C * S >= 2)");
    if (D > 0x7FFFFFFFLL) return fail(BMM_ERR_INVALID, std::string(what) + ": C * S too large");
    return BMM_OK;
}

int bmm_loo(const void *X, int32_t N, int32_t P, int32_t K, int32_t S, int32_t C, const double *theta, const double *pi,
            const double *r_eff, uint32_t flags, int32_t device, double *elpd_loo, double *lpd, double *pareto_k,
            double *n_eff) {
    TRY(loglik_args(X, N, P, K, S, C, theta, pi, "loo"));
    const long long D = (long long)C * S;
    // tail length of each observation, loo's n_pareto_tail; no smoothing below 5
    std::vector<int> Mi(N);
    for (int i = 0; i < N; ++i) {
        const double re = r_eff ? r_eff[i] : 1.0;
        if (!(re > 0.0) || !std::isfinite(re)) return fail(BMM_ERR_INVALID, "loo: r_eff must be finite and > 0");
        const double m = std::min(std::ceil(0.2 * (double)D), std::ceil(3 * std::sqrt((double)D / re)));
        if (m > bmm::LOO_MAX_TAIL) {
            char msg[256];
            snprintf(msg, sizeof msg, "loo: the Pareto tail of %lld draws at r_eff = %g has %.0f draws; at most %d are supported "
                     "(D <= 29826161 at r_eff = 1)", D, re, m, bmm::LOO_MAX_TAIL);
            return fail(BMM_ERR_INVALID, msg);
        }
        Mi[i] = (int)m;
    }
    if (device < 0 || bmm_device_count() <= device) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    std::vector<uint32_t> bits;
    int W;
    TRY(input_rows(X, N, P, flags, bits, W));
    // de-duplicate on (row, M): r_eff changes only the tail length, and n_eff's r_eff factor is applied per observation
    std::vector<uint32_t> keys((size_t)N * (W + 1));
    for (int i = 0; i < N; ++i) {
        std::memcpy(&keys[(size_t)i * (W + 1)], &bits[(size_t)i * W], (size_t)W * 4);
        keys[(size_t)i * (W + 1) + W] = (uint32_t)Mi[i];
    }
    std::vector<uint32_t>().swap(bits);
    std::vector<int> rowid, wt;
    std::vector<uint32_t> urows;
    dedup_rows(keys.data(), N, W + 1, rowid, wt, urows);
    std::vector<uint32_t>().swap(keys);
    const int U = (int)wt.size();
    std::vector<uint32_t> rowbits((size_t)U * W);
    std::vector<int> Mu(U);
    for (int u = 0; u < U; ++u) {
        std::memcpy(&rowbits[(size_t)u * W], &urows[(size_t)u * (W + 1)], (size_t)W * 4);
        Mu[u] = (int)urows[(size_t)u * (W + 1) + W];
    }
    LoglikMat lm;
    TRY(lm.init(rowbits, U, W, P, K, S, C, theta, pi, flags, device));
    // per chunk: the long-tail rows (chunk-local index, M, offset into the chunk's tail storage) and the widest tails
    const int rows = lm.rows, nch = (U + rows - 1) / rows;
    std::vector<int> lrow, lM, l0(nch + 1), short_m(nch, 0), long_m(nch, 0);
    std::vector<long long> ltoff;
    long long max_tail = 0;
    int max_nlong = 0;
    for (int c = 0; c < nch; ++c) {
        l0[c] = (int)lrow.size();
        long long toff = 0;
        for (int u = c * rows; u < std::min(U, (c + 1) * rows); ++u) {
            if (Mu[u] > bmm::LOO_SHORT_MAX_M) {
                lrow.push_back(u - c * rows);
                lM.push_back(Mu[u]);
                ltoff.push_back(toff);
                toff += Mu[u];
                long_m[c] = std::max(long_m[c], Mu[u]);
            } else {
                short_m[c] = std::max(short_m[c], Mu[u]);
            }
        }
        max_tail = std::max(max_tail, toff);
        max_nlong = std::max(max_nlong, (int)lrow.size() - l0[c]);
    }
    l0[nch] = (int)lrow.size();
    const int nblk = bmm::loo_long_blocks(D);
    DevBuf dM, dlrow, dlM, dltoff, sel, hist, tail, part, out;
    TRY(upload(dM, Mu.data(), Mu.size()));
    if (max_nlong) {
        TRY(upload(dlrow, lrow.data(), lrow.size()));
        TRY(upload(dlM, lM.data(), lM.size()));
        TRY(upload(dltoff, ltoff.data(), ltoff.size()));
        CU(sel.alloc((size_t)max_nlong * sizeof(bmm::LooSel), false));
        CU(hist.alloc((size_t)max_nlong * 256 * 4, false));
        CU(tail.alloc((size_t)max_tail * 8, false));
        CU(part.alloc((size_t)max_nlong * nblk * 4 * 8, false));
    }
    CU(out.alloc((size_t)4 * U * 8, false));
    double *dE = out.as<double>(), *dL = dE + U, *dK = dL + U, *dN = dK + U;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    struct EvPair { cudaEvent_t a, b; ~EvPair() { cudaEventDestroy(a); cudaEventDestroy(b); } } evs{e0, e1};
    CU(cudaEventRecord(e0, 0));
    TRY(lm.tables());
    for (int c = 0; c < nch; ++c) {
        const int u0 = c * rows, n = std::min(rows, U - u0), nl = l0[c + 1] - l0[c];
        TRY(lm.produce(u0, n));
        const double *L = lm.L.as<double>();
        CU(bmm::launch_loo_short(n, D, short_m[c], L, dM.as<int>() + u0, dE + u0, dL + u0, dK + u0, dN + u0, 0));
        if (nl)
            CU(bmm::launch_loo_long(n, D, nl, long_m[c], L, dlrow.as<int>() + l0[c], dlM.as<int>() + l0[c],
                                    dltoff.as<long long>() + l0[c], sel.as<bmm::LooSel>(), hist.as<unsigned>(),
                                    tail.as<double>(), part.as<double>(), dE + u0, dL + u0, dK + u0, dN + u0, 0));
    }
    CU(cudaEventRecord(e1, 0));
    CU(cudaEventSynchronize(e1));
    CU(cudaEventElapsedTime(&g_loo_ms, e0, e1));
    g_loo_tensor = lm.tensor;
    TRY(lm.status());
    std::vector<double> res((size_t)4 * U);
    CU(cudaMemcpy(res.data(), out.p, res.size() * 8, cudaMemcpyDeviceToHost));
    for (int i = 0; i < N; ++i) {
        const int u = rowid[i];
        if (elpd_loo) elpd_loo[i] = res[u];
        if (lpd) lpd[i] = res[(size_t)U + u];
        if (pareto_k) pareto_k[i] = res[(size_t)2 * U + u];
        if (n_eff) n_eff[i] = res[(size_t)3 * U + u] * (r_eff ? r_eff[i] : 1.0);
    }
    return BMM_OK;
}

int bmm_loo_kernel_ms(float *ms, int32_t *tensor) {
    if (!ms || !tensor) return fail(BMM_ERR_INVALID, "ms / tensor is NULL");
    *ms = g_loo_ms;
    *tensor = g_loo_tensor;
    return BMM_OK;
}

int bmm_loglik_matrix(const void *X, int32_t N, int32_t P, int32_t K, int32_t S, int32_t C, const double *theta,
                      const double *pi, uint32_t flags, int32_t device, double *out) {
    TRY(loglik_args(X, N, P, K, S, C, theta, pi, "loglik_matrix"));
    if (!out) return fail(BMM_ERR_INVALID, "loglik_matrix: out is NULL");
    if (device < 0 || bmm_device_count() <= device) return fail(BMM_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    const long long D = (long long)C * S;
    std::vector<uint32_t> bits;
    int W;
    TRY(input_rows(X, N, P, flags, bits, W));
    std::vector<int> rowid, wt;
    std::vector<uint32_t> rowbits;
    dedup_rows(bits.data(), N, W, rowid, wt, rowbits);
    std::vector<uint32_t>().swap(bits);
    const int U = (int)wt.size();
    LoglikMat lm;
    TRY(lm.init(rowbits, U, W, P, K, S, C, theta, pi, flags, device));
    TRY(lm.tables());
    std::vector<double> h;
    for (int u0 = 0; u0 < U; u0 += lm.rows) {
        const int n = std::min(lm.rows, U - u0);
        TRY(lm.produce(u0, n));
        h.resize((size_t)n * D);
        CU(cudaMemcpy(h.data(), lm.L.p, h.size() * 8, cudaMemcpyDeviceToHost));
        TRY(lm.status());
        for (int i = 0; i < N; ++i) {
            const int u = rowid[i] - u0;
            if (u < 0 || u >= n) continue;
            double *o = out + (size_t)D * i;
            for (long long g = 0; g < D; ++g) o[g] = h[(size_t)g * n + u];
        }
    }
    return BMM_OK;
}

// One uncollapsed z-sweep's matrices at a given state: a 2-sample replay run whose "recorded"
// parameters are the caller's (theta, pi).
int bmm_full_condprob(const int32_t *X, int32_t N, int32_t P, int32_t K, const double *theta, const double *pi,
                      int32_t precision, uint32_t flags, double *loglik, double *probs) {
    if (!X || !theta || !pi) return fail(BMM_ERR_INVALID, "bad condprob arguments");
    const size_t KP = (size_t)K * P, NK = (size_t)N * K;
    std::vector<double> rth(KP * 2), rpi((size_t)K * 2), ral(2, 1.0), ru((size_t)2 * N * std::max(K - 1, 1), 0.5);
    for (size_t e = 0; e < KP; ++e) rth[e] = rth[KP + e] = theta[e];
    for (int k = 0; k < K; ++k) rpi[2 * (size_t)k] = rpi[2 * (size_t)k + 1] = pi[k];  // 2 x K cm
    bmm_replay rp{ru.data(), std::max(K - 1, 1), rpi.data(), rth.data(), ral.data()};
    bmm_args a{};
    a.X = X; a.N = N; a.P = P; a.nsamples = 2; a.K = K; a.alpha = 1.0; a.beta = 0.5; a.gamma = 0.5; a.a = 1; a.b = 1;
    a.burnin = 0; a.n_chains = 1; a.precision = precision; a.flags = flags; a.replay = &rp;
    bmm_init in{pi, theta, nullptr};
    std::vector<double> pb(probs ? NK * 2 : 0), lb(loglik ? NK * 2 : 0);
    bmm_out o{};
    o.probs = probs ? pb.data() : nullptr;
    o.loglik = loglik ? lb.data() : nullptr;
    int rc = run_once(BMM_SAMPLER_FULL, &a, &in, &o);
    if (rc) return rc;
    if (probs) std::copy(pb.begin() + NK, pb.end(), probs);
    if (loglik) std::copy(lb.begin() + NK, lb.end(), loglik);
    return BMM_OK;
}

}  // extern "C"
#pragma GCC visibility pop
