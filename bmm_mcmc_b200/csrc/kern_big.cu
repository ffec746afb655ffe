// Uncollapsed samplers for ONE chain over many observations (BASELINE configs C4 / C5): the z-sweep is
// data-parallel over observations, so the whole GPU (and, N-sharded, several GPUs) works on one
// sweep.  Replaces, per sweep,
//   z-sweep               /root/reference/src/full_gibbs.cpp:87-157, stickbreaking.cpp:70-140
//   sufficient statistics full_gibbs.cpp:182-200, stickbreaking.cpp:164-186
//   pi / sticks / theta / alpha draws  full_gibbs.cpp:10-27,202-230, stickbreaking.cpp:187-235, utils.cpp:6-14
//
// Launch sequence per sweep j (all on one stream):
//   big_sweep_kernel   grid-wide: one observation per thread; bit-packed row -> K conditional
//                      probabilities -> categorical draw -> 1-byte allocation; counts c_k, V_kd as
//                      shared-memory histograms flushed once per block with global atomics.
//   [all-reduce]       N-sharded runs only: int32 counts summed over ranks (dist.cu).
//   big_param_kernel   theta_kd ~ Beta, gamma / stick draws, one thread per parameter (Philox keyed by
//                      parameter index, so every rank draws identical values: no broadcast).
//   big_finish_kernel  one block: pi (normalise / stick-breaking), alpha (Escobar-West), log tables for
//                      the next sweep, history rows, zeroing of the next sweep's count buffer.
//
// The per-observation Philox counter is the GLOBAL observation index, and the reduced quantities are
// integers, so the chain is bit-identical for any number of GPUs and identical to the
// chain-per-block kernel (kern_full.cu) for the same seed.
//
// Template parameter R is the type of the probability arithmetic: double follows the reference's
// operation order exactly (d-ordered log-likelihood sum, exp(log pi + loglh), running normaliser);
// float is the CUDA-core fast path (BMM_FP32).  The tensor-core path lives in kern_big_tc.cu.
#include <cstdlib>

#include "kernels.h"
#include "common.cuh"
#include "ws_table.cuh"

namespace bmm {
namespace {

constexpr int BIG_THREADS = 256;
constexpr int REPLAY_MAXK = 64;

template <typename R> __device__ __forceinline__ R exp_r(R x);
template <> __device__ __forceinline__ double exp_r<double>(double x) { return exp(x); }
template <> __device__ __forceinline__ float exp_r<float>(float x) { return __expf(x); }

template <typename R>
struct BigSmem {
    R *w1, *w0, *lpi;
    int *cnt;
};

template <typename R>
__host__ __device__ inline size_t big_layout(int K, int P, bool tables_in_smem, char *base, BigSmem<R> *s) {
    const size_t KP = (size_t)K * P;
    size_t off = 0;
    R *w1 = nullptr, *w0 = nullptr, *lpi = nullptr;
    int *cnt = nullptr;
    if (tables_in_smem) {
        w1 = (R *)(base + off); off += KP * sizeof(R);
        w0 = (R *)(base + off); off += KP * sizeof(R);
        lpi = (R *)(base + off); off += (size_t)K * sizeof(R);
        off = (off + 7) & ~(size_t)7;
        cnt = (int *)(base + off); off += (K + KP) * sizeof(int);
    }
    if (s) { s->w1 = w1; s->w0 = w0; s->lpi = lpi; s->cnt = cnt; }
    return (off + 15) & ~(size_t)15;
}

// loglh_k(x) = sum_d x_d log theta_kd + (1 - x_d) log(1 - theta_kd), summed in d order (full_gibbs.cpp:92-103)
template <typename R>
__device__ __forceinline__ R row_loglik(const uint32_t *__restrict__ xb, int P, int K, int k, const R *w1, const R *w0) {
    R ll = 0;
    for (int d0 = 0; d0 < P; d0 += 32) {
        const uint32_t word = xb[d0 >> 5];
        const int dn = min(32, P - d0);
        for (int b = 0; b < dn; ++b) {
            const int d = d0 + b;
            ll += ((word >> b) & 1u) ? w1[k + K * d] : w0[k + K * d];
        }
    }
    return ll;
}

template <typename R, bool REPLAY>
__global__ void __launch_bounds__(BIG_THREADS) big_sweep_kernel(const BigParams p, const int j) {
    extern __shared__ __align__(16) char smem_raw[];
    BigSmem<R> s;
    big_layout<R>(p.K, p.P, p.tables_in_smem, smem_raw, &s);
    const int K = p.K, P = p.P, W = p.W, KP = K * P, tid = threadIdx.x;
    int *gcnt = p.counts + (size_t)(j & 1) * (K + KP);
    const R *w1, *w0, *lpi;
    if (p.tables_in_smem) {
        for (int t = tid; t < KP; t += blockDim.x) { s.w1[t] = (R)p.w1[t]; s.w0[t] = (R)p.w0[t]; }
        for (int t = tid; t < K; t += blockDim.x) s.lpi[t] = (R)p.lpi[t];
        for (int t = tid; t < K + KP; t += blockDim.x) s.cnt[t] = 0;
        __syncthreads();
        w1 = s.w1; w0 = s.w0; lpi = s.lpi;
    } else {
        w1 = (const R *)p.w1; w0 = (const R *)p.w0; lpi = (const R *)p.lpi;  // R == double on this path
    }
    int *cnt = p.tables_in_smem ? s.cnt : gcnt;
    const bool stable = (p.flags & 1u) != 0;  // BMM_FLAG_STABLE_SOFTMAX
    const uint2 key = make_uint2((uint32_t)p.seed, (uint32_t)p.chain_offset);
    const uint32_t sid = ST_Z ^ ((uint32_t)(p.seed >> 32) << 8);
    uint8_t *zrow = p.zhist ? p.zhist + (size_t)(p.keep_history ? j : 0) * p.N_local : nullptr;

    for (long long i = (long long)blockIdx.x * blockDim.x + tid; i < p.N_local; i += (long long)gridDim.x * blockDim.x) {
        const uint32_t *xb = p.xbits + (size_t)i * W;
        const unsigned long long gi = (unsigned long long)p.row_offset + (unsigned long long)i;
        R mx = 0;
        if (stable) {
            mx = -INFINITY;
            for (int k = 0; k < K; ++k) mx = max(mx, lpi[k] + row_loglik<R>(xb, P, K, k, w1, w0));
        }
        R cum = 0;
        for (int k = 0; k < K; ++k) cum += exp_r<R>(lpi[k] + row_loglik<R>(xb, P, K, k, w1, w0) - mx);
        if (!(cum > 0) || !isfinite(cum)) *p.status = -9;  // BMM_ERR_PROB
        int z;
        if (REPLAY) {
            double pr[REPLAY_MAXK];
            for (int k = 0; k < K; ++k) pr[k] = (double)(exp_r<R>(lpi[k] + row_loglik<R>(xb, P, K, k, w1, w0) - mx) / cum);
            z = rmultinom1_replay(K, [&](int k) { return pr[k]; },
                                  p.ru + ((size_t)j * p.N_local + i) * p.ru_slots);
        } else {
            const uint4 rnd = philox4x32_10(make_uint4((uint32_t)(gi >> 2), (uint32_t)(gi >> 34), sid, (uint32_t)j), key);
            const double u = u32_unit(philox_word(rnd, (int)(gi & 3)));
            R c2 = 0;
            z = K - 1;
            for (int k = 0; k < K - 1; ++k) {
                c2 += exp_r<R>(lpi[k] + row_loglik<R>(xb, P, K, k, w1, w0) - mx) / cum;
                if (u < (double)c2) { z = k; break; }
            }
            // In float the prefix sum of the first K - 1 probabilities can fall a few ulp short of a u near 1: the draw
            // then lands on K - 1 whatever its weight.  Fall back to the last cluster with weight instead.
            if (sizeof(R) == 4 && z == K - 1)
                while (z > 0 && !(exp_r<R>(lpi[z] + row_loglik<R>(xb, P, K, z, w1, w0) - mx) > (R)0)) --z;
        }
        if (p.probs_f32) {
            for (int k = 0; k < K; ++k)
                p.probs_f32[(size_t)i * K + k] = (float)(exp_r<R>(lpi[k] + row_loglik<R>(xb, P, K, k, w1, w0) - mx) / cum);
        }
        if (p.probs_out || p.loglik_out) {
            for (int k = 0; k < K; ++k) {
                const R ll = row_loglik<R>(xb, P, K, k, w1, w0);
                if (p.loglik_out) p.loglik_out[(size_t)j * p.N_local * K + i + (size_t)p.N_local * k] = (double)ll;
                if (p.probs_out) p.probs_out[(size_t)j * p.N_local * K + i + (size_t)p.N_local * k] = (double)(exp_r<R>(lpi[k] + ll - mx) / cum);
            }
        }
        if (zrow) zrow[i] = (uint8_t)(z + 1);
        atomicAdd(&cnt[z], 1);
        for (int d0 = 0; d0 < P; d0 += 32) {
            uint32_t word = xb[d0 >> 5];
            if (P - d0 < 32) word &= (1u << (P - d0)) - 1u;
            while (word) {
                const int b = __ffs(word) - 1;
                word &= word - 1;
                atomicAdd(&cnt[K + z + K * (d0 + b)], 1);
            }
        }
    }
    if (p.tables_in_smem) {
        __syncthreads();
        for (int t = tid; t < K + KP; t += blockDim.x) {
            const int v = s.cnt[t];
            if (v) atomicAdd(&gcnt[t], v);
        }
    }
}

constexpr int UPD_THREADS = 256;

// diagnostic stamps of the update kernel (ns): per sweep parity [0] block 0 start, [1] block 0 has its counts, [2] block 0
// end, [3] last block start, [4] last block end
__device__ unsigned long long g_upd_trace[16];
__device__ __forceinline__ void upd_stamp(int j, int slot) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_upd_trace[8 * (j & 1) + slot] = t;
}

// One launch per sweep, after the z-sweep: blocks 0..K-1 own one cluster each (theta_k., its log tables and, for
// the tensor path, row k of the operand image), block K draws pi / sticks / alpha, writes the history rows and
// zeroes the next sweep's count buffer.  On an N-sharded run over peer memory every thread sums, over the ranks, the
// inbox words it needs, re-reading a word until it carries this exchange's number (kernels.h); the
// reduced values are integers, and every draw is keyed by its parameter index, so all ranks compute identical
// tables without a broadcast (full_gibbs.cpp:182-230, stickbreaking.cpp:164-235, utils.cpp:6-14).
__global__ void __launch_bounds__(UPD_THREADS) big_update_kernel(const BigParams p, const int j) {
    __shared__ double red[32];
    __shared__ double ag[4];
    __shared__ double sh_w0[128];
    __shared__ int sh_c[256];
    const int K = p.K, P = p.P, KP = K * P, ns = p.nsamples, S = hist_count(ns, p.burnin, p.thin), tid = threadIdx.x;
    const int sidx = hist_slot(j, p.burnin, p.thin);
    const int blk = blockIdx.x;
    const bool replay = p.rtheta != nullptr;
    int *cur = p.counts + (size_t)(j & 1) * (K + KP);
    const uint32_t chain = (uint32_t)p.chain_offset;
    const double alpha_prev = *p.alpha_cur;
    if (tid == 0 && blockIdx.x == 0) upd_stamp(j, 0);
    if (tid == 0 && blockIdx.x == gridDim.x - 1) upd_stamp(j, 3);
    // the next sweep kernel may start its prologue now; it waits for this grid before it reads the tables
    griddep_launch();
    // Inbox mode without relabelling needs nothing from the predecessor but the tagged words themselves; otherwise wait
    // until the kernel in front (sweep, all-reduce or Q update) has completed.
    if (p.x_world < 1 || p.theta_rel_out) griddep_wait();
    const int world = p.x_world;
    const int2 *slots = nullptr;         // [world][cap] words of this exchange when the counts come from the inbox
    int xs = 0;
    if (world >= 1) {
        xs = p.x_seq[0] + j;
        slots = p.x_local + x_slot_off(xs, world, 0, (size_t)p.x_cap);
    }
    auto count_of = [&](int e) -> int {       // reduced count e (c_k for e < K, V_kd at K + k + K d)
        if (!slots) return cur[e];
        int acc = 0;
        for (int r = 0; r < world; ++r) {
            const int2 *w = slots + (size_t)r * p.x_cap + e;
            int2 v = x_load(w);
            if (v.y != xs) {
                // not there yet; a peer that never publishes must not hang the GPU: give up after 20 s of wall time
                unsigned long long t0 = 0, t1;
                unsigned spins = 0;
                while ((v = x_load(w)).y != xs) {
                    if ((++spins & 1023u) == 0) {
                        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                        if (!t0) t0 = t1;
                        else if (t1 - t0 > 20000000000ull) { *p.status = -7; break; }   // BMM_ERR_NCCL: exchange failed
                    }
                }
            }
            acc += v.x;
        }
        return acc;
    };

    if (blk < K) {
        // ---------------- cluster block: theta_kd ~ Beta(beta + V_kd, gamma + c_k - V_kd) ----------------
        const int k = blk;
        const int ck = count_of(k);
        if (tid == 0 && blk == 0) upd_stamp(j, 1);
        for (int d0 = 0; d0 < P; d0 += UPD_THREADS) {
            const int d = d0 + tid;
            if (d < P) {
                const int e = k + K * d;
                const int v = count_of(K + e);
                double th;
                if (replay) th = p.rtheta[(size_t)KP * j + e];
                else {
                    Stream st(p.seed, chain, (uint32_t)j, ST_THETA, (uint32_t)(k * P + d));
                    th = st.beta(p.beta + v, p.gamma + ck - v);
                }
                const double l1 = log(th), l0 = log(1 - th);
                p.theta_cur[e] = th;
                p.w1[e] = l1;
                p.w0[e] = l0;
                if (p.theta_out && sidx >= 0) p.theta_out[(size_t)KP * sidx + e] = th;
                if (p.theta_rel_out && sidx >= 0)   // theta_rel[perm[k], :] = theta[k, :] (full_gibbs.cpp:221-223)
                    p.theta_rel_out[(size_t)KP * sidx + p.perm_cur[k] + (size_t)K * d] = th;
                if (p.ws_b1) {
                    ws_store_cell(p.ws_b1, k, d, l1, l0);
                    sh_w0[d] = l0;
                }
            }
        }
        if (p.ws_b1) {      // s0_k in a fixed order (every rank must get the same bits)
            __syncthreads();
            if (tid < 32) {
                double a = 0.0;
                for (int d = tid; d < P; d += 32) a += sh_w0[d];
                a = warp_sum_xor(a, 32);
                if (tid == 0) p.ws_s0[k] = a;
            }
        }
        if (tid == 0 && blk == 0) upd_stamp(j, 2);
        griddep_wait();     // this grid must not complete before the sweep kernel in front has (see the end of the kernel)
        return;
    }

    // ---------------- last block: pi, alpha, log pi, history rows; zero the next sweep's count buffer ----------------
    int *next = p.counts + (size_t)((j + 1) & 1) * (K + KP);
    for (int t = tid; t < K + KP; t += blockDim.x) next[t] = 0;
    if (p.counts_out)
        for (int t = tid; t < K + KP; t += blockDim.x) p.counts_out[(size_t)j * (K + KP) + t] = count_of(t);
    if (replay) {
        for (int k = tid; k < K; k += blockDim.x) p.pi_cur[k] = p.rpi[j + (size_t)ns * k];
        __syncthreads();
        if (tid == 0) *p.alpha_cur = p.ralpha[j];
    } else {
        for (int t = tid; t < K; t += blockDim.x) sh_c[t] = count_of(t);
        __syncthreads();
        for (int t = tid; t < K; t += blockDim.x) {
            if (!p.stickbreaking) {  // Dirichlet via K Gamma(alpha/K + c_k, 1) (full_gibbs.cpp:202-210)
                Stream st(p.seed, chain, (uint32_t)j, ST_PI, (uint32_t)t);
                p.gsc[t] = st.gamma(alpha_prev / K + sh_c[t]);
            } else {                 // v_k ~ Beta(1 + c_k, alpha + sum_{l>k} c_l) (stickbreaking.cpp:187-193)
                long long later = 0;
                for (int l = t + 1; l < K; ++l) later += sh_c[l];
                Stream st(p.seed, chain, (uint32_t)j, ST_STICK, (uint32_t)t);
                p.gsc[t] = st.beta(1.0 + sh_c[t], alpha_prev + (double)later);
            }
        }
        __syncthreads();
        if (!p.stickbreaking) {
            double part = 0.0;
            for (int k = tid; k < K; k += blockDim.x) part += p.gsc[k];
            part = warp_sum_xor(part, 32);
            if ((tid & 31) == 0) red[tid >> 5] = part;
            __syncthreads();
            double sum = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) sum += red[w];
            for (int k = tid; k < K; k += blockDim.x) p.pi_cur[k] = p.gsc[k] / sum;
            if (p.alpha0 == 0.0) {          // the four Gamma substreams of the alpha update, one thread each
                if (tid < 4) {
                    Stream st(p.seed, chain, (uint32_t)j, ST_ALPHA, (uint32_t)tid);
                    ag[tid] = st.gamma(alpha_gamma_shape(tid, alpha_prev, p.a, (int)p.N_global, K));
                }
                __syncthreads();
                if (tid == 0) *p.alpha_cur = alpha_combine(ag, p.a, p.b, (int)p.N_global, K);
            }
        } else {                         // stick-breaking weights (stickbreaking.cpp:195-214)
            __shared__ int kv_sh;
            if (tid == 0) {
                p.gsc[K - 1] = 1.0;
                int K_viable = 0;
                double cumprod = 1.0;
                for (int k = 0; k < K; ++k) {
                    const double pk = (k == 0) ? p.gsc[0] : cumprod * p.gsc[k];
                    p.pi_cur[k] = pk;
                    if (pk > 0.01) K_viable++;
                    cumprod *= (1 - p.gsc[k]);
                }
                kv_sh = K_viable;
            }
            __syncthreads();
            if (p.alpha0 == 0.0) {
                if (tid < 4) {
                    Stream st(p.seed, chain, (uint32_t)j, ST_ALPHA, (uint32_t)tid);
                    ag[tid] = st.gamma(alpha_gamma_shape(tid, alpha_prev, p.a, (int)p.N_global, kv_sh));
                }
                __syncthreads();
                if (tid == 0) *p.alpha_cur = alpha_combine(ag, p.a, p.b, (int)p.N_global, kv_sh);
            }
        }
    }
    __syncthreads();
    for (int k = tid; k < K; k += blockDim.x) {
        const double pk = p.pi_cur[k];
        p.lpi[k] = log(pk);
        if (p.pi_out && sidx >= 0) p.pi_out[sidx + (size_t)S * k] = pk;
    }
    if (tid == 0 && p.alpha_out && sidx >= 0) p.alpha_out[sidx] = *p.alpha_cur;
    if (tid == 0) upd_stamp(j, 4);
    // In inbox mode nothing above waited for the sweep kernel itself, only for its tagged words.  Whatever follows in the
    // stream is ordered after THIS grid, so this grid completes only once the sweep kernel has (its allocation history
    // is read by the layout kernels, its count buffer is zeroed two sweeps later).
    griddep_wait();
}

// operand image of the initial tables (sweep 1 reads theta_0); later sweeps get it from big_update_kernel
__global__ void ws_table_kernel(const BigParams p) {
    const int K = p.K, P = p.P;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < K * P; e += gridDim.x * blockDim.x)
        ws_store_cell(p.ws_b1, e % K, e / K, p.w1[e], p.w0[e]);
    if (blockIdx.x == 0)
        for (int k = threadIdx.x; k < K; k += blockDim.x) {   // any fixed order: this launch happens once per run
            double a = 0.0;
            for (int d = 0; d < P; ++d) a += p.w0[k + K * d];
            p.ws_s0[k] = a;
        }
}

// Log tables of the initial state (sweep 1 reads theta_0, pi_0); iteration 0 of the histories.
__global__ void big_init_kernel(const BigParams p) {
    const int K = p.K, P = p.P, KP = K * P, S = hist_count(p.nsamples, p.burnin, p.thin);
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < K + KP; t += gridDim.x * blockDim.x) {
        if (t < K) {
            const double pk = p.pi_cur[t];
            p.lpi[t] = log(pk);
            if (p.burnin == 0 && p.pi_out) p.pi_out[(size_t)S * t] = pk;
        } else {
            const int e = t - K;
            const double th = p.theta_cur[e];
            p.w1[e] = log(th);
            p.w0[e] = log(1 - th);
            if (p.burnin == 0 && p.theta_out) p.theta_out[e] = th;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && p.burnin == 0 && p.alpha_out) p.alpha_out[0] = *p.alpha_cur;
    (void)P;
}

// replay: state of sweep j-1 comes from the recorded run
__global__ void big_replay_load_kernel(const BigParams p, const int j) {
    const int K = p.K, P = p.P, KP = K * P, ns = p.nsamples;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < K + KP; t += gridDim.x * blockDim.x) {
        if (t < K) {
            const double pk = p.rpi[(j - 1) + (size_t)ns * t];
            p.pi_cur[t] = pk;
            p.lpi[t] = log(pk);
        } else {
            const int e = t - K;
            const double th = p.rtheta[(size_t)KP * (j - 1) + e];
            p.theta_cur[e] = th;
            p.w1[e] = log(th);
            p.w0[e] = log(1 - th);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *p.alpha_cur = p.ralpha[j - 1];
    (void)P;
}

template <typename R>
cudaError_t launch_sweep_t(const BigParams &p, int j, int grid, cudaStream_t st) {
    BigSmem<R> *none = nullptr;
    const size_t smem = big_layout<R>(p.K, p.P, p.tables_in_smem, nullptr, none);
    cudaError_t e;
    if (p.ru) {
        e = cudaFuncSetAttribute(big_sweep_kernel<R, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        big_sweep_kernel<R, true><<<grid, BIG_THREADS, smem, st>>>(p, j);
    } else {
        e = cudaFuncSetAttribute(big_sweep_kernel<R, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        big_sweep_kernel<R, false><<<grid, BIG_THREADS, smem, st>>>(p, j);
    }
    g_launches++;
    return cudaGetLastError();
}

}  // namespace

bool big_tables_fit_smem(int K, int P, int precision) {
    const size_t KP = (size_t)K * P, r = precision == 1 ? 4 : 8;
    return (2 * KP + K) * r + (K + KP) * 4 + 64 <= 96 * 1024;
}

int big_replay_max_k() { return REPLAY_MAXK; }

cudaError_t launch_big_init(const BigParams &p, cudaStream_t st) {
    const int n = p.K + p.K * p.P;
    big_init_kernel<<<min(296, (n + 255) / 256), 256, 0, st>>>(p);
    g_launches++;
    return cudaGetLastError();
}

cudaError_t launch_big_replay_load(const BigParams &p, int j, cudaStream_t st) {
    const int n = p.K + p.K * p.P;
    big_replay_load_kernel<<<min(296, (n + 255) / 256), 256, 0, st>>>(p, j);
    g_launches++;
    return cudaGetLastError();
}

cudaError_t launch_big_sweep(const BigParams &p, int j, int sm_count, cudaStream_t st) {
    static const bool no_tc = getenv("BMM_NO_TC") != nullptr;  // A/B switch: CUDA-core float path
    if (!no_tc && !(p.flags & 32u /* BMM_FLAG_NO_TENSOR */)) {
        if (big_tc_supported(p)) return launch_big_sweep_ws(p, j, sm_count, st);
        if (big_lp_supported(p)) return launch_big_sweep_lp(p, j, sm_count, st);
    }
    long long blocks = ((long long)p.N_local + BIG_THREADS - 1) / BIG_THREADS;
    const int cap = sm_count * 8;
    const int grid = (int)(blocks < 1 ? 1 : (blocks < cap ? blocks : cap));
    if (p.precision == 1) {
        // float tables are the double tables converted on load (tables_in_smem) -- the global-table
        // variant reads the double tables through R = double.
        if (p.tables_in_smem) return launch_sweep_t<float>(p, j, grid, st);
    }
    return launch_sweep_t<double>(p, j, grid, st);
}

bool pdl_enabled() {
    static const bool on = !(getenv("BMM_PDL") && getenv("BMM_PDL")[0] == '0');
    return on;
}

cudaError_t launch_big_params(const BigParams &p, int j, cudaStream_t st) {
    // keep the L1 / shared-memory split at the sweep kernel's (which needs > 200 KB): a different split between two
    // kernels of the loop makes the SMs drain and reconfigure at every kernel boundary
    static FuncAttrCache carve;
    {
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev >= 0 && dev < 64 && !carve.set[dev]) {
            cudaFuncSetAttribute(big_update_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            carve.set[dev] = 1;
        }
    }
    g_launches++;
    return launch_pdl(big_update_kernel, dim3(p.K + 1), dim3(UPD_THREADS), 0, st, p, j);
}

__global__ void x_begin_run_kernel(int *seq, int n) {
    seq[0] = seq[1];
    seq[1] += n;
}
cudaError_t launch_x_begin_run(int *seq, int n_sweeps, cudaStream_t st) {
    x_begin_run_kernel<<<1, 1, 0, st>>>(seq, n_sweeps);
    g_launches++;
    return cudaGetLastError();
}

cudaError_t upd_trace_read(unsigned long long out[16]) { return cudaMemcpyFromSymbol(out, g_upd_trace, 16 * sizeof(unsigned long long)); }

cudaError_t launch_ws_table(const BigParams &p, cudaStream_t st) {
    if (!p.ws_b1) return cudaSuccess;
    ws_table_kernel<<<16, 256, 0, st>>>(p);
    g_launches++;
    return cudaGetLastError();
}

}  // namespace bmm
