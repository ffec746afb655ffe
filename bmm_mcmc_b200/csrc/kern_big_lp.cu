// Large-P / large-K tensor-core path of the grid sampler (BASELINE config C5: N = 1e6, P = 4096,
// K = 128).  Same algebra as kern_big_ws.cu -- loglh = X D^T + b on tcgen05 with D split into two
// fp16 terms, sufficient statistics as [X]^T onehot(z) -- but P no longer fits one shared-memory tile,
// so the contraction runs as a pipelined k-loop and the statistics as a second kernel:
//
//   lp_table_kernel    per sweep: D (log2 units) split into fp16 hi|lo (22 significant bits; the 0/1 rows are
//                      exact in fp16), written to global memory already in the shared-memory operand image
//                      ([64-feature step][16-B chunk][2*128 rows][16 B]), so a stage is one contiguous 32 KB block.
//   lp_sweep_kernel    persistent, a 256-observation super-tile (two 128-row tiles) at a time per CTA, 3-stage
//                      mbarrier pipeline of 64 features:
//                        warps 0-7  expand 64 bits per observation and step into the two fp16 A tiles of the
//                                   stage; after a super-tile's last step they run its epilogue: three passes
//                                   over TMEM (max, sum, inverse-CDF walk; 128 logits do not fit the register
//                                   file), 1-byte allocation to HBM;
//                        warp 8     one thread streams the B stage with cp.async.bulk (mbarrier tx count);
//                        warp 9     one thread issues 8 tcgen05.mma (M128 N256 K16) per step: both tiles
//                                   against the SAME B stage, into two 128 x 256 fp32 accumulators (all of TMEM).
//                      Sharing a B stage between two tiles halves the table traffic out of L2, which bounded
//                      the one-tile version (every tile re-reads the 2 MB table: 9.3 TB/s at 1.77 ms).
//   (counts)           V_kd, c_k from the allocations: kern_big_counts.cu (counting sort + bit-sliced counters
//                      on the packed rows; a tcgen05 [X]^T onehot(z) kernel used to sit here and was 10x slower).
//
// Replaces /root/reference/src/full_gibbs.cpp:87-157,182-200 (stickbreaking.cpp:70-140,164-186) at sizes
// where the reference itself cannot run (its unstabilised exp underflows at P = 4096, full_gibbs.cpp:106).
#include <cuda_fp16.h>

#include "common.cuh"
#include "kernels.h"
#include "umma.cuh"

namespace bmm {
namespace {

constexpr int LP_KC = 128;                  // clusters, padded
constexpr int LP_NCOL = 2 * LP_KC;          // accumulator columns per tile: hi | lo
constexpr int LP_DK = 64;                   // features per pipeline step
constexpr int LP_TM = 2;                    // 128-observation tiles sharing one B stage (a 256-row super-tile)
constexpr int LP_A_TILE = 8 * 2048;         // [8 chunks][128 rows][16 B]
constexpr int LP_A_STAGE = LP_TM * LP_A_TILE;
constexpr int LP_B_STAGE = 8 * LP_NCOL * 16;  // [8 chunks][256 rows][16 B]
constexpr int LP_STAGE = LP_A_STAGE + LP_B_STAGE;
constexpr int LP_NS = 3;                    // pipeline stages (64 KB each)
constexpr int LP_ROWT = LP_TM * 128;        // row threads: warps 0-7 write A stages, then run the epilogue
constexpr int LP_THREADS = LP_ROWT + 64;    // + warp 8 B streamer, warp 9 MMA issuer
constexpr double LOG2E_D = 1.4426950408889634;

// ---- per-sweep tables -----------------------------------------------------------------------------
// The conditional probabilities only depend on differences between clusters, so both D_kd and b_k
// are centred over k (exact in double) before they are rounded: the fp32 accumulator then carries a
// zero-mean random walk of magnitude ~sqrt(P) instead of a drift of magnitude ~P, which is what keeps
// the probabilities within 1e-4 of fp64 at P = 4096.
__global__ void lp_table_kernel(const BigParams p) {
    const int K = p.K, P = p.P;
    unsigned char *img = (unsigned char *)p.lp_table;
    const int Ppad = (P + LP_DK - 1) / LP_DK * LP_DK;   // features beyond P: zero weights (their bits are zero too)
    for (int d = blockIdx.x * blockDim.x + threadIdx.x; d < Ppad; d += gridDim.x * blockDim.x) {
        const bool real = d < P;
        const double *w1 = p.w1 + (size_t)K * (real ? d : 0), *w0 = p.w0 + (size_t)K * (real ? d : 0);
        // theta_kd drawn as exactly 0 or 1 gives log 0 = -inf; the reference then computes 0 * -inf = NaN and
        // dies (full_gibbs.cpp:97).  Here such a weight is clamped to +-1e4 (a factor 2^-10000 = 0), which is
        // the limit the reference's formula is reaching for, and the centring only uses finite entries.
        double mean = 0.0;
        int nfin = 0;
        for (int k = 0; k < K; ++k) { const double D = w1[k] - w0[k]; if (isfinite(D)) { mean += D; ++nfin; } }
        mean = nfin ? mean / nfin : 0.0;
        unsigned char *col = img + (size_t)(d >> 3) * LP_NCOL * 16 + (d & 7) * 2;
        for (int k = 0; k < LP_KC; ++k) {
            double D = (real && k < K) ? (w1[k] - w0[k] - mean) * LOG2E_D : 0.0;
            D = fmin(fmax(D, -1.0e4), 1.0e4);
            if (D != D) D = 0.0;
            const __half hi = __double2half(D);
            const __half lo = __double2half(D - (double)__half2float(hi));
            *(__half *)(col + (0 * LP_KC + k) * 16) = hi;
            *(__half *)(col + (1 * LP_KC + k) * 16) = lo;
        }
    }
}

// b_k = log2(e) * (log pi_k + sum_d log(1 - theta_kd)) in double; centred and rounded by the sweep kernel
__global__ void lp_bias_kernel(const BigParams p) {
    __shared__ double red[4];
    const int k = blockIdx.x, K = p.K, P = p.P;
    double s = 0.0;
    if (k < K) for (int d = threadIdx.x; d < P; d += blockDim.x) s += p.w0[k + (size_t)K * d];
    s = warp_sum_xor(s, 32);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) p.lp_bias[k] = k < K ? (p.lpi[k] + red[0] + red[1] + red[2] + red[3]) * LOG2E_D : 0.0;
}

// ---- the sweep ------------------------------------------------------------------------------------
struct LpSmem {
    static constexpr int BIAS_OFF = LP_STAGE * LP_NS;
    static constexpr int BAR_OFF = BIAS_OFF + LP_KC * 4;
    static constexpr int TOTAL = BAR_OFF + (2 * LP_NS + 2) * 8 + 16;
};

// logits of 32 clusters [c0, c0+32) of this thread's observation: hi + lo + bias
__device__ __forceinline__ void lp_logits32(uint32_t acc, uint32_t lane_sel, int c0, const float *bias, float (&l)[32]) {
    uint32_t v[32], w[32];
    tmem_ld32(acc + lane_sel + (uint32_t)c0, v);
    tmem_ld32(acc + lane_sel + (uint32_t)(LP_KC + c0), w);
    tmem_ld_wait();
#pragma unroll
    for (int q = 0; q < 32; ++q) l[q] = (__uint_as_float(v[q]) + __uint_as_float(w[q])) + bias[c0 + q];
}

__global__ void __launch_bounds__(LP_THREADS, 1) lp_sweep_kernel(const BigParams p, const int j) {
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5;
    const int K = p.K, W = p.W;
    const int nsteps = (p.P + LP_DK - 1) / LP_DK;   // the last step may be partial: missing words read as zero bits
    float *bias = (float *)(smem + LpSmem::BIAS_OFF);
    uint64_t *bars = (uint64_t *)(smem + LpSmem::BAR_OFF);   // full[NS], empty[NS], accfull, accempty
    uint32_t *tmem_slot = (uint32_t *)(bars + 2 * LP_NS + 2);
    const uint32_t full0 = smem_u32(&bars[0]), empty0 = smem_u32(&bars[LP_NS]);
    const uint32_t accfull = smem_u32(&bars[2 * LP_NS]), accempty = smem_u32(&bars[2 * LP_NS + 1]);
    constexpr int BW = LP_ROWT / 32, MW = BW + 1;   // B-streamer warp, MMA warp

    if (warp == BW) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == MW * 32) {
        for (int s = 0; s < LP_NS; ++s) {
            mbar_init(full0 + 8 * s, LP_ROWT + 1);   // row threads + the bulk-copy thread
            mbar_init(empty0 + 8 * s, 1);            // tcgen05.commit
        }
        mbar_init(accfull, 1); mbar_init(accempty, LP_ROWT);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    {   // shift by the largest finite b_k (a cluster with pi_k = 0 has b_k = -inf and simply never wins)
        double top = -INFINITY;
        for (int k = 0; k < K; ++k) { const double b = p.lp_bias[k]; if (isfinite(b)) top = fmax(top, b); }
        if (!isfinite(top)) top = 0.0;
        for (int k = tid; k < LP_KC; k += LP_THREADS) {
            const double b = k < K ? p.lp_bias[k] - top : -INFINITY;
            bias[k] = b == b ? (float)b : -INFINITY;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t acc = *tmem_slot;
    const long long nsuper = ((long long)p.N_local + LP_ROWT - 1) / LP_ROWT;   // super-tiles of 256 observations
    const long long mine = blockIdx.x < nsuper ? (nsuper - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;   // of this CTA
    bool ok = true;

    if (warp < BW) {
        // ================= rows -> fp16 A stages, and the epilogue of the finished super-tile =================
        const int h = tid >> 7, r = tid & 127;            // tile within the super-tile, row = TMEM lane
        const uint32_t lane_sel = (uint32_t)((warp & 3) * 32) << 16, acch = acc + (uint32_t)(h * LP_NCOL);
        const uint2 key = make_uint2((uint32_t)p.seed, (uint32_t)p.chain_offset);
        const uint32_t sid = ST_Z ^ ((uint32_t)(p.seed >> 32) << 8);
        uint8_t *zrow = p.zhist + (size_t)(p.keep_history ? j : 0) * p.N_local;
        auto row_of = [&](long long it) { return ((long long)blockIdx.x + it * gridDim.x) * LP_ROWT + tid; };
        // two 32-bit words per step; rows are only 4-byte aligned when W is odd, so the words are read singly
        auto load_step = [&](long long it, int c) {
            uint2 v = make_uint2(0u, 0u);
            const long long i = row_of(it);
            if (it < mine && i < p.N_local) {
                const uint32_t *xb = p.xbits + (size_t)i * W;
                if ((W & 1) == 0) { if (2 * c < W) v = *(const uint2 *)(xb + 2 * c); }   // 8-byte aligned rows
                else {
                    if (2 * c < W) v.x = xb[2 * c];
                    if (2 * c + 1 < W) v.y = xb[2 * c + 1];
                }
            }
            return v;
        };
        auto epilogue = [&](long long it) {
            const long long i = row_of(it);
            const bool valid = i < p.N_local;
            const unsigned long long gi = (unsigned long long)p.row_offset + (unsigned long long)i;
            const uint4 rnd = philox4x32_10(make_uint4((uint32_t)(gi >> 2), (uint32_t)(gi >> 34), sid, (uint32_t)j), key);
            const float u = u32_unit_f(philox_word(rnd, (int)(gi & 3)));
            ok = mbar_wait(accfull, (uint32_t)(it & 1));
            if (!ok) return;
            tc_fence_after();
            float l[32];
            float mx = -INFINITY;
            for (int c0 = 0; c0 < LP_KC; c0 += 32) {
                lp_logits32(acch, lane_sel, c0, bias, l);
#pragma unroll
                for (int q = 0; q < 32; ++q) mx = fmaxf(mx, l[q]);
            }
            float sum = 0.f;
            for (int c0 = 0; c0 < LP_KC; c0 += 32) {
                lp_logits32(acch, lane_sel, c0, bias, l);
#pragma unroll
                for (int q = 0; q < 32; ++q) sum += ex2_ftz(l[q] - mx);
            }
            if (!(sum > 0.f) || !isfinite(sum)) *p.status = -9;  // BMM_ERR_PROB
            const float target = u * sum, inv = 1.f / sum;
            float run = 0.f;
            int z = 0;
            for (int c0 = 0; c0 < LP_KC; c0 += 32) {
                lp_logits32(acch, lane_sel, c0, bias, l);
#pragma unroll
                for (int q = 0; q < 32; ++q) {
                    const float e = ex2_ftz(l[q] - mx);
                    run += e;
                    z += (run <= target) ? 1 : 0;
                    if (p.probs_out && valid && c0 + q < K)
                        p.probs_out[(size_t)j * p.N_local * K + i + (size_t)p.N_local * (c0 + q)] = (double)(e * inv);
                    l[q] = e * inv;
                }
                if (p.probs_f32 && valid) {        // this observation's row of P, 16 bytes at a time when aligned
                    float *dst = p.probs_f32 + (size_t)i * K + c0;
                    if ((K & 3) == 0) {
#pragma unroll
                        for (int q = 0; q < 32; q += 4)
                            if (c0 + q < K) *(float4 *)(dst + q) = make_float4(l[q], l[q + 1], l[q + 2], l[q + 3]);
                    } else {
#pragma unroll
                        for (int q = 0; q < 32; ++q)
                            if (c0 + q < K) dst[q] = l[q];
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(accempty);             // the accumulators may be overwritten by the next super-tile
            // This walk adds the same values in the same order as the total, so at the last cluster with weight run == sum
            // > target = u * sum for every u < 1 (u32_unit_f stays below 1): clusters of weight 0 after it are never
            // counted, and the clamp only guards against a NaN total.
            z = min(z, K - 1);
            if (valid) zrow[i] = (uint8_t)(z + 1);
        };
        // Stages are produced in one flat sequence over (super-tile, step).  The epilogue of a super-tile runs after
        // the first `pre` stages of the next one are in the ring, so the MMAs restart as soon as the accumulators
        // are released (those stages only wait for MMAs of the finished super-tile: no cycle through accempty).
        const int pre = nsteps < LP_NS ? nsteps : LP_NS;
        const long long nstage = mine * nsteps;
        long long it = 0, itp = 0;             // super-tile of stage g / of the stage being prefetched (g + 2)
        int c = 0, cp = 0;                     // step within it
        auto advance = [&](long long &t, int &k) { if (++k == nsteps) { k = 0; ++t; } };
        uint2 nxt = load_step(itp, cp);
        advance(itp, cp);
        uint2 nxt2 = load_step(itp, cp);
        advance(itp, cp);
        for (long long g = 0; g < nstage && ok; ++g) {
            const uint2 cur = nxt;
            nxt = nxt2;
            nxt2 = load_step(itp, cp);
            advance(itp, cp);
            uint4 ex[8];
#pragma unroll
            for (int ch = 0; ch < 8; ++ch) {
                const uint32_t byte = (ch < 4 ? cur.x : cur.y) >> ((ch & 3) * 8);
                ex[ch] = make_uint4(bits2_f16x2(byte), bits2_f16x2(byte >> 2), bits2_f16x2(byte >> 4), bits2_f16x2(byte >> 6));
            }
            const int s = (int)(g % LP_NS);
            const long long n = g / LP_NS;
            if (n > 0) ok = mbar_wait(empty0 + 8 * s, (uint32_t)((n - 1) & 1));
            if (!ok) break;
            unsigned char *A = smem + s * LP_STAGE + h * LP_A_TILE;
#pragma unroll
            for (int ch = 0; ch < 8; ++ch) *(uint4 *)(A + ch * 2048 + r * 16) = ex[ch];
            fence_async_smem();
            mbar_arrive(full0 + 8 * s);
            if (it > 0 && c == pre - 1) epilogue(it - 1);
            advance(it, c);
        }
        if (ok && mine > 0) epilogue(mine - 1);
    } else if (warp == BW) {
      if (tid == BW * 32) {
        // ================= B stage streamer =================
        const unsigned char *img = (const unsigned char *)p.lp_table;
        const long long nstage = mine * nsteps;
        int c = 0;
        for (long long g = 0; g < nstage && ok; ++g) {
            const int s = (int)(g % LP_NS);
            const long long n = g / LP_NS;
            if (n > 0) ok = mbar_wait(empty0 + 8 * s, (uint32_t)((n - 1) & 1));
            if (!ok) break;
            const uint32_t dst = smem_u32(smem + s * LP_STAGE + LP_A_STAGE);
            mbar_arrive_expect_tx(full0 + 8 * s, LP_B_STAGE);
            bulk_g2s(dst, img + (size_t)c * LP_B_STAGE, LP_B_STAGE, full0 + 8 * s);
            if (++c == nsteps) c = 0;
        }
      }
      __syncwarp();
    } else {
      {
        // ================= MMA issuer: per step 4 x K16 for each of the two tiles against the same B stage =================
        // (all 32 lanes walk the loop, one elected lane issues: umma.cuh::elect_one)
        constexpr uint32_t IDESC = umma_idesc_f16(128, LP_NCOL, 0, 0);
        long long g = 0;
        for (long long it = 0; it < mine && ok; ++it) {
            if (it > 0) ok = __all_sync(0xffffffffu, mbar_wait(accempty, (uint32_t)((it - 1) & 1)));
            tc_fence_after();
            for (int c = 0; c < nsteps && ok; ++c, ++g) {
                const int s = (int)(g % LP_NS);
                ok = __all_sync(0xffffffffu, mbar_wait(full0 + 8 * s, (uint32_t)((g / LP_NS) & 1)));
                if (!ok) break;
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t a0 = smem_u32(smem + s * LP_STAGE), b0 = a0 + LP_A_STAGE;
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
#pragma unroll
                        for (int h = 0; h < LP_TM; ++h)
                            umma_f16(acc + (uint32_t)(h * LP_NCOL), umma_desc(a0 + h * LP_A_TILE + kk * 2 * 2048, 2048, 128),
                                      umma_desc(b0 + kk * 2 * (LP_NCOL * 16), LP_NCOL * 16, 128), IDESC, (c | kk) ? 1u : 0u);
                    umma_commit(empty0 + 8 * s);
                    if (c == nsteps - 1) umma_commit(accfull);
                }
                __syncwarp();
            }
        }
      }
      __syncwarp();
    }
    if (!ok) *p.status = -10;  // BMM_ERR_TIMEOUT
    tc_fence_before();
    __syncthreads();
    if (warp == BW) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(acc), "r"(512) : "memory");
    }
}

}  // namespace

// float path, K <= 128 clusters, any P (padded to a multiple of 64 with zero weights)
bool big_lp_supported(const BigParams &p) {
    return p.precision == 1 && p.K <= LP_KC && p.ru == nullptr &&
           p.loglik_out == nullptr && p.lp_table != nullptr;
}

size_t big_lp_table_bytes(int P) { return (size_t)((P + LP_DK - 1) / LP_DK * LP_DK) / 8 * LP_NCOL * 16; }

cudaError_t launch_big_sweep_lp(const BigParams &p, int j, int sm_count, cudaStream_t st) {
    static FuncAttrCache attr;
    if (cudaError_t e = attr.ensure_smem(lp_sweep_kernel, (int)LpSmem::TOTAL)) return e;
    lp_table_kernel<<<(p.P + 63) / 64, 64, 0, st>>>(p);   // one thread per (padded) feature
    lp_bias_kernel<<<LP_KC, 128, 0, st>>>(p);
    const long long ntiles = ((long long)p.N_local + LP_ROWT - 1) / LP_ROWT;
    const int ctas = (int)(ntiles < sm_count ? ntiles : sm_count);
    lp_sweep_kernel<<<ctas, LP_THREADS, LpSmem::TOTAL, st>>>(p, j);
    g_launches += 3;
    // counts of this sweep from the allocations just written (kern_big_counts.cu)
    const uint8_t *zrow = p.zhist + (size_t)(p.keep_history ? j : 0) * p.N_local;
    return launch_big_counts(p.N_local, p.K, p.P, p.W, p.xbits, zrow, p.counts + (size_t)(j & 1) * (p.K + (size_t)p.K * p.P),
                             p.cnt_ws, sm_count, st);
}

}  // namespace bmm
