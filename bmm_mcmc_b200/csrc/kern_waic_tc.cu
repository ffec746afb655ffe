// Tensor-core WAIC pass for K <= 32, P <= 112 (the shapes of kern_big_ws.cu).  The loop order is the reverse of the
// z-sweep: a CTA owns 128-row tiles of the distinct rows and walks all D = C S draws over each tile.
//
//   waic_tc_tables_kernel   per draw g: the fp16 hi | lo operand image of D_kd = log2 theta_kd - log2(1 - theta_kd)
//                           (ws_table.cuh, 1 KB per 8 variables) and the bias b_k = log2 pi_k + sum_d log2(1 - theta_kd)
//   waic_tc_kernel          warps 0-3   expand the tile's packed rows to the fp16 A operand once per tile; then the
//                                       epilogue: TMEM lane = row, l = ln 2 * log2 sum_k 2^(hi + lo + b_k) per draw
//                                       (fp32 ex2 / lg2), running Welford and log-sum-exp moments in fp64 registers,
//                                       written once per chain; the warp's fp64 share of the trace per draw
//                           warp 4      streams the draws' images through a ring of WT_NB shared-memory stages
//                                       (cp.async.bulk)
//                           warp 5      one elected lane issues X [hi|lo]^T into two alternating 64-column TMEM
//                                       accumulators, so draw g + 1 multiplies while draw g is in the epilogue
//
// Every wait on an mbarrier is bounded; a time-out sets *status = BMM_ERR_TIMEOUT.  The partials have the layout of the
// fp64 path (kern_predict.cu) with one slice per chain, and waic_merge_kernel / waic_sum_kernel combine them in a fixed
// order: the results do not depend on the grid size.
//
// With LMAT = true (launch_loglik_tc) the epilogue stores l itself, L[g U + u] over the D draws of one pooled chain (the
// log-likelihood matrix PSIS-LOO reads, kern_loo.cu), lane = row so a warp's store is 256 contiguous bytes, and keeps no
// moments.  The WAIC instantiation (LMAT = false) is unchanged.
#include <cstdlib>
#include <cuda_fp16.h>

#include "kernels.h"
#include "umma.cuh"
#include "ws_table.cuh"

namespace bmm {
namespace {

constexpr int WT_NB = 4;        // image ring stages (one epilogue warpgroup: any depth keeps a stage with its consumer)
constexpr int WT_NA = 2;        // TMEM accumulators of WS_PARTS * WS_KC = 64 columns
constexpr int WT_THREADS = 192;
constexpr int WS_CHUNK = 2048;  // one 8-variable chunk of a 128-row A tile (the kern_big_ws.cu layout)

__global__ void waic_tc_tables_kernel(int K, int P, const double *__restrict__ theta, const double *__restrict__ pi,
                                      long long D, unsigned char *__restrict__ img, float *__restrict__ bias) {
    const int nch = ws_nch(P);
    const size_t ib = (size_t)nch * WS_B1_ROW;
    const long long g = blockIdx.x;
    unsigned char *B = img + (size_t)g * ib;
    for (int e = threadIdx.x; e < (int)(ib / 16); e += blockDim.x) ((uint4 *)B)[e] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();
    const double *th = theta + (size_t)K * P * g;
    for (int e = threadIdx.x; e < K * P; e += blockDim.x) {
        const double t = th[e];
        ws_store_cell(B, e % K, e / K, log(t), log(1.0 - t));
    }
    for (int k = threadIdx.x; k < WS_KC; k += blockDim.x) {
        float b = -INFINITY;
        if (k < K) {
            double a = log(pi[(size_t)g + (size_t)D * k]);
            for (int d = 0; d < P; ++d) a += log(1.0 - th[k + (size_t)K * d]);
            a *= 1.4426950408889634;
            b = a == a ? (float)fmax(a, -3.0e38) : -INFINITY;
        }
        bias[(size_t)g * WS_KC + k] = b;
    }
}

template <int NCH>
struct WtLayout {
    static constexpr int IMG = NCH * WS_B1_ROW;
    static constexpr int RING_OFF = NCH * WS_CHUNK;
    static constexpr int BAR_OFF = RING_OFF + WT_NB * IMG;
    static constexpr int NBAR = 2 * WT_NB + 2 * WT_NA + 1;
    static constexpr int TOTAL = BAR_OFF + NBAR * 8 + 16;
    // at most four CTAs per SM: each holds WT_NA * 64 of the SM's 512 TMEM columns
    static constexpr int LAUNCH = TOTAL > 50 * 1024 ? TOTAL : 50 * 1024;
};

template <int NCH, bool LMAT>
__global__ void __launch_bounds__(WT_THREADS) waic_tc_kernel(int U, int W, int S, int C, const uint32_t *__restrict__ rowbits,
                                                             const int *__restrict__ wt, const unsigned char *__restrict__ img,
                                                             const float *__restrict__ bias, double *__restrict__ stat,
                                                             double *__restrict__ tpart, int *__restrict__ status) {
    using L = WtLayout<NCH>;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5;
    const int D = C * S;
    uint64_t *bars = (uint64_t *)(smem + L::BAR_OFF);
    uint32_t *tmem_slot = (uint32_t *)(bars + L::NBAR);
    const uint32_t b_full = smem_u32(bars), b_free = b_full + 8 * WT_NB;
    const uint32_t acc_full = b_free + 8 * WT_NB, acc_free = acc_full + 8 * WT_NA, a_full = acc_free + 8 * WT_NA;
    if (warp == 5) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"(WT_NA * 64) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 128) {
        for (int s = 0; s < WT_NB; ++s) { mbar_init(b_full + 8 * s, 1); mbar_init(b_free + 8 * s, 1); }
        for (int a = 0; a < WT_NA; ++a) { mbar_init(acc_full + 8 * a, 1); mbar_init(acc_free + 8 * a, 128); }
        mbar_init(a_full, 128);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int ntiles = (U + 127) / 128;
    const int T = (int)blockIdx.x < ntiles ? (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const long long steps = (long long)T * D;
    bool ok = true;

    if (warp == 4) {
        // ================= image ring producer =================
        int slot = 0, g = 0;
        uint32_t ph = 0;
        for (long long n = 0; n < steps; ++n) {
            if (n >= WT_NB) ok = mbar_wait(b_free + 8 * slot, ph ^ 1u);
            ok = __all_sync(0xffffffffu, ok);
            if (!ok) break;
            if (elect_one()) {
                mbar_arrive_expect_tx(b_full + 8 * slot, L::IMG);
                bulk_g2s(smem_u32(smem + L::RING_OFF + slot * L::IMG), img + (size_t)g * L::IMG, L::IMG, b_full + 8 * slot);
            }
            __syncwarp();
            if (++g == D) g = 0;
            if (++slot == WT_NB) { slot = 0; ph ^= 1u; }
        }
    } else if (warp == 5) {
        // ================= MMA issuer =================
        constexpr uint32_t IDESC = umma_idesc_f16(128, WS_PARTS * WS_KC, 0, 0);
        const uint64_t da0 = umma_desc(smem_u32(smem), WS_CHUNK, 128);
        const uint64_t db0 = umma_desc(smem_u32(smem + L::RING_OFF), WS_B1_ROW, 128);
        int slot = 0, a = 0;
        uint32_t ph_b = 0, ph_a = 0;
        long long n = 0;
        for (int kt = 0; kt < T && ok; ++kt) {
            ok = __all_sync(0xffffffffu, mbar_wait(a_full, (uint32_t)(kt & 1)));
            if (!ok) break;
            for (int g = 0; g < D; ++g, ++n) {
                ok = mbar_wait(b_full + 8 * slot, ph_b);
                if (ok && n >= WT_NA) ok = mbar_wait(acc_free + 8 * a, ph_a ^ 1u);
                ok = __all_sync(0xffffffffu, ok);
                if (!ok) break;
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t db = db0 + (uint64_t)((slot * L::IMG) >> 4);
#pragma unroll
                    for (int kk = 0; kk < NCH / 2; ++kk)
                        umma_f16(tmem_base + (uint32_t)(a * WS_PARTS * WS_KC), da0 + (uint64_t)((kk * 2 * WS_CHUNK) >> 4),
                                 db + (uint64_t)((kk * 2 * WS_B1_ROW) >> 4), IDESC, kk ? 1u : 0u);
                    umma_commit(b_free + 8 * slot);
                    umma_commit(acc_full + 8 * a);
                }
                __syncwarp();
                if (++slot == WT_NB) { slot = 0; ph_b ^= 1u; }
                if (++a == WT_NA) { a = 0; ph_a ^= 1u; }
            }
        }
    } else {
        // ================= A expansion + epilogue (warps 0-3) =================
        const int t = tid, lane = tid & 31;
        const uint32_t lane_sel = (uint32_t)(warp * 32) << 16;
        constexpr int NW = (NCH + 3) / 4;
        const long long G = 4LL * ntiles;
        int a = 0;
        uint32_t ph_a = 0;
        for (int kt = 0; kt < T && ok; ++kt) {
            const int tile = (int)blockIdx.x + kt * (int)gridDim.x;
            const int u = tile * 128 + t;
            const bool valid = u < U;
            // this thread's A row (the MMAs of the previous tile are complete: this thread saw their last commit)
            uint32_t xw[NW];
#pragma unroll
            for (int w = 0; w < NW; ++w) xw[w] = (valid && w < W) ? rowbits[(size_t)u * W + w] : 0u;
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                const uint32_t y = __byte_perm(xw[c >> 2], 0u, 0x4440u + (c & 3)) * 0x8001u;
                *(uint4 *)(smem + c * WS_CHUNK + t * 16) =
                    make_uint4((y & 0x10001u) * 0x3C00u, ((y >> 2) & 0x10001u) * 0x3C00u,
                               ((y >> 4) & 0x10001u) * 0x3C00u, ((y >> 6) & 0x10001u) * 0x3C00u);
            }
            fence_async_smem();
            mbar_arrive(a_full);
            const double w = (!LMAT && valid) ? (double)wt[u] : 0.0;
            double st[WAIC_STAT];
            waic_stat_init(st);
            int c = 0, s = 0;
            for (int g = 0; g < D; ++g) {
                ok = mbar_wait(acc_full + 8 * a, ph_a);
                if (!ok) break;
                tc_fence_after();
                float l2[WS_KC];
                {
                    uint32_t v[32];
                    tmem_ld32(tmem_base + lane_sel + (uint32_t)(a * WS_PARTS * WS_KC), v);
                    tmem_ld_wait();
#pragma unroll
                    for (int q = 0; q < WS_KC; ++q) l2[q] = __uint_as_float(v[q]);
                    tmem_ld32(tmem_base + lane_sel + (uint32_t)(a * WS_PARTS * WS_KC + WS_KC), v);
                    tmem_ld_wait();
                    const float4 *b4 = (const float4 *)(bias + (size_t)g * WS_KC);
#pragma unroll
                    for (int q = 0; q < WS_KC / 4; ++q) {
                        const float4 b = __ldg(b4 + q);
                        l2[4 * q] += __uint_as_float(v[4 * q]) + b.x;
                        l2[4 * q + 1] += __uint_as_float(v[4 * q + 1]) + b.y;
                        l2[4 * q + 2] += __uint_as_float(v[4 * q + 2]) + b.z;
                        l2[4 * q + 3] += __uint_as_float(v[4 * q + 3]) + b.w;
                    }
                }
                tc_fence_before();
                mbar_arrive(acc_free + 8 * a);
                float mx = l2[0];
#pragma unroll
                for (int q = 1; q < WS_KC; ++q) mx = fmaxf(mx, l2[q]);
                double l = -INFINITY;
                if (mx > -INFINITY) {
                    float sum = 0.f;
#pragma unroll
                    for (int q = 0; q < WS_KC; ++q) sum += ex2_ftz(l2[q] - mx);
                    float lg;
                    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(sum));
                    l = ((double)mx + (double)lg) * 0.6931471805599453;
                }
                if constexpr (LMAT) {
                    if (valid) stat[(size_t)g * U + u] = l;
                    if (++a == WT_NA) { a = 0; ph_a ^= 1u; }
                    continue;
                }
                waic_push(st, l);
                double v = valid ? w * l : 0.0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (lane == 0) tpart[(size_t)g * G + 4LL * tile + warp] = v;
                if (++s == S) {
                    if (valid)
                        for (int e = 0; e < WAIC_STAT; ++e) stat[((size_t)c * U + u) * WAIC_STAT + e] = st[e];
                    waic_stat_init(st);
                    s = 0;
                    ++c;
                }
                if (++a == WT_NA) { a = 0; ph_a ^= 1u; }
            }
        }
    }
    if (!ok) *status = -10;   // BMM_ERR_TIMEOUT
    tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(WT_NA * 64) : "memory");
    }
}

template <int NCH, bool LMAT>
cudaError_t launch_tc_nch(int U, int W, int S, int C, const uint32_t *rowbits, const int *wt, const unsigned char *img,
                          const float *bias, double *stat, double *tpart, int *status, int sm_count, cudaStream_t st) {
    using L = WtLayout<NCH>;
    static FuncAttrCache attr;
    if (cudaError_t e = attr.ensure_smem(waic_tc_kernel<NCH, LMAT>, (int)L::LAUNCH)) return e;
    int per_sm = 0;
    if (cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, waic_tc_kernel<NCH, LMAT>, WT_THREADS, (size_t)L::LAUNCH))
        return e;
    const long long ntiles = ((long long)U + 127) / 128;
    long long ctas = (long long)sm_count * (per_sm < 1 ? 1 : per_sm);
    if (ctas > ntiles) ctas = ntiles;
    if (const char *e = getenv("BMM_GRID_MAX_CTAS")) { const int cap = atoi(e); if (cap > 0 && ctas > cap) ctas = cap; }   // tests: many tiles per CTA
    if (ctas < 1) ctas = 1;
    waic_tc_kernel<NCH, LMAT><<<(unsigned)ctas, WT_THREADS, (size_t)L::LAUNCH, st>>>(U, W, S, C, rowbits, wt, img, bias, stat, tpart, status);
    g_launches++;
    return cudaGetLastError();
}

}  // namespace

bool waic_tc_supported(int K, int P) { return K <= WS_KC && P <= 112; }
size_t waic_tc_img_bytes(int P) { return (size_t)ws_nch(P) * WS_B1_ROW; }

cudaError_t launch_waic_tc_tables(int K, int P, long long D, const double *theta, const double *pi, unsigned char *img,
                                  float *bias, cudaStream_t st) {
    waic_tc_tables_kernel<<<(unsigned)D, 128, 0, st>>>(K, P, theta, pi, D, img, bias);
    g_launches++;
    return cudaGetLastError();
}

cudaError_t launch_waic_tc(int U, int P, int W, int K, int S, int C, const uint32_t *rowbits, const int *wt,
                           const unsigned char *img, const float *bias, double *stat, double *tpart, int *status,
                           int sm_count, cudaStream_t st) {
    (void)K;
    switch (ws_nch(P)) {
        case 2: return launch_tc_nch<2, false>(U, W, S, C, rowbits, wt, img, bias, stat, tpart, status, sm_count, st);
        case 4: return launch_tc_nch<4, false>(U, W, S, C, rowbits, wt, img, bias, stat, tpart, status, sm_count, st);
        case 6: return launch_tc_nch<6, false>(U, W, S, C, rowbits, wt, img, bias, stat, tpart, status, sm_count, st);
        case 8: return launch_tc_nch<8, false>(U, W, S, C, rowbits, wt, img, bias, stat, tpart, status, sm_count, st);
        case 10: return launch_tc_nch<10, false>(U, W, S, C, rowbits, wt, img, bias, stat, tpart, status, sm_count, st);
        case 12: return launch_tc_nch<12, false>(U, W, S, C, rowbits, wt, img, bias, stat, tpart, status, sm_count, st);
        default: return launch_tc_nch<14, false>(U, W, S, C, rowbits, wt, img, bias, stat, tpart, status, sm_count, st);
    }
}

cudaError_t launch_loglik_tc(int Uc, int P, int W, long long D, const uint32_t *rowbits, const unsigned char *img,
                             const float *bias, double *L, int *status, int sm_count, cudaStream_t st) {
    switch (ws_nch(P)) {
        case 2: return launch_tc_nch<2, true>(Uc, W, (int)D, 1, rowbits, nullptr, img, bias, L, nullptr, status, sm_count, st);
        case 4: return launch_tc_nch<4, true>(Uc, W, (int)D, 1, rowbits, nullptr, img, bias, L, nullptr, status, sm_count, st);
        case 6: return launch_tc_nch<6, true>(Uc, W, (int)D, 1, rowbits, nullptr, img, bias, L, nullptr, status, sm_count, st);
        case 8: return launch_tc_nch<8, true>(Uc, W, (int)D, 1, rowbits, nullptr, img, bias, L, nullptr, status, sm_count, st);
        case 10: return launch_tc_nch<10, true>(Uc, W, (int)D, 1, rowbits, nullptr, img, bias, L, nullptr, status, sm_count, st);
        case 12: return launch_tc_nch<12, true>(Uc, W, (int)D, 1, rowbits, nullptr, img, bias, L, nullptr, status, sm_count, st);
        default: return launch_tc_nch<14, true>(Uc, W, (int)D, 1, rowbits, nullptr, img, bias, L, nullptr, status, sm_count, st);
    }
}

}  // namespace bmm
