// Warp-specialised tensor-core z-sweep for K <= 32, P <= 112 (BASELINE config C4): two contractions on
// tcgen05 (loglh = X D^T; counts = [X|1]^T onehot(z)), with the work of one 128-observation tile split
// over dedicated warps connected by mbarrier rings, so the bit expansion, the tensor pipe and the
// per-observation epilogue run concurrently instead of in lockstep (the ncu profile of the earlier
// single-role kernel showed its four warpgroups convoying: ALU phase and tensor phase did not overlap).
//
//   warps 0-3    producers: packed row -> fp16 A stage (ring of NS stages) -> arrive full_A
//   warp  4      one thread issues GEMM1(k) into accumulator k % NA, tcgen05.commit publishes it
//   warp  5      one thread issues GEMM2(k) from A stage + one-hot stage; its commits free both stages
//   warps 8-19   three epilogue warpgroups (tile k goes to warpgroup k % 3): TMEM lane = observation,
//                softmax, Philox inverse-CDF draw, 1-byte allocation, one-hot row -> B2 stage
//
// Replaces /root/reference/src/full_gibbs.cpp:87-157,182-200 (stickbreaking.cpp:70-140,164-186).
#include <cstdlib>
#include <cuda_fp16.h>

#include "common.cuh"
#include "kernels.h"
#include "umma.cuh"
#include "ws_table.cuh"

namespace bmm {
namespace {

#ifndef WS_NA_CFG
#define WS_NA_CFG 4
#endif
#ifndef WS_NB_CFG
#define WS_NB_CFG 6
#endif
#ifndef WS_NEPI_CFG
#define WS_NEPI_CFG 3
#endif
constexpr int WS_NA = WS_NA_CFG;      // GEMM1 accumulators (64 TMEM columns each)
constexpr int WS_NB = WS_NB_CFG;      // one-hot stages: a multiple of WS_NEPI, so that a stage always comes back to the same warpgroup
constexpr int WS_NEPI = WS_NEPI_CFG;  // epilogue warpgroups (4 at 80 registers/thread measured no faster)
constexpr int WS_THREADS = 256 + 128 * WS_NEPI;
constexpr int WS_REP = 16;    // replicas of the count vector the CTAs flush into

// Phase stamps of the last launch (CTA 0; %globaltimer, ns): [0] entry, [1] tables loaded / pipeline start, [2] first
// tile's allocation drawn, [3] last tile drawn (epilogue warpgroup 0), [4] counts flushed, [5] exit.  Diagnostic only
// (bmm_debug_ws_trace): six timer reads per launch.
__device__ unsigned long long g_ws_trace[16];     // [sweep parity][8]
__device__ int g_ws_trace_j;
__device__ unsigned long long g_ws_cta[2 * 160];  // per CTA of the last launch: entry and "counts flushed" stamps, + SM id
__device__ __forceinline__ void ws_stamp(int slot) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_ws_trace[8 * (g_ws_trace_j & 1) + slot] = t;
}
constexpr int WS_CHUNK = 2048;
constexpr int WS_B2_BYTES = (WS_KC / 8) * WS_CHUNK;   // 8 KB

// shared memory: [A ring][B2 ring][B1 table][bias][barriers][tmem slot].  GEMM2 reads 16 chunks (M = 128)
// from an A stage that only holds NCH + 1: the rows beyond are whatever follows (other stages, one-hot
// rows, the weight table -- all finite fp16) and land in accumulator lanes that are never read.
// A stages: as many as fit (at most 9).  A stage is held from the bit expansion until GEMM2 of its tile has run, i.e.
// across the whole epilogue of that tile, so the ring has to cover ~5 tile times of latency; with the 5 stages of the
// first version the epilogue warps spent 30 % of their samples waiting for an accumulator (profiles/r01_ncu_big_sweep_ws.txt).
template <int NCH>
struct WsLayout {
    static constexpr int A_STAGE = (NCH + 1) * WS_CHUNK;
    static constexpr int FIXED = WS_NB * WS_B2_BYTES + NCH * WS_B1_ROW + WS_KC * 4 + 64 * 8 + 16;
    static constexpr int NS_FIT = (226 * 1024 - FIXED) / A_STAGE;
    static constexpr int WS_NS = NS_FIT > 9 ? 9 : NS_FIT;
    static constexpr int B2_OFF = WS_NS * A_STAGE;
    static constexpr int B1_OFF = B2_OFF + WS_NB * WS_B2_BYTES;
    static constexpr int BIAS_OFF = B1_OFF + NCH * WS_B1_ROW;
    static constexpr int BAR_OFF = BIAS_OFF + WS_KC * 4;
    static constexpr int NBAR = 2 * WS_NS + 2 * WS_NA + 2 * WS_NB + 1;
    static constexpr int TOTAL = BAR_OFF + NBAR * 8 + 16;
    static_assert(WS_NS >= 4, "too few A stages");
    static_assert(NBAR <= 64, "barrier block");
    static_assert(B1_OFF + NCH * WS_B1_ROW - (WS_NS - 1) * A_STAGE >= 16 * WS_CHUNK, "GEMM2 over-read must stay inside the operand data");
};

template <int NCH>
__global__ void __launch_bounds__(WS_THREADS, 1) big_sweep_ws_kernel(const BigParams p, const int j) {
    using L = WsLayout<NCH>;
    constexpr int WS_NS = L::WS_NS;
    extern __shared__ __align__(128) unsigned char smem[];
    const int tid = threadIdx.x, warp = tid >> 5;
    const int K = p.K, P = p.P, W = p.W;
    constexpr int ONES = NCH * 8;
    constexpr int NW = (NCH + 3) / 4;
    unsigned char *B1 = smem + L::B1_OFF;
    float *bias = (float *)(smem + L::BIAS_OFF);
    uint64_t *bars = (uint64_t *)(smem + L::BAR_OFF);
    uint32_t *tmem_slot = (uint32_t *)(bars + L::NBAR);
    const uint32_t full_a = smem_u32(bars), free_a = full_a + 8 * WS_NS;
    const uint32_t acc_full = free_a + 8 * WS_NS, acc_free = acc_full + 8 * WS_NA;
    const uint32_t b2_full = acc_free + 8 * WS_NA, b2_free = b2_full + 8 * WS_NB;
    const uint32_t all_done = b2_free + 8 * WS_NB;

    // ---- prologue ----
    if (blockIdx.x == 0 && tid == 0) { g_ws_trace_j = j; ws_stamp(0); }
    if (tid == 0 && blockIdx.x < 160) {
        unsigned long long t; unsigned sm;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
        g_ws_cta[2 * blockIdx.x] = ((t & 0x3FFFFFFFFFFFFFull) << 10) | sm;
    }
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_u32(tmem_slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 192) {
        for (int s = 0; s < WS_NS; ++s) { mbar_init(full_a + 8 * s, 128); mbar_init(free_a + 8 * s, 1); }
        for (int a = 0; a < WS_NA; ++a) { mbar_init(acc_full + 8 * a, 1); mbar_init(acc_free + 8 * a, 128); }
        for (int b = 0; b < WS_NB; ++b) { mbar_init(b2_full + 8 * b, 128); mbar_init(b2_free + 8 * b, 1); }
        mbar_init(all_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // everything above overlaps the tail of the update kernel in front (programmatic dependent launch); its
    // tables, log pi and the zeroed count buffer are needed from here on
    griddep_wait();
    // weight table: the operand image the update kernel wrote (ws_table.cuh), 16 bytes per thread and step
    for (int e = tid; e < NCH * WS_B1_ROW / 16; e += WS_THREADS) *(uint4 *)(B1 + e * 16) = __ldcg((const uint4 *)p.ws_b1 + e);
    for (int k = tid; k < WS_KC; k += WS_THREADS) {
        float b = -INFINITY;
        if (k < K) {
            const double bb = (p.lpi[k] + p.ws_s0[k]) * 1.4426950408889634;
            b = bb == bb ? (float)fmax(bb, -3.0e38) : -INFINITY;
        }
        bias[k] = b;
    }
    // the ones column of [X | 1] (chunk NCH of every A stage) and zeroed one-hot stages
    for (int e = tid; e < WS_NS * 128; e += WS_THREADS)
        *(uint4 *)(smem + (e / 128) * L::A_STAGE + NCH * WS_CHUNK + (e % 128) * 16) = make_uint4(0x3C00u, 0u, 0u, 0u);
    for (int e = tid; e < WS_NB * WS_B2_BYTES / 16; e += WS_THREADS) *(uint4 *)(smem + L::B2_OFF + e * 16) = make_uint4(0u, 0u, 0u, 0u);
    fence_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t acc2 = tmem_base + WS_NA * WS_PARTS * WS_KC;
    if (blockIdx.x == 0 && tid == 0) ws_stamp(1);
    const long long ntiles = ((long long)p.N_local + 127) / 128;
    const int T = blockIdx.x < ntiles ? (int)((ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;   // tiles of this CTA
    bool ok = true;

    if (warp < 4) {
        // ================= producers =================
        const int t = tid;
        auto load_row = [&](long long k, uint32_t (&xw)[NW]) {
            const long long i = (blockIdx.x + k * gridDim.x) * 128 + t;
#pragma unroll
            for (int w = 0; w < NW; ++w) xw[w] = 0u;
            if (k < T && i < p.N_local) {
                const uint32_t *xb = p.xbits + (size_t)i * W;
                if (NW == 2 && W == 2) { const uint2 v = *(const uint2 *)xb; xw[0] = v.x; xw[NW - 1] = v.y; }
                else {
#pragma unroll
                    for (int w = 0; w < NW; ++w) if (w < W) xw[w] = xb[w];
                }
            }
        };
        // rows of the next PF tiles are kept in flight: one tile lasts ~0.3 us, a DRAM round trip ~0.8 us
        constexpr int PF = 4;
        uint32_t ring[PF][NW];
#pragma unroll
        for (int d = 0; d < PF; ++d) load_row(d, ring[d]);
        int s = 0;
        uint32_t ph = 0;            // pass number & 1; the n-th reuse of a stage waits for completion n - 1 of its "free" barrier
        bool first_pass = true;
        for (int k0 = 0; k0 < T && ok; k0 += PF) {
#pragma unroll
            for (int d = 0; d < PF; ++d) {
                const int k = k0 + d;
                if (k >= T || !ok) break;
                // 8 bits -> 8 fp16 (0.0 / 1.0): y = byte * 0x8001 puts bit i at i and at i + 15, so (y >> 2p) & 0x10001 holds
                // bits 2p, 2p + 1 in the two halves; times 0x3C00 = fp16 1.0 (14 instructions per byte)
                uint4 ex[NCH];
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    const uint32_t y = __byte_perm(ring[d][c >> 2], 0u, 0x4440u + (c & 3)) * 0x8001u;
                    ex[c] = make_uint4((y & 0x10001u) * 0x3C00u, ((y >> 2) & 0x10001u) * 0x3C00u,
                                       ((y >> 4) & 0x10001u) * 0x3C00u, ((y >> 6) & 0x10001u) * 0x3C00u);
                }
                load_row(k + PF, ring[d]);
                if (!first_pass) ok = mbar_wait(free_a + 8 * s, ph ^ 1u);
                if (!ok) break;
                unsigned char *A = smem + s * L::A_STAGE;
#pragma unroll
                for (int c = 0; c < NCH; ++c) *(uint4 *)(A + c * WS_CHUNK + t * 16) = ex[c];
                fence_async_smem();
                mbar_arrive(full_a + 8 * s);
                if (++s == WS_NS) { s = 0; ph ^= 1u; first_pass = false; }
            }
        }
    } else if (warp == 4) {
        // ================= GEMM1 issuer =================
        // (one thread per GEMM: a single thread issuing both was the bottleneck -- ~300 dependent
        //  instructions per tile; descriptors are base + constant offset in the 16-byte address field)
        // all 32 lanes walk the loop (uniform control flow), one elected lane issues
        {
            constexpr uint32_t IDESC1 = umma_idesc_f16(128, WS_PARTS * WS_KC, 0, 0);
            const uint64_t da0 = umma_desc(smem_u32(smem), WS_CHUNK, 128), db0 = umma_desc(smem_u32(B1), WS_B1_ROW, 128);
            int s = 0, a = 0;
            uint32_t ph_s = 0, ph_a = 0;
            for (int k = 0; k < T; ++k) {
                ok = mbar_wait(full_a + 8 * s, ph_s);
                if (ok && k >= WS_NA) ok = mbar_wait(acc_free + 8 * a, ph_a ^ 1u);
                ok = __all_sync(0xffffffffu, ok);
                if (!ok) break;
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t da = da0 + (uint64_t)((s * L::A_STAGE) >> 4);
#pragma unroll
                    for (int kk = 0; kk < NCH / 2; ++kk)
                        umma_f16(tmem_base + (uint32_t)(a * WS_PARTS * WS_KC), da + (uint64_t)((kk * 2 * WS_CHUNK) >> 4),
                                  db0 + (uint64_t)((kk * 2 * WS_B1_ROW) >> 4), IDESC1, kk ? 1u : 0u);
                    umma_commit(acc_full + 8 * a);
                }
                __syncwarp();
                if (++s == WS_NS) { s = 0; ph_s ^= 1u; }
                if (++a == WS_NA) { a = 0; ph_a ^= 1u; }
            }
        }
        __syncwarp();
    } else if (warp == 5) {
        // ================= GEMM2 issuer =================
        {
            constexpr uint32_t IDESC2 = umma_idesc_f16(128, WS_KC, 1, 1);
            const uint64_t da0 = umma_desc(smem_u32(smem), 128, WS_CHUNK), db0 = umma_desc(smem_u32(smem + L::B2_OFF), 128, WS_CHUNK);
            int s = 0, b = 0;
            uint32_t ph_b = 0;
            for (int q = 0; q < T; ++q) {
                ok = __all_sync(0xffffffffu, mbar_wait(b2_full + 8 * b, ph_b));
                if (!ok) break;
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t da = da0 + (uint64_t)((s * L::A_STAGE) >> 4), db = db0 + (uint64_t)((b * WS_B2_BYTES) >> 4);
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk)
                        umma_f16(acc2, da + (uint64_t)((kk * 256) >> 4), db + (uint64_t)((kk * 256) >> 4), IDESC2, (q > 0 || kk > 0) ? 1u : 0u);
                    umma_commit(free_a + 8 * s);
                    umma_commit(b2_free + 8 * b);
                }
                __syncwarp();
                if (++s == WS_NS) s = 0;
                if (++b == WS_NB) { b = 0; ph_b ^= 1u; }
            }
            if (elect_one()) umma_commit(all_done);
        }
        __syncwarp();
    } else if (warp >= 8) {
        // ================= epilogue warpgroups =================
        const int e = (warp - 8) >> 2, t = (tid - 256) & 127, wq = warp & 3, lane = tid & 31;
        const uint32_t lane_sel = (uint32_t)(wq * 32) << 16;
        const uint2 key = make_uint2((uint32_t)p.seed, (uint32_t)p.chain_offset);
        const uint32_t sid = ST_Z ^ ((uint32_t)(p.seed >> 32) << 8);
        uint8_t *zrow = p.zhist ? p.zhist + (size_t)(p.keep_history ? j : 0) * p.N_local : nullptr;
        const float2 *bias2 = (const float2 *)bias;
        // One Philox block carries the uniforms of four consecutive observations, and a warp's 32 rows of a tile use 8
        // blocks: each lane evaluates ONE block per four tiles of its warpgroup (lane = 8 * tile slot + block) and the
        // words are handed out by shuffles, instead of every lane evaluating its own block for every tile.
        const bool shared_rng = (p.row_offset & 3) == 0;
        uint4 rnd4 = make_uint4(0u, 0u, 0u, 0u);
        // The label this thread last stored in each one-hot stage.  Tile k uses stage k % NB and warpgroup k % NEPI; only with
        // NB a multiple of NEPI is row t of a stage always written by the same thread -- with 4 stages under 3 warpgroups a
        // stage went round the warpgroups, each cleared only its own previous entry, and from the fifth tile of a CTA on the
        // rows carried stale ones into the count contraction (caught by test_grid_tensor_kernels_many_tiles_per_cta).
        unsigned long long prevz = ~0ull;
        static_assert(WS_NB <= 8 && WS_NB % WS_NEPI == 0 && WS_NB >= WS_NEPI, "prevz holds one byte per one-hot stage; stages must not migrate between warpgroups");
        int a = e % WS_NA, b = e % WS_NB;                       // tile k uses accumulator k % NA, one-hot stage k % NB
        uint32_t ph_a = (uint32_t)((e / WS_NA) & 1), ph_b = (uint32_t)((e / WS_NB) & 1);
        int it = 0;
        for (int k = e; k < T && ok; k += WS_NEPI, ++it) {
            const long long i = ((long long)blockIdx.x + (long long)k * gridDim.x) * 128 + t;
            const bool valid = i < p.N_local;
            const unsigned long long gi = (unsigned long long)p.row_offset + (unsigned long long)i;
            uint32_t uw;
            if (shared_rng) {
                if ((it & 3) == 0) {
                    const int kk = k + WS_NEPI * (lane >> 3);          // the tile this lane's block belongs to
                    const unsigned long long g0 = (unsigned long long)p.row_offset +
                        (unsigned long long)(((long long)blockIdx.x + (long long)kk * gridDim.x) * 128 + wq * 32 + 4 * (lane & 7));
                    rnd4 = philox4x32_10(make_uint4((uint32_t)(g0 >> 2), (uint32_t)(g0 >> 34), sid, (uint32_t)j), key);
                }
                const int src = 8 * (it & 3) + (lane >> 2);
                const uint32_t w0 = __shfl_sync(0xffffffffu, rnd4.x, src), w1 = __shfl_sync(0xffffffffu, rnd4.y, src);
                const uint32_t w2 = __shfl_sync(0xffffffffu, rnd4.z, src), w3 = __shfl_sync(0xffffffffu, rnd4.w, src);
                uw = (lane & 2) ? ((lane & 1) ? w3 : w2) : ((lane & 1) ? w1 : w0);
            } else {
                const uint4 rnd = philox4x32_10(make_uint4((uint32_t)(gi >> 2), (uint32_t)(gi >> 34), sid, (uint32_t)j), key);
                uw = philox_word(rnd, (int)(gi & 3));
            }
            const float u = u32_unit_f(uw);
            ok = mbar_wait(acc_full + 8 * a, ph_a);
            if (!ok) break;
            tc_fence_after();
            // logits: hi part + bias, then + lo part, two lanes of fp32 per instruction (FADD2)
            unsigned long long lp[WS_KC / 2];
            {
                uint32_t v[32];
                tmem_ld32(tmem_base + lane_sel + (uint32_t)(a * WS_PARTS * WS_KC), v);
                tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < WS_KC / 2; ++q) {
                    const float2 bq = bias2[q];
                    lp[q] = f2_add(f2_pack(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])), f2_pack(bq.x, bq.y));
                }
                tmem_ld32(tmem_base + lane_sel + (uint32_t)(a * WS_PARTS * WS_KC + WS_KC), v);
                tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < WS_KC / 2; ++q)
                    lp[q] = f2_add(lp[q], f2_pack(__uint_as_float(v[2 * q]), __uint_as_float(v[2 * q + 1])));
            }
            tc_fence_before();
            mbar_arrive(acc_free + 8 * a);      // accumulator a may be overwritten by GEMM1(k + NA)
            float l[WS_KC];
#pragma unroll
            for (int q = 0; q < WS_KC / 2; ++q) f2_unpack(lp[q], l[2 * q], l[2 * q + 1]);
            // maximum with the three-input instruction (FMNMX3): 10 + 4 + 2 instead of 31
            float mx;
            {
                float m[10];
#pragma unroll
                for (int q = 0; q < 10; ++q) m[q] = fmax3(l[3 * q], l[3 * q + 1], l[3 * q + 2]);
                const float m0 = fmax3(m[0], m[1], m[2]), m1 = fmax3(m[3], m[4], m[5]), m2 = fmax3(m[6], m[7], m[8]);
                const float m3 = fmax3(m[9], l[30], l[31]);
                mx = fmaxf(fmax3(m0, m1, m2), m3);
            }
            {
                const unsigned long long nmx = f2_pack(-mx, -mx);
#pragma unroll
                for (int q = 0; q < WS_KC / 2; ++q) { lp[q] = f2_add(lp[q], nmx); f2_unpack(lp[q], l[2 * q], l[2 * q + 1]); }
            }
            // Unnormalised probabilities e_q = 2^(l_q - max) and their prefix sums.  The draw needs
            // z = #{q : e_0 + ... + e_q <= u * total}; the prefix sums are kept per group of 8 (four independent
            // dependency chains instead of one of 32) and each group is compared with the target minus the mass
            // of the groups before it.
            float run = 0.f;
            float off[WS_KC / 8];        // mass of the groups before group g
            if (p.probs_out == nullptr && p.probs_f32 == nullptr) {
#pragma unroll
                for (int g = 0; g < WS_KC / 8; ++g) {
                    float c = 0.f;
#pragma unroll
                    for (int q = 8 * g; q < 8 * g + 8; ++q) { c += ex2_ftz(l[q]); l[q] = c; }
                }
#pragma unroll
                for (int g = 0; g < WS_KC / 8; ++g) { off[g] = run; run += l[8 * g + 7]; }
            } else {
                float sum = 0.f;
#pragma unroll
                for (int q = 0; q < WS_KC; ++q) { l[q] = ex2_ftz(l[q]); sum += l[q]; }
                const float inv = 1.f / sum;
                if (valid && p.probs_out) {
#pragma unroll
                    for (int q = 0; q < WS_KC; ++q)
                        if (q < K) p.probs_out[(size_t)j * p.N_local * K + i + (size_t)p.N_local * q] = (double)(l[q] * inv);
                }
                if (valid && p.probs_f32) {    // this observation's row of P, 16 bytes at a time when aligned
                    float *dst = p.probs_f32 + (size_t)i * K;
                    if ((K & 3) == 0) {
#pragma unroll
                        for (int q = 0; q < WS_KC; q += 4)
                            if (q < K) *(float4 *)(dst + q) = make_float4(l[q] * inv, l[q + 1] * inv, l[q + 2] * inv, l[q + 3] * inv);
                    } else {
#pragma unroll
                        for (int q = 0; q < WS_KC; ++q)
                            if (q < K) dst[q] = l[q] * inv;
                    }
                }
#pragma unroll
                for (int g = 0; g < WS_KC / 8; ++g) {
                    float c = 0.f;
#pragma unroll
                    for (int q = 8 * g; q < 8 * g + 8; ++q) { c += l[q]; l[q] = c; }
                }
#pragma unroll
                for (int g = 0; g < WS_KC / 8; ++g) { off[g] = run; run += l[8 * g + 7]; }
            }
            if (!(run > 0.f) || !isfinite(run)) *p.status = -9;  // BMM_ERR_PROB
            // d_q = (target - off_g) - c_q, two per FFMA2; its sign bit says "not counted" and is shifted into a per-group
            // mask with one funnel shift per element (a compare + select + add costs three)
            const float target = u * run;
            const unsigned long long neg1 = f2_pack(-1.f, -1.f);
            int over = 0;
#pragma unroll
            for (int g = 0; g < WS_KC / 8; ++g) {
                const float tg = target - off[g];
                const unsigned long long tg2 = f2_pack(tg, tg);
                uint32_t mask = 0u;
#pragma unroll
                for (int q = 8 * g; q < 8 * g + 8; q += 2) {
                    float d0, d1;
                    f2_unpack(f2_fma(f2_pack(l[q], l[q + 1]), neg1, tg2), d0, d1);
                    mask = __funnelshift_l(__float_as_uint(d0), mask, 1);
                    mask = __funnelshift_l(__float_as_uint(d1), mask, 1);
                }
                over += __popc(mask);
            }
            int z = min(WS_KC - over, K - 1);
            // (target - off_g) - c_q can round to >= 0 for the last cluster with weight, and then also for the clusters of
            // weight 0 after it (a pi_k = 0, or an underflowed 2^l), which would be counted too.  That takes a target within
            // a few ulp of the total, i.e. u > 1 - 2^-16 (one row in 65 536, so the check stays off the common path): the
            // draw then falls back to the last cluster with weight, found from where the group prefix sums grow.
            if (u > 0x1.fffep-1f) {
                int last = 0;
#pragma unroll
                for (int q = 0; q < WS_KC; ++q) last = l[q] > ((q & 7) ? l[q - 1] : 0.f) ? q : last;
                z = min(z, last);
            }
            if (valid && zrow) zrow[i] = (uint8_t)(z + 1);
            if (blockIdx.x == 0 && tid == 256) { if (k == 0) ws_stamp(2); if (k + WS_NEPI >= T) ws_stamp(3); }
            if (k >= WS_NB) ok = mbar_wait(b2_free + 8 * b, ph_b ^ 1u);
            if (!ok) break;
            {   // one-hot row of this observation in stage b: clear the entry this thread set there last time (the
                // stages start zeroed and row t of a stage is only ever written by this thread), set the new one
                unsigned char *row = smem + L::B2_OFF + b * WS_B2_BYTES + t * 16;
                const uint32_t pz = (uint32_t)(prevz >> (8 * b)) & 0xFFu;
                if (pz != 0xFFu) *(unsigned short *)(row + (pz >> 3) * WS_CHUNK + (pz & 7u) * 2) = 0;
                const unsigned long long nz = valid ? (unsigned long long)z : 0xFFull;
                if (valid) *(unsigned short *)(row + (z >> 3) * WS_CHUNK + (z & 7) * 2) = 0x3C00;
                prevz = (prevz & ~(0xFFull << (8 * b))) | (nz << (8 * b));
            }
            fence_async_smem();
            mbar_arrive(b2_full + 8 * b);
            a += WS_NEPI; if (a >= WS_NA) { a -= WS_NA; ph_a ^= 1u; }
            b += WS_NEPI; if (b >= WS_NB) { b -= WS_NB; ph_b ^= 1u; }
        }
    }
    griddep_launch();   // the update kernel may be scheduled as CTAs drain; it waits on the tagged inbox words
    // ---- flush the counts: TMEM lane d of acc2 holds V_kd (d < P) or c_k (d == ONES) ----
    if (warp >= 8 && warp < 12) {
        const int t = tid - 256;
        if (ok && T > 0) ok = mbar_wait(all_done, 0u);
        if (ok && T > 0) {
            tc_fence_after();
            // The CTA's counts are staged in shared memory (the A ring is idle by now) in the layout of the count
            // vector, c_k then V_kd at K + k + K d, and added to global memory by ONE bulk reduction below.
            int *stage = (int *)smem;
            uint32_t v[32];
            tmem_ld32(acc2 + ((uint32_t)((warp & 3) * 32) << 16), v);
            tmem_ld_wait();
            if (t < P || t == ONES) {
#pragma unroll
                for (int q = 0; q < 32; ++q) {
                    const int n = (int)(__uint_as_float(v[q]) + 0.5f);
                    if (q < K) stage[t == ONES ? q : K + q + K * t] = n;
                }
            }
            fence_async_smem();
        }
    }
    if (!ok) *p.status = -10;  // BMM_ERR_TIMEOUT
    tc_fence_before();
    __syncthreads();
    if (blockIdx.x == 0 && tid == 0) ws_stamp(4);
    if (tid == 0 && blockIdx.x < 160) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_ws_cta[2 * blockIdx.x + 1] = t;
    }
    // ---- the last CTA to get here sums the replicas into the count vector and, in inbox mode, pushes the sums as
    //      tagged words into every rank's inbox (its own included) ----
    {
        __shared__ int last_sh;
        // Every CTA adds its counts to one of WS_REP replicas of the count vector with a single cp.reduce.async.bulk
        // (UBLKRED: the copy engine performs the additions at the L2 in 16-byte pieces).  The first version issued 2080
        // scalar atomics per CTA into ONE copy: all 148 CTAs hit the same 65 cache lines at the same moment and the
        // fence behind them took 13 us per launch (7.6 us with 16 replicas), measured with the phase stamps.
        if (tid == 0) {
            const int n = K + K * P, nstride = (n + 3) & ~3;
            int *rep = p.ws_rep + (size_t)(blockIdx.x % WS_REP) * nstride;
            if (ok && T > 0) {
                const int nb = (n & ~3) * 4;
                if (nb) {
                    asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.s32 [%0], [%1], %2;"
                                 :: "l"(rep), "r"(smem_u32(smem)), "r"(nb) : "memory");
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
                for (int e = n & ~3; e < n; ++e) atomicAdd(&rep[e], ((const int *)smem)[e]);
                asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            }
            __threadfence();             // this CTA's additions are performed before its ticket
            if (blockIdx.x == 0) ws_stamp(6);
            const unsigned ticket = atomicAdd(p.x_done, 1u);
            last_sh = ticket == gridDim.x - 1;
            if (last_sh) *p.x_done = 0u;         // ready for the next launch (stream order)
        }
        __syncthreads();
        if (blockIdx.x == 0 && tid == 0) ws_stamp(7);
        if (last_sh) {
            __threadfence();
            const int n = K + K * P, nstride = (n + 3) & ~3, world = p.x_world, s = world >= 1 ? p.x_seq[0] + j : 0;
            int *gcnt = p.counts + (size_t)(j & 1) * n;
            const size_t off = world >= 1 ? x_slot_off(s, world, p.x_rank, (size_t)p.x_cap) : 0;
            // this is a serial step of the whole GPU: four elements per thread with all their replica loads in flight at once
            // (64 independent L2 loads), not one dependent round trip after another
            for (int e0 = tid; e0 < n; e0 += 4 * WS_THREADS) {
                int v[4] = {0, 0, 0, 0};
#pragma unroll
                for (int r = 0; r < WS_REP; ++r)
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int e = e0 + q * WS_THREADS;
                        if (e < n) v[q] += __ldcg(p.ws_rep + (size_t)r * nstride + e);
                    }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int e = e0 + q * WS_THREADS;
                    if (e < n) {
                        gcnt[e] = v[q];
                        for (int r = 0; r < world; ++r) x_store(p.x_peer[r] + off + e, v[q], s);   // (count, tag) in one 8-byte store
                    }
                }
#pragma unroll
                for (int r = 0; r < WS_REP; ++r)
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int e = e0 + q * WS_THREADS;
                        if (e < n) p.ws_rep[(size_t)r * nstride + e] = 0;          // zero for the next sweep
                    }
            }
        }
    }
    if (blockIdx.x == 0 && tid == 0) ws_stamp(5);
    if (warp == 4) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(512) : "memory");
    }
}

template <int NCH>
cudaError_t launch_ws_nch(const BigParams &p, int j, int sm_count, cudaStream_t st) {
    using L = WsLayout<NCH>;
    static FuncAttrCache attr;
    if (cudaError_t e = attr.ensure_smem(big_sweep_ws_kernel<NCH>, (int)L::TOTAL)) return e;
    const long long ntiles = ((long long)p.N_local + 127) / 128;
    long long ctas = ntiles < sm_count ? ntiles : sm_count;
    if (const char *e = getenv("BMM_GRID_MAX_CTAS")) { const int cap = atoi(e); if (cap > 0 && ctas > cap) ctas = cap; }   // tests: many tiles per CTA
    if (ctas < 1) ctas = 1;
    g_launches++;
    return launch_pdl(big_sweep_ws_kernel<NCH>, dim3((unsigned)ctas), dim3(WS_THREADS), (size_t)L::TOTAL, st, p, j);
}

}  // namespace

bool big_tc_supported(const BigParams &p) {
    return p.precision == 1 && p.K <= 32 && p.P <= 112 && p.W <= 4 && p.ru == nullptr && p.loglik_out == nullptr;
}

size_t ws_b1_bytes(int P) { return (size_t)ws_nch(P) * WS_B1_ROW; }
size_t ws_rep_bytes(int K, int P) { return (size_t)WS_REP * (((size_t)K + (size_t)K * P + 3) & ~(size_t)3) * sizeof(int); }

cudaError_t ws_cta_read(unsigned long long out[320]) { return cudaMemcpyFromSymbol(out, g_ws_cta, 320 * sizeof(unsigned long long)); }
cudaError_t ws_trace_read(unsigned long long out[16]) { return cudaMemcpyFromSymbol(out, g_ws_trace, 16 * sizeof(unsigned long long)); }

cudaError_t launch_big_sweep_ws(const BigParams &p, int j, int sm_count, cudaStream_t st) {
    if (!p.ws_b1 || !p.ws_s0) return cudaErrorInvalidValue;
    switch (ws_nch(p.P)) {
        case 2: return launch_ws_nch<2>(p, j, sm_count, st);
        case 4: return launch_ws_nch<4>(p, j, sm_count, st);
        case 6: return launch_ws_nch<6>(p, j, sm_count, st);
        case 8: return launch_ws_nch<8>(p, j, sm_count, st);
        case 10: return launch_ws_nch<10>(p, j, sm_count, st);
        case 12: return launch_ws_nch<12>(p, j, sm_count, st);
        default: return launch_ws_nch<14>(p, j, sm_count, st);
    }
}

}  // namespace bmm
