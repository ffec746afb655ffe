// PSIS-LOO (Vehtari, Gelman & Gabry 2017; the algorithm of R's loo package, tests/loo_ref.py) over a chunk of the
// log-likelihood matrix L[g Uc + u] (draw-major, fp64) that kern_predict.cu / kern_waic_tc.cu write.  For distinct row u
// with r_g = -l_g over the D pooled draws and tail length M (M = 0 when loo would not smooth, M < 5):
//
//   cut      the (M + 1)-th largest r; the tail is the M largest r (every r > cut, then copies of cut)
//   tail     sorted ascending, lw_j = t_j - max r; unless it is flat (max - min < eps / 100), the generalized Pareto fit
//            of Zhang & Stephens (gpdfit) to x_j = exp(lw_j) - exp(cut - max r) gives k and sigma, and a finite k
//            replaces lw_j by log(qgpd((j + 0.5) / M) + exp(cut - max r)), truncated at 0
//   outputs  with S1 = sum exp(lw) and S2 = sum exp(2 lw) over all draws (non-tail draws keep lw = r - max r):
//            elpd_loo = -log S1 - max r + log(D - M + sum_tail exp(lw~_j - lw_j)), because w~ + l is the same
//            -log S1 - max r for every non-tail draw; lpd = log mean exp l; neff = S1^2 / S2 (r_eff is applied on the host)
//
// Two kernels cover the two regimes, every row independent and every sum in a fixed order (no floating-point atomics),
// so the results do not depend on the chunk or the grid size:
//   loo_short_kernel   M <= 64: one thread per row, reading the chunk coalesced twice (a heap of the M + 1 largest r in
//                      shared memory, then the sums below cut); the fit runs in fp64 registers over shared memory
//   long rows          M > 64: radix select of the (M + 1)-th largest r on order-preserving 64-bit keys, 8 bits per pass
//                      (integer histograms, several CTAs per row), a gather of the tail with per-CTA partial sums merged
//                      in block order, and one CTA per row that sorts the tail (bitonic, shared memory) and fits it
#include "kernels.h"

namespace bmm {
namespace {

constexpr double LOO_FLAT = 2.220446049250313e-16 / 100;   // R's .Machine$double.eps / 100
constexpr int SHORT_THREADS = 128;
constexpr int LONG_THREADS = 256;
constexpr int FIT_THREADS = 512;
constexpr int MAX_GRID = 30 + 128;                          // gpdfit grid points at M = LOO_MAX_TAIL

// order-preserving map of a double to uint64 (larger value, larger key) and back
__device__ __forceinline__ unsigned long long okey(double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double okey_inv(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k));
}

__device__ __forceinline__ double qgpd(double p, double k, double sigma) {
    if (sigma != sigma || sigma <= 0.0) return NAN;
    return sigma * expm1(-k * log1p(-p)) / k;
}

// gpdfit's grid point j (1-based) of m, its log-likelihood from kappa = mean log1p(-theta x), and the weakly informative
// prior adjustment of k
__device__ __forceinline__ double gpd_theta(int j, int m, double xn, double xstar) {
    return 1.0 / xn + (1.0 - sqrt((double)m / (j - 0.5))) / 3.0 / xstar;
}
__device__ __forceinline__ double gpd_lx(double theta, double kappa, int n) {
    const double a = -theta;
    return n * (log(a / kappa) - kappa - 1.0);
}
__device__ __forceinline__ double gpd_adjust(double k, int n) {
    k = k * n / (n + 10) + 10 * 0.5 / (n + 10);
    return k != k ? INFINITY : k;
}

// the smoothed, truncated log weight of tail position j of M (ascending), and its contributions e1, e2, e3
__device__ __forceinline__ void tail_terms(int j, int M, double lw, bool smooth, double k, double sigma, double ec,
                                           double &e1, double &e2, double &e3) {
    double s = lw;
    if (smooth) {
        s = log(qgpd(((double)(j + 1) - 0.5) / M, k, sigma) + ec);
        if (s > 0.0) s = 0.0;
    }
    const double e = exp(s);
    e1 += e;
    e2 += e * e;
    e3 += exp(s - lw);
}

// Row results from the row's statistics: rmax / rmin of r, cut, the sums over draws with r < cut (s_lt, s2_lt of
// exp(r - rmax) and its square, their count n_lt), s_l = sum exp(rmin - r) over all draws, and the tail sums.
__device__ __forceinline__ void loo_finish(long long D, int M, double rmax, double rmin, double cut, double s_lt,
                                           double s2_lt, double n_lt, double s_l, double e1, double e2, double e3, double k,
                                           double *elpd, double *lpd, double *khat, double *neff) {
    const double ncut = (double)D - n_lt - M;          // copies of cut outside the tail
    const double ec = exp(cut - rmax);
    const double S1 = s_lt + ncut * ec + e1, S2 = s2_lt + ncut * (ec * ec) + e2;
    double el = -log(S1) - rmax + log((double)(D - M) + e3), ne = S1 * S1 / S2;
    if (rmax == INFINITY) { el = NAN; ne = NAN; k = INFINITY; }   // some l = -inf: lw = nan, as the definition gives
    *elpd = el;
    *neff = ne;
    *khat = k;
    *lpd = rmin == INFINITY ? -INFINITY : -rmin + log(s_l) - log((double)D);
}

// ---------------------------------------------------------------------------------------------------------------------
// short rows.  Per thread, shared memory column t of H = M + 1 heap slots then M fit slots: hs[i * 128 + t].
__global__ void __maxnreg__(96) loo_short_kernel(int Uc, long long D, const double *__restrict__ L,
                                                 const int *__restrict__ Mrow, double *__restrict__ elpd,
                                                 double *__restrict__ lpd, double *__restrict__ khat,
                                                 double *__restrict__ neff) {
    extern __shared__ double hs[];
    const int t = threadIdx.x, u = blockIdx.x * SHORT_THREADS + t;
    if (u >= Uc) return;
    const int M0 = Mrow[u];
    if (M0 > LOO_SHORT_MAX_M) return;
    const int M = M0 >= 5 ? M0 : 0, H = M + 1;
    double *h = hs + t;
#define HP(i) h[(size_t)(i) * SHORT_THREADS]
    double rmax = -INFINITY, rmin = INFINITY;
    int n = 0;
    const double *col = L + u;
    for (long long g0 = 0; g0 < D; g0 += 8) {
        double v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = g0 + q < D ? __ldg(col + (size_t)(g0 + q) * Uc) : 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if (g0 + q >= D) break;
            const double r = 0.0 - v[q];
            rmax = fmax(rmax, r);
            rmin = fmin(rmin, r);
            if (n < H) {                                   // min-heap of the H largest r
                int i = n++;
                while (i > 0) {
                    const int p = (i - 1) >> 1;
                    const double pv = HP(p);
                    if (pv <= r) break;
                    HP(i) = pv;
                    i = p;
                }
                HP(i) = r;
            } else if (r > HP(0)) {
                int i = 0;
                for (;;) {
                    int c = 2 * i + 1;
                    if (c >= H) break;
                    if (c + 1 < H && HP(c + 1) < HP(c)) ++c;
                    if (HP(c) >= r) break;
                    HP(i) = HP(c);
                    i = c;
                }
                HP(i) = r;
            }
        }
    }
    const double cut = HP(0);
    double s_lt = 0.0, s2_lt = 0.0, n_lt = 0.0, s_l = 0.0;
    for (long long g0 = 0; g0 < D; g0 += 8) {
        double v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = g0 + q < D ? __ldg(col + (size_t)(g0 + q) * Uc) : 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if (g0 + q >= D) break;
            const double r = 0.0 - v[q];
            if (r < cut) {
                const double e = exp(r - rmax);
                s_lt += e;
                s2_lt += e * e;
                n_lt += 1.0;
            }
            s_l += exp(rmin - r);
        }
    }
    // heap sort: HP(0) largest ... HP(M) = cut; tail position j (ascending) is HP(M - 1 - j)
    for (int end = H - 1; end > 0; --end) {
        const double r = HP(end);
        HP(end) = HP(0);
        int i = 0;
        for (;;) {
            int c = 2 * i + 1;
            if (c >= end) break;
            if (c + 1 < end && HP(c + 1) < HP(c)) ++c;
            if (HP(c) >= r) break;
            HP(i) = HP(c);
            i = c;
        }
        HP(i) = r;
    }
    double k = INFINITY, sigma = 0.0, e1 = 0.0, e2 = 0.0, e3 = 0.0;
    bool smooth = false;
    const double ec = exp(cut - rmax);
    if (M > 0 && !(fabs((HP(0) - rmax) - (HP(M - 1) - rmax)) < LOO_FLAT)) {
        // x_j ascending in fit slot H + j
        for (int j = 0; j < M; ++j) HP(H + j) = exp(HP(M - 1 - j) - rmax) - ec;
        const int m = 30 + (int)floor(sqrt((double)M));
        const double xn = HP(H + M - 1), xstar = HP(H + (int)floor(M / 4.0 + 0.5) - 1);
        double lmx = -INFINITY, ws = 0.0, wt = 0.0;
        for (int j = 1; j <= m; ++j) {
            const double th = gpd_theta(j, m, xn, xstar), a = -th;
            double kap = 0.0;
            for (int i = 0; i < M; ++i) kap += log1p(a * HP(H + i));
            const double l = gpd_lx(th, kap / M, M);
            if (l > lmx) {
                const double sc = exp(lmx - l);
                ws = ws * sc + 1.0;
                wt = wt * sc + th;
                lmx = l;
            } else if (!(l == -INFINITY)) {
                const double e = exp(l - lmx);
                ws += e;
                wt += th * e;
            }
        }
        const double th_hat = wt / ws;
        double kk = 0.0;
        for (int i = 0; i < M; ++i) kk += log1p(-th_hat * HP(H + i));
        kk /= M;
        sigma = -kk / th_hat;
        k = gpd_adjust(kk, M);
        smooth = isfinite(k);
    }
    for (int j = 0; j < M; ++j) tail_terms(j, M, HP(M - 1 - j) - rmax, smooth, k, sigma, ec, e1, e2, e3);
#undef HP
    loo_finish(D, M, rmax, rmin, cut, s_lt, s2_lt, n_lt, s_l, e1, e2, e3, k, elpd + u, lpd + u, khat + u, neff + u);
}

// ---------------------------------------------------------------------------------------------------------------------
// long rows: row r of the chunk's long-row list is chunk row lrow[r] with tail length lM[r] and tail storage at ltoff[r].
__global__ void loo_long_init_kernel(int nlong, const int *__restrict__ lM, LooSel *__restrict__ sel, unsigned *__restrict__ hist) {
    const int r = blockIdx.x;
    if (threadIdx.x == 0) {
        LooSel s;
        s.prefix = 0ull;
        s.kmax = 0ull;
        s.kmin = ~0ull;
        s.rank = (unsigned)lM[r] + 1u;
        s.gt = 0u;
        s.tcount = 0u;
        s.pad = 0u;
        sel[r] = s;
    }
    hist[(size_t)r * 256 + threadIdx.x] = 0u;
}

__device__ __forceinline__ void long_range(long long D, int nblk, long long &g0, long long &g1) {
    const long long per = (D + nblk - 1) / nblk;
    g0 = blockIdx.y * per;
    g1 = min(D, g0 + per);
}

// digit (key >> shift) & 255 of the keys that match the selected prefix above it; pass 0 also finds max / min
__global__ void __launch_bounds__(LONG_THREADS) loo_long_hist_kernel(int pass, int Uc, long long D, int nblk,
                                                                     const double *__restrict__ L,
                                                                     const int *__restrict__ lrow, LooSel *__restrict__ sel,
                                                                     unsigned *__restrict__ hist) {
    __shared__ unsigned h[256];
    const int r = blockIdx.x, t = threadIdx.x;
    h[t] = 0u;
    __syncthreads();
    const int shift = 56 - 8 * pass;
    const unsigned long long pre = sel[r].prefix;
    const double *col = L + lrow[r];
    long long g0, g1;
    long_range(D, nblk, g0, g1);
    unsigned long long mx = 0ull, mn = ~0ull;
    for (long long g = g0 + t; g < g1; g += LONG_THREADS) {
        const unsigned long long key = okey(0.0 - col[(size_t)g * Uc]);
        if (pass == 0) {
            mx = key > mx ? key : mx;
            mn = key < mn ? key : mn;
            atomicAdd(&h[key >> 56], 1u);
        } else if (((key ^ pre) >> (shift + 8)) == 0ull) {
            atomicAdd(&h[(key >> shift) & 255u], 1u);
        }
    }
    __syncthreads();
    if (h[t]) atomicAdd(&hist[(size_t)r * 256 + t], h[t]);
    if (pass == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long a = __shfl_xor_sync(0xffffffffu, mx, o), b = __shfl_xor_sync(0xffffffffu, mn, o);
            mx = a > mx ? a : mx;
            mn = b < mn ? b : mn;
        }
        if ((t & 31) == 0) {
            atomicMax(&sel[r].kmax, mx);
            atomicMin(&sel[r].kmin, mn);
        }
    }
}

// one thread per row: the digit bin that holds the rank-th largest key; keys in higher bins are counted in gt
__global__ void loo_long_select_kernel(int pass, int nlong, LooSel *__restrict__ sel, unsigned *__restrict__ hist) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nlong) return;
    const int shift = 56 - 8 * pass;
    unsigned *hr = hist + (size_t)r * 256;
    LooSel s = sel[r];
    unsigned cum = 0u;
    for (int b = 255; b >= 0; --b) {
        const unsigned c = hr[b];
        if (cum + c >= s.rank) {
            s.prefix |= (unsigned long long)b << shift;
            s.rank -= cum;
            s.gt += cum;
            break;
        }
        cum += c;
    }
    for (int b = 0; b < 256; ++b) hr[b] = 0u;
    sel[r] = s;
}

template <int NV>
__device__ __forceinline__ void block_sum(double (&v)[NV], double *red) {   // red: NV * 32 doubles
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int e = 0; e < NV; ++e) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[e] += __shfl_xor_sync(0xffffffffu, v[e], o);
        if (lane == 0) red[e * 32 + warp] = v[e];
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < NV; ++e) {
        double a = 0.0;
        for (int w = 0; w < nw; ++w) a += red[e * 32 + w];
        v[e] = a;
    }
    __syncthreads();
}

// the draws above cut go to the row's tail storage (in any order: the fit sorts them); per CTA, the sums below cut
__global__ void __launch_bounds__(LONG_THREADS) loo_long_gather_kernel(int Uc, long long D, int nblk,
                                                                       const double *__restrict__ L,
                                                                       const int *__restrict__ lrow,
                                                                       const long long *__restrict__ ltoff,
                                                                       LooSel *__restrict__ sel, double *__restrict__ tail,
                                                                       double *__restrict__ part) {
    __shared__ double red[4 * 32];
    const int r = blockIdx.x, t = threadIdx.x;
    const unsigned long long ck = sel[r].prefix;
    const double rmax = okey_inv(sel[r].kmax), rmin = okey_inv(sel[r].kmin);
    const double *col = L + lrow[r];
    double *tr = tail + ltoff[r];
    long long g0, g1;
    long_range(D, nblk, g0, g1);
    double v[4] = {0.0, 0.0, 0.0, 0.0};
    for (long long g = g0 + t; g < g1; g += LONG_THREADS) {
        const double x = 0.0 - col[(size_t)g * Uc];
        const unsigned long long key = okey(x);
        if (key > ck) {
            tr[atomicAdd(&sel[r].tcount, 1u)] = x;
        } else if (key < ck) {
            const double e = exp(x - rmax);
            v[0] += e;
            v[1] += e * e;
            v[2] += 1.0;
        }
        v[3] += exp(rmin - x);
    }
    block_sum<4>(v, red);
    if (t == 0)
        for (int e = 0; e < 4; ++e) part[((size_t)r * nblk + blockIdx.y) * 4 + e] = v[e];
}

// one CTA per long row: sort the tail, fit, smooth, finish.  Dynamic shared memory: P2 doubles (P2 = the power of two
// >= M of the widest row of the launch); the sorted tail goes back to global memory and x takes its place.
__global__ void __maxnreg__(96) loo_long_fit_kernel(long long D, int nblk, const int *__restrict__ lrow,
                                                    const int *__restrict__ lM, const long long *__restrict__ ltoff,
                                                    const LooSel *__restrict__ sel,
                                                    const double *__restrict__ part, double *__restrict__ tail,
                                                    double *__restrict__ elpd, double *__restrict__ lpd,
                                                    double *__restrict__ khat, double *__restrict__ neff) {
    extern __shared__ double sx[];
    __shared__ double red[4 * 32];
    __shared__ double lth[MAX_GRID], thg[MAX_GRID];
    __shared__ double th_hat_s;
    const int r = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int M = lM[r];
    int P2 = 1;
    while (P2 < M) P2 <<= 1;
    const LooSel s = sel[r];
    const double cut = okey_inv(s.prefix), rmax = okey_inv(s.kmax), rmin = okey_inv(s.kmin);
    double *tr = tail + ltoff[r];
    for (int i = t; i < P2; i += FIT_THREADS) sx[i] = i < (int)s.gt ? tr[i] : (i < M ? cut : INFINITY);
    __syncthreads();
    for (int kk = 2; kk <= P2; kk <<= 1)
        for (int j = kk >> 1; j > 0; j >>= 1) {
            for (int i = t; i < P2; i += FIT_THREADS) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const double a = sx[i], b = sx[ixj];
                    if ((a > b) == ((i & kk) == 0)) { sx[i] = b; sx[ixj] = a; }
                }
            }
            __syncthreads();
        }
    const bool flat = fabs((sx[M - 1] - rmax) - (sx[0] - rmax)) < LOO_FLAT;
    const double ec = exp(cut - rmax);
    __syncthreads();
    for (int i = t; i < M; i += FIT_THREADS) {
        tr[i] = sx[i];
        sx[i] = exp(sx[i] - rmax) - ec;
    }
    __syncthreads();
    double k = INFINITY, sigma = 0.0;
    if (!flat) {
        const int m = 30 + (int)floor(sqrt((double)M));
        const double xn = sx[M - 1], xstar = sx[(int)floor(M / 4.0 + 0.5) - 1];
        for (int j = warp; j < m; j += FIT_THREADS / 32) {
            const double th = gpd_theta(j + 1, m, xn, xstar), a = -th;
            double kap = 0.0;
            for (int i = lane; i < M; i += 32) kap += log1p(a * sx[i]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) kap += __shfl_xor_sync(0xffffffffu, kap, o);
            if (lane == 0) {
                thg[j] = th;
                lth[j] = gpd_lx(th, kap / M, M);
            }
        }
        __syncthreads();
        if (t == 0) {                                     // softmax of the grid's log-likelihoods, as logSumExp does
            double lmx = -INFINITY;
            for (int j = 0; j < m; ++j) lmx = fmax(lmx, lth[j]);
            double ws = 0.0, wt = 0.0;
            for (int j = 0; j < m; ++j) {
                const double e = exp(lth[j] - lmx);
                ws += e;
                wt += thg[j] * e;
            }
            th_hat_s = wt / ws;
        }
        __syncthreads();
        const double th_hat = th_hat_s;
        double v[1] = {0.0};
        for (int i = t; i < M; i += FIT_THREADS) v[0] += log1p(-th_hat * sx[i]);
        block_sum<1>(v, red);
        const double kk = v[0] / M;
        sigma = -kk / th_hat;
        k = gpd_adjust(kk, M);
    }
    const bool smooth = !flat && isfinite(k);
    double e[3] = {0.0, 0.0, 0.0};
    for (int i = t; i < M; i += FIT_THREADS) tail_terms(i, M, tr[i] - rmax, smooth, k, sigma, ec, e[0], e[1], e[2]);
    block_sum<3>(e, red);
    if (t == 0) {
        double p[4] = {0.0, 0.0, 0.0, 0.0};
        for (int b = 0; b < nblk; ++b)
            for (int q = 0; q < 4; ++q) p[q] += part[((size_t)r * nblk + b) * 4 + q];
        const int u = lrow[r];
        loo_finish(D, M, rmax, rmin, cut, p[0], p[1], p[2], p[3], e[0], e[1], e[2], k, elpd + u, lpd + u, khat + u, neff + u);
    }
}

}  // namespace

int loo_long_blocks(long long D) {
    const long long b = (D + 8191) / 8192;
    return (int)(b < 1 ? 1 : (b > 512 ? 512 : b));
}

cudaError_t launch_loo_short(int Uc, long long D, int max_m, const double *L, const int *Mrow, double *elpd, double *lpd,
                             double *khat, double *neff, cudaStream_t st) {
    const int m = max_m >= 5 ? max_m : 0;
    const int smem = (2 * m + 1) * SHORT_THREADS * 8;
    static FuncAttrCache attr;
    if (cudaError_t e = attr.ensure_smem(loo_short_kernel, smem)) return e;
    loo_short_kernel<<<(Uc + SHORT_THREADS - 1) / SHORT_THREADS, SHORT_THREADS, smem, st>>>(Uc, D, L, Mrow, elpd, lpd, khat, neff);
    g_launches++;
    return cudaGetLastError();
}

cudaError_t launch_loo_long(int Uc, long long D, int nlong, int max_m, const double *L, const int *lrow, const int *lM,
                            const long long *ltoff, LooSel *sel, unsigned *hist, double *tail, double *part, double *elpd,
                            double *lpd, double *khat, double *neff, cudaStream_t st) {
    if (nlong < 1) return cudaSuccess;
    const int nblk = loo_long_blocks(D);
    const dim3 grid((unsigned)nlong, (unsigned)nblk);
    loo_long_init_kernel<<<nlong, 256, 0, st>>>(nlong, lM, sel, hist);
    for (int pass = 0; pass < 8; ++pass) {
        loo_long_hist_kernel<<<grid, LONG_THREADS, 0, st>>>(pass, Uc, D, nblk, L, lrow, sel, hist);
        loo_long_select_kernel<<<(nlong + 127) / 128, 128, 0, st>>>(pass, nlong, sel, hist);
    }
    loo_long_gather_kernel<<<grid, LONG_THREADS, 0, st>>>(Uc, D, nblk, L, lrow, ltoff, sel, tail, part);
    int P2 = 1;
    while (P2 < max_m) P2 <<= 1;
    static FuncAttrCache attr;
    if (cudaError_t e = attr.ensure_smem(loo_long_fit_kernel, P2 * 8)) return e;
    loo_long_fit_kernel<<<nlong, FIT_THREADS, (size_t)P2 * 8, st>>>(D, nblk, lrow, lM, ltoff, sel, part, tail, elpd, lpd,
                                                                    khat, neff);
    g_launches += 19;
    return cudaGetLastError();
}

}  // namespace bmm
