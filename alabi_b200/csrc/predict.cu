// K3: batched GP prediction over M query points, and K4: fused acquisition
// utilities + argmin.
//
// Replaces george GP.predict(y, X*, return_var) as alabi calls it
// (alabi/core.py:85,95,1441,1486,1601,1812) and the per-point scipy loops over
// bape/agp/jones_utility (alabi/utility.py:629-946, core.py:1587-1667).
//
//   mean      mu_q = amp * sum_j k(x*_q, x_j) alpha_j + mean.  The cross
//             covariance is built on the fly: training points are staged in
//             shared memory, every thread keeps two query points in registers.
//   variance  sigma^2_q = amp - | L^-1 k*_q |^2.  Pass 1 also stores the cross
//             covariance panel P[j][q] (query index contiguous, coalesced);
//             pass 2 is a DMMA GEMM  L^-1 (N x N, lower) x P (N x 128)  per CTA
//             whose epilogue squares and column-reduces the product in
//             registers; nothing but sigma^2 is written back.  White noise is
//             not added (george semantics).
//   few       m <= 8 queries (the reference's M = 1 calls inside optimisers and samplers):
//             few_* kernels spread one query over the GPU and reproduce the batched
//             kernels' summation order, so a query has the same bits in any batch.
#include <float.h>
#include <algorithm>
#include "handle.h"
#include "dmma_gemm.cuh"

namespace {

constexpr int NB = AB_NB;
constexpr int TS = 128;        // training points per shared-memory tile
constexpr int QPB = 256;       // queries per CTA (128 threads x 2)
constexpr int JCHUNK = 512;    // training points per grid.y slice (fixed: results do not depend on batching)

template <int KIND, int D, bool STORE>
__global__ void __launch_bounds__(128)
predict_mean_kernel(const double* __restrict__ Xq, int64_t m, int64_t q_off, const double* __restrict__ Xs,
                    const double* __restrict__ alpha, int64_t n, int64_t npad, KernParams kp, double mean,
                    double* __restrict__ mu, double* __restrict__ P, int64_t ldp, int nsplit,
                    double* __restrict__ partial, int64_t part_ld) {
    __shared__ __align__(16) double sX[TS * D];
    __shared__ double sAl[TS];
    const int tid = threadIdx.x, d = kp.d;
    const int64_t qa = (int64_t)blockIdx.x * QPB + tid, qb = qa + 128;   // local to this panel
    double xa[D], xb[D];
#pragma unroll
    for (int k = 0; k < D; k++) {
        xa[k] = (k < d && q_off + qa < m) ? Xq[(q_off + qa) * d + k] * kp.inv_len[k] : 0.0;
        xb[k] = (k < d && q_off + qb < m) ? Xq[(q_off + qb) * d + k] * kp.inv_len[k] : 0.0;
    }
    // training range of this split
    const int64_t jtot = STORE ? npad : n;      // the panel also needs the (zero) padding rows
    int64_t jbeg = 0, jend = jtot;
    if (nsplit > 1) {            // fixed chunks of JCHUNK training points: the summation order
        jbeg = (int64_t)blockIdx.y * JCHUNK;     // depends on N only, never on the batch size
        jend = jbeg + JCHUNK < jtot ? jbeg + JCHUNK : jtot;
    }
    double ma = 0.0, mb = 0.0;
    for (int64_t j0 = jbeg; j0 < jend; j0 += TS) {
        __syncthreads();
        for (int idx = tid; idx < TS * D; idx += 128) {
            int jj = idx / D, k = idx - jj * D;
            sX[idx] = (k < d && j0 + jj < npad) ? Xs[(j0 + jj) * d + k] : 0.0;
        }
        if (tid < TS) sAl[tid] = (j0 + tid < n) ? alpha[j0 + tid] : 0.0;
        __syncthreads();
        const int tn = (int)((jend - j0 < TS) ? (jend - j0) : TS);
        for (int jj = 0; jj < tn; jj++) {
            double ra = 0.0, rb = 0.0;
#pragma unroll
            for (int k = 0; k < D; k += 2) {
                double2 x = *reinterpret_cast<const double2*>(&sX[jj * D + k]);
                double da0 = xa[k] - x.x, da1 = xa[k + 1] - x.y;
                double db0 = xb[k] - x.x, db1 = xb[k + 1] - x.y;
                ra = fma(da0, da0, ra); ra = fma(da1, da1, ra);
                rb = fma(db0, db0, rb); rb = fma(db1, db1, rb);
            }
            double ka = ab_radial<KIND>(ra, kp.alpha, kp.inv2a), kb = ab_radial<KIND>(rb, kp.alpha, kp.inv2a);
            const double al = sAl[jj];
            ma = fma(ka, al, ma);
            mb = fma(kb, al, mb);
            if (STORE) {
                const bool valid = (j0 + jj) < n;
                P[(j0 + jj) * ldp + qa] = valid ? kp.amp * ka : 0.0;
                P[(j0 + jj) * ldp + qb] = valid ? kp.amp * kb : 0.0;
            }
        }
    }
    if (nsplit > 1) {
        partial[(int64_t)blockIdx.y * part_ld + qa] = ma;
        partial[(int64_t)blockIdx.y * part_ld + qb] = mb;
    } else {
        if (q_off + qa < m) mu[q_off + qa] = fma(kp.amp, ma, mean);
        if (q_off + qb < m) mu[q_off + qb] = fma(kp.amp, mb, mean);
    }
}

// mu[q_off + q] = amp * sum_splits partial[split][q] + mean  for q < cnt (fixed order)
__global__ void combine_splits_kernel(const double* __restrict__ partial, int64_t part_ld, int64_t cnt, int nsplit,
                                      double amp, double mean, double* __restrict__ mu, int64_t q_off) {
    int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= cnt) return;
    double s = 0.0;
    for (int p = 0; p < nsplit; p++) s += partial[(int64_t)p * part_ld + q];
    mu[q_off + q] = fma(amp, s, mean);
}

// Per-thread sums of squares of one 128 x 128 product tile: blk[j][e] = sum over the 8
// m-fragments of acc^2 (a chain that starts at zero for every row block).
__device__ __forceinline__ void tile_thread_sq(const abg::Acc& acc, double (&blk)[4][2]) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
        blk[j][0] = blk[j][1] = 0.0;
#pragma unroll
        for (int a = 0; a < 8; a++) {
            blk[j][0] = fma(acc.v[a][j][0], acc.v[a][j][0], blk[j][0]);
            blk[j][1] = fma(acc.v[a][j][1], acc.v[a][j][1], blk[j][1]);
        }
    }
}

// sigma^2 of the 128 queries of a tile from the per-thread totals: shuffle tree over the
// 8 row groups of a warp, then the two warp rows through shared memory (`red`: 256 doubles).
__device__ __forceinline__ void tile_finish_var(double (&tot)[4][2], double* red, int64_t q, int64_t m, double amp,
                                                double* __restrict__ var) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < 4; j++)
#pragma unroll
        for (int e = 0; e < 2; e++) {
            double v = tot[j][e];
            v += __shfl_xor_sync(0xffffffffu, v, 4);
            v += __shfl_xor_sync(0xffffffffu, v, 8);
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            tot[j][e] = v;
        }
    if (lane < 4) {
#pragma unroll
        for (int j = 0; j < 4; j++)
#pragma unroll
            for (int e = 0; e < 2; e++) red[(warp >> 2) * 128 + (warp & 3) * 32 + j * 8 + lane * 2 + e] = tot[j][e];
    }
    __syncthreads();
    if (threadIdx.x < 128 && q < m) var[q] = amp - (red[threadIdx.x] + red[128 + threadIdx.x]);
}

// Per-thread block values (tile_thread_sq) of row block i of L^-1 P for the query tile at Bp.
// NL = number of 8-row groups of the LAST row block (last = true) that hold training points (rows
// >= n of L^-1 are identity padding and k* is zero there, so their products are exactly zero and
// skipping them changes no bit of the result).
template <int NL>
__device__ __forceinline__ void var_row_block(const double* __restrict__ Linv, int64_t ld, int i, bool last,
                                              const double* __restrict__ Bp, int64_t ldp, double* smem,
                                              double (&blk)[4][2]) {
    abg::Acc acc;
    acc.zero();
    if (NL < 16 && last)
        abg::Main::mainloop<true, false, true, abg::NoGate, NL>(acc, Linv + (int64_t)i * NB * ld, ld, Bp, ldp,
                                                               (i + 1) * (NB / abg::BK), smem);
    else
        abg::mainloop<true, false, true>(acc, Linv + (int64_t)i * NB * ld, ld, Bp, ldp, (i + 1) * (NB / abg::BK), smem);
    tile_thread_sq(acc, blk);
}

// the 8 block values of this thread for one (row block, query tile) item of the split schedules,
// where var_combine_kernel reads them
__device__ __forceinline__ void store_part(double* __restrict__ part, int64_t item, const double (&blk)[4][2]) {
    double* dst = part + (item * abg::THREADS + threadIdx.x) * 8;
#pragma unroll
    for (int j = 0; j < 4; j++) *reinterpret_cast<double2*>(dst + 2 * j) = make_double2(blk[j][0], blk[j][1]);
}

// sigma^2 for the 128 queries of this CTA:  amp - sum_i ( sum_k Linv[i][k] P[k][q] )^2.
// Canonical summation order (shared with the split path below, so both give identical
// bits): per thread, per row block a chain over the m-fragments starting at zero; the
// block values added in block order; then the reduction tree of tile_finish_var.
template <int NL>
__global__ void __launch_bounds__(abg::THREADS, 1)
predict_var_kernel(const double* __restrict__ Linv, int64_t ld, int T, const double* __restrict__ P, int64_t ldp,
                   int64_t m, int64_t q_off, double amp, double* __restrict__ var) {
    extern __shared__ __align__(16) double smem[];
    const double* Bp = P + (int64_t)blockIdx.x * abg::BN;
    double tot[4][2];
#pragma unroll
    for (int j = 0; j < 4; j++) tot[j][0] = tot[j][1] = 0.0;
    for (int i = 0; i < T; i++) {
        double blk[4][2];
        var_row_block<NL>(Linv, ld, i, i == T - 1, Bp, ldp, smem, blk);
#pragma unroll
        for (int j = 0; j < 4; j++) { tot[j][0] += blk[j][0]; tot[j][1] += blk[j][1]; }
    }
    tile_finish_var(tot, smem, q_off + (int64_t)blockIdx.x * abg::BN + threadIdx.x, m, amp, var);
}

// Few query tiles (one-point calls of the acquisition polish, small batches): the loop
// over row blocks of predict_var_kernel would run serially on a handful of SMs, so the
// row blocks are spread over grid.y.  Each CTA stores its per-thread block values
// (8 per thread); var_combine_kernel adds them in block order and finishes exactly like
// predict_var_kernel.
__global__ void __launch_bounds__(abg::THREADS, 1)
predict_var_split_kernel(const double* __restrict__ Linv, int64_t ld, const double* __restrict__ P, int64_t ldp,
                         double* __restrict__ part) {
    extern __shared__ __align__(16) double smem[];
    const int i = blockIdx.y;
    double blk[4][2];
    var_row_block<16>(Linv, ld, i, false, P + (int64_t)blockIdx.x * abg::BN, ldp, smem, blk);
    store_part(part, (int64_t)i * gridDim.x + blockIdx.x, blk);
}

// Full panels with many row blocks: predict_var_kernel gives one CTA the whole row-block loop of its
// 128 queries, so the CTA streams its own 128-column slice of the panel (N x 128 x 8 B = 8 MB at
// N = 8192) once per row block, and 148 such slices do not fit the L2: ncu shows 40 GB of DRAM
// reads per 18 944-query wave against 1.5 GB of algorithmic bytes.  Here the work of ONE query tile
// is spread over ceil(T / 2) CTAs that are ADJACENT in launch order (blockIdx.x = row-block pair
// (p, T - 1 - p): T + 1 k blocks each, so all CTAs carry equal work), so the few tiles in flight
// share their panel slices through the L2 and L^-1 is streamed once per group of tiles.  Per-thread
// block values go to `part` exactly like predict_var_split_kernel; var_combine_kernel finishes in
// the canonical order, so the bits equal predict_var_kernel's.
template <int NL>
__global__ void __launch_bounds__(abg::THREADS, 1)
predict_var_pair_kernel(const double* __restrict__ Linv, int64_t ld, int T, int ntq, const double* __restrict__ P,
                        int64_t ldp, double* __restrict__ part) {
    extern __shared__ __align__(16) double smem[];
    // persistent: one CTA per SM walks the (tile, pair) items round-robin, pair index fastest, so the
    // CTAs that run at the same time work on neighbouring items = the same few query tiles
    const int npairs = (T + 1) / 2;
    const long long nitems = (long long)npairs * ntq;
    for (long long item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int p = (int)(item % npairs), q = (int)(item / npairs);
        const double* Bp = P + (int64_t)q * abg::BN;
        for (int h = 0; h < 2; h++) {
            const int i = (h == 0) ? p : T - 1 - p;
            if (h == 1 && i == p) break;                         // middle row block of an odd T
            double blk[4][2];
            var_row_block<NL>(Linv, ld, i, i == T - 1, Bp, ldp, smem, blk);
            store_part(part, (int64_t)i * ntq + q, blk);
        }
    }
}

// one CTA (256 threads) per query tile
__global__ void __launch_bounds__(abg::THREADS)
var_combine_kernel(const double* __restrict__ part, int T, int64_t m, int64_t q_off, double amp,
                   double* __restrict__ var) {
    __shared__ double red[256];
    double tot[4][2];
#pragma unroll
    for (int j = 0; j < 4; j++) tot[j][0] = tot[j][1] = 0.0;
    for (int i = 0; i < T; i++) {
        const double* src = part + (((int64_t)i * gridDim.x + blockIdx.x) * abg::THREADS + threadIdx.x) * 8;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const double2 v = *reinterpret_cast<const double2*>(src + 2 * j);
            tot[j][0] += v.x;
            tot[j][1] += v.y;
        }
    }
    tile_finish_var(tot, red, q_off + (int64_t)blockIdx.x * abg::BN + threadIdx.x, m, amp, var);
}

// ---------------------------------------------------------------------------
// Gradients of the predictive mean and variance w.r.t. the query point
// (alabi/utility.py:558-621 `grad_gp_mean_prediction` / `grad_gp_var_prediction`,
// which difference the kernel numerically and form a dense K^-1 per call):
//   d mu / dx      =        sum_j alpha_j        d k*_j / dx
//   d sigma^2 / dx = -2     sum_j (K^-1 k*)_j    d k*_j / dx
//   d k*_j / dx_k  = amp k'(r^2) 2 (x_k - x_jk) / M_k          (analytic)
// K^-1 k* for a panel of queries is two triangular DMMA GEMMs with L^-1.
// ---------------------------------------------------------------------------
// C(i, q-tile) = sum_k op(Linv)(i, k) B(k, q-tile);  TRANS = false: Linv (k <= i, diagonal
// block triangular), TRANS = true: Linv^T (k >= i).  B, C: [row][query], query contiguous.
template <bool TRANS>
__global__ void __launch_bounds__(abg::THREADS, 1)
tri_gemm_kernel(const double* __restrict__ Linv, int64_t ld, int T, const double* __restrict__ B, int64_t ldb,
                double* __restrict__ C) {
    extern __shared__ __align__(16) double smem[];
    const int i = blockIdx.y;
    const double* Bp = B + (int64_t)blockIdx.x * abg::BN;
    abg::Acc acc;
    acc.zero();
    if (!TRANS)
        abg::mainloop<true, false, true>(acc, Linv + (int64_t)i * NB * ld, ld, Bp, ldb, (i + 1) * (NB / abg::BK), smem);
    else
        abg::mainloop<false, false>(acc, Linv + (int64_t)i * NB * ld + (int64_t)i * NB, ld, Bp + (int64_t)i * NB * ldb, ldb,
                                    (T - i) * (NB / abg::BK), smem);
    abg::store_tile(acc, C + (int64_t)i * NB * ldb + (int64_t)blockIdx.x * abg::BN, ldb, 1.0, 0.0);
}

// one query per thread; partial[(split * 2D + k) * part_ld + q] = sum over the split's
// training points of alpha_j g_j diff_k (k < D) and V_jq g_j diff_k (D <= k < 2D)
template <int KIND, int D>
__global__ void __launch_bounds__(128)
predict_grad_kernel(const double* __restrict__ Xq, int64_t m, int64_t q_off, const double* __restrict__ Xs,
                    const double* __restrict__ alpha, const double* __restrict__ V, int64_t ldp, int64_t n,
                    int64_t npad, KernParams kp, double* __restrict__ partial, int64_t part_ld) {
    __shared__ __align__(16) double sX[TS * D];
    __shared__ double sAl[TS];
    const int tid = threadIdx.x, d = kp.d;
    const int64_t q = (int64_t)blockIdx.x * 128 + tid;
    double x[D], gm[D], gv[D];
#pragma unroll
    for (int k = 0; k < D; k++) {
        x[k] = (k < d && q_off + q < m) ? Xq[(q_off + q) * d + k] * kp.inv_len[k] : 0.0;
        gm[k] = gv[k] = 0.0;
    }
    const int64_t jbeg = (int64_t)blockIdx.y * JCHUNK;
    const int64_t jend = jbeg + JCHUNK < n ? jbeg + JCHUNK : n;
    for (int64_t j0 = jbeg; j0 < jend; j0 += TS) {
        __syncthreads();
        for (int idx = tid; idx < TS * D; idx += 128) {
            int jj = idx / D, k = idx - jj * D;
            sX[idx] = (k < d && j0 + jj < npad) ? Xs[(j0 + jj) * d + k] : 0.0;
        }
        if (tid < TS) sAl[tid] = (j0 + tid < n) ? alpha[j0 + tid] : 0.0;
        __syncthreads();
        const int tn = (int)((jend - j0 < TS) ? (jend - j0) : TS);
        for (int jj = 0; jj < tn; jj++) {
            double df[D], r2 = 0.0;
#pragma unroll
            for (int k = 0; k < D; k++) {
                df[k] = x[k] - sX[jj * D + k];
                r2 = fma(df[k], df[k], r2);
            }
            const double g = ab_radial_grad<KIND>(r2, kp.alpha, kp.inv2a);
            const double c1 = sAl[jj] * g, c2 = V[(j0 + jj) * ldp + q] * g;
#pragma unroll
            for (int k = 0; k < D; k++) {
                gm[k] = fma(c1, df[k], gm[k]);
                gv[k] = fma(c2, df[k], gv[k]);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < D; k++) {
        partial[((int64_t)blockIdx.y * 2 * D + k) * part_ld + q] = gm[k];
        partial[((int64_t)blockIdx.y * 2 * D + D + k) * part_ld + q] = gv[k];
    }
}

__global__ void grad_combine_kernel(const double* __restrict__ partial, int64_t part_ld, int64_t cnt, int nsplit, int D,
                                    int d, KernParams kp, double* __restrict__ dmu, double* __restrict__ dvar,
                                    int64_t q_off) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= cnt * d) return;
    const int64_t q = idx / d;
    const int k = (int)(idx - q * d);
    double sm = 0.0, sv = 0.0;
    for (int p = 0; p < nsplit; p++) {
        sm += partial[((int64_t)p * 2 * D + k) * part_ld + q];
        sv += partial[((int64_t)p * 2 * D + D + k) * part_ld + q];
    }
    const double f = 2.0 * kp.amp * kp.inv_len[k];
    dmu[(q_off + q) * d + k] = f * sm;
    dvar[(q_off + q) * d + k] = -2.0 * f * sv;
}

// ---------------------------------------------------------------------------
// K4 utilities.  Expression order follows the reference exactly
// (alabi/utility.py:489-504, 696, 804, 926-939).
// ---------------------------------------------------------------------------
struct UtilParams {
    int kind, d;                  // 0 bape, 1 agp, 2 jones
    double y_best, zeta;
    double lo[AB_MAX_DIM], hi[AB_MAX_DIM];
};

__device__ __forceinline__ double utility_value(const UtilParams& up, double mu, double var) {
    if (up.kind == 0) {
        double lse = (var <= 0.0) ? -INFINITY : var + log(1.0 - exp(0.0 - var));
        return -((2.0 * mu + var) + lse);
    }
    if (up.kind == 1) return -(mu + 0.5 * log(2.0 * 3.141592653589793 * 2.718281828459045 * var));
    double sd = sqrt(var);
    if (!(sd > 0.0)) return 0.0;
    double dd = mu - up.y_best - up.zeta;
    double z = dd / sd;
    double cdf = 0.5 * erfc(-z * 0.7071067811865476);
    double pdf = exp(-(z * z) / 2.0) / 2.5066282746310002;
    return -(dd * cdf + sd * pdf);
}

__global__ void __launch_bounds__(256)
utility_kernel(const double* __restrict__ Xq, const double* __restrict__ mu, const double* __restrict__ var,
               int64_t m, UtilParams up, double* __restrict__ util, double* __restrict__ bval,
               long long* __restrict__ bidx) {
    __shared__ double sv[8];
    __shared__ long long si[8];
    int64_t q = (int64_t)blockIdx.x * 256 + threadIdx.x;
    double u = INFINITY;
    if (q < m) {
        bool inside = true;
        for (int k = 0; k < up.d; k++) {
            double x = Xq[q * up.d + k];
            inside = inside && (x > up.lo[k]) && (x < up.hi[k]);     // strict, like lnprior_uniform
        }
        u = inside ? utility_value(up, mu[q], var[q]) : INFINITY;
        if (util) util[q] = u;
    }
    // argmin over finite values, lowest index on ties
    double bv = (q < m && isfinite(u)) ? u : INFINITY;
    long long bi = (q < m && isfinite(u)) ? (long long)q : -1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        double ov = __shfl_xor_sync(0xffffffffu, bv, o);
        long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi >= 0 && (bi < 0 || ov < bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = bv; si[threadIdx.x >> 5] = bi; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; w++)
            if (si[w] >= 0 && (bi < 0 || sv[w] < bv || (sv[w] == bv && si[w] < bi))) { bv = sv[w]; bi = si[w]; }
        bval[blockIdx.x] = bv;
        bidx[blockIdx.x] = bi;
    }
}

__global__ void __launch_bounds__(256)
argmin_final_kernel(const double* __restrict__ bval, const long long* __restrict__ bidx, int nb,
                    double* __restrict__ out_val, long long* __restrict__ out_idx) {
    __shared__ double sv[256];
    __shared__ long long si[256];
    double bv = INFINITY;
    long long bi = -1;
    for (int p = threadIdx.x; p < nb; p += 256) {
        double ov = bval[p];
        long long oi = bidx[p];
        if (oi >= 0 && (bi < 0 || ov < bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    sv[threadIdx.x] = bv;
    si[threadIdx.x] = bi;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 256; w++)
            if (si[w] >= 0 && (bi < 0 || sv[w] < bv || (sv[w] == bv && si[w] < bi))) { bv = sv[w]; bi = si[w]; }
        *out_val = bv;
        *out_idx = bi;
    }
}

// ---------------------------------------------------------------------------
// Few queries (m <= FEW_MQ: the one-point calls of the acquisition polish, host-driven
// samplers).  The batched kernels above give one query to one THREAD (mean) and 128 queries
// to one DMMA tile (variance), so a single query costs as much as 256 / 128 of them and runs
// as long serial chains: 225 us at N = 1000, 670 us at N = 4000.  This path spreads ONE
// query over the machine and reproduces the batched kernels' operations in their canonical
// order, so a query keeps identical bits in any batch:
//   few_cross_kernel   one training point per thread: k*_j for every query (same r^2 chain,
//                      same radial function), panel P[j][q]; then one thread per query runs
//                      the 512-point FMA chain of its split from shared memory
//   few_gemv_kernel    z = L^-1 k*: one warp per 32 rows, lane = row, sequential FMA chain over
//                      k ascending -- the order in which DMMA.8x8x4 accumulates a row of the
//                      product (k4-steps in order, k0..k3 chained inside an instruction)
//   few_finish_kernel  squares of z summed exactly like tile_thread_sq / tile_finish_var
//                      (per (warp row, row group): chain over the 8 m-fragments per row
//                      block, blocks in order, xor tree over the row groups, warp rows 0 + 1),
//                      and the split sums of the mean in split order
// ---------------------------------------------------------------------------
constexpr int FEW_MQ = 8;
constexpr int FEW_ST = 4;                           // cp.async ring depth of few_gemv_kernel (8 stages measured: no gain, the warp is issue / chain bound)
constexpr int FEW_GEMV_SMEM = FEW_ST * (32 * 34 + 32 * FEW_MQ) * 8;

template <int KIND, int D>
__global__ void __launch_bounds__(JCHUNK)
few_cross_kernel(const double* __restrict__ Xq, int m, const double* __restrict__ Xs, const double* __restrict__ alpha,
                 int64_t n, int64_t npad, KernParams kp, double* __restrict__ P, double* __restrict__ partial) {
    __shared__ double sQ[FEW_MQ][D];
    __shared__ double sK[FEW_MQ][JCHUNK];
    __shared__ double sAl[JCHUNK];
    const int tid = threadIdx.x, d = kp.d;
    const int64_t j = (int64_t)blockIdx.x * JCHUNK + tid;
    if (tid < FEW_MQ * D) {
        const int q = tid / D, k = tid - q * D;
        sQ[q][k] = (k < d && q < m) ? Xq[(int64_t)q * d + k] * kp.inv_len[k] : 0.0;
    }
    double x[D];
#pragma unroll
    for (int k = 0; k < D; k++) x[k] = (k < d && j < npad) ? Xs[j * d + k] : 0.0;
    sAl[tid] = (j < n) ? alpha[j] : 0.0;
    __syncthreads();
    for (int q = 0; q < FEW_MQ; q++) {
        double kq = 0.0;
        if (q < m) {
            double r = 0.0;
#pragma unroll
            for (int k = 0; k < D; k++) {
                const double df = sQ[q][k] - x[k];
                r = fma(df, df, r);
            }
            kq = ab_radial<KIND>(r, kp.alpha, kp.inv2a);
        }
        sK[q][tid] = kq;
        if (P && j < npad) P[j * FEW_MQ + q] = (q < m && j < n) ? kp.amp * kq : 0.0;
    }
    __syncthreads();
    if (tid < m) {
        const int64_t jtot = P ? npad : n;          // as predict_mean_kernel: the panel pass also walks the padding
        const int64_t jbeg = (int64_t)blockIdx.x * JCHUNK;
        const int tn = (int)((jtot - jbeg < JCHUNK) ? (jtot - jbeg) : JCHUNK);
        double ma = 0.0;
        for (int jj = 0; jj < tn; jj++) ma = fma(sK[tid][jj], sAl[jj], ma);
        partial[(int64_t)blockIdx.x * FEW_MQ + tid] = ma;
    }
}

template <int MQ>
__global__ void __launch_bounds__(32)
few_gemv_kernel(const double* __restrict__ Linv, int64_t ld, const double* __restrict__ P, double* __restrict__ Z) {
    constexpr int ST = FEW_ST, LP = 34;             // stages; row pitch (double2 reads of 8 lanes hit 32 distinct banks)
    extern __shared__ __align__(16) double few_smem[];
    double (*sL)[32 * LP] = reinterpret_cast<double (*)[32 * LP]>(few_smem);
    double (*sP)[32 * FEW_MQ] = reinterpret_cast<double (*)[32 * FEW_MQ]>(few_smem + ST * 32 * LP);
    const int lane = threadIdx.x;
    const int64_t r0 = (int64_t)blockIdx.x * 32;
    const int nt = (int)blockIdx.x + 1;             // 32-wide k tiles up to and including the diagonal one
    auto issue = [&](int t) {
        if (t < nt) {
            const int st = t % ST;
            const int64_t k0 = (int64_t)t * 32;
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const int c = lane + 32 * i, row = c >> 4, c16 = c & 15;
                abg::cp_async16(&sL[st][row * LP + 2 * c16], Linv + (r0 + row) * ld + k0 + 2 * c16);
            }
#pragma unroll
            for (int i = 0; i < FEW_MQ / 2 / 2; i++) {       // 32 rows x 4 chunks of 16 B: the whole FEW_MQ-wide panel rows
                const int c = lane + 32 * i * 2;
                abg::cp_async16(&sP[st][2 * c], P + k0 * FEW_MQ + 2 * c);
                abg::cp_async16(&sP[st][2 * (c + 32)], P + k0 * FEW_MQ + 2 * (c + 32));
            }
        }
        abg::cp_async_commit();
    };
    double z[MQ];
#pragma unroll
    for (int q = 0; q < MQ; q++) z[q] = 0.0;
#pragma unroll
    for (int t = 0; t < ST - 1; t++) issue(t);
    for (int t = 0; t < nt; t++) {
        abg::cp_async_wait<ST - 2>();
        __syncwarp();
        issue(t + ST - 1);
        const double* bl = &sL[t % ST][lane * LP];
        const double* bp = sP[t % ST];
        const int lim = (t == nt - 1) ? lane + 1 : 32;      // diagonal tile: k <= row
#pragma unroll 4
        for (int kk = 0; kk < 32; kk += 2) {
            const double2 a = *reinterpret_cast<const double2*>(bl + kk);
            if (kk < lim) {
#pragma unroll
                for (int q = 0; q < MQ; q++) z[q] = fma(a.x, bp[kk * FEW_MQ + q], z[q]);
            }
            if (kk + 1 < lim) {
#pragma unroll
                for (int q = 0; q < MQ; q++) z[q] = fma(a.y, bp[(kk + 1) * FEW_MQ + q], z[q]);
            }
        }
        __syncwarp();
    }
    abg::cp_async_wait<0>();
#pragma unroll
    for (int q = 0; q < MQ; q++) Z[(int64_t)q * ld + r0 + lane] = z[q];
}

// 128 threads: thread = (query q, warp row wm, row group g)
__global__ void __launch_bounds__(16 * FEW_MQ)
few_finish_kernel(const double* __restrict__ Z, int64_t npad, int T, const double* __restrict__ partial, int nsplit,
                  int m, double amp, double mean, double* __restrict__ mu, double* __restrict__ var) {
    __shared__ double sR[FEW_MQ][2];
    const int tid = threadIdx.x, q = tid >> 4, wm = (tid >> 3) & 1, g = tid & 7;
    if (Z) {
        double tot = 0.0;
        const double* zq = Z + (int64_t)q * npad;
        // loads of four row blocks are issued together (they do not depend on the chain)
        for (int i0 = 0; i0 < T; i0 += 4) {
            double v[4][8];
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
                for (int a = 0; a < 8; a++)
                    v[u][a] = (q < m && i0 + u < T) ? zq[(int64_t)(i0 + u) * NB + wm * 64 + a * 8 + g] : 0.0;
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (i0 + u < T) {
                    double blk = 0.0;
#pragma unroll
                    for (int a = 0; a < 8; a++) blk = fma(v[u][a], v[u][a], blk);
                    tot += blk;
                }
            }
        }
        tot += __shfl_xor_sync(0xffffffffu, tot, 1);
        tot += __shfl_xor_sync(0xffffffffu, tot, 2);
        tot += __shfl_xor_sync(0xffffffffu, tot, 4);
        if (g == 0) sR[q][wm] = tot;
    }
    __syncthreads();
    if (tid < m) {
        double s = 0.0;
        for (int p = 0; p < nsplit; p++) s += partial[(int64_t)p * FEW_MQ + tid];
        mu[tid] = fma(amp, s, mean);
        if (Z) var[tid] = amp - (sR[tid][0] + sR[tid][1]);
    }
}

// v = L^-T z for the few-query gradient path: lane = column i, chain over k ascending from the
// diagonal (the order of tri_gemm_kernel<true>); Linv rows are read as coalesced 256-byte pieces
template <int MQ>
__global__ void __launch_bounds__(32)
few_gemv_t_kernel(const double* __restrict__ Linv, int64_t ld, const double* __restrict__ Z, double* __restrict__ V) {
    constexpr int ST = 4;
    __shared__ __align__(16) double sL[ST][32 * 32];
    __shared__ __align__(16) double sZ[ST][MQ * 32];
    const int lane = threadIdx.x;
    const int64_t i0 = (int64_t)blockIdx.x * 32;
    const int nt = (int)((ld - i0) / 32);           // k tiles from the diagonal one to the last row
    auto issue = [&](int t) {
        if (t < nt) {
            const int st = t % ST;
            const int64_t k0 = i0 + (int64_t)t * 32;
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const int c = lane + 32 * i, row = c >> 4, c16 = c & 15;
                abg::cp_async16(&sL[st][row * 32 + 2 * c16], Linv + (k0 + row) * ld + i0 + 2 * c16);
            }
            for (int c = lane; c < MQ * 16; c += 32) {
                const int q = c >> 4, c16 = c & 15;
                abg::cp_async16(&sZ[st][q * 32 + 2 * c16], Z + (int64_t)q * ld + k0 + 2 * c16);
            }
        }
        abg::cp_async_commit();
    };
    double v[MQ];
#pragma unroll
    for (int q = 0; q < MQ; q++) v[q] = 0.0;
#pragma unroll
    for (int t = 0; t < ST - 1; t++) issue(t);
    for (int t = 0; t < nt; t++) {
        abg::cp_async_wait<ST - 2>();
        __syncwarp();
        issue(t + ST - 1);
        const double* bl = sL[t % ST];
        const double* bz = sZ[t % ST];
        const int first = (t == 0) ? lane : 0;      // diagonal tile: k >= column
#pragma unroll 4
        for (int kk = 0; kk < 32; kk++) {
            if (kk >= first) {
                const double a = bl[kk * 32 + lane];
#pragma unroll
                for (int q = 0; q < MQ; q++) v[q] = fma(a, bz[q * 32 + kk], v[q]);
            }
        }
        __syncwarp();
    }
    abg::cp_async_wait<0>();
#pragma unroll
    for (int q = 0; q < MQ; q++) V[(int64_t)q * ld + i0 + lane] = v[q];
}

// derivative reduction of predict_grad_kernel for few queries: one CTA per 512-point split;
// per 64-point piece all threads evaluate k'(r^2) for (query, point), then one thread per
// (query, mean | variance, dimension) extends its FMA chain over the piece in point order
template <int KIND, int D>
__global__ void __launch_bounds__(512)
few_grad_kernel(const double* __restrict__ Xq, int m, const double* __restrict__ Xs, const double* __restrict__ alpha,
                const double* __restrict__ V, int64_t ldv, int64_t n, int64_t npad, KernParams kp,
                double* __restrict__ gpart) {
    constexpr int PS = 64;
    __shared__ double sQ[FEW_MQ][D];
    __shared__ double sX[PS * D];
    __shared__ double sG[FEW_MQ][PS], sV[FEW_MQ][PS], sAl[PS];
    const int tid = threadIdx.x, d = kp.d;
    if (tid < FEW_MQ * D) {
        const int q = tid / D, k = tid - q * D;
        sQ[q][k] = (k < d && q < m) ? Xq[(int64_t)q * d + k] * kp.inv_len[k] : 0.0;
    }
    const int64_t jbeg = (int64_t)blockIdx.x * JCHUNK;
    const int64_t jend = jbeg + JCHUNK < n ? jbeg + JCHUNK : n;
    const int cq = tid / (2 * D), crem = tid - cq * 2 * D, ckind = crem / D, ck = crem - ckind * D;
    const bool chain = cq < m && ck < d;
    const int ejj = tid & (PS - 1), eq = tid / PS;       // evaluation role: (point, query)
    double acc = 0.0;
    for (int64_t j0 = jbeg; j0 < jend; j0 += PS) {
        __syncthreads();
        for (int idx = tid; idx < PS * D; idx += 512) {
            const int jj = idx / D, k = idx - jj * D;
            sX[idx] = (k < d && j0 + jj < npad) ? Xs[(j0 + jj) * d + k] : 0.0;
        }
        if (tid < PS) sAl[tid] = (j0 + tid < n) ? alpha[j0 + tid] : 0.0;
        __syncthreads();
        {
            double g = 0.0, vv = 0.0;
            if (eq < m && j0 + ejj < n) {
                double r2 = 0.0;
#pragma unroll
                for (int k = 0; k < D; k++) {
                    const double df = sQ[eq][k] - sX[ejj * D + k];
                    r2 = fma(df, df, r2);
                }
                g = ab_radial_grad<KIND>(r2, kp.alpha, kp.inv2a);
                vv = V[(int64_t)eq * ldv + j0 + ejj];
            }
            sG[eq][ejj] = g;
            sV[eq][ejj] = vv;
        }
        __syncthreads();
        if (chain) {
            const int tn = (int)((jend - j0 < PS) ? (jend - j0) : PS);
            for (int jj = 0; jj < tn; jj++) {
                const double df = sQ[cq][ck] - sX[jj * D + ck];
                const double c = (ckind == 0 ? sAl[jj] : sV[cq][jj]) * sG[cq][jj];
                acc = fma(c, df, acc);
            }
        }
    }
    if (chain) gpart[((int64_t)blockIdx.x * 2 * D + ckind * D + ck) * FEW_MQ + cq] = acc;
}

__global__ void few_grad_finish_kernel(const double* __restrict__ gpart, int nsplit, int D, int m, KernParams kp,
                                       double* __restrict__ dmu, double* __restrict__ dvar) {
    const int d = kp.d, idx = threadIdx.x;
    if (idx >= m * d) return;
    const int q = idx / d, k = idx - q * d;
    double sm = 0.0, sv = 0.0;
    for (int p = 0; p < nsplit; p++) {
        sm += gpart[((int64_t)p * 2 * D + k) * FEW_MQ + q];
        sv += gpart[((int64_t)p * 2 * D + D + k) * FEW_MQ + q];
    }
    const double f = 2.0 * kp.amp * kp.inv_len[k];
    dmu[(int64_t)q * d + k] = f * sm;
    dvar[(int64_t)q * d + k] = -2.0 * f * sv;
}

// f(std::integral_constant<int, MQ>{}) for the query count MQ of the few-query kernels that covers m
template <class F>
auto dispatch_mq(int m, F&& f) {
    if (m == 1) return f(std::integral_constant<int, 1>{});
    if (m == 2) return f(std::integral_constant<int, 2>{});
    if (m <= 4) return f(std::integral_constant<int, 4>{});
    return f(std::integral_constant<int, 8>{});
}

// mean (and variance, and their gradients w.r.t. the query) of m <= FEW_MQ queries;
// 2 (mean), 3 (+ variance) or 6 (+ gradients) launches
int launch_few(ab_gp* h, const double* Xq, int m, double* mu, double* var, double* dmu = nullptr, double* dvar = nullptr) {
    cudaStream_t s = h->stream;
    const int T = (int)(h->npad / NB);
    const int nsplit = (int)(((var ? h->npad : h->n) + JCHUNK - 1) / JCHUNK);
    const int nsplit_g = (int)((h->n + JCHUNK - 1) / JCHUNK);
    const size_t need = ((size_t)h->npad * FEW_MQ * 3 + (size_t)nsplit * FEW_MQ + (size_t)nsplit_g * 2 * AB_MAX_DIM * FEW_MQ) * sizeof(double);
    int rc = ab_ensure_scratch(h, need);
    if (rc) return rc;
    double* P = var ? h->scratch : nullptr;                      // npad x FEW_MQ
    double* Z = h->scratch + (size_t)h->npad * FEW_MQ;           // FEW_MQ x npad
    double* V = Z + (size_t)h->npad * FEW_MQ;                    // FEW_MQ x npad
    double* partial = V + (size_t)h->npad * FEW_MQ;
    double* gpart = partial + (size_t)nsplit * FEW_MQ;
    ab_prof_begin(h, AB_PROF_PREDICT_PANEL);
    AB_DISPATCH_KIND(h->kp.kind, ab_dispatch_dim(h->d, [&](auto D) {
        few_cross_kernel<KIND, D><<<nsplit, JCHUNK, 0, s>>>(Xq, m, h->Xs, h->alpha, h->n, h->npad, h->kp, P, partial);
    }));
    ab_prof_end(h, AB_PROF_PREDICT_PANEL);
    AB_CHECK_LAUNCH();
    const unsigned nb = (unsigned)(h->npad / 32);
    if (var) {
        ab_prof_begin(h, AB_PROF_PREDICT_VAR);
        rc = dispatch_mq(m, [&](auto MQ) {
            AB_CUDA(cudaFuncSetAttribute(few_gemv_kernel<MQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, FEW_GEMV_SMEM));
            few_gemv_kernel<MQ><<<nb, 32, FEW_GEMV_SMEM, s>>>(h->Linv, h->npad, P, Z);
            return 0;
        });
        ab_prof_end(h, AB_PROF_PREDICT_VAR);
        if (rc) return rc;
        AB_CHECK_LAUNCH();
    }
    few_finish_kernel<<<1, 16 * FEW_MQ, 0, s>>>(var ? Z : nullptr, h->npad, T, partial, nsplit, m, h->kp.amp, h->mean, mu, var);
    AB_CHECK_LAUNCH();
    ab_count_launches(var ? 3 : 2);
    if (var && dmu && dvar) {
        dispatch_mq(m, [&](auto MQ) { few_gemv_t_kernel<MQ><<<nb, 32, 0, s>>>(h->Linv, h->npad, Z, V); });
        AB_DISPATCH_KIND(h->kp.kind, ab_dispatch_dim(h->d, [&](auto D) {
            few_grad_kernel<KIND, D><<<nsplit_g, 512, 0, s>>>(Xq, m, h->Xs, h->alpha, V, h->npad, h->n, h->npad, h->kp, gpart);
        }));
        few_grad_finish_kernel<<<1, FEW_MQ * AB_MAX_DIM, 0, s>>>(gpart, nsplit_g, ab_padded_dim(h->d), m, h->kp, dmu, dvar);
        AB_CHECK_LAUNCH();
        ab_count_launches(3);
    }
    return 0;
}

// f(std::integral_constant<int, NL>{}) for nl = 1..16 (the NL of predict_var_kernel)
template <int NL = 1, class F>
int dispatch_nl(int nl, F&& f) {
    if constexpr (NL < 16) {
        if (nl == NL) return f(std::integral_constant<int, NL>{});
        return dispatch_nl<NL + 1>(nl, f);
    } else {
        return f(std::integral_constant<int, 16>{});
    }
}

// chunks of JCHUNK training points the panel pass splits the training range into (grid.y)
int panel_splits(const ab_gp* h) { return (int)((h->npad + JCHUNK - 1) / JCHUNK); }

}  // namespace

// The panel pass of queries [q0, q0 + cnt): their means, and with P their cross-covariance panel
// P[j][q] (npad x ldp, ldp >= cnt rounded up to QPB).  predict_mean_kernel covers the training range
// in panel_splits(h) fixed chunks (more CTAs, a summation order fixed by N); combine_splits_kernel
// adds the chunk partials (panel_splits(h) x ldp) in chunk order.
static int launch_panel(ab_gp* h, const double* Xq, int64_t m, int64_t q0, int64_t cnt, double* mu, double* P,
                        int64_t ldp, double* partial) {
    cudaStream_t s = h->stream;
    const int nsplit = panel_splits(h);
    const dim3 grid((unsigned)((cnt + QPB - 1) / QPB), (unsigned)nsplit);
    ab_prof_begin(h, AB_PROF_PREDICT_PANEL);
    AB_DISPATCH_KIND(h->kp.kind, ab_dispatch_dim(h->d, [&](auto D) {
        if (P)
            predict_mean_kernel<KIND, D, true><<<grid, 128, 0, s>>>(Xq, m, q0, h->Xs, h->alpha, h->n, h->npad, h->kp,
                                                                    h->mean, mu, P, ldp, nsplit, partial, ldp);
        else
            predict_mean_kernel<KIND, D, false><<<grid, 128, 0, s>>>(Xq, m, q0, h->Xs, h->alpha, h->n, h->npad, h->kp,
                                                                     h->mean, mu, P, ldp, nsplit, partial, ldp);
    }));
    if (nsplit > 1)
        combine_splits_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, s>>>(partial, ldp, cnt, nsplit, h->kp.amp, h->mean,
                                                                            mu, q0);
    ab_prof_end(h, AB_PROF_PREDICT_PANEL);
    AB_CHECK_LAUNCH();
    ab_count_launches(nsplit > 1 ? 2 : 1);
    return 0;
}

// sigma^2 for `cnt` queries of the panel P: one CTA per 128 queries looping over the row
// blocks, or the row blocks spread over the grid (few query tiles, or full panels with many
// row blocks), their per-thread block values in `part` (T x ldp x 16)
static int launch_variance(ab_gp* h, int T, const double* P, int64_t ldp, int64_t m, int64_t q0, int64_t cnt,
                           double* var, double* part) {
    cudaStream_t s = h->stream;
    const unsigned ntq = (unsigned)((cnt + abg::BN - 1) / abg::BN);
    const int nl = (int)((h->n - (int64_t)(T - 1) * NB + 7) / 8);        // 1..16 row groups in the last block
    // row-block pairs of a tile on adjacent CTAs from N >= 6144 (measured: 0.2 % slower at N = 8192 for a quarter of the DRAM traffic, 3 % slower at N = 4000)
    if (T >= 48 && (int)ntq * 2 > h->nsm) {
        const long long nitems = (long long)((T + 1) / 2) * ntq;
        const unsigned grid = (unsigned)(nitems < h->nsm ? nitems : h->nsm);
        const int rc = dispatch_nl(nl, [&](auto NL) {
            AB_CUDA(cudaFuncSetAttribute(predict_var_pair_kernel<NL>, cudaFuncAttributeMaxDynamicSharedMemorySize, abg::SMEM_BYTES));
            predict_var_pair_kernel<NL><<<grid, abg::THREADS, abg::SMEM_BYTES, s>>>(h->Linv, h->npad, T, (int)ntq, P, ldp, part);
            return 0;
        });
        if (rc) return rc;
        var_combine_kernel<<<ntq, abg::THREADS, 0, s>>>(part, T, m, q0, h->kp.amp, var);
        ab_count_launches(2);
    } else if (T > 1 && (int)ntq * 2 <= h->nsm) {
        AB_CUDA(cudaFuncSetAttribute(predict_var_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, abg::SMEM_BYTES));
        predict_var_split_kernel<<<dim3(ntq, T), abg::THREADS, abg::SMEM_BYTES, s>>>(h->Linv, h->npad, P, ldp, part);
        var_combine_kernel<<<ntq, abg::THREADS, 0, s>>>(part, T, m, q0, h->kp.amp, var);
        ab_count_launches(2);
    } else {
        const int rc = dispatch_nl(nl, [&](auto NL) {
            AB_CUDA(cudaFuncSetAttribute(predict_var_kernel<NL>, cudaFuncAttributeMaxDynamicSharedMemorySize, abg::SMEM_BYTES));
            predict_var_kernel<NL><<<ntq, abg::THREADS, abg::SMEM_BYTES, s>>>(h->Linv, h->npad, T, P, ldp, m, q0, h->kp.amp, var);
            return 0;
        });
        if (rc) return rc;
        ab_count_launches(1);
    }
    AB_CHECK_LAUNCH();
    return 0;
}

// queries per variance panel: one wave of CTAs (148 SMs x 128 queries)
static const int64_t kPanelQueries = 148 * 128;

// queries per variance panel for the current training-set size: whole waves of variance CTAs, as many
// as fit a ~2 GB cross-covariance panel
int64_t ab_predict_panel_queries(ab_gp* h) {
    int64_t waves = (int64_t)((2ULL << 30) / ((size_t)h->npad * kPanelQueries * sizeof(double)));
    if (waves < 1) waves = 1;
    if (waves > 16) waves = 16;
    return waves * kPanelQueries;
}

int ab_launch_predict(ab_gp* h, const double* Xq, int64_t m, double* mu, double* var) {
    if (m <= 0) return 0;
    if (m <= FEW_MQ && h->few_path) return launch_few(h, Xq, (int)m, mu, var);
    const int nsplit = panel_splits(h);
    if (!var) {
        const int64_t ldp = (m + QPB - 1) / QPB * QPB;
        if (nsplit > 1) {
            const int rc = ab_ensure_scratch(h, (size_t)nsplit * ldp * sizeof(double));
            if (rc) return rc;
        }
        return launch_panel(h, Xq, m, 0, m, mu, nullptr, ldp, nsplit > 1 ? h->scratch : nullptr);
    }
    // mean + variance, processed in panels
    const int T = (int)(h->npad / NB);
    const int64_t mq = std::min(m, ab_predict_panel_queries(h));
    const int64_t ldp = (mq + QPB - 1) / QPB * QPB;                 // multiple of 256 (and of 128)
    const size_t panel_elems = (size_t)h->npad * ldp;
    int rc = ab_ensure_scratch(h, (panel_elems + (size_t)nsplit * ldp + (size_t)T * ldp * 16) * sizeof(double));
    if (rc) return rc;
    double* P = h->scratch;
    double* partial = h->scratch + panel_elems;
    double* vpart = partial + (size_t)nsplit * ldp;
    for (int64_t q0 = 0; q0 < m; q0 += mq) {
        const int64_t cnt = (m - q0 < mq) ? (m - q0) : mq;
        rc = launch_panel(h, Xq, m, q0, cnt, mu, P, ldp, partial);
        if (rc) return rc;
        ab_prof_begin(h, AB_PROF_PREDICT_VAR);
        rc = launch_variance(h, T, P, ldp, m, q0, cnt, var, vpart);
        ab_prof_end(h, AB_PROF_PREDICT_VAR);
        if (rc) return rc;
    }
    return 0;
}

// mean, variance and their gradients w.r.t. the query coordinates (row-major m x d)
int ab_launch_predict_grad(ab_gp* h, const double* Xq, int64_t m, double* mu, double* var, double* dmu, double* dvar) {
    if (m <= 0) return 0;
    if (m <= FEW_MQ && h->few_path) return launch_few(h, Xq, (int)m, mu, var, dmu, dvar);
    cudaStream_t s = h->stream;
    const int d = h->d, Dp = ab_padded_dim(d);
    AB_CUDA(cudaFuncSetAttribute(tri_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, abg::SMEM_BYTES));
    AB_CUDA(cudaFuncSetAttribute(tri_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, abg::SMEM_BYTES));
    const int T = (int)(h->npad / NB);
    int64_t mq = m < 1024 ? m : 1024;                              // queries per panel
    const int64_t ldp = (mq + QPB - 1) / QPB * QPB;
    const int nsplit = panel_splits(h);
    const size_t panel = (size_t)h->npad * ldp;
    int rc = ab_ensure_scratch(h, (3 * panel + (size_t)nsplit * ldp * (1 + 2 * Dp) + (size_t)T * ldp * 16) * sizeof(double));
    if (rc) return rc;
    double* P = h->scratch;
    double* W = P + panel;
    double* V = W + panel;
    double* partial = V + panel;                                   // [nsplit][ldp] mean partials
    double* gpartial = partial + (size_t)nsplit * ldp;             // [nsplit][2 Dp][ldp]
    for (int64_t q0 = 0; q0 < m; q0 += mq) {
        const int64_t cnt = (m - q0 < mq) ? (m - q0) : mq;
        rc = launch_panel(h, Xq, m, q0, cnt, mu, P, ldp, partial);
        if (rc) return rc;
        const unsigned ntq = (unsigned)((cnt + abg::BN - 1) / abg::BN);
        rc = launch_variance(h, T, P, ldp, m, q0, cnt, var, gpartial + (size_t)nsplit * 2 * Dp * ldp);
        if (rc) return rc;
        tri_gemm_kernel<false><<<dim3(ntq, T), abg::THREADS, abg::SMEM_BYTES, s>>>(h->Linv, h->npad, T, P, ldp, W);
        tri_gemm_kernel<true><<<dim3(ntq, T), abg::THREADS, abg::SMEM_BYTES, s>>>(h->Linv, h->npad, T, W, ldp, V);
        AB_CHECK_LAUNCH();
        dim3 ggrid((unsigned)((cnt + 127) / 128), (unsigned)nsplit);
        AB_DISPATCH_KIND(h->kp.kind, ab_dispatch_dim(d, [&](auto D) {
            predict_grad_kernel<KIND, D><<<ggrid, 128, 0, s>>>(Xq, m, q0, h->Xs, h->alpha, V, ldp, h->n, h->npad, h->kp,
                                                               gpartial, ldp);
        }));
        grad_combine_kernel<<<(unsigned)((cnt * d + 255) / 256), 256, 0, s>>>(gpartial, ldp, cnt, nsplit, Dp, d, h->kp, dmu,
                                                                            dvar, q0);
        AB_CHECK_LAUNCH();
        ab_count_launches(4);
    }
    return 0;
}

int ab_launch_utility(ab_gp* h, int kind, const double* Xq, const double* mu, const double* var, int64_t m,
                      const double* h_bounds, double y_best, double zeta, double* util, int64_t* h_argmin,
                      double* h_min) {
    UtilParams up;
    up.kind = kind;
    up.d = h->d;
    up.y_best = y_best;
    up.zeta = zeta;
    for (int k = 0; k < h->d; k++) { up.lo[k] = h_bounds[2 * k]; up.hi[k] = h_bounds[2 * k + 1]; }
    int nb = (int)((m + 255) / 256);
    int rc = ab_ensure_scratch(h, (size_t)nb * 16 + 64);
    if (rc) return rc;
    double* bval = h->scratch + 8;
    long long* bidx = reinterpret_cast<long long*>(h->scratch + 8 + nb);
    utility_kernel<<<nb, 256, 0, h->stream>>>(Xq, mu, var, m, up, util, bval, bidx);
    argmin_final_kernel<<<1, 256, 0, h->stream>>>(bval, bidx, nb, h->scratch, reinterpret_cast<long long*>(h->scratch + 1));
    AB_CHECK_LAUNCH();
    ab_count_launches(2);
    AB_CUDA(cudaMemcpyAsync(h->h_pinned, h->scratch, 16, cudaMemcpyDeviceToHost, h->stream));
    AB_CUDA(cudaStreamSynchronize(h->stream));
    *h_min = h->h_pinned[0];
    *h_argmin = (int64_t) * reinterpret_cast<long long*>(h->h_pinned + 1);
    return 0;
}

// ---------------------------------------------------------------------------
// Full predictive covariance (george GP.predict(y, t, return_cov=True)):
//   Sigma = K(t, t) - W^T W,  W = L^-1 P,  P[j][q] = amp k(x_j, t_q)
// Stages: panel + mean (predict_mean_kernel, as ab_launch_predict), W (tri_gemm_kernel<false>),
// the prior block K(t, t) straight into the caller's matrix (cov_kernel), the SYRK below over the
// lower 128 x 128 tile pairs, the diagonal from W in the canonical order of predict_var_kernel
// (so diag(Sigma) has the bits of predict(return_var=True)), and a mirror of the lower triangle.
// Every entry (a, b) depends on queries a and b only, through a k order fixed by N.
// ---------------------------------------------------------------------------
namespace {

// C[a-tile][b-tile] -= sum_k W[k][a] W[k][b] for the tile pair (a, b), b <= a, of blockIdx.x.
// nk: BK chunks of the k range (fixed by N: rows of W past the training points are zero).
// Masked element stores: the same expression for every element, ragged tile or not.
__global__ void __launch_bounds__(abg::THREADS, 1)
syrk_lower_kernel(const double* __restrict__ W, int64_t ldw, int nk, double* __restrict__ C, int64_t ldc,
                  int64_t m) {
    extern __shared__ __align__(16) double smem[];
    int a, b;
    abg::tri_decode(blockIdx.x, a, b);
    abg::Acc acc;
    acc.zero();
    abg::mainloop<false, false>(acc, W + (int64_t)a * abg::BM, ldw, W + (int64_t)b * abg::BN, ldw, nk, smem);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int64_t r = (int64_t)a * abg::BM + abg::acc_row(i);
#pragma unroll
        for (int j = 0; j < 4; j++)
#pragma unroll
            for (int e = 0; e < 2; e++) {
                const int64_t c = (int64_t)b * abg::BN + abg::acc_col(j) + e;
                if (r < m && c < m) {
                    double* p = C + r * ldc + c;
                    *p = *p - acc.v[i][j][e];
                }
            }
    }
}

// sigma^2 of the 128 queries of blockIdx.x from W (npad x ldw): the W tiles are read back in the
// accumulator layout store_tile wrote them from (alpha = 1: the accumulator's bits), then squared
// and summed exactly like predict_var_kernel / var_combine_kernel
__global__ void __launch_bounds__(abg::THREADS)
var_from_w_kernel(const double* __restrict__ W, int64_t ldw, int T, int64_t m, double amp, double* __restrict__ var) {
    __shared__ double red[256];
    double tot[4][2];
#pragma unroll
    for (int j = 0; j < 4; j++) tot[j][0] = tot[j][1] = 0.0;
    const double* Wq = W + (int64_t)blockIdx.x * abg::BN;
    for (int i = 0; i < T; i++) {
        abg::Acc acc;
#pragma unroll
        for (int a = 0; a < 8; a++) {
            const double* row = Wq + ((int64_t)i * NB + abg::acc_row(a)) * ldw;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const double2 v = *reinterpret_cast<const double2*>(row + abg::acc_col(j));
                acc.v[a][j][0] = v.x;
                acc.v[a][j][1] = v.y;
            }
        }
        double blk[4][2];
        tile_thread_sq(acc, blk);
#pragma unroll
        for (int j = 0; j < 4; j++) { tot[j][0] += blk[j][0]; tot[j][1] += blk[j][1]; }
    }
    tile_finish_var(tot, red, (int64_t)blockIdx.x * abg::BN + threadIdx.x, m, amp, var);
}

__global__ void set_diag_kernel(const double* __restrict__ v, int64_t m, double* __restrict__ C, int64_t ldc) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q < m) C[q * ldc + q] = v[q];
}

}  // namespace

// C = op-free lower triangular product L B (tri_gemm_kernel<false>): L is T x T blocks of 128 with
// leading dimension ld, lower, with the upper part of its diagonal blocks zero (L^-1, or a Cholesky
// factor of the dataflow kernel); B and C are (T 128) x ldb, the first ntiles 128-column tiles are
// computed.  Every column of C depends on the same column of B only.
int ab_launch_tri_gemm_lower(ab_gp* h, const double* L, int64_t ld, int T, const double* B, int64_t ldb, int ntiles,
                             double* C) {
    AB_CUDA(cudaFuncSetAttribute(tri_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, abg::SMEM_BYTES));
    tri_gemm_kernel<false><<<dim3((unsigned)ntiles, (unsigned)T), abg::THREADS, abg::SMEM_BYTES, h->stream>>>(L, ld, T, B,
                                                                                                             ldb, C);
    AB_CHECK_LAUNCH();
    ab_count_launches(1);
    return 0;
}

// mean mu (m) and covariance C (m x m, leading dimension ldc >= m) of the m queries Xq; needs L^-1.
// Workspace: P and W (npad x ldp each, ldp = m rounded up to 256) from the handle scratch.
int ab_launch_predict_cov(ab_gp* h, const double* Xq, int64_t m, double* mu, double* C, int64_t ldc) {
    if (m <= 0) return 0;
    cudaStream_t s = h->stream;
    const int d = h->d, T = (int)(h->npad / NB);
    const int64_t ldp = (m + QPB - 1) / QPB * QPB;
    const int nsplit = panel_splits(h);
    const int ntq = (int)((m + abg::BN - 1) / abg::BN);
    const size_t panel = (size_t)h->npad * ldp;
    int rc = ab_ensure_scratch(h, (2 * panel + (size_t)nsplit * ldp + ldp + (size_t)m * d) * sizeof(double));
    if (rc) {
        cudaGetLastError();                    // a failed allocation is reported once, by the return code
        return rc;
    }
    double* P = h->scratch;
    double* W = P + panel;
    double* partial = W + panel;
    double* dv = partial + (size_t)nsplit * ldp;
    double* XT = dv + ldp;
    // 1. panel P and mean
    rc = launch_panel(h, Xq, m, 0, m, mu, P, ldp, partial);
    if (rc) return rc;
    // 2. W = L^-1 P
    ab_prof_begin(h, AB_PROF_PREDICT_VAR);
    rc = ab_launch_tri_gemm_lower(h, h->Linv, h->npad, T, P, ldp, ntq, W);
    if (rc) return rc;
    // 3. prior block K(t, t) into C
    rc = ab_launch_scale_points(h, Xq, m, XT, m);
    if (rc) return rc;
    rc = ab_launch_cross_cov(h, XT, m, m, XT, m, m, C, ldc);
    if (rc) return rc;
    // 4. C -= W^T W on the lower tile pairs; k over the training rows rounded up to BK
    const int nk = (int)((h->n + abg::BK - 1) / abg::BK);
    AB_CUDA(cudaFuncSetAttribute(syrk_lower_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, abg::SMEM_BYTES));
    syrk_lower_kernel<<<(unsigned)(ntq * (ntq + 1) / 2), abg::THREADS, abg::SMEM_BYTES, s>>>(W, ldp, nk, C, ldc, m);
    AB_CHECK_LAUNCH();
    // 5. the diagonal: sigma^2 with the bits of the variance path
    var_from_w_kernel<<<(unsigned)ntq, abg::THREADS, 0, s>>>(W, ldp, T, m, h->kp.amp, dv);
    set_diag_kernel<<<(unsigned)((m + 255) / 256), 256, 0, s>>>(dv, m, C, ldc);
    AB_CHECK_LAUNCH();
    ab_count_launches(5);
    // 6. exact symmetry
    rc = ab_launch_mirror_lower_n(h, C, ldc, m);
    ab_prof_end(h, AB_PROF_PREDICT_VAR);
    return rc;
}
