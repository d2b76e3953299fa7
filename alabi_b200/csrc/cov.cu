// K1: fused anisotropic-distance + covariance-matrix builder (FP64).
//
// Replaces george's `kernel.get_value(x)` + white-noise diagonal inside
// `GP.compute` (reference call sites alabi/gp_utils.py:243, alabi/core.py:1158).
// One CTA computes a 64 x 64 tile from per-dimension-major ("SoA") scaled
// inputs staged in shared memory; every thread owns a 4 x 4 block and writes
// 32-byte row segments, so a half-warp writes 512 contiguous bytes.  In the
// symmetric case only lower tiles are computed and mirrored.
#include <vector>
#include "handle.h"
#include "dmma_gemm.cuh"

namespace {

__global__ void scale_inputs_kernel(const double* __restrict__ X, int64_t n, int64_t npad, int d,
                                    KernParams kp, double* __restrict__ Xs, double* __restrict__ XsT) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= npad * d) return;
    int64_t i = idx / d;
    int k = (int)(idx - i * d);
    double v = (i < n) ? X[idx] * kp.inv_len[k] : 0.0;
    Xs[idx] = v;
    XsT[(int64_t)k * npad + i] = v;
}

// arbitrary point set (m x d, row-major) -> scaled SoA (d x ldm)
__global__ void scale_points_kernel(const double* __restrict__ X, int64_t m, int d, KernParams kp,
                                    double* __restrict__ XT, int64_t ldm) {
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= m * d) return;
    int64_t i = idx / d;
    int k = (int)(idx - i * d);
    XT[(int64_t)k * ldm + i] = X[idx] * kp.inv_len[k];
}

// Rows come from point set A (SoA: AT[k * lda + i]), columns from set B.
// symmetric != 0: A == B, blockIdx.x enumerates lower tiles, diagonal gets
// diag_add, optional mirror; rows/cols >= n_valid become identity when
// pad_identity (padding of the blocked factorisation).
template <int KIND>
__global__ void __launch_bounds__(256, 4)
cov_kernel(const double* __restrict__ AT, int64_t lda, int64_t na, const double* __restrict__ BT, int64_t ldb,
           int64_t nb, int64_t n_valid, KernParams kp, double* __restrict__ K, int64_t ld, int symmetric,
           int mirror, int pad_identity) {
    __shared__ __align__(16) double sA[AB_MAX_DIM][64];
    __shared__ __align__(16) double sB[AB_MAX_DIM][64];
    int ti, tj;
    if (symmetric) abg::tri_decode(blockIdx.x, ti, tj);
    else { ti = blockIdx.y; tj = blockIdx.x; }
    const int64_t i0 = (int64_t)ti * 64, j0 = (int64_t)tj * 64;
    const int tid = threadIdx.x;
    const int d = kp.d;
    for (int idx = tid; idx < 64 * d; idx += 256) {
        int k = idx >> 6, r = idx & 63;
        sA[k][r] = (i0 + r < na) ? AT[(int64_t)k * lda + i0 + r] : 0.0;
        sB[k][r] = (j0 + r < nb) ? BT[(int64_t)k * ldb + j0 + r] : 0.0;
    }
    __syncthreads();
    const int tx = tid & 15, ty = tid >> 4;
    double r2[4][4];
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
        for (int c = 0; c < 4; c++) r2[r][c] = 0.0;
    for (int k = 0; k < d; k++) {
        double2 a01 = *reinterpret_cast<const double2*>(&sA[k][ty * 4]);
        double2 a23 = *reinterpret_cast<const double2*>(&sA[k][ty * 4 + 2]);
        double2 b01 = *reinterpret_cast<const double2*>(&sB[k][tx * 4]);
        double2 b23 = *reinterpret_cast<const double2*>(&sB[k][tx * 4 + 2]);
        double a[4] = {a01.x, a01.y, a23.x, a23.y};
        double b[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
        for (int r = 0; r < 4; r++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                double df = a[r] - b[c];
                r2[r][c] = fma(df, df, r2[r][c]);
            }
    }
    double v[4][4];
#pragma unroll
    for (int r = 0; r < 4; r++)
#pragma unroll
        for (int c = 0; c < 4; c++) {
            int64_t gi = i0 + ty * 4 + r, gj = j0 + tx * 4 + c;
            double x = kp.amp * ab_radial<KIND, false>(r2[r][c], kp.alpha, kp.inv2a);
            if (symmetric) {
                if (gi == gj) x += kp.diag_add;
                if (pad_identity && (gi >= n_valid || gj >= n_valid)) x = (gi == gj) ? 1.0 : 0.0;
            }
            v[r][c] = x;
        }
    const bool full = (i0 + 64 <= na) && (j0 + 64 <= nb) && ((ld & 1) == 0) &&
                      ((reinterpret_cast<uintptr_t>(K) & 15) == 0);
    if (full) {
#pragma unroll
        for (int r = 0; r < 4; r++) {
            double* p = K + (i0 + ty * 4 + r) * ld + j0 + tx * 4;
            *reinterpret_cast<double2*>(p) = make_double2(v[r][0], v[r][1]);
            *reinterpret_cast<double2*>(p + 2) = make_double2(v[r][2], v[r][3]);
        }
        if (symmetric && mirror && ti != tj) {
#pragma unroll
            for (int c = 0; c < 4; c++) {
                double* p = K + (j0 + tx * 4 + c) * ld + i0 + ty * 4;
                *reinterpret_cast<double2*>(p) = make_double2(v[0][c], v[1][c]);
                *reinterpret_cast<double2*>(p + 2) = make_double2(v[2][c], v[3][c]);
            }
        }
    } else {
#pragma unroll
        for (int r = 0; r < 4; r++)
#pragma unroll
            for (int c = 0; c < 4; c++) {
                int64_t gi = i0 + ty * 4 + r, gj = j0 + tx * 4 + c;
                if (gi < na && gj < nb) {
                    K[gi * ld + gj] = v[r][c];
                    if (symmetric && mirror && ti != tj) K[gj * ld + gi] = v[r][c];
                }
            }
    }
}

// Factorisation path (padded matrix, full tiles, lower triangle only): one CTA walks a
// strip of up to `seg` tiles of one tile row.  The row inputs are loaded once, the
// column inputs of tile t + 1 arrive by cp.async while tile t is evaluated, and the
// stores of tile t drain behind the arithmetic of tile t + 1, so the FP64 pipe does not
// idle through a load / barrier / store sequence per 64 x 64 tile.
template <int KIND>
__global__ void __launch_bounds__(256, 3)
cov_strip_kernel(const double* __restrict__ XT, int64_t ldx, int64_t n_valid, KernParams kp,
                 double* __restrict__ K, int64_t ld, int seg, const int2* __restrict__ items) {
    __shared__ __align__(16) double sA[AB_MAX_DIM][64];
    __shared__ __align__(16) double sB[2][AB_MAX_DIM][64];
    const int ti = items[blockIdx.x].x, t0 = items[blockIdx.x].y;
    const int t1 = (t0 + seg < ti + 1) ? t0 + seg : ti + 1;            // tiles [t0, t1) of row ti
    const int tid = threadIdx.x, d = kp.d;
    const int64_t i0 = (int64_t)ti * 64;
    auto issue_B = [&](int tj, int buf) {
        for (int idx = tid; idx < 32 * d; idx += 256) {
            const int k = idx >> 5, r2 = (idx & 31) * 2;
            abg::cp_async16(&sB[buf][k][r2], XT + (int64_t)k * ldx + (int64_t)tj * 64 + r2);
        }
        abg::cp_async_commit();
    };
    issue_B(t0, 0);
    for (int idx = tid; idx < 64 * d; idx += 256) {
        const int k = idx >> 6, r = idx & 63;
        sA[k][r] = XT[(int64_t)k * ldx + i0 + r];
    }
    const int tx = tid & 15, ty = tid >> 4;
    for (int tj = t0; tj < t1; tj++) {
        const int buf = (tj - t0) & 1;
        if (tj + 1 < t1) issue_B(tj + 1, buf ^ 1);
        else abg::cp_async_commit();
        abg::cp_async_wait<1>();
        __syncthreads();
        const int64_t j0 = (int64_t)tj * 64;
        double r2[4][4];
#pragma unroll
        for (int r = 0; r < 4; r++)
#pragma unroll
            for (int c = 0; c < 4; c++) r2[r][c] = 0.0;
        for (int k = 0; k < d; k++) {
            const double2 a01 = *reinterpret_cast<const double2*>(&sA[k][ty * 4]);
            const double2 a23 = *reinterpret_cast<const double2*>(&sA[k][ty * 4 + 2]);
            const double2 b01 = *reinterpret_cast<const double2*>(&sB[buf][k][tx * 4]);
            const double2 b23 = *reinterpret_cast<const double2*>(&sB[buf][k][tx * 4 + 2]);
            const double a[4] = {a01.x, a01.y, a23.x, a23.y};
            const double b[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
            for (int r = 0; r < 4; r++)
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const double df = a[r] - b[c];
                    r2[r][c] = fma(df, df, r2[r][c]);
                }
        }
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int64_t gi = i0 + ty * 4 + r;
            double v[4];
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int64_t gj = j0 + tx * 4 + c;
                double x = kp.amp * ab_radial<KIND, false>(r2[r][c], kp.alpha, kp.inv2a);
                if (gi == gj) x += kp.diag_add;
                if (gi >= n_valid || gj >= n_valid) x = (gi == gj) ? 1.0 : 0.0;
                v[c] = x;
            }
            double* p = K + gi * ld + j0 + tx * 4;
            *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
            *reinterpret_cast<double2*>(p + 2) = make_double2(v[2], v[3]);
        }
        __syncthreads();                                   // buffer `buf` is refilled by tile tj + 2
    }
}

}  // namespace

int ab_launch_scale_inputs(ab_gp* h) {
    int64_t tot = h->npad * h->d;
    scale_inputs_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(h->X, h->n, h->npad, h->d, h->kp,
                                                                            h->Xs, h->XsT);
    AB_CHECK_LAUNCH();
    return 0;
}

// Symmetric training covariance.  pad_identity: build the npad x npad padded
// matrix (ld >= npad) for the factorisation; else the plain n x n matrix.
int ab_launch_cov(ab_gp* h, double* K, int64_t ld, int mirror, int pad_identity) {
    int64_t rows = pad_identity ? h->npad : h->n;
    int64_t nt = (rows + 63) / 64;
    int64_t ntiles = nt * (nt + 1) / 2;
    if (pad_identity && !mirror && (ld & 1) == 0 && (reinterpret_cast<uintptr_t>(K) & 15) == 0) {
        // strips of tiles: long enough to amortise the row inputs, short enough to fill the GPU
        int seg = (int)(ntiles / ((int64_t)h->nsm * 6));
        seg = seg < 1 ? 1 : (seg > 16 ? 16 : seg);
        if (h->cov_items_nt != (int)nt || h->cov_items_seg != seg) {
            std::vector<int2> items;
            for (int ti = (int)nt - 1; ti >= 0; ti--)                 // longest rows first
                for (int t0 = 0; t0 <= ti; t0 += seg) items.push_back(make_int2(ti, t0));
            if (h->cov_items) cudaFree(h->cov_items);
            h->cov_items = nullptr;
            AB_CUDA(cudaMalloc(&h->cov_items, items.size() * sizeof(int2)));
            AB_CUDA(cudaMemcpyAsync(h->cov_items, items.data(), items.size() * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
            AB_CUDA(cudaStreamSynchronize(h->stream));
            h->cov_items_nt = (int)nt;
            h->cov_items_seg = seg;
            h->cov_items_count = (int)items.size();
        }
        ab_prof_begin(h, AB_PROF_COV);
        AB_DISPATCH_KIND(h->kp.kind, (cov_strip_kernel<KIND><<<(unsigned)h->cov_items_count, 256, 0, h->stream>>>(
                                         h->XsT, h->npad, h->n, h->kp, K, ld, seg, reinterpret_cast<const int2*>(h->cov_items))));
        ab_prof_end(h, AB_PROF_COV);
        ab_count_launches(1);
        AB_CHECK_LAUNCH();
        return 0;
    }
    ab_prof_begin(h, AB_PROF_COV);
    AB_DISPATCH_KIND(h->kp.kind, (cov_kernel<KIND><<<(unsigned)ntiles, 256, 0, h->stream>>>(
                                     h->XsT, h->npad, rows, h->XsT, h->npad, rows, h->n, h->kp, K, ld, 1, mirror,
                                     pad_identity)));
    ab_prof_end(h, AB_PROF_COV);
    ab_count_launches(1);
    AB_CHECK_LAUNCH();
    return 0;
}

// General cross covariance amp * k(A, B) for SoA point sets already scaled.
int ab_launch_cross_cov(ab_gp* h, const double* AT, int64_t lda, int64_t na, const double* BT, int64_t ldb,
                        int64_t nb, double* K, int64_t ld) {
    dim3 grid((unsigned)((nb + 63) / 64), (unsigned)((na + 63) / 64));
    AB_DISPATCH_KIND(h->kp.kind, (cov_kernel<KIND><<<grid, 256, 0, h->stream>>>(AT, lda, na, BT, ldb, nb, 0, h->kp, K,
                                                                              ld, 0, 0, 0)));
    AB_CHECK_LAUNCH();
    return 0;
}

int ab_launch_scale_points(ab_gp* h, const double* X, int64_t m, double* XT, int64_t ldm) {
    int64_t tot = m * h->d;
    if (tot <= 0) return 0;
    scale_points_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(X, m, h->d, h->kp, XT, ldm);
    AB_CHECK_LAUNCH();
    return 0;
}
