// Bordered Cholesky update: append ONE training point to a factorised GP in O(N^2).
//
// Replaces the full refactorisation the reference performs after every active-
// learning step (`_fit_gp` -> `gp.compute`, alabi/core.py:1780 -> 1158) when only a
// point was appended and the hyper-parameters are unchanged (SURVEY 8f.4):
//
//     K' = [ K   k ]      L' = [ L    0 ]     l = L^-1 k,
//          [ k^T c ]           [ l^T  s ]     s = sqrt(c - l.l),  c = amp k(0) + diag
//
// In the padded layout row n of L is an identity row, so the update overwrites that
// row, rebuilds the inverse of the one diagonal block that contains it, and leaves
// every other tile untouched.  When n is a multiple of 128 the padded matrix first
// grows by one identity block (re-layout with the new leading dimension).
#include "handle.h"
#include "alabi_b200.h"

namespace {

constexpr int NB = AB_NB;

// k_j = amp * k(x_j, x_new) for j < n0, zero padding above; Xs already holds the new
// point as row n0 (scaled)
template <int KIND>
__global__ void append_cross_kernel(const double* __restrict__ Xs, int64_t n0, int64_t npad, int d, KernParams kp,
                                    double* __restrict__ out) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= npad) return;
    double v = 0.0;
    if (j < n0) {
        double r2 = 0.0;
        for (int k = 0; k < d; k++) {
            const double df = Xs[j * d + k] - Xs[n0 * d + k];
            r2 = fma(df, df, r2);
        }
        v = kp.amp * ab_radial<KIND>(r2, kp.alpha, kp.inv2a);
    }
    out[j] = v;
}

// s^2 = c - |l|^2; on success write row n0 of L (info stays 0), else info = n0 + 1
template <int KIND>
__global__ void __launch_bounds__(1024)
append_row_kernel(double* __restrict__ L, int64_t ld, int64_t n0, const double* __restrict__ l, KernParams kp,
                  int* __restrict__ info) {
    __shared__ double sh[32];
    __shared__ double s_lam;
    double s = 0.0;
    for (int64_t j = threadIdx.x; j < n0; j += 1024) s = fma(l[j], l[j], s);
    s = ab_warp_sum(s);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double q = 0.0;
        for (int w = 0; w < 32; w++) q += sh[w];
        const double lam2 = kp.amp * ab_radial<KIND>(0.0, kp.alpha, kp.inv2a) + kp.diag_add - q;
        if (!(lam2 > 0.0)) { *info = (int)(n0 + 1); s_lam = -1.0; }
        else s_lam = sqrt(lam2);
    }
    __syncthreads();
    const double lam = s_lam;
    if (lam < 0.0) return;
    for (int64_t j = threadIdx.x; j < n0; j += 1024) L[n0 * ld + j] = l[j];
    if (threadIdx.x == 0) L[n0 * ld + n0] = lam;
}

// New row of L^-1 after the bordered update:  Linv'[n0][j] = -(1/s) sum_{i<n0} l_i Linv[i][j],
// Linv'[n0][n0] = 1/s.  Column j per thread (rows are read coalesced), the row range split
// over grid.y into fixed chunks; linv_row_finish adds the chunk sums in order.
constexpr int LR_CHUNK = 1024;
__global__ void __launch_bounds__(128)
linv_row_partial_kernel(const double* __restrict__ Linv, int64_t ld, int64_t n0, const double* __restrict__ l,
                        double* __restrict__ part, int64_t part_ld) {
    const int64_t j = (int64_t)blockIdx.x * 128 + threadIdx.x;
    const int64_t i0 = (int64_t)blockIdx.y * LR_CHUNK;
    int64_t i1 = i0 + LR_CHUNK < n0 ? i0 + LR_CHUNK : n0;
    double s = 0.0;
    if (j < n0) {
        int64_t ib = i0 > j ? i0 : j;                      // Linv is lower triangular: rows i >= j
        for (int64_t i = ib; i < i1; i++) s = fma(l[i], Linv[i * ld + j], s);
    }
    part[(int64_t)blockIdx.y * part_ld + j] = s;
}
__global__ void linv_row_finish_kernel(double* __restrict__ Linv, int64_t ld, int64_t n0, const double* __restrict__ L,
                                       const double* __restrict__ part, int64_t part_ld, int nchunk) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const double inv_s = 1.0 / L[n0 * ld + n0];
    if (j < n0) {
        double s = 0.0;
        for (int c = 0; c < nchunk; c++) s += part[(int64_t)c * part_ld + j];
        Linv[n0 * ld + j] = -inv_s * s;
    } else if (j == n0) {
        Linv[n0 * ld + n0] = inv_s;
    }
}

// new identity block rows [npad0, npad1) of the re-laid-out factor
__global__ void pad_identity_rows_kernel(double* __restrict__ L, int64_t ld, int64_t r0) {
    const int64_t row = r0 + blockIdx.x;
    for (int64_t c = threadIdx.x; c < ld; c += blockDim.x) L[row * ld + c] = (c == row) ? 1.0 : 0.0;
}

__global__ void identity_block_kernel(double* __restrict__ D) {
    for (int idx = threadIdx.x; idx < NB * NB; idx += blockDim.x) D[idx] = ((idx >> 7) == (idx & (NB - 1))) ? 1.0 : 0.0;
}

template <typename T>
int grow(T** p, size_t old_count, size_t new_count, cudaStream_t s) {
    T* q = nullptr;
    AB_CUDA(cudaMalloc(&q, new_count * sizeof(T)));
    cudaError_t e = cudaSuccess;
    if (*p && old_count) e = cudaMemcpyAsync(q, *p, old_count * sizeof(T), cudaMemcpyDeviceToDevice, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) {          // the old buffer stays in place, the new one is released
        cudaFree(q);
        ab_set_error("grow: copy failed: %s", cudaGetErrorString(e));
        return -100 - (int)e;
    }
    if (*p) AB_CUDA(cudaFree(*p));
    *p = q;
    return 0;
}

// one more identity block: npad -> npad + 128 (new leading dimension)
int grow_padded(ab_gp* h) {
    const int64_t np0 = h->npad, np1 = np0 + NB;
    cudaStream_t s = h->stream;
    const int d = h->d;
    // capacity: grow geometrically so that a long active-learning run re-allocates rarely
    int64_t cap = h->cap_pad;
    if (np1 > cap) {
        cap = np1 + (np1 / 4 + NB - 1) / NB * NB;
        int rc = grow(&h->X, (size_t)h->n * d, (size_t)cap * h->cap_d, s);
        if (rc) return rc;
        double* bufs_free[] = {h->Xs, h->XsT, h->alpha, h->z, h->work};
        for (double* b : bufs_free) if (b) AB_CUDA(cudaFree(b));
        h->Xs = h->XsT = h->alpha = h->z = h->work = nullptr;
        AB_CUDA(cudaMalloc(&h->Xs, (size_t)cap * h->cap_d * sizeof(double)));
        AB_CUDA(cudaMalloc(&h->XsT, (size_t)cap * h->cap_d * sizeof(double)));
        AB_CUDA(cudaMalloc(&h->alpha, (size_t)cap * sizeof(double)));
        AB_CUDA(cudaMalloc(&h->z, (size_t)cap * sizeof(double)));
        AB_CUDA(cudaMalloc(&h->work, (size_t)cap * sizeof(double)));
        rc = grow(&h->Dinv, (size_t)np0 * NB, (size_t)cap * NB, s);
        if (!rc) rc = grow(&h->logdet_parts, (size_t)np0 / NB, (size_t)cap / NB, s);
        if (rc) return rc;
    }
    // factor: new buffer (when the capacity grew) or a second buffer of the same capacity;
    // rows are re-laid-out from leading dimension np0 to np1
    double* Lnew = nullptr;
    AB_CUDA(cudaMalloc(&Lnew, (size_t)cap * cap * sizeof(double)));
    AB_CUDA(cudaMemsetAsync(Lnew, 0, (size_t)np1 * np1 * sizeof(double), s));
    AB_CUDA(cudaMemcpy2DAsync(Lnew, (size_t)np1 * sizeof(double), h->L, (size_t)np0 * sizeof(double),
                              (size_t)np0 * sizeof(double), (size_t)np0, cudaMemcpyDeviceToDevice, s));
    pad_identity_rows_kernel<<<NB, 256, 0, s>>>(Lnew, np1, np0);
    identity_block_kernel<<<1, 256, 0, s>>>(h->Dinv + (size_t)np0 * NB);
    AB_CUDA(cudaMemsetAsync(h->logdet_parts + np0 / NB, 0, sizeof(double), s));
    AB_CHECK_LAUNCH();
    AB_CUDA(cudaStreamSynchronize(s));
    AB_CUDA(cudaFree(h->L));
    h->L = Lnew;
    h->cap_pad = cap;
    h->npad = np1;
    // the inverse buffers follow the capacity lazily (ensure_inverse_buffers)
    h->have_linv = h->have_kinv = false;
    if (h->inv_cap_pad < cap) h->inv_cap_pad = 0;
    return 0;
}

}  // namespace

extern "C" int ab_gp_append_point(ab_gp* h, const double* d_x) {
    if (!h || !d_x) { ab_set_error("ab_gp_append_point: null argument"); return -1; }
    if (!h->factored || !h->have_kernel) { ab_set_error("ab_gp_append_point: not factorised"); return -2; }
    AB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int64_t n0 = h->n;
    int rc;
    if (n0 == h->npad) {
        rc = grow_padded(h);
        if (rc) return rc;
    }
    const int64_t ld = h->npad;
    AB_CUDA(cudaMemcpyAsync(h->X + (size_t)n0 * h->d, d_x, (size_t)h->d * sizeof(double), cudaMemcpyDeviceToDevice, s));
    h->n = n0 + 1;
    rc = ab_launch_scale_inputs(h);                       // Xs, XsT with the new row (N d work)
    if (rc) { h->n = n0; return rc; }
    AB_DISPATCH_KIND(h->kp.kind, (append_cross_kernel<KIND><<<(unsigned)((ld + 255) / 256), 256, 0, s>>>(
                                     h->Xs, n0, ld, h->d, h->kp, h->work)));
    AB_CUDA(cudaMemsetAsync(h->d_info, 0, sizeof(int), s));
    *reinterpret_cast<int*>(h->h_pinned + 10) = 0;
    if (ld / NB >= 2) {
        rc = ab_launch_trsv_dataflow(h, h->work, 0);      // forward only: z = L^-1 k
    } else {
        rc = ab_launch_trsv_single(h, h->work);
    }
    if (rc) { h->n = n0; return rc; }
    AB_DISPATCH_KIND(h->kp.kind, (append_row_kernel<KIND><<<1, 1024, 0, s>>>(h->L, ld, n0, h->z, h->kp, h->d_info)));
    AB_CHECK_LAUNCH();
    rc = ab_launch_rebuild_dinv_block(h, (int)(n0 / NB));
    if (rc) { h->n = n0; return rc; }
    ab_count_launches(5);
    bool keep_linv = false;
    if (h->have_linv && h->Linv) {
        // L^-1 follows in O(N^2) as well (its row n0 was the identity row of the padding)
        const int nchunk = (int)((n0 + LR_CHUNK - 1) / LR_CHUNK);
        rc = ab_ensure_scratch(h, 256 + ((size_t)(nchunk > 0 ? nchunk : 1) * ld + (size_t)(2 * (ld / NB) + 64)) * sizeof(double));
        if (rc) { h->n = n0; return rc; }
        double* part = h->scratch + 32 + (2 * (ld / NB) + 64);       // behind the solve's control words
        if (nchunk > 0)
            linv_row_partial_kernel<<<dim3((unsigned)(ld / 128), (unsigned)nchunk), 128, 0, s>>>(h->Linv, ld, n0, h->z, part, ld);
        linv_row_finish_kernel<<<(unsigned)((n0 + 1 + 255) / 256), 256, 0, s>>>(h->Linv, ld, n0, h->L, part, ld, nchunk);
        AB_CHECK_LAUNCH();
        ab_count_launches(2);
        keep_linv = true;
    }
    AB_CUDA(cudaMemcpyAsync(h->h_pinned + 8, h->d_info, sizeof(int), cudaMemcpyDeviceToHost, s));
    AB_CUDA(cudaStreamSynchronize(s));
    h->have_linv = keep_linv;
    h->have_kinv = h->have_alpha = false;
    if (*reinterpret_cast<int*>(h->h_pinned + 10) != 0) {
        ab_set_error("dataflow triangular solve watchdog fired");
        h->factored = false;
        return -5;
    }
    const int info = *reinterpret_cast<int*>(h->h_pinned + 8);
    if (info != 0) {                                       // not positive definite with the new point
        h->info = info;
        h->factored = false;
        h->have_linv = false;
        ab_set_error("matrix not positive definite after appending a point: pivot %d", info);
        return info;
    }
    return 0;
}
