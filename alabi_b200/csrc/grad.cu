// K2 (gradient): fused hyper-parameter gradient of the log marginal likelihood.
//
//   grad_theta = 1/2 sum_ij (alpha_i alpha_j - Kinv_ij) dK_ij/dtheta
//
// Replaces george GP.grad_log_likelihood (alabi/core.py:1261), which materialises
// dK as an N x N x P array (49 GB at N = 16384, d = 20).  Here K^-1 is read
// exactly once (lower tiles, weight 2 off the diagonal) and all P = d + 3
// trace terms (d + 4 for the rational quadratic kernel) are accumulated in
// registers; distances and kernel derivatives are recomputed on the fly from
// the scaled inputs in shared memory.
// Output order: [mean, white_noise, log_constant, log_M_0 .. log_M_{d-1}], and
// [mean, white_noise, log_constant, log_alpha, log_M_0 .. log_M_{d-1}] for the
// rational quadratic kernel (george's parameter order).
#include "handle.h"
#include "dmma_gemm.cuh"

namespace {

constexpr int NB = AB_NB;
// trace terms a kernel family adds to [white_noise, log_constant, log_M...]: the rational
// quadratic kernel's log_alpha
template <int KIND> constexpr int kExtra = (KIND == 3) ? 1 : 0;

template <int KIND, int DMAX>
__global__ void __launch_bounds__(256, (DMAX <= 8) ? 3 : ((DMAX <= 20) ? 2 : 1))
grad_tiles_kernel(const double* __restrict__ Kinv, int64_t ld, const double* __restrict__ XsT, int64_t npad,
                  int64_t n, const double* __restrict__ alpha, KernParams kp, double* __restrict__ partials) {
    extern __shared__ __align__(16) double sm[];
    double* sXi = sm;                      // [DMAX][NB]
    double* sXj = sm + DMAX * NB;          // [DMAX][NB]
    double* sAi = sm + 2 * DMAX * NB;      // [NB]
    double* sAj = sAi + NB;                // [NB]
    double* sred = sAj + NB;               // [8][DMAX + 2 + NX]
    constexpr int NX = kExtra<KIND>, RS = DMAX + 2 + NX;
    int ti, tj;
    abg::tri_decode(blockIdx.x, ti, tj);
    const int64_t i0 = (int64_t)ti * NB, j0 = (int64_t)tj * NB;
    const int tid = threadIdx.x, d = kp.d;
    for (int idx = tid; idx < d * NB; idx += 256) {
        int k = idx >> 7, r = idx & (NB - 1);
        sXi[k * NB + r] = XsT[(int64_t)k * npad + i0 + r];
        sXj[k * NB + r] = XsT[(int64_t)k * npad + j0 + r];
    }
    if (tid < NB) { sAi[tid] = alpha[i0 + tid]; sAj[tid] = alpha[j0 + tid]; }
    __syncthreads();
    const int c = tid & (NB - 1), half = tid >> 7;
    const double wt = (ti == tj) ? 1.0 : 2.0;
    double s_tr = 0.0, s_c = 0.0, s_a = 0.0, s_m[DMAX];
    double xj[DMAX];
#pragma unroll
    for (int k = 0; k < DMAX; k++) { s_m[k] = 0.0; xj[k] = (k < d) ? sXj[k * NB + c] : 0.0; }
    const double aj = sAj[c];
    const bool col_ok = (j0 + c) < n;
    for (int r = half; r < NB; r += 2) {
        const int64_t gi = i0 + r;
        if (gi >= n || !col_ok) continue;
        double d2[DMAX], r2 = 0.0;
#pragma unroll
        for (int k = 0; k < DMAX; k++) {
            if (k < d) {
                double df = sXi[k * NB + r] - xj[k];
                d2[k] = df * df;
                r2 += d2[k];
            } else d2[k] = 0.0;
        }
        const double a = wt * (sAi[r] * aj - Kinv[gi * ld + j0 + c]);
        double kv, gv, av;
        ab_radial_both<KIND, true>(r2, kp.alpha, kp.inv2a, kv, gv, av);   // one exponential for k and dk/d(r^2)
        s_c = fma(a, kp.amp * kv, s_c);
        if (NX) s_a = fma(a, kp.amp * av, s_a);
        const double gk = -a * kp.amp * gv;
#pragma unroll
        for (int k = 0; k < DMAX; k++)
            if (k < d) s_m[k] = fma(gk, d2[k], s_m[k]);
        if (gi == j0 + c) s_tr += a;
    }
    // block reduction in a fixed order
    const int lane = tid & 31, warp = tid >> 5;
    double v;
    v = ab_warp_sum(s_tr); if (lane == 0) sred[warp * RS + 0] = v;
    v = ab_warp_sum(s_c);  if (lane == 0) sred[warp * RS + 1] = v;
    if (NX) { v = ab_warp_sum(s_a); if (lane == 0) sred[warp * RS + 2] = v; }
#pragma unroll
    for (int k = 0; k < DMAX; k++) {
        if (k < d) { v = ab_warp_sum(s_m[k]); if (lane == 0) sred[warp * RS + 2 + NX + k] = v; }
    }
    __syncthreads();
    if (tid < d + 2 + NX) {
        double s = 0.0;
        for (int w = 0; w < 8; w++) s += sred[w * RS + tid];
        partials[(int64_t)blockIdx.x * (AB_MAX_DIM + 2 + NX) + tid] = s;
    }
}

template <int NX>
__global__ void __launch_bounds__(256)
grad_final_kernel(const double* __restrict__ partials, int ntiles, const double* __restrict__ alpha, int64_t n,
                  int d, double wn_scale, double* __restrict__ out) {
    __shared__ double sh[8];
    const int tid = threadIdx.x;
    // out[0] = sum alpha (mean gradient)
    double s = 0.0;
    for (int64_t i = tid; i < n; i += 256) s += alpha[i];
    s = ab_warp_sum(s);
    if ((tid & 31) == 0) sh[tid >> 5] = s;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; w++) t += sh[w];
        out[0] = t;
    }
    // tile partials: output w, w + 8, ... by warp w; lanes stride over the tiles, fixed-order tree
    const int lane = tid & 31, warp = tid >> 5;
    for (int o = warp; o < d + 2 + NX; o += 8) {
        double t = 0.0;
        for (int p = lane; p < ntiles; p += 32) t += partials[(int64_t)p * (AB_MAX_DIM + 2 + NX) + o];
        t = ab_warp_sum(t);
        if (lane == 0) out[1 + o] = 0.5 * t * (o == 0 ? wn_scale : 1.0);
    }
}

}  // namespace

// Needs h->Kinv and h->alpha.  Leaves d + 3 doubles (d + 4 for the rational quadratic kernel) in
// h->h_pinned (async copy).
int ab_launch_grad(ab_gp* h) {
    const int T = (int)(h->npad / NB);
    const int ntiles = T * (T + 1) / 2;
    const int nx = (h->kp.kind == 3) ? kExtra<3> : 0;
    size_t need = (size_t)ntiles * (AB_MAX_DIM + 2 + nx) * sizeof(double) + 64 * sizeof(double);
    int rc = ab_ensure_scratch(h, need);
    if (rc) return rc;
    double* partials = h->scratch + 64;
    cudaStream_t s = h->stream;
    // the per-dimension loops are unrolled over the template dimension: instantiate the padded
    // dimension of the problem, not AB_MAX_DIM (d = 10 ran 32-long predicated loops with 230 registers)
    rc = ab_dispatch_dim(h->d, [&](auto DM) {
        AB_DISPATCH_KIND(h->kp.kind, {
            const int smem = (2 * DM * NB + 2 * NB + 8 * (DM + 2 + kExtra<KIND>)) * 8;
            AB_CUDA(cudaFuncSetAttribute(grad_tiles_kernel<KIND, DM>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
            grad_tiles_kernel<KIND, DM><<<ntiles, 256, smem, s>>>(h->Kinv, h->npad, h->XsT, h->npad, h->n, h->alpha,
                                                                  h->kp, partials);
        });
        return 0;
    });
    if (rc) return rc;
    AB_CHECK_LAUNCH();
    if (nx) grad_final_kernel<1><<<1, 256, 0, s>>>(partials, ntiles, h->alpha, h->n, h->d, exp(h->white_noise), h->scratch);
    else grad_final_kernel<0><<<1, 256, 0, s>>>(partials, ntiles, h->alpha, h->n, h->d, exp(h->white_noise), h->scratch);
    AB_CHECK_LAUNCH();
    AB_CUDA(cudaMemcpyAsync(h->h_pinned, h->scratch, (h->d + 3 + nx) * sizeof(double), cudaMemcpyDeviceToHost, s));
    return 0;
}
