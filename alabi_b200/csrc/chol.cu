// K2 around the factorisation: the factor itself is the dataflow kernel in
// chol_dataflow.cu; this file holds what the log-likelihood, its gradient and the
// predictive variance need from an existing factor L:
//   * the triangular inverse L^-1 (recursive halving, DMMA GEMMs) and K^-1 = L^-T L^-1;
//   * the rebuild of the diagonal-block inverses D_k^-1 and log-determinant parts of
//     an imported or bordered factor (potf2_inv_kernel);
//   * the triangular solves of a one-block factor, the residual and the final sums.
// The block triangular solves of larger factors live in trsv_dataflow.cu.
//
// With chol_dataflow.cu, replaces george BasicSolver.compute / apply_inverse /
// get_inverse (scipy cholesky + cho_solve) reached from alabi/gp_utils.py:243,
// alabi/core.py:1158, 1248, 1261, 1430.  Matrix layout: row-major, lower triangle,
// padded to a multiple of AB_NB = 128 with an identity block so every tile is full.
#include <vector>
#include "handle.h"
#include "dmma_gemm.cuh"
#include "potf2.cuh"

namespace {

constexpr int NB = AB_NB;

// grid = number of diagonal blocks; the matrix already holds L (an imported or bordered
// factor): rebuild D^-1 and the log-determinant parts with the sweep of potf2.cuh.
// CTA b works on the block at offset b * NB (the argument o is overwritten).
__global__ void __launch_bounds__(256, 1)
potf2_inv_kernel(double* __restrict__ A, int64_t ld, int64_t o, double* __restrict__ Dinv,
                 double* __restrict__ logdet_part, int* __restrict__ info) {
    o = (int64_t)blockIdx.x * NB;
    Dinv += (int64_t)blockIdx.x * NB * NB;
    logdet_part += blockIdx.x;
    __shared__ abp::SweepShared sh;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    if (tid == 0) abp::mbar_init((unsigned)__cvta_generic_to_shared(&sh.mbar), 256);
    __syncthreads();
    double a[8][8], b[8][8];
#pragma unroll
    for (int r = 0; r < 8; r++)
#pragma unroll
        for (int c = 0; c < 8; c++) {
            // only the lower block triangle (r >= c) is ever referenced: the rest
            // must not occupy registers
            if (r >= c) {
                const int i = ty + 16 * r, k = tx + 16 * c;
                a[r][c] = (k <= i) ? A[(o + i) * ld + o + k] : 0.0;
                b[r][c] = (k == i) ? 1.0 : 0.0;
            }
        }
    unsigned phase = 0;
    abp::potf2_sweep<false, 8>(a, b, sh, tx, ty, o, info, phase);
    double* sdiag = sh.sdiag;
    double* sinv = sh.sinv;
    if (tid < 32) {
        double s = 0.0;
        for (int j = tid; j < NB; j += 32) s += 2.0 * log(sdiag[j]);
        s = ab_warp_sum(s);
        if (tid == 0) *logdet_part = s;
    }
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const int i = ty + 16 * r;
        const double si = sinv[i];
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const int k = tx + 16 * c;
            Dinv[i * NB + k] = (r >= c && k <= i) ? b[r][c] * si : 0.0;
        }
    }
}

// ---------------------------------------------------------------------------
// blocked triangular solves for z = L^-1 r and alpha = L^-T z
// ---------------------------------------------------------------------------
// forward step k: every CTA recomputes z_k = D_k^-1 r_k; CTA 0 stores it, CTA b >= 1
// applies r_{k+b} -= L_{k+b,k} z_k.
__global__ void __launch_bounds__(256)
trsv_fwd_kernel(const double* __restrict__ L, int64_t ld, const double* __restrict__ Dinv, int k,
                double* __restrict__ r, double* __restrict__ z) {
    __shared__ double sr[NB], sz[NB];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t o = (int64_t)k * NB;
    if (tid < NB) sr[tid] = r[o + tid];
    __syncthreads();
    const double* D = Dinv + (int64_t)k * NB * NB;
    for (int row = warp; row < NB; row += 8) {
        double s = 0.0;
#pragma unroll
        for (int c = lane; c < NB; c += 32) s = fma(D[row * NB + c], sr[c], s);
        s = ab_warp_sum(s);
        if (lane == 0) sz[row] = s;
    }
    __syncthreads();
    if (blockIdx.x == 0) {
        if (tid < NB) z[o + tid] = sz[tid];
        return;
    }
    const int64_t rb = o + (int64_t)blockIdx.x * NB;
    for (int row = warp; row < NB; row += 8) {
        const double* Lr = L + (rb + row) * ld + o;
        double s = 0.0;
#pragma unroll
        for (int c = lane; c < NB; c += 32) s = fma(Lr[c], sz[c], s);
        s = ab_warp_sum(s);
        if (lane == 0) r[rb + row] -= s;
    }
}

// backward step k: alpha_k = D_k^-T z_k (CTA 0 stores), CTA b >= 1 applies
// z_{b-1} -= L_{k,b-1}^T alpha_k.
__global__ void __launch_bounds__(NB)
trsv_bwd_kernel(const double* __restrict__ L, int64_t ld, const double* __restrict__ Dinv, int k,
                double* __restrict__ z, double* __restrict__ alpha) {
    __shared__ double sz[NB], sa[NB];
    const int tid = threadIdx.x;
    const int64_t o = (int64_t)k * NB;
    sz[tid] = z[o + tid];
    __syncthreads();
    const double* D = Dinv + (int64_t)k * NB * NB;
    double s0 = 0.0, s1 = 0.0;
#pragma unroll 4
    for (int c = 0; c < NB; c += 2) {
        s0 = fma(D[c * NB + tid], sz[c], s0);
        s1 = fma(D[(c + 1) * NB + tid], sz[c + 1], s1);
    }
    sa[tid] = s0 + s1;
    __syncthreads();
    if (blockIdx.x == 0) {
        alpha[o + tid] = sa[tid];
        return;
    }
    const int64_t cb = (int64_t)(blockIdx.x - 1) * NB;
    const double* Lp = L + o * ld + cb + tid;
    s0 = s1 = 0.0;
#pragma unroll 4
    for (int c = 0; c < NB; c += 2) {
        s0 = fma(Lp[(int64_t)c * ld], sa[c], s0);
        s1 = fma(Lp[(int64_t)(c + 1) * ld], sa[c + 1], s1);
    }
    z[cb + tid] -= s0 + s1;
}

__global__ void residual_kernel(const double* __restrict__ y, int64_t n, int64_t npad, double mean,
                                double* __restrict__ r) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < npad) r[i] = (i < n) ? y[i] - mean : 0.0;
}

// single CTA, fixed summation order: out[0] = sum v^2, out[1] = sum parts
__global__ void __launch_bounds__(1024)
final_sums_kernel(const double* __restrict__ v, int64_t n, const double* __restrict__ parts, int nparts,
                  double* __restrict__ out) {
    __shared__ double sh[32];
    double s = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) s = fma(v[i], v[i], s);
    s = ab_warp_sum(s);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double q = 0.0;
        for (int w = 0; w < 32; w++) q += sh[w];
        double ld = 0.0;
        for (int p = 0; p < nparts; p++) ld += parts[p];
        out[0] = q;
        out[1] = ld;
    }
}

// ---------------------------------------------------------------------------
// triangular inverse by recursive halving and K^-1 = L^-T L^-1
// ---------------------------------------------------------------------------
struct InvNode { int r0, h, n2, tile_begin; };          // block units
struct InvLevel { int nnodes; InvNode nodes[64]; };

__global__ void copy_diag_blocks_kernel(const double* __restrict__ Dinv, double* __restrict__ Linv, int64_t ld) {
    const int64_t o = (int64_t)blockIdx.x * NB;
    const double* D = Dinv + (int64_t)blockIdx.x * NB * NB;
    for (int idx = threadIdx.x; idx < NB * NB; idx += blockDim.x) {
        int i = idx >> 7, j = idx & (NB - 1);
        Linv[(o + i) * ld + o + j] = D[idx];
    }
}

// PASS 1: W21 = L21 * Linv11 ; PASS 2: Linv21 = -Linv22 * W21
template <int PASS>
__global__ void __launch_bounds__(abg::THREADS, 1)
trinv_kernel(const double* __restrict__ L, double* __restrict__ Linv, double* __restrict__ W, int64_t ld,
             const __grid_constant__ InvLevel lv) {
    extern __shared__ __align__(16) double smem[];
    int nd = 0;
    for (int q = 1; q < lv.nnodes; q++)
        if ((int)blockIdx.x >= lv.nodes[q].tile_begin) nd = q;
    const InvNode node = lv.nodes[nd];
    const int p = blockIdx.x - node.tile_begin;
    const int i = p / node.h, j = p % node.h;
    const int64_t rowi = (int64_t)(node.r0 + node.h + i) * NB, colj = (int64_t)(node.r0 + j) * NB;
    abg::Acc acc;
    acc.zero();
    if (PASS == 1) {
        const double* Ap = L + rowi * ld + colj;                 // k starts at block j
        const double* Bp = Linv + colj * ld + colj;
        abg::mainloop<true, false>(acc, Ap, ld, Bp, ld, (node.h - j) * (NB / abg::BK), smem);
        abg::store_tile(acc, W + rowi * ld + colj, ld, 1.0, 0.0);
    } else {
        const int64_t k0 = (int64_t)(node.r0 + node.h) * NB;
        const double* Ap = Linv + rowi * ld + k0;
        const double* Bp = W + k0 * ld + colj;
        abg::mainloop<true, false>(acc, Ap, ld, Bp, ld, (i + 1) * (NB / abg::BK), smem);
        abg::store_tile(acc, Linv + rowi * ld + colj, ld, -1.0, 0.0);
    }
}

// Kinv(i, j) = sum_{k >= i} Linv(k, i)^T Linv(k, j), j <= i
__global__ void __launch_bounds__(abg::THREADS, 1)
kinv_kernel(const double* __restrict__ Linv, double* __restrict__ Kinv, int64_t ld, int T) {
    extern __shared__ __align__(16) double smem[];
    int i, j;
    abg::tri_decode(blockIdx.x, i, j);
    abg::Acc acc;
    acc.zero();
    const double* Ap = Linv + (int64_t)i * NB * ld + (int64_t)i * NB;
    const double* Bp = Linv + (int64_t)i * NB * ld + (int64_t)j * NB;
    abg::mainloop<false, false>(acc, Ap, ld, Bp, ld, (T - i) * (NB / abg::BK), smem);
    abg::store_tile(acc, Kinv + (int64_t)i * NB * ld + (int64_t)j * NB, ld, 1.0, 0.0);
}

__global__ void mirror_lower_kernel(double* __restrict__ A, int64_t ld, int64_t n) {
    __shared__ double t[32][33];
    int bi = blockIdx.y, bj = blockIdx.x;
    if (bj >= bi) return;                       // strictly-lower tiles -> upper
    int x = threadIdx.x, y = threadIdx.y;
    for (int yy = y; yy < 32; yy += 8) {
        int64_t r = (int64_t)bi * 32 + yy, c = (int64_t)bj * 32 + x;
        t[yy][x] = (r < n && c < n) ? A[r * ld + c] : 0.0;
    }
    __syncthreads();
    for (int yy = y; yy < 32; yy += 8) {
        int64_t r = (int64_t)bj * 32 + yy, c = (int64_t)bi * 32 + x;
        if (r < n && c < n) A[r * ld + c] = t[x][yy];
    }
}
__global__ void mirror_diag_tiles_kernel(double* __restrict__ A, int64_t ld, int64_t n) {
    int64_t o = (int64_t)blockIdx.x * 32;
    for (int idx = threadIdx.x; idx < 32 * 32; idx += blockDim.x) {
        int i = idx >> 5, j = idx & 31;
        if (j > i && o + j < n) A[(o + i) * ld + o + j] = A[(o + j) * ld + o + i];
    }
}

template <typename F>
int set_smem(F f, int bytes) {
    AB_CUDA(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    return 0;
}

// cudaFuncSetAttribute is per device: remember which devices are configured
int configure_once() {
    static unsigned long long done_mask = 0;
    int dev = 0;
    AB_CUDA(cudaGetDevice(&dev));
    const bool done = dev < 64 && ((done_mask >> dev) & 1ULL);
    if (done) return 0;
    int rc = 0;
    rc |= set_smem(trinv_kernel<1>, abg::SMEM_BYTES);
    rc |= set_smem(trinv_kernel<2>, abg::SMEM_BYTES);
    rc |= set_smem(kinv_kernel, abg::SMEM_BYTES);
    if (rc) return rc;
    if (dev < 64) done_mask |= 1ULL << dev;
    return 0;
}

// returns the height of the subtree rooted at blocks [r0, r0 + nblk)
int inv_tree(int r0, int nblk, std::vector<std::vector<InvNode>>& levels) {
    if (nblk <= 1) return 0;
    int h = nblk / 2, n2 = nblk - h;
    int ha = inv_tree(r0, h, levels), hb = inv_tree(r0 + h, n2, levels);
    int ht = 1 + (ha > hb ? ha : hb);
    if ((int)levels.size() < ht + 1) levels.resize(ht + 1);
    levels[ht].push_back(InvNode{r0, h, n2, 0});
    return ht;
}
}  // namespace

int ab_launch_rebuild_dinv(ab_gp* h) {
    int rc = configure_once();
    if (rc) return rc;
    const int T = (int)(h->npad / NB);
    potf2_inv_kernel<<<T, 256, 0, h->stream>>>(h->L, h->npad, 0, h->Dinv, h->logdet_parts, h->d_info);
    AB_CHECK_LAUNCH();
    return 0;
}

// inverse and log-determinant part of ONE diagonal block of an existing factor
int ab_launch_rebuild_dinv_block(ab_gp* h, int kb) {
    int rc = configure_once();
    if (rc) return rc;
    const int64_t o = (int64_t)kb * NB;
    potf2_inv_kernel<<<1, 256, 0, h->stream>>>(h->L + o * h->npad + o, h->npad, 0, h->Dinv + o * NB,
                                               h->logdet_parts + kb, h->d_info);
    AB_CHECK_LAUNCH();
    return 0;
}

// one-block factor: z = D_0^-1 r (r is not modified)
int ab_launch_trsv_single(ab_gp* h, const double* r) {
    AB_CUDA(cudaMemcpyAsync(h->alpha, r, NB * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));   // alpha: scratch here
    trsv_fwd_kernel<<<1, 256, 0, h->stream>>>(h->L, h->npad, h->Dinv, 0, h->alpha, h->z);
    AB_CHECK_LAUNCH();
    return 0;
}

// z = L^-1 (y - mean), alpha = L^-T z, quad = |z|^2, logdet = sum parts.
// Leaves {quad, logdet} in h->h_pinned[0..1] after a stream sync by the caller.
int ab_launch_solve_alpha(ab_gp* h, const double* y) {
    const int T = (int)(h->npad / NB);
    const int64_t ld = h->npad;
    cudaStream_t s = h->stream;
    residual_kernel<<<(unsigned)((h->npad + 255) / 256), 256, 0, s>>>(y, h->n, h->npad, h->mean, h->work);
    if (T >= 2) {
        int rc = ab_launch_trsv_dataflow(h, h->work, 1);          // both sweeps, one cooperative launch
        if (rc) return rc;
    } else {
        for (int k = 0; k < T; k++) trsv_fwd_kernel<<<T - k, 256, 0, s>>>(h->L, ld, h->Dinv, k, h->work, h->z);
        AB_CUDA(cudaMemcpyAsync(h->work, h->z, h->npad * sizeof(double), cudaMemcpyDeviceToDevice, s));
        for (int k = T - 1; k >= 0; k--) trsv_bwd_kernel<<<k + 1, NB, 0, s>>>(h->L, ld, h->Dinv, k, h->work, h->alpha);
    }
    final_sums_kernel<<<1, 1024, 0, s>>>(h->z, h->npad, h->logdet_parts, T, h->scratch);
    AB_CHECK_LAUNCH();
    AB_CUDA(cudaMemcpyAsync(h->h_pinned, h->scratch, 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
    return 0;
}

int ab_launch_build_linv(ab_gp* h) {
    int rc = configure_once();
    if (rc) return rc;
    const int T = (int)(h->npad / NB);
    const int64_t ld = h->npad;
    cudaStream_t s = h->stream;
    copy_diag_blocks_kernel<<<T, 256, 0, s>>>(h->Dinv, h->Linv, ld);
    std::vector<std::vector<InvNode>> levels;
    inv_tree(0, T, levels);
    for (size_t ht = 1; ht < levels.size(); ht++) {
        auto& nodes = levels[ht];
        for (size_t b = 0; b < nodes.size(); b += 64) {
            InvLevel lv;
            lv.nnodes = (int)((nodes.size() - b < 64) ? nodes.size() - b : 64);
            int tiles = 0;
            for (int q = 0; q < lv.nnodes; q++) {
                lv.nodes[q] = nodes[b + q];
                lv.nodes[q].tile_begin = tiles;
                tiles += lv.nodes[q].h * lv.nodes[q].n2;
            }
            trinv_kernel<1><<<tiles, abg::THREADS, abg::SMEM_BYTES, s>>>(h->L, h->Linv, h->Kinv, ld, lv);
            trinv_kernel<2><<<tiles, abg::THREADS, abg::SMEM_BYTES, s>>>(h->L, h->Linv, h->Kinv, ld, lv);
        }
    }
    AB_CHECK_LAUNCH();
    return 0;
}

int ab_launch_build_kinv(ab_gp* h) {
    int rc = configure_once();
    if (rc) return rc;
    const int T = (int)(h->npad / NB);
    kinv_kernel<<<T * (T + 1) / 2, abg::THREADS, abg::SMEM_BYTES, h->stream>>>(h->Linv, h->Kinv, h->npad, T);
    AB_CHECK_LAUNCH();
    return 0;
}

int ab_launch_mirror_lower(ab_gp* h, double* A, int64_t ld) { return ab_launch_mirror_lower_n(h, A, ld, h->npad); }

// strict lower triangle of the leading n x n block of A -> upper
int ab_launch_mirror_lower_n(ab_gp* h, double* A, int64_t ld, int64_t n) {
    unsigned nt = (unsigned)((n + 31) / 32);
    mirror_lower_kernel<<<dim3(nt, nt), dim3(32, 8), 0, h->stream>>>(A, ld, n);
    mirror_diag_tiles_kernel<<<nt, 256, 0, h->stream>>>(A, ld, n);
    AB_CHECK_LAUNCH();
    return 0;
}
