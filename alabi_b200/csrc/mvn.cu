// Draws from a multivariate normal N(mean, Sigma + jitter I) on the device: george's
// GP.sample_conditional / GP.sample (george/gp.py), which draw through NumPy's
// multivariate_normal (an SVD of Sigma on the host).
//
//   mvn_pad_kernel       lower tiles of Sigma + jitter I into an mpad x mpad workspace, identity
//                        padding (the layout of cv_batch.cu's cvb_cov_kernel); Sigma is not modified
//   chol_dataflow_kernel (batched form with one matrix, chol_dataflow.cu): L_Sigma, or the first
//                        non-positive pivot
//   mvn_normals_kernel   Z[i][s] ~ N(0, 1): Philox4x32-10, key = seed, counter = (i, s / 2, 0,
//                        AB_STREAM_MVN), Box-Muller as in nested.cu
//   tri_gemm_kernel<false>  Y = L_Sigma Z (FP64 DMMA; column s of Y depends on column s of Z only,
//                        so the first k draws of any batch are the k draws of a smaller one)
//   mvn_finish_kernel    out[s][q] = mean[q] + Y[q][s]
#include <cmath>
#include <vector>
#include "handle.h"
#include "alabi_b200.h"
#include "philox.cuh"

int ab_launch_factor_dataflow_batch(ab_gp* h, double* d_A, int64_t strideA, int T, int nmat, double* d_Dinv,
                                    double* d_logdet_parts, int* d_info, int* d_ctrl, const int2* d_tasks);
void ab_build_batch_tasks(int T, int nmat, std::vector<int2>& tasks);

namespace {

constexpr int NB = AB_NB;

// A[r][c] for the 32 x 32 block (blockIdx.y, blockIdx.x) when it lies in a lower 128-tile
__global__ void __launch_bounds__(256)
mvn_pad_kernel(const double* __restrict__ S, int64_t m, int64_t ldc, double jitter, double* __restrict__ A,
               int64_t mpad) {
    const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
    if (c0 / NB > r0 / NB) return;                      // strictly upper tile: never read by the factor
    for (int k = threadIdx.y; k < 32; k += 8) {
        const int64_t r = r0 + k, c = c0 + threadIdx.x;
        double v;
        if (r < m && c < m) v = S[r * ldc + c] + (r == c ? jitter : 0.0);
        else v = (r == c) ? 1.0 : 0.0;
        A[r * mpad + c] = v;
    }
}

// one thread per (row i, sample pair p); rows >= m and samples >= ns are zero
__global__ void __launch_bounds__(256)
mvn_normals_kernel(int64_t m, int64_t mpad, int64_t ns, int64_t lds, unsigned seed_lo, unsigned seed_hi,
                   double* __restrict__ Z) {
    const int64_t npair = lds / 2;
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= mpad * npair) return;
    const int64_t i = idx / npair, p = idx - i * npair;
    double z0 = 0.0, z1 = 0.0;
    if (i < m && 2 * p < ns) {
        const abr::U4 r = abr::philox((unsigned)i, (unsigned)p, 0u, (unsigned)AB_STREAM_MVN, seed_lo, seed_hi);
        const double u1 = 1.0 - abr::u53(r.x, r.y), u2 = abr::u53(r.z, r.w);     // u1 in (0, 1]
        const double rad = sqrt(-2.0 * log(u1));
        double sn, cs;
        sincospi(2.0 * u2, &sn, &cs);
        z0 = rad * cs;
        z1 = (2 * p + 1 < ns) ? rad * sn : 0.0;
    }
    *reinterpret_cast<double2*>(Z + i * lds + 2 * p) = make_double2(z0, z1);
}

// out[s][q] = mean[q] + Y[q][s] through a 32 x 32 transpose in shared memory
__global__ void __launch_bounds__(256)
mvn_finish_kernel(const double* __restrict__ Y, int64_t lds, int64_t m, int64_t ns, const double* __restrict__ mean,
                  double* __restrict__ out) {
    __shared__ double t[32][33];
    const int64_t q0 = (int64_t)blockIdx.y * 32, s0 = (int64_t)blockIdx.x * 32;
    for (int k = threadIdx.y; k < 32; k += 8) {
        const int64_t q = q0 + k, s = s0 + threadIdx.x;
        t[k][threadIdx.x] = (q < m && s < ns) ? Y[q * lds + s] : 0.0;
    }
    __syncthreads();
    for (int k = threadIdx.y; k < 32; k += 8) {
        const int64_t s = s0 + k, q = q0 + threadIdx.x;
        if (q < m && s < ns) out[s * m + q] = mean ? mean[q] + t[threadIdx.x][k] : t[threadIdx.x][k];
    }
}

}  // namespace

extern "C" int ab_mvn_sample(ab_gp* h, const double* d_cov, int64_t m, int64_t ldc, const double* d_mean, double jitter,
                             int64_t nsamples, uint64_t seed, double* d_out, int* h_info) {
    if (!h || !d_cov || !d_out || !h_info) { ab_set_error("ab_mvn_sample: null argument"); return -1; }
    if (m < 1 || ldc < m || nsamples < 1) {
        ab_set_error("ab_mvn_sample: need m >= 1, ldc >= m and nsamples >= 1 (m=%lld ldc=%lld nsamples=%lld)",
                     (long long)m, (long long)ldc, (long long)nsamples);
        return -1;
    }
    if (!(std::isfinite(jitter) && jitter >= 0.0)) { ab_set_error("ab_mvn_sample: jitter %g is not finite and >= 0", jitter); return -1; }
    const int64_t mpad = (m + NB - 1) / NB * NB;
    const int T = (int)(mpad / NB);
    if (T > 4095) { ab_set_error("ab_mvn_sample: m = %lld is too large", (long long)m); return -1; }
    *h_info = 0;
    AB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int64_t lds = (nsamples + NB - 1) / NB * NB;            // whole 128-column tiles of the product
    const int ntasks = T * (T + 1) / 2;
    const size_t need = ((size_t)mpad * mpad + (size_t)mpad * NB + (size_t)T + 2 * (size_t)mpad * lds) * sizeof(double) +
                        (size_t)ntasks * sizeof(int2) + (size_t)(T + 3) * sizeof(int) + 8 * 256;
    int rc = ab_ensure_scratch(h, need);
    if (rc) {
        cudaGetLastError();                    // a failed allocation is reported once, by the return code
        return rc;
    }
    Carver cv{reinterpret_cast<char*>(h->scratch), h->scratch_bytes};
    double* A = static_cast<double*>(cv.take((size_t)mpad * mpad * sizeof(double)));
    double* Dinv = static_cast<double*>(cv.take((size_t)mpad * NB * sizeof(double)));
    double* logdet = static_cast<double*>(cv.take((size_t)T * sizeof(double)));
    double* Z = static_cast<double*>(cv.take((size_t)mpad * lds * sizeof(double)));
    double* Y = static_cast<double*>(cv.take((size_t)mpad * lds * sizeof(double)));
    int2* tasks = static_cast<int2*>(cv.take((size_t)ntasks * sizeof(int2)));
    int* info = static_cast<int*>(cv.take(sizeof(int)));
    int* ctrl = static_cast<int*>(cv.take((size_t)(T + 2) * sizeof(int)));
    if (!A || !Dinv || !logdet || !Z || !Y || !tasks || !info || !ctrl) { ab_set_error("ab_mvn_sample: workspace layout"); return -1; }

    // 1. Sigma + jitter I, padded
    const unsigned nb32 = (unsigned)(mpad / 32);
    mvn_pad_kernel<<<dim3(nb32, nb32), dim3(32, 8), 0, s>>>(d_cov, m, ldc, jitter, A, mpad);
    AB_CHECK_LAUNCH();
    // 2. factor (one matrix of the batched dataflow Cholesky)
    std::vector<int2> th;
    ab_build_batch_tasks(T, 1, th);
    AB_CUDA(cudaMemcpyAsync(tasks, th.data(), th.size() * sizeof(int2), cudaMemcpyHostToDevice, s));
    rc = ab_launch_factor_dataflow_batch(h, A, 0, T, 1, Dinv, logdet, info, ctrl, tasks);
    if (rc) return rc;
    int st[2] = {0, 0};
    AB_CUDA(cudaMemcpyAsync(&st[0], info, sizeof(int), cudaMemcpyDeviceToHost, s));
    AB_CUDA(cudaMemcpyAsync(&st[1], ctrl + 1, sizeof(int), cudaMemcpyDeviceToHost, s));
    AB_CUDA(cudaStreamSynchronize(s));                            // also: `th` may go out of scope
    if (st[1] != 0) { ab_set_error("dataflow Cholesky watchdog fired (dependency wait exceeded its limit)"); return -5; }
    if (st[0] != 0) {
        *h_info = st[0];
        ab_set_error("ab_mvn_sample: covariance not positive definite: pivot %d", st[0]);
        return st[0];
    }
    // 3. standard normals
    const int64_t nthr = mpad * (lds / 2);
    mvn_normals_kernel<<<(unsigned)((nthr + 255) / 256), 256, 0, s>>>(m, mpad, nsamples, lds, (unsigned)(seed & 0xFFFFFFFFu),
                                                                      (unsigned)(seed >> 32), Z);
    AB_CHECK_LAUNCH();
    // 4. Y = L_Sigma Z
    rc = ab_launch_tri_gemm_lower(h, A, mpad, T, Z, lds, (int)(lds / NB), Y);
    if (rc) return rc;
    // 5. out = mean + Y^T
    mvn_finish_kernel<<<dim3((unsigned)((nsamples + 31) / 32), (unsigned)((m + 31) / 32)), dim3(32, 8), 0, s>>>(
        Y, lds, m, nsamples, d_mean, d_out);
    AB_CHECK_LAUNCH();
    ab_count_launches(4);
    return 0;
}
