// k-fold cross-validation of hyper-parameter candidates as ONE batched device job (SURVEY 8f-1).
//
// The reference's default hyper-parameter search (`hyperopt_method="cv"`, alabi/core.py:751 ->
// gp_utils.optimize_gp_kfold_cv, alabi/gp_utils.py:511-1231) scores 100 + 50 + 25 candidates on 5
// folds each: 875 independent jobs "factorise K(theta_c) on the fold's training rows, check the
// log-likelihood, predict the mean at the held-out rows" (worker: gp_utils.py:511-637), run one
// after another (or over a multiprocessing pool).  Here a whole stage is four launches:
//
//   cvb_gather_kernel   per job: training / validation rows gathered from X, scaled by the
//                       candidate's metric; residuals y - mean
//   cvb_cov_kernel      per job and lower tile: K = amp k(r^2) + (yerr^2 + e^wn) I, identity padding
//   chol_dataflow_kernel (batched form, chol_dataflow.cu): the tiles of ALL matrices in one
//                       dependency-ordered task list, so the waits of one small factorisation are
//                       filled with the tiles of the others
//   cvb_solve_predict_kernel  per job (one CTA): z = L^-1 r, alpha = L^-T z by blocks with the
//                       diagonal-block inverses, log-likelihood, predictive mean at the held-out rows
//
// Jobs are processed in chunks sized to a workspace budget.  Results per job: predictions, the
// log-likelihood and the Cholesky status (first non-positive pivot, 0 = ok).
#include <cmath>
#include <vector>
#include "handle.h"
#include "alabi_b200.h"

int ab_launch_factor_dataflow_batch(ab_gp* h, double* d_A, int64_t strideA, int T, int nmat, double* d_Dinv,
                                    double* d_logdet_parts, int* d_info, int* d_ctrl, const int2* d_tasks);
void ab_build_batch_tasks(int T, int nmat, std::vector<int2>& tasks);

namespace {

constexpr int NB = AB_NB;

struct CandParams {
    double amp, diag_add, mean;
    double inv_len[AB_MAX_DIM];
    double alpha, inv2a;          // rational quadratic kernel only (0 for kinds 0-2)
};

struct CvArgs {
    const double* X; const double* y; int d;
    const CandParams* cand; const int* job_cand;
    const int* ntrain; const int* nval;
    const int* train_idx; int ld_train; const int* val_idx; int ld_val;
    int npad, T;
    double* Xs;       // [job][npad][d] scaled training rows (padding rows 0)
    double* Xv;       // [job][ld_val][d] scaled validation rows
    double* r;        // [job][npad] y - mean (padding 0); overwritten by z, then alpha
    double* A;        // [job][npad][npad]
    double* Dinv;     // [job][T][128][128]
    double* logdet;   // [job][T]
    int* info;        // [job]
    double* pred;     // [job][ld_val]
    double* loglik;   // [job]
    int job0;         // first job of this chunk (indices into the per-job arrays)
};

__global__ void __launch_bounds__(256)
cvb_gather_kernel(const CvArgs a) {
    const int jl = blockIdx.y, job = a.job0 + jl, d = a.d;
    const CandParams& c = a.cand[a.job_cand[job]];
    const int nt = a.ntrain[job], nv = a.nval[job];
    for (int idx = blockIdx.x * 256 + threadIdx.x; idx < a.npad * d; idx += gridDim.x * 256) {
        const int row = idx / d, k = idx - row * d;
        double v = 0.0;
        if (row < nt) v = a.X[(int64_t)a.train_idx[(int64_t)job * a.ld_train + row] * d + k] * c.inv_len[k];
        a.Xs[((int64_t)jl * a.npad) * d + idx] = v;
    }
    for (int row = blockIdx.x * 256 + threadIdx.x; row < a.npad; row += gridDim.x * 256)
        a.r[(int64_t)jl * a.npad + row] = (row < nt) ? a.y[a.train_idx[(int64_t)job * a.ld_train + row]] - c.mean : 0.0;
    for (int idx = blockIdx.x * 256 + threadIdx.x; idx < nv * d; idx += gridDim.x * 256) {
        const int row = idx / d, k = idx - row * d;
        a.Xv[((int64_t)jl * a.ld_val) * d + idx] = a.X[(int64_t)a.val_idx[(int64_t)job * a.ld_val + row] * d + k] * c.inv_len[k];
    }
}

// one 128 x 128 lower tile (ti >= tj) of one job's covariance matrix; 256 threads, thread = (row
// pair, 16-column strip) with the column points staged in shared memory
template <int KIND>
__global__ void __launch_bounds__(256)
cvb_cov_kernel(const CvArgs a) {
    extern __shared__ __align__(16) double cov_sm[];          // 2 x 128 x (d + 1) doubles
    const int jl = blockIdx.y, job = a.job0 + jl, d = a.d, tid = threadIdx.x;
    double* const sR = cov_sm;
    double* const sCo = cov_sm + NB * (d + 1);
    int ti, tj;
    {   // linear tile index -> (ti, tj), tj <= ti
        int p = blockIdx.x, r = 0;
        while ((r + 1) * (r + 2) / 2 <= p) r++;
        ti = r; tj = p - r * (r + 1) / 2;
    }
    const CandParams& c = a.cand[a.job_cand[job]];
    const int nt = a.ntrain[job];
    const double* Xs = a.Xs + (int64_t)jl * a.npad * d;
    const int pitch = d + 1;
    for (int idx = tid; idx < NB * d; idx += 256) {
        const int row = idx / d, k = idx - row * d;
        sR[row * pitch + k] = Xs[(int64_t)(ti * NB + row) * d + k];
        sCo[row * pitch + k] = Xs[(int64_t)(tj * NB + row) * d + k];
    }
    __syncthreads();
    double* A = a.A + (int64_t)jl * a.npad * a.npad;
    const int cx = tid & 15, ry = tid >> 4;               // 16 x 16 threads, 8 x 8 elements each
    for (int rr = 0; rr < 8; rr++) {
        const int lr = ry + 16 * rr, gi = ti * NB + lr;
        for (int cc = 0; cc < 8; cc++) {
            const int lc = cx + 16 * cc, gj = tj * NB + lc;
            double v;
            if (gi < nt && gj < nt) {
                double r2 = 0.0;
                for (int k = 0; k < d; k++) {
                    const double df = sR[lr * pitch + k] - sCo[lc * pitch + k];
                    r2 = fma(df, df, r2);
                }
                v = c.amp * ab_radial<KIND>(r2, c.alpha, c.inv2a) + ((gi == gj) ? c.diag_add : 0.0);
            } else {
                v = (gi == gj) ? 1.0 : 0.0;                  // identity padding
            }
            A[(int64_t)gi * a.npad + gj] = v;
        }
    }
}

// one CTA per job: both triangular solves by 128-blocks, log-likelihood, mean at the held-out rows
template <int KIND>
__global__ void __launch_bounds__(256)
cvb_solve_predict_kernel(const CvArgs a) {
    __shared__ double sv[NB], ss[NB], red[256];
    const int jl = blockIdx.x, job = a.job0 + jl, tid = threadIdx.x, d = a.d;
    const int npad = a.npad, T = a.T;
    const CandParams& c = a.cand[a.job_cand[job]];
    const int nt = a.ntrain[job], nv = a.nval[job];
    const double* L = a.A + (int64_t)jl * npad * npad;
    const double* Dinv = a.Dinv + (int64_t)jl * T * NB * NB;
    double* x = a.r + (int64_t)jl * npad;                   // r -> z -> alpha in place
    if (a.info[jl] != 0) {                                   // not positive definite: the job failed
        if (tid == 0) a.loglik[job] = -INFINITY;
        for (int v = tid; v < nv; v += 256) a.pred[(int64_t)job * a.ld_val + v] = NAN;
        return;
    }
    const int row = tid & 127, half = tid >> 7;              // two threads per row split the columns
    // ---- forward: z_k = D_k^-1 (r_k - sum_{j<k} L_kj z_j) --------------------------------
    for (int k = 0; k < T; k++) {
        double s = 0.0;
        const double* Lrow = L + (int64_t)(k * NB + row) * npad;
        for (int col = half; col < k * NB; col += 2) s = fma(Lrow[col], x[col], s);
        red[tid] = s;
        __syncthreads();
        if (tid < NB) ss[tid] = x[k * NB + tid] - (red[tid] + red[tid + 128]);
        __syncthreads();
        if (tid < NB) {
            const double* Dr = Dinv + ((int64_t)k * NB + tid) * NB;
            double zz = 0.0;
            for (int q = 0; q <= tid; q++) zz = fma(Dr[q], ss[q], zz);
            sv[tid] = zz;
        }
        __syncthreads();
        if (tid < NB) x[k * NB + tid] = sv[tid];
        __syncthreads();
    }
    // ---- quadratic form and log-determinant --------------------------------------------------
    double q = 0.0;
    for (int i = tid; i < npad; i += 256) q = fma(x[i], x[i], q);
    red[tid] = q;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) red[tid] += red[tid + o];
        __syncthreads();
    }
    if (tid == 0) {
        double ld = 0.0;
        for (int k = 0; k < T; k++) ld += a.logdet[(int64_t)jl * T + k];
        a.loglik[job] = -0.5 * red[0] - 0.5 * ld - 0.5 * (double)nt * 1.8378770664093453;
    }
    __syncthreads();
    // ---- backward: alpha_k = D_k^-T (z_k - sum_{j>k} L_jk^T alpha_j) ---------------------------
    for (int k = T - 1; k >= 0; k--) {
        double s = 0.0;                                      // thread (col = row, half): rows split in two
        for (int rr = (k + 1) * NB + half; rr < npad; rr += 2) s = fma(L[(int64_t)rr * npad + k * NB + row], x[rr], s);
        red[tid] = s;
        __syncthreads();
        if (tid < NB) ss[tid] = x[k * NB + tid] - (red[tid] + red[tid + 128]);
        __syncthreads();
        if (tid < NB) {
            double al = 0.0;
            for (int rr = tid; rr < NB; rr++) al = fma(Dinv[((int64_t)k * NB + rr) * NB + tid], ss[rr], al);
            sv[tid] = al;
        }
        __syncthreads();
        if (tid < NB) x[k * NB + tid] = sv[tid];
        __syncthreads();
    }
    // ---- predictive mean at the held-out rows --------------------------------------------------
    const double* Xs = a.Xs + (int64_t)jl * npad * d;
    const double* Xv = a.Xv + (int64_t)jl * a.ld_val * d;
    for (int v = tid; v < nv; v += 256) {
        double xv[AB_MAX_DIM];
        for (int k = 0; k < d; k++) xv[k] = Xv[(int64_t)v * d + k];
        double m = 0.0;
        for (int j = 0; j < nt; j++) {
            double r2 = 0.0;
            for (int k = 0; k < d; k++) {
                const double df = xv[k] - Xs[(int64_t)j * d + k];
                r2 = fma(df, df, r2);
            }
            m = fma(ab_radial<KIND>(r2, c.alpha, c.inv2a), x[j], m);
        }
        a.pred[(int64_t)job * a.ld_val + v] = fma(c.amp, m, c.mean);
    }
}

// bytes of workspace one job needs (matrix, diagonal-block inverses, scaled inputs, vectors, control words)
size_t job_bytes(int npad, int d, int ld_val) {
    const int T = npad / NB;
    size_t b = ((size_t)npad * npad + (size_t)npad * NB + (size_t)npad * d + (size_t)ld_val * d + (size_t)npad + T) * sizeof(double);
    b += (size_t)(T * (T + 1) / 2) * sizeof(int2) + (size_t)(T + 2) * sizeof(int) + 64;
    return (b + 255) / 256 * 256;
}

}  // namespace

extern "C" int ab_gp_cv_batch(ab_gp* h, const double* d_X, const double* d_y, int64_t n, int d, int kernel_id, int ncand,
                              const double* h_params, int njobs, const int* h_job_cand, const int* h_ntrain,
                              const int* h_nval, const int* d_train_idx, int ld_train, const int* d_val_idx, int ld_val,
                              double* d_pred, double* h_loglik, int* h_status, void* d_work, size_t work_bytes) {
    if (!h || !d_X || !d_y || !h_params || !h_job_cand || !h_ntrain || !h_nval || !d_train_idx || !d_val_idx || !d_pred ||
        !h_loglik || !h_status) { ab_set_error("ab_gp_cv_batch: null argument"); return -1; }
    if (n < 2 || d < 1 || d > AB_MAX_DIM || kernel_id < 0 || kernel_id > AB_KERNEL_RATQUAD || ncand < 1 || njobs < 1 || ld_train < 1 || ld_val < 1) {
        ab_set_error("ab_gp_cv_batch: bad argument"); return -1;
    }
    AB_CUDA(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    int nt_max = 0;
    for (int j = 0; j < njobs; j++) {
        if (h_ntrain[j] < 1 || h_ntrain[j] > ld_train || h_nval[j] < 0 || h_nval[j] > ld_val || h_job_cand[j] < 0 ||
            h_job_cand[j] >= ncand) { ab_set_error("ab_gp_cv_batch: bad job %d", j); return -1; }
        if (h_ntrain[j] > nt_max) nt_max = h_ntrain[j];
    }
    const int npad = (nt_max + NB - 1) / NB * NB, T = npad / NB;
    // candidates: [mean, white_noise, amp, log_M...], [mean, white_noise, amp, log_alpha, log_M...] (RQ)
    const int nx = (kernel_id == AB_KERNEL_RATQUAD) ? 1 : 0;
    std::vector<CandParams> cp(ncand);
    for (int c = 0; c < ncand; c++) {
        const double* p = h_params + (size_t)c * (3 + nx + d);
        cp[c].mean = p[0];
        cp[c].diag_add = exp(p[1]);
        cp[c].amp = p[2];
        for (int k = 0; k < AB_MAX_DIM; k++) cp[c].inv_len[k] = (k < d) ? exp(-0.5 * p[3 + nx + k]) : 0.0;
        cp[c].alpha = nx ? exp(p[3]) : 0.0;
        cp[c].inv2a = nx ? 0.5 / cp[c].alpha : 0.0;
        if (nx && !(std::isfinite(cp[c].alpha) && cp[c].alpha > 0.0 && std::isfinite(cp[c].inv2a))) {
            ab_set_error("ab_gp_cv_batch: candidate %d: alpha = exp(%g) is not finite and positive", c, p[3]);
            return -1;
        }
    }
    // the caller's workspace decides how many jobs are factorised per launch
    const size_t fixed = sizeof(CandParams) * ncand + (size_t)njobs * (3 * sizeof(int) + sizeof(double)) + 4096;
    const size_t per_job = job_bytes(npad, d, ld_val);
    if (!d_work || work_bytes < fixed + per_job) {
        ab_set_error("ab_gp_cv_batch: workspace too small (%zu bytes; one job needs %zu + %zu)", work_bytes, per_job, fixed);
        return -3;
    }
    int chunk = (int)((work_bytes - fixed) / per_job);
    if (chunk > njobs) chunk = njobs;
    const int ntiles = T * (T + 1) / 2;
    Carver cv{static_cast<char*>(d_work), work_bytes};
    void* bCand = cv.take(sizeof(CandParams) * ncand);
    int* bJc = static_cast<int*>(cv.take(sizeof(int) * njobs));
    int* bNt = static_cast<int*>(cv.take(sizeof(int) * njobs));
    int* bNv = static_cast<int*>(cv.take(sizeof(int) * njobs));
    double* bLl = static_cast<double*>(cv.take(sizeof(double) * njobs));
    double* bA = static_cast<double*>(cv.take(sizeof(double) * chunk * npad * npad));
    double* bD = static_cast<double*>(cv.take(sizeof(double) * chunk * npad * NB));
    double* bXs = static_cast<double*>(cv.take(sizeof(double) * chunk * npad * d));
    double* bXv = static_cast<double*>(cv.take(sizeof(double) * chunk * ld_val * d));
    double* bR = static_cast<double*>(cv.take(sizeof(double) * chunk * npad));
    double* bLd = static_cast<double*>(cv.take(sizeof(double) * chunk * T));
    int* bInfo = static_cast<int*>(cv.take(sizeof(int) * chunk));
    int* bCtrl = static_cast<int*>(cv.take(sizeof(int) * (2 + (size_t)chunk * T)));
    int2* bTasks = static_cast<int2*>(cv.take(sizeof(int2) * (size_t)chunk * ntiles));
    if (!bCand || !bJc || !bNt || !bNv || !bLl || !bA || !bD || !bXs || !bXv || !bR || !bLd || !bInfo || !bCtrl || !bTasks) {
        ab_set_error("ab_gp_cv_batch: workspace layout does not fit (%zu bytes)", work_bytes);
        return -3;
    }
    int rc = 0;
    AB_CUDA(cudaMemcpyAsync(bCand, cp.data(), sizeof(CandParams) * ncand, cudaMemcpyHostToDevice, s));
    AB_CUDA(cudaMemcpyAsync(bJc, h_job_cand, sizeof(int) * njobs, cudaMemcpyHostToDevice, s));
    AB_CUDA(cudaMemcpyAsync(bNt, h_ntrain, sizeof(int) * njobs, cudaMemcpyHostToDevice, s));
    AB_CUDA(cudaMemcpyAsync(bNv, h_nval, sizeof(int) * njobs, cudaMemcpyHostToDevice, s));
    std::vector<int2> tasks;
    int tasks_for = -1;
    std::vector<int> info_h(njobs, 0), abort_h(1, 0);
    CvArgs a{};
    a.X = d_X; a.y = d_y; a.d = d;
    a.cand = static_cast<const CandParams*>(bCand); a.job_cand = bJc;
    a.ntrain = bNt; a.nval = bNv;
    a.train_idx = d_train_idx; a.ld_train = ld_train; a.val_idx = d_val_idx; a.ld_val = ld_val;
    a.npad = npad; a.T = T;
    a.Xs = bXs; a.Xv = bXv; a.r = bR; a.A = bA; a.Dinv = bD; a.logdet = bLd;
    a.info = bInfo; a.pred = d_pred; a.loglik = bLl;
    for (int j0 = 0; j0 < njobs; j0 += chunk) {
        const int nj = (njobs - j0 < chunk) ? (njobs - j0) : chunk;
        a.job0 = j0;
        if (tasks_for != nj) {
            AB_CUDA(cudaStreamSynchronize(s));              // the previous chunk may still read the list
            ab_build_batch_tasks(T, nj, tasks);
            AB_CUDA(cudaMemcpyAsync(bTasks, tasks.data(), sizeof(int2) * tasks.size(), cudaMemcpyHostToDevice, s));
            AB_CUDA(cudaStreamSynchronize(s));              // `tasks` may be rebuilt for a smaller last chunk
            tasks_for = nj;
        }
        int gx = (npad * d + 255) / 256;
        if (gx > 64) gx = 64;
        cvb_gather_kernel<<<dim3(gx, nj), 256, 0, s>>>(a);
        const int cov_smem = 2 * NB * (d + 1) * (int)sizeof(double);
        AB_DISPATCH_KIND(kernel_id, {
            AB_CUDA(cudaFuncSetAttribute(cvb_cov_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, cov_smem));
            cvb_cov_kernel<KIND><<<dim3(ntiles, nj), 256, cov_smem, s>>>(a);
        });
        AB_CHECK_LAUNCH();
        rc = ab_launch_factor_dataflow_batch(h, a.A, (int64_t)npad * npad, T, nj, a.Dinv, a.logdet, a.info, bCtrl, bTasks);
        if (rc) return rc;
        AB_DISPATCH_KIND(kernel_id, (cvb_solve_predict_kernel<KIND><<<nj, 256, 0, s>>>(a)));
        AB_CHECK_LAUNCH();
        ab_count_launches(3);
        AB_CUDA(cudaMemcpyAsync(info_h.data() + j0, a.info, sizeof(int) * nj, cudaMemcpyDeviceToHost, s));
        AB_CUDA(cudaMemcpyAsync(abort_h.data(), bCtrl + 1, sizeof(int), cudaMemcpyDeviceToHost, s));
        AB_CUDA(cudaStreamSynchronize(s));
        if (abort_h[0] != 0) { ab_set_error("batched Cholesky watchdog fired (dependency wait exceeded its limit)"); return -5; }
    }
    AB_CUDA(cudaMemcpyAsync(h_loglik, bLl, sizeof(double) * njobs, cudaMemcpyDeviceToHost, s));
    AB_CUDA(cudaStreamSynchronize(s));
    for (int j = 0; j < njobs; j++) h_status[j] = info_h[j];
    return 0;
}

// workspace (bytes) that lets ab_gp_cv_batch factorise `njobs` jobs of at most `ntrain_max` training
// rows in one launch; any size from one job's worth upwards works (more launches)
extern "C" size_t ab_gp_cv_workspace_bytes(int ntrain_max, int d, int ld_val, int ncand, int njobs) {
    const int npad = (ntrain_max + NB - 1) / NB * NB;
    return sizeof(CandParams) * (size_t)ncand + (size_t)njobs * (3 * sizeof(int) + sizeof(double)) + 8192 +
           (size_t)njobs * job_bytes(npad, d, ld_val) + 16 * 256;
}
