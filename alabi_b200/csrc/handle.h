// Opaque GP handle behind the C ABI (include/alabi_b200.h).  One handle is bound
// to one device and one stream; it owns the factor / inverse workspaces.
#pragma once
#include <vector>
#include "common.cuh"

enum { AB_PROF_COV = 0, AB_PROF_FACTOR = 1, AB_PROF_PREDICT_PANEL = 2, AB_PROF_PREDICT_VAR = 3,
       AB_PROF_ENSEMBLE = 4, AB_PROF_FAMILIES = 5 };

struct ab_gp {
    int device = 0;
    int nsm = 148;                        // SM count of the device
    cudaStream_t stream = nullptr;        // caller's stream (borrowed)
    cudaStream_t copy_stream = nullptr;   // device-to-host copies that overlap the next kernels on `stream` (owned)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;

    int64_t n = 0, npad = 0;              // training points, padded to AB_NB
    int d = 0;
    KernParams kp{};                      // kernel id, amplitude, metric, diagonal term
    double mean = 0.0, white_noise = -12.0, yerr2 = 0.0;
    double log_M[AB_MAX_DIM] = {0};

    double* X = nullptr;                  // n x d   training inputs (as given)
    double* Xs = nullptr;                 // npad x d inputs scaled by exp(-0.5 log_M) (pad rows = 0)
    double* XsT = nullptr;                // d x npad transpose of Xs (coalesced per-dimension reads)
    double* L = nullptr;                  // npad x npad lower Cholesky factor (row-major)
    double* Dinv = nullptr;               // (npad/NB) x NB x NB inverses of the diagonal blocks of L
    double* Linv = nullptr;               // npad x npad L^-1 (lower; lazily built)
    double* Kinv = nullptr;               // npad x npad K^-1 (lower tiles + full diagonal tiles; lazy)
    double* alpha = nullptr;              // npad  K^-1 (y - mean)
    double* z = nullptr;                  // npad  L^-1 (y - mean)
    double* work = nullptr;               // npad scratch
    double* logdet_parts = nullptr;       // npad/NB partial log-determinants
    double* scratch = nullptr;            // generic scratch (predict panels, partial sums)
    size_t scratch_bytes = 0;
    double* io = nullptr;                 // staging for the host-buffer entry points
    size_t io_bytes = 0;
    int64_t cap_pad = 0;                  // allocated capacity (padded points) of the O(n^2) buffers
    int cap_d = 0;
    int64_t inv_cap_pad = 0;              // capacity of Linv / Kinv
    bool have_inputs = false, have_kernel = false, scaled = false;
    int* d_info = nullptr;                // first non-positive pivot (1-based), 0 = SPD
    double* h_pinned = nullptr;           // small pinned host staging buffer (>= 4 KB)

    // optional per-kernel-family device timing (bench.py roofline): event pairs
    // recorded on h->stream around the launches of one family
    bool profiling = false;
    std::vector<cudaEvent_t> prof_ev[AB_PROF_FAMILIES];

    bool few_path = true;                 // m <= 8 queries: the spread-one-query kernels of predict.cu (false: batched kernels)
    void* df_tasks = nullptr;             // dataflow task list (device) for df_tasks_T block rows
    int df_tasks_T = 0;
    void* cov_items = nullptr;            // work list of cov_strip_kernel for cov_items_nt tile rows
    int cov_items_nt = 0, cov_items_seg = 0, cov_items_count = 0;
    bool factored = false, have_linv = false, have_kinv = false, have_alpha = false;
    int info = 0;
    double logdet = 0.0, quad = 0.0;
    // ab_ensemble_launch -> ab_ensemble_finish
    bool ens_pending = false;
};

int ab_ensure_scratch(ab_gp* h, size_t bytes);
// carve `bytes` (256-aligned) out of a workspace; nullptr when it does not fit
struct Carver {
    char* p; size_t left;
    void* take(size_t bytes) {
        bytes = (bytes + 255) / 256 * 256;
        if (bytes > left) return nullptr;
        void* r = p; p += bytes; left -= bytes;
        return r;
    }
};
void ab_count_launches(long long n);
// RAII-less scope helpers: record an event before / after a kernel family
void ab_prof_begin(ab_gp* h, int family);
void ab_prof_end(ab_gp* h, int family);

// cov.cu
int ab_launch_cov(ab_gp* h, double* K, int64_t ld, int mirror, int pad_identity);
int ab_launch_scale_inputs(ab_gp* h);
int ab_launch_scale_points(ab_gp* h, const double* X, int64_t m, double* XT, int64_t ldm);
int ab_launch_cross_cov(ab_gp* h, const double* AT, int64_t lda, int64_t na, const double* BT, int64_t ldb,
                        int64_t nb, double* K, int64_t ld);
int ab_launch_factor_dataflow(ab_gp* h);   // chol_dataflow.cu
// chol.cu
int ab_launch_trsv_dataflow(ab_gp* h, const double* r, int backward);   // trsv_dataflow.cu
int ab_launch_trsv_single(ab_gp* h, const double* r);      // chol.cu: z = D_0^-1 r for a one-block factor
int ab_launch_rebuild_dinv_block(ab_gp* h, int kb);        // chol.cu
int ab_launch_rebuild_dinv(ab_gp* h);
int ab_launch_solve_alpha(ab_gp* h, const double* y);
int ab_launch_build_linv(ab_gp* h);
int ab_launch_build_kinv(ab_gp* h);
int ab_launch_mirror_lower(ab_gp* h, double* A, int64_t ld);
int ab_launch_mirror_lower_n(ab_gp* h, double* A, int64_t ld, int64_t n);
// grad.cu
int ab_launch_grad(ab_gp* h);
// predict.cu
int ab_launch_predict(ab_gp* h, const double* Xq, int64_t m, double* mu, double* var);
int64_t ab_predict_panel_queries(ab_gp* h);
int ab_launch_predict_cov(ab_gp* h, const double* Xq, int64_t m, double* mu, double* C, int64_t ldc);
int ab_launch_tri_gemm_lower(ab_gp* h, const double* L, int64_t ld, int T, const double* B, int64_t ldb, int ntiles,
                             double* C);
int ab_launch_predict_grad(ab_gp* h, const double* Xq, int64_t m, double* mu, double* var, double* dmu, double* dvar);
int ab_launch_utility(ab_gp* h, int kind, const double* Xq, const double* mu, const double* var, int64_t m,
                      const double* h_bounds, double y_best, double zeta, double* util,
                      int64_t* h_argmin, double* h_min);
