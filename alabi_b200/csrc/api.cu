// extern "C" boundary of libalabi_b200.so (declared in include/alabi_b200.h).
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <cmath>
#include "handle.h"
#include "alabi_b200.h"

static thread_local char g_err[1024] = "";

void ab_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

#include <atomic>
static std::atomic<long long> g_launches{0};
void ab_count_launches(long long n) { g_launches += n; }

static void prof_mark(ab_gp* h, int family) {
    if (!h->profiling) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, h->stream);
    h->prof_ev[family].push_back(e);
}
void ab_prof_begin(ab_gp* h, int family) { prof_mark(h, family); }
void ab_prof_end(ab_gp* h, int family) { prof_mark(h, family); }

#define AB_REQUIRE(cond, code, ...)            \
    do {                                       \
        if (!(cond)) {                         \
            ab_set_error(__VA_ARGS__);         \
            return (code);                     \
        }                                      \
    } while (0)

int ab_ensure_scratch(ab_gp* h, size_t bytes) {
    if (bytes < 4096) bytes = 4096;
    if (h->scratch_bytes >= bytes) return 0;
    if (h->scratch) AB_CUDA(cudaFree(h->scratch));
    h->scratch = nullptr;
    h->scratch_bytes = 0;
    AB_CUDA(cudaMalloc(&h->scratch, bytes));
    h->scratch_bytes = bytes;
    return 0;
}

static int ensure_io(ab_gp* h, size_t bytes) {
    if (h->io_bytes >= bytes) return 0;
    if (h->io) AB_CUDA(cudaFree(h->io));
    h->io = nullptr;
    h->io_bytes = 0;
    AB_CUDA(cudaMalloc(&h->io, bytes));
    h->io_bytes = bytes;
    return 0;
}

template <typename T>
static int re_alloc(T** p, size_t count) {
    if (*p) AB_CUDA(cudaFree(*p));
    *p = nullptr;
    AB_CUDA(cudaMalloc(p, count * sizeof(T)));
    return 0;
}

static int ensure_inverse_buffers(ab_gp* h) {
    if (h->inv_cap_pad >= h->npad && h->Linv && h->Kinv) return 0;
    int rc = re_alloc(&h->Linv, (size_t)h->cap_pad * h->cap_pad);
    if (rc) return rc;
    rc = re_alloc(&h->Kinv, (size_t)h->cap_pad * h->cap_pad);
    if (rc) return rc;
    h->inv_cap_pad = h->cap_pad;
    return 0;
}

static int ensure_linv(ab_gp* h) {
    if (h->have_linv) return 0;
    int rc = ensure_inverse_buffers(h);
    if (rc) return rc;
    rc = ab_launch_build_linv(h);
    if (rc) return rc;
    h->have_linv = true;
    h->have_kinv = false;
    return 0;
}

static int ensure_kinv(ab_gp* h) {
    int rc = ensure_linv(h);
    if (rc) return rc;
    if (h->have_kinv) return 0;
    rc = ab_launch_build_kinv(h);
    if (rc) return rc;
    h->have_kinv = true;
    return 0;
}

static int create_resources(ab_gp* h) {
    int lo = 0, hi = 0;
    AB_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    AB_CUDA(cudaStreamCreateWithPriority(&h->copy_stream, cudaStreamNonBlocking, hi));
    AB_CUDA(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    AB_CUDA(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    AB_CUDA(cudaMalloc(&h->d_info, sizeof(int)));
    AB_CUDA(cudaMallocHost(&h->h_pinned, 8192));   // [0, 512): scalars / flags / partial sums; [512, 1024): few-query staging
    return ab_ensure_scratch(h, 1 << 20);
}

extern "C" {

int ab_version(void) { return 100; }
int ab_sizeof_ensemble_config(void) { return (int)sizeof(ab_ensemble_config); }
const char* ab_last_error(void) { return g_err; }

int ab_device_sm_count(int device) {
    int n = 0;
    AB_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device));
    return n;
}

int ab_gp_create(ab_gp** out, int device, void* cuda_stream) {
    AB_REQUIRE(out != nullptr, -1, "ab_gp_create: null out");
    int ndev = 0;
    AB_CUDA(cudaGetDeviceCount(&ndev));
    AB_REQUIRE(device >= 0 && device < ndev, -1, "ab_gp_create: device %d not available (%d devices)", device, ndev);
    AB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    AB_CUDA(cudaGetDeviceProperties(&prop, device));
    AB_REQUIRE(prop.major == 10, -4, "alabi_b200 needs an sm_100a device (B200); found sm_%d%d", prop.major, prop.minor);
    ab_gp* h = new ab_gp();
    h->device = device;
    h->nsm = prop.multiProcessorCount;
    h->stream = (cudaStream_t)cuda_stream;
    int rc = create_resources(h);
    if (rc) {                   // nothing half-built survives a failed create
        ab_gp_destroy(h);
        return rc;
    }
    *out = h;
    return 0;
}

int ab_gp_destroy(ab_gp* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    double* bufs[] = {h->X, h->Xs, h->XsT, h->L, h->Dinv, h->Linv, h->Kinv, h->alpha, h->z, h->work,
                      h->logdet_parts, h->scratch, h->io};
    for (double* b : bufs)
        if (b) cudaFree(b);
    if (h->d_info) cudaFree(h->d_info);
    if (h->df_tasks) cudaFree(h->df_tasks);
    if (h->cov_items) cudaFree(h->cov_items);
    if (h->h_pinned) cudaFreeHost(h->h_pinned);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    cudaEvent_t evs[] = {h->ev_fork, h->ev_join};
    for (cudaEvent_t e : evs)
        if (e) cudaEventDestroy(e);
    for (auto& fam : h->prof_ev)
        for (cudaEvent_t e : fam) cudaEventDestroy(e);
    delete h;
    return 0;
}

int ab_gp_set_few_query_path(ab_gp* h, int enabled) {
    AB_REQUIRE(h, -1, "null handle");
    h->few_path = enabled != 0;
    return 0;
}

int ab_gp_set_inputs(ab_gp* h, const double* d_X, int64_t n, int d) {
    AB_REQUIRE(h && d_X, -1, "ab_gp_set_inputs: null argument");
    AB_REQUIRE(n >= 1 && d >= 1 && d <= AB_MAX_DIM, -1, "ab_gp_set_inputs: need n >= 1 and 1 <= d <= %d (n=%lld d=%d)",
               AB_MAX_DIM, (long long)n, d);
    AB_CUDA(cudaSetDevice(h->device));
    int64_t npad = (n + AB_NB - 1) / AB_NB * AB_NB;
    if (npad > h->cap_pad || d > h->cap_d) {
        AB_CUDA(cudaStreamSynchronize(h->stream));
        int64_t cap = npad > h->cap_pad ? npad : h->cap_pad;
        int cd = d > h->cap_d ? d : h->cap_d;
        // the capacities describe what is allocated: zero them first, so a failure half-way
        // (buffers freed and nulled) can never be mistaken for a usable allocation later
        h->cap_pad = 0;
        h->cap_d = 0;
        h->have_inputs = h->scaled = h->factored = h->have_linv = h->have_kinv = h->have_alpha = false;
        int rc = 0;
        if (!rc) rc = re_alloc(&h->X, (size_t)cap * cd);
        if (!rc) rc = re_alloc(&h->Xs, (size_t)cap * cd);
        if (!rc) rc = re_alloc(&h->XsT, (size_t)cap * cd);
        if (!rc) rc = re_alloc(&h->L, (size_t)cap * cap);
        if (!rc) rc = re_alloc(&h->Dinv, (size_t)cap * AB_NB);
        if (!rc) rc = re_alloc(&h->alpha, (size_t)cap);
        if (!rc) rc = re_alloc(&h->z, (size_t)cap);
        if (!rc) rc = re_alloc(&h->work, (size_t)cap);
        if (!rc) rc = re_alloc(&h->logdet_parts, (size_t)cap / AB_NB);
        if (rc) return rc;
        h->cap_pad = cap;
        h->cap_d = cd;
    }
    h->n = n;
    h->npad = npad;
    h->d = d;
    AB_CUDA(cudaMemcpyAsync(h->X, d_X, (size_t)n * d * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    h->have_inputs = true;
    h->scaled = h->factored = h->have_linv = h->have_kinv = h->have_alpha = false;
    return 0;
}

static int set_kernel(ab_gp* h, int kernel_id, double amp, double alpha, const double* h_log_M, double mean,
                      double white_noise, double yerr2) {
    h->kp.kind = kernel_id;
    h->kp.d = h->d;
    h->kp.amp = amp;
    h->kp.diag_add = yerr2 + exp(white_noise);
    for (int k = 0; k < AB_MAX_DIM; k++) {
        h->log_M[k] = (k < h->d) ? h_log_M[k] : 0.0;
        h->kp.inv_len[k] = (k < h->d) ? exp(-0.5 * h_log_M[k]) : 0.0;
    }
    h->kp.alpha = alpha;
    h->kp.inv2a = (alpha > 0.0) ? 0.5 / alpha : 0.0;
    h->mean = mean;
    h->white_noise = white_noise;
    h->yerr2 = yerr2;
    h->have_kernel = true;
    h->scaled = h->factored = h->have_linv = h->have_kinv = h->have_alpha = false;
    return 0;
}

int ab_gp_set_kernel(ab_gp* h, int kernel_id, double amp, const double* h_log_M, double mean, double white_noise,
                     double yerr2) {
    AB_REQUIRE(h && h_log_M, -1, "ab_gp_set_kernel: null argument");
    AB_REQUIRE(kernel_id >= 0 && kernel_id <= 2, -1, "ab_gp_set_kernel: unknown kernel id %d", kernel_id);
    AB_REQUIRE(h->have_inputs, -2, "ab_gp_set_kernel: call ab_gp_set_inputs first");
    return set_kernel(h, kernel_id, amp, 0.0, h_log_M, mean, white_noise, yerr2);
}

int ab_gp_set_kernel_rq(ab_gp* h, double amp, double log_alpha, const double* h_log_M, double mean,
                        double white_noise, double yerr2) {
    AB_REQUIRE(h && h_log_M, -1, "ab_gp_set_kernel_rq: null argument");
    const double alpha = exp(log_alpha);
    AB_REQUIRE(std::isfinite(alpha) && alpha > 0.0 && std::isfinite(0.5 / alpha), -1,
               "ab_gp_set_kernel_rq: alpha = exp(%g) is not finite and positive (or 1 / (2 alpha) overflows)", log_alpha);
    AB_REQUIRE(h->have_inputs, -2, "ab_gp_set_kernel_rq: call ab_gp_set_inputs first");
    return set_kernel(h, AB_KERNEL_RATQUAD, amp, alpha, h_log_M, mean, white_noise, yerr2);
}

static int ensure_scaled(ab_gp* h) {
    AB_REQUIRE(h->have_inputs && h->have_kernel, -2, "inputs and kernel must be set first");
    if (h->scaled) return 0;
    int rc = ab_launch_scale_inputs(h);
    if (rc) return rc;
    h->scaled = true;
    return 0;
}

int ab_gp_build_cov(ab_gp* h, double* d_K, int with_diag) {
    AB_REQUIRE(h && d_K, -1, "ab_gp_build_cov: null argument");
    AB_CUDA(cudaSetDevice(h->device));
    int rc = ensure_scaled(h);
    if (rc) return rc;
    double keep = h->kp.diag_add;
    if (!with_diag) h->kp.diag_add = 0.0;
    rc = ab_launch_cov(h, d_K, h->n, 1, 0);
    h->kp.diag_add = keep;
    return rc;
}

int ab_gp_cross_cov(ab_gp* h, const double* d_X1, int64_t m1, const double* d_X2, int64_t m2, double* d_K) {
    AB_REQUIRE(h && d_X1 && d_X2 && d_K, -1, "ab_gp_cross_cov: null argument");
    AB_REQUIRE(h->have_kernel, -2, "ab_gp_cross_cov: kernel not set");
    AB_CUDA(cudaSetDevice(h->device));
    int rc = ab_ensure_scratch(h, (size_t)(m1 + m2) * h->d * sizeof(double));
    if (rc) return rc;
    double* AT = h->scratch;
    double* BT = h->scratch + (size_t)m1 * h->d;
    rc = ab_launch_scale_points(h, d_X1, m1, AT, m1);
    if (rc) return rc;
    rc = ab_launch_scale_points(h, d_X2, m2, BT, m2);
    if (rc) return rc;
    return ab_launch_cross_cov(h, AT, m1, m1, BT, m2, m2, d_K, m2);
}

int ab_gp_factor(ab_gp* h) {
    AB_REQUIRE(h, -1, "null handle");
    AB_CUDA(cudaSetDevice(h->device));
    int rc = ensure_scaled(h);
    if (rc) return rc;
    h->factored = h->have_linv = h->have_kinv = h->have_alpha = false;
    rc = ab_launch_cov(h, h->L, h->npad, 0, 1);
    if (rc) return rc;
    *reinterpret_cast<int*>(h->h_pinned + 9) = 0;
    rc = ab_launch_factor_dataflow(h);
    if (rc) return rc;
    AB_CUDA(cudaMemcpyAsync(h->h_pinned + 8, h->d_info, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    AB_CUDA(cudaStreamSynchronize(h->stream));
    if (*reinterpret_cast<int*>(h->h_pinned + 9) != 0) {
        ab_set_error("dataflow Cholesky watchdog fired (dependency wait exceeded its limit)");
        return -5;
    }
    h->info = *reinterpret_cast<int*>(h->h_pinned + 8);
    if (h->info != 0) {
        ab_set_error("matrix not positive definite: pivot %d", h->info);
        return h->info;
    }
    h->factored = true;
    return 0;
}

int ab_gp_set_targets(ab_gp* h, const double* d_y) {
    AB_REQUIRE(h && d_y, -1, "ab_gp_set_targets: null argument");
    AB_REQUIRE(h->factored, -2, "ab_gp_set_targets: not factorised (call ab_gp_factor)");
    AB_CUDA(cudaSetDevice(h->device));
    *reinterpret_cast<int*>(h->h_pinned + 10) = 0;
    int rc = ab_launch_solve_alpha(h, d_y);
    if (rc) return rc;
    AB_CUDA(cudaStreamSynchronize(h->stream));
    if (*reinterpret_cast<int*>(h->h_pinned + 10) != 0) {
        ab_set_error("dataflow triangular solve watchdog fired (dependency wait exceeded its limit)");
        return -5;
    }
    h->quad = h->h_pinned[0];
    h->logdet = h->h_pinned[1];
    h->have_alpha = true;
    return 0;
}

int ab_gp_log_determinant(ab_gp* h, double* h_out) {
    AB_REQUIRE(h && h_out, -1, "null argument");
    AB_REQUIRE(h->factored, -2, "not factorised");
    AB_CUDA(cudaSetDevice(h->device));
    AB_CUDA(cudaMemcpyAsync(h->h_pinned + 16, h->logdet_parts, (h->npad / AB_NB) * sizeof(double),
                            cudaMemcpyDeviceToHost, h->stream));
    AB_CUDA(cudaStreamSynchronize(h->stream));
    double s = 0.0;
    for (int64_t k = 0; k < h->npad / AB_NB; k++) s += h->h_pinned[16 + k];
    *h_out = s;
    return 0;
}

int ab_gp_log_likelihood(ab_gp* h, const double* d_y, double* h_out) {
    AB_REQUIRE(h_out, -1, "null argument");
    int rc = ab_gp_set_targets(h, d_y);
    if (rc) return rc;
    *h_out = -0.5 * h->quad - 0.5 * h->logdet - 0.5 * (double)h->n * 1.8378770664093453;   // ln(2 pi)
    return 0;
}

int ab_gp_grad_log_likelihood(ab_gp* h, const double* d_y, double* h_out) {
    AB_REQUIRE(h && h_out, -1, "null argument");
    int rc = 0;
    if (d_y) {                       // NULL: reuse the alpha of the last ab_gp_set_targets / log_likelihood
        rc = ab_gp_set_targets(h, d_y);
        if (rc) return rc;
    }
    AB_REQUIRE(h->have_alpha, -2, "ab_gp_grad_log_likelihood: targets not set");
    AB_CUDA(cudaSetDevice(h->device));
    rc = ensure_kinv(h);
    if (rc) return rc;
    rc = ab_launch_grad(h);
    if (rc) return rc;
    AB_CUDA(cudaStreamSynchronize(h->stream));
    memcpy(h_out, h->h_pinned, (h->d + 3 + (h->kp.kind == AB_KERNEL_RATQUAD ? 1 : 0)) * sizeof(double));
    return 0;
}

int ab_gp_predict(ab_gp* h, const double* d_Xq, int64_t m, double* d_mu, double* d_var) {
    AB_REQUIRE(h && d_Xq && d_mu, -1, "ab_gp_predict: null argument");
    AB_REQUIRE(h->have_alpha, -2, "ab_gp_predict: targets not set (call ab_gp_factor + ab_gp_set_targets)");
    AB_CUDA(cudaSetDevice(h->device));
    if (d_var) {
        int rc = ensure_linv(h);
        if (rc) return rc;
    }
    return ab_launch_predict(h, d_Xq, m, d_mu, d_var);
}

int ab_gp_predict_cov(ab_gp* h, const double* d_Xq, int64_t m, double* d_mu, double* d_cov, int64_t ldc) {
    AB_REQUIRE(h && d_Xq && d_mu && d_cov, -1, "ab_gp_predict_cov: null argument");
    AB_REQUIRE(m >= 0 && ldc >= m && ldc >= 1, -1, "ab_gp_predict_cov: need m >= 0 and ldc >= max(m, 1) (m=%lld ldc=%lld)",
               (long long)m, (long long)ldc);
    AB_REQUIRE(h->have_alpha, -2, "ab_gp_predict_cov: targets not set (call ab_gp_factor + ab_gp_set_targets)");
    AB_CUDA(cudaSetDevice(h->device));
    int rc = ensure_linv(h);
    if (rc) return rc;
    return ab_launch_predict_cov(h, d_Xq, m, d_mu, d_cov, ldc);
}

int ab_gp_predict_grad(ab_gp* h, const double* d_Xq, int64_t m, double* d_mu, double* d_var, double* d_dmu,
                       double* d_dvar) {
    AB_REQUIRE(h && d_Xq && d_mu && d_var && d_dmu && d_dvar, -1, "ab_gp_predict_grad: null argument");
    AB_REQUIRE(h->have_alpha, -2, "ab_gp_predict_grad: targets not set (call ab_gp_factor + ab_gp_set_targets)");
    AB_CUDA(cudaSetDevice(h->device));
    int rc = ensure_linv(h);
    if (rc) return rc;
    return ab_launch_predict_grad(h, d_Xq, m, d_mu, d_var, d_dmu, d_dvar);
}

int ab_gp_predict_host(ab_gp* h, const double* h_Xq, int64_t m, double* h_mu, double* h_var) {
    AB_REQUIRE(h && h_Xq && h_mu, -1, "ab_gp_predict_host: null argument");
    AB_REQUIRE(h->have_alpha, -2, "ab_gp_predict_host: targets not set");
    AB_CUDA(cudaSetDevice(h->device));
    size_t nx = (size_t)m * h->d;
    int rc = ensure_io(h, (nx + 2 * (size_t)m) * sizeof(double));
    if (rc) return rc;
    double* dq = h->io;
    double* dmu = h->io + nx;
    double* dvar = h_var ? dmu + m : nullptr;
    if (m <= 8) {
        // one-point calls of optimisers / samplers: inputs and results travel through the handle's
        // page-locked block (one asynchronous copy each way instead of three pageable ones)
        double* st = h->h_pinned + 512;
        memcpy(st, h_Xq, nx * sizeof(double));
        AB_CUDA(cudaMemcpyAsync(dq, st, nx * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        rc = ab_gp_predict(h, dq, m, dmu, dvar);
        if (rc) return rc;
        AB_CUDA(cudaMemcpyAsync(st + 256, dmu, (size_t)(h_var ? 2 : 1) * m * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        AB_CUDA(cudaStreamSynchronize(h->stream));
        memcpy(h_mu, st + 256, (size_t)m * sizeof(double));
        if (h_var) memcpy(h_var, st + 256 + m, (size_t)m * sizeof(double));
        return 0;
    }
    AB_CUDA(cudaMemcpyAsync(dq, h_Xq, nx * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    const int64_t chunk = h_var ? ab_predict_panel_queries(h) : m;
    if (m <= chunk) {
        rc = ab_gp_predict(h, dq, m, dmu, dvar);
        if (rc) return rc;
        AB_CUDA(cudaMemcpyAsync(h_mu, dmu, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (h_var) AB_CUDA(cudaMemcpyAsync(h_var, dvar, (size_t)m * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        AB_CUDA(cudaStreamSynchronize(h->stream));
        return 0;
    }
    // Large batches: the same panels ab_gp_predict would form (identical launches, identical
    // bits), but the results of panel c - 1 travel to the host on the handle's second stream
    // while panel c is computed; the (possibly blocking, pageable) copy is issued after the
    // next panel has been enqueued.
    cudaEvent_t ev[2] = {h->ev_fork, h->ev_join};
    auto copy_out = [&](int64_t off, int64_t cnt, cudaEvent_t e) -> int {
        AB_CUDA(cudaStreamWaitEvent(h->copy_stream, e, 0));
        AB_CUDA(cudaMemcpyAsync(h_mu + off, dmu + off, (size_t)cnt * sizeof(double), cudaMemcpyDeviceToHost, h->copy_stream));
        AB_CUDA(cudaMemcpyAsync(h_var + off, dvar + off, (size_t)cnt * sizeof(double), cudaMemcpyDeviceToHost, h->copy_stream));
        return 0;
    };
    int64_t prev_off = -1, prev_cnt = 0;
    int c = 0;
    for (int64_t off = 0; off < m; off += chunk, c++) {
        const int64_t cnt = (m - off < chunk) ? (m - off) : chunk;
        rc = ab_gp_predict(h, dq + (size_t)off * h->d, cnt, dmu + off, dvar + off);
        if (rc) return rc;
        AB_CUDA(cudaEventRecord(ev[c & 1], h->stream));
        if (prev_off >= 0) {
            rc = copy_out(prev_off, prev_cnt, ev[(c - 1) & 1]);
            if (rc) return rc;
        }
        prev_off = off;
        prev_cnt = cnt;
    }
    rc = copy_out(prev_off, prev_cnt, ev[(c - 1) & 1]);
    if (rc) return rc;
    AB_CUDA(cudaStreamSynchronize(h->copy_stream));
    AB_CUDA(cudaStreamSynchronize(h->stream));
    return 0;
}

int ab_utility_eval(ab_gp* h, int utility_id, const double* d_Xq, const double* d_mu, const double* d_var,
                    int64_t m, const double* h_bounds, double y_best, double zeta, double* d_util,
                    int64_t* h_argmin, double* h_min) {
    AB_REQUIRE(h && d_Xq && d_mu && d_var && h_bounds && h_argmin && h_min, -1, "ab_utility_eval: null argument");
    AB_REQUIRE(utility_id >= 0 && utility_id <= 2, -1, "unknown utility id %d", utility_id);
    AB_REQUIRE(m >= 1, -1, "need at least one candidate");
    AB_CUDA(cudaSetDevice(h->device));
    return ab_launch_utility(h, utility_id, d_Xq, d_mu, d_var, m, h_bounds, y_best, zeta, d_util, h_argmin, h_min);
}

int ab_gp_utility_argmin(ab_gp* h, int utility_id, const double* d_Xq, int64_t m, const double* h_bounds,
                         double y_best, double zeta, double* d_util, int64_t* h_argmin, double* h_min) {
    AB_REQUIRE(h && d_Xq && h_bounds && h_argmin && h_min, -1, "ab_gp_utility_argmin: null argument");
    AB_REQUIRE(m >= 1, -1, "need at least one candidate");
    AB_CUDA(cudaSetDevice(h->device));
    int rc = ensure_io(h, 2 * (size_t)m * sizeof(double));
    if (rc) return rc;
    double* dmu = h->io;
    double* dvar = h->io + m;
    rc = ab_gp_predict(h, d_Xq, m, dmu, dvar);
    if (rc) return rc;
    return ab_utility_eval(h, utility_id, d_Xq, dmu, dvar, m, h_bounds, y_best, zeta, d_util, h_argmin, h_min);
}

long long ab_launch_counter(void) { return g_launches.load(); }

// returns the previous setting (0 / 1)
int ab_gp_set_profiling(ab_gp* h, int enabled) {
    AB_REQUIRE(h, -1, "null handle");
    const int prev = h->profiling ? 1 : 0;
    h->profiling = enabled != 0;
    return prev;
}

// Sum of the device time (ms) between the begin/end marks of one kernel family
// since the last call, and the number of marked launches.  Synchronises.
int ab_gp_profile_read(ab_gp* h, int family, double* h_ms, long long* h_count) {
    AB_REQUIRE(h && h_ms && h_count, -1, "null argument");
    AB_REQUIRE(family >= 0 && family < AB_PROF_FAMILIES, -1, "bad family");
    AB_CUDA(cudaSetDevice(h->device));
    AB_CUDA(cudaStreamSynchronize(h->stream));
    auto& v = h->prof_ev[family];
    double ms = 0.0;
    for (size_t i = 0; i + 1 < v.size(); i += 2) {
        float t = 0.f;
        AB_CUDA(cudaEventElapsedTime(&t, v[i], v[i + 1]));
        ms += t;
    }
    *h_ms = ms;
    *h_count = (long long)(v.size() / 2);
    for (cudaEvent_t e : v) cudaEventDestroy(e);
    v.clear();
    return 0;
}

int64_t ab_gp_padded_size(ab_gp* h) { return h ? h->npad : -1; }

int ab_gp_get_factor(ab_gp* h, double* d_L) {
    AB_REQUIRE(h && d_L, -1, "null argument");
    AB_REQUIRE(h->factored, -2, "not factorised");
    AB_CUDA(cudaSetDevice(h->device));
    AB_CUDA(cudaMemcpyAsync(d_L, h->L, (size_t)h->npad * h->npad * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    return 0;
}

int ab_gp_get_block_inverses(ab_gp* h, double* d_Dinv) {
    AB_REQUIRE(h && d_Dinv, -1, "null argument");
    AB_REQUIRE(h->factored, -2, "not factorised");
    AB_CUDA(cudaSetDevice(h->device));
    AB_CUDA(cudaMemcpyAsync(d_Dinv, h->Dinv, (size_t)h->npad * AB_NB * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    return 0;
}

int ab_gp_get_alpha(ab_gp* h, double* d_alpha) {
    AB_REQUIRE(h && d_alpha, -1, "null argument");
    AB_REQUIRE(h->have_alpha, -2, "targets not set");
    AB_CUDA(cudaSetDevice(h->device));
    AB_CUDA(cudaMemcpyAsync(d_alpha, h->alpha, (size_t)h->n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    return 0;
}

int ab_gp_get_inverse(ab_gp* h, double* d_Kinv) {
    AB_REQUIRE(h && d_Kinv, -1, "null argument");
    AB_REQUIRE(h->factored, -2, "not factorised");
    AB_CUDA(cudaSetDevice(h->device));
    int rc = ensure_kinv(h);
    if (rc) return rc;
    rc = ab_launch_mirror_lower(h, h->Kinv, h->npad);
    if (rc) return rc;
    AB_CUDA(cudaMemcpy2DAsync(d_Kinv, (size_t)h->n * sizeof(double), h->Kinv, (size_t)h->npad * sizeof(double),
                              (size_t)h->n * sizeof(double), (size_t)h->n, cudaMemcpyDeviceToDevice, h->stream));
    return 0;
}

// Adopt a factor and alpha computed elsewhere (another GPU, after an NCCL
// broadcast).  The diagonal-block inverses are rebuilt locally from L.
int ab_gp_import_state(ab_gp* h, const double* d_L, const double* d_alpha) {
    return ab_gp_import_state_full(h, d_L, nullptr, d_alpha);
}

// d_Dinv != NULL: adopt the sender's diagonal-block inverses as well, so that everything
// derived from the factor (L^-1, K^-1, variances) has the SAME bits on every GPU; NULL:
// rebuild them locally (same values up to rounding).
int ab_gp_import_state_full(ab_gp* h, const double* d_L, const double* d_Dinv, const double* d_alpha) {
    AB_REQUIRE(h && d_L && d_alpha, -1, "null argument");
    AB_CUDA(cudaSetDevice(h->device));
    int rc = ensure_scaled(h);
    if (rc) return rc;
    AB_CUDA(cudaMemcpyAsync(h->L, d_L, (size_t)h->npad * h->npad * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    AB_CUDA(cudaMemsetAsync(h->alpha, 0, (size_t)h->npad * sizeof(double), h->stream));
    AB_CUDA(cudaMemcpyAsync(h->alpha, d_alpha, (size_t)h->n * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    rc = ab_launch_rebuild_dinv(h);                    // also the log-determinant parts
    if (rc) return rc;
    if (d_Dinv)
        AB_CUDA(cudaMemcpyAsync(h->Dinv, d_Dinv, (size_t)h->npad * AB_NB * sizeof(double), cudaMemcpyDeviceToDevice, h->stream));
    h->factored = true;
    h->have_alpha = true;
    h->have_linv = h->have_kinv = false;
    return 0;
}

}  // extern "C"
