// Constrained random walks for nested sampling on the surrogate (SURVEY 8f-2).
//
// The reference hands SurrogateModel.surrogate_log_likelihood to dynesty
// (alabi/core.py:2549-2706), which replaces the worst live point by a point drawn inside the
// hard constraint L > L_min — with sample="rwalk": `walks` Metropolis steps in the unit cube from
// a random live point, one likelihood call (one GP predict, one re-factorisation in the reference,
// core.py:1430) per step.  Here a whole batch of such walks is ONE launch: every chain proposes
// u' = u + scale * C z (C = Cholesky factor of the live points' covariance, z ~ N(0, I) from
// Philox + Box-Muller), maps it through the prior transform (uniform box, or the inverse normal
// CDF for ut.prior_transform_normal dimensions), evaluates the surrogate mean exactly like the
// sampler kernel of ensemble.cu (theta scaler, axis-aligned metric, kernel sum against alpha,
// y scaler) and accepts iff the point is inside the cube and L > L_min.
//
// Work decomposition: one CTA = 32 chains (lane e of every warp owns chain e), the 8 warps split
// the training points, which sit SoA in shared memory (resident when they fit, else chunked).
// The partial sums of the warps are added in warp order, so a chain's log-likelihood does not
// depend on the batch it runs in.
#include <cmath>
#include "handle.h"
#include "alabi_b200.h"
#include "philox.cuh"

namespace {

constexpr int NW = 8;                // warps per CTA
constexpr int NTHREADS = NW * 32;

struct WalkArgs {
    double* u; double* logl; double* theta; int* naccept;
    const double* chol;              // d x d lower factor (row-major), device
    const double* XsT; const double* alpha; long long n, npad;
    KernParams kp; double mean;
    int nchains, d, walks, ch;
    double scale, lmin;
    unsigned seed_lo, seed_hi;
    long long counter, chain_offset;
    double lo[AB_MAX_DIM], width[AB_MAX_DIM], pr_mu[AB_MAX_DIM], pr_sd[AB_MAX_DIM];
    double t_scale[AB_MAX_DIM], t_off[AB_MAX_DIM];
    int y_kind; double y_scale, y_off;
};

using abr::U4;
using abr::philox;
using abr::u53;

template <int KIND, int D>
__global__ void __launch_bounds__(NTHREADS)
nested_walk_kernel(const __grid_constant__ WalkArgs A) {
    extern __shared__ __align__(16) double sm[];
    const int CH = A.ch;
    double* sX = sm;                  // [D][CH]
    double* sAl = sm + D * CH;        // [CH]
    __shared__ double sQs[32][D + 1]; // scaled proposal of chain e (pitch D + 1: conflict-free column reads)
    __shared__ double sPart[NW][32];
    __shared__ double sC[AB_MAX_DIM * AB_MAX_DIM];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int d = A.d;
    const long long chain = (long long)blockIdx.x * 32 + lane;
    const bool resident = A.n <= CH;
    const bool owner = (warp == 0) && chain < A.nchains;

    for (int i = tid; i < d * d; i += NTHREADS) sC[i] = A.chol[i];
    auto load_chunk = [&](long long c0) {
        for (int idx = tid; idx < D * CH; idx += NTHREADS) {
            int k = idx / CH, jj = idx - k * CH;
            sX[idx] = (k < d && c0 + jj < A.n) ? A.XsT[(long long)k * A.npad + c0 + jj] : 0.0;
        }
        for (int jj = tid; jj < CH; jj += NTHREADS) sAl[jj] = (c0 + jj < A.n) ? A.alpha[c0 + jj] : 0.0;
    };
    if (resident) load_chunk(0);

    // chain state (owner lanes)
    double u[D], un[D], th[D];
    double logl = 0.0;
    int nacc = 0;
    if (owner) {
#pragma unroll
        for (int k = 0; k < D; k++) u[k] = (k < d) ? A.u[chain * d + k] : 0.0;
        logl = A.logl[chain];
    }
    __syncthreads();

    for (int step = 0; step < A.walks; step++) {
        // ---- proposal (owner lanes) -------------------------------------------------------
        int inside = 0;
        if (owner) {
            double z[D];
#pragma unroll
            for (int k = 0; k < D; k += 2) {
                if (k >= d) { z[k] = 0.0; if (k + 1 < D) z[k + 1] = 0.0; continue; }
                // one Philox call per pair of normals: Box-Muller on two 53-bit uniforms
                U4 r = philox((unsigned)(A.chain_offset + chain), (unsigned)step, (unsigned)(k >> 1),
                              (unsigned)A.counter, A.seed_lo, A.seed_hi);
                const double u1 = 1.0 - u53(r.x, r.y), u2 = u53(r.z, r.w);     // u1 in (0, 1]
                const double rad = sqrt(-2.0 * log(u1));
                double sn, cs;
                sincospi(2.0 * u2, &sn, &cs);
                z[k] = rad * cs;
                if (k + 1 < D) z[k + 1] = rad * sn;
            }
            inside = 1;
#pragma unroll
            for (int k = 0; k < D; k++) {
                if (k < d) {
                    double s = 0.0;
                    for (int j = 0; j <= k; j++) s = fma(sC[k * d + j], z[j], s);
                    un[k] = u[k] + A.scale * s;
                    if (!(un[k] > 0.0 && un[k] < 1.0)) inside = 0;
                } else {
                    un[k] = 0.0;
                }
            }
#pragma unroll
            for (int k = 0; k < D; k++) {
                double t = 0.0;
                if (k < d && inside) {
                    // ut.prior_transform_uniform: (hi - lo) * u + lo;  ut.prior_transform_normal: norm.ppf(u, mu, sd)
                    t = (A.pr_sd[k] > 0.0) ? __dadd_rn(__dmul_rn(normcdfinv(un[k]), A.pr_sd[k]), A.pr_mu[k])
                                           : __dadd_rn(__dmul_rn(A.width[k], un[k]), A.lo[k]);
                }
                th[k] = t;
                sQs[lane][k] = (k < d) ? fma(t, A.t_scale[k], A.t_off[k]) * A.kp.inv_len[k] : 0.0;
            }
        } else if (warp == 0) {
#pragma unroll
            for (int k = 0; k < D; k++) sQs[lane][k] = 0.0;
        }
        __syncthreads();
        // ---- surrogate mean of the 32 proposals: warps split the training points ------------
        double qv[D];
#pragma unroll
        for (int k = 0; k < D; k++) qv[k] = sQs[lane][k];
        double acc = 0.0;
        auto eval = [&](int cn) {
            const int per = cn / NW;                 // cn is a multiple of 32 >= NW
            const int j0 = warp * per, j1 = j0 + per;
#pragma unroll 2
            for (int j = j0; j < j1; j += 2) {
                double r0 = 0.0, r1 = 0.0;
#pragma unroll
                for (int k = 0; k < D; k++) {
                    const double2 xx = *reinterpret_cast<const double2*>(&sX[k * CH + j]);
                    const double d0 = qv[k] - xx.x, d1 = qv[k] - xx.y;
                    r0 = fma(d0, d0, r0);
                    r1 = fma(d1, d1, r1);
                }
                const double2 al = *reinterpret_cast<const double2*>(&sAl[j]);
                acc = fma(ab_radial<KIND>(r0, A.kp.alpha, A.kp.inv2a), al.x, acc);
                acc = fma(ab_radial<KIND>(r1, A.kp.alpha, A.kp.inv2a), al.y, acc);
            }
        };
        if (resident) {
            eval(CH);
        } else {
            for (long long c0 = 0; c0 < A.n; c0 += CH) {
                __syncthreads();
                load_chunk(c0);
                __syncthreads();
                eval(CH);
            }
        }
        sPart[warp][lane] = acc;
        __syncthreads();
        // ---- accept / reject (owner lanes) ---------------------------------------------------------
        if (owner && inside) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < NW; w++) s += sPart[w][lane];
            const double ys = fma(A.kp.amp, s, A.mean);
            const double y = (A.y_kind == 0) ? fma(ys, A.y_scale, A.y_off)
                           : (A.y_kind == 1) ? -pow(10.0, ys) : pow(10.0, ys);
            if (y > A.lmin) {
#pragma unroll
                for (int k = 0; k < D; k++) u[k] = un[k];
                logl = y;
                nacc++;
                for (int k = 0; k < d; k++) A.theta[chain * d + k] = th[k];
            }
        }
        __syncthreads();
    }
    if (owner) {
        for (int k = 0; k < d; k++) A.u[chain * d + k] = u[k];
        A.logl[chain] = logl;
        A.naccept[chain] = nacc;
    }
}

template <int KIND, int D>
int launch_walk(ab_gp* h, WalkArgs& A) {
    auto kern = nested_walk_kernel<KIND, D>;
    const size_t budget = 160 * 1024;
    int ch;
    if ((size_t)A.n * (D + 1) * 8 <= budget) {
        ch = (int)((A.n + 31) / 32 * 32);
    } else {
        ch = (int)(budget / ((D + 1) * 8)) / 32 * 32;
    }
    if (ch < 32) ch = 32;
    A.ch = ch;
    const size_t smem = (size_t)ch * (D + 1) * 8;
    AB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned grid = (unsigned)((A.nchains + 31) / 32);
    kern<<<grid, NTHREADS, smem, h->stream>>>(A);
    AB_CHECK_LAUNCH();
    ab_count_launches(1);
    return 0;
}

}  // namespace

extern "C" int ab_nested_walk(ab_gp* h, const ab_nested_config* cfg, double* d_u, double* d_logl, double* d_theta,
                              int* d_naccept) {
    if (!h || !cfg || !d_u || !d_logl || !d_theta || !d_naccept) { ab_set_error("ab_nested_walk: null argument"); return -1; }
    if (!h->have_alpha) { ab_set_error("ab_nested_walk: targets not set (call ab_gp_set_targets)"); return -2; }
    if (cfg->nchains < 1 || cfg->walks < 0) { ab_set_error("ab_nested_walk: bad configuration"); return -1; }
    AB_CUDA(cudaSetDevice(h->device));
    const int d = h->d;
    int rc = ab_ensure_scratch(h, (size_t)AB_MAX_DIM * AB_MAX_DIM * sizeof(double) + 4096);
    if (rc) return rc;
    // proposal covariance factor: a copy from pageable memory returns once the source has been
    // staged, so the caller's struct may be reused right away
    double* dchol = h->scratch + 64;
    AB_CUDA(cudaMemcpyAsync(dchol, cfg->chol, (size_t)d * d * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    WalkArgs A{};
    A.u = d_u; A.logl = d_logl; A.theta = d_theta; A.naccept = d_naccept; A.chol = dchol;
    A.XsT = h->XsT; A.alpha = h->alpha; A.n = h->n; A.npad = h->npad; A.kp = h->kp; A.mean = h->mean;
    A.nchains = cfg->nchains; A.d = d; A.walks = cfg->walks;
    A.scale = cfg->scale; A.lmin = cfg->lmin;
    A.seed_lo = (unsigned)(cfg->seed & 0xffffffffULL); A.seed_hi = (unsigned)(cfg->seed >> 32);
    A.counter = cfg->counter; A.chain_offset = cfg->chain_offset;
    for (int k = 0; k < d; k++) {
        A.lo[k] = cfg->lo[k]; A.width[k] = cfg->hi[k] - cfg->lo[k];
        A.pr_mu[k] = cfg->prior_mu[k]; A.pr_sd[k] = cfg->use_normal_prior ? cfg->prior_sd[k] : 0.0;
        A.t_scale[k] = cfg->theta_scale[k]; A.t_off[k] = cfg->theta_offset[k];
    }
    A.y_kind = cfg->y_kind; A.y_scale = cfg->y_scale; A.y_off = cfg->y_offset;
#define AB_NW(DD) AB_DISPATCH_KIND(h->kp.kind, rc = (launch_walk<KIND, DD>(h, A)))
    if (d <= 2) AB_NW(2);
    else if (d <= 4) AB_NW(4);
    else if (d <= 8) AB_NW(8);
    else if (d <= 12) AB_NW(12);
    else if (d <= 16) AB_NW(16);
    else if (d <= 20) AB_NW(20);
    else if (d <= 24) AB_NW(24);
    else AB_NW(32);
#undef AB_NW
    return rc;
}

extern "C" int ab_sizeof_nested_config(void) { return (int)sizeof(ab_nested_config); }
