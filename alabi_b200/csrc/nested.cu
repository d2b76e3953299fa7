// Constrained moves for nested sampling on the surrogate (SURVEY 8f-2).
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
// sample="rslice" (dynesty's random-direction slice sampling) is a second kernel on the same
// parts: each of `slices` steps draws a direction v = scale * C z / |z| and samples the slice
// {x : L(T(u + x v)) > L_min} by stepping out and shrinking (Neal 2003), see nested_rslice_kernel.
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

// Step-out moves and failed shrink draws allowed per slice; a chain that would need more stops
// at the end point of its last completed slice (include/alabi_b200.h, ab_nested_rslice).
constexpr int RSLICE_MAX_EXPAND = 1024;
constexpr int RSLICE_MAX_CONTRACT = 256;

struct WalkArgs {
    double* u; double* logl; double* theta;
    int* counts;                     // walk: accepted steps per chain; rslice: 4 counts per chain
    const double* chol;              // d x d lower factor (row-major), device
    const double* XsT; const double* alpha; long long n, npad;
    KernParams kp; double mean;
    int nchains, d, walks, ch;       // walks: walk steps, or slices for rslice
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

// normals 2p and 2p + 1 of step `step` of chain `cid`: one Philox call, Box-Muller on two 53-bit
// uniforms
__device__ __forceinline__ void normal_pair(const WalkArgs& A, unsigned cid, int step, int p, double& z0, double& z1) {
    U4 r = philox(cid, (unsigned)step, (unsigned)p, (unsigned)A.counter, A.seed_lo, A.seed_hi);
    const double u1 = 1.0 - u53(r.x, r.y), u2 = u53(r.z, r.w);     // u1 in (0, 1]
    const double rad = sqrt(-2.0 * log(u1));
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    z0 = rad * cs;
    z1 = rad * sn;
}

// ut.prior_transform_uniform: (hi - lo) * u + lo;  ut.prior_transform_normal: norm.ppf(u, mu, sd)
__device__ __forceinline__ double prior_theta(const WalkArgs& A, int k, double u) {
    return (A.pr_sd[k] > 0.0) ? __dadd_rn(__dmul_rn(normcdfinv(u), A.pr_sd[k]), A.pr_mu[k])
                              : __dadd_rn(__dmul_rn(A.width[k], u), A.lo[k]);
}

// training points [c0, c0 + CH) into shared memory, zero-padded
template <int D>
__device__ __forceinline__ void load_points(const WalkArgs& A, double* sX, double* sAl, int CH, long long c0, int tid, int d) {
    for (int idx = tid; idx < D * CH; idx += NTHREADS) {
        int k = idx / CH, jj = idx - k * CH;
        sX[idx] = (k < d && c0 + jj < A.n) ? A.XsT[(long long)k * A.npad + c0 + jj] : 0.0;
    }
    for (int jj = tid; jj < CH; jj += NTHREADS) sAl[jj] = (c0 + jj < A.n) ? A.alpha[c0 + jj] : 0.0;
}

// acc += this warp's share of sum_j k(qv, x_j) alpha_j over the CH points in shared memory
template <int KIND, int D>
__device__ __forceinline__ void partial_sum(const WalkArgs& A, const double* sX, const double* sAl, int CH,
                                            const double (&qv)[D], int warp, double& acc) {
    const int per = CH / NW;                     // CH is a multiple of 32 >= NW
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
}

// surrogate log-likelihood of chain `lane` from the warps' partial sums (added in warp order)
__device__ __forceinline__ double surrogate_y(const WalkArgs& A, const double (*sPart)[32], int lane) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < NW; w++) s += sPart[w][lane];
    const double ys = fma(A.kp.amp, s, A.mean);
    return (A.y_kind == 0) ? fma(ys, A.y_scale, A.y_off)
         : (A.y_kind == 1) ? -pow(10.0, ys) : pow(10.0, ys);
}

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
    if (resident) load_points<D>(A, sX, sAl, CH, 0, tid, d);

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
                double z1;
                normal_pair(A, (unsigned)(A.chain_offset + chain), step, k >> 1, z[k], z1);
                if (k + 1 < D) z[k + 1] = z1;
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
                const double t = (k < d && inside) ? prior_theta(A, k, un[k]) : 0.0;
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
        auto eval = [&](int cn) { partial_sum<KIND, D>(A, sX, sAl, cn, qv, warp, acc); };
        if (resident) {
            eval(CH);
        } else {
            for (long long c0 = 0; c0 < A.n; c0 += CH) {
                __syncthreads();
                load_points<D>(A, sX, sAl, CH, c0, tid, d);
                __syncthreads();
                eval(CH);
            }
        }
        sPart[warp][lane] = acc;
        __syncthreads();
        // ---- accept / reject (owner lanes) ---------------------------------------------------------
        if (owner && inside) {
            const double y = surrogate_y(A, sPart, lane);
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
        A.counts[chain] = nacc;
    }
}

// Random-direction slice sampling (dynesty's sample="rslice"), `A.walks` slices per chain.
// Slice s of chain c:
//   direction  z ~ N(0, I_d) from the walk's normals at step = s, v = (C z) * (scale / |z|)
//   window     r0 = u53 of Philox block j0 = ceil(d/2) (words 0, 1); x_l = -r0, x_r = 1 - r0
//   step out   while F(x_l) > lmin: x_l -= 1; then while F(x_r) > lmin: x_r += 1  (one nexpand each)
//   shrink     draw i = 0, 1, ...: x = x_l + u_i (x_r - x_l), u_i from block j0 + 1 + i;
//              F(x) > lmin accepts u <- u + x v, else x_l = x (x < 0) or x_r = x (x > 0)  (one ncontract)
// with F(x) = L(T(u + x v)) inside (0, 1)^d and -inf (no evaluation) outside.  The window and
// point arithmetic is separately rounded (no contraction), so a CPU replay takes the same branches.
//
// Rounds: every unfinished owner lane advances its state machine to its next in-cube proposal
// (out-of-cube steps are free and taken at once), the 8 warps evaluate the <= 32 proposals, the
// owners consume the results.  The CTA ends when no lane is unfinished.  A chain only sees its own
// draws and likelihood values, so its result does not depend on the batch or its neighbours.
template <int KIND, int D>
__global__ void __launch_bounds__(NTHREADS)
nested_rslice_kernel(const __grid_constant__ WalkArgs A) {
    extern __shared__ __align__(16) double sm[];
    const int CH = A.ch;
    double* sX = sm;                  // [D][CH]
    double* sAl = sm + D * CH;        // [CH]
    __shared__ double sQs[32][D + 1]; // scaled proposal of chain e
    __shared__ double sU[32][D + 1];  // current point of chain e (unit cube)
    __shared__ double sV[32][D + 1];  // slice direction of chain e
    __shared__ double sPart[NW][32];
    __shared__ double sC[AB_MAX_DIM * AB_MAX_DIM];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int d = A.d;
    const long long chain = (long long)blockIdx.x * 32 + lane;
    const bool resident = A.n <= CH;
    const bool owner = (warp == 0) && chain < A.nchains;
    const unsigned cid = (unsigned)(A.chain_offset + chain);
    const int j0 = (d + 1) / 2;       // first Philox block after the direction's normals

    for (int i = tid; i < d * d; i += NTHREADS) sC[i] = A.chol[i];
    if (resident) load_points<D>(A, sX, sAl, CH, 0, tid, d);
    if (warp == 0) {
        for (int k = 0; k < D; k++) {
            sQs[lane][k] = 0.0;
            sV[lane][k] = 0.0;
            sU[lane][k] = (owner && k < d) ? A.u[chain * d + k] : 0.0;
        }
    }

    // chain state (owner lanes)
    int s = 0, phase = 0, i = 0, nexp_s = 0, ncon_s = 0, nexp = 0, ncon = 0, nev = 0;
    double xl = 0.0, xr = 0.0, x = 0.0, logl = owner ? A.logl[chain] : 0.0;
    bool done = !owner || A.walks == 0, pending = false;
    __syncthreads();

    auto uniform = [&](int j) {
        const U4 r = philox(cid, (unsigned)s, (unsigned)j, (unsigned)A.counter, A.seed_lo, A.seed_hi);
        return u53(r.x, r.y);
    };
    auto shrink_draw = [&]() { return __dadd_rn(xl, __dmul_rn(uniform(j0 + 1 + i), __dadd_rn(xr, -xl))); };
    auto begin_slice = [&]() {
        double z[D];
#pragma unroll
        for (int k = 0; k < D; k += 2) {
            if (k >= d) { z[k] = 0.0; if (k + 1 < D) z[k + 1] = 0.0; continue; }
            double z1;
            normal_pair(A, cid, s, k >> 1, z[k], z1);
            if (k + 1 < D) z[k + 1] = z1;
        }
        double nz = 0.0;             // |z| over the d dimensions (for odd d the last pair also fills z[d])
#pragma unroll
        for (int k = 0; k < D; k++) if (k < d) nz = fma(z[k], z[k], nz);
        const double f = A.scale / sqrt(nz);
#pragma unroll
        for (int k = 0; k < D; k++) {
            if (k < d) {
                double c = 0.0;
                for (int j = 0; j <= k; j++) c = fma(sC[k * d + j], z[j], c);
                sV[lane][k] = c * f;
            }
        }
        const double r0 = uniform(j0);
        xl = -r0; xr = __dadd_rn(1.0, -r0); x = xl;
        phase = 0; i = 0; nexp_s = 0; ncon_s = 0;
    };
    // u + x v into sQs (scaled) when it lies inside the unit cube; false: F(x) = -inf
    auto propose = [&]() {
        for (int k = 0; k < d; k++) {
            const double p = __dadd_rn(sU[lane][k], __dmul_rn(x, sV[lane][k]));
            if (!(p > 0.0 && p < 1.0)) return false;
        }
        for (int k = 0; k < d; k++) {
            const double p = __dadd_rn(sU[lane][k], __dmul_rn(x, sV[lane][k]));
            sQs[lane][k] = fma(prior_theta(A, k, p), A.t_scale[k], A.t_off[k]) * A.kp.inv_len[k];
        }
        return true;
    };
    // outcome ok = F(x) > lmin of the current x: next x, the next slice, or the end of the chain
    auto advance = [&](bool ok, double y) {
        if (phase < 2) {                                   // stepping out: 0 left, 1 right
            if (ok) {
                if (nexp_s == RSLICE_MAX_EXPAND) { done = true; return; }
                nexp_s++; nexp++;
                if (phase == 0) { xl = __dadd_rn(xl, -1.0); x = xl; }
                else { xr = __dadd_rn(xr, 1.0); x = xr; }
            } else if (phase == 0) {
                phase = 1; x = xr;
            } else {
                phase = 2; x = shrink_draw();
            }
        } else if (ok) {                                   // shrinking: accept
            for (int k = 0; k < d; k++) {
                const double p = __dadd_rn(sU[lane][k], __dmul_rn(x, sV[lane][k]));
                sU[lane][k] = p;
                A.theta[chain * d + k] = prior_theta(A, k, p);
            }
            logl = y;
            if (++s == A.walks) done = true;
            else begin_slice();
        } else {                                           // shrinking: reject
            ncon_s++; ncon++;
            if (x < 0.0) xl = x;
            else if (x > 0.0) xr = x;
            if (ncon_s == RSLICE_MAX_CONTRACT) { done = true; return; }
            i++; x = shrink_draw();
        }
    };
    auto next_proposal = [&]() {
        pending = false;
        while (!done) {
            if (propose()) { pending = true; nev++; return; }
            advance(false, 0.0);
        }
    };

    if (!done) { begin_slice(); next_proposal(); }
    while (__syncthreads_or(pending)) {
        double qv[D];
#pragma unroll
        for (int k = 0; k < D; k++) qv[k] = sQs[lane][k];
        double acc = 0.0;
        auto eval = [&](int cn) { partial_sum<KIND, D>(A, sX, sAl, cn, qv, warp, acc); };
        if (resident) {
            eval(CH);
        } else {
            for (long long c0 = 0; c0 < A.n; c0 += CH) {
                __syncthreads();
                load_points<D>(A, sX, sAl, CH, c0, tid, d);
                __syncthreads();
                eval(CH);
            }
        }
        sPart[warp][lane] = acc;
        __syncthreads();
        if (pending) {                                     // owner lanes only
            const double y = surrogate_y(A, sPart, lane);
            advance(y > A.lmin, y);
            next_proposal();
        }
    }
    if (owner) {
        for (int k = 0; k < d; k++) A.u[chain * d + k] = sU[lane][k];
        A.logl[chain] = logl;
        int* c = A.counts + chain * 4;
        c[0] = s; c[1] = nexp; c[2] = ncon; c[3] = nev;
    }
}

template <int D>
int launch_nested(ab_gp* h, WalkArgs& A, void (*kern)(const WalkArgs)) {
    int ch;
    if (ab_resident(A.n, D)) {
        ch = (int)((A.n + 31) / 32 * 32);
    } else {
        ch = (int)(AB_RESIDENT_SMEM / ((D + 1) * 8)) / 32 * 32;
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

// argument checks and kernel arguments shared by both entry points
int nested_args(const char* what, ab_gp* h, const ab_nested_config* cfg, double* d_u, double* d_logl, double* d_theta,
                int* d_counts, WalkArgs& A) {
    if (!h || !cfg || !d_u || !d_logl || !d_theta || !d_counts) { ab_set_error("%s: null argument", what); return -1; }
    if (!h->have_alpha) { ab_set_error("%s: targets not set (call ab_gp_set_targets)", what); return -2; }
    if (cfg->nchains < 1 || cfg->walks < 0) { ab_set_error("%s: bad configuration", what); return -1; }
    AB_CUDA(cudaSetDevice(h->device));
    const int d = h->d;
    int rc = ab_ensure_scratch(h, (size_t)AB_MAX_DIM * AB_MAX_DIM * sizeof(double) + 4096);
    if (rc) return rc;
    // proposal covariance factor: a copy from pageable memory returns once the source has been
    // staged, so the caller's struct may be reused right away
    double* dchol = h->scratch + 64;
    AB_CUDA(cudaMemcpyAsync(dchol, cfg->chol, (size_t)d * d * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    A = WalkArgs{};
    A.u = d_u; A.logl = d_logl; A.theta = d_theta; A.counts = d_counts; A.chol = dchol;
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
    return 0;
}

int dispatch_nested(ab_gp* h, WalkArgs& A, bool rslice) {
    return ab_dispatch_dim(A.d, [&](auto D) {
        int rc = 0;
        AB_DISPATCH_KIND(h->kp.kind, rc = (launch_nested<D>(h, A, rslice ? nested_rslice_kernel<KIND, D>
                                                                          : nested_walk_kernel<KIND, D>)));
        return rc;
    });
}

}  // namespace

extern "C" int ab_nested_walk(ab_gp* h, const ab_nested_config* cfg, double* d_u, double* d_logl, double* d_theta,
                              int* d_naccept) {
    WalkArgs A;
    int rc = nested_args("ab_nested_walk", h, cfg, d_u, d_logl, d_theta, d_naccept, A);
    return rc ? rc : dispatch_nested(h, A, false);
}

extern "C" int ab_nested_rslice(ab_gp* h, const ab_nested_config* cfg, double* d_u, double* d_logl, double* d_theta,
                                int* d_counts) {
    WalkArgs A;
    int rc = nested_args("ab_nested_rslice", h, cfg, d_u, d_logl, d_theta, d_counts, A);
    return rc ? rc : dispatch_nested(h, A, true);
}

extern "C" int ab_sizeof_nested_config(void) { return (int)sizeof(ab_nested_config); }
