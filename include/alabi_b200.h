/* alabi_b200 — C ABI of the B200-native GP surrogate hot path.
 *
 * The reference (jbirky/alabi) has no FFI layer: the seam is the object
 * protocol it consumes from george / emcee (SURVEY.md 8b).  Every entry point
 * below names the reference call it replaces.  A maintainer binds this library
 * with ctypes (INTEGRATION.md shows the stub); alabi_b200/_lib.py is that
 * binding and alabi_b200/gp.py / ensemble.py mirror the george / emcee objects
 * on top of it.
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer owned by the caller (a
 *     torch tensor's data_ptr()); h_* is a host pointer; FP64, row-major,
 *     C-contiguous.
 *   - a handle is bound to one device and one stream (the caller's, borrowed),
 *     is not re-entrant, and owns K / L / L^-1 / K^-1 / alpha workspaces.
 *   - return value: 0 = ok; > 0 = numerical status (factorisation: 1-based index
 *     of the first non-positive pivot, LAPACK dpotrf style; sampler: 1 = NaN
 *     log-probability); < 0 = bad argument or CUDA error, text in
 *     ab_last_error().  Nothing throws or exits across the ABI.
 *   - hyper-parameters follow george's vector
 *       [mean:value, white_noise:value, kernel:k1:log_constant,
 *        kernel:k2:metric:log_M_0_0, ...]        (docs/source/save_reload.py:117-120)
 *     but are passed unpacked; white_noise is ln(variance), log_M is ln(l^2).
 */
#ifndef ALABI_B200_H
#define ALABI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AB_MAX_DIM_PUBLIC 32

/* kernel ids: george.kernels.{ExpSquared,Matern32,Matern52}Kernel, alabi/core.py:998-1014 */
#define AB_KERNEL_EXPSQUARED 0
#define AB_KERNEL_MATERN32 1
#define AB_KERNEL_MATERN52 2
#define AB_KERNEL_RATQUAD 3      /* george RationalQuadraticKernel: set with ab_gp_set_kernel_rq */

/* utility ids: alabi/utility.py:729 (bape), :629 (agp), :853 (jones) */
#define AB_UTILITY_BAPE 0
#define AB_UTILITY_AGP 1
#define AB_UTILITY_JONES 2

/* Philox counter streams of the sampler (restated in oracle/philox.py) */
#define AB_STREAM_SPLIT 0
#define AB_STREAM_PARTNER 1
#define AB_STREAM_MOVE 2
/* Philox counter stream of the multivariate-normal draws of ab_mvn_sample */
#define AB_STREAM_MVN 3

typedef struct ab_gp ab_gp;

int ab_version(void);
/* sizeof(ab_ensemble_config) as compiled: a binding checks its mirror of the struct against it */
int ab_sizeof_ensemble_config(void);
const char* ab_last_error(void);
/* multiprocessor count of `device`, < 0 on error (also proves a usable GPU) */
int ab_device_sm_count(int device);

/* instrumentation used by bench.py: number of kernels this library has launched
 * in the process, and per-family device time between CUDA events recorded on
 * the handle's stream (family: 0 cov, 1 factor, 2 predict panel/mean,
 * 3 predict variance GEMM, 4 ensemble) */
long long ab_launch_counter(void);
/* measured issue-rate peak of the FP64 tensor pipe (DMMA.8x8x4), TFLOP/s */
int ab_fp64_tensor_peak(int device, double* h_tflops);
/* measured issue-rate peak of plain FP64 FMA (DFMA), TFLOP/s: the roof of the kernel-evaluation
 * loops (covariance build, predictive mean, sampler) */
int ab_fp64_fma_peak(int device, double* h_tflops);
int ab_gp_set_profiling(ab_gp* h, int enabled);   /* returns the previous setting (0 / 1) */
int ab_gp_profile_read(ab_gp* h, int family, double* h_ms, long long* h_count);

/* ---- lifecycle: george.GP(kernel, fit_mean, mean, white_noise, fit_white_noise)
 *      alabi/gp_utils.py:233, alabi/core.py:1141 ------------------------------- */
int ab_gp_create(ab_gp** out, int device, void* cuda_stream);
int ab_gp_destroy(ab_gp* h);
/* predictions of <= 8 queries (GP.predict with M = 1 inside optimisers and samplers,
 * alabi/utility.py:629-946) use kernels that spread one query over the GPU and reproduce the
 * batched kernels' bits; 0 sends them through the batched kernels (cross-check), default 1 */
int ab_gp_set_few_query_path(ab_gp* h, int enabled);

/* Append ONE training point (d doubles on the device, same space as X) to a
 * factorised model in O(N^2): bordered Cholesky update instead of the full
 * refactorisation `_fit_gp` -> `gp.compute` performs after every active-learning
 * step (alabi/core.py:1780 -> 1158) when the hyper-parameters are unchanged.
 * Returns 0, or k > 0 (= n + 1) when the bordered matrix is not positive definite
 * (the handle is then left un-factorised, like a failed ab_gp_factor). */
int ab_gp_append_point(ab_gp* h, const double* d_x);

/* training inputs of gp.compute(x): X is n x d (copied).  alabi/gp_utils.py:243 */
int ab_gp_set_inputs(ab_gp* h, const double* d_X, int64_t n, int d);

/* kernel id + unpacked george parameter vector (gp.set_parameter_vector,
 * alabi/core.py:705,1152).  amp = exp(log_constant) (1.0 without amplitude);
 * h_log_M has d entries; yerr2 is george's yerr^2 (0 in alabi). Marks the
 * factorisation dirty. */
int ab_gp_set_kernel(ab_gp* h, int kernel_id, double amp, const double* h_log_M, double mean,
                     double white_noise, double yerr2);

/* ab_gp_set_kernel for george's RationalQuadraticKernel (AB_KERNEL_RATQUAD, the kernel with a
 * parameter of its own): k(r^2) = (1 + r^2 / (2 alpha))^(-alpha), alpha = exp(log_alpha),
 * r^2 = sum_k dx_k^2 / M_k.  Returns -1 when exp(log_alpha) is not finite and positive.
 * ab_gp_set_kernel rejects kernel id 3: this is the only way to select it. */
int ab_gp_set_kernel_rq(ab_gp* h, double amp, double log_alpha, const double* h_log_M, double mean,
                        double white_noise, double yerr2);

/* K1: kernel.get_value(x) [+ diagonal]: full symmetric n x n matrix into d_K
 * (ld = n).  with_diag != 0 adds yerr2 + exp(white_noise) like GP.compute. */
int ab_gp_build_cov(ab_gp* h, double* d_K, int with_diag);
/* kernel.get_value(x1, x2) (alabi/utility.py:549-550,607): m1 x m2 into d_K */
int ab_gp_cross_cov(ab_gp* h, const double* d_X1, int64_t m1, const double* d_X2, int64_t m2, double* d_K);

/* K1 + K2: gp.compute / gp.recompute — build K, Cholesky.  Returns 0 or the
 * 1-based index of the first non-positive pivot (george raises LinAlgError;
 * quiet=True callers map it to -inf / zero gradient). */
int ab_gp_factor(ab_gp* h);
int ab_gp_log_determinant(ab_gp* h, double* h_out);

/* alpha = K^-1 (y - mean) (george GP._compute_alpha); d_y has n entries. */
int ab_gp_set_targets(ab_gp* h, const double* d_y);
/* gp.log_likelihood(y): -1/2 r^T K^-1 r - 1/2 logdet - n/2 ln 2pi.  alabi/core.py:1248 */
int ab_gp_log_likelihood(ab_gp* h, const double* d_y, double* h_out);
/* gp.grad_log_likelihood(y): h_out[0..d+2] = d/d[mean, white_noise, log_constant,
 * log_M_0..]; for AB_KERNEL_RATQUAD h_out[0..d+3] = d/d[mean, white_noise, log_constant,
 * log_alpha, log_M_0..] (george's order); the caller drops frozen entries.  d_y == NULL reuses the alpha of
 * the preceding ab_gp_set_targets / ab_gp_log_likelihood.  alabi/core.py:1261 */
int ab_gp_grad_log_likelihood(ab_gp* h, const double* d_y, double* h_out);

/* K3: gp.predict(y, t, return_var).  d_var may be NULL (mean only).
 * alabi/core.py:85,95,1441,1486,1601 */
int ab_gp_predict(ab_gp* h, const double* d_Xq, int64_t m, double* d_mu, double* d_var);

/* gp.predict(y, t, return_cov=True) (george's default call; the oracle's GP.predict): the
 * predictive mean d_mu (m) and the full predictive covariance
 *   d_cov = K(t, t) - K(t, X) K^-1 K(X, t)     (m x m, leading dimension ldc >= m, white noise not added)
 * from L^-1 by FP64 DMMA products (W = L^-1 K(X, t), then K(t, t) - W^T W on the lower tiles).
 * d_mu has the bits of ab_gp_predict's mean, diag(d_cov) the bits of its variance, d_cov is exactly
 * symmetric, and entry (a, b) depends on queries a and b only (the same bits in any batch).
 * Device workspace: 16 npad m bytes (m rounded up to 256); when it cannot be allocated the call
 * returns -102 (cudaErrorMemoryAllocation) and computes nothing. */
int ab_gp_predict_cov(ab_gp* h, const double* d_Xq, int64_t m, double* d_mu, double* d_cov, int64_t ldc);

/* Draws from N(mean, cov + jitter I), george's GP.sample_conditional / GP.sample (which go through
 * numpy.random.multivariate_normal): d_cov is m x m (leading dimension ldc >= m, lower triangle
 * read, not modified), d_mean m values or NULL (zero mean), d_out nsamples x m (george's (size, M)
 * layout).  cov + jitter I is factorised by the dataflow Cholesky; returns 0, or the 1-based index of
 * the first non-positive pivot (also in *h_info; nothing is written to d_out then).  Normals:
 * Philox4x32-10, key = seed, counter = (row, sample / 2, 0, AB_STREAM_MVN), Box-Muller; draw s
 * depends on column s of the normals only, so the first k draws of any call are the draws of a call
 * with nsamples = k and the same seed. */
int ab_mvn_sample(ab_gp* h, const double* d_cov, int64_t m, int64_t ldc, const double* d_mean /* or NULL */,
                  double jitter, int64_t nsamples, uint64_t seed, double* d_out /* nsamples x m */, int* h_info);

/* gp.predict plus the gradients of mean and variance w.r.t. the query point:
 * d_dmu, d_dvar are m x d row-major.  Replaces grad_gp_mean_prediction /
 * grad_gp_var_prediction (alabi/utility.py:558-621), which difference the kernel
 * numerically (h = 1e-6) and form a dense K^-1 per call; here the kernel derivative
 * is analytic and K^-1 k* is two triangular DMMA GEMMs with L^-1. */
int ab_gp_predict_grad(ab_gp* h, const double* d_Xq, int64_t m, double* d_mu, double* d_var, double* d_dmu,
                       double* d_dvar);
/* same with HOST buffers (pageable or pinned): copies in, predicts, copies out */
int ab_gp_predict_host(ab_gp* h, const double* h_Xq, int64_t m, double* h_mu, double* h_var);

/* K4: bape/agp/jones utility over a candidate batch + argmin over the finite
 * values (lowest index on ties; -1 if none).  h_bounds = d pairs (lo, hi) in
 * the same (scaled) space as the candidates; d_util may be NULL.
 * Replaces the scipy restarts of find_next_point, alabi/core.py:1587-1667. */
int ab_gp_utility_argmin(ab_gp* h, int utility_id, const double* d_Xq, int64_t m, const double* h_bounds,
                         double y_best, double zeta, double* d_util, int64_t* h_argmin, double* h_min);
/* elementwise utility from given mean / variance (no GP evaluation) */
int ab_utility_eval(ab_gp* h, int utility_id, const double* d_Xq, const double* d_mu, const double* d_var,
                    int64_t m, const double* h_bounds, double y_best, double zeta, double* d_util,
                    int64_t* h_argmin, double* h_min);

/* factor / solver state export and import (broadcast L and alpha to other
 * GPUs; gp._alpha, gp.solver.get_inverse() — alabi/utility.py:577-610) */
int64_t ab_gp_padded_size(ab_gp* h);
int ab_gp_get_factor(ab_gp* h, double* d_L /* npad x npad */);
int ab_gp_get_alpha(ab_gp* h, double* d_alpha /* n */);
int ab_gp_get_inverse(ab_gp* h, double* d_Kinv /* n x n, full symmetric */);
int ab_gp_import_state(ab_gp* h, const double* d_L /* npad x npad */, const double* d_alpha /* n */);
/* inverses of the 128 x 128 diagonal blocks of L ((npad/128) x 128 x 128), and an import that
 * adopts them: with L, D^-1 and alpha from the training GPU every replica derives L^-1, K^-1
 * and variances with identical bits (sharded results == single-GPU results) */
int ab_gp_get_block_inverses(ab_gp* h, double* d_Dinv);
int ab_gp_import_state_full(ab_gp* h, const double* d_L, const double* d_Dinv /* or NULL */, const double* d_alpha);

/* K5: emcee.EnsembleSampler(...).run_mcmc over lnprob = surrogate mean + uniform
 * (optionally times independent normal) prior (alabi/core.py:2073-2100, 2319-2325). */
#define AB_MAX_PEERS 15
typedef struct ab_ensemble_config {
    int nwalkers;
    int nsteps;            /* ensemble steps to run in this call */
    int thin_by;           /* store every thin_by-th step (>= 1) */
    int init_logp;         /* 1: evaluate log-prob of d_coords first */
    int randomize_split;   /* 1: coin per walker pair, 0: parity split */
    int warps_per_unit;    /* 0 = auto; 1/2/4/8 = that many warps per unit inside 8-warp CTAs */
    int y_kind;            /* y = ys*y_scale + y_offset (0), -10^ys (1), 10^ys (2) */
    int reserved;          /* must be 0 */
    double a;              /* stretch scale (emcee default 2.0) */
    uint64_t seed;
    int64_t first_step;    /* step counter of the first step (continuing chains) */
    int64_t walker_offset; /* global id of walker 0 (sub-ensembles on other GPUs) */
    double y_scale, y_offset;
    double lo[AB_MAX_DIM_PUBLIC], hi[AB_MAX_DIM_PUBLIC];                    /* prior box, unscaled theta */
    double theta_scale[AB_MAX_DIM_PUBLIC], theta_offset[AB_MAX_DIM_PUBLIC]; /* theta_scaled = theta*scale + offset */
    /* optional independent normal priors on top of the box (ut.lnprior_normal,
     * alabi/utility.py:370-378): use_normal_prior != 0 adds norm.logpdf(theta_k; prior_mu[k],
     * prior_sd[k]) for every k with prior_sd[k] > 0 (prior_sd[k] <= 0: uniform dimension) */
    int use_normal_prior;
    int schedule;          /* small ensembles (2 proposals per unit, training set resident in shared memory):
                            * 0 = dataflow (a proposal waits for its partner's versioned record only; default),
                            * 1 = a grid barrier per half-step.  Identical chains.  3 = as 0, and keep 2-proposal units
                            * even when the training set does not fit shared memory (development: the automatic
                            * choice there is the wide unit with short chunks spread over the GPU) */
    double prior_mu[AB_MAX_DIM_PUBLIC], prior_sd[AB_MAX_DIM_PUBLIC];
    /* Fused all_gather of chain blocks (sub-ensembles sharded over GPUs, SURVEY 8e): the stored rows
     * are written as columns [chain_walker_offset, + nwalkers) of rows of chain_row_walkers walkers
     * (0 = nwalkers: a private block), into d_chain / d_logp_chain AND into the same places of
     * n_chain_peers other buffers (peer memory of the other GPUs, ab_peer_open) by the sampler kernel
     * itself, so the collective costs no launch and no pass over the chain after the run.  The caller
     * synchronises the ranks (all kernels finished) before anybody reads a gathered buffer. */
    int64_t chain_row_walkers;
    int64_t chain_walker_offset;
    int n_chain_peers;     /* 0 .. AB_MAX_PEERS */
    int reserved3;
    void* chain_peers[AB_MAX_PEERS];
    void* logp_chain_peers[AB_MAX_PEERS];
} ab_ensemble_config;

/* d_coords (nwalkers x d) and d_logp (nwalkers) are in/out state; d_naccept is
 * accumulated.  d_chain ((nsteps/thin_by) x nwalkers x d) and d_logp_chain may
 * be NULL, as may the proposal record d_rec_q (nsteps x nwalkers x d) /
 * d_rec_lp (nsteps x nwalkers) used by the parity tests. */
int ab_ensemble_run(ab_gp* h, const ab_ensemble_config* cfg, double* d_coords, double* d_logp,
                    long long* d_naccept, double* d_chain, double* d_logp_chain, double* d_rec_q,
                    double* d_rec_lp);
/* The same run in two calls: ab_ensemble_launch enqueues the whole chain on the handle's stream
 * and returns; ab_ensemble_finish waits for it and returns 0, or 1 when a log-probability was NaN
 * (emcee raises ValueError there).  Between the two the host is free, e.g. to page-lock the
 * buffers the chain is copied into.  One run in flight per handle. */
int ab_ensemble_launch(ab_gp* h, const ab_ensemble_config* cfg, double* d_coords, double* d_logp,
                       long long* d_naccept, double* d_chain, double* d_logp_chain, double* d_rec_q,
                       double* d_rec_lp);
int ab_ensemble_finish(ab_gp* h);
/* The same run with the stored chain delivered to HOST buffers (what emcee's backend holds after
 * run_mcmc, alabi/core.py:2325 -> sampler.get_chain()): the run is cut into `nblocks` consecutive
 * pieces (identical chain: the random streams are counter based) that are enqueued back to back;
 * the stored rows of piece b travel to h_chain ((nsteps/thin_by) x nwalkers x d) and h_logp_chain
 * on the handle's second stream while piece b + 1 runs.  d_chain / d_logp_chain are device staging
 * of the same shapes.  Host buffers may be page-locked (asynchronous copies) or pageable.
 * Returns 0, 1 (NaN log-probability) or < 0. */
int ab_ensemble_run_host(ab_gp* h, const ab_ensemble_config* cfg, double* d_coords, double* d_logp,
                         long long* d_naccept, double* d_chain, double* d_logp_chain, double* h_chain,
                         double* h_logp_chain, int nblocks);

/* Nested sampling on the surrogate: a batch of constrained random walks in the unit cube
 * (dynesty's sample="rwalk" replacement step; the reference passes surrogate_log_likelihood and a
 * prior transform to dynesty.(Dynamic)NestedSampler, alabi/core.py:2549-2706).  Chain c starts at
 * d_u[c] (unit cube) with log-likelihood d_logl[c] and makes `walks` Metropolis steps
 * u' = u + scale * chol z, z ~ N(0, I); u' is accepted iff it lies inside (0, 1)^d and the surrogate
 * mean at prior_transform(u') exceeds lmin.  Prior transform: (hi - lo) u + lo per dimension
 * (ut.prior_transform_uniform), or mu + sd * ndtri(u) where use_normal_prior != 0 and
 * prior_sd[k] > 0 (ut.prior_transform_normal).  Random numbers: Philox4x32-10, key = seed,
 * counter = (chain_offset + c, step, pair of dimensions, counter).  On return d_u / d_logl hold
 * the end points, d_theta (nchains x d) their images under the prior transform (rows of chains
 * that never moved are left untouched) and d_naccept the accepted steps per chain. */
typedef struct ab_nested_config {
    int nchains;
    int walks;
    int y_kind;            /* as in ab_ensemble_config */
    int use_normal_prior;
    double scale;
    double lmin;
    uint64_t seed;
    int64_t counter;
    int64_t chain_offset;
    double y_scale, y_offset;
    double lo[AB_MAX_DIM_PUBLIC], hi[AB_MAX_DIM_PUBLIC];
    double prior_mu[AB_MAX_DIM_PUBLIC], prior_sd[AB_MAX_DIM_PUBLIC];
    double theta_scale[AB_MAX_DIM_PUBLIC], theta_offset[AB_MAX_DIM_PUBLIC];
    double chol[AB_MAX_DIM_PUBLIC * AB_MAX_DIM_PUBLIC];   /* d x d, row-major, lower triangular */
} ab_nested_config;
int ab_sizeof_nested_config(void);
int ab_nested_walk(ab_gp* h, const ab_nested_config* cfg, double* d_u, double* d_logl, double* d_theta,
                   int* d_naccept);
/* The same replacement step by random-direction slice sampling (dynesty's sample="rslice"), with
 * the same configuration, argument checks and return codes; cfg->walks is the number of slices.
 * Slice s of chain c (F(x) = surrogate mean at prior_transform(u + x v) inside (0, 1)^d, -inf and
 * no evaluation outside):
 *   direction  z as the walk's normals at step = s; v = (chol z) * (scale / |z|)
 *   window     r0 = u53(words 0, 1) of Philox block j0 = ceil(d / 2), counter
 *              (chain_offset + c, s, j0, counter); x_l = -r0, x_r = 1 - r0
 *   step out   while F(x_l) > lmin: x_l -= 1; then while F(x_r) > lmin: x_r += 1 (one nexpand each)
 *   shrink     draw i = 0, 1, ...: x = x_l + u_i (x_r - x_l), u_i = u53(words 0, 1) of block
 *              j0 + 1 + i; F(x) > lmin accepts u <- u + x v, otherwise x_l = x (x < 0) or
 *              x_r = x (x > 0) (one ncontract)
 * Window and point arithmetic is rounded operation by operation (no fused multiply-add).  Caps:
 * a slice that needs more than 1024 expansions or more than 256 contractions ends its chain at the
 * end point of the last completed slice, so every launch ends.  On return d_u / d_logl / d_theta are as for ab_nested_walk and d_counts (nchains x 4)
 * holds per chain: slices completed (< walks for a chain stopped by a cap), nexpand, ncontract and
 * surrogate evaluations.  A chain's result does not depend on the other chains of the batch. */
int ab_nested_rslice(ab_gp* h, const ab_nested_config* cfg, double* d_u, double* d_logl, double* d_theta,
                     int* d_counts);

/* ---- NCCL helpers (SURVEY 8b / 8e): one process per GPU; the factor is trained once and
 *      broadcast over NVLink, argmin records and chain blocks are all_gathered.  The reference has
 *      no counterpart (its parallelism is multiprocessing pools, alabi/core.py:309-314).  NCCL is
 *      resolved at run time (dlopen of libnccl.so.2, e.g. the copy PyTorch already loaded); without
 *      it the calls return -6.  A communicator is bound to one device and one stream; calls are
 *      asynchronous on that stream except where stated. ---- */
#define AB_NCCL_ID_BYTES 128
typedef struct ab_comm ab_comm;
int ab_nccl_unique_id(unsigned char* h_id /* AB_NCCL_ID_BYTES, made on one rank and handed to all */);
int ab_nccl_init(ab_comm** out, int world, int rank, const unsigned char* h_id, int device, void* cuda_stream);
int ab_nccl_destroy(ab_comm* c);
int ab_nccl_sync(ab_comm* c);                                         /* waits for the communicator's stream */
int ab_nccl_broadcast(ab_comm* c, void* d_buf, int64_t nbytes, int root);
int ab_nccl_allgather(ab_comm* c, const void* d_send, void* d_recv /* world x nbytes_per_rank */, int64_t nbytes_per_rank);
/* factor state (L, diagonal-block inverses, log-determinant parts, alpha) of the trained handle of
 * rank `root` into the handles of all ranks, in place, no staging copies; every rank must have set
 * the same inputs and hyper-parameters (ab_gp_set_inputs / ab_gp_set_kernel).  Returns after the
 * transfer has completed. */
int ab_nccl_broadcast_gp(ab_comm* c, ab_gp* h, int root);

/* Peer memory between the processes of one box (one process per GPU): a device buffer that the
 * sampler kernels of the other ranks write their chain blocks into (ab_ensemble_config.chain_peers).
 * ab_peer_alloc allocates it (cudaMalloc) and fills the 64-byte handle that travels to the other
 * processes by any host channel; ab_peer_open maps another rank's buffer into this process (CUDA IPC,
 * peer access over NVLink / NVSwitch enabled on first use); ab_peer_close unmaps it, ab_peer_free
 * releases the owner's allocation (after every rank has closed it). */
#define AB_PEER_HANDLE_BYTES 64
int ab_peer_alloc(int device, size_t bytes, void** d_ptr, unsigned char* h_handle);
int ab_peer_open(int device, const unsigned char* h_handle, void** d_ptr);
int ab_peer_close(int device, void* d_ptr);
int ab_peer_free(int device, void* d_ptr);

/* k-fold cross-validation of hyper-parameter candidates as one batched job
 * (gp_utils.optimize_gp_kfold_cv and its per-candidate worker, alabi/gp_utils.py:511-637, 640-1231;
 * the default hyper-parameter search of init_gp, alabi/core.py:751).  Job b = (candidate
 * h_job_cand[b], one fold): the GP with that candidate's hyper-parameters is factorised on the
 * rows d_train_idx[b][0 .. h_ntrain[b]) of X (n x d, device), the log-likelihood of y on those rows
 * goes to h_loglik[b], the predictive mean at the rows d_val_idx[b][0 .. h_nval[b]) to
 * d_pred[b][...] (leading dimensions ld_train / ld_val), and h_status[b] is 0 or the 1-based index
 * of the first non-positive pivot (the reference scores such a fold as failed).  h_params holds,
 * per candidate, 3 + d doubles: mean, white_noise (ln variance), amp = exp(log_constant), log_M[d];
 * for kernel_id AB_KERNEL_RATQUAD 4 + d doubles: mean, white_noise, amp, log_alpha, log_M[d].
 * All jobs of a call are factorised by ONE batched dataflow-Cholesky launch per workspace chunk:
 * d_work / work_bytes is caller-owned device scratch (ab_gp_cv_workspace_bytes gives the size that
 * takes all jobs in one launch; anything from one job's worth upwards works with more launches).
 * The handle supplies device, stream and nothing else: its own model state is not touched. */
int ab_gp_cv_batch(ab_gp* h, const double* d_X, const double* d_y, int64_t n, int d, int kernel_id, int ncand,
                   const double* h_params, int njobs, const int* h_job_cand, const int* h_ntrain,
                   const int* h_nval, const int* d_train_idx, int ld_train, const int* d_val_idx, int ld_val,
                   double* d_pred, double* h_loglik, int* h_status, void* d_work, size_t work_bytes);
size_t ab_gp_cv_workspace_bytes(int ntrain_max, int d, int ld_val, int ncand, int njobs);

#ifdef __cplusplus
}
#endif
#endif
