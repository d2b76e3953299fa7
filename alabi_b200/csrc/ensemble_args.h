// Arguments of the ensemble sampler kernel, shared by the translation units that instantiate the
// kernel (ensemble_k0 / k1 / k2.cu: one kernel family each, compiled in parallel) and ensemble.cu,
// which fills them from ab_ensemble_config and owns the C entry points.
#pragma once
#include "handle.h"
#include "alabi_b200.h"

#define AB_ENS_RING 32             // versions of a walker's position the dataflow schedule keeps
#define AB_ENS_THROTTLE 15         // steps between its (non-blocking) progress barriers: 2 * 15 + 1 <= 32
#define AB_ENS_MAXSEG 64           // segments a streamed wide unit may be cut into (ranged schedule)

struct EnsArgs {
    // state and outputs
    double* coords; double* logp; long long* naccept;
    double* chain; double* logp_chain; double* rec_q; double* rec_lp;
    unsigned long long* barrier; int* nan_flag;
    // surrogate
    const double* XsT; const double* alpha; long long n, npad;
    KernParams kp; double mean;
    // sampler configuration
    int nwalkers, d, nsteps, thin_by, init_logp, randomize_split, ws, ch;
    // streamed wide unit, `ranged` != 0: the work of a half-step is the list of (unit, chunk of
    // training points) pairs, cut into equal CONTIGUOUS ranges, one per CTA, so every SM carries the
    // same load whatever the number of units (128 units on 148 SMs would leave 14 % idle).  A unit
    // whose chunks fall into several ranges is finished by the CTA that delivers its last segment:
    // segment sums meet in slice_part (fixed segment order), completions are counted in slice_cnt.
    int ranged, max_units;
    int maxseg;                   // segments per unit the slice_part layout provides for
    int ch_hint;                  // > 0 ("spread" mode, small ensembles on a large training set): chunk length to use, ranged
    double* slice_part; unsigned* slice_cnt;
    // stored rows: walker w of stored row r sits at r * chain_ld + chain_off + w of chain_dst[0] (= chain)
    // and of the n_dst - 1 peer buffers behind it (fused all_gather of chain blocks)
    long long chain_ld, chain_off;
    int n_dst, chain_vec;         // chain_vec: d is even and every destination is 16-byte aligned (double2 row stores)
    double* chain_dst[AB_MAX_PEERS + 1]; double* logp_dst[AB_MAX_PEERS + 1];
    // dataflow schedule (FLOW kernels): ring of AB_ENS_RING versions of every walker's position,
    // one 16-byte line {lo, flag, hi, flag} per coordinate, flag = version + 1 (0 = never written)
    uint4* ring;
    double a;
    unsigned seed_lo, seed_hi;
    long long first_step, walker_offset;
    double lo[AB_MAX_DIM], hi[AB_MAX_DIM], t_scale[AB_MAX_DIM], t_off[AB_MAX_DIM];
    int y_kind; double y_scale, y_off;
    // independent normal priors (use_normal: any; pr_sd[k] <= 0: dimension k is uniform);
    // pr_c[k] = log sqrt(2 pi) + log sd, the constant of norm.logpdf
    int use_normal;
    double pr_mu[AB_MAX_DIM], pr_sd[AB_MAX_DIM], pr_lsd[AB_MAX_DIM];
};

// one per kernel family (KIND = 0 ExpSquared, 1 Matern-3/2, 2 Matern-5/2): picks the padded dimension
// and the unit shape, launches on the handle's stream.  Defined in ensemble_k<KIND>.cu.
int ab_ens_launch_k0(ab_gp* h, EnsArgs& A, int n_half, int p, bool small_cta, int ws);
int ab_ens_launch_k1(ab_gp* h, EnsArgs& A, int n_half, int p, bool small_cta, int ws);
int ab_ens_launch_k2(ab_gp* h, EnsArgs& A, int n_half, int p, bool small_cta, int ws);
int ab_ens_launch_k3(ab_gp* h, EnsArgs& A, int n_half, int p, bool small_cta, int ws);
