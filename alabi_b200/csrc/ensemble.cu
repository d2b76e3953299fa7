// K5: emcee-compatible ensemble stretch-move sampler, fully on device.
//
// Replaces emcee.EnsembleSampler.run_mcmc over SurrogateModel.lnprob
// (alabi/core.py:2073-2100, 2319-2325): the red/blue stretch move, every
// walker's surrogate log-probability (uniform prior box + GP predictive mean,
// K3 mean-only) and the accept/reject step run inside ONE persistent
// cooperative kernel; the two dependent half-updates of a step are separated
// by a grid barrier, never by a host round trip.
//
// Work decomposition: small ensembles use "units" of 1, 2, 4 or 8 warps that evaluate
// P = 2 proposals at a time, lanes striding over the training points; large
// ensembles use the wide unit (P = 32: one lane per proposal, the warps of a CTA split
// the training points and read them as shared-memory broadcasts).  Training points are
// SoA in shared memory, resident for the whole run when they fit, else streamed in
// double-buffered cp.async chunks; proposals sit in registers.
//
// Random numbers: Philox4x32-10 keyed by the seed, counter = (global walker id,
// step, stream, 0) — restated on the CPU in oracle/philox.py so a device chain
// can be replayed exactly.  The red/blue split flips one fair coin per walker
// pair (2i, 2i+1): balanced, position independent, no compaction needed.
//
// This file: the C entry points; the kernel lives in ensemble_kernel.cuh (instantiated per kernel
// family by ensemble_k0 / k1 / k2.cu).
#include <cmath>
#include <vector>
#include "ensemble_args.h"

// Enqueue one sampler kernel on the handle's stream.  `first`: clear the barrier counter and the
// NaN flag; later pieces of the same run clear the barrier counter only.
static int ens_enqueue(ab_gp* h, const ab_ensemble_config* cfg, double* d_coords, double* d_logp,
                       long long* d_naccept, double* d_chain, double* d_logp_chain, double* d_rec_q,
                       double* d_rec_lp, bool first) {
    if (!h->have_alpha) { ab_set_error("ab_ensemble_run: targets not set (call ab_gp_set_targets)"); return -2; }
    if (cfg->nwalkers < 2 || cfg->nsteps < 0 || cfg->thin_by < 1) { ab_set_error("bad ensemble configuration"); return -1; }
    if (cfg->reserved != 0) { ab_set_error("ab_ensemble_run: ab_ensemble_config.reserved must be 0"); return -1; }
    // scratch: [0, 4096) barrier word and NaN flag; then the completion counters and the
    // segment sums of split wide units (3 kinds of half-step x units x AB_ENS_MAXSEG segments x 32 proposals)
    const int max_units = (cfg->nwalkers + 31) / 32;
    const size_t cnt_bytes = ((size_t)3 * max_units * sizeof(unsigned) + 255) / 256 * 256;
    // proposals per half-step
    int n_half = (cfg->nwalkers + 1) / 2;
    if (cfg->init_logp && cfg->nsteps == 0) n_half = cfg->nwalkers;
    const int nsm = h->nsm;
    // proposals per unit: 2 (small ensembles, many units), 32 = one lane per proposal once
    // there are enough proposals for one 32-wide unit per SM
    int p = (n_half >= 16 * nsm) ? 32 : 2;
    // dataflow schedule (ab_ensemble_config.schedule 0 = automatic, 1 = grid barriers): small ensembles
    // whose half-steps are latency bound; the launcher drops it when the training set is not resident
    const bool resident_small = ab_resident(h->n, ab_padded_dim(h->d));
    // Small ensemble on a training set that does not fit shared memory (emcee's default 10 x ndim walkers on
    // an N = 8192 surrogate): a 2-proposal unit would stream all N points through ONE CTA per half-step
    // (86 us per step at N = 8192, d = 10, whatever the walker count).  "Spread" mode runs the wide unit
    // instead with SHORT chunks, so that the (unit, chunk) pairs of a half-step cover the GPU: every CTA
    // evaluates 32 proposals against 128-512 points, the segment sums meet in global memory and the CTA
    // that delivers a unit's last segment accepts (the ranged schedule of the large ensembles).
    int ch_hint = 0, maxseg = AB_ENS_MAXSEG;
    if (p == 2 && !resident_small && cfg->schedule != 3) {
        p = 32;
        const long long units = (n_half + 31) / 32;
        ch_hint = 128;
        for (int c = 512; c >= 128; c /= 2)
            if (h->npad % c == 0 && units * (h->npad / c) >= 2LL * nsm) { ch_hint = c; break; }
        maxseg = (int)(h->npad / ch_hint) + 2;
        if (maxseg < AB_ENS_MAXSEG) maxseg = AB_ENS_MAXSEG;
    }
    const size_t part_bytes = (size_t)3 * max_units * maxseg * 32 * sizeof(double);
    const bool flow = p == 2 && cfg->schedule != 1 && cfg->nsteps > 0 && resident_small;
    const size_t ring_bytes = flow ? (size_t)AB_ENS_RING * cfg->nwalkers * h->d * sizeof(uint4) : 0;
    int rc = ab_ensure_scratch(h, 4096 + cnt_bytes + part_bytes + ring_bytes);
    if (rc) return rc;
    EnsArgs A{};
    if (flow) {
        A.ring = reinterpret_cast<uint4*>(reinterpret_cast<char*>(h->scratch) + 4096 + cnt_bytes + part_bytes);
        AB_CUDA(cudaMemsetAsync(A.ring, 0, ring_bytes, h->stream));
    }
    A.max_units = max_units;
    A.maxseg = maxseg;
    A.ch_hint = ch_hint;
    A.slice_cnt = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(h->scratch) + 4096);
    A.slice_part = reinterpret_cast<double*>(reinterpret_cast<char*>(h->scratch) + 4096 + cnt_bytes);
    if (first) AB_CUDA(cudaMemsetAsync(A.slice_cnt, 0, cnt_bytes, h->stream));
    A.coords = d_coords; A.logp = d_logp; A.naccept = d_naccept;
    A.chain = d_chain; A.logp_chain = d_logp_chain; A.rec_q = d_rec_q; A.rec_lp = d_rec_lp;
    if (cfg->n_chain_peers < 0 || cfg->n_chain_peers > AB_MAX_PEERS || cfg->chain_row_walkers < 0 || cfg->chain_walker_offset < 0 ||
        (cfg->chain_row_walkers > 0 && cfg->chain_walker_offset + cfg->nwalkers > cfg->chain_row_walkers) ||
        (cfg->chain_row_walkers == 0 && (cfg->chain_walker_offset != 0 || cfg->n_chain_peers != 0))) {
        ab_set_error("ab_ensemble_run: bad chain layout (chain_row_walkers / chain_walker_offset / n_chain_peers)"); return -1;
    }
    A.chain_ld = cfg->chain_row_walkers > 0 ? cfg->chain_row_walkers : cfg->nwalkers;
    A.chain_off = cfg->chain_walker_offset;
    A.n_dst = d_chain ? 1 + cfg->n_chain_peers : 0;
    A.chain_dst[0] = d_chain; A.logp_dst[0] = d_logp_chain;
    for (int q = 0; q < cfg->n_chain_peers; q++) {
        if (!cfg->chain_peers[q] || !cfg->logp_chain_peers[q]) { ab_set_error("ab_ensemble_run: null peer buffer"); return -1; }
        A.chain_dst[1 + q] = static_cast<double*>(cfg->chain_peers[q]);
        A.logp_dst[1 + q] = static_cast<double*>(cfg->logp_chain_peers[q]);
    }
    A.chain_vec = (h->d % 2 == 0) ? 1 : 0;
    for (int q = 0; q < A.n_dst; q++)
        if (reinterpret_cast<uintptr_t>(A.chain_dst[q]) & 15) A.chain_vec = 0;
    A.barrier = reinterpret_cast<unsigned long long*>(h->scratch);
    A.nan_flag = reinterpret_cast<int*>(h->scratch + 1);
    AB_CUDA(cudaMemsetAsync(h->scratch, 0, first ? 16 : 8, h->stream));
    A.XsT = h->XsT; A.alpha = h->alpha; A.n = h->n; A.npad = h->npad; A.kp = h->kp; A.mean = h->mean;
    A.nwalkers = cfg->nwalkers; A.d = h->d; A.nsteps = cfg->nsteps; A.thin_by = cfg->thin_by;
    A.init_logp = cfg->init_logp; A.randomize_split = cfg->randomize_split; A.a = cfg->a;
    A.seed_lo = (unsigned)(cfg->seed & 0xffffffffULL); A.seed_hi = (unsigned)(cfg->seed >> 32);
    A.first_step = cfg->first_step; A.walker_offset = cfg->walker_offset;
    for (int k = 0; k < h->d; k++) {
        A.lo[k] = cfg->lo[k]; A.hi[k] = cfg->hi[k];
        A.t_scale[k] = cfg->theta_scale[k]; A.t_off[k] = cfg->theta_offset[k];
    }
    A.y_kind = cfg->y_kind; A.y_scale = cfg->y_scale; A.y_off = cfg->y_offset;
    A.use_normal = 0;
    if (cfg->use_normal_prior) {
        for (int k = 0; k < h->d; k++) {
            A.pr_mu[k] = cfg->prior_mu[k]; A.pr_sd[k] = cfg->prior_sd[k];
            if (cfg->prior_sd[k] > 0.0) {
                if (!std::isfinite(cfg->prior_mu[k]) || !std::isfinite(cfg->prior_sd[k])) {
                    ab_set_error("ab_ensemble_run: non-finite normal prior"); return -1;
                }
                A.pr_lsd[k] = std::log(cfg->prior_sd[k]);
                A.use_normal = 1;
            }
        }
    }
    // warps per unit: all 8 warps on one unit while that still fills the GPU
    const int units_half = (n_half + p - 1) / p;
    int ws = 1;
    if (p == 32) ws = 16;                      // wide unit = the whole CTA (16 warps)
    else if (cfg->warps_per_unit > 0) ws = cfg->warps_per_unit;
    else while (ws < 8 && units_half * ws * 2 <= nsm * 8) ws *= 2;   // the half-step in ONE pass of one 8-warp CTA per SM
    if (ws != 1 && ws != 2 && ws != 4 && ws != 8 && !(p == 32 && ws == 16)) { ab_set_error("warps_per_unit must be 0, 1, 2, 4 or 8"); return -1; }
    A.ws = ws;
    // 4-warp CTAs (one unit each, several per SM) when 8-warp CTAs would run several units in lockstep
    // and every unit still gets a co-resident CTA
    const bool small_cta = p == 2 && cfg->warps_per_unit == 0 && ws < 8;
    rc = (h->kp.kind == 0) ? ab_ens_launch_k0(h, A, n_half, p, small_cta, ws)
       : (h->kp.kind == 1) ? ab_ens_launch_k1(h, A, n_half, p, small_cta, ws)
       : (h->kp.kind == 2) ? ab_ens_launch_k2(h, A, n_half, p, small_cta, ws)
                           : ab_ens_launch_k3(h, A, n_half, p, small_cta, ws);
    return rc;
}

extern "C" int ab_ensemble_launch(ab_gp* h, const ab_ensemble_config* cfg, double* d_coords, double* d_logp,
                                  long long* d_naccept, double* d_chain, double* d_logp_chain, double* d_rec_q,
                                  double* d_rec_lp) {
    if (!h || !cfg) { ab_set_error("null argument"); return -1; }
    if (h->ens_pending) { ab_set_error("ab_ensemble_launch: the previous run was not finished (ab_ensemble_finish)"); return -1; }
    AB_CUDA(cudaSetDevice(h->device));
    int rc = ens_enqueue(h, cfg, d_coords, d_logp, d_naccept, d_chain, d_logp_chain, d_rec_q, d_rec_lp, true);
    if (rc) return rc;
    AB_CUDA(cudaMemcpyAsync(h->h_pinned, h->scratch, 16, cudaMemcpyDeviceToHost, h->stream));
    h->ens_pending = true;
    return 0;
}

// The same chain delivered to HOST buffers.  The run is cut into `nblocks` consecutive pieces
// (the random streams are counter based, so the chain does not depend on the cut); every piece is
// enqueued at once on the handle's stream, and the stored rows of piece b travel to the host on
// the handle's second stream while piece b + 1 runs.  h_chain / h_logp_chain may be page-locked
// (the copies are then asynchronous) or pageable.
extern "C" int ab_ensemble_run_host(ab_gp* h, const ab_ensemble_config* cfg, double* d_coords, double* d_logp,
                                    long long* d_naccept, double* d_chain, double* d_logp_chain, double* h_chain,
                                    double* h_logp_chain, int nblocks) {
    if (!h || !cfg || !d_chain || !d_logp_chain || !h_chain || !h_logp_chain) { ab_set_error("null argument"); return -1; }
    if (h->ens_pending) { ab_set_error("ab_ensemble_run_host: the previous run was not finished (ab_ensemble_finish)"); return -1; }
    if (cfg->thin_by < 1 || cfg->nsteps < 0 || cfg->nsteps % cfg->thin_by != 0) {
        ab_set_error("ab_ensemble_run_host: nsteps must be a multiple of thin_by"); return -1;
    }
    if (cfg->chain_row_walkers != 0 || cfg->n_chain_peers != 0) {
        ab_set_error("ab_ensemble_run_host: gathered chain layouts go through ab_ensemble_launch"); return -1;
    }
    AB_CUDA(cudaSetDevice(h->device));
    const long long rows = cfg->nsteps / cfg->thin_by, nw = cfg->nwalkers, d = h->d;
    if (nblocks < 1) nblocks = 1;
    if (nblocks > 64) nblocks = 64;
    if ((long long)nblocks > rows) nblocks = rows > 0 ? (int)rows : 1;
    const long long rpb = rows > 0 ? (rows + nblocks - 1) / nblocks : 0;
    std::vector<cudaEvent_t> evs;
    int rc = 0;
    bool first = true;
    long long done = 0;
    struct Piece { long long row0, nrows; };
    std::vector<Piece> pieces;
    do {
        const long long nr = (rows - done < rpb) ? (rows - done) : rpb;
        ab_ensemble_config c = *cfg;
        c.nsteps = (int)(nr * cfg->thin_by);
        c.first_step = cfg->first_step + done * cfg->thin_by;
        c.init_logp = first ? cfg->init_logp : 0;
        rc = ens_enqueue(h, &c, d_coords, d_logp, d_naccept, d_chain + done * nw * d, d_logp_chain + done * nw, nullptr,
                         nullptr, first);
        if (rc) break;
        cudaEvent_t e;
        if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) { ab_set_error("cudaEventCreate failed"); rc = -100; break; }
        cudaEventRecord(e, h->stream);
        evs.push_back(e);
        pieces.push_back({done, nr});
        done += nr;
        first = false;
    } while (done < rows);
    if (!rc) {
        cudaMemcpyAsync(h->h_pinned, h->scratch, 16, cudaMemcpyDeviceToHost, h->stream);
        for (size_t b = 0; b < pieces.size() && !rc; b++) {
            const Piece& p = pieces[b];
            cudaError_t e = cudaStreamWaitEvent(h->copy_stream, evs[b], 0);
            if (e == cudaSuccess && p.nrows > 0) {
                e = cudaMemcpyAsync(h_chain + p.row0 * nw * d, d_chain + p.row0 * nw * d, (size_t)(p.nrows * nw * d) * sizeof(double),
                                    cudaMemcpyDeviceToHost, h->copy_stream);
                if (e == cudaSuccess)
                    e = cudaMemcpyAsync(h_logp_chain + p.row0 * nw, d_logp_chain + p.row0 * nw, (size_t)(p.nrows * nw) * sizeof(double),
                                        cudaMemcpyDeviceToHost, h->copy_stream);
            }
            if (e != cudaSuccess) { ab_set_error("ab_ensemble_run_host: copy failed: %s", cudaGetErrorString(e)); rc = -100 - (int)e; }
        }
    }
    cudaStreamSynchronize(h->copy_stream);
    cudaError_t es = cudaStreamSynchronize(h->stream);
    for (cudaEvent_t e : evs) cudaEventDestroy(e);
    if (rc) return rc;
    if (es != cudaSuccess) { ab_set_error("ab_ensemble_run_host: %s", cudaGetErrorString(es)); return -100 - (int)es; }
    if (reinterpret_cast<int*>(h->h_pinned + 1)[0] == 2) {
        ab_set_error("ensemble sampler: a partner record did not arrive within the watchdog time (dataflow schedule); "
                     "the chain of this run is invalid");
        return -7;
    }
    if (reinterpret_cast<int*>(h->h_pinned + 1)[0] != 0) {
        ab_set_error("Probability function returned NaN");
        return 1;
    }
    return 0;
}

extern "C" int ab_ensemble_finish(ab_gp* h) {
    if (!h) { ab_set_error("null argument"); return -1; }
    if (!h->ens_pending) { ab_set_error("ab_ensemble_finish: no run was launched"); return -1; }
    h->ens_pending = false;
    AB_CUDA(cudaSetDevice(h->device));
    AB_CUDA(cudaStreamSynchronize(h->stream));
    if (reinterpret_cast<int*>(h->h_pinned + 1)[0] == 2) {
        ab_set_error("ensemble sampler: a partner record did not arrive within the watchdog time (dataflow schedule); "
                     "the chain of this run is invalid");
        return -7;
    }
    if (reinterpret_cast<int*>(h->h_pinned + 1)[0] != 0) {
        ab_set_error("Probability function returned NaN");
        return 1;
    }
    return 0;
}

extern "C" int ab_ensemble_run(ab_gp* h, const ab_ensemble_config* cfg, double* d_coords, double* d_logp,
                               long long* d_naccept, double* d_chain, double* d_logp_chain, double* d_rec_q,
                               double* d_rec_lp) {
    int rc = ab_ensemble_launch(h, cfg, d_coords, d_logp, d_naccept, d_chain, d_logp_chain, d_rec_q, d_rec_lp);
    if (rc) return rc;
    return ab_ensemble_finish(h);
}
