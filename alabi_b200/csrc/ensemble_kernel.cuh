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
// This header holds the kernel and its launchers; ensemble_k0 / k1 / k2.cu instantiate one kernel
// family each (so the three compile in parallel), ensemble.cu holds the C entry points.
#pragma once
#include <stdio.h>
#include <cmath>
#include <vector>
#include "ensemble_args.h"

namespace {

constexpr int kWideUnroll = 2;    // point pairs per iteration of the wide unit's inner loop (1 and 4 measured: profiles/r02b_sampler_unroll_variants.txt)

// warps per CTA (EW): 8; 16 was measured slower on the c2 workload (longer proposal and compute phases)


struct U4 { unsigned x, y, z, w; };

__device__ __forceinline__ U4 philox4x32_10(unsigned c0, unsigned c1, unsigned c2, unsigned c3, unsigned k0, unsigned k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return U4{c0, c1, c2, c3};
}
__device__ __forceinline__ double u53(unsigned hi, unsigned lo) {
    return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6)) / 9007199254740992.0;
}

// walker of pair i that belongs to set s at this step
__device__ __forceinline__ int member_of(const EnsArgs& A, int i, int s, unsigned step_lo) {
    int bit = 0;
    if (A.randomize_split && 2 * i + 1 < A.nwalkers)
        bit = philox4x32_10((unsigned)(A.walker_offset + 2 * i), step_lo, AB_STREAM_SPLIT, 0, A.seed_lo, A.seed_hi).x & 1u;
    return 2 * i + (bit ^ s);
}

// grid barrier split in two: arrive as soon as this CTA's updates are published,
// wait only when the next half-step needs the other CTAs' updates.  Release / acquire
// on the counter itself orders the walker updates (no separate fences).
template <class Sync>
__device__ __forceinline__ void grid_arrive(unsigned long long* counter, unsigned long long& target, Sync csync) {
    csync();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        asm volatile("red.release.gpu.global.add.u64 [%0], %1;" ::"l"(counter), "l"(1ULL) : "memory");
    }
}
template <class Sync>
__device__ __forceinline__ void grid_wait(unsigned long long* counter, unsigned long long target, Sync csync) {
    if (threadIdx.x == 0) {
        unsigned long long v;
        do {
            asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(counter) : "memory");
        } while (v < target);
    }
    csync();
}

// CHT > 0: the chunk length is a compile-time constant (the streamed wide unit at 512 points per
// chunk): the shared-memory row addresses bX[k * CH + j] of the inner loop become immediate offsets
// instead of one integer multiply-add per dimension and point pair.  CHT = 0: run-time A.ch.
//
// FLOW (small ensembles, resident training set): the grid barrier between half-steps is replaced
// by dataflow on the one remote input of a proposal, its partner's position.  The pair (2i, 2i+1)
// is always updated by the same lanes of the same CTA, so a walker's own state is ordered by
// program order; the partner is read from a ring of versioned records that the updating lane
// publishes with its accept decision: one 16-byte line {lo, flag, hi, flag} per coordinate
// (8-byte halves are single-copy atomic, so a line whose two flags carry the wanted version holds
// that version's value: the data IS the signal, one L2 round trip instead of counter + poll +
// load).  Version v of walker w (its position after v steps) lives in slot v mod AB_ENS_RING; a
// half-step (t, 0) reads version t of its partner, (t, 1) version t + 1 -- exactly the positions
// the barrier schedule reads, so the chain has identical bits.  A progress barrier every
// AB_ENS_THROTTLE steps, arrived at once and waited for one period later, keeps any two CTAs less
// than 2 * AB_ENS_THROTTLE steps apart, so a slot is never overwritten while a reader needs it.
//
// Small units (P = 2) carry one extra warp, the PREP warp: it draws the random-stream part
// (walker, partner, stretch factor, accept threshold: three Philox blocks and two logarithms, ~1 us
// as a serial chain) of the CTA's work items TWO items ahead of the EW compute warps, into a ring of
// three buffers, so that chain never sits between a half-step's accept and the next gather and has a
// whole item period to finish, however short the kernel evaluations are.  The compute warps
// synchronise among themselves on named barrier 1; barrier 2 (all warps) opens every work item: the
// prep warp arrives there with the item's buffer filled.
template <int KIND, int D, int EW, int P, int CHT = 0, bool FLOW = false>
__global__ void __launch_bounds__(EW * 32 + (P == 32 ? 0 : 32), ((P == 32 && EW == 8) || EW == 4) ? 2 : 1)
ensemble_kernel(const __grid_constant__ EnsArgs A) {
    constexpr int ETHREADS = EW * 32;               // compute threads
    constexpr bool PW = (P != 32);                  // prep warp present (warp EW)
    constexpr int ATHREADS = ETHREADS + (PW ? 32 : 0);
    extern __shared__ __align__(16) double sm[];
    const int CH = CHT > 0 ? CHT : A.ch;
    double* sX = sm;                 // [D][CH]
    double* sAl = sm + D * CH;       // [CH]
    // P proposals per unit (2: small ensembles, more units)
    // P = 32 ("wide"): ONE unit per CTA whose proposal e belongs to LANE e of every warp; the
    // eight warps split the training points and read them as shared-memory broadcasts, so
    // there is no cross-lane reduction and the proposal / accept phases use all 32 lanes.
    constexpr bool WIDE = (P == 32);
    constexpr int NU = WIDE ? 1 : EW;            // units per CTA the per-unit arrays must hold
    __shared__ double sQ[NU][P][D], sQs[NU][P][D];
    __shared__ double sS[NU][P][D];              // current position of the walker being updated
    constexpr int NPB = PW ? 3 : 1;               // prep buffers
    __shared__ double sPart[EW][P], sLogZ[NPB][NU][P], sLogU[NPB][NU][P], sLps[NU][P], sZZ[NPB][NU][P];
    __shared__ int sW[NPB][NU][P], sInside[NU][P], sPartner[NPB][NU][P];
    __shared__ double sPrior[NU][P];             // ln of the normal part of the prior at the proposal
    __shared__ int sSliceLast;                   // split units: this CTA delivered the last slice of its unit
    __shared__ int sOut[WIDE ? P : 1];           // wide unit: proposal left the prior box (cooperative gather)
    __shared__ int sAccF[WIDE ? P : 1];          // wide unit: accept flags and stored log-probabilities of the unit,
    __shared__ double sLpOut[WIDE ? P : 1];      // handed from the proposal lanes to the cooperative row stores

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int WS = A.ws, G = EW / WS;
    const bool is_prep = PW && warp == EW;
    // barrier among the compute warps (the prep warp runs on its own clock)
    auto csync = [&]() {
        if constexpr (PW) asm volatile("bar.sync 1, %0;" ::"r"(ETHREADS) : "memory");
        else __syncthreads();
    };
    auto item_sync = [&]() {                     // opens a work item: compute warps + prep warp
        if constexpr (PW) asm volatile("bar.sync 2, %0;" ::"r"(ATHREADS) : "memory");
    };
    const int unit = is_prep ? 0 : warp / WS, wiu = is_prep ? -1 : warp - unit * WS;   // (the prep warp leaves before the item loop)
    const int d = A.d, nw = A.nwalkers;
    const bool resident = A.n <= CH;
    const bool prop_lane = (wiu == 0 && lane < P);
    unsigned long long bar_target = 0;

    // resident: the whole training set (rows >= n zero-filled) is loaded once
    auto load_resident = [&]() {
        for (int idx = tid; idx < D * CH; idx += ATHREADS) {
            int k = idx / CH, jj = idx - k * CH;
            sX[idx] = (k < d && jj < A.n) ? A.XsT[(long long)k * A.npad + jj] : 0.0;
        }
        for (int jj = tid; jj < CH; jj += ATHREADS) sAl[jj] = (jj < A.n) ? A.alpha[jj] : 0.0;
    };
    // streamed: chunks of CH points (CH divides npad; padding rows of XsT and alpha
    // are zero) through a double-buffered cp.async ring: buffer = [D][CH] + [CH]
    const int BUF = (D + 1) * CH;
    auto issue_chunk = [&](long long c0, int buf) {
        double* bX = sm + buf * BUF;
        for (int idx = tid; idx < (D + 1) * (CH / 2) && !is_prep; idx += ETHREADS) {
            int k = idx / (CH / 2), j2 = (idx - k * (CH / 2)) * 2;
            const double* src = (k < D) ? ((k < d) ? A.XsT + (long long)k * A.npad + c0 + j2 : nullptr)
                                        : A.alpha + c0 + j2;
            double* dst = bX + k * CH + j2;
            if (src) {
                unsigned sa = (unsigned)__cvta_generic_to_shared(dst);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(src) : "memory");
            } else {
                dst[0] = 0.0; dst[1] = 0.0;
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (resident) { load_resident(); __syncthreads(); }
    // bulk-copy ring of the streamed wide unit: one mbarrier per (buffer, warp); the rows k >= d of both
    // buffers (padding dimensions) are zeroed once, no copy ever touches them
    __shared__ __align__(8) unsigned long long wbar[2][WIDE ? EW : 1];
    unsigned wphase = 0;                             // bit b: parity of this warp's next wait on buffer b
    if (WIDE && !resident) {
        if (tid < 2 * EW) {
            const unsigned ba = (unsigned)__cvta_generic_to_shared(&wbar[tid / EW][tid % EW]);
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ba) : "memory");
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int idx = tid; idx < 2 * (D - d) * CH; idx += ETHREADS) {
            const int b2 = idx / ((D - d) * CH), rem = idx - b2 * (D - d) * CH;
            sm[b2 * ((D + 1) * CH) + d * CH + rem] = 0.0;
        }
        __syncthreads();
    }
    unsigned long long flow_prev_target = 0;
    bool flow_have_prev = false;
    if constexpr (FLOW) {
        // version 0 = the initial positions (the log-prob pass of step -1 does not move them)
        for (long long idx = (long long)blockIdx.x * ATHREADS + tid; idx < (long long)nw * d; idx += (long long)gridDim.x * ATHREADS) {
            const double v = A.coords[idx];
            const unsigned lo = (unsigned)__double2loint(v), hi = (unsigned)__double2hiint(v);
            asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(A.ring + idx), "r"(lo), "r"(1u), "r"(hi), "r"(1u) : "memory");
        }
    }

    // Everything of a proposal that depends on the random stream only (which walker,
    // which partner, the stretch factor, the accept threshold): computed by the
    // proposal lanes BEFORE they wait on the grid barrier of the previous half-step.
    // (u, e): unit and proposal slot the calling lane prepares, pb: prep buffer it writes
    auto prep_to = [&](int step, int split, int b, int u, int e, int pb) {
        const int item = (b * G + u) * P + e;
        const int n_items = (step < 0) ? nw : (split == 0 ? (nw + 1) / 2 : nw / 2);
        const int n_other = (split == 0) ? nw / 2 : (nw + 1) / 2;
        int w = -1, partner = -1;
        double zz = 1.0, logz = 0.0, logu = 0.0;
        if (item < n_items) {
            if (step < 0) {
                w = item;
            } else {
                const unsigned step_lo = (unsigned)(A.first_step + step);
                w = member_of(A, item, split, step_lo);
                if (n_other > 0) {
                    const unsigned gw = (unsigned)(A.walker_offset + w);
                    U4 rp = philox4x32_10(gw, step_lo, AB_STREAM_PARTNER, 0, A.seed_lo, A.seed_hi);
                    int jj = (int)__umulhi(rp.x, (unsigned)n_other);
                    partner = member_of(A, jj, 1 - split, step_lo);
                    U4 rm = philox4x32_10(gw, step_lo, AB_STREAM_MOVE, 0, A.seed_lo, A.seed_hi);
                    double uz = u53(rm.x, rm.y), ua = u53(rm.z, rm.w);
                    double tz = __dadd_rn(__dmul_rn(A.a - 1.0, uz), 1.0);
                    zz = __ddiv_rn(__dmul_rn(tz, tz), A.a);
                    logz = (d - 1.0) * log(zz);
                    logu = log(ua);
                }
            }
        }
        sW[pb][u][e] = w; sPartner[pb][u][e] = partner; sZZ[pb][u][e] = zz; sLogZ[pb][u][e] = logz; sLogU[pb][u][e] = logu;
    };
    // wide unit: every proposal lane prepares its own slot in place
    auto prep = [&](int step, int split, int b) {
        if (prop_lane) prep_to(step, split, b, unit, lane, 0);
    };
    // small units: the prep warp's lane l serves slot (l / P, l % P) of the CTA's work item `b` of (step, split)
    auto prep_warp = [&](int step, int split, int b, int pb) {
        if (is_prep && lane < G * P) prep_to(step, split, b, lane / P, lane % P, pb);
    };
    // the work item of this CTA that follows item `it` of half-step (step, split); false: none left
    auto next_item = [&](int& step, int& split, int& it) -> bool {
        it += gridDim.x;
        for (;;) {
            if (step >= A.nsteps) return false;
            const int n_items = (step < 0) ? nw : (split == 0 ? (nw + 1) / 2 : nw / 2);
            if (it < (n_items + P * G - 1) / (P * G)) return true;
            if (step < 0 || split == 1) { step++; split = 0; } else split = 1;
            it = blockIdx.x;
        }
    };
    int pbuf = 0;                                    // prep buffer of the current work item

    const int first = A.init_logp ? -1 : 0;
    // contiguous ranges of (unit, chunk) pairs: CTA c owns [c W / G, (c + 1) W / G)
    auto range_begin = [&](long long W, long long c) -> long long { return c * W / (long long)gridDim.x; };
    auto range_owner = [&](long long W, long long w) -> int {
        long long c = w * (long long)gridDim.x / W;
        while (c + 1 < (long long)gridDim.x && range_begin(W, c + 1) <= w) c++;
        while (c > 0 && range_begin(W, c) > w) c--;
        return (int)c;
    };
    // unit this CTA starts the given half-step with (its random-stream part is prepared early)
    auto first_unit = [&](int step, int split) -> int {
        if (!(WIDE && !resident && A.ranged != 0)) return (int)blockIdx.x;
        const int n_items = (step < 0) ? nw : (split == 0 ? (nw + 1) / 2 : nw / 2);
        const int nbatch = (n_items + P * G - 1) / (P * G);
        const int nchunks = (int)(A.npad / CH);
        return (int)(range_begin((long long)nbatch * nchunks, blockIdx.x) / nchunks);
    };
    if constexpr (PW) {
        if (is_prep) {
            // the prep warp's whole life: stay two work items ahead of the compute warps
            int s0 = first, p0 = 0, i0 = (int)blockIdx.x - (int)gridDim.x;
            bool more = next_item(s0, p0, i0);
            int prepared = 0, opened = 0;
            for (int a2 = 0; a2 < 2 && more; a2++) {
                prep_warp(s0, p0, i0, prepared % 3);
                prepared++;
                more = next_item(s0, p0, i0);
            }
            while (opened < prepared) {
                item_sync();                          // item `opened` starts: its buffer is complete
                opened++;
                if (more) {                           // buffer (opened + 1) % 3 was last read by item opened - 2
                    prep_warp(s0, p0, i0, prepared % 3);
                    prepared++;
                    more = next_item(s0, p0, i0);
                }
            }
            return;
        }
    } else {
        if (first < A.nsteps) prep(first, 0, first_unit(first, 0));
    }
    for (int step = first; step < A.nsteps; step++) {
        const int nsplit = (step < 0) ? 1 : 2;
        // row of the stored chain this step writes (-1: not stored)
        const long long store_row = (A.chain && step >= 0 && (step + 1) % A.thin_by == 0)
                                        ? (long long)((step + 1) / A.thin_by - 1) : -1;
        for (int split = 0; split < nsplit; split++) {
            const int n_items = (step < 0) ? nw : (split == 0 ? (nw + 1) / 2 : nw / 2);
            const int nbatch = (n_items + P * G - 1) / (P * G);
            const int slot = (step < 0) ? 2 : split;             // completion counters / segment sums of this kind of half-step
            const bool ranged = WIDE && !resident && A.ranged != 0;
            const int nchunks = resident ? 1 : (int)(A.npad / CH);
            const long long Wtot = (long long)nbatch * nchunks;  // (unit, chunk) pairs of this half-step
            const long long w_begin = ranged ? range_begin(Wtot, blockIdx.x) : 0, w_end = ranged ? range_begin(Wtot, blockIdx.x + 1) : 0;
            long long wcur = w_begin;
            int it = blockIdx.x;
            bool first_seg = true;
            for (;;) {
                int b, c_lo = 0, c_hi = nchunks, seg = 0, nseg = 1;
                if (ranged) {
                    if (wcur >= w_end) break;
                    b = (int)(wcur / nchunks);
                    const long long u0 = (long long)b * nchunks, u1 = u0 + nchunks;
                    c_lo = (int)(wcur - u0);
                    c_hi = (int)((w_end < u1 ? w_end : u1) - u0);
                    const int cta0 = range_owner(Wtot, u0), cta1 = range_owner(Wtot, u1 - 1);
                    seg = (int)blockIdx.x - cta0;
                    nseg = cta1 - cta0 + 1;
                    wcur = u0 + c_hi;
                } else {
                    if (it >= nbatch) break;
                    b = it;
                    it += gridDim.x;
                }
                if (!PW && !first_seg) prep(step, split, b);         // wide: further units of this CTA inline
                first_seg = false;
                item_sync();                                         // small units: this item's prep buffer is complete
                // ---- gather (proposal lanes): own state and partner position, proposal ----
                bool first_chunk_issued = false;
                if constexpr (WIDE) {
                    // streamed wide unit: the first chunk of this item is requested before the gather, so it
                    // arrives while the proposal lanes fetch the walkers (the warp's buffers are free: its
                    // reads of the previous item ended before the barriers in between)
                    if (!resident && c_lo < c_hi) {
                        const int per = CH / EW, j0 = warp * per;
                        const unsigned ba = (unsigned)__cvta_generic_to_shared(&wbar[0][warp]);
                        const unsigned row_bytes = (unsigned)per * 8u;
                        const long long off = (long long)c_lo * CH + j0;
                        if (lane == 0)
                            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ba), "r"((unsigned)(d + 1) * row_bytes) : "memory");
                        __syncwarp();
                        for (int k = lane; k <= d; k += 32) {
                            const double* src = (k < d) ? A.XsT + (long long)k * A.npad + off : A.alpha + off;
                            const unsigned da = (unsigned)__cvta_generic_to_shared(sm + (k < d ? k : D) * CH + j0);
                            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                         ::"r"(da), "l"(src), "r"(row_bytes), "r"(ba) : "memory");
                        }
                        first_chunk_issued = true;
                    }
                }
                // (the compile-time-chunk kernel of the large ensembles keeps the per-lane gather: with the
                // cooperative one its inner loop was scheduled 5 % slower, for a gather that is 1 % of its time)
                if constexpr (WIDE && CHT == 0) {
                    // Wide unit: the WHOLE CTA gathers.  Element (e, k) = coordinate k of proposal e goes to one
                    // thread, so a walker's row is one coalesced request and the 32 x d proposals are formed in
                    // parallel (as scattered 8-byte loads of the 32 proposal lanes the gather took ~7000 cycles
                    // per segment: a third of a half-step in spread mode).  The arithmetic of a coordinate is the
                    // same separately rounded sequence as below; "outside the box" is collected as a flag per
                    // proposal (threads that find a violation store the same value).
                    if (tid < P) sOut[tid] = 0;
                    csync();
                    for (int idx = tid; idx < P * D; idx += ETHREADS) {
                        const int e = idx / D, k = idx - e * D;
                        const int w = sW[0][0][e], partner = sPartner[0][0][e];
                        double q = 0.0, qs = 0.0, sv = 0.0;
                        if (w >= 0 && k < d) {
                            sv = __ldcg(&A.coords[(long long)w * d + k]);
                            if (step >= 0 && partner >= 0) {
                                const double cv = __ldcg(&A.coords[(long long)partner * d + k]);
                                q = __dsub_rn(cv, __dmul_rn(__dsub_rn(cv, sv), sZZ[0][0][e]));
                            } else {
                                q = sv;                                  // step < 0 or no partner: the current position
                            }
                            if (!((q > A.lo[k]) && (q < A.hi[k]))) sOut[e] = 1;
                            qs = fma(q, A.t_scale[k], A.t_off[k]) * A.kp.inv_len[k];
                        }
                        sS[0][e][k] = sv;
                        sQ[0][e][k] = q;
                        sQs[0][e][k] = qs;
                    }
                    csync();
                    if (prop_lane) {
                        const int e = lane, w = sW[0][0][e], partner = sPartner[0][0][e];
                        int inside = 1;
                        if (w >= 0) {
                            if (step >= 0) sLps[0][e] = __ldcg(&A.logp[w]);
                            if (step >= 0 && partner < 0) inside = -1;  // no complementary walker: keep the state
                            else if (sOut[e]) inside = 0;
                            if (A.use_normal) {
                                // scipy's norm.logpdf term by term, in dimension order (oracle/utility.py)
                                double pr = 0.0;
                                for (int k = 0; k < d; k++) {
                                    if (A.pr_sd[k] > 0.0) {
                                        const double z = __ddiv_rn(__dsub_rn(sQ[0][e][k], A.pr_mu[k]), A.pr_sd[k]);
                                        pr = __dadd_rn(pr, __dsub_rn(__dsub_rn(-__dmul_rn(z, z) * 0.5, 0.9189385332046727),
                                                                     A.pr_lsd[k]));
                                    }
                                }
                                sPrior[0][e] = pr;
                            }
                        }
                        sInside[0][e] = inside;
                    }
                } else if (prop_lane) {
                    const int e = lane, w = sW[pbuf][unit][e], partner = sPartner[pbuf][unit][e];
                    int inside = 1;
                    if (w >= 0) {
                        // all global loads first (one L2 round trip), then the arithmetic
                        double cs[D], ss[D];
                        const long long ow = (long long)w * d, op = (long long)(partner >= 0 ? partner : w) * d;
                        const bool from_ring = FLOW && step >= 0 && partner >= 0;
#pragma unroll
                        for (int k = 0; k < D; k++) {
                            ss[k] = (k < d) ? __ldcg(&A.coords[ow + k]) : 0.0;
                            cs[k] = (k < d && !from_ring) ? __ldcg(&A.coords[op + k]) : 0.0;
                        }
                        if (step >= 0) sLps[unit][e] = __ldcg(&A.logp[w]);
                        if constexpr (FLOW) {
                            if (from_ring) {
                                // partner's position after `step` (split 0) or `step + 1` (split 1) updates
                                const unsigned need = (unsigned)step + (split == 0 ? 1u : 2u);
                                const uint4* line = A.ring + ((long long)((need - 1u) % AB_ENS_RING) * nw + partner) * d;
                                bool ok;
                                unsigned spins = 0;
                                long long wd0 = 0;
                                do {
                                    ok = true;
#pragma unroll
                                    for (int k = 0; k < D; k++) {
                                        if (k < d) {
                                            unsigned x0, x1, x2, x3;
                                            asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                                                         : "=r"(x0), "=r"(x1), "=r"(x2), "=r"(x3) : "l"(line + k) : "memory");
                                            ok = ok && (x1 == need) && (x3 == need);
                                            cs[k] = __hiloint2double((int)x2, (int)x0);
                                        }
                                    }
                                    // watchdog: a record that never arrives (it cannot, by the dependency order; this
                                    // guards the GPU against a fault elsewhere) raises flag 2 after ~2 s, and every
                                    // poll loop leaves as soon as it sees the flag: the run ends with an error
                                    if (!ok && (++spins & 0x3fffu) == 0) {
                                        if (wd0 == 0) wd0 = clock64();
                                        if (*((volatile int*)A.nan_flag) == 2 || clock64() - wd0 > 4000000000LL) {
                                            atomicExch(A.nan_flag, 2);
                                            break;
                                        }
                                    }
                                } while (!ok);
                            }
                        }
                        const double zz = sZZ[pbuf][unit][e];
                        if (step >= 0 && partner < 0) inside = -1;      // no complementary walker: keep the state
#pragma unroll
                        for (int k = 0; k < D; k++) {
                            if (k < d) {
                                // step < 0 or no partner: cs == ss, the proposal is the current position
                                const double q = (step >= 0 && partner >= 0)
                                                     ? __dsub_rn(cs[k], __dmul_rn(__dsub_rn(cs[k], ss[k]), zz)) : ss[k];
                                sS[unit][e][k] = ss[k];
                                sQ[unit][e][k] = q;
                                if (inside >= 0 && !((q > A.lo[k]) && (q < A.hi[k]))) inside = 0;
                                sQs[unit][e][k] = fma(q, A.t_scale[k], A.t_off[k]) * A.kp.inv_len[k];
                            }
                        }
                        if (A.use_normal) {
                            // scipy's norm.logpdf term by term, in dimension order (oracle/utility.py)
                            double pr = 0.0;
                            for (int k = 0; k < d; k++) {
                                if (A.pr_sd[k] > 0.0) {
                                    const double z = __ddiv_rn(__dsub_rn(sQ[unit][e][k], A.pr_mu[k]), A.pr_sd[k]);
                                    pr = __dadd_rn(pr, __dsub_rn(__dsub_rn(-__dmul_rn(z, z) * 0.5, 0.9189385332046727),
                                                                 A.pr_lsd[k]));
                                }
                            }
                            sPrior[unit][e] = pr;
                        }
                    }
                    for (int k = (w < 0 ? 0 : d); k < D; k++) { sQ[unit][e][k] = 0.0; sQs[unit][e][k] = 0.0; }
                    sInside[unit][e] = inside;
                }
                csync();
                // ---- surrogate mean of the two proposals of this unit ------------
                if constexpr (WIDE) {
                    double qv[D];
#pragma unroll
                    for (int k = 0; k < D; k++) qv[k] = sQs[0][lane][k];
                    double accw = 0.0;
                    // cn is a multiple of 32 (resident: CH, rows >= n are zero with alpha = 0); every
                    // 128-bit broadcast read serves two training points
                    auto eval_wide = [&](const double* bX, const double* bAl, int cn) {
                        const int per = cn / EW;
                        const int j0 = warp * per, j1 = j0 + per;
#pragma unroll kWideUnroll
                        for (int j = j0; j < j1; j += 2) {
                            // two partial sums per point (even / odd dimensions): with the two points of
                            // a load and the unroll that is 8 independent FMA chains per lane
                            double r0 = 0.0, r1 = 0.0, s0 = 0.0, s1 = 0.0;
#pragma unroll
                            for (int k = 0; k < D; k += 2) {
                                const double2 xa = *reinterpret_cast<const double2*>(&bX[k * CH + j]);
                                const double2 xb = *reinterpret_cast<const double2*>(&bX[(k + 1) * CH + j]);
                                const double d0 = qv[k] - xa.x, d1 = qv[k] - xa.y;
                                const double e0 = qv[k + 1] - xb.x, e1 = qv[k + 1] - xb.y;
                                r0 = fma(d0, d0, r0);
                                r1 = fma(d1, d1, r1);
                                s0 = fma(e0, e0, s0);
                                s1 = fma(e1, e1, s1);
                            }
                            const double2 al = *reinterpret_cast<const double2*>(&bAl[j]);
                            accw = fma(ab_radial<KIND>(r0 + s0, A.kp.alpha, A.kp.inv2a), al.x, accw);
                            accw = fma(ab_radial<KIND>(r1 + s1, A.kp.alpha, A.kp.inv2a), al.y, accw);
                        }
                    };
                    if (resident) {
                        eval_wide(sX, sAl, CH);
                    } else {
                        // every warp streams ITS slice of a chunk (the CH / EW points it evaluates) through
                        // its own two-deep ring: no CTA barrier in the chunk loop, a warp that falls behind
                        // delays nobody
                        const int per = CH / EW, j0 = warp * per;
                        // row slices of `per` points (256 B at per = 32) by bulk copies: lane k issues row k (lane d
                        // the alpha row), completion on the warp's own mbarrier of that buffer
                        auto issue_bulk = [&](long long c0, int buf) {
                            const unsigned ba = (unsigned)__cvta_generic_to_shared(&wbar[buf][warp]);
                            const unsigned row_bytes = (unsigned)per * 8u;
                            if (lane == 0)
                                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ba), "r"((unsigned)(d + 1) * row_bytes) : "memory");
                            __syncwarp();
                            for (int k = lane; k <= d; k += 32) {
                                const double* src = (k < d) ? A.XsT + (long long)k * A.npad + c0 + j0 : A.alpha + c0 + j0;
                                const unsigned da = (unsigned)__cvta_generic_to_shared(sm + buf * BUF + (k < d ? k : D) * CH + j0);
                                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                             ::"r"(da), "l"(src), "r"(row_bytes), "r"(ba) : "memory");
                            }
                        };
                        auto wait_bulk = [&](int buf) {
                            const unsigned ba = (unsigned)__cvta_generic_to_shared(&wbar[buf][warp]);
                            const unsigned par = (wphase >> buf) & 1u;
                            unsigned ok;
                            do {
                                asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                                             : "=r"(ok) : "r"(ba), "r"(par) : "memory");
                            } while (!ok);
                            wphase ^= 1u << buf;
                        };
                        if (c_lo < c_hi && !first_chunk_issued) issue_bulk((long long)c_lo * CH, 0);
                        for (int c = c_lo; c < c_hi; c++) {
                            const int buf = (c - c_lo) & 1;
                            if (c + 1 < c_hi) issue_bulk((long long)(c + 1) * CH, buf ^ 1);     // that buffer was read out before the
                            wait_bulk(buf);                                                    // __syncwarp that closed chunk c - 1
                            const double* bX = sm + buf * BUF;
                            eval_wide(bX, bX + D * CH, CH);
                            __syncwarp();
                        }
                    }
                    sPart[warp][lane] = accw;
                } else {
                double q[P][D], acc[P];
#pragma unroll
                for (int e = 0; e < P; e++) {
                    acc[e] = 0.0;
#pragma unroll
                    for (int k = 0; k < D; k++) q[e][k] = sQs[unit][e][k];
                }
                auto eval_points = [&](const double* bX, const double* bAl, int cn) {
#pragma unroll 2
                    for (int jj = wiu * 32 + lane; jj < cn; jj += 32 * WS) {
                        double r[P];
#pragma unroll
                        for (int e = 0; e < P; e++) r[e] = 0.0;
#pragma unroll
                        for (int k = 0; k < D; k++) {
                            const double x = bX[k * CH + jj];
#pragma unroll
                            for (int e = 0; e < P; e++) {
                                const double df = q[e][k] - x;
                                r[e] = fma(df, df, r[e]);
                            }
                        }
                        const double al = bAl[jj];
#pragma unroll
                        for (int e = 0; e < P; e++) acc[e] = fma(ab_radial<KIND>(r[e], A.kp.alpha, A.kp.inv2a), al, acc[e]);
                    }
                };
                if (resident) {
                    eval_points(sX, sAl, (int)A.n);
                } else {
                    const int nch = (int)(A.npad / CH);
                    issue_chunk(0, 0);
                    for (int c = 0; c < nch; c++) {
                        if (c + 1 < nch) issue_chunk((long long)(c + 1) * CH, (c + 1) & 1);
                        else asm volatile("cp.async.commit_group;" ::: "memory");
                        asm volatile("cp.async.wait_group 1;" ::: "memory");
                        csync();
                        const double* bX = sm + (c & 1) * BUF;
                        eval_points(bX, bX + D * CH, CH);
                        csync();             // buffer c & 1 is refilled by chunk c + 2
                    }
                }
#pragma unroll
                for (int e = 0; e < P; e++) {
                    acc[e] = ab_warp_sum(acc[e]);
                    if (lane == 0) sPart[warp][e] = acc[e];
                }
                }
                csync();
                // ---- split units: publish this slice's sums; the CTA that completes the unit goes on ----
                bool finisher = true;
                if (WIDE && nseg > 1) {
                    double* part = A.slice_part + (((long long)slot * A.max_units + b) * A.maxseg) * 32;
                    if (prop_lane) {
                        double sp = 0.0;
#pragma unroll
                        for (int x = 0; x < EW; x++) sp += sPart[x][lane];          // warps in order
                        __stcg(&part[seg * 32 + lane], sp);
                    }
                    csync();
                    if (tid == 0) {
                        // one acq_rel counter update instead of a fence by every thread on either side: release is
                        // cumulative over the segment sums stored before the barrier, acquire orders the finisher's
                        // reads (behind the next barrier) after the other segments' stores
                        unsigned old;
                        asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;"
                                     : "=r"(old) : "l"(&A.slice_cnt[(long long)slot * A.max_units + b]) : "memory");
                        sSliceLast = ((old + 1u) % (unsigned)nseg == 0u) ? 1 : 0;   // nseg is the same in every half-step of this kind
                    }
                    csync();
                    finisher = sSliceLast != 0;
                }
                // ---- accept / reject ------------------------------------------------
                if (prop_lane && finisher) {
                    const int e = lane, w = sW[pbuf][unit][e];
                    if (w >= 0) {
                        double s = 0.0;
                        if (WIDE && nseg > 1) {
                            const double* part = A.slice_part + (((long long)slot * A.max_units + b) * A.maxseg) * 32;
                            for (int x = 0; x < nseg; x++) s += __ldcg(&part[x * 32 + e]);   // segments in order
                        } else {
                        double pv[EW];                       // independent loads, then the fixed-order sum
#pragma unroll
                        for (int x = 0; x < EW; x++) pv[x] = (x < WS) ? sPart[unit * WS + x][e] : 0.0;
#pragma unroll
                        for (int x = 0; x < EW; x++) s += pv[x];
                        }
                        double ys = fma(A.kp.amp, s, A.mean);
                        double y = (A.y_kind == 0) ? fma(ys, A.y_scale, A.y_off)
                                 : (A.y_kind == 1) ? -pow(10.0, ys) : pow(10.0, ys);
                        const int inside = sInside[unit][e];
                        if (A.use_normal) y = __dadd_rn(y, sPrior[unit][e]);
                        double lp_q = (inside == 1) ? y : -INFINITY;
                        if (inside == 1 && isnan(y)) atomicCAS(A.nan_flag, 0, 1);      // (keeps a watchdog flag 2)
                        if (step < 0) {
                            A.logp[w] = lp_q;
                        } else {
                            double lp_s = sLps[unit][e];
                            bool acc = (inside >= 0) && ((sLogZ[pbuf][unit][e] + lp_q - lp_s) > sLogU[pbuf][unit][e]);
                            if constexpr (FLOW) {
                                // the record other CTAs wait for goes out before anything else
                                const unsigned fl = (unsigned)step + 2u;
                                uint4* line = A.ring + ((long long)((fl - 1u) % AB_ENS_RING) * nw + w) * d;
                                for (int k = 0; k < d; k++) {
                                    const double v = acc ? sQ[unit][e][k] : sS[unit][e][k];
                                    asm volatile("st.relaxed.gpu.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(line + k),
                                                 "r"((unsigned)__double2loint(v)), "r"(fl), "r"((unsigned)__double2hiint(v)), "r"(fl) : "memory");
                                }
                            }
                            if (acc) {
                                for (int k = 0; k < d; k++) A.coords[(long long)w * d + k] = sQ[unit][e][k];
                                A.logp[w] = lp_q;
                                atomicAdd(reinterpret_cast<unsigned long long*>(A.naccept + w), 1ULL);
                                lp_s = lp_q;
                            }
                            if (A.rec_q && inside >= 0) {
                                long long r = (long long)step * nw + w;
                                for (int k = 0; k < d; k++) A.rec_q[r * d + k] = sQ[unit][e][k];
                                A.rec_lp[r] = lp_q;
                            }
                            if constexpr (WIDE) {
                                sAccF[e] = acc ? 1 : 0;                      // rows are stored by the whole CTA below
                                sLpOut[e] = lp_s;
                            } else if (store_row >= 0) {
                                const long long r = store_row * A.chain_ld + A.chain_off + w;
#pragma unroll 1
                                for (int pd = 0; pd < A.n_dst; pd++) {       // own buffer, then the peers' (NVLink stores)
                                    double* cdst = A.chain_dst[pd] + r * d;
                                    for (int k = 0; k < d; k++) cdst[k] = acc ? sQ[unit][e][k] : sS[unit][e][k];
                                    A.logp_dst[pd][r] = lp_s;
                                }
                            }
                        }
                    }
                }
                if constexpr (WIDE) {
                    // Stored rows of the unit's 32 walkers, written by ALL warps: 16-byte stores, the d / 2
                    // chunks of a walker's row on consecutive lanes (whole 32-byte sectors per row instead of
                    // d scattered 8-byte stores per lane -- what the peer destinations over NVLink need: as
                    // scalar stores of the proposal lanes the fused all_gather cost 14 % of the kernel at 8 GPUs)
                    if (store_row >= 0 && finisher) {
                        csync();                                         // sAccF / sLpOut / sQ / sS of this unit are complete
                        const long long rbase = store_row * A.chain_ld + A.chain_off;
                        if (A.chain_vec) {
                            const int half = d >> 1, per_dst = P * half;
                            for (int idx = tid; idx < A.n_dst * per_dst; idx += ETHREADS) {
                                const int pd = idx / per_dst, rem = idx - pd * per_dst, e = rem / half, c2 = (rem - e * half) * 2;
                                const int w = sW[0][0][e];
                                if (w < 0) continue;
                                const double* srow = sAccF[e] ? &sQ[0][e][0] : &sS[0][e][0];
                                *reinterpret_cast<double2*>(A.chain_dst[pd] + (rbase + w) * d + c2) = make_double2(srow[c2], srow[c2 + 1]);
                            }
                        } else {
                            const int per_dst = P * d;
                            for (int idx = tid; idx < A.n_dst * per_dst; idx += ETHREADS) {
                                const int pd = idx / per_dst, rem = idx - pd * per_dst, e = rem / d, k = rem - e * d;
                                const int w = sW[0][0][e];
                                if (w < 0) continue;
                                A.chain_dst[pd][(rbase + w) * d + k] = sAccF[e] ? sQ[0][e][k] : sS[0][e][k];
                            }
                        }
                        for (int idx = tid; idx < A.n_dst * P; idx += ETHREADS) {
                            const int pd = idx / P, e = idx - pd * P, w = sW[0][0][e];
                            if (w >= 0) A.logp_dst[pd][rbase + w] = sLpOut[e];
                        }
                    }
                }
                // wide: the proposal lanes own sW.. of their unit, the next prep / gather by the same
                // lanes follows in program order; small units: the next item's values sit in the other
                // prep buffer since the barrier after the compute phase.  sQs / sPart readers are fenced
                // by the two __syncthreads above and the one that opens grid_arrive / the next gather
                csync();
                if constexpr (PW) pbuf = (pbuf + 1) % 3;
            }
            const bool flow_step = FLOW && step >= 0;
            if (!flow_step) grid_arrive(A.barrier, bar_target, csync);
            {   // random-stream part of the next half-step, overlapped with the barrier
                int nstep = step, nsp = split + 1;
                if (nsp >= nsplit) { nstep = step + 1; nsp = 0; }
                if (!PW && nstep < A.nsteps) prep(nstep, nsp, first_unit(nstep, nsp));
            }
            if (!flow_step) {
                grid_wait(A.barrier, bar_target, csync);
            } else if (split == 1 && (step + 1) % AB_ENS_THROTTLE == 0) {
                // progress barrier: wait for the one arrived at a period ago (everybody has finished
                // step + 1 - AB_ENS_THROTTLE), then arrive at this one
                if (flow_have_prev) grid_wait(A.barrier, flow_prev_target, csync);
                grid_arrive(A.barrier, bar_target, csync);
                flow_prev_target = bar_target;
                flow_have_prev = true;
            }
        }
    }
}

// one_pass_only: return 1 without launching unless every unit of a half-step gets its own co-resident CTA
template <int KIND, int D, int P, int EW = 8>
int launch_ens_p(ab_gp* h, EnsArgs& A, int n_half, bool one_pass_only = false) {
    constexpr int ETHREADS = EW * 32 + (P == 32 ? 0 : 32);     // small units: + the prep warp
    void (*kern)(const EnsArgs) = ensemble_kernel<KIND, D, EW, P>;
    // shared memory: resident when the whole training set fits, else two chunk buffers
    const bool resident = ab_resident(A.n, D);
    int ch;
    size_t smem;
    if (resident) {
        ch = (int)((A.n + 31) / 32 * 32);
        if (ch < 32) ch = 32;
        smem = (size_t)ch * (D + 1) * 8;
    } else {
        // divides npad; two buffers of at most ~48 KB each (two CTAs per SM) or ~100 KB each (the
        // 16-warp wide unit has the SM to itself: longer chunks, fewer CTA barriers per point)
        const size_t per_buf = (EW == 16) ? 100 * 1024 : 48 * 1024;
        ch = 128;
        while (ch * 2 <= 1024 && A.npad % (ch * 2) == 0 && (size_t)(ch * 2) * (D + 1) * 8 <= per_buf) ch *= 2;
        if (P == 32 && A.ch_hint > 0 && A.ch_hint <= ch && A.npad % A.ch_hint == 0) ch = A.ch_hint;
        smem = 2 * (size_t)ch * (D + 1) * 8;
    }
    A.ch = ch;
    if constexpr (P == 32 && EW == 16) {
        if (!resident && ch == 512 && A.ch_hint == 0) kern = ensemble_kernel<KIND, D, EW, P, 512>;
    }
    if constexpr (P == 2) {
        // dataflow schedule: resident training set, a ring was provided by the caller
        if (A.ring && resident) kern = ensemble_kernel<KIND, D, EW, P, 0, true>;
        else A.ring = nullptr;
    } else {
        A.ring = nullptr;
    }
    AB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    AB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, ETHREADS, smem));
    if (per_sm < 1) { ab_set_error("ensemble kernel does not fit on an SM (smem %zu)", smem); return -3; }
    int G = EW / A.ws;
    int nbatch = (n_half + P * G - 1) / (P * G);
    const int grid_max = per_sm * h->nsm;
    if (one_pass_only && grid_max < nbatch) return 1;
    int grid = grid_max;
    A.ranged = 0;
    if (P == 32 && !resident) {
        // streamed wide unit: equal contiguous ranges of (unit, chunk) pairs per CTA when every CTA
        // gets at least 4 chunks and no unit is cut into more than AB_ENS_MAXSEG segments
        const long long nch = A.npad / ch;
        const long long share = (long long)nbatch * nch / grid_max;
        if (share >= 4 && nch / share + 2 <= A.maxseg) A.ranged = 1;
        if (A.ch_hint > 0 && nch + 2 <= A.maxseg) {
            // spread mode: few units, so the (unit, chunk) pairs themselves are dealt over the CTAs; every CTA
            // must own at least one pair in every kind of half-step (an empty range would be counted as a
            // segment that never arrives), so the grid is capped at the pairs of the smaller half-step
            A.ranged = 1;
            const long long small_items = (A.nsteps > 0) ? (A.nwalkers / 2 > 0 ? A.nwalkers / 2 : 1) : A.nwalkers;
            const long long w_min = ((small_items + P - 1) / P) * nch;
            if ((long long)grid > w_min) grid = (int)w_min;
        }
    }
    if (!A.ranged && grid > nbatch) grid = nbatch;
    if (grid < 1) grid = 1;
    void* args[] = {(void*)&A};
    ab_prof_begin(h, AB_PROF_ENSEMBLE);
    AB_CUDA(cudaLaunchCooperativeKernel((void*)kern, dim3(grid), dim3(ETHREADS), args, smem, h->stream));
    ab_prof_end(h, AB_PROF_ENSEMBLE);
    ab_count_launches(1);
    return 0;
}

// n_half: proposals of the larger half-step (or all walkers for a log-prob-only call)
// small_cta: try 4-warp CTAs first; else (or when they would not all be co-resident) 8-warp CTAs, ws8 warps per unit
template <int KIND, int D>
int launch_ens(ab_gp* h, EnsArgs& A, int n_half, int p, bool small_cta, int ws8) {
    // wide unit: 16 warps split the training points (4 warps per scheduler hide the FP64 dependency
    // latency that 2 leave exposed: ncu, c5 share, FP64 pipe 56 % with 8 warps); one CTA per SM
    if (p == 32) return launch_ens_p<KIND, D, 32, 16>(h, A, n_half);
    if (small_cta) {
        // One 4-warp unit (+ prep warp) per CTA, two or more CTAs per SM: units that would share an
        // 8-warp CTA in lockstep instead run as independent CTAs, so one unit's publish -> poll latency
        // is covered by its neighbour's kernel evaluations on the same SM.
        uint4* ring = A.ring;
        A.ws = 4;
        const int rc = launch_ens_p<KIND, D, 2, 4>(h, A, n_half, true);
        if (rc != 1) return rc;
        A.ring = ring;
    }
    A.ws = ws8;
    return launch_ens_p<KIND, D, 2>(h, A, n_half);
}

// padded-dimension dispatch of one kernel family
template <int KIND>
int launch_ens_kind(ab_gp* h, EnsArgs& A, int n_half, int p, bool small_cta, int ws) {
    return ab_dispatch_dim(h->d, [&](auto D) { return launch_ens<KIND, D>(h, A, n_half, p, small_cta, ws); });
}

}  // namespace
