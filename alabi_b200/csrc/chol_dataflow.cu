// K2, dataflow form: the whole blocked Cholesky in ONE persistent kernel.
//
// Replaces george BasicSolver.compute (scipy cholesky) reached from
// alabi/gp_utils.py:243, alabi/core.py:1158,1430:
//
//   * one task per 128 x 128 tile (i, j), j <= i, of the lower triangle, handed
//     out in column-major order through an atomic counter (one CTA per SM);
//   * task (i, j) is LEFT-looking: it accumulates  S = sum_{k<j} L_ik L_jk^T  in one
//     long-K DMMA main loop (the tile of K is read once and written once, instead
//     of being re-read and re-written by every trailing update), then
//         i == j :  L_jj = chol(A_jj - S), D_j^-1 = L_jj^-1   (register-tiled sweep)
//         i  > j :  L_ij = (A_ij - S) D_j^-T                  (DMMA, A operand resident in smem)
//   * dependencies are per block row: prog[r] = number of final tiles in row r
//     (tiles of a row become final left to right).  The main loop waits on
//     prog[i] > k and prog[j] > k just before it prefetches k block k, so a task
//     runs ahead through every k block that is already final — look-ahead falls
//     out of the task order, there are no launch gaps and no wave quantisation.
//
// Deadlock freedom: tasks are popped in an order in which every dependency has
// a smaller index, and only resident CTAs hold tasks, so the lowest-index
// unfinished task can always run.  Every wait loop also carries a watchdog
// (about 2 s) that raises an abort flag instead of hanging the GPU.
#include <vector>
#include "handle.h"
#include "dmma_gemm.cuh"
#include "potf2.cuh"

namespace {

constexpr int NB = AB_NB;
using Core = abg::Main;
constexpr int LDC = NB + 4;                              // resident C tile [128][132]
constexpr int C_ELEMS = NB * LDC;
constexpr int BSTAGE = NB * Core::LDK;                   // one Dinv chunk [128][20]
constexpr int DF_SMEM_BYTES = (C_ELEMS + Core::STAGES * BSTAGE) * 8;     // 217088
static_assert(DF_SMEM_BYTES >= Core::SMEM_BYTES && DF_SMEM_BYTES <= 227 * 1024, "shared memory plan");

constexpr int LDH = 64 + 4;                              // 64 x 64 blocks staged in the B ring

// 64 x 64 x 64 product from shared memory on 8 warps (32 x 16 each):
//   acc[m][n] = sum_k A[m][k] * (B_KMAJOR ? B[n][k] : B[k][n]);   lda, ldb == 4 (mod 16)
// TRI prunes k4-steps whose operand block is structurally zero (warp-uniform):
//   1: B zero for k > n     2: B zero for k < n     3: A zero for k > m
template <bool B_KMAJOR, int TRI>
__device__ __forceinline__ void gemm64(double (&acc)[4][2][2], const double* A, int lda, const double* B, int ldb,
                                       int warp, int lane) {
    const int g = lane >> 2, t = lane & 3, wm = warp >> 2, wn = warp & 3;
#pragma unroll
    for (int f = 0; f < 4; f++)
#pragma unroll
        for (int q = 0; q < 2; q++) acc[f][q][0] = acc[f][q][1] = 0.0;
#pragma unroll 4
    for (int k4 = 0; k4 < 16; k4++) {
        const int k0 = k4 * 4;
        if (TRI == 1 && k0 > wn * 16 + 15) continue;
        if (TRI == 2 && k0 + 3 < wn * 16) continue;
        if (TRI == 3 && k0 > wm * 32 + 31) continue;
        double fa[4], fb[2];
#pragma unroll
        for (int f = 0; f < 4; f++) fa[f] = A[(wm * 32 + f * 8 + g) * lda + k0 + t];
#pragma unroll
        for (int q = 0; q < 2; q++)
            fb[q] = B_KMAJOR ? B[(wn * 16 + q * 8 + g) * ldb + k0 + t] : B[(k0 + t) * ldb + wn * 16 + q * 8 + g];
#pragma unroll
        for (int f = 0; f < 4; f++) {
            if (TRI == 3 && k0 > wm * 32 + f * 8 + 7) continue;
#pragma unroll
            for (int q = 0; q < 2; q++) {
                if (TRI == 1 && k0 > wn * 16 + q * 8 + 7) continue;
                if (TRI == 2 && k0 + 3 < wn * 16 + q * 8) continue;
                abg::dmma884(acc[f][q][0], acc[f][q][1], fa[f], fb[q]);
            }
        }
    }
}

// One matrix or a BATCH of equally sized matrices (k-fold cross-validation jobs,
// cv_batch.cu): matrix b lives at A + b strideA, its diagonal-block inverses at Dinv + b strideD,
// its per-block-row words (prog, logdet_parts) at + b T, its status at info + b.  A task is
// (i | b << 12, j); the task list orders the tiles of ALL matrices column by column, so every
// dependency still has a smaller task index and different matrices fill each other's waits.
struct DfArgs {
    double* A; int64_t ld; int T;
    double* Dinv; double* logdet_parts; int* info;
    int* prog;                    // [T] final tiles per block row (per matrix)
    unsigned int* next_task;      // task counter
    int* abort_flag;
    const int2* tasks; int ntasks;
    int64_t strideA, strideD;     // batch strides in doubles
};

__device__ __forceinline__ int ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// wait until prog[row] > k; `seen` caches the last value this warp observed.  Called
// convergently by whole warps: lane 0 polls (ld.acquire.gpu), the result is broadcast,
// and the trailing __syncwarp + fence orders every lane's later loads after it.
struct Waiter {
    const int* prog; int* abort_flag; bool aborted;
    __device__ __forceinline__ void wait(int row, int k, int& seen) {
        if (seen > k || aborted) return;
        int v = seen, ab = 0;
        if ((threadIdx.x & 31) == 0) {
            long long t0 = 0;
            unsigned spins = 0;
            for (;;) {
                v = ld_acquire(prog + row);
                if (v > k) break;
                if ((++spins & 255u) == 0) {
                    if (t0 == 0) t0 = clock64();
                    if (*((volatile int*)abort_flag) != 0 || clock64() - t0 > 4000000000LL) {
                        atomicExch(abort_flag, 1);
                        ab = 1;
                        break;
                    }
                }
            }
            __threadfence();
        }
        __syncwarp();
        seen = __shfl_sync(0xffffffffu, v, 0);
        aborted = __shfl_sync(0xffffffffu, ab, 0) != 0;
    }
};

// gate of the accumulation loop: chunk c belongs to k block c / KB, final once both
// block rows i and j have progressed past it
struct RowGate {
    Waiter* w; int i, j; int seen_i, seen_j;
    __device__ __forceinline__ bool ready(int c) {
        if ((c % Core::KB) != 0) return true;                 // same k block as the chunk before it
        const int k = c / Core::KB;
        if (seen_i > k && seen_j > k) return true;
        if (w->aborted) return true;
        int vi = seen_i, vj = seen_j;
        if ((threadIdx.x & 31) == 0) {
            if (vi <= k) vi = ld_acquire(w->prog + i);
            if (vj <= k) vj = ld_acquire(w->prog + j);
            __threadfence();
        }
        __syncwarp();
        seen_i = __shfl_sync(0xffffffffu, vi, 0);
        seen_j = __shfl_sync(0xffffffffu, vj, 0);
        return seen_i > k && seen_j > k;
    }
    __device__ __forceinline__ void wait(int c) {
        const int k = c / Core::KB;
        w->wait(i, k, seen_i);
        w->wait(j, k, seen_j);
    }
};

__global__ void __launch_bounds__(Core::THREADS, 1)
chol_dataflow_kernel(const __grid_constant__ DfArgs a) {
    extern __shared__ __align__(16) double smem[];
    __shared__ abp::SweepShared sh;
    __shared__ int s_task;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3, wm = warp / Core::WN, wn = warp % Core::WN;
    const int wm64 = warp >> 2, wn64 = warp & 3;          // gemm64 warp grid
    Waiter w{a.prog, a.abort_flag, false};
    double* sC = smem;
    double* sBring = smem + C_ELEMS;
    double* const sdiag = sh.sdiag;
    double* const sinv = sh.sinv;
    unsigned sweep_phase = 0;
    if (tid == 0) abp::mbar_init((unsigned)__cvta_generic_to_shared(&sh.mbar), Core::THREADS);
    __syncthreads();

    for (;;) {
        if (tid == 0) s_task = (int)atomicAdd(a.next_task, 1u);
        __syncthreads();
        const int task = s_task;
        if (task >= a.ntasks) break;
        const int tx_ = a.tasks[task].x, j = a.tasks[task].y;
        const int i = tx_ & 4095, mb = tx_ >> 12;                // block row, matrix of the batch
        double* const Ab = a.A + (int64_t)mb * a.strideA;
        double* const Db = a.Dinv + (int64_t)mb * a.strideD;
        double* const logdet_b = a.logdet_parts + (int64_t)mb * a.T;
        int* const info_b = a.info + mb;
        int* const prog_b = a.prog + (int64_t)mb * a.T;
        w.prog = prog_b;
        const int64_t row0 = (int64_t)i * NB, col0 = (int64_t)j * NB;
        int seen_i = 0, seen_j = 0;
        // the tile of K itself is only needed after the long accumulation: pull it into L2 now
        for (int c = tid; c < NB * 8; c += Core::THREADS)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(Ab + (row0 + (c >> 3)) * a.ld + col0 + (c & 7) * 16));

        // ---- S = sum_{k<j} L_ik L_jk^T, gated per k block --------------------------
        abg::Acc acc;
        acc.zero();
        if (j > 0) {
            RowGate gate{&w, i, j, 0, 0};
            Core::mainloop_gated<true, true>(acc, Ab + row0 * a.ld, a.ld, Ab + col0 * a.ld, a.ld, j * Core::KB, smem,
                                             gate, i == j);
            seen_i = gate.seen_i;
            seen_j = gate.seen_j;
        }
        // ---- C = A_ij - S, staged in shared memory ------------------------------------
        // (A_ij still holds the covariance values written before this launch)
#pragma unroll
        for (int f = 0; f < 8; f++) {
            const int r = Core::gated_row(wm, f) + g;               // row / column mapping of mainloop_gated
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int c = Core::gated_col(wn, q) + 2 * t;
                const double2 v = *reinterpret_cast<const double2*>(Ab + (row0 + r) * a.ld + col0 + c);
                double2 o;
                o.x = v.x - acc.v[f][q][0];
                o.y = v.y - acc.v[f][q][1];
                *reinterpret_cast<double2*>(sC + r * LDC + c) = o;
            }
        }
        __syncthreads();

        if (i == j) {
            // ---- diagonal tile: Cholesky + inverse by 2 x 2 recursion on 64 x 64 blocks ----
            //   [A11    ]   L11 = chol(A11), D11 = L11^-1          (register-tiled sweep, 64 columns)
            //   [A21 A22]   L21 = A21 D11^T ; A22 -= L21 L21^T     (DMMA from shared memory)
            //               L22 = chol(A22), D22 = L22^-1          (second sweep)
            //               (L^-1)21 = -D22 (L21 D11)              (two DMMA products)
            // D11 lives in the unused upper-right quadrant of sC, D22 and L21 D11 in the B ring.
            const int tx = tid & 15, ty = tid >> 4;
            double* Aj = Ab + col0 * a.ld + col0;
            double* Dj = Db + (int64_t)j * NB * NB;
            double* sD11 = sC + 64;                       // [n][k], ld LDC
            double* sD22 = sBring;                        // [m][k], ld LDH
            double* sM1 = sBring + 64 * LDH;              // [k][n], ld LDH
            double logdet = 0.0;
            for (int half = 0; half < 2; half++) {
                const int ob = half * 64;
                double pa[4][4], pb[4][4];
#pragma unroll
                for (int r = 0; r < 4; r++)
#pragma unroll
                    for (int c = 0; c < 4; c++)
                        if (r >= c) {
                            const int ii = ty + 16 * r, kk = tx + 16 * c;
                            pa[r][c] = (kk <= ii) ? sC[(ob + ii) * LDC + ob + kk] : 0.0;
                            pb[r][c] = (kk == ii) ? 1.0 : 0.0;
                        }
                abp::potf2_sweep<true, 4>(pa, pb, sh, tx, ty, col0 + ob, info_b, sweep_phase);
                if (tid < 32) {
                    double s = 0.0;
                    for (int q = tid; q < 64; q += 32) s += 2.0 * log(sdiag[q]);
                    logdet += ab_warp_sum(s);
                }
                double* sDh = half == 0 ? sD11 : sD22;
                const int ldh = half == 0 ? LDC : LDH;
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    const int ii = ty + 16 * r;
                    const double si = sinv[ii];
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        const int kk = tx + 16 * c;
                        double lv = 0.0, dv = 0.0;
                        if (r >= c) {
                            lv = (kk < ii) ? pa[r][c] * sinv[kk] : ((kk == ii) ? sdiag[ii] : 0.0);
                            dv = (kk <= ii) ? pb[r][c] * si : 0.0;
                        }
                        Aj[(int64_t)(ob + ii) * a.ld + ob + kk] = lv;
                        Dj[(ob + ii) * NB + ob + kk] = dv;
                        sDh[ii * ldh + kk] = dv;
                        if (half == 0) {                   // upper-right quadrants of L and L^-1 are zero
                            Aj[(int64_t)ii * a.ld + 64 + kk] = 0.0;
                            Dj[ii * NB + 64 + kk] = 0.0;
                        }
                    }
                }
                __syncthreads();
                if (half == 0) {
                    // L21 = A21 D11^T
                    double acc2[4][2][2];
                    gemm64<true, 1>(acc2, sC + 64 * LDC, LDC, sD11, LDC, warp, lane);
                    __syncthreads();                       // every warp has read A21
#pragma unroll
                    for (int f = 0; f < 4; f++)
#pragma unroll
                        for (int q = 0; q < 2; q++) {
                            const int r = wm64 * 32 + f * 8 + g, c = wn64 * 16 + q * 8 + 2 * t;
                            const double2 v = make_double2(acc2[f][q][0], acc2[f][q][1]);
                            *reinterpret_cast<double2*>(sC + (64 + r) * LDC + c) = v;
                            *reinterpret_cast<double2*>(Aj + (int64_t)(64 + r) * a.ld + c) = v;
                        }
                    __syncthreads();
                    // A22 -= L21 L21^T
                    gemm64<true, 0>(acc2, sC + 64 * LDC, LDC, sC + 64 * LDC, LDC, warp, lane);
#pragma unroll
                    for (int f = 0; f < 4; f++)
#pragma unroll
                        for (int q = 0; q < 2; q++) {
                            const int r = wm64 * 32 + f * 8 + g, c = wn64 * 16 + q * 8 + 2 * t;
                            double2* p = reinterpret_cast<double2*>(sC + (64 + r) * LDC + 64 + c);
                            double2 v = *p;
                            v.x -= acc2[f][q][0];
                            v.y -= acc2[f][q][1];
                            *p = v;
                        }
                    __syncthreads();
                }
            }
            if (tid == 0) logdet_b[j] = logdet;
            {
                // (L^-1)21 = -D22 (L21 D11)
                double acc2[4][2][2];
                gemm64<false, 2>(acc2, sC + 64 * LDC, LDC, sD11, LDC, warp, lane);       // M1 = L21 D11
#pragma unroll
                for (int f = 0; f < 4; f++)
#pragma unroll
                    for (int q = 0; q < 2; q++) {
                        const int r = wm64 * 32 + f * 8 + g, c = wn64 * 16 + q * 8 + 2 * t;
                        *reinterpret_cast<double2*>(sM1 + r * LDH + c) = make_double2(acc2[f][q][0], acc2[f][q][1]);
                    }
                __syncthreads();
                gemm64<false, 3>(acc2, sD22, LDH, sM1, LDH, warp, lane);
#pragma unroll
                for (int f = 0; f < 4; f++)
#pragma unroll
                    for (int q = 0; q < 2; q++) {
                        const int r = wm64 * 32 + f * 8 + g, c = wn64 * 16 + q * 8 + 2 * t;
                        *reinterpret_cast<double2*>(Dj + (64 + r) * NB + c) = make_double2(-acc2[f][q][0], -acc2[f][q][1]);
                    }
            }
        } else {
            // ---- off-diagonal tile: L_ij = C D_j^-T (A operand resident, D_j^-1 streamed) ----
            w.wait(j, j, seen_j);                                    // diagonal tile of column j is final
            const double* Dj = Db + (int64_t)j * NB * NB;
            abg::Acc out;
            out.zero();
            const int cb = (wm == 0) ? wn : 3 - wn;                  // output column block of this warp
            constexpr int NK = NB / Core::BK;
#pragma unroll
            for (int s = 0; s < Core::STAGES - 1; s++) {
                Core::load_operand<true, NB>(sBring + s * BSTAGE, Dj + s * Core::BK, NB, tid);
                abg::cp_async_commit();
            }
            for (int kc = 0; kc < NK; kc++) {
                abg::cp_async_wait<Core::STAGES - 2>();
                __syncthreads();
                const double* sB = sBring + (kc % Core::STAGES) * BSTAGE;
                const int nx = kc + Core::STAGES - 1;
                if (nx < NK) Core::load_operand<true, NB>(sBring + (nx % Core::STAGES) * BSTAGE, Dj + nx * Core::BK, NB, tid);
                abg::cp_async_commit();
                // D_j^-1 is lower triangular: output column c only needs k <= c.  Column blocks
                // are dealt so that the two warps of every scheduler hold blocks cb and 3 - cb
                // (equal work per scheduler); n-fragments are pruned at 8-column granularity.
#pragma unroll
                for (int kk = 0; kk < Core::BK / 4; kk++) {
                    const int k0 = kc * Core::BK + kk * 4;
                    if (k0 > cb * 32 + 31) continue;                 // warp-uniform
                    double fa[8], fb[4];
#pragma unroll
                    for (int f = 0; f < 8; f++) fa[f] = sC[(wm * 64 + f * 8 + g) * LDC + k0 + t];
#pragma unroll
                    for (int f = 0; f < 4; f++) fb[f] = sB[(cb * 32 + f * 8 + g) * Core::LDK + kk * 4 + t];
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        if (k0 > cb * 32 + q * 8 + 7) continue;
#pragma unroll
                        for (int f = 0; f < 8; f++) abg::dmma884(out.v[f][q][0], out.v[f][q][1], fa[f], fb[q]);
                    }
                }
            }
            abg::cp_async_wait<0>();
#pragma unroll
            for (int f = 0; f < 8; f++) {
                const int r = wm * 64 + f * 8 + g;
#pragma unroll
                for (int q = 0; q < 4; q++)
                    *reinterpret_cast<double2*>(Ab + (row0 + r) * a.ld + col0 + cb * 32 + q * 8 + 2 * t) =
                        make_double2(out.v[f][q][0], out.v[f][q][1]);
            }
        }
        // ---- publish: the tile (and D_j^-1) is final -------------------------------------
        __threadfence();
        __syncthreads();
        if (tid == 0) st_release(prog_b + i, j + 1);
    }
}

// Factorisation of `nmat` matrices of T x T tiles (leading dimension T * 128), matrix b at
// A + b * strideA etc. as described at DfArgs.  ctrl: 2 + nmat * T ints ([0] task counter,
// [1] abort word, then prog), zeroed here with the info words; tasks: nmat * T (T + 1) / 2
// entries.  Only the handle's own factor is timed (`profile`).
int launch_dataflow(ab_gp* h, double* A, int64_t strideA, int T, int nmat, double* Dinv, double* logdet_parts,
                    int* info, int* ctrl, const int2* tasks, bool profile) {
    static unsigned long long configured = 0;   // per-device bit: cudaFuncSetAttribute is per device
    if (h->device >= 64 || !((configured >> h->device) & 1ULL)) {
        AB_CUDA(cudaFuncSetAttribute(chol_dataflow_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, DF_SMEM_BYTES));
        if (h->device < 64) configured |= 1ULL << h->device;
    }
    const long long ntasks = (long long)nmat * T * (T + 1) / 2;
    cudaStream_t s = h->stream;
    AB_CUDA(cudaMemsetAsync(ctrl, 0, (2 + (size_t)nmat * T) * sizeof(int), s));
    AB_CUDA(cudaMemsetAsync(info, 0, (size_t)nmat * sizeof(int), s));
    DfArgs a;
    a.A = A; a.ld = (int64_t)T * NB; a.T = T;
    a.Dinv = Dinv; a.logdet_parts = logdet_parts; a.info = info;
    a.next_task = reinterpret_cast<unsigned int*>(ctrl);
    a.abort_flag = ctrl + 1;
    a.prog = ctrl + 2;
    a.tasks = tasks; a.ntasks = (int)ntasks;
    a.strideA = strideA; a.strideD = (int64_t)T * NB * NB;
    const int grid = ntasks < h->nsm ? (int)ntasks : h->nsm;
    if (profile) ab_prof_begin(h, AB_PROF_FACTOR);
    chol_dataflow_kernel<<<grid, Core::THREADS, DF_SMEM_BYTES, s>>>(a);
    if (profile) ab_prof_end(h, AB_PROF_FACTOR);
    ab_count_launches(1);
    AB_CHECK_LAUNCH();
    return 0;
}

}  // namespace

// The handle's factor: L, Dinv and logdet_parts of the handle, d_info; the abort word goes to
// h_pinned[9].  The control block sits in scratch; the task list is cached per size.
int ab_launch_factor_dataflow(ab_gp* h) {
    const int T = (int)(h->npad / NB);
    const int ntasks = T * (T + 1) / 2;
    int rc = ab_ensure_scratch(h, (2 + (size_t)T) * sizeof(int));
    if (rc) return rc;
    if (h->df_tasks_T != T) {                      // column-major task list for this T (host -> device once per size)
        std::vector<int2> tasks;
        tasks.reserve(ntasks);
        for (int j = 0; j < T; j++)
            for (int i = j; i < T; i++) tasks.push_back(make_int2(i, j));
        if (h->df_tasks) cudaFree(h->df_tasks);
        h->df_tasks = nullptr;
        AB_CUDA(cudaMalloc(&h->df_tasks, (size_t)ntasks * sizeof(int2)));
        AB_CUDA(cudaMemcpyAsync(h->df_tasks, tasks.data(), (size_t)ntasks * sizeof(int2), cudaMemcpyHostToDevice, h->stream));
        AB_CUDA(cudaStreamSynchronize(h->stream));
        h->df_tasks_T = T;
    }
    int* ctrl = reinterpret_cast<int*>(h->scratch);
    rc = launch_dataflow(h, h->L, 0, T, 1, h->Dinv, h->logdet_parts, h->d_info, ctrl,
                         reinterpret_cast<const int2*>(h->df_tasks), true);
    if (rc) return rc;
    AB_CUDA(cudaMemcpyAsync(h->h_pinned + 9, ctrl + 1, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    return 0;
}

// Batched factorisation (cv_batch.cu): d_ctrl at least 2 + nmat * T ints, d_tasks filled by
// ab_build_batch_tasks.  Asynchronous on h->stream; the abort word is d_ctrl[1].
int ab_launch_factor_dataflow_batch(ab_gp* h, double* d_A, int64_t strideA, int T, int nmat, double* d_Dinv,
                                    double* d_logdet_parts, int* d_info, int* d_ctrl, const int2* d_tasks) {
    if (T < 1 || T > 4095 || nmat < 1 || nmat >= (1 << 19)) { ab_set_error("batched factorisation: bad shape"); return -1; }
    return launch_dataflow(h, d_A, strideA, T, nmat, d_Dinv, d_logdet_parts, d_info, d_ctrl, d_tasks, false);
}

// task list of a batch: column by column over all matrices (host vector)
void ab_build_batch_tasks(int T, int nmat, std::vector<int2>& tasks) {
    tasks.clear();
    tasks.reserve((size_t)nmat * T * (T + 1) / 2);
    for (int j = 0; j < T; j++)
        for (int b = 0; b < nmat; b++)
            for (int i = j; i < T; i++) tasks.push_back(make_int2(i | (b << 12), j));
}
