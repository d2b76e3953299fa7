// FP64 tensor-core GEMM core for sm_100a: Core<BK, STAGES, ORDER, WM, WN> = a (64 WM) x
// (32 WN) CTA tile (128 x 128 in the product configuration), cp.async multi-stage
// pipeline, DMMA.8x8x4 (mma.sync.m8n8k4.f64) warp tiles of 64x32.  Three main loops:
// mainloop (plain, optional triangular / padded-row pruning), mainloop_gated (operands
// produced by other CTAs of the same kernel), plus the tile store / index helpers.
//
// On sm_100a every f64 mma shape lowers to DMMA.8x8x4 (checked with cuobjdump),
// tcgen05 has no f64 kind, so this warp-level path IS the FP64 tensor pipe.
//
// Each operand tile may be "K-major" (global layout [row][k], k contiguous) or
// "K-strided" (global layout [k][row], row contiguous).  Shared-memory leading
// dimensions are chosen == 4 (mod 16) doubles so that the 16 lanes of a
// half-warp (4 groupIDs x 4 threadID_in_group) hit 16 distinct 8-byte banks.
#pragma once
#include <type_traits>
#include "common.cuh"

namespace abg {

constexpr int BM = 128, BN = 128, THREADS = 256;

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
        : "+d"(c0), "+d"(c1)
        : "d"(a), "d"(b));
}

struct NoGate {
    __device__ __forceinline__ void operator()(int) const {}
};

struct Acc {
    double v[8][4][2];   // [m-frag][n-frag][2]; 64x32 warp tile
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) v[i][j][0] = v[i][j][1] = 0.0;
    }
};

// BK_: k extent of one pipeline stage; STAGES_: cp.async ring depth; ORDER_ = 1
// issues the first k4-step of a chunk BEFORE the prefetch of the next chunk, so
// the tensor pipe is fed right after the barrier.
// WM_ x WN_ warps of 64 x 32 each: CTA tile (64 WM_) x (32 WN_), 32 WM_ WN_ threads
// (2 x 4 = the 128 x 128 tile of the big GEMMs; 1 x 2 = the 64 x 64 tile of the
// Cholesky panel operations, which have too few 128-tiles to fill 148 SMs).
template <int BK_, int STAGES_, int ORDER_, int WM_ = 2, int WN_ = 4>
struct Core {
    static constexpr int BK = BK_, STAGES = STAGES_, WM = WM_, WN = WN_, THREADS = 32 * WM * WN, MF = 8, NF = 4;
    static constexpr int TM = 64 * WM, TN = 32 * WN;
    static constexpr int LDK = BK + 4;            // K-major tile   [rows][BK + 4]
    static constexpr int LDRA = TM + 4, LDRB = TN + 4;   // K-strided tiles [BK][rows + 4]
    static constexpr int A_ELEMS = (TM * LDK > BK * LDRA) ? TM * LDK : BK * LDRA;
    static constexpr int B_ELEMS = (TN * LDK > BK * LDRB) ? TN * LDK : BK * LDRB;
    static constexpr int OPER_ELEMS = A_ELEMS;    // offset of the B operand inside a stage
    static constexpr int STAGE_ELEMS = A_ELEMS + B_ELEMS;
    static constexpr int SMEM_BYTES = STAGES * STAGE_ELEMS * 8;
    static constexpr int KB = 128 / BK;           // chunks per 128-wide k block
    // first row of m-fragment f of warp row wm.  (Warps w and w + 4 share a scheduler and
    // are the two warp rows of one warp column, so contiguous rows already balance a
    // triangular A block across schedulers; interleaving them was measured slower.)
    static __device__ __forceinline__ int frag_row(int wm, int f) { return wm * 64 + f * 8; }
    // mainloop_gated interleaves rows AND columns (see there)
    static __device__ __forceinline__ int gated_row(int wm, int f) { return (f * WM + wm) * 8; }
    using Acc = abg::Acc;
    static_assert(LDK % 16 == 4 && LDRA % 16 == 4 && LDRB % 16 == 4, "leading dimensions must be 4 (mod 16) doubles");
    static_assert(SMEM_BYTES <= 227 * 1024, "pipeline does not fit shared memory");
    static_assert(STAGES >= 2 && STAGES <= 5, "mainloop_gated counts at most STAGES - 1 pending groups");

    // Copy one ROWS x BK operand chunk global -> shared (all threads, 16 B per cp.async).
    template <bool KMAJOR, int ROWS>
    static __device__ __forceinline__ void load_operand(double* s, const double* g, int64_t ld, int tid) {
        constexpr int CHUNKS = ROWS * BK / 2, LDR = ROWS + 4;
        static_assert(CHUNKS % THREADS == 0, "operand chunk count must divide evenly");
        static_assert(LDR % 16 == 4, "K-strided leading dimension must be 4 (mod 16) doubles");
#pragma unroll
        for (int i = 0; i < CHUNKS / THREADS; i++) {
            int c = tid + i * THREADS;
            if (KMAJOR) {
                int row = c / (BK / 2), c16 = c % (BK / 2);
                cp_async16(s + row * LDK + c16 * 2, g + (int64_t)row * ld + c16 * 2);
            } else {
                int k = c / (ROWS / 2), c16 = c % (ROWS / 2);
                cp_async16(s + k * LDR + c16 * 2, g + (int64_t)k * ld + c16 * 2);
            }
        }
    }

    // acc += A_tile(128 x nk*BK) * B_tile(128 x nk*BK)^T.
    //   AK: A is K-major, pointer at element [row0][k0]; else pointer at [k0][row0].
    //   BKM: same for B.
    // All 256 threads must call; smem must hold SMEM_BYTES.  Ends with the pipeline
    // drained and a __syncthreads(), so smem can be reused by the caller.
    //   TRI_A: the last 128-wide k block multiplies a LOWER-TRIANGULAR 128 x 128 A
    //   block (A[r][k] = 0 for k > r): m-fragments whose rows all lie above the
    //   current k4-step are skipped (warp-uniform test).
    //   gate(c) is called by every thread right before it issues the loads of chunk c
    //   (the dataflow Cholesky waits there for the producer of that k block).
    //   MLIM < 16: only the first MLIM 8-row m-fragments of the 128-row A tile matter (the
    //   rest is padding whose products are exactly zero); the per-warp-row fragment counts
    //   are compile-time constants, selected once per chunk by the warp row.
    template <bool AK, bool BKM, bool TRI_A = false, typename Gate = NoGate, int MLIM = 16>
    static __device__ __forceinline__ void mainloop(Acc& acc, const double* __restrict__ A, int64_t lda,
                                                    const double* __restrict__ B, int64_t ldb, int nk,
                                                    double* smem, Gate gate = Gate()) {
        const int tid = threadIdx.x;
        const int lane = tid & 31, warp = tid >> 5;
        const int g = lane >> 2, t = lane & 3;
        const int wm = warp / WN, wn = warp % WN;
        const int64_t a_step = AK ? (int64_t)BK : (int64_t)BK * lda;
        const int64_t b_step = BKM ? (int64_t)BK : (int64_t)BK * ldb;

#pragma unroll
        for (int s = 0; s < STAGES - 1; s++) {
            if (s < nk) {
                gate(s);
                load_operand<AK, TM>(smem + s * STAGE_ELEMS, A + s * a_step, lda, tid);
                load_operand<BKM, TN>(smem + s * STAGE_ELEMS + OPER_ELEMS, B + s * b_step, ldb, tid);
            }
            cp_async_commit();
        }
        for (int kc = 0; kc < nk; kc++) {
            cp_async_wait<STAGES - 2>();
            __syncthreads();
            const double* sA = smem + (kc % STAGES) * STAGE_ELEMS;
            const double* sB = sA + OPER_ELEMS;
            auto prefetch = [&]() {
                int nx = kc + STAGES - 1;
                if (nx < nk) {
                    int st = nx % STAGES;
                    gate(nx);
                    load_operand<AK, TM>(smem + st * STAGE_ELEMS, A + nx * a_step, lda, tid);
                    load_operand<BKM, TN>(smem + st * STAGE_ELEMS + OPER_ELEMS, B + nx * b_step, ldb, tid);
                }
                cp_async_commit();
            };
            if (ORDER_ == 0) prefetch();
            // one k4-step: fragment loads, then 32 DMMAs (TRI: only the m-fragments that
            // reach down to k offset `ktri` of the triangular block)
            auto k4step = [&](int kk, auto tri, int ktri, auto nfc) {
                constexpr int NF = decltype(nfc)::value;             // m-fragments of this warp row that matter
                double a[8], b[4];
#pragma unroll
                for (int f = 0; f < NF; f++)
                    a[f] = AK ? sA[(frag_row(wm, f) + g) * LDK + kk * 4 + t]
                              : sA[(kk * 4 + t) * LDRA + frag_row(wm, f) + g];
#pragma unroll
                for (int f = 0; f < 4; f++)
                    b[f] = BKM ? sB[(wn * 32 + f * 8 + g) * LDK + kk * 4 + t]
                               : sB[(kk * 4 + t) * LDRB + wn * 32 + f * 8 + g];
#pragma unroll
                for (int i = 0; i < NF; i++) {
                    if (decltype(tri)::value && ktri > frag_row(wm, i) + 7) continue;
#pragma unroll
                    for (int j = 0; j < 4; j++) dmma884(acc.v[i][j][0], acc.v[i][j][1], a[i], b[j]);
                }
            };
            auto chunk = [&](auto nfc) {
                if (TRI_A && kc >= nk - KB) {        // chunk inside the triangular diagonal block
                    const int k0 = (kc - (nk - KB)) * BK;
                    if (k0 > frag_row(wm, 7) + 7) {  // nothing left for this warp's rows
                        if (ORDER_ == 1) prefetch();
                    } else {
#pragma unroll
                        for (int kk = 0; kk < BK / 4; kk++) {
                            k4step(kk, std::true_type{}, k0 + kk * 4, nfc);
                            if (ORDER_ == 1 && kk == 0) prefetch();
                        }
                    }
                } else {
#pragma unroll
                    for (int kk = 0; kk < BK / 4; kk++) {
                        k4step(kk, std::false_type{}, -1, nfc);
                        if (ORDER_ == 1 && kk == 0) prefetch();
                    }
                }
            };
            if constexpr (MLIM >= 16 || WM != 2) {
                chunk(std::integral_constant<int, 8>{});
            } else {
                if (wm == 0) chunk(std::integral_constant<int, (MLIM < 8 ? MLIM : 8)>{});
                else chunk(std::integral_constant<int, (MLIM > 8 ? MLIM - 8 : 0)>{});
            }
        }
        cp_async_wait<0>();
        __syncthreads();
    }

    // Main loop for operands that other CTAs are still producing (dataflow Cholesky):
    // gate.ready(c) is a non-blocking test "chunk c may be loaded", gate.wait(c) blocks.
    // Loads run ahead only while the gate is open; the loop blocks only when the chunk
    // it must multiply next has not been issued, i.e. after everything already in
    // shared memory has been consumed.  cp.async groups are counted per thread (one
    // group per chunk), so warps may open the gate at different times.
    // Column mapping differs from mainloop(): n-fragment q of warp column wn covers the
    // 8 columns gated_col(wn, q) = 8 (wn + WN q) (interleaved), so that `lower_only`
    // (a diagonal tile: only columns <= rows matter) halves the work of EVERY warp in
    // the upper row half instead of idling half of them.
    static __device__ __forceinline__ int gated_col(int wn, int q) { return 8 * (wn + WN * q); }

    template <bool AK, bool BKM, typename Gate>
    static __device__ __forceinline__ void mainloop_gated(Acc& acc, const double* __restrict__ A, int64_t lda,
                                                          const double* __restrict__ B, int64_t ldb, int nk,
                                                          double* smem, Gate& gate, bool lower_only) {
        const int tid = threadIdx.x;
        const int lane = tid & 31, warp = tid >> 5;
        const int g = lane >> 2, t = lane & 3;
        const int wm = warp / WN, wn = warp % WN;
        const int64_t a_step = AK ? (int64_t)BK : (int64_t)BK * lda;
        const int64_t b_step = BKM ? (int64_t)BK : (int64_t)BK * ldb;
        static_assert(WN == 4 && TN == 128, "gated column interleave assumes 4 warp columns of 32");
        // rows and columns are both interleaved: m-fragment i holds rows 16 i + 8 wm, n-fragment q
        // columns 32 q + 8 wn.  For a diagonal tile only (i, q) with 32 q <= 16 i + 15 matter.
        const bool skip_upper = lower_only;
        int issued = 0;
        auto issue = [&](int c) {
            const int st = c % STAGES;
            load_operand<AK, TM>(smem + st * STAGE_ELEMS, A + c * a_step, lda, tid);
            load_operand<BKM, TN>(smem + st * STAGE_ELEMS + OPER_ELEMS, B + c * b_step, ldb, tid);
            cp_async_commit();
            issued = c + 1;
        };
        for (int kc = 0; kc < nk; kc++) {
            if (issued <= kc) {
                gate.wait(kc);
                issue(kc);
            }
            switch (issued - kc - 1) {                 // groups younger than chunk kc's
                case 0: cp_async_wait<0>(); break;
                case 1: cp_async_wait<1>(); break;
                case 2: cp_async_wait<2>(); break;
                default: cp_async_wait<STAGES - 2>(); break;
            }
            __syncthreads();
            const double* sA = smem + (kc % STAGES) * STAGE_ELEMS;
            const double* sB = sA + OPER_ELEMS;
#pragma unroll
            for (int kk = 0; kk < BK / 4; kk++) {
                double a[8], b[4];
#pragma unroll
                for (int f = 0; f < 8; f++)
                    a[f] = AK ? sA[(gated_row(wm, f) + g) * LDK + kk * 4 + t]
                              : sA[(kk * 4 + t) * LDRA + gated_row(wm, f) + g];
#pragma unroll
                for (int f = 0; f < 4; f++)
                    b[f] = BKM ? sB[(gated_col(wn, f) + g) * LDK + kk * 4 + t]
                               : sB[(kk * 4 + t) * LDRB + gated_col(wn, f) + g];
                if (skip_upper) {                      // diagonal tile: fragments strictly above the diagonal are skipped
#pragma unroll
                    for (int i = 0; i < 8; i++)
#pragma unroll
                        for (int j = 0; j < 4; j++)
                            if (32 * j <= 16 * i + 15) dmma884(acc.v[i][j][0], acc.v[i][j][1], a[i], b[j]);
                } else {
#pragma unroll
                    for (int i = 0; i < 8; i++)
#pragma unroll
                        for (int j = 0; j < 4; j++) dmma884(acc.v[i][j][0], acc.v[i][j][1], a[i], b[j]);
                }
                if (kk == 0) {
                    // slot of chunk nx held chunk nx - STAGES, consumed before this iteration's barrier
                    while (issued < nk && issued < kc + STAGES && gate.ready(issued)) issue(issued);
                }
            }
        }
        cp_async_wait<0>();
        __syncthreads();
    }

    // Element (row, col) owned by acc.v[i][j][e] inside the CTA tile.
    static __device__ __forceinline__ int acc_row(int i) {
        int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        return frag_row(warp / WN, i) + (lane >> 2);
    }
    static __device__ __forceinline__ int acc_col(int j) {
        int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        return (warp % WN) * 32 + j * 8 + (lane & 3) * 2;   // + e
    }

    // C[tile] = alpha * acc + beta * C[tile]   (C row-major, 16-byte vector accesses)
    static __device__ __forceinline__ void store_tile(const Acc& acc, double* __restrict__ C, int64_t ldc,
                                                      double alpha, double beta) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            int r = acc_row(i);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                double2* p = reinterpret_cast<double2*>(C + (int64_t)r * ldc + acc_col(j));
                double2 o;
                if (beta != 0.0) {
                    double2 c = *p;
                    o.x = alpha * acc.v[i][j][0] + beta * c.x;
                    o.y = alpha * acc.v[i][j][1] + beta * c.y;
                } else {
                    o.x = alpha * acc.v[i][j][0];
                    o.y = alpha * acc.v[i][j][1];
                }
                *p = o;
            }
        }
    }
};

// configuration used by the product kernels
using Main = Core<16, 4, 1>;            // 128 x 128 tile, 256 threads, 160 KB
constexpr int BK = Main::BK, STAGES = Main::STAGES;
constexpr int SMEM_BYTES = Main::SMEM_BYTES;

template <bool AK, bool BKM, bool TRI_A = false>
__device__ __forceinline__ void mainloop(Acc& acc, const double* __restrict__ A, int64_t lda,
                                         const double* __restrict__ B, int64_t ldb, int nk, double* smem) {
    Main::mainloop<AK, BKM, TRI_A>(acc, A, lda, B, ldb, nk, smem);
}

__device__ __forceinline__ int acc_row(int i) { return Main::acc_row(i); }
__device__ __forceinline__ int acc_col(int j) { return Main::acc_col(j); }
__device__ __forceinline__ void store_tile(const Acc& acc, double* __restrict__ C, int64_t ldc, double alpha, double beta) {
    Main::store_tile(acc, C, ldc, alpha, beta);
}

// linear index p -> (i, j) with 0 <= j <= i  (row-major lower triangle)
__device__ __forceinline__ void tri_decode(int p, int& i, int& j) {
    int r = (int)((sqrtf(8.0f * (float)p + 1.0f) - 1.0f) * 0.5f);
    while ((r + 1) * (r + 2) / 2 <= p) r++;
    while (r * (r + 1) / 2 > p) r--;
    i = r;
    j = p - r * (r + 1) / 2;
}

}  // namespace abg
