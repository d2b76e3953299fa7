// Diagonal-block step of the blocked Cholesky: factor an SPD block and invert the
// factor, in ONE register-tiled sweep by a single CTA (the diagonal tasks of
// chol_dataflow.cu; chol.cu's potf2_inv_kernel runs it on an existing factor).
//
// 256 threads form a 16 x 16 grid; thread (ty, tx) owns the 8 x 8 cyclic
// sub-matrix rows {ty + 16 r}, columns {tx + 16 c} of both A (-> L) and B
// (identity -> L^-1) in registers.  Step j broadcasts column j of A and row j of
// B through shared memory (one __syncthreads per step, double buffered) and
// every thread applies the two rank-1 updates
//      A[i][k] -= A[i][j] A[k][j] / p_j          (j < k <= i)
//      B[i][c] -= A[i][j] B[j][c] / p_j          (c <= j < i)
// Columns/rows are scaled by 1/sqrt(p_j) only at the end, so the sweep has no
// second dependent phase.  The outer loop over j / 16 is unrolled so that all
// register-array indices are static and the triangular structure prunes work at
// compile time.
#pragma once
#include <type_traits>
#include "common.cuh"

namespace abp {

constexpr int NB = AB_NB;

// 1/x to ~1 ulp: MUFU.RCP64H seed + two Newton steps (no slow-path call on the
// critical path of the column sweep; x is a positive pivot here)
__device__ __forceinline__ double fast_rcp(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    return r;
}

// split-phase CTA barrier in shared memory (mbarrier): threads arrive right after
// they have published the next pivot column and wait only when they need it
__device__ __forceinline__ void mbar_init(unsigned addr, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(addr), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned addr) {
    asm volatile("{ .reg .b64 st; mbarrier.arrive.shared::cta.b64 st, [%0]; }" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned addr, unsigned parity) {
    unsigned ok;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
    } while (!ok);
}

struct SweepShared {
    double colA[2][NB], rowB[2][NB], sdiag[NB], sinv[NB];
    unsigned long long mbar;          // initialised once per kernel with count = 256
};

// One column step with in-kernel look-ahead.  Column j = 16 JR + jm was published
// (into buffer j & 1) during step j - 1; this step first applies its update to
// column j + 1 of A and row j + 1 of B (block index JRN), publishes them and
// arrives on the barrier, and only then applies the bulk of the rank-1 updates,
// so the barrier / shared-memory / reciprocal latency of step j + 1 is hidden
// behind the bulk of step j.  JRN == 8: last column, nothing to publish.
template <bool FACTOR, int R, int JR, int JRN>
__device__ __forceinline__ void potf2_step(double (&a)[R][R], double (&b)[R][R], SweepShared& sh, int jm, int tx,
                                           int ty, int64_t o, int* info, unsigned mbar, unsigned& phase) {
    const int j = JR * 16 + jm, buf = jm & 1;
    mbar_wait(mbar, phase & 1u);
    phase++;
    double p = sh.colA[buf][j];
    if (FACTOR && !(p > 0.0)) {                 // LAPACK dpotrf: ajj <= 0 or NaN -> info = j + 1
        if (tx == 0 && ty == 0) atomicCAS(info, 0, (int)(o + j + 1));
        p = 1.0;
    }
    if (tx == 0 && ty == 0) sh.sdiag[j] = p;    // sqrt / reciprocal of the pivots: after the sweep
    const double ip = fast_rcp(p);
    // everything this step reads from shared memory, before the arrive (the buffer is
    // rewritten by step j + 1 of a faster thread only after every thread has arrived).
    // The triangular structure is enforced by zeroing OPERANDS, not by predicating the
    // FMAs: valid entries (A: i >= k > j, B: c <= j < i) only ever consume valid
    // entries; entries outside those regions may hold garbage and are never read back.
    double ai[R], ak[R], xk[R];
#pragma unroll
    for (int r = JR; r < R; r++) ai[r] = sh.colA[buf][ty + 16 * r];
    if (FACTOR) {
#pragma unroll
        for (int c = JR; c < R; c++) ak[c] = sh.colA[buf][tx + 16 * c] * ip;
        ak[JR] = (tx > jm) ? ak[JR] : 0.0;                      // columns k <= j are final
    }
#pragma unroll
    for (int c = 0; c <= JR; c++) xk[c] = sh.rowB[buf][tx + 16 * c] * ip;
    xk[JR] = (tx <= jm) ? xk[JR] : 0.0;                         // B[j][c] = 0 for c > j
    const double ab_jr = (ty > jm) ? ai[JR] : 0.0;              // rows i <= j of B are final

    if (JRN < R) {
        constexpr int N = JRN < R ? JRN : R - 1;
        const int jn = (JRN == JR) ? jm + 1 : 0;
        if (FACTOR) {
#pragma unroll
            for (int r = N; r < R; r++) a[r][N] = fma(-ai[r], ak[N], a[r][N]);
        }
        if (tx == jn) {
#pragma unroll
            for (int r = N; r < R; r++) sh.colA[buf ^ 1][ty + 16 * r] = a[r][N];
        }
#pragma unroll
        for (int c = 0; c <= JR; c++) b[N][c] = fma(-(N == JR ? ab_jr : ai[N]), xk[c], b[N][c]);
        if (ty == jn) {
#pragma unroll
            for (int c = 0; c <= N; c++) sh.rowB[buf ^ 1][tx + 16 * c] = b[N][c];
        }
        mbar_arrive(mbar);
    }
    if (FACTOR) {
#pragma unroll
        for (int c = JR; c < R; c++)
            if (c != JRN) {
#pragma unroll
                for (int r = c; r < R; r++) a[r][c] = fma(-ai[r], ak[c], a[r][c]);
            }
    }
#pragma unroll
    for (int r = JR; r < R; r++)
        if (r != JRN) {
#pragma unroll
            for (int c = 0; c <= JR; c++) b[r][c] = fma(-(r == JR ? ab_jr : ai[r]), xk[c], b[r][c]);
        }
}

template <bool FACTOR, int R, int JR>
__device__ __forceinline__ void sweep16(double (&a)[R][R], double (&b)[R][R], SweepShared& sh, int tx, int ty,
                                        int64_t o, int* info, unsigned mbar, unsigned& phase) {
    for (int jm = 0; jm < 15; jm++) potf2_step<FACTOR, R, JR, JR>(a, b, sh, jm, tx, ty, o, info, mbar, phase);
    potf2_step<FACTOR, R, JR, JR + 1>(a, b, sh, 15, tx, ty, o, info, mbar, phase);
    if constexpr (JR + 1 < R) sweep16<FACTOR, R, JR + 1>(a, b, sh, tx, ty, o, info, mbar, phase);
}

// Whole 16 R-column sweep on the register-tiled block (a: block -> unscaled L columns,
// b: identity -> unscaled L^-1 rows); R = 8: 128 x 128, R = 4: 64 x 64 (same 16 x 16
// thread grid, R x R cyclic entries per thread).  On return sh.sdiag = diag(L),
// sh.sinv = 1 / diag(L) (after a __syncthreads inside).  All 256 threads; `phase` is
// the running count of completed barrier phases of sh.mbar (kept by the caller).
template <bool FACTOR, int R = 8>
__device__ __forceinline__ void potf2_sweep(double (&a)[R][R], double (&b)[R][R], SweepShared& sh, int tx, int ty,
                                            int64_t o, int* info, unsigned& phase) {
    const unsigned mbar = (unsigned)__cvta_generic_to_shared(&sh.mbar);
    // publish column 0 of A and row 0 of B
    if (tx == 0) {
#pragma unroll
        for (int r = 0; r < R; r++) sh.colA[0][ty + 16 * r] = a[r][0];
    }
    if (ty == 0) sh.rowB[0][tx] = b[0][0];
    mbar_arrive(mbar);
    sweep16<FACTOR, R, 0>(a, b, sh, tx, ty, o, info, mbar, phase);
    __syncthreads();
    if (threadIdx.x < 16 * R) {                       // pivots -> diagonal of L and its reciprocal
        const double dj = FACTOR ? sqrt(sh.sdiag[threadIdx.x]) : sh.sdiag[threadIdx.x];
        sh.sdiag[threadIdx.x] = dj;
        sh.sinv[threadIdx.x] = 1.0 / dj;
    }
    __syncthreads();
}

}  // namespace abp
