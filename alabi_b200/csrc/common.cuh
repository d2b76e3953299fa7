// Shared device/host helpers for the alabi_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <type_traits>

#define AB_MAX_DIM 32     // maximum input dimension (per-dimension metric)
#define AB_NB 128         // block size of every blocked dense algorithm; matrices are padded to it

#if defined(__CUDA_ARCH__) && !defined(__CUDA_ARCH_FEAT_SM100_ALL)
#error "alabi_b200 kernels are written for sm_100a (compile with -gencode arch=compute_100a,code=sm_100a)"
#endif

// Stationary kernel with an axis-aligned metric.  Coordinates are pre-scaled by
// 1/sqrt(M_k) so r^2 is a plain squared distance (george: r^2 = sum dx_k^2 / M_k;
// reference call site alabi/core.py:998-1014).
struct KernParams {
    int kind;                     // 0 ExpSquared, 1 Matern32, 2 Matern52, 3 RationalQuadratic
    int d;
    double amp;                   // exp(log_constant), 1 without an amplitude
    double diag_add;              // yerr^2 + exp(white_noise)
    double inv_len[AB_MAX_DIM];   // exp(-0.5 log_M_k)
    double alpha;                 // RationalQuadratic: exp(log_alpha); 0 for kinds 0-2
    double inv2a;                 // RationalQuadratic: 1 / (2 alpha); 0 for kinds 0-2
};

// 2^(j/64), j = 0..63, correctly rounded (global memory, L1 resident: 512 B)
static __device__ const double ab_exp2_tab[64] = {
    0x1.0000000000000p+0, 0x1.02c9a3e778061p+0, 0x1.059b0d3158574p+0, 0x1.0874518759bc8p+0,
    0x1.0b5586cf9890fp+0, 0x1.0e3ec32d3d1a2p+0, 0x1.11301d0125b51p+0, 0x1.1429aaea92de0p+0,
    0x1.172b83c7d517bp+0, 0x1.1a35beb6fcb75p+0, 0x1.1d4873168b9aap+0, 0x1.2063b88628cd6p+0,
    0x1.2387a6e756238p+0, 0x1.26b4565e27cddp+0, 0x1.29e9df51fdee1p+0, 0x1.2d285a6e4030bp+0,
    0x1.306fe0a31b715p+0, 0x1.33c08b26416ffp+0, 0x1.371a7373aa9cbp+0, 0x1.3a7db34e59ff7p+0,
    0x1.3dea64c123422p+0, 0x1.4160a21f72e2ap+0, 0x1.44e086061892dp+0, 0x1.486a2b5c13cd0p+0,
    0x1.4bfdad5362a27p+0, 0x1.4f9b2769d2ca7p+0, 0x1.5342b569d4f82p+0, 0x1.56f4736b527dap+0,
    0x1.5ab07dd485429p+0, 0x1.5e76f15ad2148p+0, 0x1.6247eb03a5585p+0, 0x1.6623882552225p+0,
    0x1.6a09e667f3bcdp+0, 0x1.6dfb23c651a2fp+0, 0x1.71f75e8ec5f74p+0, 0x1.75feb564267c9p+0,
    0x1.7a11473eb0187p+0, 0x1.7e2f336cf4e62p+0, 0x1.82589994cce13p+0, 0x1.868d99b4492edp+0,
    0x1.8ace5422aa0dbp+0, 0x1.8f1ae99157736p+0, 0x1.93737b0cdc5e5p+0, 0x1.97d829fde4e50p+0,
    0x1.9c49182a3f090p+0, 0x1.a0c667b5de565p+0, 0x1.a5503b23e255dp+0, 0x1.a9e6b5579fdbfp+0,
    0x1.ae89f995ad3adp+0, 0x1.b33a2b84f15fbp+0, 0x1.b7f76f2fb5e47p+0, 0x1.bcc1e904bc1d2p+0,
    0x1.c199bdd85529cp+0, 0x1.c67f12e57d14bp+0, 0x1.cb720dcef9069p+0, 0x1.d072d4a07897cp+0,
    0x1.d5818dcfba487p+0, 0x1.da9e603db3285p+0, 0x1.dfc97337b9b5fp+0, 0x1.e502ee78b3ff6p+0,
    0x1.ea4afa2a490dap+0, 0x1.efa1bee615a27p+0, 0x1.f50765b6e4540p+0, 0x1.fa7c1819e90d8p+0};

// Branch-free FP64 exp(x) for x <= 0 (the only arguments the kernels produce):
// n = rint(64 x / ln 2) = 64 m + j, r = x - n ln2/64 (Cody-Waite, |r| <= 0.0055),
// exp(x) = 2^m 2^(j/64) (1 + r + r^2/2 + .. + r^5/120)  (remainder 4e-17): ten FP64
// instructions and one L1 table load.  Relative error about 1 ulp; exp(x) < 1e-307
// flushes to 0.  No slow-path call, no divergence.
__device__ __forceinline__ double ab_exp_neg(double x) {
    const double SHIFT = 6755399441055744.0;                 // 1.5 * 2^52
    const double t = fma(x, 92.33248261689366, SHIFT);       // 64 / ln 2
    const int n = __double2loint(t);
    const double nf = t - SHIFT;
    double r = fma(nf, -0x1.62e42fee00000p-7, x);            // ln2/64, high part (32 bits)
    r = fma(nf, -0x1.a39ef35793c76p-39, r);                  // low part
    double q = fma(r, 8.3333333333333332e-03, 4.1666666666666664e-02);
    q = fma(q, r, 1.6666666666666666e-01);
    q = fma(q, r, 0.5);
    q = fma(q, r, 1.0);
    q *= r;
    const double tj = __ldg(&ab_exp2_tab[n & 63]);
    const double p = fma(tj, q, tj);
    const double res = __hiloint2double(__double2hiint(p) + ((n >> 6) << 20), __double2loint(p));
    // x > -707 (x <= 0) as an integer compare of the high word of |x| (707.0 = 0x4086180000000000): no
    // FP64 issue slot; NaN compares false, as before
    return ((__double2hiint(x) & 0x7fffffff) < 0x40861800) ? res : 0.0;
}

// exp(-r2 / 2) for r2 >= 0 with the SAME bits as ab_exp_neg(-0.5 * r2), two FP64 issue slots cheaper
// (the squared-exponential kernel of K1 / K3 / K5: 53 -> 51 FP64 instructions per evaluation at d = 20).
// The factor -1/2 moves into the constants: t = r2 (-32 / ln 2) + SHIFT is the same product; the
// reduced argument is carried as u = -2 r = r2 + nf (2 ln2 / 64) (exact, like r), and the Horner
// coefficients absorb (-1/2)^k, so every intermediate is the old one times a power of two and the
// final product q u equals the old q r bit for bit (no rounding differs under power-of-two scaling).
__device__ __forceinline__ double ab_exp_neg_half(double r2) {
    const double SHIFT = 6755399441055744.0;                 // 1.5 * 2^52
    const double t = fma(r2, -46.16624130844683, SHIFT);     // -32 / ln 2 = -0.5 * 92.33248261689366
    const int n = __double2loint(t);
    const double nf = t - SHIFT;
    double u = fma(nf, 0x1.62e42fee00000p-6, r2);            // 2 * ln2/64, high part
    u = fma(nf, 0x1.a39ef35793c76p-38, u);                   // low part
    double q = fma(u, -8.3333333333333332e-03 * 0.03125, 4.1666666666666664e-02 * 0.0625);
    q = fma(q, u, -1.6666666666666666e-01 * 0.125);
    q = fma(q, u, 0.125);
    q = fma(q, u, -0.5);
    q *= u;
    const double tj = __ldg(&ab_exp2_tab[n & 63]);
    const double p = fma(tj, q, tj);
    const double res = __hiloint2double(__double2hiint(p) + ((n >> 6) << 20), __double2loint(p));
    // r2 < 1414 (= 0x4096180000000000), i.e. -r2/2 > -707; NaN compares false
    return ((__double2hiint(r2) & 0x7fffffff) < 0x40961800) ? res : 0.0;
}

// Table-free variant of ab_exp_neg for kernels with few resident warps (cov, gradient
// tiles), where the L1 latency of the table load is not hidden:
// n = rint(x log2 e), f = x - n ln2 (Cody-Waite), degree-13 Taylor on |f| <= 0.347
// (remainder 4e-18), scaling by 2^n through the exponent field; exp(x) < 1e-307
// flushes to 0.  Relative error ~2e-16, no slow-path call, no divergence.
__device__ __forceinline__ double ab_exp_neg_poly(double x) {
    const double SHIFT = 6755399441055744.0;                 // 1.5 * 2^52
    double t = fma(x, 1.4426950408889634, SHIFT);
    int n = __double2loint(t);
    double nf = t - SHIFT;
    double f = fma(nf, -6.93147180369123816490e-01, x);
    f = fma(nf, -1.90821492927058770002e-10, f);
    double p = 1.6059043836821613e-10;                       // 1/13!
    p = fma(p, f, 2.0876756987868100e-09);                   // 1/12!
    p = fma(p, f, 2.5052108385441720e-08);                   // 1/11!
    p = fma(p, f, 2.7557319223985893e-07);                   // 1/10!
    p = fma(p, f, 2.7557319223985888e-06);                   // 1/9!
    p = fma(p, f, 2.4801587301587302e-05);                   // 1/8!
    p = fma(p, f, 1.9841269841269841e-04);                   // 1/7!
    p = fma(p, f, 1.3888888888888889e-03);                   // 1/6!
    p = fma(p, f, 8.3333333333333332e-03);                   // 1/5!
    p = fma(p, f, 4.1666666666666664e-02);                   // 1/4!
    p = fma(p, f, 1.6666666666666666e-01);                   // 1/3!
    p = fma(p, f, 0.5);
    p = fma(p, f, 1.0);
    p = fma(p, f, 1.0);
    double r = __hiloint2double(__double2hiint(p) + (n << 20), __double2loint(p));
    return ((__double2hiint(x) & 0x7fffffff) < 0x40861800) ? r : 0.0;   // x > -707 (x <= 0), integer compare; NaN -> 0
}

// Branch-free sqrt(x) for finite x >= 0: MUFU.RSQ64H seed, two Newton steps on
// 1/sqrt, one correction of the root (<= 1 ulp); x < 1e-290 returns 0.
__device__ __forceinline__ double ab_sqrt_pos(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    const double hx = 0.5 * x;
    double e = fma(-hx * y, y, 0.5);
    y = fma(y, e, y);
    e = fma(-hx * y, y, 0.5);
    y = fma(y, e, y);
    double s = x * y;
    s = fma(0.5 * y, fma(-s, s, x), s);
    return (x > 1e-290) ? s : 0.0;
}

// TAB = true: table-based exp (fewest FP64 instructions; needs enough resident warps to
// hide one L1 load), false: polynomial-only exp.  Both are ~1 ulp.
template <bool TAB>
__device__ __forceinline__ double ab_exp_sel(double x) { return TAB ? ab_exp_neg(x) : ab_exp_neg_poly(x); }
// exp(-r2 / 2), r2 >= 0
template <bool TAB>
__device__ __forceinline__ double ab_exp_half_sel(double r2) { return TAB ? ab_exp_neg_half(r2) : ab_exp_neg_poly(-0.5 * r2); }

// The radial profiles k(r^2).  alpha and inv2a = 1 / (2 alpha) are read by the rational quadratic
// kernel (KIND 3) only, k = (1 + r^2 / (2 alpha))^(-alpha) = exp(-alpha log1p(x)), x = r^2 inv2a;
// kinds 0-2 ignore them.
template <int KIND, bool TAB = true>
__device__ __forceinline__ double ab_radial(double r2, double alpha, double inv2a) {
    if (KIND == 0) return ab_exp_half_sel<TAB>(r2);
    if (KIND == 1) { double r = ab_sqrt_pos(3.0 * r2); return (1.0 + r) * ab_exp_sel<TAB>(-r); }
    if (KIND == 3) return ab_exp_sel<TAB>(-alpha * log1p(r2 * inv2a));
    double r = ab_sqrt_pos(5.0 * r2);
    return (1.0 + r + r * r * 0.3333333333333333) * ab_exp_sel<TAB>(-r);
}

// dk/d(r^2)
template <int KIND, bool TAB = true>
__device__ __forceinline__ double ab_radial_grad(double r2, double alpha, double inv2a) {
    if (KIND == 0) return -0.5 * ab_exp_half_sel<TAB>(r2);
    if (KIND == 1) { double r = ab_sqrt_pos(3.0 * r2); return -1.5 * ab_exp_sel<TAB>(-r); }
    if (KIND == 3) {
        const double x = r2 * inv2a;
        return -0.5 * ab_exp_sel<TAB>(-alpha * log1p(x)) / (1.0 + x);
    }
    double r = ab_sqrt_pos(5.0 * r2);
    return -5.0 * (1.0 + r) * ab_exp_sel<TAB>(-r) * 0.16666666666666666;
}

// g(x) = log1p(x) - x / (1 + x) >= 0 for x >= 0, the rational quadratic kernel's dk/dlog(alpha) =
// -alpha k g(x).  For small x the two terms cancel: evaluated directly, g's relative error is about
// 5 eps / x (log1p and the quotient each carry ~1 ulp of a number ~x, g ~ x^2 / 2), which is total
// for x < eps.  Below x = 1/16 the alternating series g = sum_{n>=2} (-1)^n (n-1)/n x^n is used
// instead: through x^15 its truncation is below 2 (15/16) x^14 ~ 3e-17 relative at x = 1/16, and
// the direct form's error at the switch is <= 80 eps ~ 2e-14 relative.  inv1px = 1 / (1 + x).
__device__ __forceinline__ double ab_rq_g(double x, double l, double inv1px) {
    double p = -0.93333333333333333;                   // -14/15 (x^15)
    p = fma(p, x, 0.92857142857142857);                // 13/14
    p = fma(p, x, -0.92307692307692308);               // -12/13
    p = fma(p, x, 0.91666666666666667);                // 11/12
    p = fma(p, x, -0.90909090909090909);               // -10/11
    p = fma(p, x, 0.9);                                // 9/10
    p = fma(p, x, -0.88888888888888889);               // -8/9
    p = fma(p, x, 0.875);                              // 7/8
    p = fma(p, x, -0.85714285714285714);               // -6/7
    p = fma(p, x, 0.83333333333333333);                // 5/6
    p = fma(p, x, -0.8);                               // -4/5
    p = fma(p, x, 0.75);                               // 3/4
    p = fma(p, x, -0.66666666666666667);               // -2/3
    p = fma(p, x, 0.5);                                // 1/2 (x^2)
    const double series = p * x * x;
    return (x < 0.0625) ? series : l - x * inv1px;
}

// k(r^2) and dk/d(r^2) from ONE exponential (the gradient kernels need both); for the rational
// quadratic kernel also av = dk/dlog(alpha) = -alpha k g(x), from the same log1p and exponential and
// one reciprocal (kinds 0-2 set av = 0)
template <int KIND, bool TAB = true>
__device__ __forceinline__ void ab_radial_both(double r2, double alpha, double inv2a, double& kv, double& gv,
                                               double& av) {
    av = 0.0;
    if (KIND == 0) {
        const double e = ab_exp_half_sel<TAB>(r2);
        kv = e; gv = -0.5 * e;
    } else if (KIND == 1) {
        const double r = ab_sqrt_pos(3.0 * r2), e = ab_exp_sel<TAB>(-r);
        kv = (1.0 + r) * e; gv = -1.5 * e;
    } else if (KIND == 3) {
        const double x = r2 * inv2a, l = log1p(x), e = ab_exp_sel<TAB>(-alpha * l);
        const double inv1px = 1.0 / (1.0 + x);
        kv = e; gv = -0.5 * e * inv1px; av = -alpha * e * ab_rq_g(x, l, inv1px);
    } else {
        const double r = ab_sqrt_pos(5.0 * r2), e = ab_exp_sel<TAB>(-r);
        kv = (1.0 + r + r * r * 0.3333333333333333) * e; gv = -5.0 * (1.0 + r) * e * 0.16666666666666666;
    }
}

// The input dimensions the kernels are compiled for.  A kernel templated on D handles d <= D only
// (coordinates past D would be dropped), so every launcher picks D here.
inline int ab_padded_dim(int d) {
    return d <= 2 ? 2 : d <= 4 ? 4 : d <= 8 ? 8 : d <= 12 ? 12 : d <= 16 ? 16 : d <= 20 ? 20 : d <= 24 ? 24 : 32;
}

// f(std::integral_constant<int, D>{}) for the padded dimension D of d
template <class F>
auto ab_dispatch_dim(int d, F&& f) {
    switch (ab_padded_dim(d)) {
        case 2: return f(std::integral_constant<int, 2>{});
        case 4: return f(std::integral_constant<int, 4>{});
        case 8: return f(std::integral_constant<int, 8>{});
        case 12: return f(std::integral_constant<int, 12>{});
        case 16: return f(std::integral_constant<int, 16>{});
        case 20: return f(std::integral_constant<int, 20>{});
        case 24: return f(std::integral_constant<int, 24>{});
        default: return f(std::integral_constant<int, 32>{});
    }
}

// Shared memory the samplers give a training set they keep resident: n points of D padded coordinates
// plus alpha.  A set within the budget is loaded once per run; a larger one is streamed in chunks.
constexpr size_t AB_RESIDENT_SMEM = 160 * 1024;
inline bool ab_resident(long long n, int D) { return (size_t)n * (D + 1) * 8 <= AB_RESIDENT_SMEM; }

#define AB_DISPATCH_KIND(kind, ...)                                   \
    do {                                                              \
        if ((kind) == 0) { constexpr int KIND = 0; __VA_ARGS__; }     \
        else if ((kind) == 1) { constexpr int KIND = 1; __VA_ARGS__; }\
        else if ((kind) == 2) { constexpr int KIND = 2; __VA_ARGS__; }\
        else { constexpr int KIND = 3; __VA_ARGS__; }                 \
    } while (0)

__device__ __forceinline__ double ab_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// error plumbing (api.cu owns the storage)
void ab_set_error(const char* fmt, ...);
#define AB_CUDA(call)                                                             \
    do {                                                                          \
        cudaError_t e_ = (call);                                                  \
        if (e_ != cudaSuccess) {                                                  \
            ab_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return -100 - (int)e_;                                                \
        }                                                                         \
    } while (0)
#define AB_CHECK_LAUNCH() AB_CUDA(cudaGetLastError())
