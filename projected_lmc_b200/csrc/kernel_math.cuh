// Stationary kernel profiles k(s) and dk/ds as functions of the squared scaled distance s (gpytorch 1.11
// RBFKernel / MaternKernel / RQKernel semantics, reached from handle_covar_, projected_lmc.py:151-167):
//   RBF exp(-s/2);  Matern: r = sqrt(max(s, 1e-30)),  nu=5/2 (1 + sqrt5 r + 5/3 r^2) exp(-sqrt5 r),
//   nu=3/2 (1 + sqrt3 r) exp(-sqrt3 r),  nu=1/2 exp(-r);  RQ (1 + s / (2 alpha))^-alpha, alpha per latent.
//
// The Gram build and the gradient sweep are bound by the FP64 instruction rate of the transform, not by HBM
// (ncu, profiles/r02_ncu_summary.md: 141 instructions per Gram entry with libdevice's exp/sqrt, FP64 pipe 26 %
// active, issue slots 51 %).  exp and sqrt are therefore written out for the argument ranges that occur here:
//   * exp(x), x <= 0:  n = rint(x 32/ln2), r = x - n ln2/32 (two-term Cody-Waite, |r| <= 0.0109),
//     e^r - 1 by a degree-6 polynomial (remainder 3e-18), times the table value 2^(j/32), j = n mod 32, exponent
//     n div 32 added to the exponent field: 13 FP64 instructions, 1 L1-resident load, < 1 ulp (checked against
//     libm on the host by tests/test_kernel_math_cpu.py);
//   * sqrt(s), s >= 1e-30:  MUFU.RSQ64H seed (rsqrt.approx.ftz.f64) and two coupled Newton steps (Goldschmidt form)
//     plus one residual correction: 9 FP64 instructions, <= 1 ulp.
// The same code compiles for the host (seed from float rsqrt) so that the accuracy claims are tested without a GPU.
#pragma once
#include "plmc_common.cuh"

#include <cmath>
#include <cstring>

namespace plmc {

// max(a, b) for non-NaN arguments.  fmax() on doubles has no hardware instruction on sm_100a: it expands to
// DSETP.MAX + SEL + FSEL + a NaN-quieting LOP3 per half (~7 instructions, ncu source page of gram_kernel); a
// compare-and-select is 3.
__host__ __device__ __forceinline__ double dmax(double a, double b) { return (a > b) ? a : b; }

#define PLMC_EXP_TABLE                                                                                                \
    {1.0, 1.0218971486541166, 1.0442737824274138, 1.0671404006768237, 1.0905077326652577, 1.1143867425958924,         \
     1.1387886347566916, 1.1637248587775775, 1.189207115002721, 1.215247359980469, 1.241857812073484,                 \
     1.2690509571917332, 1.2968395546510096, 1.3252366431597413, 1.3542555469368927, 1.383909881963832,               \
     1.4142135623730951, 1.4451808069770467, 1.4768261459394993, 1.5091644275934228, 1.5422108254079407,              \
     1.5759808451078865, 1.6104903319492543, 1.645755478153965, 1.681792830507429, 1.718619298122478,                 \
     1.7562521603732995, 1.7947090750031072, 1.8340080864093424, 1.8741676341103, 1.9152065613971474,                 \
     1.9571441241754002}

// device copy in GLOBAL memory, read with __ldg: the index differs between the lanes of a warp, which a __constant__
// bank would serialise; the 256-byte table is two L1 lines
static __device__ const double d_exp_table[32] = PLMC_EXP_TABLE;
static const double h_exp_table[32] = PLMC_EXP_TABLE;

// exp(x) for x <= 0 (x > 0 is outside the contract; the callers have checked their inputs for NaN).  Branch-free:
// the argument is clamped at -707 and results below e^-707 are flushed to 0 by a select (kernel values that
// small are irrelevant next to the noise floor e^-9 on the diagonal).
__host__ __device__ __forceinline__ double exp_nonpos(double x0) {
    const double x = dmax(x0, -707.0);
    const double MAGIC = 6755399441055744.0;                 // 1.5 * 2^52: low word of (t + MAGIC) is rint(t)
    const double tm = fma(x, 46.16624130844683, MAGIC);      // x * 32 / ln 2
    const double nd = tm - MAGIC;
#ifdef __CUDA_ARCH__
    const int n = __double2loint(tm);
#else
    long long bits;
    memcpy(&bits, &tm, 8);
    const int n = (int)(unsigned)(bits & 0xFFFFFFFFll);
#endif
    double r = fma(nd, -0.021660849392446835, x);            // ln2/32, leading 36 bits: n * L_hi is exact
    r = fma(nd, -5.145609244655338e-14, r);
    double p = 1.0 / 720.0;
    p = fma(p, r, 1.0 / 120.0);
    p = fma(p, r, 1.0 / 24.0);
    p = fma(p, r, 1.0 / 6.0);
    p = fma(p, r, 0.5);
    p = fma(p, r, 1.0);
    p = p * r;                                               // e^r - 1
#ifdef __CUDA_ARCH__
    const double T = __ldg(&d_exp_table[n & 31]);
    const double v = fma(T, p, T);
    const double r2 = __hiloint2double(__double2hiint(v) + ((n >> 5) << 20), __double2loint(v));
#else
    const double T = h_exp_table[n & 31];
    const double v = fma(T, p, T);
    const double r2 = ldexp(v, n >> 5);
#endif
    return (x0 < -707.0) ? 0.0 : r2;
}

// sqrt(s) for 1e-300 < s < 1e300
__host__ __device__ __forceinline__ double sqrt_pos(double s) {
    double y;
#ifdef __CUDA_ARCH__
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(s));
#else
    y = (double)(1.0f / sqrtf((float)s));
    if (!(y > 0.0) || y > 1e30) y = 1.0 / sqrt(s);           // outside float range (host test only)
#endif
    double g = s * y, h = 0.5 * y;
    double r = fma(-h, g, 0.5);
    g = fma(g, r, g);
    h = fma(h, r, h);
    r = fma(-h, g, 0.5);
    g = fma(g, r, g);
    h = fma(h, r, h);
    const double d = fma(-g, g, s);                          // residual: g <- g + d / (2 g)
    return fma(d, h, g);
}

// sqrt(s) and 1/sqrt(s) from ONE coupled Goldschmidt iteration (the Cholesky leaf's pivot step, csrc/potrf_leaf.cuh):
// root to <= 1 ulp, reciprocal to <= 2 ulp (checked on the host by tests/test_kernel_math_cpu.py).  s <= 0 or NaN
// gives NaN for both, like sqrt() of a negative number.
__host__ __device__ __forceinline__ void sqrt_and_reciprocal(double s, double& root, double& inv) {
    double y;
#ifdef __CUDA_ARCH__
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(s));
#else
    y = (double)(1.0f / sqrtf((float)s));
    if (!(y > 0.0) || y > 1e30) y = 1.0 / sqrt(s);           // outside float range (host test only)
#endif
    double g = s * y, h = 0.5 * y;
    double r = fma(-h, g, 0.5);
    g = fma(g, r, g);
    h = fma(h, r, h);
    r = fma(-h, g, 0.5);
    g = fma(g, r, g);
    h = fma(h, r, h);
    const double d = fma(-g, g, s);                          // residual: g <- g + d / (2 g)
    g = fma(d, h, g);
    r = fma(-h, g, 0.5);                                     // h <- 1 / (2 g) for the corrected root
    h = fma(h, r, h);
    const bool ok = s > 0.0;
#ifdef __CUDA_ARCH__
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
#else
    const double qnan = NAN;
#endif
    root = ok ? g : qnan;
    inv = ok ? h + h : qnan;
}

// log(1 + x) for finite x >= 0, table-driven like exp_nonpos.  u = 1 + x is split as u = 2^e m with
// m within 1/64 of c_j = 1 + j/32 (j = the mantissa's leading 5 bits, rounded), so that
//   log1p(x) = e ln2 + log(c_j) + log1p(r),   r = (m - c_j + c 2^-e) / c_j,   |r| <= 1/64,
// where c = x - (u - 1) is the rounding error of u (exact for x < 2^53): without it small x would lose their low
// bits in 1 + x, and the RQ kernel at large alpha (alpha log1p(s / 2 alpha) -> s / 2) would not reach the RBF
// value.  r is carried as r_hi + r_lo (the division residual by one FMA), log1p(r_hi) by its Taylor series to
// r^9 (remainder <= 2^-60 / 10) plus r_lo (1 - r_hi), and e ln2 + log(c_j) + r_hi is summed with its rounding
// error.  About 25 FP64 instructions, 2 L1-resident loads; < 1.2 ulp against a correctly rounded log1p (the
// residue above 1/2 ulp is the rounding of e ln2 + log(c_j); tests/test_rq_kernel_cpu.py).
// Per j: {1 / c_j rounded, log(c_j) leading part}, and the trailing part of log(c_j).
#define PLMC_LOG_TABLE_A                                                                                            \
    {{1.0, 0.0}, {0.9696969696969697, 0.030771658666753687}, {0.9411764705882353, 0.06062462181643484},           \
     {0.9142857142857143, 0.08961215868968714}, {0.8888888888888888, 0.11778303565638346},                        \
     {0.8648648648648649, 0.1451820098444979}, {0.8421052631578947, 0.17185025692665923},                         \
     {0.8205128205128205, 0.19782574332991987}, {0.8, 0.22314355131420976},                                       \
     {0.7804878048780488, 0.24783616390458127}, {0.7619047619047619, 0.27193371548364176},                        \
     {0.7441860465116279, 0.2954642128938359}, {0.7272727272727273, 0.3184537311185346},                          \
     {0.7111111111111111, 0.3409265869705932}, {0.6956521739130435, 0.3629054936893685},                          \
     {0.6808510638297872, 0.38441169891033206}, {0.6666666666666666, 0.4054651081081644},                         \
     {0.6530612244897959, 0.4260843953109001}, {0.64, 0.44628710262841953},                                       \
     {0.6274509803921569, 0.46608972992459924}, {0.6153846153846154, 0.4855078157817008},                         \
     {0.6037735849056604, 0.5045560107523953}, {0.5925925925925926, 0.5232481437645479},                          \
     {0.5818181818181818, 0.5415972824327444}, {0.5714285714285714, 0.5596157879354227},                          \
     {0.5614035087719298, 0.5773153650348236}, {0.5517241379310345, 0.5947071077466928},                          \
     {0.5423728813559322, 0.6118015411059929}, {0.5333333333333333, 0.6286086594223741},                          \
     {0.5245901639344263, 0.6451379613735847}, {0.5161290322580645, 0.661398482245365},                           \
     {0.5079365079365079, 0.6773988235918061}}
#define PLMC_LOG_TABLE_B                                                                                            \
    {0.0, 1.0431732029005968e-18, 2.6424025938726934e-18, -5.4268129336647135e-18, -1.1971685747593677e-18,       \
     8.242418783022475e-18, -6.0224538210113705e-18, 1.2821194372980142e-17, -9.091270597324799e-18,              \
     -1.2432209578702523e-17, 7.83319637697442e-19, -2.16461086040599e-17, 2.7114779367326236e-17,                \
     1.7467136443544747e-17, -2.1492361455310972e-17, -1.612149700764673e-17, -2.8811380259626426e-18,            \
     -2.499176776547466e-17, -1.8182541194649598e-17, -1.4116523239904406e-17, -1.6618350693852048e-17,           \
     -2.4888518873597905e-17, -3.1833882216350925e-17, -3.748764246125639e-17, 2.685492580212308e-17,             \
     -8.903591846974013e-18, 1.3751689964323675e-17, -3.7397759448726e-17, 4.3538742607970387e-17,                \
     9.346960920120906e-19, -7.603333785634003e-18, -2.0978183882652005e-18}

static __device__ const double2 d_log_table_a[32] = PLMC_LOG_TABLE_A;
static __device__ const double d_log_table_b[32] = PLMC_LOG_TABLE_B;
static const double h_log_table_a[32][2] = PLMC_LOG_TABLE_A;
static const double h_log_table_b[32] = PLMC_LOG_TABLE_B;

__host__ __device__ __forceinline__ long long plmc_double_bits(double v) {
#ifdef __CUDA_ARCH__
    return __double_as_longlong(v);
#else
    long long b;
    memcpy(&b, &v, 8);
    return b;
#endif
}

__host__ __device__ __forceinline__ double plmc_bits_double(long long b) {
#ifdef __CUDA_ARCH__
    return __longlong_as_double(b);
#else
    double v;
    memcpy(&v, &b, 8);
    return v;
#endif
}

__host__ __device__ __forceinline__ double log1p_nonneg(double x) {
    const double u = 1.0 + x;
    const double c = x - (u - 1.0);                           // 1 + x = u + c exactly
    const long long ix = plmc_double_bits(u) + (1ll << 46);   // round the mantissa to 5 bits
    const int e = (int)(ix >> 52) - 1023;
    const int j = (int)(ix >> 47) & 31;
    const double m = plmc_bits_double(plmc_double_bits(u) - ((long long)e << 52));   // u 2^-e, |m - c_j| <= 1/64
    const double cj = plmc_bits_double(0x3FF0000000000000ll | ((long long)j << 47));
    const double c2 = c * plmc_bits_double((long long)(1023 - e) << 52);              // c 2^-e
#ifdef __CUDA_ARCH__
    const double2 ta = __ldg(&d_log_table_a[j]);
    const double inv = ta.x, thi = ta.y, tlo = __ldg(&d_log_table_b[j]);
#else
    const double inv = h_log_table_a[j][0], thi = h_log_table_a[j][1], tlo = h_log_table_b[j];
#endif
    const double dm = m - cj;                                 // exact
    const double rh = dm * inv;
    const double rl = (fma(-rh, cj, dm) + c2) * inv;          // r = rh + rl to ~2^-100 relative
    double p = 1.0 / 9.0;                                     // log1p(rh) = rh + rh^2 P(rh)
    p = fma(p, rh, -1.0 / 8.0);
    p = fma(p, rh, 1.0 / 7.0);
    p = fma(p, rh, -1.0 / 6.0);
    p = fma(p, rh, 1.0 / 5.0);
    p = fma(p, rh, -1.0 / 4.0);
    p = fma(p, rh, 1.0 / 3.0);
    p = fma(p, rh, -0.5);
    const double MAGIC = 6755399441055744.0;                  // e as a double without an integer conversion
    const double ed = plmc_bits_double(plmc_double_bits(MAGIC) + e) - MAGIC;
    const double hi = fma(ed, 0.6931471805598903, thi);       // ln2 leading 42 bits: e ln2_hi is exact
    const double lo = fma(ed, 5.497923018708371e-14, tlo);
    const double w = hi + rh;
    const double err = (hi - w) + rh;                         // |hi| >= |rh| whenever hi != 0: exact
    return w + fma(rh * rh, p, fma(-rl, rh, rl) + lo + err);   // log1p(rh + rl) = log1p(rh) + rl (1 - rh) + ...
}

// 1 / b for b >= 1 (the RQ base): MUFU.RCP64H seed and two Newton steps, <= 1 ulp
__host__ __device__ __forceinline__ double rcp_ge1(double b) {
    double y;
#ifdef __CUDA_ARCH__
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(b));
#else
    y = (double)(1.0f / (float)b);
    if (!(y > 0.0) || y < 1e-30) y = 1.0 / b;                 // outside float range (host test only)
#endif
    double r = fma(-b, y, 1.0);
    y = fma(y, r, y);
    r = fma(-b, y, 1.0);
    return fma(y, r, y);
}

// Shape parameter of a kernel, read once per latent: the RQ exponent alpha and 1 / (2 alpha) (so that the
// per-entry x = s / (2 alpha) is one multiplication).  Unused by kernels 0-3.
struct KernelShape {
    double alpha, half_inv;
};

__host__ __device__ __forceinline__ KernelShape kernel_shape(double alpha) { return KernelShape{alpha, 0.5 / alpha}; }

template <int KID>
__host__ __device__ __forceinline__ double kernel_value(double s, KernelShape sh = KernelShape{0.0, 0.0}) {
    if (KID == 4) return exp_nonpos(-sh.alpha * log1p_nonneg(s * sh.half_inv));
    if (KID == 0) return exp_nonpos(-0.5 * s);
    if (KID == 1) {
        const double u = 5.0 * dmax(s, 1e-30);               // (sqrt5 r)^2
        const double a = sqrt_pos(u);
        return (1.0 + a + u * (1.0 / 3.0)) * exp_nonpos(-a);
    }
    if (KID == 2) {
        const double a = sqrt_pos(3.0 * dmax(s, 1e-30));
        return (1.0 + a) * exp_nonpos(-a);
    }
    return exp_nonpos(-sqrt_pos(dmax(s, 1e-30)));
}

// k(s) and dk/ds
template <int KID>
__host__ __device__ __forceinline__ void kernel_value_grad(double s, double& k, double& dk) {
    if (KID == 0) {
        k = exp_nonpos(-0.5 * s);
        dk = -0.5 * k;
        return;
    }
    if (KID == 1) {
        const double u = 5.0 * dmax(s, 1e-30);
        const double a = sqrt_pos(u);
        const double e = exp_nonpos(-a);
        k = (1.0 + a + u * (1.0 / 3.0)) * e;
        dk = -(5.0 / 6.0) * (1.0 + a) * e;
    } else if (KID == 2) {
        const double a = sqrt_pos(3.0 * dmax(s, 1e-30));
        const double e = exp_nonpos(-a);
        k = (1.0 + a) * e;
        dk = -1.5 * e;
    } else {
        const double r = sqrt_pos(dmax(s, 1e-30));
        k = exp_nonpos(-r);
        dk = (s > 1e-30) ? -0.5 * k / r : 0.0;
    }
}

// k(s), dk/ds and dk/d(shape).  RQ (gpytorch 1.11 RQKernel): with x = s / (2 alpha), b = 1 + x, L = log1p(x):
//   k = b^-alpha = exp(-alpha L),  dk/ds = -k / (2 b),  dk/dalpha = k (x / b - L).
// Kernels 0-3 have no shape parameter (dk/dshape = 0) and compile exactly as the two-output form above.
template <int KID>
__host__ __device__ __forceinline__ void kernel_value_grad(double s, double& k, double& dk, double& dka,
                                                           KernelShape sh) {
    if (KID == 4) {
        const double x = s * sh.half_inv;
        const double L = log1p_nonneg(x);
        k = exp_nonpos(-sh.alpha * L);
        const double ib = rcp_ge1(1.0 + x);
        dk = (-0.5 * k) * ib;
        dka = k * fma(x, ib, -L);
        return;
    }
    kernel_value_grad<KID>(s, k, dk);
    dka = 0.0;
}

}  // namespace plmc
