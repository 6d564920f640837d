// ndchg.cu -- C ABI (include/ndchg.h) of the omnibus change detection: one thread per pixel walks the reference's
// control flow (nd/_change.pyx:224-260) with the reference's arithmetic types.  The marginal tests of one starting
// point l grow by one time step at a time, so their sums / determinant product are kept running (the same
// left-to-right accumulation order as recomputing every subset from scratch, hence identical values).
// The walk and the probability kernel are templates over the accumulator of one covariance layout: `Acc<T>` is the
// reference's dual-pol statistic; `AccDiag<T, P>` (single-pol and the diagonal-only layouts) and `AccQuad<T>`
// (quad-pol) generalise it, reading the data type and computing everything else in double (include/ndchg.h).
// `change_direction_kernel` is a post-pass over the walk's change map that classifies each change as an increase,
// a decrease or indefinite; the walk kernels do not know about it.
#include "../../include/ndchg.h"
#include "../../include/ndnlm.h"

#include <cmath>
#include <cstdarg>
#include <cstdio>

#include <cuda_runtime.h>
#include <math_constants.h>

static thread_local char g_chg_err[512] = "";
static int chg_fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_chg_err, sizeof(g_chg_err), fmt, ap);
    va_end(ap);
    return code;
}

namespace ndchg {

// separate, correctly rounded operations in the data type (no FMA contraction: the reference is plain C)
__device__ __forceinline__ float mul_(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add_(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub_(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double mul_(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add_(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double sub_(double a, double b) { return __dsub_rn(a, b); }

// Regularised lower incomplete gamma P(a, y) for INTEGER a >= 1 and y > 0, in double:
//   y <= a:  P = e^-y y^a / a!  * sum_{m>=0} y^m / ((a+1)...(a+m))
//   y >  a:  P = 1 - e^-y y^(a-1) / (a-1)! * sum_{i=0}^{a-1} (a-1)...(a-i) / y^i
__device__ double gamma_p_int(const int a, const double y) {
    if (y <= double(a)) {
        double term = 1.0, sum = 1.0;
        for (int m = 1; m < 100000; ++m) {
            term *= y / double(a + m);
            sum += term;
            if (term < sum * 1e-17) break;
        }
        return exp(double(a) * log(y) - y - lgamma(double(a) + 1.0)) * sum;
    }
    double term = 1.0, sum = 1.0;
    for (int i = 1; i < a; ++i) {
        term *= double(a - i) / y;
        sum += term;
        if (term < sum * 1e-17) break;
    }
    return 1.0 - exp(double(a - 1) * log(y) - y - lgamma(double(a))) * sum;
}

// gsl_cdf_chisq_P(x, nu) with nu = 2 a
__device__ __forceinline__ double chisq_p(const double x, const int a) {
    if (x != x) return x;
    if (!(x > 0.0)) return 0.0;
    return gamma_p_int(a, 0.5 * x);
}

// The double-precision constants, operation by operation in the reference's order (explicit intrinsics: no FMA
// contraction, `x**2` is pow(x, 2) = the correctly rounded x*x).
__device__ __forceinline__ double rho_(const double p, const double k, const double n) {
    // 1 - (2 * p**2 - 1) / (6 * (k - 1) * p) * (k/n - 1/(n*k))                              nd/_change.pyx:26-30
    const double A = __dsub_rn(__dmul_rn(2.0, __dmul_rn(p, p)), 1.0);
    const double B = __dmul_rn(__dmul_rn(6.0, __dsub_rn(k, 1.0)), p);
    const double C = __dsub_rn(__ddiv_rn(k, n), __ddiv_rn(1.0, __dmul_rn(n, k)));
    return __dsub_rn(1.0, __dmul_rn(__ddiv_rn(A, B), C));
}
__device__ __forceinline__ double omega2_(const double p, const double k, const double n, const double rho) {
    // p**2 * (p**2 - 1) / (24 * rho**2) * (k/(n**2) - 1/((n*k)**2)) - p**2 * (k - 1) / 4 * (1 - 1/rho)**2   :33-39
    const double p2 = __dmul_rn(p, p);
    const double nk = __dmul_rn(n, k);
    const double left = __dmul_rn(__ddiv_rn(__dmul_rn(p2, __dsub_rn(p2, 1.0)), __dmul_rn(24.0, __dmul_rn(rho, rho))),
                                  __dsub_rn(__ddiv_rn(k, __dmul_rn(n, n)), __ddiv_rn(1.0, __dmul_rn(nk, nk))));
    const double x = __dsub_rn(1.0, __ddiv_rn(1.0, rho));
    const double right = __dmul_rn(__ddiv_rn(__dmul_rn(p2, __dsub_rn(k, 1.0)), 4.0), __dmul_rn(x, x));
    return __dsub_rn(left, right);
}

// running state of `_z` (nd/_change.pyx:45-79) over a growing subset
template <typename T>
struct Acc {
    using value_type = T;
    T c11, c12r, c12i, c22;
    double prod;
    __device__ void reset() { c11 = c12r = c12i = c22 = T(0); prod = 1.0; }
    __device__ void push(const T* q, const long long s3) { push(q[0], q[s3], q[2 * s3], q[3 * s3]); }
    __device__ void push(const T a, const T br, const T bi, const T d) {
        const T det = sub_(mul_(a, d), add_(mul_(br, br), mul_(bi, bi)));
        prod = __dmul_rn(prod, double(det));
        c11 = add_(c11, a);
        c12r = add_(c12r, br);
        c12i = add_(c12i, bi);
        c22 = add_(c22, d);
    }
    // single_pixel_omnibus (nd/_change.pyx:139-160) of the k steps pushed so far
    __device__ T probability(const int k, const unsigned n) const {
        const double kd = double(k), nd = double(n);
        const T det_of_sum = sub_(mul_(c11, c22), add_(mul_(c12r, c12r), mul_(c12i, c12i)));
        const T pk = mul_(T(2), T(k));                                                     // `p*k` in `floating`
        // n * (p*k*log(k) + log(prod_of_dets) - k*log(det_of_sum))                            nd/_change.pyx:74
        const double logQ = __dmul_rn(nd, __dsub_rn(__dadd_rn(__dmul_rn(double(pk), log(kd)), log(prod)),
                                                    __dmul_rn(kd, log(double(det_of_sum)))));
        const double rho = rho_(2.0, kd, nd);
        const T rho_t = T(rho);
        const T z = T(__dmul_rn(double(mul_(T(-2), rho_t)), logQ));
        const double omega2 = omega2_(2.0, kd, nd, rho);
        const int a = 2 * (k - 1);                                                         // f / 2 with f = (k-1) p^2
        const T P1 = T(chisq_p(double(z), a));
        const T P2 = T(chisq_p(double(z), a + 2));
        return T(__dadd_rn(double(P1), __dmul_rn(omega2, double(sub_(P2, P1)))));
    }
};

// Regularised lower incomplete gamma P(a, y) for REAL a > 0, in double (the layouts other than dual-pol have
// half-integer shapes): series for y < a + 1, Legendre's continued fraction for Q = 1 - P otherwise (modified Lentz).
// The algorithm of oracle/gsl_shim/gsl_shim.h; the prefactor exp(-y + a ln y - lgamma(a)) loses ~a ulps, and
// the probabilities stay within 1e-12 of scipy's up to a = 283.5 (quad-pol, k = 64; tests/test_change_pol.py).
__device__ double gamma_p(const double a, const double y) {
    if (isinf(y)) return 1.0;
    const double lg = lgamma(a);
    if (y < a + 1.0) {
        double ap = a, sum = 1.0 / a, del = sum;
        for (int m = 0; m < 100000; ++m) {
            ap += 1.0;
            del *= y / ap;
            sum += del;
            if (fabs(del) < fabs(sum) * 1e-17) break;
        }
        return sum * exp(-y + a * log(y) - lg);
    }
    const double tiny = 1e-300;
    double b = y + 1.0 - a, c = 1.0 / tiny, d = 1.0 / b, h = d;
    for (int i = 1; i < 100000; ++i) {
        const double an = -double(i) * (double(i) - a);
        b += 2.0;
        d = an * d + b;
        if (fabs(d) < tiny) d = tiny;
        c = b + an / c;
        if (fabs(c) < tiny) c = tiny;
        d = 1.0 / d;
        const double del = d * c;
        h *= del;
        if (fabs(del - 1.0) < 1e-16) break;
    }
    return 1.0 - exp(-y + a * log(y) - lg) * h;
}

// chi-square CDF with f = 2 a degrees of freedom; NaN stays NaN, x <= 0 gives 0
__device__ __forceinline__ double chisq_p_real(const double x, const double a) {
    if (x != x) return x;
    if (!(x > 0.0)) return 0.0;
    return gamma_p(a, 0.5 * x);
}

// The generalised statistic of the layouts other than dual-pol, in double from the sum of ln det X_i and
// det sum_i X_i over k steps.  Full covariance (FULL): the reference's f = (k-1) p^2, rho, omega2 at p; diagonal
// only: f = (k-1) p, rho at p = 1, omega2 = -f/4 (1 - 1/rho)^2 (lnQ is the sum of p single-band lnQs).
template <int P, bool FULL>
__device__ __forceinline__ double omnibus_p(const int k, const unsigned n, const double sum_logdet, const double det_of_sum) {
    const double p = P, kd = double(k), nd = double(n);
    const double logQ = nd * (p * kd * log(kd) + sum_logdet - kd * log(det_of_sum));
    const double rho = rho_(FULL ? p : 1.0, kd, nd);
    const double f = FULL ? (kd - 1.0) * p * p : (kd - 1.0) * p;
    const double x = 1.0 - 1.0 / rho;
    const double omega2 = FULL ? omega2_(p, kd, nd, rho) : -f / 4.0 * (x * x);
    const double z = -2.0 * rho * logQ;
    const double P1 = chisq_p_real(z, 0.5 * f);
    const double P2 = chisq_p_real(z, 0.5 * f + 2.0);
    return P1 + omega2 * (P2 - P1);
}

// diagonal of a P x P covariance: single-pol (P = 1, where the diagonal and the full statistic coincide) and the
// intensity-only layouts [C11, C22] / [C11, C22, C33]; det is the product of the diagonal
template <typename T, int P>
struct AccDiag {
    using value_type = T;
    double c[P];
    double logdets;
    __device__ void reset() {
        for (int b = 0; b < P; ++b) c[b] = 0.0;
        logdets = 0.0;
    }
    __device__ void push(const T* q, const long long s3) {
        double det = 1.0;
        for (int b = 0; b < P; ++b) {
            const double v = double(q[b * s3]);
            det *= v;
            c[b] += v;
        }
        logdets += log(det);
    }
    __device__ T probability(const int k, const unsigned n) const {
        double det = 1.0;
        for (int b = 0; b < P; ++b) det *= c[b];
        return T(omnibus_p<P, P == 1>(k, n, logdets, det));
    }
};

// 3 x 3 Hermitian covariance [C11, Re C12, Im C12, Re C13, Im C13, C22, Re C23, Im C23, C33]
template <typename T>
struct AccQuad {
    using value_type = T;
    double c[9];
    double logdets;
    // a, d, g the real diagonal, b = C12, c = C13, e = C23: a d g + 2 Re(b e conj(c)) - a|e|^2 - d|c|^2 - g|b|^2
    __device__ static double det(const double* m) {
        const double a = m[0], br = m[1], bi = m[2], cr = m[3], ci = m[4], d = m[5], er = m[6], ei = m[7], g = m[8];
        const double be_re = br * er - bi * ei, be_im = br * ei + bi * er;
        return a * d * g + 2.0 * (be_re * cr + be_im * ci) - a * (er * er + ei * ei) - d * (cr * cr + ci * ci) -
               g * (br * br + bi * bi);
    }
    __device__ void reset() {
        for (int b = 0; b < 9; ++b) c[b] = 0.0;
        logdets = 0.0;
    }
    __device__ void push(const T* q, const long long s3) {
        double m[9];
        for (int b = 0; b < 9; ++b) {
            m[b] = double(q[b * s3]);
            c[b] += m[b];
        }
        logdets += log(det(m));
    }
    __device__ T probability(const int k, const unsigned n) const { return T(omnibus_p<3, true>(k, n, logdets, det(c))); }
};

template <typename A>
__global__ void __launch_bounds__(128)
change_detection_kernel(const typename A::value_type* __restrict__ values, const long long rows, const long long cols,
                        const int k, const long long s0, const long long s1, const long long s2, const long long s3,
                        unsigned char* __restrict__ result, const double alpha, const unsigned n) {
    using T = typename A::value_type;
    const long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= rows * cols) return;
    const long long i = pix / cols, j = pix - i * cols;
    const T* ts = values + i * s0 + j * s1;
    unsigned char* res = result + pix * k;
    for (int t = 0; t < k; ++t) res[t] = 0;
    auto push = [&](A& acc, const int t) { acc.push(ts + (long long)t * s2, s3); };
    int l = 0, r = 0;
    A acc;
    while (true) {                                                                         // nd/_change.pyx:238-260
        acc.reset();
        for (int t = l; t < k; ++t) push(acc, t);
        if (!(double(acc.probability(k - l, n)) > alpha)) break;                           // global hypothesis H0_l
        acc.reset();
        push(acc, l);
        for (int jj = 2; jj < k - l + 1; ++jj) {                                           // marginal hypotheses
            push(acc, l + jj - 1);
            r = jj - 1;
            if (double(acc.probability(jj, n)) > alpha) {
                res[l + r] = 1;
                break;
            }
        }
        l = l + r;
        if (l >= k - 1) break;
    }
}

template <typename A>
__global__ void __launch_bounds__(128)
omnibus_probability_kernel(const typename A::value_type* __restrict__ values, const long long rows, const long long cols,
                           const int k, const long long s0, const long long s1, const long long s2, const long long s3,
                           typename A::value_type* __restrict__ prob, const unsigned n) {
    using T = typename A::value_type;
    const long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= rows * cols) return;
    const long long i = pix / cols, j = pix - i * cols;
    const T* ts = values + i * s0 + j * s1;
    A acc;
    acc.reset();
    for (int t = 0; t < k; ++t) acc.push(ts + (long long)t * s2, s3);
    prob[pix] = acc.probability(k, n);
}

// Loewner order of D = X_t - mean of the segment before it (include/ndchg.h).  Every operation is a separate,
// correctly rounded double operation in the order of oracle/omnibus_direction_oracle.py::classify, so the codes match the
// oracle exactly; AccQuad::det is deliberately not reused (written without intrinsics, nvcc contracts it into FMAs).
__host__ __device__ constexpr int pol_bands(const int pol) {
    return pol == NDCHG_POL_DUAL ? 4 : pol == NDCHG_POL_SINGLE ? 1 : pol == NDCHG_POL_QUAD ? 9 : pol == NDCHG_POL_DUAL_DIAGONAL ? 2 : 3;
}

template <int POL>
__device__ __forceinline__ unsigned char classify(const double* D) {
    if constexpr (POL == NDCHG_POL_DUAL || POL == NDCHG_POL_QUAD) {
        // Sylvester's criterion on the leading principal minors; C22 is band 3 (dual) or 5 (quad)
        constexpr int i22 = POL == NDCHG_POL_DUAL ? 3 : 5;
        const double m1 = D[0];
        const double m2 = __dsub_rn(__dmul_rn(D[0], D[i22]), __dadd_rn(__dmul_rn(D[1], D[1]), __dmul_rn(D[2], D[2])));
        if constexpr (POL == NDCHG_POL_DUAL) {
            if (m1 > 0.0 && m2 > 0.0) return NDCHG_DIR_INCREASE;
            if (m1 < 0.0 && m2 > 0.0) return NDCHG_DIR_DECREASE;
        } else {
            const double a = D[0], br = D[1], bi = D[2], cr = D[3], ci = D[4], d = D[5], er = D[6], ei = D[7], g = D[8];
            // ((a*d)*g + 2*re_bec) - a*(|e|^2) - d*(|c|^2) - g*(|b|^2), re_bec = Re(b e conj(c))
            const double re_bec = __dadd_rn(__dmul_rn(__dsub_rn(__dmul_rn(br, er), __dmul_rn(bi, ei)), cr),
                                            __dmul_rn(__dadd_rn(__dmul_rn(br, ei), __dmul_rn(bi, er)), ci));
            double m3 = __dadd_rn(__dmul_rn(__dmul_rn(a, d), g), __dmul_rn(2.0, re_bec));
            m3 = __dsub_rn(m3, __dmul_rn(a, __dadd_rn(__dmul_rn(er, er), __dmul_rn(ei, ei))));
            m3 = __dsub_rn(m3, __dmul_rn(d, __dadd_rn(__dmul_rn(cr, cr), __dmul_rn(ci, ci))));
            m3 = __dsub_rn(m3, __dmul_rn(g, __dadd_rn(__dmul_rn(br, br), __dmul_rn(bi, bi))));
            if (m1 > 0.0 && m2 > 0.0 && m3 > 0.0) return NDCHG_DIR_INCREASE;
            if (m1 < 0.0 && m2 > 0.0 && m3 < 0.0) return NDCHG_DIR_DECREASE;
        }
        return NDCHG_DIR_INDEFINITE;
    } else {
        // single and the intensity-only diagonals: signs of the diagonal, no products (nothing can underflow)
        bool up = true, down = true;
        for (int b = 0; b < pol_bands(POL); ++b) {
            up = up && D[b] > 0.0;
            down = down && D[b] < 0.0;
        }
        return up ? NDCHG_DIR_INCREASE : down ? NDCHG_DIR_DECREASE : NDCHG_DIR_INDEFINITE;
    }
}

// Post-pass after change_detection_kernel on the same stream: rewrites each pixel's 0 / 1 change vector in place
// with the direction codes.  A pixel without a change returns before reading `values`; otherwise its series is read
// once, up to its last change.  The segment before a change starts at the previous change (the walk restarts there).
template <typename T, int POL>
__global__ void __launch_bounds__(128)
change_direction_kernel(const T* __restrict__ values, const long long rows, const long long cols, const int k,
                        const long long s0, const long long s1, const long long s2, const long long s3,
                        unsigned char* __restrict__ result) {
    constexpr int B = pol_bands(POL);
    const long long pix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= rows * cols) return;
    unsigned char* res = result + pix * k;
    int last = -1;
    for (int t = 0; t < k; ++t)
        if (res[t]) last = t;
    if (last < 0) return;
    const long long i = pix / cols, j = pix - i * cols;
    const T* ts = values + i * s0 + j * s1;
    double S[B];
    for (int b = 0; b < B; ++b) S[b] = 0.0;
    int m = 0;
    for (int t = 0; t <= last; ++t) {
        const T* q = ts + (long long)t * s2;
        if (res[t]) {                                        // the walk never marks t = 0, so m >= 1 here
            double D[B];
            const double md = double(m);
            for (int b = 0; b < B; ++b) {
                D[b] = __dsub_rn(double(q[b * s3]), __ddiv_rn(S[b], md));
                S[b] = 0.0;
            }
            res[t] = classify<POL>(D);
            m = 0;
        }
        for (int b = 0; b < B; ++b) S[b] = __dadd_rn(S[b], double(q[b * s3]));
        ++m;
    }
}

// ---- equivalent number of looks (ndchg_enl, include/ndchg.h) -----------------------------------------------------
// g(L, s) = ln L - psi(L - s) and dg = d/dL g = 1/L - psi'(L - s), for L - s > 0: psi and psi' by the recurrence
// psi(x) = psi(x + m) - sum_{j<m} 1/(x + j) up to y = x + m >= 10, then the asymptotic series of ln y - psi(y) and
// psi'(y) (Bernoulli numbers up to B14; the first omitted term is < 5e-17 at y = 10).  ln L - ln y is formed as
// -log1p((m - s) / L), so g keeps its relative accuracy at large L, where it is ~ (s + 1/2) / L and the plain
// difference ln L - psi(L - s) would cancel.
__device__ __forceinline__ void ln_minus_digamma(const double L, const int s, double& g, double& dg) {
    const double x = L - double(s);
    double r = 0.0, r2 = 0.0;
    int m = 0;
    while (x + double(m) < 10.0) {
        const double inv = 1.0 / (x + double(m));
        r += inv;
        r2 += inv * inv;
        ++m;
    }
    const double iy = 1.0 / (x + double(m)), iy2 = iy * iy;
    // ln y - psi(y) = 1/(2y) + 1/(12y^2) - 1/(120y^4) + 1/(252y^6) - 1/(240y^8) + 1/(132y^10) - 691/(32760y^12) + 1/(12y^14)
    const double lnpsi = 0.5 * iy + iy2 * (1.0 / 12 + iy2 * (-1.0 / 120 + iy2 * (1.0 / 252 + iy2 * (-1.0 / 240 +
                         iy2 * (1.0 / 132 + iy2 * (-691.0 / 32760 + iy2 * (1.0 / 12)))))));
    // psi'(y) = 1/y + 1/(2y^2) + 1/(6y^3) - 1/(30y^5) + 1/(42y^7) - 1/(30y^9) + 5/(66y^11) - 691/(2730y^13) + 7/(6y^15)
    const double trigamma = iy + iy2 * (0.5 + iy * (1.0 / 6 + iy2 * (-1.0 / 30 + iy2 * (1.0 / 42 + iy2 * (-1.0 / 30 +
                            iy2 * (5.0 / 66 + iy2 * (-691.0 / 2730 + iy2 * (7.0 / 6))))))));
    g = -log1p(double(m - s) / L) + r + lnpsi;
    dg = 1.0 / L - (trigamma + r2);
}

// G(L) and G'(L): full layouts (p x p complex Wishart) G = sum_{i<P} (ln L - psi(L - i)) on L > P - 1; diagonal
// layouts (P independent Gamma channels) G = P (ln L - psi(L)) on L > 0.
template <int P, bool FULL>
__device__ __forceinline__ void enl_G(const double L, double& G, double& dG) {
    if constexpr (FULL) {
        G = dG = 0.0;
        for (int i = 0; i < P; ++i) {
            double g, dg;
            ln_minus_digamma(L, i, g, dg);
            G += g;
            dG += dg;
        }
    } else {
        ln_minus_digamma(L, 0, G, dG);
        G *= P;
        dG *= P;
    }
}

// The root of h(L) = G(L) - G(N L) = delta (h falls strictly from +inf to 0 on the domain), to a relative 1e-13:
// Newton from the large-L approximation h ~ c (1 - 1/N) / L (c = P^2 / 2 full, P / 2 diagonal), kept inside the
// bracket [lo, hi] of the iterates seen so far (bisection, or doubling while no upper bound is known).
template <int P, bool FULL>
__device__ double enl_solve(const double delta, const double N) {
    double lo = FULL ? double(P - 1) : 0.0, hi = CUDART_INF;
    const double c = FULL ? 0.5 * P * P : 0.5 * P;
    double L = lo + c * (1.0 - 1.0 / N) / delta;
    for (int it = 0; it < 200; ++it) {
        double G1, dG1, GN, dGN;
        enl_G<P, FULL>(L, G1, dG1);
        enl_G<P, FULL>(N * L, GN, dGN);
        const double f = (G1 - GN) - delta, df = dG1 - N * dGN;
        if (f == 0.0) return L;
        if (f > 0.0) lo = L;
        else hi = L;
        double next = L - f / df;
        if (!(next > lo && next < hi)) next = isinf(hi) ? 2.0 * L : 0.5 * (lo + hi);
        if (fabs(next - L) <= 1e-13 * next || hi - lo <= 1e-15 * lo) return next;
        L = next;
    }
    return L;
}

// One CTA: an output tile of ENL_TR x ENL_TC pixels x KT time steps.  The input rows of the tile plus the w - 1
// halo rows are read one at a time, in segments of ENL_SEG pixels; a thread per sample reads its bands (contiguous
// for C-contiguous input, as are the KT samples of a pixel), forms ln det and stores the B + 1 doubles in shared
// memory.  The horizontal window sums of the row (w terms each, added left to right) go to H and are added to the
// vertical sums V of every output row whose window contains the input row, in row order: each window sum is a
// direct sum of w x w terms, never a running add / subtract.  Then every thread solves its outputs.
constexpr int ENL_TR = 16, ENL_TC = 32, ENL_SEG = 64, ENL_THREADS = 256;

template <typename T, int POL>
struct EnlTile {
    static constexpr int B = pol_bands(POL);
    static constexpr int E = B + 1;                                      // bands, then ln det
    static constexpr int KT = (32 / int(sizeof(T)) + B - 1) / B;         // >= 32 bytes of each pixel per row read
    static constexpr size_t smem = sizeof(double) * E * KT * (size_t(ENL_TR) * ENL_TC + ENL_TC + ENL_SEG);
};

template <int POL>
__device__ __forceinline__ double sample_det(const double* x) {
    if constexpr (POL == NDCHG_POL_DUAL) {
        return x[0] * x[3] - (x[1] * x[1] + x[2] * x[2]);
    } else if constexpr (POL == NDCHG_POL_QUAD) {
        return AccQuad<double>::det(x);
    } else {
        double d = 1.0;
        for (int b = 0; b < pol_bands(POL); ++b) d *= x[b];
        return d;
    }
}

template <typename T, int POL>
__global__ void __launch_bounds__(ENL_THREADS)
enl_kernel(const T* __restrict__ values, const long long rows, const long long cols, const int k, const long long s0,
           const long long s1, const long long s2, const long long s3, const int w, T* __restrict__ enl) {
    using Tile = EnlTile<T, POL>;
    constexpr int B = Tile::B, E = Tile::E, KT = Tile::KT;
    extern __shared__ double smem[];
    double* V = smem;                                                    // [ENL_TR][ENL_TC][KT][E]
    double* H = V + ENL_TR * ENL_TC * KT * E;                            // [ENL_TC][KT][E]
    double* S = H + ENL_TC * KT * E;                                     // [ENL_SEG][KT][E]
    const int tid = threadIdx.x, hw = w / 2;
    const int t0 = blockIdx.x * KT;
    const long long j0 = (long long)blockIdx.y * ENL_TC, i0 = (long long)blockIdx.z * ENL_TR;
    for (int e = tid; e < ENL_TR * ENL_TC * KT * E; e += ENL_THREADS) V[e] = 0.0;
    // columns whose window lies inside the image, and the input columns they read
    const long long cin0 = j0 - hw < 0 ? 0 : j0 - hw;
    const long long cin1 = j0 + ENL_TC + hw < cols ? j0 + ENL_TC + hw : cols;          // exclusive
    const long long rin0 = i0 - hw < 0 ? 0 : i0 - hw;
    const long long rin1 = i0 + ENL_TR + hw < rows ? i0 + ENL_TR + hw : rows;
    for (long long R = rin0; R < rin1; ++R) {
        __syncthreads();                                                 // the previous row's H is no longer read
        for (int e = tid; e < ENL_TC * KT * E; e += ENL_THREADS) H[e] = 0.0;
        for (long long cs = cin0; cs < cin1; cs += ENL_SEG) {
            __syncthreads();                                             // S and H free, H zeroed
            const int nseg = int(cin1 - cs < ENL_SEG ? cin1 - cs : ENL_SEG);
            for (int q = tid; q < nseg * KT; q += ENL_THREADS) {
                const int p = q / KT, tt = q - p * KT;
                double* x = S + q * E;
                if (t0 + tt < k) {
                    const T* src = values + R * s0 + (cs + p) * s1 + (long long)(t0 + tt) * s2;
                    bool finite = true;
                    for (int b = 0; b < B; ++b) {
                        x[b] = double(src[b * s3]);
                        finite = finite && isfinite(x[b]);
                    }
                    const double det = sample_det<POL>(x);
                    x[B] = finite && det > 0.0 ? log(det) : CUDART_NAN;
                }
            }
            __syncthreads();
            for (int e = tid; e < ENL_TC * KT * E; e += ENL_THREADS) {
                const int c = e / (KT * E), rest = e - c * (KT * E);
                const long long j = j0 + c;
                if (j < hw || j >= cols - hw) continue;                  // border column: no window
                // this segment's part of the window cols j - hw .. j + hw, left to right
                const long long a = j - hw > cs ? j - hw : cs;
                const long long z = j + hw + 1 < cs + nseg ? j + hw + 1 : cs + nseg;
                double sum = H[e];
                for (long long jj = a; jj < z; ++jj) sum += S[int(jj - cs) * KT * E + rest];
                H[e] = sum;
            }
        }
        __syncthreads();
        // add the row's window sums to the output rows i = i0 + r with |i - R| <= hw (only those rows are touched)
        const int r0 = R - hw - i0 > 0 ? int(R - hw - i0) : 0;
        const int r1 = R + hw - i0 < ENL_TR - 1 ? int(R + hw - i0) : ENL_TR - 1;
        constexpr int ROW = ENL_TC * KT * E;
        for (int e = r0 * ROW + tid; e < (r1 + 1) * ROW; e += ENL_THREADS) V[e] += H[e % ROW];
    }
    __syncthreads();
    const double N = double(w) * double(w);
    for (int o = tid; o < ENL_TR * ENL_TC * KT; o += ENL_THREADS) {
        const int r = o / (ENL_TC * KT), c = (o / KT) % ENL_TC, tt = o % KT;
        const long long i = i0 + r, j = j0 + c;
        const int t = t0 + tt;
        if (i >= rows || j >= cols || t >= k) continue;
        double out = CUDART_NAN;
        if (i >= hw && i < rows - hw && j >= hw && j < cols - hw) {
            const double* v = V + o * E;
            double M[B];
#pragma unroll
            for (int b = 0; b < B; ++b) M[b] = v[b] / N;
            const double detM = sample_det<POL>(M), delta = log(detM) - v[B] / N;
            if (!(detM > 0.0) || delta != delta) out = CUDART_NAN;
            else if (delta <= 0.0) out = CUDART_INF;                     // no speckle
            else if (delta < CUDART_INF) {
                constexpr int P = POL == NDCHG_POL_SINGLE ? 1 : POL == NDCHG_POL_DUAL || POL == NDCHG_POL_DUAL_DIAGONAL ? 2 : 3;
                out = enl_solve<P, POL == NDCHG_POL_SINGLE || POL == NDCHG_POL_DUAL || POL == NDCHG_POL_QUAD>(delta, N);
            }
        }
        enl[(i * cols + j) * k + t] = T(out);
    }
}

// ---- refined Lee filter (ndchg_refined_lee, include/ndchg.h) ------------------------------------------------------
// One CTA: a LEE_T x LEE_T tile of output pixels of one time step, one thread per pixel.  The time step is
// blockIdx.x, so the CTAs of neighbouring steps, which read the same pixel records, run close together.  The
// (LEE_T + N - 1)^2 input samples of the tile and its halo are staged in shared memory in double, band-planar, with
// the span as plane B; then the s x s box mean of the span at each of the (LEE_T + 2c)^2 subwindow centres the tile
// uses is formed once (nine output pixels read each).  Each thread then selects its mask and forms its masked sums
// over the whole N x N window, adding only the offsets inside the mask: all threads of a warp read the same offset
// at the same time, so the shared-memory reads stay conflict-free whichever masks the threads chose.
constexpr int LEE_T = 16, LEE_THREADS = LEE_T * LEE_T;

// number of diagonal bands of a layout, and the band of the d-th one
__host__ __device__ constexpr int lee_diagonals(const int pol) {
    return pol == NDCHG_POL_SINGLE ? 1 : pol == NDCHG_POL_DUAL || pol == NDCHG_POL_DUAL_DIAGONAL ? 2 : 3;
}
__host__ __device__ constexpr int lee_diagonal_band(const int pol, const int d) {
    return pol == NDCHG_POL_DUAL ? 3 * d : pol == NDCHG_POL_QUAD ? (d == 0 ? 0 : d == 1 ? 5 : 8) : d;
}

__host__ __device__ constexpr size_t lee_smem(const int bands, const int N) {
    return sizeof(double) * (size_t(bands + 1) * (LEE_T + N - 1) * (LEE_T + N - 1) +
                             size_t(LEE_T + N - (N - 1) / 2) * (LEE_T + N - (N - 1) / 2));
}

// scipy's 'reflect' (half-sample symmetric) index, one reflection deep; clamped so that the staged positions no
// output reads (beyond the last tile's pixels) stay inside the image
__device__ __forceinline__ long long lee_reflect(long long r, const long long n) {
    r = r < 0 ? -r - 1 : r >= n ? 2 * n - 1 - r : r;
    return r < 0 ? 0 : r >= n ? n - 1 : r;
}

__device__ __forceinline__ double add3_(const double a, const double b, const double c) { return add_(add_(a, b), c); }

template <typename T, int POL>
__global__ void __launch_bounds__(LEE_THREADS)
refined_lee_kernel(const T* __restrict__ values, const long long rows, const long long cols, const int k,
                   const long long s0, const long long s1, const long long s2, const long long s3, const int N,
                   const double looks, T* __restrict__ out) {
    constexpr int B = pol_bands(POL), P = lee_diagonals(POL);
    const int h = N / 2, s = (N - 1) / 2, c = (N - s) / 2;
    const int S = LEE_T + N - 1, BX = LEE_T + 2 * c;
    extern __shared__ double smem[];
    double* X = smem;                                                    // [B + 1][S][S]: the bands, then the span
    double* Y = X + B * S * S;
    double* box = Y + S * S;                                             // [BX][BX]
    const int tid = threadIdx.x, t = blockIdx.x;
    const long long i0 = (long long)blockIdx.z * LEE_T, j0 = (long long)blockIdx.y * LEE_T;
    for (int q = tid; q < S * S; q += LEE_THREADS) {
        const int a = q / S, b = q - a * S;
        const T* src = values + lee_reflect(i0 - h + a, rows) * s0 + lee_reflect(j0 - h + b, cols) * s1 + (long long)t * s2;
        double x[B];
#pragma unroll
        for (int band = 0; band < B; ++band) {
            x[band] = double(src[band * s3]);
            X[band * S * S + q] = x[band];
        }
        double y = x[lee_diagonal_band(POL, 0)];
#pragma unroll
        for (int d = 1; d < P; ++d) y = add_(y, x[lee_diagonal_band(POL, d)]);
        Y[q] = y;
    }
    __syncthreads();
    // box[p][q]: the mean of the span over staged rows p .. p + s - 1, columns q .. q + s - 1, i.e. the subwindow
    // centred at staged (p + h - c, q + h - c), since c + (s - 1) / 2 = h
    const double ss = double(s * s);
    for (int q = tid; q < BX * BX; q += LEE_THREADS) {
        const int a = q / BX, b = q - a * BX;
        double acc = 0.0;
        for (int u = 0; u < s; ++u)
            for (int v = 0; v < s; ++v) acc = add_(acc, Y[(a + u) * S + b + v]);
        box[q] = __ddiv_rn(acc, ss);
    }
    __syncthreads();
    const int ty = tid / LEE_T, tx = tid - ty * LEE_T;
    const long long i = i0 + ty, j = j0 + tx;
    if (i >= rows || j >= cols) return;
    // pixel (ty, tx) is staged at (ty + h, tx + h); its subwindow (u, v) is box[ty + u c][tx + v c]
    const double* mb = box + ty * BX + tx;
    const double m00 = mb[0], m01 = mb[c], m02 = mb[2 * c];
    const double m10 = mb[c * BX], m11 = mb[c * BX + c], m12 = mb[c * BX + 2 * c];
    const double m20 = mb[2 * c * BX], m21 = mb[2 * c * BX + c], m22 = mb[2 * c * BX + 2 * c];
    const double G0 = fabs(sub_(add3_(m02, m12, m22), add3_(m00, m10, m20)));
    const double G1 = fabs(sub_(add3_(m20, m21, m22), add3_(m00, m01, m02)));
    const double G2 = fabs(sub_(add3_(m01, m02, m12), add3_(m10, m20, m21)));
    const double G3 = fabs(sub_(add3_(m00, m01, m10), add3_(m12, m21, m22)));
    int e = 0;
    double Ge = G0;
    if (G1 > Ge) { e = 1; Ge = G1; }
    if (G2 > Ge) { e = 2; Ge = G2; }
    if (G3 > Ge) e = 3;
    const double first = e == 0 ? m10 : e == 1 ? m01 : e == 2 ? m02 : m00;
    const double second = e == 0 ? m12 : e == 1 ? m21 : e == 2 ? m20 : m22;
    // the mask is sg * (ay dy + ax dx) <= 0
    const int sg = fabs(sub_(second, m11)) < fabs(sub_(first, m11)) ? -1 : 1;
    const int ay = e == 0 ? 0 : sg, ax = e == 0 ? sg : e == 1 ? 0 : e == 2 ? -sg : sg;
    const double* Yw = Y + ty * S + tx;                                  // the window's top-left sample
    double sy = 0.0;
    for (int dy = 0; dy < N; ++dy)
        for (int dx = 0; dx < N; ++dx) {
            const double v = add_(sy, Yw[dy * S + dx]);
            sy = ay * (dy - h) + ax * (dx - h) <= 0 ? v : sy;
        }
    const double n = double(N * (N + 1) / 2);
    const double ybar = __ddiv_rn(sy, n);
    double vy = 0.0, sx[B];
#pragma unroll
    for (int band = 0; band < B; ++band) sx[band] = 0.0;
    for (int dy = 0; dy < N; ++dy)
        for (int dx = 0; dx < N; ++dx) {
            const bool in = ay * (dy - h) + ax * (dx - h) <= 0;
            const int o = dy * S + dx;
            const double dv = sub_(Yw[o], ybar);
            const double v = add_(vy, mul_(dv, dv));
            vy = in ? v : vy;
#pragma unroll
            for (int band = 0; band < B; ++band) {
                const double w = add_(sx[band], Yw[o + (band - B) * S * S]);
                sx[band] = in ? w : sx[band];
            }
        }
    const double var_y = __ddiv_rn(vy, n);
    const double sv2 = __ddiv_rn(1.0, looks);
    const double var_x = __ddiv_rn(sub_(var_y, mul_(mul_(ybar, ybar), sv2)), add_(1.0, sv2));
    const double wgt = var_x > 0.0 ? __ddiv_rn(var_x, var_y) : 0.0;
    T* o = out + ((i * cols + j) * k + t) * B;
    const int centre = (h * S + h) - B * S * S;                          // the pixel's own sample, band 0, from Yw
#pragma unroll
    for (int band = 0; band < B; ++band) {
        const double M = __ddiv_rn(sx[band], n);
        o[band] = T(add_(M, mul_(wgt, sub_(Yw[centre + band * S * S], M))));
    }
}

// ---- H / A / alpha decomposition (ndchg_h_a_alpha, include/ndchg.h) ----------------------------------------------
// One thread per sample (pixel, step), with 64-bit sample and element indices.  The bands are first scaled by a
// power of two (exact) so that their largest magnitude lies in [1, 2): squares and determinants can then neither
// overflow nor underflow, and the eigenvalues are scaled back exactly.  Quad layouts diagonalise the Pauli coherency
// matrix T by cyclic complex Jacobi; alpha needs only |e_i[0]|^2, the first row of the accumulated rotation V
// (T = V diag(lambda) V^H), so that row is all that is kept.  Dual layouts use the closed form of the 2 x 2 matrix.
constexpr int HAA_THREADS = 256, HAA_MAX_SWEEPS = 16;
constexpr double HAA_TAU = 1e-9;

__host__ __device__ constexpr int haa_outputs(const int pol) {
    return pol == NDCHG_POL_QUAD || pol == NDCHG_POL_QUAD_DIAGONAL ? 6 : 4;
}

// (x, y) <- (c x - s ph y, s x + c ph y): columns p and q of a row times the rotation of haa_rotate
__device__ __forceinline__ void haa_rot(double2& x, double2& y, const double c, const double s, const double2 ph) {
    const double2 py = make_double2(ph.x * y.x - ph.y * y.y, ph.x * y.y + ph.y * y.x);
    const double2 nx = make_double2(c * x.x - s * py.x, c * x.y - s * py.y);
    y = make_double2(s * x.x + c * py.x, s * x.y + c * py.y);
    x = nx;
}

__device__ __forceinline__ double2 haa_conj(const double2 a) { return make_double2(a.x, -a.y); }

// One Jacobi rotation J of the plane (P, Q), P < Q, that zeroes T[P][Q] = m e^(i phi): J = diag(1, e^(-i phi)) R
// on (P, Q) with the real rotation R = [[c, s], [-s, c]] of Numerical Recipes' jacobi, T <- J^H T J, V <- V J.
// d: the real diagonal; u[r]: the upper entry of the plane without index r (u[2] = T01, u[1] = T02, u[0] = T12);
// v: row 0 of V.
template <int P, int Q>
__device__ __forceinline__ void haa_rotate(double d[3], double2 u[3], double2 v[3]) {
    constexpr int R = 3 - P - Q;
    const double m = hypot(u[R].x, u[R].y);
    if (m == 0.0) return;
    const double2 ph = make_double2(u[R].x / m, -u[R].y / m);
    const double theta = (d[Q] - d[P]) / (2.0 * m);
    const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + hypot(theta, 1.0));
    const double c = 1.0 / hypot(t, 1.0), s = t * c;
    d[P] -= t * m;
    d[Q] += t * m;
    u[R] = make_double2(0.0, 0.0);
    // row R of T holds T[R][P] and T[R][Q]; below the diagonal they are the conjugates of the stored upper entries
    double2 rp = R > P ? haa_conj(u[Q]) : u[Q], rq = R > Q ? haa_conj(u[P]) : u[P];
    haa_rot(rp, rq, c, s, ph);
    u[Q] = R > P ? haa_conj(rp) : rp;
    u[P] = R > Q ? haa_conj(rq) : rq;
    haa_rot(v[P], v[Q], c, s, ph);
}

template <typename T, int POL>
__global__ void __launch_bounds__(HAA_THREADS)
h_a_alpha_kernel(const T* __restrict__ values, const long long cols, const long long k, const long long samples,
                 const long long s0, const long long s1, const long long s2, const long long s3, T* __restrict__ out) {
    constexpr int B = pol_bands(POL), NO = haa_outputs(POL);
    constexpr bool QUAD = POL == NDCHG_POL_QUAD || POL == NDCHG_POL_QUAD_DIAGONAL;
    constexpr int K = QUAD ? 3 : 2;                                      // matrix size
    const long long g = (long long)blockIdx.x * HAA_THREADS + threadIdx.x;
    if (g >= samples) return;
    const long long pix = g / k, t = g - pix * k, i = pix / cols, j = pix - i * cols;
    const T* src = values + i * s0 + j * s1 + t * s2;
    T* o = out + g * NO;
    double x[B], amax = 0.0;
    bool finite = true;
#pragma unroll
    for (int b = 0; b < B; ++b) {
        x[b] = double(src[b * s3]);
        finite = finite && isfinite(x[b]);
        amax = fmax(amax, fabs(x[b]));
    }
    if (!finite) {
#pragma unroll
        for (int q = 0; q < NO; ++q) o[q] = T(CUDART_NAN);
        return;
    }
    const int e = amax > 0.0 ? ilogb(amax) : 0;
#pragma unroll
    for (int b = 0; b < B; ++b) x[b] = scalbn(x[b], -e);
    double lam[K], w[K];                                                 // eigenvalues (descending), |e_i[0]|^2
    bool tie[K - 1];
    if constexpr (QUAD) {
        // C3 = [C11, C12, C13, C22, C23, C33]; the diagonal layout has no off-diagonal bands
        const double c11 = x[0], c22 = x[POL == NDCHG_POL_QUAD ? 5 : 1], c33 = x[POL == NDCHG_POL_QUAD ? 8 : 2];
        const double c12r = POL == NDCHG_POL_QUAD ? x[1] : 0.0, c12i = POL == NDCHG_POL_QUAD ? x[2] : 0.0;
        const double c13r = POL == NDCHG_POL_QUAD ? x[3] : 0.0, c13i = POL == NDCHG_POL_QUAD ? x[4] : 0.0;
        const double c23r = POL == NDCHG_POL_QUAD ? x[6] : 0.0, c23i = POL == NDCHG_POL_QUAD ? x[7] : 0.0;
        const double r2 = 0.70710678118654752440;                        // 1 / sqrt(2)
        double d[3] = {0.5 * (c11 + 2.0 * c13r + c33), 0.5 * (c11 - 2.0 * c13r + c33), c22};
        double2 u[3] = {make_double2((c12r - c23r) * r2, (c12i + c23i) * r2),          // T23 = (C12 - conj C23) / sqrt 2
                        make_double2((c12r + c23r) * r2, (c12i - c23i) * r2),          // T13 = (C12 + conj C23) / sqrt 2
                        make_double2(0.5 * (c11 - c33), -c13i)};                         // T12 = (C11 - C33) / 2 - i Im C13
        double2 v[3] = {make_double2(1.0, 0.0), make_double2(0.0, 0.0), make_double2(0.0, 0.0)};
        // until the off-diagonal Frobenius norm is <= eps ||T||_F
        constexpr double eps2 = 2.220446049250313e-16 * 2.220446049250313e-16;
        for (int sweep = 0; sweep < HAA_MAX_SWEEPS; ++sweep) {
            const double off = 2.0 * (u[0].x * u[0].x + u[0].y * u[0].y + u[1].x * u[1].x + u[1].y * u[1].y +
                                      u[2].x * u[2].x + u[2].y * u[2].y);
            if (off <= eps2 * (d[0] * d[0] + d[1] * d[1] + d[2] * d[2] + off)) break;
            haa_rotate<0, 1>(d, u, v);
            haa_rotate<0, 2>(d, u, v);
            haa_rotate<1, 2>(d, u, v);
        }
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            lam[q] = d[q];
            w[q] = v[q].x * v[q].x + v[q].y * v[q].y;
        }
        // sort descending, |e[0]|^2 along
#define HAA_ORDER(a, b)                                                                 \
        if (lam[a] < lam[b]) {                                                          \
            const double tl = lam[a], tw = w[a];                                        \
            lam[a] = lam[b]; w[a] = w[b]; lam[b] = tl; w[b] = tw;                       \
        }
        HAA_ORDER(0, 1) HAA_ORDER(1, 2) HAA_ORDER(0, 1)
#undef HAA_ORDER
    } else {
        // C2 = [[C11, C12], [conj C12, C22]]: lambda = (C11 + C22) / 2 +- r, r = hypot((C11 - C22) / 2, |C12|);
        // lambda2 = det / lambda1 (no cancellation); |e_1[0]|^2 = (lambda1 - C22) / (2 r), |e_2[0]|^2 =
        // (lambda1 - C11) / (2 r), each side formed without cancellation, (lambda1 - C11)(lambda1 - C22) = |C12|^2
        const double c11 = x[0], c22 = x[POL == NDCHG_POL_DUAL ? 3 : 1];
        const double b2 = POL == NDCHG_POL_DUAL ? x[1] * x[1] + x[2] * x[2] : 0.0;
        const double delta = 0.5 * (c11 - c22), r = hypot(delta, sqrt(b2));
        lam[0] = 0.5 * (c11 + c22) + r;
        lam[1] = lam[0] > 0.0 ? (c11 * c22 - b2) / lam[0] : lam[0];      // lambda1 <= 0: s = 0 below
        const double a1 = delta >= 0.0 ? delta + r : b2 / (r - delta);   // lambda1 - C22
        const double a2 = delta >= 0.0 ? b2 / (delta + r) : r - delta;   // lambda1 - C11
        w[0] = a1 / (2.0 * r);
        w[1] = a2 / (2.0 * r);
    }
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < K; ++q) {
        lam[q] = fmax(lam[q], 0.0);
        s += lam[q];
    }
#pragma unroll
    for (int q = 0; q < K - 1; ++q) tie[q] = lam[q] - lam[q + 1] <= HAA_TAU * s;
    double H = CUDART_NAN, A = CUDART_NAN, alpha = CUDART_NAN;
    if (s > 0.0) {
        // the tie clusters share the mean of their |e[0]|^2: the (0, 0) entry of the cluster's projector / m
        if constexpr (K == 2) {
            if (tie[0]) w[0] = w[1] = 0.5;
        } else {
            if (tie[0] && tie[1]) w[0] = w[1] = w[2] = (w[0] + w[1] + w[2]) / 3.0;
            else if (tie[0]) w[0] = w[1] = 0.5 * (w[0] + w[1]);
            else if (tie[1]) w[1] = w[2] = 0.5 * (w[1] + w[2]);
        }
        H = 0.0;
        alpha = 0.0;
#pragma unroll
        for (int q = 0; q < K; ++q) {
            const double p = lam[q] / s;
            if (p > 0.0) H -= p * log(p);
            alpha += p * acos(fmin(fmax(sqrt(w[q]), 0.0), 1.0));
        }
        H /= K == 3 ? 1.0986122886681098 : 0.69314718055994531;         // ln 3, ln 2
        alpha *= 57.295779513082321;                                     // 180 / pi
        if constexpr (K == 3) A = lam[1] <= HAA_TAU * s ? 0.0 : (lam[1] - lam[2]) / (lam[1] + lam[2]);
    }
    int q = 0;
    o[q++] = T(H);
    if constexpr (K == 3) o[q++] = T(A);
    o[q++] = T(alpha);
#pragma unroll
    for (int r = 0; r < K; ++r) o[q++] = T(scalbn(lam[r], e));
}

// ---- H / alpha zones and the Wishart classification (ndchg_h_alpha_zones, ndchg_wishart_classify) -----------------
// Zones: h_a_alpha_kernel runs unchanged into device scratch (ZONE_CHUNK samples at a time), then one thread per
// sample reads its H, A, alpha.  Wishart: three kernels per iteration on one stream.  `wishart_assign_kernel` reads
// the cube once: one CTA owns a fixed chunk of WIS_CHUNK consecutive samples (the partition depends on the sample
// count only, never on the device), each warp 32 samples at a time.  A lane takes the argmin of its sample, then the
// warp stages its 32 (label, bands) in shared memory and lane e of lane group q adds accumulator column e (a band,
// or the count) of samples q, q + Q, ... in lane order into the group's own K x (B + 1) copy.  The copies are added
// in (warp, group) order into one partial per chunk; `wishart_reduce_kernel` adds the chunk partials of every
// accumulator in a fixed tree, and `wishart_centres_kernel` (one warp) turns the sums into the next (g, w) table.
// No floating-point atomics, so the sums are bit-identical from run to run, on any B200 and for any strides.
constexpr int WIS_THREADS = 256, WIS_WARPS = WIS_THREADS / 32, WIS_GROUPS = 16, WIS_MAX_CLASSES = 32;
constexpr long long WIS_CHUNK = (long long)WIS_THREADS * WIS_GROUPS;    // samples per CTA, i.e. per chunk of the sums
constexpr long long ZONE_CHUNK = 1LL << 24;
constexpr int WIS_REDUCE_THREADS = 256;

// lane groups of a warp in the accumulation: Q groups of B + 1 lanes
__host__ __device__ constexpr int wis_groups(const int pol) { return 32 / (pol_bands(pol) + 1); }

__host__ __device__ constexpr size_t wis_smem(const int pol, const int K) {
    return sizeof(double) * size_t(WIS_WARPS) * wis_groups(pol) * K * (pol_bands(pol) + 1);
}

// device state of one ndchg_wishart_classify call; the sums and the chunk partials follow it in the same scratch
struct WisState {
    unsigned long long changed;                      // samples whose label changed in the current pass
    unsigned long long valid;                        // valid samples (counted in iteration 0)
    unsigned done;                                   // the loop has stopped: every later launch returns at once
    unsigned bad;                                    // an initial label > K
    unsigned active;                                 // active classes after the last centres kernel
    int act[WIS_MAX_CLASSES];
    double g[WIS_MAX_CLASSES];                       // ln det V_m
    double w[WIS_MAX_CLASSES * 9];                   // [K][B]: the weights of the distance
};

template <typename T, int POL>
__global__ void __launch_bounds__(HAA_THREADS)
h_alpha_zone_kernel(const T* __restrict__ haa, const long long n, const int anisotropy, unsigned char* __restrict__ zones) {
    constexpr bool QUAD = POL == NDCHG_POL_QUAD || POL == NDCHG_POL_QUAD_DIAGONAL;
    const long long g = (long long)blockIdx.x * HAA_THREADS + threadIdx.x;
    if (g >= n) return;
    const T* o = haa + g * haa_outputs(POL);
    const double H = double(o[0]), alpha = double(o[QUAD ? 2 : 1]);
    unsigned char z = 0;
    if (!isnan(H) && !isnan(alpha)) {
        if (H >= 0.9) z = alpha >= 55.0 ? 1 : alpha >= 40.0 ? 2 : 3;
        else if (H >= 0.5) z = alpha >= 50.0 ? 4 : alpha >= 40.0 ? 5 : 6;
        else z = alpha >= 47.5 ? 7 : alpha >= 42.5 ? 8 : 9;
        if (QUAD && anisotropy && double(o[1]) > 0.5) z += 9;
    }
    zones[g] = z;
}

// sets `bad` (and `done`) if any initial label exceeds K
__global__ void __launch_bounds__(256)
wishart_check_kernel(const unsigned char* __restrict__ labels, const long long n, const int K, WisState* st) {
    bool bad = false;
    for (long long g = (long long)blockIdx.x * 256 + threadIdx.x; g < n; g += (long long)gridDim.x * 256) bad |= labels[g] > K;
    if (__syncthreads_or(bad) && threadIdx.x == 0) {
        st->bad = 1;
        st->done = 1;
    }
}

// One pass over the cube.  ASSIGN = false is iteration 0: the initial labels are kept (invalid samples set to 0) and
// the valid samples are counted; ASSIGN = true takes the argmin and counts the changed labels.  Either way the pass
// accumulates, per label, the band sums and the count of its valid samples into partials[a * nchunk + chunk].
// FLAT: the (rows, cols, k) axes collapse into one of stride s2, so sample g starts at element g * s2.
template <typename T, int POL, bool ASSIGN>
__global__ void __launch_bounds__(WIS_THREADS)
wishart_assign_kernel(const T* __restrict__ values, const long long cols, const long long k, const long long samples,
                      const long long s0, const long long s1, const long long s2, const long long s3, const bool flat,
                      unsigned char* __restrict__ labels, WisState* __restrict__ st, const int K,
                      double* __restrict__ partials, const long long nchunk) {
    constexpr int B = pol_bands(POL), E = B + 1, Q = wis_groups(POL);
    __shared__ double tab_g[WIS_MAX_CLASSES], tab_w[WIS_MAX_CLASSES * B];
    __shared__ int tab_act[WIS_MAX_CLASSES];
    __shared__ T stage[WIS_WARPS][32][B];
    __shared__ unsigned char slab[WIS_WARPS][32];
    __shared__ unsigned long long cta_count;
    extern __shared__ double acc[];                                      // [WIS_WARPS][Q][K][E]
    if (st->done) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (ASSIGN) {
        for (int q = tid; q < K * B; q += WIS_THREADS) tab_w[q] = st->w[q];
        if (tid < K) {
            tab_g[tid] = st->g[tid];
            tab_act[tid] = st->act[tid];
        }
    }
    for (int q = tid; q < WIS_WARPS * Q * K * E; q += WIS_THREADS) acc[q] = 0.0;
    if (tid == 0) cta_count = 0;
    __syncthreads();
    double* myacc = acc + warp * Q * K * E;
    const int grp = lane / E, col = lane - grp * E;                       // the lane's copy and accumulator column
    unsigned count = 0;
    const long long base = (long long)blockIdx.x * WIS_CHUNK + warp * (32 * WIS_GROUPS);
    for (int r = 0; r < WIS_GROUPS; ++r) {
        const long long g = base + r * 32 + lane;
        int lab = 0;
        if (g < samples) {
            long long off;
            if (flat) {
                off = g * s2;
            } else {
                const long long pix = g / k, t = g - pix * k, i = pix / cols, j = pix - i * cols;
                off = i * s0 + j * s1 + t * s2;
            }
            const T* src = values + off;
            double x[B];
            bool finite = true;
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const T v = src[b * s3];
                stage[warp][lane][b] = v;
                x[b] = double(v);
                finite = finite && isfinite(x[b]);
            }
            double tr = x[lee_diagonal_band(POL, 0)];
#pragma unroll
            for (int d = 1; d < lee_diagonals(POL); ++d) tr = add_(tr, x[lee_diagonal_band(POL, d)]);
            const int old = labels[g];
            if (finite && tr > 0.0) {
                if (ASSIGN) {
                    double best = CUDART_INF;
                    for (int m = 0; m < K; ++m) {
                        if (!tab_act[m]) continue;
                        const double* w = tab_w + m * B;
                        double d = tab_g[m];
#pragma unroll
                        for (int b = 0; b < B; ++b) d = add_(d, mul_(w[b], x[b]));
                        if (d < best) {
                            best = d;
                            lab = m + 1;
                        }
                    }
                    if (lab != old) {
                        labels[g] = (unsigned char)lab;
                        ++count;
                    }
                } else {
                    lab = old;
                    ++count;
                }
            } else if (!ASSIGN && old != 0) {
                labels[g] = 0;
            }
        }
        slab[warp][lane] = (unsigned char)lab;
        __syncwarp();
        if (grp < Q) {
            double* a = myacc + grp * K * E + col;
            for (int s = grp; s < 32; s += Q) {
                const int m = slab[warp][s];
                if (m) a[(m - 1) * E] = add_(a[(m - 1) * E], col < B ? double(stage[warp][s][col < B ? col : 0]) : 1.0);
            }
        }
        __syncwarp();
    }
    count = __reduce_add_sync(0xffffffffu, count);
    if (lane == 0 && count) atomicAdd(&cta_count, (unsigned long long)count);
    __syncthreads();
    if (tid == 0 && cta_count) atomicAdd(ASSIGN ? &st->changed : &st->valid, cta_count);
    for (int a = tid; a < K * E; a += WIS_THREADS) {
        double s = 0.0;
        for (int c = 0; c < WIS_WARPS * Q; ++c) s = add_(s, acc[c * K * E + a]);
        partials[a * nchunk + blockIdx.x] = s;
    }
}

// sums[a] = the chunk partials of accumulator a = blockIdx.x, added in a fixed tree
__global__ void __launch_bounds__(WIS_REDUCE_THREADS)
wishart_reduce_kernel(const double* __restrict__ partials, const long long nchunk, double* __restrict__ sums,
                      const WisState* __restrict__ st) {
    __shared__ double red[WIS_REDUCE_THREADS];
    if (st->done) return;
    const int tid = threadIdx.x;
    const double* p = partials + blockIdx.x * nchunk;
    double s = 0.0;
    for (long long c = tid; c < nchunk; c += WIS_REDUCE_THREADS) s = add_(s, p[c]);
    red[tid] = s;
    __syncthreads();
    for (int h = WIS_REDUCE_THREADS / 2; h > 0; h >>= 1) {
        if (tid < h) red[tid] = add_(red[tid], red[tid + h]);
        __syncthreads();
    }
    if (tid == 0) sums[blockIdx.x] = red[0];
}

// One warp, thread m = class m + 1: the mean V, det V, the active flag, W = adj(V) / det V and the (g, w) table of
// the next pass; writes the outputs and decides whether the loop stops after iteration `it`.
template <int POL>
__global__ void __launch_bounds__(32)
wishart_centres_kernel(WisState* __restrict__ st, const double* __restrict__ sums, const int K, const unsigned it,
                       const unsigned max_iter, const double tol, double* __restrict__ centres,
                       long long* __restrict__ counts, unsigned* __restrict__ iterations) {
    constexpr int B = pol_bands(POL), E = B + 1, P = lee_diagonals(POL);
    if (st->done) return;
    const int m = threadIdx.x;
    bool act = false;
    if (m < K) {
        const double n = sums[m * E + B];
        double V[B];
#pragma unroll
        for (int b = 0; b < B; ++b) V[b] = __ddiv_rn(sums[m * E + b], n);
        double tr = V[lee_diagonal_band(POL, 0)];
#pragma unroll
        for (int d = 1; d < P; ++d) tr = add_(tr, V[lee_diagonal_band(POL, d)]);
        const double q = __ddiv_rn(tr, double(P));
        const double qp = P == 2 ? mul_(q, q) : mul_(mul_(q, q), q);
        double det, w[B];
        if constexpr (POL == NDCHG_POL_DUAL) {
            const double a = V[0], br = V[1], bi = V[2], d = V[3];
            det = sub_(mul_(a, d), add_(mul_(br, br), mul_(bi, bi)));
            w[0] = __ddiv_rn(d, det);
            w[1] = mul_(-2.0, __ddiv_rn(br, det));
            w[2] = mul_(-2.0, __ddiv_rn(bi, det));
            w[3] = __ddiv_rn(a, det);
        } else if constexpr (POL == NDCHG_POL_QUAD) {
            const double a = V[0], br = V[1], bi = V[2], cr = V[3], ci = V[4], d = V[5], er = V[6], ei = V[7], g = V[8];
            const double re_bec = add_(mul_(sub_(mul_(br, er), mul_(bi, ei)), cr), mul_(add_(mul_(br, ei), mul_(bi, er)), ci));
            const double e2 = add_(mul_(er, er), mul_(ei, ei)), c2 = add_(mul_(cr, cr), mul_(ci, ci));
            const double b2 = add_(mul_(br, br), mul_(bi, bi));
            det = add_(mul_(mul_(a, d), g), mul_(2.0, re_bec));
            det = sub_(det, mul_(a, e2));
            det = sub_(det, mul_(d, c2));
            det = sub_(det, mul_(g, b2));
            // adj(V) / det: W12 = (c conj(e) - b g) / det, W13 = (b e - c d) / det, W23 = (c conj(b) - a e) / det
            w[0] = __ddiv_rn(sub_(mul_(d, g), e2), det);
            w[5] = __ddiv_rn(sub_(mul_(a, g), c2), det);
            w[8] = __ddiv_rn(sub_(mul_(a, d), b2), det);
            w[1] = mul_(2.0, __ddiv_rn(sub_(add_(mul_(cr, er), mul_(ci, ei)), mul_(br, g)), det));
            w[2] = mul_(2.0, __ddiv_rn(sub_(sub_(mul_(ci, er), mul_(cr, ei)), mul_(bi, g)), det));
            w[3] = mul_(2.0, __ddiv_rn(sub_(sub_(mul_(br, er), mul_(bi, ei)), mul_(cr, d)), det));
            w[4] = mul_(2.0, __ddiv_rn(sub_(add_(mul_(br, ei), mul_(bi, er)), mul_(ci, d)), det));
            w[6] = mul_(2.0, __ddiv_rn(sub_(add_(mul_(cr, br), mul_(ci, bi)), mul_(a, er)), det));
            w[7] = mul_(2.0, __ddiv_rn(sub_(sub_(mul_(ci, br), mul_(cr, bi)), mul_(a, ei)), det));
        } else {
            det = V[0];
#pragma unroll
            for (int b = 1; b < B; ++b) det = mul_(det, V[b]);
#pragma unroll
            for (int b = 0; b < B; ++b) w[b] = __ddiv_rn(1.0, V[b]);
        }
        act = n >= 1.0 && det > mul_(1e-12, qp);
#pragma unroll
        for (int b = 0; b < B; ++b) {
            centres[m * B + b] = act ? V[b] : CUDART_NAN;
            st->w[m * B + b] = act ? w[b] : 0.0;
        }
        st->g[m] = act ? log(det) : 0.0;
        st->act[m] = act;
        counts[m] = (long long)n;
    }
    const unsigned nact = __popc(__ballot_sync(0xffffffffu, act));
    if (m == 0) {
        const unsigned long long changed = st->changed;
        st->active = nact;
        st->changed = 0;
        *iterations = it;
        if (it >= max_iter || nact == 0 || (it >= 1 && double(changed) <= __dmul_rn(tol, double(st->valid)))) st->done = 1;
    }
}

}  // namespace ndchg

struct ChgDeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit ChgDeviceGuard(const void* ptr) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess || attr.type != cudaMemoryTypeDevice) {
            cudaGetLastError();
            ok = false;
            return;
        }
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != attr.device && cudaSetDevice(attr.device) != cudaSuccess) ok = false;
        if (prev == attr.device) prev = -1;
    }
    ~ChgDeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

static int check_args(const void* values, const int64_t* shape, const int64_t* strides, int dtype, const void* out, uint32_t n) {
    if (!values || !shape || !strides || !out) return chg_fail(NDNLM_EINVAL, "null argument");
    if (dtype != NDCHG_F32 && dtype != NDCHG_F64) return chg_fail(NDNLM_EDTYPE, "No matching signature found (only float32 / float64 data is supported)");
    if (shape[0] < 1 || shape[1] < 1 || shape[0] * shape[1] > 0x7fffffffLL * 128) return chg_fail(NDNLM_EINVAL, "shape out of range");
    if (shape[2] < 2 || shape[2] > 0x7fffffffLL) return chg_fail(NDNLM_EINVAL, "the omnibus test needs at least 2 time steps");
    if (n < 1) return chg_fail(NDNLM_EINVAL, "the number of looks n must be >= 1");
    return NDNLM_OK;
}

template <typename A>
static int launch_change(const void* values, const int64_t* shape, const int64_t* strides, uint8_t* result, double alpha,
                         uint32_t n, void* stream) {
    const long long pixels = shape[0] * shape[1];
    const unsigned grid = unsigned((pixels + 127) / 128);
    ndchg::change_detection_kernel<A><<<grid, 128, 0, (cudaStream_t)stream>>>(
        (const typename A::value_type*)values, shape[0], shape[1], int(shape[2]), strides[0], strides[1], strides[2],
        strides[3], result, alpha, n);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "launch failed: %s", cudaGetErrorString(e));
    return NDNLM_OK;
}

template <typename A>
static int launch_probability(const void* values, const int64_t* shape, const int64_t* strides, void* prob, uint32_t n,
                              void* stream) {
    const long long pixels = shape[0] * shape[1];
    const unsigned grid = unsigned((pixels + 127) / 128);
    ndchg::omnibus_probability_kernel<A><<<grid, 128, 0, (cudaStream_t)stream>>>(
        (const typename A::value_type*)values, shape[0], shape[1], int(shape[2]), strides[0], strides[1], strides[2],
        strides[3], (typename A::value_type*)prob, n);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "launch failed: %s", cudaGetErrorString(e));
    return NDNLM_OK;
}

// calls f(A()) with the accumulator of layout `pol` (other than dual-pol, which has its own entry points) for data type T
template <typename T, typename F>
static int with_layout(int pol, F&& f) {
    switch (pol) {
        case NDCHG_POL_SINGLE: return f(ndchg::AccDiag<T, 1>());
        case NDCHG_POL_QUAD: return f(ndchg::AccQuad<T>());
        case NDCHG_POL_DUAL_DIAGONAL: return f(ndchg::AccDiag<T, 2>());
        case NDCHG_POL_QUAD_DIAGONAL: return f(ndchg::AccDiag<T, 3>());
        default: return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    }
}

static int check_pol(int pol, uint32_t n) {
    if (pol < NDCHG_POL_DUAL || pol > NDCHG_POL_QUAD_DIAGONAL) return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    if (pol == NDCHG_POL_QUAD && n < 3)
        return chg_fail(NDNLM_EINVAL, "quad-pol needs n >= 3 looks (the sample covariance of fewer looks is singular)");
    return NDNLM_OK;
}

extern "C" int ndchg_change_detection(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype,
                                      uint8_t* result, double alpha, uint32_t n, void* stream) {
    int rc = check_args(values, shape, strides, dtype, result, n);
    if (rc) return rc;
    ChgDeviceGuard guard(result);
    if (!guard.ok) return chg_fail(NDNLM_EINVAL, "result is not a CUDA device pointer");
    if (dtype == NDCHG_F64) return launch_change<ndchg::Acc<double>>(values, shape, strides, result, alpha, n, stream);
    return launch_change<ndchg::Acc<float>>(values, shape, strides, result, alpha, n, stream);
}

extern "C" int ndchg_omnibus_probability(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype,
                                         void* prob, uint32_t n, void* stream) {
    int rc = check_args(values, shape, strides, dtype, prob, n);
    if (rc) return rc;
    ChgDeviceGuard guard(prob);
    if (!guard.ok) return chg_fail(NDNLM_EINVAL, "prob is not a CUDA device pointer");
    if (dtype == NDCHG_F64) return launch_probability<ndchg::Acc<double>>(values, shape, strides, prob, n, stream);
    return launch_probability<ndchg::Acc<float>>(values, shape, strides, prob, n, stream);
}

extern "C" int ndchg_change_detection_pol(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype,
                                          int pol, uint8_t* result, double alpha, uint32_t n, void* stream) {
    int rc = check_args(values, shape, strides, dtype, result, n);
    if (!rc) rc = check_pol(pol, n);
    if (rc) return rc;
    if (pol == NDCHG_POL_DUAL) return ndchg_change_detection(values, shape, strides, dtype, result, alpha, n, stream);
    ChgDeviceGuard guard(result);
    if (!guard.ok) return chg_fail(NDNLM_EINVAL, "result is not a CUDA device pointer");
    auto go = [&](auto acc) { return launch_change<decltype(acc)>(values, shape, strides, result, alpha, n, stream); };
    return dtype == NDCHG_F64 ? with_layout<double>(pol, go) : with_layout<float>(pol, go);
}

extern "C" int ndchg_omnibus_probability_pol(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype,
                                             int pol, void* prob, uint32_t n, void* stream) {
    int rc = check_args(values, shape, strides, dtype, prob, n);
    if (!rc) rc = check_pol(pol, n);
    if (rc) return rc;
    if (pol == NDCHG_POL_DUAL) return ndchg_omnibus_probability(values, shape, strides, dtype, prob, n, stream);
    ChgDeviceGuard guard(prob);
    if (!guard.ok) return chg_fail(NDNLM_EINVAL, "prob is not a CUDA device pointer");
    auto go = [&](auto acc) { return launch_probability<decltype(acc)>(values, shape, strides, prob, n, stream); };
    return dtype == NDCHG_F64 ? with_layout<double>(pol, go) : with_layout<float>(pol, go);
}

template <typename T, int POL>
static int launch_direction(const void* values, const int64_t* shape, const int64_t* strides, uint8_t* result, void* stream) {
    const long long pixels = shape[0] * shape[1];
    const unsigned grid = unsigned((pixels + 127) / 128);
    ndchg::change_direction_kernel<T, POL><<<grid, 128, 0, (cudaStream_t)stream>>>(
        (const T*)values, shape[0], shape[1], int(shape[2]), strides[0], strides[1], strides[2], strides[3], result);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "launch failed: %s", cudaGetErrorString(e));
    return NDNLM_OK;
}

template <typename T>
static int launch_direction(int pol, const void* values, const int64_t* shape, const int64_t* strides, uint8_t* result,
                            void* stream) {
    switch (pol) {
        case NDCHG_POL_DUAL: return launch_direction<T, NDCHG_POL_DUAL>(values, shape, strides, result, stream);
        case NDCHG_POL_SINGLE: return launch_direction<T, NDCHG_POL_SINGLE>(values, shape, strides, result, stream);
        case NDCHG_POL_QUAD: return launch_direction<T, NDCHG_POL_QUAD>(values, shape, strides, result, stream);
        case NDCHG_POL_DUAL_DIAGONAL: return launch_direction<T, NDCHG_POL_DUAL_DIAGONAL>(values, shape, strides, result, stream);
        case NDCHG_POL_QUAD_DIAGONAL: return launch_direction<T, NDCHG_POL_QUAD_DIAGONAL>(values, shape, strides, result, stream);
        default: return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    }
}

extern "C" int ndchg_change_direction(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype,
                                      int pol, uint8_t* result, double alpha, uint32_t n, void* stream) {
    int rc = check_args(values, shape, strides, dtype, result, n);
    if (!rc) rc = check_pol(pol, n);
    if (rc) return rc;
    ChgDeviceGuard guard(result);
    if (!guard.ok) return chg_fail(NDNLM_EINVAL, "result is not a CUDA device pointer");
    rc = ndchg_change_detection_pol(values, shape, strides, dtype, pol, result, alpha, n, stream);
    if (rc) return rc;
    return dtype == NDCHG_F64 ? launch_direction<double>(pol, values, shape, strides, result, stream)
                              : launch_direction<float>(pol, values, shape, strides, result, stream);
}

template <typename T, int POL>
static int launch_enl(const void* values, const int64_t* shape, const int64_t* strides, uint32_t window, void* enl,
                      void* stream) {
    using Tile = ndchg::EnlTile<T, POL>;
    const dim3 grid(unsigned((shape[2] + Tile::KT - 1) / Tile::KT), unsigned((shape[1] + ndchg::ENL_TC - 1) / ndchg::ENL_TC),
                    unsigned((shape[0] + ndchg::ENL_TR - 1) / ndchg::ENL_TR));
    if (grid.y > 65535 || grid.z > 65535) return chg_fail(NDNLM_EINVAL, "image of %lld x %lld pixels is too large for ndchg_enl",
                                                          (long long)shape[0], (long long)shape[1]);
    cudaError_t e = cudaFuncSetAttribute(ndchg::enl_kernel<T, POL>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(Tile::smem));
    if (e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "shared memory of %zu bytes: %s", Tile::smem, cudaGetErrorString(e));
    ndchg::enl_kernel<T, POL><<<grid, ndchg::ENL_THREADS, Tile::smem, (cudaStream_t)stream>>>(
        (const T*)values, shape[0], shape[1], int(shape[2]), strides[0], strides[1], strides[2], strides[3], int(window), (T*)enl);
    e = cudaGetLastError();
    if (e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "launch failed: %s", cudaGetErrorString(e));
    return NDNLM_OK;
}

template <typename T>
static int launch_enl(int pol, const void* values, const int64_t* shape, const int64_t* strides, uint32_t window, void* enl,
                      void* stream) {
    switch (pol) {
        case NDCHG_POL_DUAL: return launch_enl<T, NDCHG_POL_DUAL>(values, shape, strides, window, enl, stream);
        case NDCHG_POL_SINGLE: return launch_enl<T, NDCHG_POL_SINGLE>(values, shape, strides, window, enl, stream);
        case NDCHG_POL_QUAD: return launch_enl<T, NDCHG_POL_QUAD>(values, shape, strides, window, enl, stream);
        case NDCHG_POL_DUAL_DIAGONAL: return launch_enl<T, NDCHG_POL_DUAL_DIAGONAL>(values, shape, strides, window, enl, stream);
        case NDCHG_POL_QUAD_DIAGONAL: return launch_enl<T, NDCHG_POL_QUAD_DIAGONAL>(values, shape, strides, window, enl, stream);
        default: return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    }
}

extern "C" int ndchg_enl(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol,
                         uint32_t window, void* enl, void* stream) {
    if (!values || !shape || !strides || !enl) return chg_fail(NDNLM_EINVAL, "null argument");
    if (dtype != NDCHG_F32 && dtype != NDCHG_F64) return chg_fail(NDNLM_EDTYPE, "No matching signature found (only float32 / float64 data is supported)");
    if (pol < NDCHG_POL_DUAL || pol > NDCHG_POL_QUAD_DIAGONAL) return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    if (shape[0] < 1 || shape[1] < 1) return chg_fail(NDNLM_EINVAL, "shape out of range");
    if (shape[2] < 1 || shape[2] > 0x7fffffffLL) return chg_fail(NDNLM_EINVAL, "the ENL needs at least 1 time step");
    if (window < 3 || window % 2 == 0) return chg_fail(NDNLM_EINVAL, "the window must be odd and >= 3, got %u", window);
    if (window > shape[0] || window > shape[1])
        return chg_fail(NDNLM_EINVAL, "the window (%u) must not exceed the image (%lld x %lld)", window, (long long)shape[0],
                        (long long)shape[1]);
    ChgDeviceGuard guard(enl);
    if (!guard.ok) return chg_fail(NDNLM_EINVAL, "enl is not a CUDA device pointer");
    return dtype == NDCHG_F64 ? launch_enl<double>(pol, values, shape, strides, window, enl, stream)
                              : launch_enl<float>(pol, values, shape, strides, window, enl, stream);
}

template <typename T, int POL>
static int launch_refined_lee(const void* values, const int64_t* shape, const int64_t* strides, uint32_t window,
                              double looks, void* out, void* stream) {
    const dim3 grid(unsigned(shape[2]), unsigned((shape[1] + ndchg::LEE_T - 1) / ndchg::LEE_T),
                    unsigned((shape[0] + ndchg::LEE_T - 1) / ndchg::LEE_T));
    if (grid.y > 65535 || grid.z > 65535)
        return chg_fail(NDNLM_EINVAL, "image of %lld x %lld pixels is too large for ndchg_refined_lee", (long long)shape[0],
                        (long long)shape[1]);
    const size_t smem = ndchg::lee_smem(ndchg::pol_bands(POL), int(window));
    cudaError_t e = cudaFuncSetAttribute(ndchg::refined_lee_kernel<T, POL>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "shared memory of %zu bytes: %s", smem, cudaGetErrorString(e));
    ndchg::refined_lee_kernel<T, POL><<<grid, ndchg::LEE_THREADS, smem, (cudaStream_t)stream>>>(
        (const T*)values, shape[0], shape[1], int(shape[2]), strides[0], strides[1], strides[2], strides[3], int(window),
        looks, (T*)out);
    e = cudaGetLastError();
    if (e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "launch failed: %s", cudaGetErrorString(e));
    return NDNLM_OK;
}

template <typename T>
static int launch_refined_lee(int pol, const void* values, const int64_t* shape, const int64_t* strides, uint32_t window,
                              double looks, void* out, void* stream) {
    switch (pol) {
        case NDCHG_POL_DUAL: return launch_refined_lee<T, NDCHG_POL_DUAL>(values, shape, strides, window, looks, out, stream);
        case NDCHG_POL_SINGLE: return launch_refined_lee<T, NDCHG_POL_SINGLE>(values, shape, strides, window, looks, out, stream);
        case NDCHG_POL_QUAD: return launch_refined_lee<T, NDCHG_POL_QUAD>(values, shape, strides, window, looks, out, stream);
        case NDCHG_POL_DUAL_DIAGONAL:
            return launch_refined_lee<T, NDCHG_POL_DUAL_DIAGONAL>(values, shape, strides, window, looks, out, stream);
        case NDCHG_POL_QUAD_DIAGONAL:
            return launch_refined_lee<T, NDCHG_POL_QUAD_DIAGONAL>(values, shape, strides, window, looks, out, stream);
        default: return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    }
}

// true if the bytes `values` spans (any strides, including negative ones) meet the C-contiguous output of `outs`
// values of `oelem` bytes per sample
static bool lee_overlap(const void* values, const int64_t* shape, const int64_t* strides, int bands, size_t elem, const void* out,
                        int outs, size_t oelem) {
    const int64_t n[4] = {shape[0], shape[1], shape[2], bands};
    const char* lo = (const char*)values;
    const char* hi = lo + elem;
    for (int d = 0; d < 4; ++d) {
        const int64_t ext = (n[d] - 1) * strides[d] * int64_t(elem);
        if (ext < 0) lo += ext;
        else hi += ext;
    }
    const char* olo = (const char*)out;
    const char* ohi = olo + shape[0] * shape[1] * shape[2] * outs * int64_t(oelem);
    return lo < ohi && olo < hi;
}

extern "C" int ndchg_refined_lee(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol,
                                 uint32_t window, double looks, void* out, void* stream) {
    if (!values || !shape || !strides || !out) return chg_fail(NDNLM_EINVAL, "null argument");
    if (pol < NDCHG_POL_DUAL || pol > NDCHG_POL_QUAD_DIAGONAL) return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    if (window != 7 && window != 11 && window != 15)
        return chg_fail(NDNLM_EINVAL, "the window must be 7, 11 or 15 (4 m + 3), got %u", window);
    if (shape[0] < 1 || shape[1] < 1) return chg_fail(NDNLM_EINVAL, "shape out of range");
    if (window > shape[0] || window > shape[1])
        return chg_fail(NDNLM_EINVAL, "the window (%u) must not exceed the image (%lld x %lld)", window, (long long)shape[0],
                        (long long)shape[1]);
    if (shape[2] < 1 || shape[2] > 0x7fffffffLL) return chg_fail(NDNLM_EINVAL, "the refined Lee filter needs at least 1 time step");
    if (!(looks > 0.0) || !std::isfinite(looks))
        return chg_fail(NDNLM_EINVAL, "the number of looks must be finite and > 0, got %g", looks);
    if (dtype != NDCHG_F32 && dtype != NDCHG_F64) return chg_fail(NDNLM_EDTYPE, "No matching signature found (only float32 / float64 data is supported)");
    if (lee_overlap(values, shape, strides, ndchg::pol_bands(pol), dtype == NDCHG_F64 ? 8 : 4, out, ndchg::pol_bands(pol),
                    dtype == NDCHG_F64 ? 8 : 4))
        return chg_fail(NDNLM_EINVAL, "out must not overlap values");
    ChgDeviceGuard guard(out);
    if (!guard.ok) return chg_fail(NDNLM_EINVAL, "out is not a CUDA device pointer");
    return dtype == NDCHG_F64 ? launch_refined_lee<double>(pol, values, shape, strides, window, looks, out, stream)
                              : launch_refined_lee<float>(pol, values, shape, strides, window, looks, out, stream);
}

template <typename T, int POL>
static int launch_h_a_alpha(const void* values, const int64_t* shape, const int64_t* strides, void* out, void* stream) {
    const long long samples = shape[0] * shape[1] * shape[2];
    const long long blocks = (samples + ndchg::HAA_THREADS - 1) / ndchg::HAA_THREADS;
    if (blocks > 0x7fffffffLL) return chg_fail(NDNLM_EINVAL, "%lld samples are too many for ndchg_h_a_alpha", samples);
    ndchg::h_a_alpha_kernel<T, POL><<<unsigned(blocks), ndchg::HAA_THREADS, 0, (cudaStream_t)stream>>>(
        (const T*)values, shape[1], shape[2], samples, strides[0], strides[1], strides[2], strides[3], (T*)out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "launch failed: %s", cudaGetErrorString(e));
    return NDNLM_OK;
}

template <typename T>
static int launch_h_a_alpha(int pol, const void* values, const int64_t* shape, const int64_t* strides, void* out, void* stream) {
    switch (pol) {
        case NDCHG_POL_DUAL: return launch_h_a_alpha<T, NDCHG_POL_DUAL>(values, shape, strides, out, stream);
        case NDCHG_POL_QUAD: return launch_h_a_alpha<T, NDCHG_POL_QUAD>(values, shape, strides, out, stream);
        case NDCHG_POL_DUAL_DIAGONAL: return launch_h_a_alpha<T, NDCHG_POL_DUAL_DIAGONAL>(values, shape, strides, out, stream);
        case NDCHG_POL_QUAD_DIAGONAL: return launch_h_a_alpha<T, NDCHG_POL_QUAD_DIAGONAL>(values, shape, strides, out, stream);
        default: return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    }
}

extern "C" int ndchg_h_a_alpha(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol,
                               void* out, void* stream) {
    if (!values || !shape || !strides || !out) return chg_fail(NDNLM_EINVAL, "null argument");
    if (pol < NDCHG_POL_DUAL || pol > NDCHG_POL_QUAD_DIAGONAL) return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    if (pol == NDCHG_POL_SINGLE)
        return chg_fail(NDNLM_EINVAL, "single-pol data have no H / A / alpha decomposition (a 1 x 1 matrix has no eigenvectors)");
    // every extent below 2^40: the element count (x 9 bands) stays far inside int64
    if (shape[0] < 1 || shape[1] < 1 || shape[0] >= (1LL << 40) || shape[1] >= (1LL << 40) ||
        double(shape[0]) * double(shape[1]) >= double(1LL << 40))
        return chg_fail(NDNLM_EINVAL, "shape out of range");
    if (shape[2] < 1 || double(shape[0]) * double(shape[1]) * double(shape[2]) >= double(1LL << 56))
        return chg_fail(NDNLM_EINVAL, "the H / A / alpha decomposition needs at least 1 time step (and fewer than 2^56 samples)");
    if (dtype != NDCHG_F32 && dtype != NDCHG_F64) return chg_fail(NDNLM_EDTYPE, "No matching signature found (only float32 / float64 data is supported)");
    if (lee_overlap(values, shape, strides, ndchg::pol_bands(pol), dtype == NDCHG_F64 ? 8 : 4, out, ndchg::haa_outputs(pol),
                    dtype == NDCHG_F64 ? 8 : 4))
        return chg_fail(NDNLM_EINVAL, "out must not overlap values");
    ChgDeviceGuard guard(out);
    if (!guard.ok) return chg_fail(NDNLM_EINVAL, "out is not a CUDA device pointer");
    return dtype == NDCHG_F64 ? launch_h_a_alpha<double>(pol, values, shape, strides, out, stream)
                              : launch_h_a_alpha<float>(pol, values, shape, strides, out, stream);
}

// the checks ndchg_h_alpha_zones and ndchg_wishart_classify share with ndchg_h_a_alpha, in its order: pol, single-pol,
// (the caller's own checks), shape and k, dtype
static int check_decomposable(int pol) {
    if (pol < NDCHG_POL_DUAL || pol > NDCHG_POL_QUAD_DIAGONAL) return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    if (pol == NDCHG_POL_SINGLE)
        return chg_fail(NDNLM_EINVAL, "single-pol data have no H / A / alpha decomposition (a 1 x 1 matrix has no eigenvectors)");
    return NDNLM_OK;
}

static int check_samples(const int64_t* shape, int dtype) {
    if (shape[0] < 1 || shape[1] < 1 || shape[0] >= (1LL << 40) || shape[1] >= (1LL << 40) ||
        double(shape[0]) * double(shape[1]) >= double(1LL << 40))
        return chg_fail(NDNLM_EINVAL, "shape out of range");
    if (shape[2] < 1 || double(shape[0]) * double(shape[1]) * double(shape[2]) >= double(1LL << 42))
        return chg_fail(NDNLM_EINVAL, "needs at least 1 time step (and fewer than 2^42 samples)");
    if (dtype != NDCHG_F32 && dtype != NDCHG_F64) return chg_fail(NDNLM_EDTYPE, "No matching signature found (only float32 / float64 data is supported)");
    return NDNLM_OK;
}

template <typename T, int POL>
static int run_zones(const void* values, const int64_t* shape, const int64_t* strides, int anisotropy, uint8_t* zones,
                     cudaStream_t st) {
    const long long rows = shape[0], cols = shape[1], k = shape[2], CH = ndchg::ZONE_CHUNK;
    const long long samples = rows * cols * k;
    T* scratch = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&scratch, sizeof(T) * size_t(samples < CH ? samples : CH) * ndchg::haa_outputs(POL), st);
    if (e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "scratch allocation failed: %s", cudaGetErrorString(e));
    // one box of samples whose outputs are contiguous: rows r0.., or columns j0.. of row i, or steps t0.. of (i, j)
    auto box = [&](long long i, long long j, long long t, long long nr, long long nc, long long nk) -> int {
        const int64_t sub[3] = {nr, nc, nk};
        const T* src = (const T*)values + i * strides[0] + j * strides[1] + t * strides[2];
        int rc = launch_h_a_alpha<T, POL>(src, sub, strides, scratch, st);
        if (rc) return rc;
        const long long n = nr * nc * nk;
        ndchg::h_alpha_zone_kernel<T, POL><<<unsigned((n + ndchg::HAA_THREADS - 1) / ndchg::HAA_THREADS), ndchg::HAA_THREADS, 0, st>>>(
            scratch, n, anisotropy, zones + (i * cols + j) * k + t);
        return NDNLM_OK;
    };
    int rc = NDNLM_OK;
    if (cols * k <= CH) {
        const long long rr = CH / (cols * k);
        for (long long i = 0; i < rows && !rc; i += rr) rc = box(i, 0, 0, rows - i < rr ? rows - i : rr, cols, k);
    } else if (k <= CH) {
        const long long cc = CH / k;
        for (long long i = 0; i < rows && !rc; ++i)
            for (long long j = 0; j < cols && !rc; j += cc) rc = box(i, j, 0, 1, cols - j < cc ? cols - j : cc, k);
    } else {
        for (long long i = 0; i < rows && !rc; ++i)
            for (long long j = 0; j < cols && !rc; ++j)
                for (long long t = 0; t < k && !rc; t += CH) rc = box(i, j, t, 1, 1, k - t < CH ? k - t : CH);
    }
    cudaFreeAsync(scratch, st);
    e = cudaGetLastError();
    if (!rc && e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "launch failed: %s", cudaGetErrorString(e));
    return rc;
}

template <typename T>
static int run_zones(int pol, const void* values, const int64_t* shape, const int64_t* strides, int anisotropy, uint8_t* zones,
                     cudaStream_t st) {
    switch (pol) {
        case NDCHG_POL_DUAL: return run_zones<T, NDCHG_POL_DUAL>(values, shape, strides, anisotropy, zones, st);
        case NDCHG_POL_QUAD: return run_zones<T, NDCHG_POL_QUAD>(values, shape, strides, anisotropy, zones, st);
        case NDCHG_POL_DUAL_DIAGONAL: return run_zones<T, NDCHG_POL_DUAL_DIAGONAL>(values, shape, strides, anisotropy, zones, st);
        case NDCHG_POL_QUAD_DIAGONAL: return run_zones<T, NDCHG_POL_QUAD_DIAGONAL>(values, shape, strides, anisotropy, zones, st);
        default: return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    }
}

extern "C" int ndchg_h_alpha_zones(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol,
                                   int anisotropy, uint8_t* zones, void* stream) {
    if (!values || !shape || !strides || !zones) return chg_fail(NDNLM_EINVAL, "null argument");
    int rc = check_decomposable(pol);
    if (rc) return rc;
    if (anisotropy != 0 && anisotropy != 1) return chg_fail(NDNLM_EINVAL, "anisotropy must be 0 or 1, got %d", anisotropy);
    if (anisotropy && pol != NDCHG_POL_QUAD && pol != NDCHG_POL_QUAD_DIAGONAL)
        return chg_fail(NDNLM_EINVAL, "anisotropy needs a quad layout (the dual layouts have no A)");
    rc = check_samples(shape, dtype);
    if (rc) return rc;
    if (lee_overlap(values, shape, strides, ndchg::pol_bands(pol), dtype == NDCHG_F64 ? 8 : 4, zones, 1, 1))
        return chg_fail(NDNLM_EINVAL, "zones must not overlap values");
    ChgDeviceGuard guard(zones);
    if (!guard.ok) return chg_fail(NDNLM_EINVAL, "zones is not a CUDA device pointer");
    return dtype == NDCHG_F64 ? run_zones<double>(pol, values, shape, strides, anisotropy, zones, (cudaStream_t)stream)
                              : run_zones<float>(pol, values, shape, strides, anisotropy, zones, (cudaStream_t)stream);
}

static bool is_device(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeDevice;
}

template <typename T, int POL>
static int run_wishart(const void* values, const int64_t* shape, const int64_t* strides, uint8_t* labels, int K,
                       uint32_t max_iter, double tol, double* centres, int64_t* counts, uint32_t* iterations, cudaStream_t st) {
    using namespace ndchg;
    constexpr int B = pol_bands(POL), E = B + 1;
    const long long rows = shape[0], cols = shape[1], k = shape[2], samples = rows * cols * k;
    const long long nchunk = (samples + WIS_CHUNK - 1) / WIS_CHUNK;
    // (rows, cols, k) collapse into one axis of stride s2: sample g starts at element g * s2
    const long long s1 = cols == 1 ? k * strides[2] : strides[1];
    const bool flat = s1 == k * strides[2] && (rows == 1 || strides[0] == cols * s1);
    const size_t state = (sizeof(WisState) + 255) / 256 * 256;
    char* scratch = nullptr;
    cudaError_t e = cudaMallocAsync((void**)&scratch, state + sizeof(double) * size_t(K * E) * (1 + nchunk), st);
    if (e != cudaSuccess) return chg_fail(NDNLM_ECUDA, "scratch allocation of the Wishart sums failed: %s", cudaGetErrorString(e));
    WisState* ws = (WisState*)scratch;
    double* sums = (double*)(scratch + state);
    double* partials = sums + K * E;
    const size_t smem = wis_smem(POL, K);
    e = cudaMemsetAsync(ws, 0, sizeof(WisState), st);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(wishart_assign_kernel<T, POL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e == cudaSuccess) e = cudaFuncSetAttribute(wishart_assign_kernel<T, POL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) {
        cudaFreeAsync(scratch, st);
        return chg_fail(NDNLM_ECUDA, "Wishart set-up failed: %s", cudaGetErrorString(e));
    }
    const long long check_blocks = (samples + 255) / 256;
    wishart_check_kernel<<<unsigned(check_blocks < 4096 ? check_blocks : 4096), 256, 0, st>>>(labels, samples, K, ws);
    auto pass = [&](unsigned it) {
        if (it == 0)
            wishart_assign_kernel<T, POL, false><<<unsigned(nchunk), WIS_THREADS, smem, st>>>(
                (const T*)values, cols, k, samples, strides[0], strides[1], strides[2], strides[3], flat, labels, ws, K, partials, nchunk);
        else
            wishart_assign_kernel<T, POL, true><<<unsigned(nchunk), WIS_THREADS, smem, st>>>(
                (const T*)values, cols, k, samples, strides[0], strides[1], strides[2], strides[3], flat, labels, ws, K, partials, nchunk);
        wishart_reduce_kernel<<<unsigned(K * E), WIS_REDUCE_THREADS, 0, st>>>(partials, nchunk, sums, ws);
        wishart_centres_kernel<POL><<<1, 32, 0, st>>>(ws, sums, K, it, max_iter, tol, centres, (long long*)counts, iterations);
    };
    // iteration 0, then one wait: a label > K or no active class is reported before any iteration is enqueued
    pass(0);
    unsigned status[3] = {0, 0, 0};                                      // done, bad, active
    e = cudaMemcpyAsync(status, &ws->done, sizeof(status), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    int rc = NDNLM_OK;
    if (e != cudaSuccess) rc = chg_fail(NDNLM_ECUDA, "iteration 0 failed: %s", cudaGetErrorString(e));
    else if (status[1]) rc = chg_fail(NDNLM_EINVAL, "an initial label exceeds classes=%d", K);
    else if (status[2] == 0)
        rc = chg_fail(NDNLM_EINVAL, "no class is active after iteration 0 (every class is empty or its mean covariance is singular)");
    // the iterations, in batches of 32: after each batch the host looks at the done flag once
    for (uint32_t it = 1; !rc && !status[0] && it <= max_iter; ++it) {
        pass(it);
        if (it % 32 == 0 && it < max_iter) {
            e = cudaMemcpyAsync(status, &ws->done, sizeof(unsigned), cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) rc = chg_fail(NDNLM_ECUDA, "iteration %u failed: %s", it, cudaGetErrorString(e));
        }
    }
    cudaFreeAsync(scratch, st);
    e = cudaGetLastError();
    if (!rc && e != cudaSuccess) rc = chg_fail(NDNLM_ECUDA, "launch failed: %s", cudaGetErrorString(e));
    return rc;
}

template <typename T>
static int run_wishart(int pol, const void* values, const int64_t* shape, const int64_t* strides, uint8_t* labels, int K,
                       uint32_t max_iter, double tol, double* centres, int64_t* counts, uint32_t* iterations, cudaStream_t st) {
    switch (pol) {
        case NDCHG_POL_DUAL:
            return run_wishart<T, NDCHG_POL_DUAL>(values, shape, strides, labels, K, max_iter, tol, centres, counts, iterations, st);
        case NDCHG_POL_QUAD:
            return run_wishart<T, NDCHG_POL_QUAD>(values, shape, strides, labels, K, max_iter, tol, centres, counts, iterations, st);
        case NDCHG_POL_DUAL_DIAGONAL:
            return run_wishart<T, NDCHG_POL_DUAL_DIAGONAL>(values, shape, strides, labels, K, max_iter, tol, centres, counts, iterations, st);
        case NDCHG_POL_QUAD_DIAGONAL:
            return run_wishart<T, NDCHG_POL_QUAD_DIAGONAL>(values, shape, strides, labels, K, max_iter, tol, centres, counts, iterations, st);
        default: return chg_fail(NDNLM_EINVAL, "unknown covariance layout pol=%d", pol);
    }
}

extern "C" int ndchg_wishart_classify(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol,
                                      uint8_t* labels, uint32_t classes, uint32_t max_iter, double tol, double* centres,
                                      int64_t* counts, uint32_t* iterations, void* stream) {
    if (!values || !shape || !strides || !labels || !centres || !counts || !iterations) return chg_fail(NDNLM_EINVAL, "null argument");
    int rc = check_decomposable(pol);
    if (!rc) rc = check_samples(shape, dtype);
    if (rc) return rc;
    if (classes < 1 || classes > ndchg::WIS_MAX_CLASSES)
        return chg_fail(NDNLM_EINVAL, "classes must be in [1, %d], got %u", ndchg::WIS_MAX_CLASSES, classes);
    if (!(tol >= 0.0 && tol <= 1.0)) return chg_fail(NDNLM_EINVAL, "tol must be in [0, 1], got %g", tol);
    if (lee_overlap(values, shape, strides, ndchg::pol_bands(pol), dtype == NDCHG_F64 ? 8 : 4, labels, 1, 1))
        return chg_fail(NDNLM_EINVAL, "labels must not overlap values");
    ChgDeviceGuard guard(labels);
    if (!guard.ok) return chg_fail(NDNLM_EINVAL, "labels is not a CUDA device pointer");
    if (!is_device(centres) || !is_device(counts) || !is_device(iterations))
        return chg_fail(NDNLM_EINVAL, "centres, counts and iterations must be CUDA device pointers");
    return dtype == NDCHG_F64 ? run_wishart<double>(pol, values, shape, strides, labels, int(classes), max_iter, tol, centres,
                                                    counts, iterations, (cudaStream_t)stream)
                              : run_wishart<float>(pol, values, shape, strides, labels, int(classes), max_iter, tol, centres,
                                                   counts, iterations, (cudaStream_t)stream);
}

extern "C" const char* ndchg_last_error(void) { return g_chg_err; }
