/*
 * ndchg.h -- C ABI of the omnibus change detection (SURVEY.md 8(f) row N4), part of libndnlm.so.
 *
 * Replaces the reference's Cython extension entry point
 *     nd/_change.pyx:266   cpdef BOOL[:, :, :] change_detection(floating[:, :, :, :] values, double alpha,
 *                                                                unsigned int n=1, unsigned int njobs=1)
 * called from `_omnibus_change_detection` (nd/change.py:67), i.e. per pixel `single_pixel_change_detection`
 * (:224-260) over `single_pixel_omnibus` (:139-160) and `_z` / `_rho` / `_omega2` / `_f` (:19-79): the
 * Conradsen et al. (2015) omnibus test on dual-pol covariance time series [C11, Re C12, Im C12, C22].
 * The reference parallelises over rows with OpenMP `prange` (:280); here one GPU thread owns one pixel.
 *
 * `values` is a DEVICE array (rows, cols, k, bands) of float32 or float64 with arbitrary element strides
 * (`strides[3]` is the band axis); `result` is a DEVICE uint8 array (rows, cols, k), C-contiguous, written
 * completely (0 / 1).  Asynchronous on `stream`; every entry returns 0 or a negative NDNLM_E* code (message:
 * ndchg_last_error()).  Argument checks come before the device-pointer check.
 *
 * Dual-pol (ndchg_change_detection, ndchg_omnibus_probability, and NDCHG_POL_DUAL of the _pol entries): bands
 * [C11, Re C12, Im C12, C22], the reference's arithmetic.  `floating` locals of the reference keep the data type
 * (float32 data -> float32 statistic), its doubles stay double.  The chi-square CDF (GSL's gsl_cdf_chisq_P in the
 * reference) is evaluated in double from the closed forms of the regularised incomplete gamma function for the
 * integer shape 2 (k - 1) the dual-pol test always has.
 *
 * Other layouts (the _pol entries), bands on the last axis in this order:
 *     NDCHG_POL_SINGLE         p = 1   [C11]
 *     NDCHG_POL_QUAD           p = 3   [C11, Re C12, Im C12, Re C13, Im C13, C22, Re C23, Im C23, C33]
 *     NDCHG_POL_DUAL_DIAGONAL  p = 2   [C11, C22]            (intensity only)
 *     NDCHG_POL_QUAD_DIAGONAL  p = 3   [C11, C22, C33]       (intensity only)
 * The same sequential procedure with lnQ = n (p k ln k + sum_i ln det X_i - k ln det sum_i X_i), z = -2 rho lnQ,
 * P = P1 + omega2 (P2 - P1), P1 = chi2cdf(z, f), P2 = chi2cdf(z, f + 4).  Full layouts: the reference's
 * f = (k-1) p^2, rho and omega2 at p.  Diagonal layouts: det = product of the diagonal, f = (k-1) p, rho at p = 1,
 * omega2 = -f/4 (1 - 1/rho)^2.  Inputs are read in the data type; sums, determinants, logs, rho, omega2, z and the
 * CDF (regularised incomplete gamma for real shape f/2: series / Legendre continued fraction) are double; only the
 * returned probability is rounded to the data type.  IEEE rules for degenerate pixels: NaN or all-zero input
 * gives a NaN statistic, i.e. no change.
 * Requirements: k >= 2, n >= 1 looks, and n >= 3 for quad-pol (the sample covariance of fewer looks is singular).
 *
 * Direction of each change (ndchg_change_direction): the walk of the layout runs unchanged (NDCHG_POL_DUAL: the
 * reference's dual-pol walk), then every change is classified by the Loewner order of the covariance after it
 * against the mean of the segment before it.  With t_1 < t_2 < ... the changes of a pixel and t_0 = 0 (the walk
 * restarts at each change), for change i: m = t_i - t_{i-1}, S = sum of double(X_s) for s = t_{i-1} .. t_i - 1 per
 * band, added left to right, M = S / m, D = double(X_t_i) - M, all in double with separate correctly rounded
 * operations (no FMA).  D is Hermitian, in the band order of the layout:
 *     single, dual / quad diagonal  increase: every diagonal entry > 0      decrease: every diagonal entry < 0
 *     dual                          increase: m1 > 0, m2 > 0                decrease: m1 < 0, m2 > 0
 *     quad                          increase: m1 > 0, m2 > 0, m3 > 0        decrease: m1 < 0, m2 > 0, m3 < 0
 * with the leading principal minors (Sylvester's criterion) m1 = D11, m2 = D11 D22 - (ReD12 ReD12 + ImD12 ImD12),
 * m3 = ((a d) g + 2 Re(b e conj(c))) - a |e|^2 - d |c|^2 - g |b|^2 evaluated left to right (a, d, g the diagonal,
 * b = D12, c = D13, e = D23; Re(b e conj(c)) = (ReB ReE - ImB ImE) ReC + (ReB ImE + ImB ReE) ImC).  Increase means
 * D is positive definite, decrease negative definite; everything else -- semidefinite, zero, NaN -- is indefinite.
 * The result holds NDCHG_DIR_NONE where there is no change, so `result != 0` is the change map of
 * ndchg_change_detection_pol with the same arguments.
 */
#ifndef NDCHG_H
#define NDCHG_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NDCHG_F32 0
#define NDCHG_F64 1

#define NDCHG_POL_DUAL 0
#define NDCHG_POL_SINGLE 1
#define NDCHG_POL_QUAD 2
#define NDCHG_POL_DUAL_DIAGONAL 3
#define NDCHG_POL_QUAD_DIAGONAL 4

#define NDCHG_DIR_NONE 0
#define NDCHG_DIR_INCREASE 1
#define NDCHG_DIR_DECREASE 2
#define NDCHG_DIR_INDEFINITE 3

int ndchg_change_detection(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype,
                           uint8_t* result, double alpha, uint32_t n, void* stream);

/* The test statistic's probability for every pixel over the whole series (`single_pixel_omnibus`,
 * nd/_change.pyx:139-160): `prob` is a DEVICE array (rows, cols) of the data type, C-contiguous. */
int ndchg_omnibus_probability(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype,
                              void* prob, uint32_t n, void* stream);

/* The same for the covariance layout `pol` (NDCHG_POL_*); NDCHG_POL_DUAL calls the two entries above. */
int ndchg_change_detection_pol(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype,
                               int pol, uint8_t* result, double alpha, uint32_t n, void* stream);
int ndchg_omnibus_probability_pol(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype,
                                  int pol, void* prob, uint32_t n, void* stream);

/* ndchg_change_detection_pol followed by the direction of every change: `result` holds NDCHG_DIR_* codes
 * instead of 0 / 1. */
int ndchg_change_direction(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol,
                           uint8_t* result, double alpha, uint32_t n, void* stream);

/* Equivalent number of looks of every sample, estimated over a square window of odd side `window` (3 <= window <=
 * min(rows, cols)) in (rows, cols); each time step on its own.  `values` as above, in the band order of `pol`; `enl`
 * is a DEVICE array (rows, cols, k) of the data type, C-contiguous, written completely.  Requires k >= 1.
 *
 * With N = window^2 and l = ln det X of every sample (det of the layout: the 2 x 2 / 3 x 3 Hermitian determinant,
 * the product of the diagonal for the diagonal layouts), for a pixel whose window lies inside the image:
 *     M = the band-wise mean over the window,   delta = ln det M - (mean of l over the window),
 * and the ENL is the root L of h(L) = G(L) - G(N L) = delta, where
 *     full layouts (single, dual, quad; d = p):  G(L) = d ln L - sum_{i=0}^{d-1} psi(L - i)   on L > d - 1,
 *     diagonal layouts (independent Gamma channels with a common L):  G(L) = p (ln L - psi(L))   on L > 0.
 * For an L-look complex Wishart sample E[ln det X] = ln det Sigma + sum_i psi(L - i) - d ln L, and the window mean of
 * N independent samples has N L looks, so E[delta] = G(L) - G(N L) exactly (no small-window bias; N -> infinity is
 * the maximum-likelihood estimator of Anfinsen et al., IEEE TGRS 2009).  h falls strictly from +inf to 0, so the
 * root is unique.  Textured (non-homogeneous) windows bias L low; spatially correlated samples (box means, filtered
 * data) bias it high, since the estimator takes the N samples of a window as independent.
 * Edge rules: pixels within window / 2 of the image border are NaN; a window containing a sample with a non-finite
 * band or det <= 0 is NaN (as is a window whose mean has det <= 0); delta <= 0 (no speckle) gives +inf.
 * Arithmetic: inputs are read in the data type, everything else is double (psi and psi' by recurrence and the
 * asymptotic series); window sums are direct sums of window^2 terms; the root is found by Newton's method inside a
 * bracket to a relative 1e-13 and rounded once to the data type. */
int ndchg_enl(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol, uint32_t window,
              void* enl, void* stream);

const char* ndchg_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* NDCHG_H */
