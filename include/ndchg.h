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

/* Refined Lee speckle filter (Lee, Grunes & de Grandi, IEEE TGRS 37(5), 1999) of every time step on its own, over
 * an N x N window, N = `window` in {7, 11, 15} (N = 4m + 3; 7 is Lee et al.'s), N <= min(rows, cols); `looks` L
 * is finite and > 0.  `values` as above, in the band order of `pol`; `out` is a DEVICE array (rows, cols, k,
 * bands) of the data type, C-contiguous, written completely, not overlapping `values`.  Requires k >= 1.
 *
 * h = N / 2, subwindow side s = (N - 1) / 2 (odd), subwindow spacing c = (N - s) / 2 (N = 7: s = 3, c = 2).  Samples
 * outside the image are scipy's 'reflect' (half-sample symmetric) images of samples inside, one reflection deep.
 * For every output pixel p, over the offsets (dy, dx) in [-h, h]^2 of its window:
 *   1. span y = the diagonal bands added left to right, C11 + C22 (+ C33); single-pol: C11.
 *   2. m[u][v], u, v in {0, 1, 2}: the mean of y over the s x s subwindow centred at ((u - 1) c, (v - 1) c),
 *      summed row-major, divided by s^2.
 *   3. G0 = |(m02 + m12 + m22) - (m00 + m10 + m20)|,  G1 = |(m20 + m21 + m22) - (m00 + m01 + m02)|,
 *      G2 = |(m01 + m02 + m12) - (m10 + m20 + m21)|,  G3 = |(m00 + m01 + m10) - (m12 + m21 + m22)|  (each
 *      three-term sum added left to right); e = 0, then e = i for i = 1, 2, 3 if Gi > Ge (the first maximum
 *      wins; NaN never wins).
 *   4. (first, second) = (m10, m12), (m01, m21), (m02, m20), (m00, m22) for e = 0 .. 3, with the masks
 *      d <= 0 / d >= 0 of d = dx, dy, dy - dx, dy + dx; the second mask iff |second - m11| < |first - m11|.
 *      A mask holds n = N (N + 1) / 2 offsets.
 *   5. over the mask, row-major (dy outer, dx inner, both ascending): ybar = sum y / n,
 *      var_y = sum (y - ybar)(y - ybar) / n, sv2 = 1 / L, var_x = (var_y - (ybar ybar) sv2) / (1 + sv2),
 *      b = var_x > 0 ? var_x / var_y : 0.
 *   6. every band: M = (sum over the mask, row-major) / n, out = M + b (x_p - M).
 * Arithmetic: inputs are read in the data type; everything else is one correctly rounded double operation at a
 * time (no FMA contraction); every sum is a direct sum in the order given (acc = acc + term from acc = 0, never a
 * running add / subtract); the result is rounded once to the data type.  NaN follows the arithmetic.  Since
 * 0 <= b < 1, every output is a convex combination of the sample and a local mean: positive semidefinite samples
 * stay positive semidefinite. */
int ndchg_refined_lee(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol,
                      uint32_t window, double looks, void* out, void* stream);

/* H / A / alpha eigen-decomposition (Cloude & Pottier, IEEE TGRS 35(1), 1997; dual-pol: Cloude, IEEE GRSL 4(2),
 * 2007) of every sample (pixel, step) on its own.  `values` as above, in the band order of `pol`, which is
 * NDCHG_POL_DUAL, NDCHG_POL_QUAD or their diagonal layouts (off-diagonal bands zero); NDCHG_POL_SINGLE is rejected
 * (a 1 x 1 matrix has no decomposition).  `out` is a DEVICE array (rows, cols, k, n) of the data type, C-contiguous,
 * written completely, not overlapping `values`: per sample, quad layouts n = 6: [H, A, alpha, l1, l2, l3]; dual
 * layouts n = 4: [H, alpha, l1, l2].  Requires k >= 1.  Checks: pol, single-pol, shape and k, dtype, overlap, then
 * the device pointer.
 *
 * Matrix: quad layouts read the lexicographic C3 of k = [S_hh, sqrt2 S_hv, S_vv] and decompose the Pauli coherency
 * matrix T = A C A^H, A = [[1, 0, 1], [1, 0, -1], [0, sqrt2, 0]] / sqrt2:
 *     T11 = (C11 + 2 Re C13 + C33) / 2,  T22 = (C11 - 2 Re C13 + C33) / 2,  T33 = C22,
 *     T12 = (C11 - C33) / 2 - i Im C13,  T13 = (C12 + conj C23) / sqrt2,  T23 = (C12 - conj C23) / sqrt2.
 * Dual layouts decompose the 2 x 2 covariance C2 itself (the first component is the first channel).  With tau = 1e-9:
 *   1. l1 >= l2 (>= l3): the eigenvalues, each clamped to max(l, 0); s = sum of them.
 *   2. A sample with a non-finite band gives NaN everywhere.  s = 0 gives NaN H, A, alpha and the (zero) eigenvalues.
 *   3. H = -sum p_i log_b p_i, p_i = l_i / s, 0 log 0 = 0, b = 3 (quad) or 2 (dual): 0 <= H <= 1.
 *   4. A = (l2 - l3) / (l2 + l3), or 0 when l2 <= tau s (quad only).
 *   5. Consecutive eigenvalues with l_i - l_{i+1} <= tau s form one cluster (chained: all three can).
 *   6. c_i = |e_i[0]|^2 of the unit eigenvector, except that every member of a cluster of m gets the (0, 0) entry of
 *      the cluster's projector / m (so alpha does not depend on the basis of a repeated eigenvalue);
 *      alpha_i = arccos(sqrt c_i) in degrees (sqrt c_i clamped to [0, 1]), alpha = sum p_i alpha_i.
 * Arithmetic: inputs are read in the data type, everything else is double, each output is rounded once.  The bands
 * are scaled by a power of two first (exact; the eigenvalues are scaled back), so no scale overflows.  Quad: cyclic
 * complex Jacobi rotations until the off-diagonal Frobenius norm is <= 2^-52 ||T||_F (at most 16 sweeps).  Dual: the
 * closed form l1 = (C11 + C22) / 2 + r, r = hypot((C11 - C22) / 2, |C12|), l2 = det / l1, and |e_1[0]|^2 =
 * (l1 - C22) / (2 r), |e_2[0]|^2 = (l1 - C11) / (2 r), each formed without cancellation.  Not bit-identical to a
 * LAPACK restatement; eigenvalues agree to ~1e-12 s where every eigenvalue gap is <= tau s or >= 1e-4 s. */
int ndchg_h_a_alpha(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol, void* out,
                    void* stream);

/* Cloude-Pottier zone of every sample in the H / alpha plane (Lee, Grunes, Ainsworth, Du, Schuler & Cloude, IEEE
 * TGRS 37(5), 1999), the initial classes of ndchg_wishart_classify.  `values` and `pol` as for ndchg_h_a_alpha
 * (NDCHG_POL_SINGLE is rejected); `zones` is a DEVICE uint8 array (rows, cols, k), C-contiguous, written completely,
 * not overlapping `values`.  The zone is a pure function of the H, A and alpha that ndchg_h_a_alpha returns for the
 * sample in the data type, compared with the thresholds in double (Lee et al.'s numbering):
 *     H >= 0.9:        1: alpha >= 55          2: 40 <= alpha < 55     3: alpha < 40 (not feasible, normally empty)
 *     0.5 <= H < 0.9:  4: alpha >= 50          5: 40 <= alpha < 50     6: alpha < 40
 *     H < 0.5:         7: alpha >= 47.5        8: 42.5 <= alpha < 47.5 9: alpha < 42.5
 * A sample with NaN H or alpha gets zone 0.  `anisotropy` = 1 (quad layouts only; 0 or 1) adds 9 where A > 0.5:
 * labels 1..18, the 16 classes of the H / A / alpha Wishart initialisation plus the two normally empty zones.  Which
 * side of each boundary a value on it belongs to is this project's convention (no bit-parity with any other tool
 * is claimed).  The dual layouts use the same plane on Cloude's dual-pol H / alpha; that is a convention too, since
 * the feasible region of the dual-pol plane differs.  Checks: pol, single-pol, anisotropy, shape and k, dtype,
 * overlap, then the device pointer.  ndchg_h_a_alpha runs into device scratch of at most 2^24 samples at a time. */
int ndchg_h_alpha_zones(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol,
                        int anisotropy, uint8_t* zones, void* stream);

/* Unsupervised Wishart classification (Lee et al., IEEE TGRS 37(5), 1999): k-means with the complex Wishart distance
 * from the initial labels `labels`, one set of K = `classes` centres for every sample (pixel, step) of the series,
 * so a label means the same on every date.  `values` as for ndchg_h_a_alpha (dual, quad and the diagonal layouts;
 * NDCHG_POL_SINGLE is rejected); p = 2 (dual layouts) or 3 (quad layouts); B bands.  `labels` is a DEVICE uint8
 * array (rows, cols, k), C-contiguous, not overlapping `values`: read (0 = unlabelled, 1..K), then overwritten with
 * the result.  `centres` (K x B doubles, row-major), `counts` (K int64) and `iterations` (one uint32) are DEVICE
 * buffers; they describe the labels returned.  Limits: 1 <= classes <= 32, tol in [0, 1].
 *   Valid samples: every band finite and the trace (the diagonal bands added left to right) > 0.  Invalid samples
 *     always get label 0, and no sum counts them.
 *   Iteration 0: V_m = the band-wise mean of the valid samples labelled m (m = 1..K).  A label > K anywhere is
 *     NDNLM_EINVAL and nothing is written.
 *   Active class: count_m >= 1 and det V_m > 1e-12 (tr V_m / p)^p, with det the Hermitian determinant of
 *     ndchg_change_direction's m2 / m3 (the product of the diagonal for the diagonal layouts) and (tr / p)^p formed
 *     as q q (q) from q = tr / p.  No active class after iteration 0 is NDNLM_EINVAL.
 *   Distance (the covariance domain; it equals the distance on the Pauli T, since T = A C A^H with A unitary):
 *     d_m(C) = ln det V_m + tr(V_m^-1 C) = g_m + sum_b w_mb x_b, with g_m = ln det V_m, W = V_m^-1 = adj(V_m) / det
 *     V_m, and w_mb = W_ii for the band C_ii, 2 Re W_ij for Re C_ij and 2 Im W_ij for Im C_ij.  Evaluated as
 *     acc = g_m, then acc = acc + w_mb x_b in band order, each a separately rounded double operation (no FMA).
 *   Iterations 1..max_iter: every valid sample takes the argmin of d_m over the active classes (a tie goes to the
 *     lowest m); the samples whose label changed (0 -> m included) are counted; the centres are recomputed from the
 *     new labels.  The loop stops after iteration i when changed <= tol * (number of valid samples), or when no class
 *     is active any more; `iterations` = the last i run (0 when max_iter = 0).
 *   Centres: K x B means in double, NaN for inactive classes; counts: the valid samples of each label.
 * Rounding: inputs are read in the data type, everything else is double; the sums of every pass are formed in a fixed
 * order (fixed chunks of samples, a fixed order inside a chunk, a fixed tree over the chunks), so a call is bit-identical
 * from run to run and for any strides of the same data.  ln is CUDA's `log`, which is not correctly rounded.
 * Checks: pol, single-pol, shape and k, dtype, classes, tol, overlap, then the device pointers.  The call waits for
 * iteration 0 on `stream` (to report a label > K or no active class) and enqueues the iterations asynchronously: a
 * device flag, set when the loop stops, turns the later launches into early returns. */
int ndchg_wishart_classify(const void* values, const int64_t shape[3], const int64_t strides[4], int dtype, int pol,
                           uint8_t* labels, uint32_t classes, uint32_t max_iter, double tol, double* centres,
                           int64_t* counts, uint32_t* iterations, void* stream);

const char* ndchg_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* NDCHG_H */
