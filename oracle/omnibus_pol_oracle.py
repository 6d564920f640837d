"""
TEST INFRASTRUCTURE ONLY.  NumPy float64 statement of the omnibus change detection for every covariance layout of
include/ndchg.h: dual-pol, single-pol, quad-pol and the intensity-only dual / quad diagonals.

No reference binary exists for the layouts beyond dual-pol, so this module is pinned by its own identities and by the
distribution of the probability under H0 (tests/test_change_pol.py).  The arithmetic is the one include/ndchg.h
specifies for them: inputs read in the data type, everything else in float64, the result rounded once to the data
type.  At pol='dual' it restates `omnibus_oracle.single_pixel_omnibus` (the pinned reference statistic) in float64,
vectorised over pixels.

`single_pixel_change_detection` / `change_detection` repeat the walk of `omnibus_oracle` (nd/_change.pyx:224-287)
with the probability function as an argument; with `omnibus_oracle.single_pixel_omnibus` they give the pinned
restatement's change maps (checked in tests/test_change_pol.py), so the control flow is the reference's.
"""
import numpy as np
from scipy.special import gammainc

from .omnibus_oracle import _f, _omega2, _rho, single_pixel_omnibus

# covariance layout -> (p, full covariance?); band order as in nd_b200.change.POLS
POLS = {'dual': (2, True), 'single': (1, True), 'quad': (3, True), 'dual_diagonal': (2, False), 'quad_diagonal': (3, False)}


def pol_det(x, pol):
    """Determinant of the covariance of every sample: x is (..., bands) float64 in the band order of `pol`."""
    if pol == 'dual':
        return x[..., 0] * x[..., 3] - (x[..., 1] ** 2 + x[..., 2] ** 2)
    if pol == 'quad':
        a, br, bi, cr, ci, d, er, ei, g = np.moveaxis(x, -1, 0)
        re_bec = (br * er - bi * ei) * cr + (br * ei + bi * er) * ci           # Re(b e conj(c))
        return a * d * g + 2 * re_bec - a * (er ** 2 + ei ** 2) - d * (cr ** 2 + ci ** 2) - g * (br ** 2 + bi ** 2)
    return np.prod(x, axis=-1)                                                     # single and the diagonals


def pol_lnQ(values, n, pol):
    """lnQ = n (p k ln k + sum_i ln det X_i - k ln det sum_i X_i) of every pixel; values is (..., k, bands)."""
    p = POLS[pol][0]
    x = np.asarray(values).astype(np.float64)
    k = x.shape[-2]
    with np.errstate(all='ignore'):
        return float(n) * (p * k * np.log(k) + np.log(pol_det(x, pol)).sum(-1) - k * np.log(pol_det(x.sum(-2), pol)))


def pol_constants(k, n, pol):
    """(f, rho, omega2): the reference's `_f` / `_rho` / `_omega2` at p for the full layouts; for the diagonal ones
    f = (k-1) p, rho at p = 1 and omega2 = -f/4 (1 - 1/rho)^2 (lnQ is a sum of p single-band lnQs)."""
    p, full = POLS[pol]
    k, n = float(k), float(n)
    if full:
        rho = _rho(p, k, n)
        return _f(p, k, n), rho, _omega2(p, k, n, rho)
    f, rho = (k - 1) * p, _rho(1, k, n)
    return f, rho, -f / 4 * (1 - 1 / rho) ** 2


def pol_z(values, n, pol):
    """z = -2 rho lnQ of every pixel, float64."""
    return -2 * pol_constants(np.shape(values)[-2], n, pol)[1] * pol_lnQ(values, n, pol)


def omnibus_probability_pol(values, n, pol):
    """P = P1 + omega2 (P2 - P1) of every pixel over its whole series; values is (..., k, bands) of float32 or
    float64, everything is float64 and the result is rounded once to the data type."""
    values = np.asarray(values)
    f, _, omega2 = pol_constants(values.shape[-2], n, pol)
    z = pol_z(values, n, pol)
    with np.errstate(all='ignore'):
        P1, P2 = [np.where(np.isnan(z), np.nan, np.where(z > 0, gammainc(nu / 2.0, z / 2.0), 0.0)) for nu in (f, f + 4)]
        return (P1 + omega2 * (P2 - P1)).astype(values.dtype)


def single_pixel_change_detection(ts, alpha, n, prob=single_pixel_omnibus):
    """nd/_change.pyx:224-260 with `prob(ts, n)`, the probability of the test over the series `ts`; returns the
    uint8 change vector of one pixel."""
    k = ts.shape[0]
    result = np.zeros(k, np.uint8)
    l = 0
    r = 0
    while True:
        if not (prob(ts[l:], n) > alpha):                                          # global hypothesis H0_l
            break
        for j in range(2, k - l + 1):                                              # marginal hypotheses
            r = j - 1
            if prob(ts[l:l + j], n) > alpha:
                result[l + r] = 1
                break
        l = l + r
        if l >= k - 1:
            break
    return result


def change_detection(values, alpha, n=1, prob=single_pixel_omnibus):
    """nd/_change.pyx:263-287 with the probability function `prob`; values is (rows, cols, k, bands)."""
    rows, cols, k = values.shape[:3]
    out = np.zeros((rows, cols, k), np.uint8)
    for i in range(rows):
        for j in range(cols):
            out[i, j] = single_pixel_change_detection(values[i, j], alpha, n, prob)
    return out


def change_detection_pol(values, alpha, n, pol):
    """`change_detection` with the statistic of layout `pol`."""
    # the probability is rounded to the data type, then compared with alpha in double, as the kernel does
    return change_detection(values, alpha, n, prob=lambda ts, n: np.float64(omnibus_probability_pol(ts, n, pol)))
