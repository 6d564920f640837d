"""
TEST INFRASTRUCTURE ONLY.  NumPy float64 statement of the equivalent-number-of-looks estimator of include/ndchg.h
(`ndchg_enl`): for every pixel whose w x w window lies inside the image, delta = ln det M - mean(ln det X) over the
window (M the band-wise window mean), and the ENL is the root L of h(L) = G(L) - G(N L) = delta with N = w^2.

It shares no code with the kernel's special functions: psi is scipy's, the window sums come from
`sliding_window_view`, and the root is found by a vectorised bisection on ln(L - L_min).  Determinants are
`omnibus_pol_oracle.pol_det`.
"""
import numpy as np
from numpy.lib.stride_tricks import sliding_window_view
from scipy.special import digamma

from .omnibus_pol_oracle import POLS, pol_det


def lower(pol):
    """Lower end of the domain of L: d - 1 for the full layouts (d = p), 0 for the diagonal ones."""
    p, full = POLS[pol]
    return p - 1.0 if full else 0.0


def G(L, pol):
    """E[ln det X] = ln det Sigma - G(L) for an L-look sample: d ln L - sum_{i<d} psi(L - i) for the full layouts,
    p (ln L - psi(L)) for the diagonal ones (independent Gamma channels with a common L)."""
    p, full = POLS[pol]
    L = np.asarray(L, np.float64)
    if full:
        return p * np.log(L) - sum(digamma(L - i) for i in range(p))
    return p * (np.log(L) - digamma(L))


def h(L, N, pol):
    """E[delta] of a window of N independent L-look samples."""
    return G(L, pol) - G(N * np.asarray(L, np.float64), pol)


def solve(delta, N, pol, iterations=64):
    """The root L of h(L, N) = delta (delta > 0), by bisection on t = ln(L - L_min) in [-40, 60]."""
    delta = np.asarray(delta, np.float64)
    lo, hi = np.full(delta.shape, -40.0), np.full(delta.shape, 60.0)
    base = lower(pol)
    with np.errstate(all='ignore'):
        for _ in range(iterations):
            mid = 0.5 * (lo + hi)
            above = h(base + np.exp(mid), N, pol) > delta                  # h falls: the root is to the right
            lo, hi = np.where(above, mid, lo), np.where(above, hi, mid)
    return base + np.exp(0.5 * (lo + hi))


def delta_map(values, w, pol):
    """delta of every full window, (rows - w + 1, cols - w + 1, k), float64; NaN where a window holds a sample with a
    non-finite band or det <= 0, or where det M <= 0."""
    x = np.asarray(values).astype(np.float64)
    N = w * w
    with np.errstate(all='ignore'):
        det = pol_det(x, pol)
        ell = np.where(np.isfinite(x).all(-1) & (det > 0), np.log(det), np.nan)
        M = sliding_window_view(x, (w, w), axis=(0, 1)).sum(axis=(-2, -1)) / N
        mean_ell = sliding_window_view(ell, (w, w), axis=(0, 1)).sum(axis=(-2, -1)) / N
        det_m = pol_det(M, pol)
        delta = np.log(det_m) - mean_ell
    return np.where((det_m > 0) & np.isfinite(delta), delta, np.nan)


def enl(values, w, pol):
    """The ENL of every sample, (rows, cols, k) in the data type of `values`: NaN within w // 2 of the border and
    where delta is NaN, +inf where delta <= 0."""
    values = np.asarray(values)
    rows, cols, k = values.shape[:3]
    delta = delta_map(values, w, pol)
    inner = np.full(delta.shape, np.nan)
    inner[delta <= 0] = np.inf
    pos = delta > 0
    inner[pos] = solve(delta[pos], float(w * w), pol)
    out = np.full((rows, cols, k), np.nan)
    r = w // 2
    out[r:rows - r, r:cols - r] = inner
    return out.astype(values.dtype)
