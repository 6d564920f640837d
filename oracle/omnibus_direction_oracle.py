"""
TEST INFRASTRUCTURE ONLY.  NumPy float64 statement of the direction of each detected change (include/ndchg.h,
`ndchg_change_direction`): the Loewner order of the covariance after the change against the mean of the segment
before it -- 1 increase (positive definite), 2 decrease (negative definite), 3 indefinite, 0 no change.

Direction depends only on the data and the change map, so `change_direction` applies to the pinned dual-pol maps
(`omnibus_oracle`) as well as to the layout oracle's (`omnibus_pol_oracle`).  Every operation is a single correctly
rounded float64 operation in a fixed order (explicit loops, no `np.sum`; the quad determinant is
`omnibus_pol_oracle.pol_det`), which the kernel repeats one for one, so the codes must match exactly.  Pinned in
tests/test_change_direction.py against eigenvalues, a hand-worked series and simulated series of known direction.
"""
import numpy as np

from .omnibus_pol_oracle import pol_det

DIR_NONE, DIR_INCREASE, DIR_DECREASE, DIR_INDEFINITE = 0, 1, 2, 3


def classify(D, pol):
    """Direction code of every Hermitian difference D (..., bands) float64 in the band order of `pol`: 1 positive
    definite, 2 negative definite, 3 otherwise (semidefinite, zero, NaN).  Full 2 x 2 / 3 x 3 layouts: Sylvester's
    criterion on the leading principal minors; single and the diagonals: the signs of the diagonal."""
    D = np.asarray(D, np.float64)
    if pol in ('dual', 'quad'):
        m1 = D[..., 0]
        m2 = pol_det(D[..., [0, 1, 2, 3 if pol == 'dual' else 5]], 'dual')
        if pol == 'dual':
            up, down = (m1 > 0) & (m2 > 0), (m1 < 0) & (m2 > 0)
        else:
            m3 = pol_det(D, 'quad')
            up, down = (m1 > 0) & (m2 > 0) & (m3 > 0), (m1 < 0) & (m2 > 0) & (m3 < 0)
    else:
        up, down = (D > 0).all(-1), (D < 0).all(-1)
    return np.where(up, DIR_INCREASE, np.where(down, DIR_DECREASE, DIR_INDEFINITE)).astype(np.uint8)


def change_direction(values, change, pol):
    """Direction codes (rows, cols, k) of the change map `change` (rows, cols, k) of `values` (rows, cols, k, bands):
    at each change t_i, D = X_{t_i} - S / m with S the left-to-right float64 sum of X over the segment since the
    previous change t_{i-1} (t_0 = 0) and m its length; 0 where there is no change."""
    x = np.asarray(values)
    change = np.asarray(change) != 0
    out = np.zeros(change.shape, np.uint8)
    S = np.zeros(x.shape[:2] + x.shape[3:], np.float64)
    m = np.zeros(x.shape[:2], np.int64)
    for t in range(x.shape[2]):
        xt = x[:, :, t].astype(np.float64)
        c = change[:, :, t]
        if c.any():                                  # the walk never marks t = 0, so m >= 1 here
            D = xt[c] - S[c] / m[c][:, None].astype(np.float64)
            out[:, :, t][c] = classify(D, pol)
            S[c] = 0.0
            m[c] = 0
        S += xt
        m += 1
    return out
