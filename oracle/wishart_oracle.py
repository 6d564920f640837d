"""
TEST INFRASTRUCTURE ONLY.  NumPy float64 statement of the H / alpha zones and of the unsupervised Wishart
classification of include/ndchg.h (`ndchg_h_alpha_zones`, `ndchg_wishart_classify`), vectorised over samples.

The zone table and the loop follow the header rule by rule: valid samples, iteration 0, the active classes, the
distance as acc = g_m, then acc = acc + w_mb x_b in band order (NumPy rounds every operation separately, as the kernel
does), the argmin with ties to the lowest class, and the stopping rule.  The class sums are NumPy sums, not the
kernel's fixed chunk order, so centres agree to rounding, not bit for bit.  Every pass also reports, per sample,
the margin between the best and the second-best distance, so tests can tell which labels rounding cannot move.
The band order is read from `nd_b200.change.POLS`.
"""
import numpy as np

from nd_b200.change import POLS

LAYOUTS = ('dual', 'quad', 'dual_diagonal', 'quad_diagonal')
# (H lower bound, [(alpha lower bound, zone), ...]) from the top of the plane down; the last alpha bound is -inf
ZONES = [(0.9, [(55.0, 1), (40.0, 2), (-np.inf, 3)]),
         (0.5, [(50.0, 4), (40.0, 5), (-np.inf, 6)]),
         (-np.inf, [(47.5, 7), (42.5, 8), (-np.inf, 9)])]


def zones(H, alpha, A=None):
    """The zone (uint8) of each (H, alpha) in the data type, compared in float64; A > 0.5 adds 9 when A is given;
    NaN H or alpha gives 0."""
    H, alpha = np.asarray(H, np.float64), np.asarray(alpha, np.float64)
    z = np.zeros(np.broadcast(H, alpha).shape, np.int64)
    done = np.isnan(H) | np.isnan(alpha)
    for h_lo, rows in ZONES:
        for a_lo, zone in rows:
            hit = ~done & (H >= h_lo) & (alpha >= a_lo)
            z[hit] = zone
            done |= hit
    if A is not None:
        z = np.where((z > 0) & (np.asarray(A, np.float64) > 0.5), z + 9, z)
    return z.astype(np.uint8)


def zones_of(haa, pol, anisotropy=False):
    """Zones from the (..., n) output of `h_a_alpha` for the layout `pol`."""
    quad = pol.startswith('quad')
    return zones(haa[..., 0], haa[..., 2 if quad else 1], haa[..., 1] if quad and anisotropy else None)


def diagonal(pol):
    """The band indices of the diagonal C11, C22 (, C33) of `pol`."""
    return [POLS[pol].index(b) for b in ('C11', 'C22', 'C33') if b in POLS[pol]]


def valid(x, pol):
    """Every band finite and the trace, added left to right, > 0."""
    x = np.asarray(x, np.float64)
    d = diagonal(pol)
    with np.errstate(invalid='ignore'):
        tr = x[..., d[0]]
        for i in d[1:]:
            tr = tr + x[..., i]
        return np.isfinite(x).all(-1) & (tr > 0)


def table(V, n, pol):
    """The pinned (g, w, det, active) of centres V (K, B) with counts n (K,): g = ln det V (0 where inactive), w the
    distance weights (K, B) from adj(V) / det V (0 where inactive)."""
    V = np.asarray(V, np.float64)
    d = diagonal(pol)
    p = len(d)
    with np.errstate(invalid='ignore', divide='ignore', over='ignore'):
        tr = V[:, d[0]]
        for i in d[1:]:
            tr = tr + V[:, i]
        q = tr / p
        qp = q * q if p == 2 else (q * q) * q
        w = np.empty_like(V)
        if pol == 'dual':
            a, br, bi, dd = V.T
            det = a * dd - (br * br + bi * bi)
            w[:, 0], w[:, 1], w[:, 2], w[:, 3] = dd / det, -2.0 * (br / det), -2.0 * (bi / det), a / det
        elif pol == 'quad':
            a, br, bi, cr, ci, dd, er, ei, g = V.T
            re_bec = (br * er - bi * ei) * cr + (br * ei + bi * er) * ci
            e2, c2, b2 = er * er + ei * ei, cr * cr + ci * ci, br * br + bi * bi
            det = (a * dd) * g + 2.0 * re_bec
            det = det - a * e2
            det = det - dd * c2
            det = det - g * b2
            w[:, 0] = (dd * g - e2) / det
            w[:, 5] = (a * g - c2) / det
            w[:, 8] = (a * dd - b2) / det
            w[:, 1] = 2.0 * (((cr * er + ci * ei) - br * g) / det)          # W12 = (c conj(e) - b g) / det
            w[:, 2] = 2.0 * (((ci * er - cr * ei) - bi * g) / det)
            w[:, 3] = 2.0 * (((br * er - bi * ei) - cr * dd) / det)         # W13 = (b e - c d) / det
            w[:, 4] = 2.0 * (((br * ei + bi * er) - ci * dd) / det)
            w[:, 6] = 2.0 * (((cr * br + ci * bi) - a * er) / det)          # W23 = (c conj(b) - a e) / det
            w[:, 7] = 2.0 * (((ci * br - cr * bi) - a * ei) / det)
        else:
            det = V[:, 0]
            for b in range(1, V.shape[1]):
                det = det * V[:, b]
            w = 1.0 / V
        active = (np.asarray(n) >= 1) & (det > 1e-12 * qp)
        g = np.where(active, np.log(np.where(active, det, 1.0)), 0.0)
    return g, np.where(active[:, None], w, 0.0), det, active


def distances(x, g, w):
    """d (n, K) in the pinned order: acc = g_m, then acc = acc + w_mb x_b for b = 0, 1, ..."""
    x = np.asarray(x, np.float64)
    acc = np.broadcast_to(g[None, :], (len(x), len(g))).copy()
    for b in range(x.shape[1]):
        acc = acc + w[None, :, b] * x[:, b, None]
    return acc


def scale(x, g, w):
    """(n, K): |g_m| + sum_b |w_mb x_b|, the magnitude the rounding errors of d_m are relative to."""
    return np.abs(g)[None, :] + np.abs(w[None, :, :] * np.asarray(x, np.float64)[:, None, :]).sum(-1)


def centres(x, labels, K):
    """Band-wise means (K, B) of the samples labelled 1..K and their counts (labels 0 are not counted)."""
    x = np.asarray(x, np.float64)
    V = np.full((K, x.shape[1]), np.nan)
    n = np.zeros(K, np.int64)
    for m in range(1, K + 1):
        sel = labels == m
        n[m - 1] = sel.sum()
        if n[m - 1]:
            V[m - 1] = x[sel].sum(0) / n[m - 1]
    return V, n


def classify(x, labels, K, pol, max_iter=10, tol=0.0):
    """The loop of `ndchg_wishart_classify` on samples x (n, B) (in the data type) from the initial labels (n,).
    Returns a dict: `labels` (uint8), `centres` (K, B; NaN where inactive), `counts`, `iterations`, `history` (the
    labels after iteration 0, 1, ...), `margin` (n,): the smallest relative margin (d2 - d1) / max_m scale_m of the
    sample over all passes (inf for invalid samples and with a single active class)."""
    x = np.asarray(x)
    labels = np.asarray(labels).astype(np.int64)
    if labels.max(initial=0) > K:
        raise ValueError('an initial label exceeds classes=%d' % K)
    ok = valid(x, pol)
    x = np.where(ok[:, None], np.asarray(x, np.float64), 0.0)
    lab = np.where(ok, labels, 0)
    history = [lab.copy()]
    V, n = centres(x, lab, K)
    g, w, _, act = table(V, n, pol)
    if not act.any():
        raise ValueError('no class is active after iteration 0')
    margin = np.full(len(x), np.inf)
    it = 0
    while it < max_iter:
        it += 1
        d = np.where(act[None, :], distances(x, g, w), np.inf)
        best = np.argmin(d, 1)
        if act.sum() > 1:
            two = np.sort(d, 1)[:, :2]
            s = np.where(act[None, :], scale(x, g, w), 0.0).max(1)
            with np.errstate(invalid='ignore'):
                margin = np.minimum(margin, np.where(ok, (two[:, 1] - two[:, 0]) / s, np.inf))
        new = np.where(ok, best + 1, 0)
        changed = int((new != lab).sum())
        lab = new
        history.append(lab.copy())
        V, n = centres(x, lab, K)
        g, w, _, act = table(V, n, pol)
        if changed <= tol * float(ok.sum()) or not act.any():
            break
    return dict(labels=lab.astype(np.uint8), centres=np.where(act[:, None], V, np.nan), counts=n, iterations=it,
                history=history, margin=margin)
