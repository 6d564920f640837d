"""
TEST INFRASTRUCTURE ONLY.  NumPy float64 statement of the H / A / alpha decomposition of include/ndchg.h
(`ndchg_h_a_alpha`), vectorised over samples.

It shares no code with the kernel: the quad layouts form T = A C A^H as a matrix product (the kernel uses the
element formulas), the eigenpairs come from LAPACK through `np.linalg.eigh` (the kernel uses Jacobi rotations or the
2 x 2 closed form), and rules 1-6 of the header follow with the same tau.  The band order is read from
`nd_b200.change.POLS`.
"""
import numpy as np

from nd_b200.change import POLS

TAU = 1e-9
LAYOUTS = ('dual', 'quad', 'dual_diagonal', 'quad_diagonal')
# lexicographic C3 -> Pauli coherency: T = A C A^H
PAULI = np.array([[1, 0, 1], [1, 0, -1], [0, np.sqrt(2), 0]]) / np.sqrt(2)


def matrices(values, pol):
    """The Hermitian matrices (..., p, p) of the bands of `pol`: C2 for the dual layouts, C3 for the quad layouts."""
    x = np.asarray(values).astype(np.float64)
    names = POLS[pol]
    p = 3 if pol.startswith('quad') else 2
    c = np.zeros(x.shape[:-1] + (p, p), complex)
    for i in range(p):
        c[..., i, i] = x[..., names.index('C%d%d' % (i + 1, i + 1))]
        for j in range(i + 1, p):
            stem = 'C%d%d' % (i + 1, j + 1)
            if stem + '__re' in names:
                c[..., i, j] = x[..., names.index(stem + '__re')] + 1j * x[..., names.index(stem + '__im')]
                c[..., j, i] = np.conj(c[..., i, j])
    return c


def components(values, pol):
    """Per sample: the clamped eigenvalues `lam` (..., p), descending, and c (..., p), |e_i[0]|^2 after the tie
    rule (rule 6), both float64; and `finite`, False where a band is not finite."""
    if pol not in LAYOUTS:
        raise ValueError('pol=%r' % (pol,))
    x = np.asarray(values).astype(np.float64)
    finite = np.isfinite(x).all(-1)
    m = matrices(np.where(finite[..., None], x, 0.0), pol)
    if pol.startswith('quad'):
        m = PAULI @ m @ PAULI.T
    w, v = np.linalg.eigh(m)
    lam = np.maximum(w[..., ::-1], 0.0)
    c = np.abs(v[..., 0, ::-1]) ** 2
    s = lam.sum(-1)
    tie = lam[..., :-1] - lam[..., 1:] <= TAU * s[..., None]
    # clusters of consecutive tied eigenvalues: label each eigenvalue by the index of its cluster's first member
    label = np.zeros(lam.shape, np.int64)
    for i in range(1, lam.shape[-1]):
        label[..., i] = np.where(tie[..., i - 1], label[..., i - 1], i)
    shared = np.empty_like(c)
    for i in range(lam.shape[-1]):
        same = label == label[..., i:i + 1]
        shared[..., i] = (c * same).sum(-1) / same.sum(-1)
    return lam, shared, finite


def h_a_alpha(values, pol='dual'):
    """(..., n) in float64: [H, A, alpha, l1, l2, l3] (quad layouts) or [H, alpha, l1, l2] (dual layouts)."""
    lam, c, finite = components(values, pol)
    p = lam.shape[-1]
    s = lam.sum(-1)
    with np.errstate(invalid='ignore', divide='ignore'):
        pi = lam / s[..., None]
        H = -np.where(pi > 0, pi * np.log(np.where(pi > 0, pi, 1.0)), 0.0).sum(-1) / np.log(p)
        alpha = (pi * np.degrees(np.arccos(np.clip(np.sqrt(c), 0.0, 1.0)))).sum(-1)
        cols = [H, alpha]
        if p == 3:
            A = np.where(lam[..., 1] <= TAU * s, 0.0, (lam[..., 1] - lam[..., 2]) / (lam[..., 1] + lam[..., 2]))
            cols = [H, A, alpha]
    cols = [np.where(s > 0, q, np.nan) for q in cols]
    out = np.concatenate([np.stack(cols, -1), lam], -1)
    return np.where(finite[..., None], out, np.nan)
