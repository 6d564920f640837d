"""
H / A / alpha decomposition (include/ndchg.h, `ndchg_h_a_alpha`; `polarimetry.h_a_alpha`, `HAAlphaDecomposition`).

The NumPy oracle (`oracle/h_a_alpha_oracle.py`, LAPACK eigenpairs) is tied to results it does not compute itself:
the canonical scattering targets, the closed forms of the dual diagonal and of rank-1 samples, the invariances of the
decomposition (roll rotation of T, scaling of C, trace), its bounds, and the adjugate formula of |e_i[0]|^2.  The CUDA
kernel (Jacobi rotations / the 2 x 2 closed form) is compared with the oracle to the tolerances of the definition:
float64 eigenvalues within 1e-12 s, H within 1e-10, alpha within 1e-8 degrees, A within 1e-10 + 1e-12 s / (l2 + l3),
wherever every eigenvalue gap is <= tau s or >= 1e-4 s; float32 within 1 ulp of the oracle rounded to float32 or
within those tolerances; NaN positions identical.
"""
import ctypes
import inspect

import numpy as np
import pytest

from nd_b200 import _lib, change, polarimetry
from nd_b200.dataset import Dataset, generate_test_dataset
from test_change_pol import P, bands, covariances
from test_refined_lee import _dataset

LAYOUTS = ['dual', 'quad', 'dual_diagonal', 'quad_diagonal']
LOOKS = [1, 2, 3, 4, 16, 50]
TAU = 1e-9
VP = ctypes.c_void_p
PAULI = np.array([[1, 0, 1], [1, 0, -1], [0, np.sqrt(2), 0]]) / np.sqrt(2)


def _oracle():
    from oracle import h_a_alpha_oracle as ho
    return ho


def _quad(C11=0.0, C12=0.0, C13=0.0, C22=0.0, C23=0.0, C33=0.0):
    return np.array([C11, np.real(C12), np.imag(C12), np.real(C13), np.imag(C13), C22, np.real(C23), np.imag(C23), C33])


def _to_bands(c, pol):
    """Bands of `pol` from Hermitian matrices (..., p, p) (the diagonal layouts keep the diagonal)."""
    return bands(c, 'quad' if pol == 'quad' else 'dual' if pol == 'dual' else pol)


def _wishart(n, looks, pol, rng):
    """n samples of `pol` at `looks` looks, each at a random power between 1e-3 and 1e3."""
    c = covariances((n,), looks, [1.0], P[pol], rng, diagonal=pol.endswith('diagonal'))[:, 0]
    return _to_bands(c, pol) * 10.0 ** rng.uniform(-3, 3, size=(n, 1))


def _unitary(p, rng):
    q, r = np.linalg.qr(rng.normal(size=(p, p)) + 1j * rng.normal(size=(p, p)))
    return q * (np.diag(r) / np.abs(np.diag(r)))


def _from_eigen(lam, pol, rng):
    """A sample of `pol` with the eigenvalues `lam` and random eigenvectors (diagonal layouts: a permuted
    diagonal); quad layouts place the eigenvalues on T, so C = A^H T A."""
    if pol.endswith('diagonal'):
        return np.asarray(lam, float)[rng.permutation(len(lam))]
    u = _unitary(len(lam), rng)
    m = u @ np.diag(lam) @ u.conj().T
    if pol == 'quad':
        m = PAULI.T @ m @ PAULI
    return _to_bands(m, pol)


def _targets(pol):
    """The canonical targets of each layout (quad: surface, dihedral, dipole, random volume, T = I)."""
    if pol == 'quad':
        return np.array([_quad(1, 0, 1, 0, 0, 1), _quad(1, 0, -1, 0, 0, 1), _quad(1), _quad(3 / 8, 0, 1 / 8, 2 / 8, 0, 3 / 8),
                         _quad(1, 0, 0, 1, 0, 1)])
    if pol == 'quad_diagonal':
        return np.array([[1.0, 0, 0], [0, 1.0, 0], [0, 0, 1.0], [1.0, 1, 1], [3, 2, 3]]) / 8
    if pol == 'dual':
        return np.array([[1.0, 0, 0, 0], [0, 0, 0, 1.0], [1, 1, 0, 1], [1, 0, 1, 1], [1, 0, 0, 1], [4, 0.5, -0.5, 1]])
    return np.array([[1.0, 0], [0, 1.0], [1, 1], [3, 1]])


def _exact_ties(pol):
    """Integer samples (exact in float32) with repeated eigenvalues: lambda2 = lambda3 > 0 and lambda1 = lambda2
    with non-trivial eigenspaces (C = l I +- k k^H), and C = c I."""
    out = []
    if pol == 'quad':
        for k in ([1, 2j, 2], [1 - 1j, 2, -1j], [3, 1 + 1j, -2j]):
            k = np.array(k)
            kk = np.outer(k, k.conj())
            n2 = int(round(np.vdot(k, k).real))
            out += [_to_bands(2 * np.eye(3) + kk, pol), _to_bands((n2 + 1) * np.eye(3) - kk, pol)]
    if pol == 'quad_diagonal':
        out += [[2.0, 2, 5], [5, 2, 2], [2, 5, 2], [7, 7, 1]]
    if pol == 'dual':
        out += [[3.0, 0, 0, 3]]
    if pol == 'dual_diagonal':
        out += [[3.0, 3], [0.5, 0.5]]
    p = P[pol]
    for c in (1.0, 0.25, 6.0):
        out.append(_to_bands(c * np.eye(p).astype(complex), pol))
    return np.array(out, float)


def _near_ties(pol, rng):
    p = P[pol]
    spectra = [[1.0003, 1.0], [1.0, 0.2]] if p == 2 else [[1.0, 0.5003, 0.5], [0.8003, 0.8, 0.3], [0.5006, 0.5003, 0.5]]
    return np.array([_from_eigen(lam, pol, rng) for lam in spectra for _ in range(4)])


def _special(pol):
    B = len(change.POLS[pol])
    v = np.ones((6, B))
    v[0, 0] = np.nan
    v[1, -1] = np.inf
    v[2, 0] = -np.inf
    v[3] = 0.0
    v[4, B // 2] = np.nan
    v[5] = -np.abs(v[5])                                  # negative diagonal: every eigenvalue clamps to 0
    if pol in ('dual', 'quad'):
        v[5, 1:B - 1] = 0.0
    return v


def _pool(pol, seed=0):
    rng = np.random.default_rng(seed)
    parts = [_wishart(120, looks, pol, rng) for looks in LOOKS]
    parts += [_targets(pol), _exact_ties(pol), _near_ties(pol, rng), _special(pol)]
    return np.concatenate(parts)


def _columns(pol):
    return polarimetry.OUTPUTS['quad' if pol.startswith('quad') else 'dual']


def _tolerance(want, pol):
    """float64 tolerance of each output (..., n) from the oracle's values."""
    cols = _columns(pol)
    lam = want[..., cols.index('lambda1'):]
    s = lam.sum(-1, keepdims=True)
    tol = np.empty_like(want)
    for q, name in enumerate(cols):
        tol[..., q] = {'entropy': 1e-10, 'alpha': 1e-8}.get(name, 0.0)
    tol[..., cols.index('lambda1'):] = 1e-12 * s
    if 'anisotropy' in cols:
        with np.errstate(invalid='ignore', divide='ignore'):
            tol[..., 1] = 1e-10 + 1e-12 * s[..., 0] / (lam[..., 1] + lam[..., 2])
    return tol


def _well_separated(want, pol):
    """Samples whose every eigenvalue gap is <= tau s or >= 1e-4 s (and whose outputs are finite)."""
    cols = _columns(pol)
    lam = want[..., cols.index('lambda1'):]
    s = lam.sum(-1, keepdims=True)
    gap = lam[..., :-1] - lam[..., 1:]
    with np.errstate(invalid='ignore'):
        return ((gap <= TAU * s) | (gap >= 1e-4 * s)).all(-1) & np.isfinite(want).all(-1)


def assert_matches_oracle(got, x, pol, min_checked=0.8):
    ho = _oracle()
    want = ho.h_a_alpha(x, pol)
    assert got.shape == want.shape and got.dtype == x.dtype
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = _well_separated(want, pol)
    assert ok.mean() >= min_checked, ok.mean()
    g, w = got[ok].astype(np.float64), want[ok]
    close = np.abs(g - w) <= _tolerance(w, pol)
    if x.dtype == np.float32:
        w32 = w.astype(np.float32)
        close |= np.abs(got[ok] - w32) <= np.spacing(np.abs(w32))
    bad = np.argwhere(~close)
    assert close.all(), [(tuple(i), g[tuple(i)], w[tuple(i)]) for i in bad[:5]]


# ---- CPU: C ABI and Python boundary --------------------------------------------------------------------
def test_c_abi_checks_arguments_before_the_device():
    L = _lib.lib()
    buf = np.zeros(8192, np.float64)
    out = np.zeros(8192, np.float64)
    def call(shape=(4, 5, 3), dtype=1, pol=0, src=None, dst=None):
        shape = list(shape)
        B = (4, 1, 9, 2, 3)[pol] if 0 <= pol <= 4 else 4
        strides = [shape[1] * shape[2] * B, shape[2] * B, B, 1]
        src = buf.ctypes.data if src is None else src
        dst = out.ctypes.data if dst is None else dst
        return L.ndchg_h_a_alpha(VP(src), _lib.i64(shape), _lib.i64(strides), dtype, pol, VP(dst), None)
    def err():
        return L.ndchg_last_error()
    for pol in (-1, 5, 99):
        assert call(pol=pol) == _lib.EINVAL and b"pol=%d" % pol in err()
    assert call(pol=1) == _lib.EINVAL and b"single-pol data have no H / A / alpha decomposition" in err()
    for shape in ((0, 5, 3), (4, 0, 3), (4, -1, 3)):
        assert call(shape=shape) == _lib.EINVAL and b"shape out of range" in err()
    for shape in ((4, 5, 0), (4, 5, -2)):
        assert call(shape=shape) == _lib.EINVAL and b"at least 1 time step" in err()
    assert call(dtype=2) == _lib.EDTYPE and b"No matching signature" in err()
    assert call(dst=buf.ctypes.data) == _lib.EINVAL and b"must not overlap" in err()
    # dual_diagonal writes 4 values per sample from 2 bands: an output ending inside the input overlaps it
    n = 4 * 5 * 3
    assert call(pol=3, src=buf.ctypes.data + 8 * 4 * n, dst=buf.ctypes.data + 8) == _lib.EINVAL and b"overlap" in err()
    assert call(pol=3, src=buf.ctypes.data + 8 * 4 * n, dst=buf.ctypes.data) == _lib.EINVAL and b"device pointer" in err()
    # quad writes 6 values per sample from 9 bands: an output starting inside the input overlaps it
    assert call(pol=2, dst=buf.ctypes.data + 8 * (9 * n - 1)) == _lib.EINVAL and b"overlap" in err()
    assert call(pol=2, dst=buf.ctypes.data + 8 * 9 * n) == _lib.EINVAL and b"device pointer" in err()
    # the checks come in this order: pol, single-pol, shape and k, dtype, overlap, device
    assert call(pol=7, shape=(4, 5, 0), dtype=2, dst=buf.ctypes.data) == _lib.EINVAL and b"pol=7" in err()
    assert call(pol=1, shape=(0, 5, 0), dtype=2, dst=buf.ctypes.data) == _lib.EINVAL and b"single-pol" in err()
    assert call(shape=(4, 5, 0), dtype=2, dst=buf.ctypes.data) == _lib.EINVAL and b"time step" in err()
    assert call(dtype=2, dst=buf.ctypes.data) == _lib.EDTYPE
    for pol in (0, 2, 3, 4):                 # valid arguments stop at the host pointer
        for dtype in (0, 1):
            assert call(pol=pol, dtype=dtype) == _lib.EINVAL and b"out is not a CUDA device pointer" in err()
    assert (out == 0).all() and (buf == 0).all()


def test_python_validates_before_the_device():
    v = np.zeros((4, 5, 2, 4), np.float32)
    with pytest.raises(ValueError, match="unknown covariance layout"):
        polarimetry.h_a_alpha(v, 'quadpol')
    with pytest.raises(ValueError, match="no H / A / alpha decomposition"):
        polarimetry.h_a_alpha(v[..., :1], 'single')
    with pytest.raises(ValueError, match=r"\(rows, cols, time, 9\)"):
        polarimetry.h_a_alpha(v, 'quad')
    with pytest.raises(ValueError, match=r"\(rows, cols, time, 4\)"):
        polarimetry.h_a_alpha(v[0])
    with pytest.raises(ValueError, match="at least 1 pixel and 1 time step"):
        polarimetry.h_a_alpha(v[:, :, :0])
    with pytest.raises(TypeError, match="No matching signature"):
        polarimetry.h_a_alpha(v.astype(np.int32))
    ds = _dataset(np.ones((4, 5, 3, 4), np.float32), 'dual')
    with pytest.raises(ValueError, match="unknown covariance layout"):
        polarimetry.HAAlphaDecomposition(pol='quadpol').apply(ds)
    with pytest.raises(ValueError, match="no H / A / alpha decomposition"):
        polarimetry.h_a_alpha_decomposition(_dataset(np.ones((4, 5, 3, 1)), 'single'), pol='single')
    with pytest.raises(ValueError, match="needs the variables"):
        polarimetry.h_a_alpha_decomposition(ds, pol='quad')
    partial = ds.copy(deep=True)
    del partial['C12__im']
    with pytest.raises(ValueError, match="missing: C12__im"):
        polarimetry.HAAlphaDecomposition().apply(partial)
    odd = _dataset(np.ones((4, 5, 3, 4), np.float32), 'dual')
    odd['C22'] = (('x', 'y', 'time'), np.ones((5, 4, 3), np.float32))
    with pytest.raises(ValueError, match="share their dims"):
        polarimetry.h_a_alpha_decomposition(odd)
    mixed = _dataset(np.ones((4, 5, 3, 4), np.float32), 'dual')
    mixed['C22'] = (('y', 'x', 'time'), np.ones((4, 5, 3)))
    with pytest.raises(ValueError, match="share one data type"):
        polarimetry.h_a_alpha_decomposition(mixed)


def test_compute_path_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    v = np.ones((4, 5, 2, 4))
    for call in (lambda: polarimetry.h_a_alpha(v), lambda: polarimetry.h_a_alpha_decomposition(_dataset(v, 'dual'))):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            call()


def test_signatures():
    assert set(polarimetry.__all__) == {'h_a_alpha', 'HAAlphaDecomposition', 'h_a_alpha_decomposition'}
    sig = inspect.signature(polarimetry.h_a_alpha).parameters
    assert list(sig) == ['values', 'pol'] and sig['pol'].default == 'dual'
    sig = inspect.signature(polarimetry.HAAlphaDecomposition.__init__).parameters
    assert list(sig) == ['self', 'pol'] and sig['pol'].kind is inspect.Parameter.KEYWORD_ONLY
    assert sig['pol'].default == 'dual'
    sig = inspect.signature(polarimetry.h_a_alpha_decomposition).parameters
    assert 'ds' in sig and sig['pol'].default == 'dual'


# ---- CPU: the oracle -----------------------------------------------------------------------------------
CANONICAL = [   # target, C3 bands, (l1, l2, l3), H, A, alpha
    ('surface', _quad(1, 0, 1, 0, 0, 1), (2, 0, 0), 0.0, 0.0, 0.0),
    ('dihedral', _quad(1, 0, -1, 0, 0, 1), (2, 0, 0), 0.0, 0.0, 90.0),
    ('horizontal dipole', _quad(1), (1, 0, 0), 0.0, 0.0, 45.0),
    ('random volume', _quad(3 / 8, 0, 1 / 8, 2 / 8, 0, 3 / 8), (0.5, 0.25, 0.25), 0.946394630357186, 0.0, 45.0),
    ('T = I', _quad(1, 0, 0, 1, 0, 1), (1, 1, 1), 1.0, 0.0, 54.735610317245346),
]


@pytest.mark.parametrize("target", CANONICAL, ids=[t[0] for t in CANONICAL])
def test_oracle_canonical_targets(target):
    ho = _oracle()
    _, c3, lam, H, A, alpha = target
    for pol, x in (('quad', c3), ('quad_diagonal', c3[[0, 5, 8]])):
        if pol == 'quad_diagonal' and np.any(c3[[1, 2, 3, 4, 6, 7]]):
            continue
        got = ho.h_a_alpha(x, pol)
        np.testing.assert_allclose(got, [H, A, alpha] + list(lam), rtol=0, atol=1e-12, err_msg=pol)


def test_oracle_dual_diagonal_closed_form():
    ho = _oracle()
    rng = np.random.default_rng(1)
    c = rng.gamma(2.0, 1.0, size=(500, 2))
    c[:5, 1] = c[:5, 0]                                           # C11 = C22: 45 degrees, H = 1
    got = ho.h_a_alpha(c, 'dual_diagonal')
    p = c / c.sum(-1, keepdims=True)
    np.testing.assert_allclose(got[:, 1], 90.0 * p[:, 1], rtol=0, atol=1e-10)
    np.testing.assert_allclose(got[:, 0], -(p * np.log2(p)).sum(-1), rtol=0, atol=1e-12)
    np.testing.assert_allclose(got[:, 2:], np.sort(c, -1)[:, ::-1], rtol=1e-15, atol=0)
    assert np.allclose(got[:5, 1], 45.0, rtol=0, atol=1e-12) and np.allclose(got[:5, 0], 1.0, rtol=0, atol=1e-15)


def test_oracle_rank_one_dual():
    ho = _oracle()
    rng = np.random.default_rng(2)
    v = rng.normal(size=(300, 2)) + 1j * rng.normal(size=(300, 2))
    c = np.einsum('ni,nj->nij', v, v.conj())
    got = ho.h_a_alpha(bands(c, 'dual'), 'dual')
    norm = np.linalg.norm(v, axis=-1)
    assert np.abs(got[:, 0]).max() < 1e-12
    np.testing.assert_allclose(got[:, 1], np.degrees(np.arccos(np.abs(v[:, 0]) / norm)), rtol=0, atol=1e-8)
    np.testing.assert_allclose(got[:, 2], norm ** 2, rtol=1e-12)
    assert (got[:, 3] <= 1e-14 * norm ** 2).all()


def _roll(c3, theta):
    """C3 of the Pauli T rolled about the line of sight: T' = R T R^T."""
    cs, sn = np.cos(2 * theta), np.sin(2 * theta)
    R = np.array([[1, 0, 0], [0, cs, sn], [0, -sn, cs]])
    T = PAULI @ c3 @ PAULI.T
    return PAULI.T @ (R @ T @ R.T) @ PAULI


@pytest.mark.parametrize("looks", [1, 2, 4, 16])
@pytest.mark.parametrize("pol", LAYOUTS)
def test_oracle_invariances_and_bounds(pol, looks):
    ho = _oracle()
    rng = np.random.default_rng(looks)
    x = _wishart(400, looks, pol, rng)
    got = ho.h_a_alpha(x, pol)
    cols = _columns(pol)
    n_ang = cols.index('lambda1')
    lam, s = got[:, n_ang:], got[:, n_ang:].sum(-1)
    diag = [change.POLS[pol].index(b) for b in ('C11', 'C22', 'C33') if b in change.POLS[pol]]
    np.testing.assert_allclose(s, x[:, diag].sum(-1), rtol=1e-12)
    assert (lam[:, :-1] >= lam[:, 1:]).all() and (lam >= 0).all()
    assert (got[:, 0] >= -1e-12).all() and (got[:, 0] <= 1 + 1e-12).all()
    alpha = got[:, cols.index('alpha')]
    assert (alpha >= 0).all() and (alpha <= 90 + 1e-12).all()
    if pol.startswith('quad'):
        assert (got[:, 1] >= 0).all() and (got[:, 1] <= 1 + 1e-12).all()
    if looks == 1 and pol in ('dual', 'quad'):                    # rank 1: H = 0, A = 0
        assert np.abs(got[:, 0]).max() < 1e-12
    for scale in (1e-6, 3.7, 2.0 ** 40):
        scaled = ho.h_a_alpha(x * scale, pol)
        np.testing.assert_allclose(scaled[:, :n_ang], got[:, :n_ang], rtol=0, atol=1e-8)
        assert (np.abs(scaled[:, n_ang:] - lam * scale) <= 1e-12 * scale * s[:, None]).all()
    if pol == 'quad':
        c3 = ho.matrices(x, pol)
        for theta in (0.3, -1.1, np.pi / 4):
            rolled = ho.h_a_alpha(_to_bands(_roll(c3, theta), pol), pol)
            assert (np.abs(rolled[:, n_ang:] - lam) <= 1e-12 * s[:, None]).all()
            np.testing.assert_allclose(rolled[:, :n_ang], got[:, :n_ang], rtol=0, atol=1e-8)


@pytest.mark.parametrize("pol", ['dual', 'quad'])
def test_oracle_alpha_equals_the_adjugate_formula(pol):
    """|e_i[0]|^2 = adj(M - l_i I)_00 / prod_{j != i} (l_j - l_i) on samples whose gaps all exceed 1e-3 s."""
    ho = _oracle()
    rng = np.random.default_rng(7)
    x = np.concatenate([_wishart(300, looks, pol, rng) for looks in (3, 4, 16)])
    lam, c, _ = ho.components(x, pol)
    m = ho.matrices(x, pol)
    if pol == 'quad':
        m = PAULI @ m @ PAULI.T
    s = lam.sum(-1)
    ok = ((lam[:, :-1] - lam[:, 1:]) > 1e-3 * s[:, None]).all(-1)
    assert ok.mean() > 0.5
    p = lam.shape[-1]
    for i in range(p):
        shifted = m - lam[:, i, None, None] * np.eye(p)
        adj00 = shifted[:, 1, 1].real if p == 2 else (shifted[:, 1, 1] * shifted[:, 2, 2] - shifted[:, 1, 2] * shifted[:, 2, 1]).real
        den = np.prod([lam[:, j] - lam[:, i] for j in range(p) if j != i], axis=0)
        np.testing.assert_allclose(c[ok, i], (adj00 / den)[ok], rtol=0, atol=1e-9)


# ---- GPU ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("pol", LAYOUTS)
def test_kernel_matches_oracle(pol, dtype):
    x = _pool(pol).astype(dtype)
    n = len(x) // 21 * 21
    got = polarimetry.h_a_alpha(x[:n].reshape(3, 7, -1, x.shape[-1]), pol)
    assert_matches_oracle(got, x[:n].reshape(3, 7, -1, x.shape[-1]), pol)
    for count in (1, 255, 257, len(x)):                           # not multiples of the 256-thread block
        part = x[:count][None, :, None]
        got = polarimetry.h_a_alpha(part, pol)
        assert_matches_oracle(got, part, pol, min_checked=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("pol", LAYOUTS)
def test_targets_and_ties_exactly(pol):
    """The canonical targets and exact ties give the stated values, float32 and float64 alike."""
    ho = _oracle()
    for dtype in (np.float64, np.float32):
        x = np.concatenate([_targets(pol), _exact_ties(pol)]).astype(dtype)[None, None]
        got = polarimetry.h_a_alpha(x, pol)
        assert_matches_oracle(got, x, pol)
    if pol == 'quad':
        got = polarimetry.h_a_alpha(np.array([t[1] for t in CANONICAL])[None, None], pol)[0, 0]
        want = np.array([[t[3], t[4], t[5]] + list(t[2]) for t in CANONICAL])
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-12)
        np.testing.assert_allclose(got, ho.h_a_alpha(np.array([t[1] for t in CANONICAL]), pol), rtol=0, atol=1e-12)


@pytest.mark.gpu
@pytest.mark.parametrize("pol", LAYOUTS)
def test_strided_views_bitwise(pol):
    import torch
    rng = np.random.default_rng(3)
    v = _wishart(37 * 53 * 4, 4, pol, rng).reshape(37, 53, 4, -1)
    n = len(_columns(pol))
    for dtype in (torch.float64, torch.float32):
        t = torch.from_numpy(v).to(dtype).cuda()
        want = polarimetry.h_a_alpha(t.cpu().numpy(), pol)
        spaced = torch.full((37, 106) + t.shape[2:], float('nan'), dtype=dtype, device='cuda')
        spaced[:, ::2] = t
        views = [t.permute(3, 0, 1, 2).contiguous().permute(1, 2, 3, 0),          # variable-major, like `to_array()`
                 t.permute(2, 0, 1, 3).contiguous().permute(1, 2, 0, 3),          # time-major
                 t.transpose(0, 1).contiguous().transpose(0, 1),                  # column-major image
                 spaced[:, ::2]]                                                  # every other pixel of a wider image
        for view in views:
            assert not view.is_contiguous()
            out = torch.empty(view.shape[:3] + (n,), dtype=dtype, device='cuda')
            rc = _lib.lib().ndchg_h_a_alpha(VP(view.data_ptr()), _lib.i64(view.shape[:3]), _lib.i64(view.stride()),
                                            0 if dtype == torch.float32 else 1, change._POL_CODES[pol],
                                            VP(out.data_ptr()), VP(torch.cuda.current_stream().cuda_stream))
            assert rc == 0, _lib.lib().ndchg_last_error()
            assert np.array_equal(out.cpu().numpy(), want, equal_nan=True)


@pytest.mark.gpu
def test_more_than_2_32_elements():
    """Quad-pol float32 (2048, 4096, 57, 9): 4,303,355,904 input elements.  The cube repeats a bank of 4096 samples;
    the first and last samples and those holding input elements 2^31 and 2^32 and output element 2^31 are checked
    against the oracle, in an output first filled with NaN."""
    import torch
    if torch.cuda.mem_get_info()[0] < 40e9:
        pytest.skip("needs 40 GB of free device memory")
    rng = np.random.default_rng(11)
    bank = _wishart(4096, 4, 'quad', rng).astype(np.float32)
    shape = (2048, 4096, 57)
    samples = shape[0] * shape[1] * shape[2]
    assert samples * 9 > 2 ** 32
    values = torch.empty((samples // 4096, 4096, 9), dtype=torch.float32, device='cuda')
    values.copy_(torch.from_numpy(bank).cuda().expand_as(values))
    out = torch.full((samples, 6), float('nan'), dtype=torch.float32, device='cuda')
    values = values.view(shape + (9,))
    rc = _lib.lib().ndchg_h_a_alpha(VP(values.data_ptr()), _lib.i64(shape), _lib.i64(values.stride()), 0,
                                    change._POL_CODES['quad'], VP(out.data_ptr()),
                                    VP(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, _lib.lib().ndchg_last_error()
    torch.cuda.synchronize()
    picks = sorted({0, 1, samples - 2, samples - 1} |
                   {e // 9 + d for e in (2 ** 31, 2 ** 32) for d in (-1, 0, 1)} | {2 ** 31 // 6 + d for d in (-1, 0, 1)})
    got = out[torch.tensor(picks, device='cuda')].cpu().numpy()
    del values, out
    torch.cuda.empty_cache()
    x = bank[np.array(picks) % 4096]
    assert_matches_oracle(got, x, 'quad')


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [('y', 'x', 'time'), ('time', 'y', 'x'), ('y', 'x')])
@pytest.mark.parametrize("pol", LAYOUTS)
def test_dataset_equals_the_array_form(pol, dims):
    k = 3 if 'time' in dims else 1
    rng = np.random.default_rng(5)
    v = _wishart(9 * 11 * k, 4, pol, rng).reshape(9, 11, k, -1).astype(np.float32)
    want = polarimetry.h_a_alpha(v, pol)
    order = [dims.index(d) for d in ('y', 'x', 'time') if d in dims]
    results = []
    for form in ('pairs', 'complex'):
        ds = _dataset(v, pol, dims, complex_c12=form == 'complex', extra=True)
        before = ds.copy(deep=True)
        out = polarimetry.HAAlphaDecomposition(pol=pol).apply(ds)
        assert ds.equals(before) and dict(ds.attrs) == dict(before.attrs)
        assert list(out.data_vars) == _columns(pol) and dict(out.attrs) == dict(ds.attrs)
        assert list(out.coords) == list(ds.coords) and all(np.array_equal(out.coords[c], ds.coords[c]) for c in ds.coords)
        for q, name in enumerate(_columns(pol)):
            assert out[name].dims == dims and out[name].dtype == np.float32, name
            got = np.transpose(out[name].values, order)
            assert np.array_equal(got, want[..., q] if 'time' in dims else want[:, :, 0, q], equal_nan=True), name
        assert polarimetry.h_a_alpha_decomposition(ds, pol=pol).equals(out)
        results.append(out)
    assert results[0].equals(results[1])


@pytest.mark.gpu
def test_dataset_with_an_extra_dim():
    rng = np.random.default_rng(6)
    v = _wishart(8 * 10 * 6, 3, 'quad', rng).reshape(8, 10, 6, 9)
    ref = generate_test_dataset(dims={'y': 8, 'band': 2, 'x': 10, 'time': 3}, var=())
    ds = Dataset(coords=ref.coords, attrs=ref.attrs)
    for b, name in enumerate(change.POLS['quad']):
        ds[name] = (('y', 'band', 'x', 'time'), np.ascontiguousarray(v[..., b].reshape(8, 10, 2, 3).transpose(0, 2, 1, 3)))
    out = polarimetry.h_a_alpha_decomposition(ds, pol='quad')
    want = polarimetry.h_a_alpha(v, 'quad')
    for q, name in enumerate(_columns('quad')):
        assert out[name].dims == ('y', 'band', 'x', 'time')
        assert np.array_equal(out[name].values, want[..., q].reshape(8, 10, 2, 3).transpose(0, 2, 1, 3))
