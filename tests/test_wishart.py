"""
H / alpha zones and the unsupervised Wishart classification (include/ndchg.h, `ndchg_h_alpha_zones`,
`ndchg_wishart_classify`; `polarimetry.h_alpha_zones`, `wishart_classify`, `WishartClassification`).

The NumPy oracle (`oracle/wishart_oracle.py`) is tied to facts it does not compute itself: the affine distance equals
ln det V + tr(V^-1 C) from LAPACK, classifying C equals classifying the Pauli T, the Wishart objective does not
increase, values on the zone boundaries land on the stated side, and a scene of canonical scatterers starts in the
expected zones and ends in classes that each hold one patch.  The CUDA kernels are compared with the oracle: zones
exactly, labels exactly wherever the oracle's margin between the best and second-best distance exceeds 1e-10
(relative to the size of the terms of the distance), counts exactly, and centres to 1e-13 (one pass) or 1e-12 (the
whole loop) relative.
"""
import ctypes

import numpy as np
import pytest

from nd_b200 import _lib, change, polarimetry
from test_change_pol import P, bands
from test_refined_lee import _dataset

LAYOUTS = ['dual', 'quad', 'dual_diagonal', 'quad_diagonal']
VP = ctypes.c_void_p
PAULI = np.array([[1, 0, 1], [1, 0, -1], [0, np.sqrt(2), 0]]) / np.sqrt(2)


def _wo():
    from oracle import wishart_oracle as wo
    return wo


def _sigmas(pol, count, rng):
    """`count` distinct well-conditioned covariances of `pol` (p x p), at powers 0.1 to 10."""
    p = P[pol]
    out = []
    for _ in range(count):
        a = rng.normal(size=(p, p)) + 1j * rng.normal(size=(p, p))
        out.append((a @ a.conj().T + 0.3 * np.eye(p)) * 10.0 ** rng.uniform(-1, 1))
    return out


def _draw(sigmas, which, looks, rng):
    """`looks`-look sample covariances (n, p, p) of the classes `which` (n,) of `sigmas`."""
    chol = np.linalg.cholesky(np.asarray(sigmas))[which]
    p = chol.shape[-1]
    w = (rng.normal(size=(len(which), looks, p)) + 1j * rng.normal(size=(len(which), looks, p))) / np.sqrt(2)
    z = np.einsum('nlj,nij->nli', w, chol)
    return np.einsum('nli,nlj->nij', z, z.conj()) / looks


def _scene(pol, n, looks=4, centres=4, seed=0):
    """n samples (n, bands) of `pol` drawn from `centres` distinct covariances, and their classes 0.."""
    rng = np.random.default_rng(seed)
    truth = rng.integers(0, centres, n)
    return bands(_draw(_sigmas(pol, centres, rng), truth, looks, rng), pol), truth


def _seeded(truth, K, rng, flip=0.2):
    """Initial labels 1..K: the true class + 1, with a fraction `flip` replaced by random labels."""
    lab = truth + 1
    swap = rng.random(len(lab)) < flip
    return np.where(swap, rng.integers(1, K + 1, len(lab)), lab).astype(np.uint8)


def _call(values, labels, K, pol, max_iter=10, tol=0.0, t=None):
    """ndchg_wishart_classify on device copies: (rc, labels, centres, counts, iterations).  `t` overrides the device
    tensor of `values` (a strided view)."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(values)).cuda() if t is None else t
    lab = torch.from_numpy(np.ascontiguousarray(labels, np.uint8)).cuda()
    B = t.shape[-1]
    centres = torch.full((K, B), -1.0, dtype=torch.float64, device='cuda')
    counts = torch.full((K,), -1, dtype=torch.int64, device='cuda')
    its = torch.full((1,), -1, dtype=torch.int32, device='cuda')
    rc = _lib.lib().ndchg_wishart_classify(VP(t.data_ptr()), _lib.i64(t.shape[:3]), _lib.i64(t.stride()),
                                           0 if t.dtype == torch.float32 else 1, change._POL_CODES[pol], VP(lab.data_ptr()),
                                           K, max_iter, tol, VP(centres.data_ptr()), VP(counts.data_ptr()),
                                           VP(its.data_ptr()), VP(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc, lab.cpu().numpy(), centres.cpu().numpy(), counts.cpu().numpy(), int(its.cpu().numpy()[0])


def _rel(a, b):
    ok = np.isfinite(b)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    return float((np.abs(a[ok] - b[ok]) / np.abs(b[ok]).max()).max()) if ok.any() else 0.0


# ---- CPU: C ABI and Python boundary --------------------------------------------------------------------
def test_c_abi_checks_arguments_before_the_device():
    L = _lib.lib()
    buf = np.zeros(8192, np.float64)
    lab = np.zeros(8192, np.uint8)
    small = np.zeros(64, np.float64)
    def strides(shape, pol):
        B = (4, 1, 9, 2, 3)[pol] if 0 <= pol <= 4 else 4
        return [shape[1] * shape[2] * B, shape[2] * B, B, 1]
    def zones(shape=(4, 5, 3), dtype=1, pol=0, anis=0, dst=None):
        dst = lab.ctypes.data if dst is None else dst
        return L.ndchg_h_alpha_zones(VP(buf.ctypes.data), _lib.i64(shape), _lib.i64(strides(shape, pol)), dtype, pol, anis,
                                     VP(dst), None)
    def classify(shape=(4, 5, 3), dtype=1, pol=0, classes=9, tol=0.0, dst=None):
        dst = lab.ctypes.data if dst is None else dst
        return L.ndchg_wishart_classify(VP(buf.ctypes.data), _lib.i64(shape), _lib.i64(strides(shape, pol)), dtype, pol,
                                        VP(dst), classes, 10, tol, VP(small.ctypes.data), VP(small.ctypes.data),
                                        VP(small.ctypes.data), None)
    def err():
        return L.ndchg_last_error()
    for call in (zones, classify):
        for pol in (-1, 5, 99):
            assert call(pol=pol) == _lib.EINVAL and b"pol=%d" % pol in err()
        assert call(pol=1) == _lib.EINVAL and b"single-pol" in err()
        for shape in ((0, 5, 3), (4, 0, 3), (4, -1, 3)):
            assert call(shape=shape) == _lib.EINVAL and b"shape out of range" in err()
        for shape in ((4, 5, 0), (4, 5, -2)):
            assert call(shape=shape) == _lib.EINVAL and b"at least 1 time step" in err()
        assert call(dtype=2) == _lib.EDTYPE and b"No matching signature" in err()
        # labels / zones inside the input, at its first and its last byte
        assert call(dst=buf.ctypes.data) == _lib.EINVAL and b"must not overlap" in err()
        assert call(dst=buf.ctypes.data + 8 * 4 * 60 - 1) == _lib.EINVAL and b"must not overlap" in err()
        assert call(dst=buf.ctypes.data + 8 * 4 * 60) == _lib.EINVAL and b"device pointer" in err()
        # the device check comes last: valid arguments stop at the host pointer
        for pol in (0, 2, 3, 4):
            for dtype in (0, 1):
                assert call(pol=pol, dtype=dtype) == _lib.EINVAL and b"is not a CUDA device pointer" in err()
    for pol in (0, 3):
        assert zones(pol=pol, anis=1) == _lib.EINVAL and b"anisotropy needs a quad layout" in err()
    assert zones(anis=2, pol=2) == _lib.EINVAL and b"anisotropy must be 0 or 1" in err()
    for pol in (2, 4):
        assert zones(pol=pol, anis=1) == _lib.EINVAL and b"device pointer" in err()
    for classes in (0, 33, 255):
        assert classify(classes=classes) == _lib.EINVAL and b"classes must be in [1, 32]" in err()
    for tol in (-1e-9, 1.000001, float('nan'), float('inf')):
        assert classify(tol=tol) == _lib.EINVAL and b"tol must be in [0, 1]" in err()
    for classes, tol in ((1, 0.0), (32, 1.0)):
        assert classify(classes=classes, tol=tol) == _lib.EINVAL and b"device pointer" in err()
    # the order: pol, single-pol, (anisotropy,) shape and k, dtype, (classes, tol,) overlap, device
    assert zones(pol=7, anis=1, shape=(0, 5, 3), dtype=2) == _lib.EINVAL and b"pol=7" in err()
    assert zones(pol=1, anis=1, shape=(0, 5, 3)) == _lib.EINVAL and b"single-pol" in err()
    assert zones(pol=0, anis=1, shape=(0, 5, 3)) == _lib.EINVAL and b"anisotropy" in err()
    assert zones(shape=(4, 5, 0), dtype=2) == _lib.EINVAL and b"time step" in err()
    assert zones(dtype=2, dst=buf.ctypes.data) == _lib.EDTYPE
    assert classify(pol=1, shape=(0, 5, 3), classes=0) == _lib.EINVAL and b"single-pol" in err()
    assert classify(shape=(0, 5, 3), dtype=2, classes=0) == _lib.EINVAL and b"shape" in err()
    assert classify(dtype=2, classes=0) == _lib.EDTYPE
    assert classify(classes=0, tol=2.0, dst=buf.ctypes.data) == _lib.EINVAL and b"classes" in err()
    assert classify(tol=2.0, dst=buf.ctypes.data) == _lib.EINVAL and b"tol" in err()
    assert (lab == 0).all() and (buf == 0).all() and (small == 0).all()


def test_python_validates_before_the_device():
    v = np.zeros((4, 5, 2, 4), np.float32)
    with pytest.raises(ValueError, match="unknown covariance layout"):
        polarimetry.h_alpha_zones(v, 'quadpol')
    with pytest.raises(ValueError, match="no H / A / alpha decomposition"):
        polarimetry.wishart_classify(v[..., :1], 'single')
    with pytest.raises(ValueError, match="anisotropy=True needs a quad layout"):
        polarimetry.h_alpha_zones(v, anisotropy=True)
    with pytest.raises(ValueError, match="init='h_a_alpha' needs a quad layout"):
        polarimetry.wishart_classify(v, init='h_a_alpha')
    with pytest.raises(ValueError, match="init must be"):
        polarimetry.wishart_classify(v, init='kmeans')
    with pytest.raises(ValueError, match="has shape"):
        polarimetry.wishart_classify(v, init=np.ones((4, 5), np.int64))
    with pytest.raises(TypeError, match="integer type"):
        polarimetry.wishart_classify(v, init=np.ones((4, 5, 2)))
    for bad in (np.zeros((4, 5, 2), np.int64), np.full((4, 5, 2), 33), np.full((4, 5, 2), -1)):
        with pytest.raises(ValueError, match=r"init labels must lie in \[0, 32\]"):
            polarimetry.wishart_classify(v, init=bad)
    with pytest.raises(ValueError, match="max_iter"):
        polarimetry.wishart_classify(v, max_iter=-1)
    with pytest.raises(ValueError, match="tol"):
        polarimetry.wishart_classify(v, tol=1.5)
    with pytest.raises(ValueError, match=r"\(rows, cols, time, 9\)"):
        polarimetry.wishart_classify(v, 'quad')
    with pytest.raises(ValueError, match="needs the variables"):
        polarimetry.wishart_classification(_dataset(np.ones((4, 5, 3, 4), np.float32), 'dual'), pol='quad')
    with pytest.raises(ValueError, match="has shape"):
        polarimetry.WishartClassification(init=np.ones((4, 5), np.int64)).apply(_dataset(np.ones((4, 5, 3, 4), np.float32), 'dual'))


def test_compute_path_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    v = np.ones((4, 5, 2, 4))
    for call in (lambda: polarimetry.h_alpha_zones(v), lambda: polarimetry.wishart_classify(v),
                 lambda: polarimetry.wishart_classification(_dataset(v, 'dual'))):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            call()


# ---- CPU: the oracle -----------------------------------------------------------------------------------
def _matrices(x, pol):
    from oracle.h_a_alpha_oracle import matrices
    return matrices(x, pol)


@pytest.mark.parametrize("pol", LAYOUTS)
def test_oracle_distance_is_logdet_plus_trace(pol):
    wo = _wo()
    x, truth = _scene(pol, 600, looks=3, centres=5, seed=1)
    V, n = wo.centres(x, truth + 1, 5)
    g, w, det, act = wo.table(V, n, pol)
    assert act.all()
    M = _matrices(V, pol)
    sign, logdet = np.linalg.slogdet(M)
    want = logdet[None, :] + np.einsum('kij,nji->nk', np.linalg.inv(M), _matrices(x, pol)).real
    assert np.allclose(sign, 1.0, rtol=0, atol=1e-12)
    np.testing.assert_allclose(np.exp(logdet), det, rtol=1e-12)
    got = wo.distances(x, g, w)
    assert (np.abs(got - want) <= 1e-12 * np.abs(want).max(1, keepdims=True)).all()


def _classify_t(T, labels, K, max_iter):
    """k-means with d = ln det V + tr(V^-1 T) on Hermitian matrices T (n, 3, 3) with LAPACK: the label history."""
    lab = labels.copy()
    history = [lab.copy()]
    for _ in range(max_iter):
        Vs = np.array([T[lab == m].mean(0) for m in range(1, K + 1)])
        d = np.linalg.slogdet(Vs)[1][None, :] + np.einsum('kij,nji->nk', np.linalg.inv(Vs), T).real
        new = np.argmin(d, 1) + 1
        changed = (new != lab).sum()
        lab = new
        history.append(lab.copy())
        if changed == 0:
            break
    return history


def test_oracle_c_and_pauli_t_give_the_same_labels():
    wo = _wo()
    rng = np.random.default_rng(2)
    x, truth = _scene('quad', 3000, looks=4, centres=4, seed=2)
    init = _seeded(truth, 4, rng, flip=0.5)
    r = wo.classify(x, init, 4, 'quad', max_iter=20)
    assert (r['margin'] > 1e-10).all() and r['iterations'] >= 3
    T = PAULI @ _matrices(x, 'quad') @ PAULI.T
    hist = _classify_t(T, init.astype(np.int64), 4, 20)
    assert len(hist) == len(r['history'])
    for a, b in zip(hist, r['history']):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("pol", LAYOUTS)
def test_oracle_objective_does_not_increase(pol):
    """sum over samples of d_label(C) with the centres of the labels, from LAPACK, after every iteration."""
    wo = _wo()
    rng = np.random.default_rng(3)
    x, truth = _scene(pol, 2000, looks=3, centres=5, seed=3)
    r = wo.classify(x, rng.integers(1, 7, len(x)), 6, pol, max_iter=30)
    assert r['iterations'] >= 3
    C = _matrices(x, pol)
    J = []
    for lab in r['history']:
        total = 0.0
        for m in np.unique(lab):
            V = C[lab == m].mean(0)
            total += (np.linalg.slogdet(V)[1] + np.einsum('ij,nji->n', np.linalg.inv(V), C[lab == m]).real).sum()
        J.append(total)
    J = np.array(J)
    assert (np.diff(J) <= 1e-9 * np.abs(J).max()).all(), J


def test_oracle_zone_boundaries():
    wo = _wo()
    up = lambda v: np.nextafter(v, np.inf)
    down = lambda v: np.nextafter(v, -np.inf)
    cases = [  # (H, alpha, zone)
        (0.9, 55.0, 1), (0.9, down(55.0), 2), (0.9, 40.0, 2), (0.9, down(40.0), 3), (1.0, 90.0, 1), (1.0, 0.0, 3),
        (down(0.9), 55.0, 4), (down(0.9), 50.0, 4), (down(0.9), down(50.0), 5), (0.5, 40.0, 5), (0.5, down(40.0), 6),
        (down(0.5), 50.0, 7), (down(0.5), 47.5, 7), (down(0.5), down(47.5), 8), (0.0, 42.5, 8), (0.0, down(42.5), 9),
        (0.0, 0.0, 9), (np.nan, 45.0, 0), (0.3, np.nan, 0), (up(0.9), up(40.0), 2)]
    H, alpha, want = (np.array(c) for c in zip(*cases))
    assert np.array_equal(wo.zones(H, alpha), want.astype(np.uint8))
    A = np.where(np.arange(len(H)) % 2 == 0, 0.5, up(0.5))
    assert np.array_equal(wo.zones(H, alpha, A), np.where((want > 0) & (A > 0.5), want + 9, want).astype(np.uint8))
    # float32 outputs are compared in double: a float32 just below 0.9 is below it
    assert wo.zones(np.float32(0.9), np.float32(55.0)) == (4 if np.float64(np.float32(0.9)) < 0.9 else 1)


def test_oracle_scatterer_scene_starts_in_its_zones_and_ends_in_pure_classes():
    """Surface, dihedral and random-volume patches of quad-pol data at 16 looks start in zone 9, zone 7 and mostly
    zones 2 / 5; the loop converges to classes that each hold one patch (the volume patch may spread over several
    classes, as Wishart k-means does on a random volume), and surface and dihedral keep one class each."""
    from oracle import h_a_alpha_oracle as ho
    wo = _wo()
    x, truth = _scatterers(2000, 16, seed=4)
    z = wo.zones_of(ho.h_a_alpha(x, 'quad'), 'quad')
    assert (z[truth == 0] == 9).mean() > 0.99 and (z[truth == 1] == 7).mean() > 0.99
    vol = z[truth == 2]
    assert np.isin(vol, [2, 5]).mean() > 0.75 and not np.isin(vol, [7, 8, 9]).any()
    r = wo.classify(x, z, 9, 'quad', max_iter=50)
    assert r['iterations'] < 50                                   # converged: no label changed in the last pass
    assert _purity(r['labels'], truth) == 1.0
    assert len(np.unique(r['labels'][truth == 0])) == 1 and len(np.unique(r['labels'][truth == 1])) == 1


def _scatterers(n, looks, seed):
    """n samples each of a surface, a dihedral and a random volume (quad C3 bands) and their patch 0 / 1 / 2."""
    rng = np.random.default_rng(seed)
    Ts = [np.diag([1.0, 0.05, 0.02]), np.diag([0.05, 1.0, 0.02]), np.diag([2.0, 1.0, 1.0]) / 4]
    sigmas = [PAULI.T @ T @ PAULI for T in Ts]
    truth = np.repeat(np.arange(3), n)
    return bands(_draw(sigmas, truth, looks, rng), 'quad'), truth


def _purity(labels, truth):
    """The fraction of samples whose class's majority patch is their own patch."""
    hits = 0
    for m in np.unique(labels):
        hits += np.bincount(truth[labels == m]).max()
    return hits / len(labels)


# ---- GPU ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("pol", LAYOUTS)
def test_zones_equal_the_oracle_on_the_kernels_own_h_a_alpha(pol, dtype):
    from test_h_a_alpha import _pool
    wo = _wo()
    x = _pool(pol).astype(dtype)
    n = len(x) // 21 * 21
    for anis in ([False, True] if pol.startswith('quad') else [False]):
        for part in [x[:n].reshape(3, 7, -1, x.shape[-1])] + [x[:c][None, :, None] for c in (1, 255, 257, len(x))]:
            got = polarimetry.h_alpha_zones(part, pol, anisotropy=anis)
            want = wo.zones_of(polarimetry.h_a_alpha(part, pol), pol, anis)
            assert got.dtype == np.uint8 and np.array_equal(got, want)
        assert (got == 0).sum() >= 5                              # NaN / inf / zero samples
        assert len(np.unique(got)) >= (8 if anis else 5)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("pol", LAYOUTS)
def test_one_pass_matches_the_oracle(pol, dtype):
    wo = _wo()
    rng = np.random.default_rng(5)
    x, truth = _scene(pol, 37 * 41 * 23, looks=4, centres=6, seed=5)
    x = x.astype(dtype)
    init = rng.integers(0, 10, len(x)).astype(np.uint8)          # 9 classes, some samples unlabelled
    rc, lab, centres, counts, its = _call(x.reshape(37, 41, 23, -1), init.reshape(37, 41, 23), 9, pol, max_iter=1)
    assert rc == 0 and its == 1
    r = wo.classify(x, init, 9, pol, max_iter=1)
    ok = r['margin'] > 1e-10
    assert ok.mean() > 0.999
    assert np.array_equal(lab.ravel()[ok], r['labels'][ok])
    if np.array_equal(lab.ravel(), r['labels']):
        assert np.array_equal(counts, r['counts'])
        assert _rel(centres, r['centres']) <= 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("pol", LAYOUTS)
def test_full_loop_equals_the_oracle(pol, dtype):
    wo = _wo()
    rng = np.random.default_rng(6)
    x, truth = _scene(pol, 64 * 50 * 7, looks=6, centres=5, seed=6)
    x = x.astype(dtype)
    init = _seeded(truth, 7, rng, flip=0.4)
    r = wo.classify(x, init, 7, pol, max_iter=25)
    assert r['margin'].min() > 1e-10 and r['iterations'] >= 3
    rc, lab, centres, counts, its = _call(x.reshape(64, 50, 7, -1), init.reshape(64, 50, 7), 7, pol, max_iter=25)
    assert rc == 0
    assert np.array_equal(lab.ravel(), r['labels']) and its == r['iterations']
    assert np.array_equal(counts, r['counts']) and _rel(centres, r['centres']) <= 1e-12
    # the Python form, and the stopping rule with tol: at most tol of the valid samples changed in the last pass
    labels, c2, its2 = polarimetry.wishart_classify(x.reshape(64, 50, 7, -1), pol, init.reshape(64, 50, 7), 25)
    assert np.array_equal(labels, lab) and np.array_equal(c2, centres, equal_nan=True) and its2 == its
    r = wo.classify(x, init, 7, pol, max_iter=25, tol=0.01)
    assert polarimetry.wishart_classify(x.reshape(64, 50, 7, -1), pol, init.reshape(64, 50, 7), 25, 0.01)[2] == r['iterations']
    assert r['iterations'] < its


@pytest.mark.gpu
@pytest.mark.parametrize("pol", LAYOUTS)
def test_edge_cases(pol):
    wo = _wo()
    rng = np.random.default_rng(7)
    x, truth = _scene(pol, 3000, looks=5, centres=3, seed=7)
    B = x.shape[1]
    # class 4 is empty; class 5 holds one rank-1 single-look sample (singular for the full layouts)
    single = bands(_draw(_sigmas(pol, 1, rng), np.zeros(1, int), 1, rng), pol)
    x = np.concatenate([x, single, np.full((1, B), np.nan), np.zeros((1, B)), -np.ones((1, B))])
    x[-1, 1:] = 0.0                                                # trace < 0, finite
    init = np.concatenate([truth + 1, [5, 2, 3, 1]]).astype(np.uint8)
    rc, lab, centres, counts, its = _call(x[None, None], init[None, None], 5, pol, max_iter=10)
    assert rc == 0
    lab = lab.ravel()
    r = wo.classify(x, init, 5, pol, max_iter=10)
    assert np.array_equal(lab, r['labels']) and np.array_equal(counts, r['counts'])
    assert (lab[-3:] == 0).all() and counts[3] == 0 and np.isnan(centres[3]).all()
    if pol in ('dual', 'quad'):                                    # the singular class loses its sample
        assert np.isnan(centres[4]).all() and lab[-4] != 5
    # a label > K: EINVAL, nothing written
    bad = init.copy()
    bad[1234] = 6
    rc, lab2, centres2, counts2, its2 = _call(x[None, None], bad[None, None], 5, pol)
    assert rc == _lib.EINVAL and b"exceeds classes=5" in _lib.lib().ndchg_last_error()
    assert np.array_equal(lab2.ravel(), bad) and (centres2 == -1).all() and (counts2 == -1).all() and its2 == -1
    # no active class after iteration 0
    rc = _call(x[None, None], np.where(init == 4, 4, 0)[None, None].astype(np.uint8), 5, pol)[0]
    assert rc == _lib.EINVAL and b"no class is active" in _lib.lib().ndchg_last_error()
    # max_iter = 0: the initial labels (invalid samples set to 0) and their centres
    rc, lab3, centres3, counts3, its3 = _call(x[None, None], init[None, None], 5, pol, max_iter=0)
    assert rc == 0 and its3 == 0 and np.array_equal(lab3.ravel(), np.where(wo.valid(x, pol), init, 0))
    assert _rel(centres3, wo.classify(x, init, 5, pol, max_iter=0)['centres']) <= 1e-13


@pytest.mark.gpu
@pytest.mark.parametrize("pol", LAYOUTS)
def test_bit_identical_across_calls_and_strides(pol):
    import torch
    x, truth = _scene(pol, 37 * 53 * 6, looks=4, centres=4, seed=8)
    v = x.reshape(37, 53, 6, -1)
    for dtype in (torch.float64, torch.float32):
        t = torch.from_numpy(v).to(dtype).cuda()
        init = polarimetry.h_alpha_zones(t.cpu().numpy(), pol)
        want = _call(None, init, 9, pol, t=t)
        assert want[0] == 0 and want[4] >= 2
        again = _call(None, init, 9, pol, t=t)
        spaced = torch.full((37, 106) + t.shape[2:], float('nan'), dtype=dtype, device='cuda')
        spaced[:, ::2] = t
        views = [t.permute(3, 0, 1, 2).contiguous().permute(1, 2, 3, 0),          # variable-major, like `to_array()`
                 t.permute(2, 0, 1, 3).contiguous().permute(1, 2, 0, 3),          # time-major
                 spaced[:, ::2]]                                                  # every other pixel of a wider image
        for got in [again] + [_call(None, init, 9, pol, t=view) for view in views]:
            assert got[0] == 0 and got[4] == want[4]
            assert np.array_equal(got[1], want[1]) and np.array_equal(got[3], want[3])
            assert np.array_equal(got[2], want[2], equal_nan=True)


@pytest.mark.gpu
def test_more_than_2_32_elements():
    """One pass on dual-diagonal float32 (2048, 4096, 300, 2): 2,516,582,400 samples, 5,033,164,800 input elements.
    The cube and the labels repeat a bank of 4096 samples, so the class means are the bank's; labels are checked
    against the oracle's pass on the bank at the ends and around sample 2^31 (input element 2^32)."""
    import torch
    if torch.cuda.mem_get_info()[0] < 40e9:
        pytest.skip("needs 40 GB of free device memory")
    wo = _wo()
    rng = np.random.default_rng(11)
    bank, truth = _scene('dual_diagonal', 4096, looks=4, centres=4, seed=11)
    bank = bank.astype(np.float32)
    init = _seeded(truth, 6, rng, flip=0.5)
    shape = (2048, 4096, 300)
    samples = shape[0] * shape[1] * shape[2]
    assert samples * 2 > 2 ** 32 and samples > 2 ** 31
    values = torch.empty((samples // 4096, 4096, 2), dtype=torch.float32, device='cuda')
    values.copy_(torch.from_numpy(bank).cuda().expand_as(values))
    labels = torch.empty((samples // 4096, 4096), dtype=torch.uint8, device='cuda')
    labels.copy_(torch.from_numpy(init).cuda().expand_as(labels))
    values = values.view(shape + (2,))
    centres = torch.empty((6, 2), dtype=torch.float64, device='cuda')
    counts = torch.empty(6, dtype=torch.int64, device='cuda')
    its = torch.empty(1, dtype=torch.int32, device='cuda')
    rc = _lib.lib().ndchg_wishart_classify(VP(values.data_ptr()), _lib.i64(shape), _lib.i64(values.stride()), 0,
                                           change._POL_CODES['dual_diagonal'], VP(labels.data_ptr()), 6, 1, 0.0,
                                           VP(centres.data_ptr()), VP(counts.data_ptr()), VP(its.data_ptr()),
                                           VP(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, _lib.lib().ndchg_last_error()
    torch.cuda.synchronize()
    picks = sorted({0, 1, samples - 2, samples - 1} | {2 ** 31 + d for d in range(-300, 300)} |
                   {2 ** 32 // 3 + d for d in range(-300, 300)})
    got = labels.view(-1)[torch.tensor(picks, device='cuda')].cpu().numpy()
    centres, counts = centres.cpu().numpy(), counts.cpu().numpy()
    del values, labels
    torch.cuda.empty_cache()
    r = wo.classify(bank, init, 6, 'dual_diagonal', max_iter=1)
    assert (r['margin'] > 1e-10).all()
    assert np.array_equal(got, r['labels'][np.array(picks) % 4096])
    assert np.array_equal(counts, r['counts'] * (samples // 4096)) and _rel(centres, r['centres']) <= 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [('y', 'x', 'time'), ('time', 'y', 'x')])
@pytest.mark.parametrize("pol", LAYOUTS)
def test_dataset_equals_the_array_form(pol, dims):
    """Every sample is classified against one set of centres and the sums follow the order of the samples, so the
    Dataset form equals the array form of the samples in the Dataset's dim order bit for bit."""
    x, _ = _scene(pol, 9 * 11 * 5, looks=4, centres=3, seed=12)
    v = x.reshape(9, 11, 5, -1).astype(np.float32)
    order = [('y', 'x', 'time').index(d) for d in dims]
    flat = np.transpose(v, order + [3]).reshape(1, 1, -1, v.shape[-1])
    want, wc, wi = polarimetry.wishart_classify(flat, pol)
    results = []
    for form in ('pairs', 'complex'):
        ds = _dataset(v, pol, dims, complex_c12=form == 'complex', extra=True)
        before = ds.copy(deep=True)
        out = polarimetry.WishartClassification(pol=pol).apply(ds)
        assert ds.equals(before)
        assert list(out.data_vars) == ['label'] and out['label'].dims == dims and out['label'].dtype == np.uint8
        assert list(out.coords) == list(ds.coords)
        assert np.array_equal(out['label'].values.ravel(), want.ravel())
        assert np.array_equal(out.attrs['wishart_centres'], wc, equal_nan=True) and out.attrs['wishart_iterations'] == wi
        assert {k: v for k, v in out.attrs.items() if not k.startswith('wishart_')} == dict(ds.attrs)
        again = polarimetry.wishart_classification(ds, pol=pol)
        assert np.array_equal(again['label'].values, out['label'].values)
        results.append(out)
    assert np.array_equal(results[0]['label'].values, results[1]['label'].values)
    # an init label array over the dims of the variables
    init = np.transpose(np.arange(9 * 11 * 5).reshape(9, 11, 5) % 4, order)
    out = polarimetry.wishart_classification(ds, pol=pol, init=init, max_iter=3)
    want, _, _ = polarimetry.wishart_classify(flat, pol, init.reshape(1, 1, -1), 3)
    assert np.array_equal(out['label'].values.ravel(), want.ravel())


@pytest.mark.gpu
def test_refined_lee_then_wishart_recovers_a_three_patch_scene():
    """4-look quad-pol surface / dihedral / volume stripes, filtered with the 7 x 7 refined Lee filter and
    classified from the H / alpha zones: >= 99 % of the pixels lie in a class whose majority is their own patch."""
    from nd_b200 import speckle
    x, truth = _scatterers(96 * 128, 4, seed=13)
    v = np.concatenate([x[truth == c].reshape(96, 128, 1, 9) for c in range(3)], axis=1)
    patch = np.repeat(np.arange(3), 128)[None, :].repeat(96, 0)
    ds = _dataset(v, 'quad', complex_c12=True)
    filtered = speckle.refined_lee_filter(ds, pol='quad', looks=4)
    out = polarimetry.wishart_classification(filtered, pol='quad', max_iter=20)
    lab = out['label'].values[..., 0]
    assert _purity(lab.ravel(), patch.ravel()) >= 0.99
