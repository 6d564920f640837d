"""
Omnibus change detection for the covariance layouts beyond dual-pol (include/ndchg.h): single-pol, quad-pol and the
intensity-only dual / quad diagonals.

No reference binary exists for these layouts.  The NumPy oracle (`oracle/omnibus_pol_oracle.py`,
`omnibus_probability_pol`) is tied to the pinned reference at pol='dual', checked by the identities of the statistic
(diagonal z = sum of single-band z, single = one band of a diagonal, quad with zero off-diagonals = quad diagonal),
and by the distribution of the probability under H0: uniform on (0, 1) when f, rho and omega2 are right.  The CUDA
kernels are compared with that oracle: probabilities to 1e-12 (float64 data) / 1.2e-7 (float32 data: the double
result rounded once), change maps identical.
"""
import ctypes
import inspect
import json
import os

import numpy as np
import pytest

from nd_b200 import _lib, change
from nd_b200.dataset import DataArray, Dataset, generate_test_dataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAYOUTS = ['single', 'quad', 'dual_diagonal', 'quad_diagonal']
P = {'dual': 2, 'single': 1, 'quad': 3, 'dual_diagonal': 2, 'quad_diagonal': 3}
# a fixed Hermitian positive definite 3 x 3 covariance (correlated channels, unequal powers)
SIGMA = np.array([[1.0, 0.3 + 0.2j, 0.1 - 0.25j], [0.3 - 0.2j, 0.7, 0.2 + 0.1j], [0.1 + 0.25j, 0.2 - 0.1j, 0.5]])


def covariances(shape, looks, scales, p, rng, diagonal=False):
    """n-look sample covariances (*shape, k, p, p) of complex Gaussian channels with covariance scales[t] * Sigma
    (its leading p x p block; only the diagonal of it for the intensity-only layouts)."""
    sigma = SIGMA[:p, :p] if not diagonal else np.diag(np.diag(SIGMA)[:p]).astype(complex)
    k = len(scales)
    w = (rng.normal(size=shape + (k, looks, p)) + 1j * rng.normal(size=shape + (k, looks, p))) / np.sqrt(2)
    z = (w @ np.linalg.cholesky(sigma).T) * np.sqrt(np.asarray(scales, np.float64))[:, None, None]
    return np.einsum('...li,...lj->...ij', z, z.conj()) / looks


def bands(c, pol):
    """The bands of layout `pol` (nd_b200.change.POLS order) from covariances (..., p, p)."""
    if pol == 'dual':
        return np.stack([c[..., 0, 0].real, c[..., 0, 1].real, c[..., 0, 1].imag, c[..., 1, 1].real], -1)
    if pol == 'quad':
        return np.stack([c[..., 0, 0].real, c[..., 0, 1].real, c[..., 0, 1].imag, c[..., 0, 2].real, c[..., 0, 2].imag,
                         c[..., 1, 1].real, c[..., 1, 2].real, c[..., 1, 2].imag, c[..., 2, 2].real], -1)
    return np.stack([c[..., i, i].real for i in range(P[pol])], -1)


def series(rows, cols, k, looks, scales, pol, seed=0, dtype=np.float64):
    """(rows, cols, k, bands) samples of layout `pol` whose scene power follows `scales[t]`."""
    rng = np.random.default_rng(seed)
    c = covariances((rows, cols), looks, scales, P[pol], rng, diagonal=pol.endswith('diagonal'))
    return bands(c, pol).astype(dtype)


# ---- CPU: C ABI and Python boundary --------------------------------------------------------------------
def test_c_abi_rejects_unknown_layout_and_quad_with_few_looks():
    L = _lib.lib()
    buf = np.zeros(64, np.float64)
    out = np.zeros(64, np.float64)
    shape, strides = _lib.i64([2, 2, 4]), _lib.i64([36, 9, 9, 1])
    vp = ctypes.c_void_p
    def both(pol, n):
        return [L.ndchg_change_detection_pol(vp(buf.ctypes.data), shape, strides, 1, pol, vp(out.ctypes.data), 0.5, n, None),
                L.ndchg_omnibus_probability_pol(vp(buf.ctypes.data), shape, strides, 1, pol, vp(out.ctypes.data), n, None)]
    for pol in (-1, 5, 99):
        for rc in both(pol, 9):
            assert rc == _lib.EINVAL and b"pol=%d" % pol in L.ndchg_last_error()
    for rc in both(2, 2):
        assert rc == _lib.EINVAL and b"n >= 3" in L.ndchg_last_error()
    for pol in range(5):                     # valid arguments pass the layout checks and stop at the host pointer
        for rc in both(pol, 3):
            assert rc == _lib.EINVAL and b"not a CUDA device pointer" in L.ndchg_last_error()
    assert both(1, 0)[0] == _lib.EINVAL and b"n must be >= 1" in L.ndchg_last_error()


def test_python_validates_layout_before_the_device():
    v = np.zeros((2, 2, 4, 9), np.float32)
    for call in (change.change_detection_pol, lambda v, n, pol: change.omnibus_probability_pol(v, n, pol)):
        args = (lambda v, n, pol: (v, 0.5, n, pol)) if call is change.change_detection_pol else (lambda v, n, pol: (v, n, pol))
        with pytest.raises(ValueError, match="unknown covariance layout"):
            call(*args(v, 9, 'quadpol'))
        with pytest.raises(ValueError, match="n >= 3"):
            call(*args(v, 2, 'quad'))
        with pytest.raises(ValueError, match="n >= 1"):
            call(*args(v[..., :1], 0, 'single'))
        with pytest.raises(ValueError, match=r"\(rows, cols, time, 2\)"):
            call(*args(v, 9, 'dual_diagonal'))
        with pytest.raises(ValueError, match=r"\(rows, cols, time, 9\)"):
            call(*args(v[..., :4], 9, 'quad'))


def test_compute_path_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    for pol in LAYOUTS + ['dual']:
        v = series(2, 2, 4, 4, [1, 1, 1, 1], pol)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            change.change_detection_pol(v, 0.5, 4, pol)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            change.omnibus_probability_pol(v, 4, pol)


def test_interface_defaults_unchanged_and_pol_keyword_only():
    sig = inspect.signature(change.OmnibusTest.__init__).parameters
    assert [sig[k].default for k in ('ml', 'n', 'alpha')] == [None, 1, 0.01]
    assert sig['pol'].kind is inspect.Parameter.KEYWORD_ONLY and sig['pol'].default is None
    assert change.OmnibusTest().pol is None and change.OmnibusTest(pol='quad').pol == 'quad'
    assert 'pol' in inspect.signature(change.omnibus).parameters
    assert list(inspect.signature(change.change_detection_pol).parameters) == ['values', 'alpha', 'n', 'pol']
    assert change.POLS['dual'] == ['C11', 'C12__re', 'C12__im', 'C22']


def test_dataset_errors_before_the_device():
    ds = generate_test_dataset(dims={'y': 4, 'x': 4, 'time': 5})                      # C11, C12, C22 only
    with pytest.raises(ValueError, match="missing: C13__re, C13__im, C23__re, C23__im, C33"):
        change.OmnibusTest(n=9, pol='quad').apply(ds)
    with pytest.raises(ValueError, match="missing: C33"):
        change.omnibus(ds, n=9, pol='quad_diagonal')
    with pytest.raises(ValueError, match="unknown covariance layout"):
        change.OmnibusTest(n=9, pol='hh').apply(ds)
    with pytest.raises(ValueError, match="n >= 3"):
        change.OmnibusTest(n=1, pol='quad').apply(ds)


# ---- CPU: the generalised oracle -----------------------------------------------------------------------
def test_oracle_dual_matches_the_pinned_restatement():
    from oracle import omnibus_oracle as oo
    from oracle import omnibus_pol_oracle as po
    for k, looks in [(2, 4), (5, 9), (12, 16), (30, 50)]:
        v = series(4, 5, k, looks, 1.0 + 0.3 * np.sin(np.arange(k)), 'dual', seed=k)
        got = po.omnibus_probability_pol(v, looks, 'dual')
        ref = np.array([[oo.single_pixel_omnibus(v[i, j], looks) for j in range(5)] for i in range(4)])
        assert np.abs(got - ref).max() < 1e-13, k


def test_oracle_walk_is_the_pinned_walk():
    """The layout oracle's walk with the reference's dual-pol statistic gives the pinned restatement's change maps."""
    from oracle import omnibus_oracle as oo
    from oracle import omnibus_pol_oracle as po
    rng = np.random.default_rng(7)
    for k, looks, alpha in [(10, 9, 0.9), (16, 4, 0.999), (7, 25, 0.5)]:
        scales = np.exp(np.cumsum(rng.choice([0.0, 0.0, 1.2, -1.0], size=k)))
        for dtype in (np.float64, np.float32):
            v = series(4, 5, k, looks, scales, 'dual', seed=k, dtype=dtype)
            want = oo.change_detection(v, alpha, looks)
            assert want.sum() > 0 and np.array_equal(po.change_detection(v, alpha, looks), want)


def test_oracle_identities():
    from oracle import omnibus_pol_oracle as po
    for k, looks in [(3, 4), (8, 16)]:
        scales = 1.0 + 0.5 * np.cos(np.arange(k))
        for pol, p in [('dual_diagonal', 2), ('quad_diagonal', 3)]:
            v = series(5, 6, k, looks, scales, pol, seed=k + p)
            z_single = sum(po.pol_z(v[..., b:b + 1], looks, 'single') for b in range(p))
            assert np.allclose(po.pol_z(v, looks, pol), z_single, rtol=1e-12, atol=1e-9)
        # single is the diagonal statistic of one band: the full formulas at p = 1 give the per-band f, rho, omega2
        f, rho, om = po.pol_constants(k, looks, 'single')
        fd, rhod, omd = po.pol_constants(k, looks, 'dual_diagonal')
        assert f == fd / 2 and rho == rhod and abs(om - omd / 2) < 1e-15
        # quad with zero off-diagonals has the lnQ of quad_diagonal
        q = series(5, 6, k, looks, scales, 'quad_diagonal', seed=k)
        full = np.zeros(q.shape[:-1] + (9,))
        full[..., [0, 5, 8]] = q
        assert np.allclose(po.pol_lnQ(full, looks, 'quad'), po.pol_lnQ(q, looks, 'quad_diagonal'), rtol=1e-13, atol=1e-10)


def test_oracle_probability_is_uniform_under_h0():
    """H0 (no change), k = 5, n = 16, 40 000 pixels, seed 0 (full layouts: a correlated Sigma; diagonal layouts:
    unequal powers).  KS distance of P to U(0, 1), against the 0.1 % critical value 1.95 / sqrt(40 000) = 0.00975:
    dual 0.0040, single 0.0035, quad 0.0044, dual_diagonal 0.0040, quad_diagonal 0.0053.  Wrong constants are
    caught: for quad_diagonal (seed 1, without omega2), rho = 1 gives 0.0122 and the full-p rho 0.0604."""
    from scipy.stats import kstest
    from oracle import omnibus_pol_oracle as po
    rng = np.random.default_rng(0)
    for pol in ['dual'] + LAYOUTS:
        c = covariances((40000,), 16, [1.0] * 5, P[pol], rng, diagonal=pol.endswith('diagonal'))
        prob = po.omnibus_probability_pol(bands(c, pol), 16, pol)
        d = kstest(prob, 'uniform').statistic
        assert d < 1.95 / np.sqrt(40000), (pol, d)


@pytest.mark.parametrize("pol", LAYOUTS)
def test_oracle_detects_a_step_change_and_nothing_else(pol):
    from oracle import omnibus_pol_oracle as po
    v = series(2, 3, 10, 9, [1.0] * 5 + [10.0] * 5, pol, seed=1)
    res = po.change_detection_pol(v, 0.9999, 9, pol)
    assert res[:, :, 5].all() and (res.sum(-1) == 1).all()
    flat = series(2, 3, 10, 9, [1.0] * 10, pol, seed=2)
    assert po.change_detection_pol(flat, 0.9999, 9, pol).sum() == 0


# ---- GPU ------------------------------------------------------------------------------------------------
TOL = {np.float64: 1e-12, np.float32: 1.2e-7}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("pol,k,looks", [(pol, k, looks) for pol in LAYOUTS for k, looks in [(2, 4), (5, 9), (12, 16), (30, 50)]]
                         + [('quad', 64, 25)])                                   # the largest gamma shape: f/2 = 283.5
def test_probability_matches_oracle(pol, k, looks, dtype):
    from oracle import omnibus_pol_oracle as po
    scales = 1.0 + 0.3 * np.sin(np.arange(k))
    v = series(6, 7, k, looks, scales, pol, seed=k, dtype=dtype)
    got = change.omnibus_probability_pol(v, looks, pol)
    ref = po.omnibus_probability_pol(v, looks, pol)
    assert got.dtype == dtype and got.shape == (6, 7)
    assert np.abs(got.astype(np.float64) - ref.astype(np.float64)).max() <= TOL[dtype]
    assert np.isfinite(ref).all() and 0.0 < np.median(ref) <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("pol", LAYOUTS)
def test_change_maps_equal_oracle(pol, dtype):
    from oracle import omnibus_pol_oracle as po
    rng = np.random.default_rng(5)
    for k, looks, alpha in [(10, 9, 0.9), (10, 9, 0.99), (16, 4, 0.999), (7, 25, 0.5)]:
        scales = np.exp(np.cumsum(rng.choice([0.0, 0.0, 0.0, 1.2, -1.0], size=k)))      # a few jumps per series
        v = series(8, 9, k, looks, scales, pol, seed=k + looks, dtype=dtype)
        got = change.change_detection_pol(v, alpha, looks, pol)
        ref = po.change_detection_pol(v, alpha, looks, pol)
        assert got.dtype == np.uint8 and got.shape == (8, 9, k)
        assert np.array_equal(got, ref), (k, looks, alpha, int((got != ref).sum()))
        assert ref.sum() > 0


@pytest.mark.gpu
def test_dual_through_the_layout_entry_is_the_reference_path():
    z = np.load(os.path.join(ROOT, "tests", "golden", "change_golden.npz"))
    meta = json.loads(str(z["__meta__"]))
    for name, m in meta.items():
        v = z[name + "__in"]
        got = change.change_detection_pol(v, m["alpha"], m["n"], 'dual')
        assert np.array_equal(got, z[name + "__change"]) and np.array_equal(got, change.change_detection(v, m["alpha"], m["n"]))
        prob = change.omnibus_probability_pol(v, m["n"], 'dual')
        assert np.array_equal(prob, change.omnibus_probability(v, n=m["n"])), name


@pytest.mark.gpu
@pytest.mark.parametrize("pol", ['quad', 'dual_diagonal'])
def test_strided_input_nan_and_zero_pixels(pol):
    from oracle import omnibus_pol_oracle as po
    v = series(5, 6, 8, 9, [1, 1, 1, 6, 6, 6, 6, 6], pol, seed=3)
    want = po.change_detection_pol(v, 0.99, 9, pol)
    assert want.sum() > 0
    view = np.moveaxis(np.ascontiguousarray(np.moveaxis(v, -1, 0)), 0, -1)        # variable-major, like `to_array()`
    assert not view.flags['C_CONTIGUOUS']
    assert np.array_equal(change.change_detection_pol(view, 0.99, 9, pol), want)
    v[1, 2, 3, 0] = np.nan                                                       # NaN: comparisons are false
    v[3, 4] = 0.0                                                                # all-zero pixel: log 0 - log 0 = NaN
    got = change.change_detection_pol(v, 0.99, 9, pol)
    assert np.array_equal(got, po.change_detection_pol(v, 0.99, 9, pol))
    assert got[1, 2].sum() == 0 and got[3, 4].sum() == 0
    prob = change.omnibus_probability_pol(v, 9, pol)
    assert np.isnan(prob[1, 2]) and np.isnan(prob[3, 4])


def quad_dataset(k=10, step=5, seed=0, shape=(6, 7)):
    """A quad-pol Dataset with complex C12 / C13 / C23 over (y, x, time), scene power x10 from `step` on."""
    rng = np.random.default_rng(seed)
    c = covariances(shape, 9, [1.0] * step + [10.0] * (k - step), 3, rng)
    ref = generate_test_dataset(dims={'y': shape[0], 'x': shape[1], 'time': k}, var=())
    ds = Dataset(coords=ref.coords, attrs=ref.attrs)
    for i in range(3):
        for j in range(i, 3):
            x = c[..., i, j] if i != j else c[..., i, j].real
            ds['C%d%d' % (i + 1, j + 1)] = (('y', 'x', 'time'), np.ascontiguousarray(x))
    return ds


@pytest.mark.gpu
def test_datasets():
    ds = quad_dataset()
    changes = change.OmnibusTest(n=9, alpha=0.9999, pol='quad').apply(ds)
    assert isinstance(changes, DataArray) and changes.name == 'change' and changes.dims == ('y', 'x', 'time')
    assert changes.dtype == bool and changes.isel(time=5).all() and (changes.sum(dim='time') == 1).all()
    assert list(changes.coords) == list(ds.coords) and dict(changes.attrs) == dict(ds.attrs)
    same = change.omnibus(ds, n=9, alpha=0.9999, pol='quad')
    assert np.array_equal(same.values, changes.values)
    ml = change.OmnibusTest(ml=3, alpha=0.9, pol='quad').apply(ds)              # multilooking: n = 9 x 9 looks
    assert ml.values.shape == changes.values.shape and ml.isel(time=5).all()
    # intensity only: a dataset holding nothing but C11 / C22
    di = Dataset(coords=ds.coords, attrs=ds.attrs)
    di['C11'], di['C22'] = ds['C11'], ds['C22']
    got = change.OmnibusTest(n=9, alpha=0.9999, pol='dual_diagonal').apply(di)
    assert got.isel(time=5).all() and (got.sum(dim='time') == 1).all()
    with pytest.raises(ValueError, match="missing: C33"):
        change.omnibus(di, n=9, pol='quad_diagonal')
    # the default stays dual-pol even when the dataset also holds C13 / C23 / C33
    assert np.array_equal(change.OmnibusTest(n=9, alpha=0.99).apply(ds).values,
                          change.OmnibusTest(n=9, alpha=0.99, pol='dual').apply(ds).values)
