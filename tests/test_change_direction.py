"""
Direction of each detected change (include/ndchg.h, `ndchg_change_direction`): 1 increase, 2 decrease, 3 indefinite,
by the Loewner order of the covariance after the change against the mean of the segment before it.

The NumPy oracle (`oracle/omnibus_direction_oracle.py`, `classify` / `change_direction`) is tied to mathematics that does
not share its code: the classifier against the eigenvalues of random Hermitian matrices, the segment bookkeeping
against a hand-worked series, and the whole against simulated series whose direction is known.  The CUDA post-pass
must give codes identical to the oracle's (every operation is correctly rounded in the same order), and its nonzero
entries must be the change map of the walk, bit for bit.
"""
import ctypes
import inspect
import json
import os

import numpy as np
import pytest

from nd_b200 import _lib, change
from nd_b200.dataset import DataArray, Dataset, generate_test_dataset
from test_change_pol import LAYOUTS, P, ROOT, bands, quad_dataset, series

POLS = ['dual'] + LAYOUTS


def _power_series(rows, cols, powers, looks, pol, seed=0, dtype=np.float64):
    """(rows, cols, k, bands) samples of `pol` from independent complex Gaussian channels whose powers at step t are
    powers[t] (one value per channel); the off-diagonals of the full layouts are sample noise around 0."""
    rng = np.random.default_rng(seed)
    pw = np.asarray(powers, np.float64)[:, :P[pol]]
    k = pw.shape[0]
    w = (rng.normal(size=(rows, cols, k, looks, P[pol])) + 1j * rng.normal(size=(rows, cols, k, looks, P[pol]))) / np.sqrt(2)
    z = w * np.sqrt(pw)[:, None, :]
    c = np.einsum('...li,...lj->...ij', z, z.conj()) / looks
    return bands(c, pol).astype(dtype)


def _oracle_codes(v, alpha, looks, pol):
    """Oracle change map of the layout (pol='dual' / None: the pinned reference walk) and its direction codes."""
    from oracle import omnibus_oracle as oo
    from oracle import omnibus_direction_oracle as do
    from oracle import omnibus_pol_oracle as po
    walk = oo.change_detection(v, alpha, looks) if pol in ('dual', None) else po.change_detection_pol(v, alpha, looks, pol)
    return walk, do.change_direction(v, walk, 'dual' if pol is None else pol)


# ---- CPU: C ABI and Python boundary --------------------------------------------------------------------
def test_c_abi_checks_arguments_like_the_layout_entries():
    L = _lib.lib()
    buf = np.zeros(64, np.float64)
    out = np.zeros(64, np.uint8)
    shape, strides = _lib.i64([2, 2, 4]), _lib.i64([36, 9, 9, 1])
    vp = ctypes.c_void_p
    def call(pol, n):
        return L.ndchg_change_direction(vp(buf.ctypes.data), shape, strides, 1, pol, vp(out.ctypes.data), 0.5, n, None)
    for pol in (-1, 5, 99):
        assert call(pol, 9) == _lib.EINVAL and b"pol=%d" % pol in L.ndchg_last_error()
    assert call(2, 2) == _lib.EINVAL and b"n >= 3" in L.ndchg_last_error()
    assert call(1, 0) == _lib.EINVAL and b"n must be >= 1" in L.ndchg_last_error()
    for pol in range(5):                     # valid arguments pass the layout checks and stop at the host pointer
        assert call(pol, 3) == _lib.EINVAL and b"result is not a CUDA device pointer" in L.ndchg_last_error()
    assert (out == 0).all()


def test_python_validates_before_the_device():
    v = np.zeros((2, 2, 4, 9), np.float32)
    with pytest.raises(ValueError, match="unknown covariance layout"):
        change.change_direction(v, 0.5, 9, 'quadpol')
    with pytest.raises(ValueError, match="n >= 3"):
        change.change_direction(v, 0.5, 2, 'quad')
    with pytest.raises(ValueError, match="n >= 1"):
        change.change_direction(v[..., :1], 0.5, 0, 'single')
    with pytest.raises(ValueError, match=r"\(rows, cols, time, 2\)"):
        change.change_direction(v, 0.5, 9, 'dual_diagonal')
    with pytest.raises(ValueError, match=r"\(rows, cols, time, 4\)"):
        change.change_direction(v, 0.5, 9)
    with pytest.raises(TypeError, match="No matching signature"):
        change.change_direction(v.astype(np.int32), 0.5, 9, 'quad')


def test_compute_path_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    for pol in POLS:
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            change.change_direction(series(2, 2, 4, 4, [1, 1, 1, 1], pol), 0.5, 4, pol)
    ds = generate_test_dataset(dims={'y': 4, 'x': 4, 'time': 5})
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        change.OmnibusTest(n=9, direction=True).apply(ds)


def test_signatures():
    sig = inspect.signature(change.OmnibusTest.__init__).parameters
    assert sig['direction'].kind is inspect.Parameter.KEYWORD_ONLY and sig['direction'].default is False
    assert change.OmnibusTest().direction is False and change.OmnibusTest(direction=True).direction is True
    assert inspect.signature(change.omnibus).parameters['direction'].default is False
    assert list(inspect.signature(change.change_direction).parameters) == ['values', 'alpha', 'n', 'pol']
    assert inspect.signature(change.change_direction).parameters['pol'].default == 'dual'
    assert list(inspect.signature(change.change_detection).parameters) == ['values', 'alpha', 'n', 'njobs']
    assert list(inspect.signature(change.change_detection_pol).parameters) == ['values', 'alpha', 'n', 'pol']
    assert list(inspect.signature(change.omnibus_probability).parameters) == ['values', 'n']
    assert list(inspect.signature(change.omnibus_probability_pol).parameters) == ['values', 'n', 'pol']
    assert change.DIRECTIONS == {'none': 0, 'increase': 1, 'decrease': 2, 'indefinite': 3}


# ---- CPU: the oracle -----------------------------------------------------------------------------------
@pytest.mark.parametrize("pol", POLS)
def test_classifier_agrees_with_eigenvalues(pol):
    """Random Hermitian D = U diag(lam) U^H with |lam| in [0.2, 3] and random signs (diagonal layouts: U = 1)."""
    from oracle import omnibus_direction_oracle as do
    rng = np.random.default_rng(11)
    p, N = P[pol], 4000
    lam = rng.uniform(0.2, 3.0, size=(N, p)) * rng.choice([-1.0, 1.0], size=(N, p))
    lam[: N // 4] = np.abs(lam[: N // 4])                                          # enough definite cases
    lam[N // 4: N // 2] = -np.abs(lam[N // 4: N // 2])
    if pol in ('dual', 'quad'):
        u, _ = np.linalg.qr(rng.normal(size=(N, p, p)) + 1j * rng.normal(size=(N, p, p)))
        D = np.einsum('nij,nj,nkj->nik', u, lam, u.conj())
    else:
        D = np.einsum('nj,jk->njk', lam, np.eye(p)).astype(complex)
    ev = np.linalg.eigvalsh(D)
    codes = do.classify(bands(D, pol), pol)
    assert np.array_equal(codes == 1, (ev > 0).all(-1)) and np.array_equal(codes == 2, (ev < 0).all(-1))
    assert np.array_equal(codes == 3, ~((ev > 0).all(-1) | (ev < 0).all(-1)))
    assert {1, 2} <= set(np.unique(codes)) and (pol == 'single' or 3 in codes)
    assert np.array_equal(do.classify(bands(-D, pol), pol), np.choose(codes, [0, 2, 1, 3]).astype(np.uint8))
    assert (do.classify(np.zeros((3, len(change.POLS[pol]))), pol) == 3).all()
    assert (do.classify(np.full((3, len(change.POLS[pol])), np.nan), pol) == 3).all()


def test_segment_restarts_at_the_last_change():
    """C11 = 1, 1, 1, 100, 100, 50 with changes at 3 and 5: the mean before 5 is 100 (since the change at 3), so 5
    is a decrease; the mean since the series start (40.6) would make it an increase."""
    from oracle import omnibus_direction_oracle as do
    v = np.array([1, 1, 1, 100, 100, 50], np.float64)[None, None, :, None]
    c = np.zeros((1, 1, 6), np.uint8)
    c[0, 0, [3, 5]] = 1
    assert do.change_direction(v, c, 'single')[0, 0].tolist() == [0, 0, 0, 1, 0, 2]


@pytest.mark.parametrize("pol", POLS)
def test_oracle_step_up_and_down(pol):
    for scales, code in (([1.0] * 5 + [10.0] * 5, 1), ([10.0] * 5 + [1.0] * 5, 2)):
        v = series(3, 4, 10, 50, scales, pol, seed=4)
        walk, codes = _oracle_codes(v, 0.9999, 50, pol)
        assert walk[:, :, 5].all() and (codes[:, :, 5] == code).all(), (pol, code)


@pytest.mark.parametrize("pol", ['dual', 'quad', 'dual_diagonal', 'quad_diagonal'])
def test_oracle_exchanged_powers_are_indefinite(pol):
    powers = [[1.0, 0.2, 0.5]] * 5 + [[0.2, 1.0, 0.5]] * 5                        # C11 falls, C22 rises
    v = _power_series(3, 4, powers, 50, pol, seed=6)
    walk, codes = _oracle_codes(v, 0.9999, 50, pol)
    assert walk[:, :, 5].all() and (codes[:, :, 5] == 3).all()


@pytest.mark.parametrize("pol", POLS)
def test_oracle_up_down_up(pol):
    v = series(3, 4, 16, 50, [1.0] * 4 + [10.0] * 4 + [1.0] * 4 + [10.0] * 4, pol, seed=8)
    walk, codes = _oracle_codes(v, 0.9999, 50, pol)
    assert walk[:, :, [4, 8, 12]].all()
    assert (codes[:, :, 4] == 1).all() and (codes[:, :, 8] == 2).all() and (codes[:, :, 12] == 1).all()


@pytest.mark.parametrize("pol", POLS)
def test_oracle_codes_mark_exactly_the_changes(pol):
    rng = np.random.default_rng(2)
    scales = np.exp(np.cumsum(rng.choice([0.0, 0.0, 1.2, -1.0], size=12)))
    v = series(5, 6, 12, 9, scales, pol, seed=3)
    walk, codes = _oracle_codes(v, 0.99, 9, pol)
    assert walk.sum() > 0 and np.array_equal(codes != 0, walk != 0)


# ---- GPU ------------------------------------------------------------------------------------------------
def _dataset(v, pol):
    """A Dataset over (y, x, time) holding the bands of `v` as the variables of `pol` (C12 as __re / __im)."""
    ref = generate_test_dataset(dims={'y': v.shape[0], 'x': v.shape[1], 'time': v.shape[2]}, var=())
    ds = Dataset(coords=ref.coords, attrs=ref.attrs)
    for b, name in enumerate(change.POLS['dual' if pol is None else pol]):
        ds[name] = (('y', 'x', 'time'), np.ascontiguousarray(v[..., b]))
    return ds


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("pol", POLS + [None])
def test_codes_equal_oracle(pol, dtype):
    """The (k, looks, alpha) settings of test_change_pol.py::test_change_maps_equal_oracle, with random multiplicative
    jumps up and down; pol=None goes through OmnibusTest(direction=True)."""
    rng = np.random.default_rng(5)
    seen = set()
    for k, looks, alpha in [(10, 9, 0.9), (10, 9, 0.99), (16, 4, 0.999), (7, 25, 0.5)]:
        scales = np.exp(np.cumsum(rng.choice([0.0, 0.0, 0.0, 1.2, -1.0], size=k)))
        v = series(8, 9, k, looks, scales, 'dual' if pol is None else pol, seed=k + looks, dtype=dtype)
        if pol is None:
            got = change.OmnibusTest(n=looks, alpha=alpha, direction=True).apply(_dataset(v, None)).values
        else:
            got = change.change_direction(v, alpha, looks, pol)
        _, want = _oracle_codes(v, alpha, looks, pol)
        assert got.dtype == np.uint8 and got.shape == (8, 9, k)
        assert np.array_equal(got, want), (k, looks, alpha, int((got != want).sum()))
        seen |= set(np.unique(got).tolist())
    assert {1, 2} <= seen and (pol == 'single' or 3 in seen), seen


@pytest.mark.gpu
def test_pinned_dual_maps():
    from oracle import omnibus_direction_oracle as do
    z = np.load(os.path.join(ROOT, "tests", "golden", "change_golden.npz"))
    meta = json.loads(str(z["__meta__"]))
    for name, m in meta.items():
        v, golden = z[name + "__in"], z[name + "__change"]
        got = change.change_direction(v, m["alpha"], m["n"], 'dual')
        assert np.array_equal(got != 0, golden != 0), name
        assert np.array_equal(got, do.change_direction(v, golden, 'dual')), name


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("pol", POLS)
def test_change_positions_unchanged(pol, dtype):
    rng = np.random.default_rng(9)
    scales = np.exp(np.cumsum(rng.choice([0.0, 0.0, 1.2, -1.0], size=14)))
    v = series(16, 20, 14, 9, scales, pol, seed=1, dtype=dtype)
    got = change.change_direction(v, 0.99, 9, pol)
    walk = change.change_detection_pol(v, 0.99, 9, pol)
    assert walk.sum() > 0 and np.array_equal((got != 0).astype(np.uint8), walk)
    if pol == 'dual':
        assert np.array_equal((got != 0).astype(np.uint8), change.change_detection(v, 0.99, 9))


@pytest.mark.gpu
@pytest.mark.parametrize("pol", POLS)
def test_strided_input_nan_and_zero_pixels(pol):
    v = series(5, 6, 8, 9, [1, 1, 1, 6, 6, 0.5, 0.5, 0.5], pol, seed=3)
    want = change.change_direction(v, 0.99, 9, pol)
    assert want.sum() > 0
    view = np.moveaxis(np.ascontiguousarray(np.moveaxis(v, -1, 0)), 0, -1)        # variable-major, like `to_array()`
    assert view.flags['C_CONTIGUOUS'] == (pol == 'single')
    assert np.array_equal(change.change_direction(view, 0.99, 9, pol), want)
    every_other = np.repeat(v, 2, axis=1)[:, ::2]                                  # pixel stride of two pixels
    assert not every_other.flags['C_CONTIGUOUS']
    assert np.array_equal(change.change_direction(every_other, 0.99, 9, pol), want)
    v[1, 2, 3, 0] = np.nan
    v[3, 4] = 0.0
    got = change.change_direction(v, 0.99, 9, pol)
    assert got[1, 2].sum() == 0 and got[3, 4].sum() == 0
    assert np.array_equal(got, _oracle_codes(v, 0.99, 9, pol)[1])


@pytest.mark.gpu
def test_datasets():
    ds = quad_dataset()
    codes = change.OmnibusTest(n=9, alpha=0.9999, pol='quad', direction=True).apply(ds)
    assert isinstance(codes, DataArray) and codes.name == 'change_direction' and codes.dims == ('y', 'x', 'time')
    assert codes.dtype == np.uint8 and list(codes.coords) == list(ds.coords) and dict(codes.attrs) == dict(ds.attrs)
    assert (codes.isel(time=5).values == 1).all()                                 # the scene gets brighter at t = 5
    boolean = change.OmnibusTest(n=9, alpha=0.9999, pol='quad').apply(ds)
    assert np.array_equal(codes.values != 0, boolean.values)
    same = change.omnibus(ds, n=9, alpha=0.9999, pol='quad', direction=True)
    assert same.name == 'change_direction' and np.array_equal(same.values, codes.values)
    ml = change.OmnibusTest(ml=3, alpha=0.9, pol='quad', direction=True).apply(ds)  # directions of the multilooked data
    assert ml.dtype == np.uint8 and ml.values.shape == codes.values.shape and (ml.isel(time=5).values == 1).all()
    assert np.array_equal(ml.values != 0, change.OmnibusTest(ml=3, alpha=0.9, pol='quad').apply(ds).values)
    # pol=None: the reference's dual-pol walk with the dual classifier
    dual = change.omnibus(ds, n=9, alpha=0.9999, direction=True)
    step = dual.isel(time=5).values                      # at 9 looks the reference walk misses the step in 1 of 42 pixels
    assert dual.name == 'change_direction' and set(np.unique(step)) == {0, 1} and (step == 1).sum() >= 40
    assert np.array_equal(dual.values != 0, change.OmnibusTest(n=9, alpha=0.9999).apply(ds).values)
