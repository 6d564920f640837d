"""
Equivalent number of looks (include/ndchg.h, `ndchg_enl`; `change.enl_map`, `EquivalentLooks`, `OmnibusTest(n='auto')`).

The NumPy oracle (`oracle/enl_oracle.py`) is tied to the statistics it states: h(L) = G(L) - G(N L) falls strictly,
the mean of delta over simulated windows of N independent L-look samples is h(L) (checked without the root finder),
and the oracle's median estimate recovers the simulated L.  The CUDA kernel must equal the oracle to 1e-10 (float64)
or 1 float32 ulp, with the same NaN and inf positions; `n='auto'` must equal `n=attrs['looks']` bit for bit.
"""
import ctypes
import functools
import inspect

import numpy as np
import pytest

from nd_b200 import _lib, change
from nd_b200.dataset import DataArray
from test_change_direction import _dataset
from test_change_pol import P, bands, covariances, series

POLS = ['dual', 'single', 'quad', 'dual_diagonal', 'quad_diagonal']
DIAGONAL = ['single', 'dual_diagonal', 'quad_diagonal']
VP = ctypes.c_void_p


def _gamma_series(shape, looks, pol, rng, powers=(1.0, 0.3, 0.5)):
    """Intensities of independent channels with Gamma(looks) speckle (any real `looks`) for the diagonal layouts."""
    p = P[pol]
    return rng.gamma(looks, 1.0 / looks, size=shape + (p,)) * np.asarray(powers)[:p]


# ---- CPU: C ABI and Python boundary --------------------------------------------------------------------
def test_c_abi_checks_arguments_before_the_device():
    L = _lib.lib()
    buf = np.zeros(4096, np.float64)
    out = np.zeros(4096, np.float64)
    def call(shape=(8, 9, 2), dtype=1, pol=0, window=3):
        shape = list(shape)
        strides = [shape[1] * shape[2] * 4, shape[2] * 4, 4, 1]
        return L.ndchg_enl(VP(buf.ctypes.data), _lib.i64(shape), _lib.i64(strides), dtype, pol, window, VP(out.ctypes.data), None)
    for pol in (-1, 5, 99):
        assert call(pol=pol) == _lib.EINVAL and b"pol=%d" % pol in L.ndchg_last_error()
    for window in (0, 1, 2, 4, 8):
        assert call(window=window) == _lib.EINVAL and b"odd and >= 3" in L.ndchg_last_error()
    assert call(window=9) == _lib.EINVAL and b"must not exceed the image (8 x 9)" in L.ndchg_last_error()
    assert call(shape=(9, 8, 2), window=9) == _lib.EINVAL and b"must not exceed the image (9 x 8)" in L.ndchg_last_error()
    assert call(shape=(8, 9, 0)) == _lib.EINVAL and b"at least 1 time step" in L.ndchg_last_error()
    assert call(dtype=2) == _lib.EDTYPE and b"No matching signature" in L.ndchg_last_error()
    for pol in range(5):                     # valid arguments stop at the host pointer
        for window in (3, 7):
            assert call(pol=pol, window=window, shape=(7, 9, 1)) == _lib.EINVAL
            assert b"enl is not a CUDA device pointer" in L.ndchg_last_error()
    assert (out == 0).all()


def test_python_validates_before_the_device():
    v = np.zeros((8, 9, 2, 4), np.float32)
    with pytest.raises(ValueError, match="unknown covariance layout"):
        change.enl_map(v, 3, 'quadpol')
    for window in (2, 4, 1, 3.5, True):
        with pytest.raises(ValueError, match="odd integer >= 3"):
            change.enl_map(v, window)
    with pytest.raises(ValueError, match=r"must not exceed the image \(8 x 9\)"):
        change.enl_map(v, 9)
    with pytest.raises(ValueError, match=r"\(rows, cols, time, 2\)"):
        change.enl_map(v, 3, 'dual_diagonal')
    with pytest.raises(TypeError, match="No matching signature"):
        change.enl_map(v.astype(np.int32), 3)
    ds = _dataset(np.ones((8, 9, 3, 4)), None)
    with pytest.raises(ValueError, match="unknown covariance layout"):
        change.EquivalentLooks(pol='quadpol').apply(ds)
    with pytest.raises(ValueError, match="needs the variables"):
        change.equivalent_looks(ds, pol='quad')
    with pytest.raises(ValueError, match="'auto'"):
        change.OmnibusTest(n='median').apply(ds)
    with pytest.raises(ValueError, match="unknown covariance layout"):
        change.OmnibusTest(n='auto', pol='quadpol').apply(ds)


def test_compute_path_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    ds = _dataset(np.ones((8, 9, 3, 4)), None)
    for call in (lambda: change.enl_map(np.ones((8, 9, 3, 4)), 7), lambda: change.equivalent_looks(ds),
                 lambda: change.OmnibusTest(n='auto').apply(ds)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            call()


def test_signatures():
    assert {'EquivalentLooks', 'equivalent_looks', 'enl_map'} <= set(change.__all__)
    assert list(inspect.signature(change.enl_map).parameters) == ['values', 'window', 'pol']
    assert inspect.signature(change.enl_map).parameters['window'].default == 7
    sig = inspect.signature(change.EquivalentLooks.__init__).parameters
    assert sig['window'].default == 7 and sig['pol'].kind is inspect.Parameter.KEYWORD_ONLY and sig['pol'].default is None
    assert inspect.signature(change.equivalent_looks).parameters['window'].default == 7
    assert inspect.signature(change.OmnibusTest.__init__).parameters['n'].default == 1
    assert change.OmnibusTest(n='auto').n == 'auto'


# ---- CPU: the oracle -----------------------------------------------------------------------------------
@pytest.mark.parametrize("pol", POLS)
def test_h_strictly_decreasing(pol):
    from oracle import enl_oracle as eo
    L = eo.lower(pol) + np.logspace(-3, 6, 400)
    for w in range(3, 16, 2):
        hv = eo.h(L, float(w * w), pol)
        assert (np.diff(hv) < 0).all() and (hv > 0).all(), w
        assert hv[0] > 100 * hv[-1]


@pytest.mark.parametrize("w", [3, 7])
@pytest.mark.parametrize("pol", POLS)
def test_mean_delta_is_h(pol, w):
    """4000 windows of N = w^2 independent samples at L = 12 (diagonal layouts also Gamma L = 4.4): the mean of
    delta is G(L) - G(N L) within 4 standard errors."""
    from oracle import enl_oracle as eo
    from oracle.omnibus_pol_oracle import pol_det
    rng = np.random.default_rng(w + len(pol))
    N, nwin = w * w, 4000
    cases = [(12, bands(covariances((nwin,), 12, [1.0] * N, P[pol], rng, diagonal=pol in DIAGONAL), pol))]
    if pol in DIAGONAL:
        cases.append((4.4, _gamma_series((nwin, N), 4.4, pol, rng)))
    for L, x in cases:
        delta = np.log(pol_det(x.mean(1), pol)) - np.log(pol_det(x, pol)).mean(1)
        se = delta.std(ddof=1) / np.sqrt(nwin)
        assert abs(delta.mean() - eo.h(L, N, pol)) < 4 * se, (L, delta.mean(), eo.h(L, N, pol), se)


@pytest.mark.parametrize("pol", POLS)
def test_oracle_recovers_looks(pol):
    """Median estimate at 128 x 128 x 4 steps, w = 7, within 3 % of L = 4, 12, 50 (and Gamma L = 4.4)."""
    from oracle import enl_oracle as eo
    cases = [(L, series(128, 128, 4, L, [1.0] * 4, pol, seed=L)) for L in (4, 12, 50)]
    if pol in DIAGONAL:
        cases.append((4.4, _gamma_series((128, 128, 4), 4.4, pol, np.random.default_rng(44))))
    for L, v in cases:
        got = np.nanmedian(eo.enl(v, 7, pol))
        assert abs(got / L - 1) < 0.03, (L, got)


@pytest.mark.parametrize("pol", POLS)
def test_oracle_edge_rules(pol):
    from oracle import enl_oracle as eo
    w, r = 5, 2
    v = series(16, 18, 3, 9, [1.0] * 3, pol, seed=2)
    e = eo.enl(v, w, pol)
    border = np.ones((16, 18), bool)
    border[r:16 - r, r:18 - r] = False
    assert np.isnan(e[border]).all() and np.isfinite(e[~border]).all()
    bad = v.copy()
    bad[5, 6, 0, 0] = np.nan                                     # non-finite band
    bad[10, 12, 1] = 0.0                                         # det 0
    bad[8, 3, 2, 0] = -1.0                                       # det < 0 (every layout: C11 < 0, others > 0 ...)
    if pol in ('dual', 'quad'):
        bad[8, 3, 2, 1] = 5.0                                    # ... and |C12|^2 > C11 C22
    e2 = eo.enl(bad, w, pol)
    want = e.copy()
    for (i, j, t) in ((5, 6, 0), (10, 12, 1), (8, 3, 2)):
        win = np.zeros((16, 18), bool)
        win[max(i - r, r):i + r + 1, max(j - r, r):j + r + 1] = True
        win[border] = False
        want[win, t] = np.nan
    assert np.array_equal(np.isnan(e2), np.isnan(want)) and np.array_equal(e2[~np.isnan(e2)], want[~np.isnan(want)])
    const = np.zeros((9, 9, 2, len(change.POLS[pol])))
    const[..., [change.POLS[pol].index(b) for b in ('C11', 'C22', 'C33') if b in change.POLS[pol]]] = 1.0
    c = eo.enl(const, 3, pol)
    assert np.isposinf(c[1:8, 1:8]).all() and np.isnan(c[0]).all()


# ---- GPU ------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _case(pol, w, shape):
    """float32-representable samples (so float32 and float64 data hold the same values) and the oracle's float64 ENL."""
    from oracle import enl_oracle as eo
    rows, cols, k = shape
    v = series(rows, cols, k, 6, [1.0, 2.0, 0.5, 1.0, 3.0][:k], pol, seed=rows + w).astype(np.float32)
    v[rows // 2, cols // 3, 0] *= 40.0                           # a bright point target
    return v, eo.enl(v.astype(np.float64), w, pol)


def _assert_matches(got, want64, dtype):
    assert got.dtype == dtype and got.shape == want64.shape
    want = want64.astype(dtype)
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(np.isinf(got), np.isinf(want))
    f = np.isfinite(want)
    if dtype == np.float64:
        rel = np.abs(got[f] - want[f]) / want[f]
        assert rel.max() <= 1e-10, rel.max()
    else:
        g, x = got[f], want[f]
        assert ((g == x) | (g == np.nextafter(x, np.inf)) | (g == np.nextafter(x, -np.inf))).all()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(37, 53, 5), (300, 520, 2), None])
@pytest.mark.parametrize("w", [3, 7, 11])
@pytest.mark.parametrize("pol", POLS)
def test_kernel_equals_oracle(pol, w, shape):
    shape = shape or (w, w, 1)
    v, want = _case(pol, w, shape)
    assert np.isfinite(want).sum() > 0
    for dtype in (np.float64, np.float32):
        _assert_matches(change.enl_map(v.astype(dtype), w, pol), want, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("pol", POLS)
def test_strided_input_bitwise(pol):
    import torch
    v, _ = _case(pol, 7, (37, 53, 5))
    for dtype in (torch.float64, torch.float32):
        t = torch.from_numpy(v).to(dtype).cuda()
        want = change.enl_map(t.cpu().numpy(), 7, pol)
        views = [t.permute(3, 0, 1, 2).contiguous().permute(1, 2, 3, 0),          # variable-major, like `to_array()`
                 t.repeat_interleave(2, dim=1)[:, ::2],                         # pixel stride of two pixels
                 t.permute(2, 0, 1, 3).contiguous().permute(1, 2, 0, 3)]        # time-major
        for view in views:
            assert not view.is_contiguous() or pol == 'single'
            out = torch.empty(view.shape[:3], dtype=dtype, device='cuda')
            rc = _lib.lib().ndchg_enl(VP(view.data_ptr()), _lib.i64(view.shape[:3]), _lib.i64(view.stride()),
                                      0 if dtype == torch.float32 else 1, change._POL_CODES[pol], 7, VP(out.data_ptr()),
                                      VP(torch.cuda.current_stream().cuda_stream))
            assert rc == 0, _lib.lib().ndchg_last_error()
            got = out.cpu().numpy()
            assert np.array_equal(got, want, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("pol", POLS)
def test_nan_zero_negative_and_constant_pixels(pol):
    from oracle import enl_oracle as eo
    v = _case(pol, 7, (37, 53, 5))[0].astype(np.float64)
    v[5, 6, 0, 0] = np.nan
    v[20, 30, 1, -1] = np.inf
    v[30, 10, 2] = 0.0
    v[12, 40, 3, 0] = -1.0
    v[:16, 40:, 4] = np.where(np.isin(np.arange(v.shape[-1]),
                                      [change.POLS[pol].index(b) for b in ('C11', 'C22', 'C33') if b in change.POLS[pol]]), 1.0, 0.0)
    want = eo.enl(v, 7, pol)
    assert np.isposinf(want[3:13, 43:50, 4]).all() and np.isnan(want[2:9, 3:10, 0]).all()
    for dtype in (np.float64, np.float32):
        _assert_matches(change.enl_map(v.astype(dtype), 7, pol), eo.enl(v.astype(dtype), 7, pol), dtype)


@pytest.mark.gpu
def test_equivalent_looks_dataset():
    v, _ = _case('quad', 7, (37, 53, 5))
    ds = _dataset(v, 'quad')
    enl = change.EquivalentLooks(pol='quad').apply(ds)
    assert isinstance(enl, DataArray) and enl.name == 'enl' and enl.dims == ('y', 'x', 'time')
    assert enl.dtype == np.float32 and list(enl.coords) == list(ds.coords) and dict(enl.attrs) == dict(ds.attrs)
    assert np.array_equal(enl.values, change.enl_map(v, 7, 'quad'), equal_nan=True)
    same = change.equivalent_looks(ds, window=5, pol='quad')
    assert np.array_equal(same.values, change.enl_map(v, 5, 'quad'), equal_nan=True)
    dual = change.equivalent_looks(_dataset(v[..., [0, 1, 2, 5]], None))                 # pol=None: dual-pol
    assert np.array_equal(dual.values, change.enl_map(v[..., [0, 1, 2, 5]], 7, 'dual'), equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("ml", [None, 3])
@pytest.mark.parametrize("direction", [False, True])
@pytest.mark.parametrize("pol", POLS + [None])
def test_auto_equals_the_looks_it_reports(pol, direction, ml):
    v = series(20, 24, 8, 9, [1, 1, 1, 1, 4, 4, 4, 4], 'dual' if pol is None else pol, seed=7)
    ds = _dataset(v, pol)
    auto = change.OmnibusTest(n='auto', ml=ml, alpha=0.99, pol=pol, direction=direction).apply(ds)
    looks, E = auto.attrs['looks'], auto.attrs['enl']
    assert isinstance(looks, int) and looks == max(int(np.floor(E)), 3 if pol == 'quad' else 1)
    seen = change._stack(ds, pol, ml)                                                   # what the walk reads
    raw = float(np.nanmedian(change.enl_map(change._stack(ds, pol), 7, 'dual' if pol is None else pol)))
    assert E == raw * (1 if ml is None else ml ** 2)                                   # with ml: before the boxcar
    fixed = change.OmnibusTest(n=looks, alpha=0.99, pol=pol, direction=direction).apply(
        ds if ml is None else _dataset(seen, pol))
    assert auto.name == fixed.name and auto.dtype == fixed.dtype and np.array_equal(auto.values, fixed.values)
    assert 'looks' not in fixed.attrs and {k: a for k, a in auto.attrs.items() if k not in ('enl', 'looks')} == dict(ds.attrs)
    same = change.omnibus(ds, n='auto', ml=ml, alpha=0.99, pol=pol, direction=direction)
    assert np.array_equal(same.values, auto.values) and same.attrs['looks'] == looks


def test_oracle_overstates_the_looks_of_boxcar_output():
    """Why n='auto' with ml estimates before the boxcar: ml x ml box means of L-look Gamma speckle have ml^2 L looks,
    but neighbouring outputs share input samples, so the estimate on them comes out far too high (an
    anti-conservative test), while ml^2 times the estimate on the input is within 3 %."""
    from scipy.ndimage import uniform_filter
    from oracle import enl_oracle as eo
    rng = np.random.default_rng(8)
    for L, ml in ((1, 3), (4, 3), (1, 5)):
        for pol in ('single', 'dual_diagonal'):
            v = _gamma_series((160, 160, 2), L, pol, rng)
            boxed = uniform_filter(v, size=(ml, ml, 1, 1), mode='constant')[ml // 2:-(ml // 2), ml // 2:-(ml // 2)]
            true = L * ml * ml
            assert np.nanmedian(eo.enl(boxed, 7, pol)) > 1.1 * true, (L, ml, pol)
            assert abs(np.nanmedian(eo.enl(v, 7, pol)) * ml * ml / true - 1) < 0.03, (L, ml, pol)


@pytest.mark.gpu
@pytest.mark.parametrize("pol", ['single', 'dual_diagonal', 'quad_diagonal'])
def test_auto_with_ml_finds_the_looks_of_the_boxcar_output(pol):
    """Gamma speckle with 1 and 4 looks, multilooked with ml = 3 by the test itself: n='auto' gives ml^2 L looks,
    not the far higher estimate a window of correlated box means would give."""
    rng = np.random.default_rng(31)
    for L in (1, 4):
        ds = _dataset(_gamma_series((96, 96, 4), L, pol, rng), pol)
        got = change.OmnibusTest(n='auto', ml=3, alpha=0.99, pol=pol).apply(ds)
        assert abs(got.attrs['looks'] - 9 * L) <= 1 and abs(got.attrs['enl'] / (9 * L) - 1) < 0.03, (L, got.attrs)
        boxed = np.nanmedian(change.enl_map(change._stack(ds, pol, 3), 7, pol))
        assert boxed > 1.1 * 9 * L


@pytest.mark.gpu
def test_auto_end_to_end_gamma_12_5():
    """dual_diagonal intensities with Gamma L = 12.5 speckle, 96 x 64 pixels x 12 steps: rows 0-63 stationary, rows
    64-95 step x3 at t = 6.  n='auto' must find 12 looks and give the change map of n=12; the stationary pixels'
    false-alarm rate of the global test at alpha = 0.99 stays within binomial bounds of 1 %."""
    rng = np.random.default_rng(125)
    k = 12
    power = np.ones((96, 64, k, 1))
    power[64:, :, 6:] = 3.0
    v = _gamma_series((96, 64, k), 12.5, 'dual_diagonal', rng) * power
    ds = _dataset(v, 'dual_diagonal')
    auto = change.OmnibusTest(n='auto', alpha=0.99, pol='dual_diagonal').apply(ds)
    assert auto.attrs['looks'] == 12 and 12.0 <= auto.attrs['enl'] < 13.0, auto.attrs
    fixed = change.OmnibusTest(n=12, alpha=0.99, pol='dual_diagonal').apply(ds)
    assert np.array_equal(auto.values, fixed.values)
    step = auto.values[64:]                             # the walk's marginal test sometimes fires a step late
    assert step.any(-1).all() and step[:, :, 5:8].any(-1).mean() > 0.98
    stationary = v[:61]
    p = change.omnibus_probability_pol(stationary, 12, 'dual_diagonal')
    npix, alpha = p.size, 0.01
    bound = 4 * np.sqrt(alpha * (1 - alpha) / npix)
    assert abs((p > 0.99).mean() - alpha) < bound, ((p > 0.99).mean(), bound)
    assert auto.values[:61].any(-1).mean() <= alpha + bound
