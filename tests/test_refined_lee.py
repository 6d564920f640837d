"""
Refined Lee speckle filter (include/ndchg.h, `ndchg_refined_lee`; `speckle.refined_lee`, `RefinedLeeFilter`).

The NumPy oracle (`oracle/refined_lee_oracle.py`) is tied to what the filter must do: constant images and noise-free
horizontal / vertical steps come back bit for bit, full-layout outputs stay positive semidefinite, speckle is
reduced, the two limits of the number of looks give the masked mean and the input, a hand-worked 7 x 7 window pins
the edge and side choice (ties included), and its edge is scipy's 'reflect'.  Every operation of the definition is
one correctly rounded double operation in a stated order, so the CUDA kernel must equal the oracle bit for bit.
"""
import ctypes
import inspect

import numpy as np
import pytest

from nd_b200 import _lib, change, speckle
from nd_b200.dataset import Dataset, generate_test_dataset
from test_change_pol import P, series

POLS = ['dual', 'single', 'quad', 'dual_diagonal', 'quad_diagonal']
FULL = ['dual', 'quad']
WINDOWS = [7, 11, 15]
VP = ctypes.c_void_p


def _oracle():
    from oracle import refined_lee_oracle as ro
    return ro


def _speckle(rows, cols, k, looks, pol, seed=0, scales=None):
    """Homogeneous L-look samples of `pol`: complex Wishart for the full layouts, Gamma intensities otherwise."""
    if pol in FULL:
        return series(rows, cols, k, looks, scales or [1.0] * k, pol, seed=seed)
    rng = np.random.default_rng(seed)
    return rng.gamma(looks, 1.0 / looks, size=(rows, cols, k, P[pol])) * np.array([1.0, 0.3, 0.5])[:P[pol]]


def _diagonal(pol):
    return [change.POLS[pol].index(b) for b in ('C11', 'C22', 'C33') if b in change.POLS[pol]]


# ---- CPU: C ABI and Python boundary --------------------------------------------------------------------
def test_c_abi_checks_arguments_before_the_device():
    L = _lib.lib()
    buf = np.zeros(8192, np.float64)
    out = np.zeros(8192, np.float64)
    def call(shape=(16, 17, 2), dtype=1, pol=0, window=7, looks=4.0, dst=None):
        shape = list(shape)
        strides = [shape[1] * shape[2] * 4, shape[2] * 4, 4, 1]
        dst = out if dst is None else dst
        return L.ndchg_refined_lee(VP(buf.ctypes.data), _lib.i64(shape), _lib.i64(strides), dtype, pol, window, looks,
                                   VP(dst.ctypes.data), None)
    def err():
        return L.ndchg_last_error()
    for pol in (-1, 5, 99):
        assert call(pol=pol) == _lib.EINVAL and b"pol=%d" % pol in err()
    for window in (0, 3, 5, 6, 9, 13, 17, 19):
        assert call(window=window) == _lib.EINVAL and b"must be 7, 11 or 15" in err()
    assert call(window=11, shape=(10, 17, 2)) == _lib.EINVAL and b"must not exceed the image (10 x 17)" in err()
    assert call(window=15, shape=(16, 14, 2)) == _lib.EINVAL and b"must not exceed the image (16 x 14)" in err()
    assert call(shape=(16, 17, 0)) == _lib.EINVAL and b"at least 1 time step" in err()
    for looks in (0.0, -1.0, float('nan'), float('inf'), -float('inf')):
        assert call(looks=looks) == _lib.EINVAL and b"looks must be finite and > 0" in err()
    assert call(dtype=2) == _lib.EDTYPE and b"No matching signature" in err()
    assert call(dst=buf) == _lib.EINVAL and b"must not overlap" in err()
    # the checks come in this order: pol, window, image size, k, looks, dtype
    assert call(pol=7, window=5, looks=0.0, dtype=2) == _lib.EINVAL and b"pol=7" in err()
    assert call(window=9, shape=(16, 17, 0), looks=0.0) == _lib.EINVAL and b"7, 11 or 15" in err()
    assert call(window=15, shape=(8, 17, 0)) == _lib.EINVAL and b"must not exceed" in err()
    assert call(shape=(16, 17, 0), looks=-1.0, dtype=2) == _lib.EINVAL and b"time step" in err()
    assert call(looks=0.0, dtype=2) == _lib.EINVAL and b"looks" in err()
    assert call(dtype=2, dst=buf) == _lib.EDTYPE
    for pol in range(5):                     # valid arguments stop at the host pointer
        for window in (7, 11, 15):
            for dtype in (0, 1):
                assert call(pol=pol, window=window, shape=(15, 17, 1), dtype=dtype, looks=0.5) == _lib.EINVAL
                assert b"out is not a CUDA device pointer" in err()
    assert (out == 0).all() and (buf == 0).all()


def test_python_validates_before_the_device():
    v = np.zeros((16, 17, 2, 4), np.float32)
    with pytest.raises(ValueError, match="unknown covariance layout"):
        speckle.refined_lee(v, 4, 7, 'quadpol')
    for window in (3, 5, 9, 13, 17, 7.0, True, '7'):
        with pytest.raises(ValueError, match="7, 11 or 15"):
            speckle.refined_lee(v, 4, window)
    for looks in (0, -1.5, float('nan'), float('inf'), 'auto', None, True):
        with pytest.raises(ValueError, match="number of looks"):
            speckle.refined_lee(v, looks)
    with pytest.raises(ValueError, match=r"must not exceed the image \(10 x 17\)"):
        speckle.refined_lee(v[:10], 4, 11)
    with pytest.raises(ValueError, match=r"\(rows, cols, time, 2\)"):
        speckle.refined_lee(v, 4, 7, 'dual_diagonal')
    with pytest.raises(TypeError, match="No matching signature"):
        speckle.refined_lee(v.astype(np.int32), 4)
    ds = _dataset(np.ones((16, 17, 3, 4), np.float32), 'dual')
    with pytest.raises(ValueError, match="unknown covariance layout"):
        speckle.RefinedLeeFilter(pol='quadpol').apply(ds)
    with pytest.raises(ValueError, match="needs the variables"):
        speckle.refined_lee_filter(ds, pol='quad')
    with pytest.raises(ValueError, match="7, 11 or 15"):
        speckle.RefinedLeeFilter(window=9).apply(ds)
    with pytest.raises(ValueError, match="number of looks"):
        speckle.RefinedLeeFilter(looks='median').apply(ds)
    with pytest.raises(ValueError, match="do not include"):
        speckle.RefinedLeeFilter(dims=('y', 'z')).apply(ds)
    odd = _dataset(np.ones((16, 17, 3, 4), np.float32), 'dual')
    odd['C22'] = (('x', 'y', 'time'), np.ones((17, 16, 3), np.float32))
    with pytest.raises(ValueError, match="share their dims"):
        speckle.refined_lee_filter(odd)
    mixed = _dataset(np.ones((16, 17, 3, 4), np.float32), 'dual')
    mixed['C22'] = (('y', 'x', 'time'), np.ones((16, 17, 3)))
    with pytest.raises(ValueError, match="share one data type"):
        speckle.refined_lee_filter(mixed)


def test_compute_path_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    v = np.ones((16, 17, 2, 4))
    ds = _dataset(v, 'dual')
    for call in (lambda: speckle.refined_lee(v, 4), lambda: speckle.refined_lee_filter(ds),
                 lambda: speckle.RefinedLeeFilter(looks='auto').apply(ds)):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            call()


def test_signatures():
    assert set(speckle.__all__) == {'refined_lee', 'RefinedLeeFilter', 'refined_lee_filter'}
    sig = inspect.signature(speckle.refined_lee).parameters
    assert list(sig) == ['values', 'looks', 'window', 'pol']
    assert sig['window'].default == 7 and sig['pol'].default == 'dual' and sig['looks'].default is inspect.Parameter.empty
    sig = inspect.signature(speckle.RefinedLeeFilter.__init__).parameters
    assert list(sig) == ['self', 'dims', 'window', 'looks', 'pol']
    assert sig['dims'].default == ('y', 'x') and sig['window'].default == 7 and sig['looks'].default == 1
    assert sig['pol'].kind is inspect.Parameter.KEYWORD_ONLY and sig['pol'].default == 'dual'
    sig = inspect.signature(speckle.refined_lee_filter).parameters
    assert sig['window'].default == 7 and sig['looks'].default == 1 and sig['pol'].default == 'dual' and 'ds' in sig


# ---- CPU: the oracle -----------------------------------------------------------------------------------
@pytest.mark.parametrize("window", WINDOWS)
@pytest.mark.parametrize("pol", POLS)
def test_oracle_constant_image_bitwise(pol, window):
    ro = _oracle()
    v = np.empty((window + 4, window + 6, 2, len(change.POLS[pol])), np.float32)
    v[...] = np.array([2.3, 0.37, -0.11, 0.05, 0.21, 1.7, -0.3, 0.13, 0.9], np.float32)[:v.shape[-1]]
    v[..., _diagonal(pol)] = np.array([2.3, 1.7, 0.9], np.float32)[:P[pol]]
    assert np.array_equal(ro.refined_lee(v, 4.0, window, pol), v)


@pytest.mark.parametrize("window", WINDOWS)
@pytest.mark.parametrize("pol", ['dual', 'quad', 'single'])
def test_oracle_steps_bitwise(pol, window):
    """Noise-free steps along each image axis, at every pixel, borders included."""
    ro = _oracle()
    base = np.array([1.0, 0.2, -0.1, 0.05, 0.3, 0.8, -0.2, 0.1, 0.6], np.float32)[:len(change.POLS[pol])]
    if pol == 'single':
        base = np.array([1.3], np.float32)
    for axis in (0, 1):
        v = np.ones((window + 17, window + 19, 2, base.size), np.float32) * base
        idx = [slice(None)] * 4
        idx[axis] = slice(window + 2, None)
        v[tuple(idx)] *= np.float32(7.5)
        v[:, :, 1] *= np.float32(0.25)
        for looks in (1.0, 4.4):
            assert np.array_equal(ro.refined_lee(v, looks, window, pol), v), (axis, looks)


@pytest.mark.parametrize("pol", POLS)
def test_oracle_keeps_covariances_valid(pol):
    """4-look speckle with a bright block and a step: the full layouts stay positive semidefinite (leading minors
    >= -1e-12 relative), every diagonal stays >= 0."""
    ro = _oracle()
    v = _speckle(40, 44, 2, 4, pol, seed=3)
    v[10:20, 5:15] *= 9.0
    v[:, 30:] *= 3.0
    out = ro.refined_lee(v, 4.0, 7, pol)
    d = _diagonal(pol)
    assert (out[..., d] >= 0).all()
    if pol in FULL:
        c11, c22 = out[..., 0], out[..., d[1]]
        m2 = c11 * c22 - (out[..., 1] ** 2 + out[..., 2] ** 2)
        assert (m2 >= -1e-12 * c11 * c22).all()
    if pol == 'quad':
        c = np.zeros(out.shape[:3] + (3, 3), complex)
        c[..., 0, 0], c[..., 1, 1], c[..., 2, 2] = out[..., 0], out[..., 5], out[..., 8]
        c[..., 0, 1] = out[..., 1] + 1j * out[..., 2]
        c[..., 0, 2] = out[..., 3] + 1j * out[..., 4]
        c[..., 1, 2] = out[..., 6] + 1j * out[..., 7]
        c[..., 1, 0], c[..., 2, 0], c[..., 2, 1] = c[..., 0, 1].conj(), c[..., 0, 2].conj(), c[..., 1, 2].conj()
        m3 = np.linalg.det(c).real
        assert (m3 >= -1e-12 * out[..., 0] * out[..., 5] * out[..., 8]).all()


@pytest.mark.parametrize("pol", POLS)
def test_oracle_reduces_speckle(pol):
    """The span's coefficient of variation on homogeneous 4-look speckle drops to well under half."""
    ro = _oracle()
    v = _speckle(64, 64, 1, 4, pol, seed=11)
    cv = lambda a: ro.span(a, pol).std() / ro.span(a, pol).mean()
    before, after = cv(v), cv(ro.refined_lee(v, 4.0, 7, pol))
    assert after < 0.4 * before, (before, after)


@pytest.mark.parametrize("pol", POLS)
def test_oracle_limits_of_the_looks(pol):
    ro = _oracle()
    v = _speckle(24, 26, 2, 4, pol, seed=5)
    st = ro.statistics(v, 1e-6, 7, pol)                          # var_x <= 0 everywhere: the masked mean
    assert (st['b'] == 0).all()
    assert np.array_equal(ro.refined_lee(v, 1e-6, 7, pol), st['M'])
    st = ro.statistics(v, 1e12, 7, pol)                          # b -> var_y / var_y = 1: the input
    assert (st['var_y'] > 0).all() and np.allclose(st['b'], 1.0, rtol=0, atol=1e-9)
    np.testing.assert_allclose(ro.refined_lee(v, 1e12, 7, pol), v, rtol=1e-8, atol=1e-9)


def test_oracle_hand_worked_window():
    """Single-pol 7 x 7 images, centre pixel (3, 3): s = 3, c = 2, the subwindows are rows / cols 0-2, 2-4, 4-6."""
    ro = _oracle()
    def centre(y, looks=4.0):
        v = np.asarray(y, np.float64)[:, :, None, None]
        m, e, second = ro.selection(v, 7, 'single')
        st = ro.statistics(v, looks, 7, 'single')
        return m[:, :, 3, 3, 0], int(e[3, 3, 0]), bool(second[3, 3, 0]), st, ro.refined_lee(v, looks, 7, 'single')[3, 3, 0, 0]
    # columns 3-6 bright: m_u0 = 1, m_u1 = (3 + 6 * 10) / 9 = 7, m_u2 = 10; G0 = 27 > G2 = G3 = 18 > G1 = 0.
    # |m12 - m11| = 3 < |m10 - m11| = 6: the second (right) half, which is all 10
    y = np.ones((7, 7))
    y[:, 3:] = 10.0
    m, e, second, st, out = centre(y)
    assert np.array_equal(m, [[1, 7, 10]] * 3) and e == 0 and second and out == 10.0
    # one bright sample at (6, 6): m22 = 2, the rest 1; G0 = G1 = G3 = 1 > G2 = 0, and the first maximum (G0) wins;
    # |m12 - m11| = |m10 - m11| = 0: the first (left) half, without the bright sample
    y = np.ones((7, 7))
    y[6, 6] = 10.0
    m, e, second, st, out = centre(y)
    assert m[2, 2] == 2 and (m.ravel()[:8] == 1).all() and e == 0 and not second and out == 1.0
    # the plane y = 7 + dy + dx: G3 = 16 > G0 = G1 = 12 > G2 = 0, e = 3; m00 = 3, m22 = 11, m11 = 7 tie: first mask,
    # dy + dx <= 0, whose 28 samples average 7 - 56 / 28 = 5
    dy, dx = np.mgrid[-3:4, -3:4]
    m, e, second, st, out = centre(7.0 + dy + dx)
    assert e == 3 and not second and st['ybar'][3, 3, 0] == 5.0
    # y = 7 + dy - dx: G2 = 16 wins, e = 2, first mask dy - dx <= 0
    m, e, second, st, out = centre(7.0 + dy - dx)
    assert e == 2 and not second and st['ybar'][3, 3, 0] == 5.0


def test_oracle_reflect_edge():
    """The edge is np.pad(mode='symmetric') = scipy.ndimage's 'reflect': filtering the padded image and cropping
    gives the same bits, and a one-hot correlation with mode='reflect' reads the same samples."""
    from scipy.ndimage import correlate
    ro = _oracle()
    for window in WINDOWS:
        h = window // 2
        v = _speckle(window + 3, window + 5, 2, 4, 'dual', seed=window)
        padded = np.pad(v, ((h, h), (h, h), (0, 0), (0, 0)), mode='symmetric')
        assert np.array_equal(ro.refined_lee(padded, 4.0, window, 'dual')[h:-h, h:-h], ro.refined_lee(v, 4.0, window, 'dual'))
        y = ro.span(v, 'dual')[..., 0]
        yp = np.pad(y, h, mode='symmetric')
        for oy, ox in ((-h, -h), (h, h), (-h, h), (2, -1)):
            k = np.zeros((window, window))
            k[h + oy, h + ox] = 1.0
            assert np.array_equal(correlate(y, k, mode='reflect'), yp[h + oy:h + oy + y.shape[0], h + ox:h + ox + y.shape[1]])


# ---- GPU ------------------------------------------------------------------------------------------------
def _dataset(v, pol, dims=('y', 'x', 'time'), complex_c12=False, extra=False):
    """A Dataset holding the bands of `v` (rows, cols, k, bands) as the variables of `pol` over `dims` (the order
    of 'y', 'x' and 'time'; without 'time', k must be 1); off-diagonals as __re / __im pairs or complex."""
    sizes = {'y': v.shape[0], 'x': v.shape[1], 'time': v.shape[2]}
    ref = generate_test_dataset(dims={d: sizes[d] for d in dims}, var=())
    ds = Dataset(coords=ref.coords, attrs=dict(ref.attrs, source='test'))
    order = [('y', 'x', 'time').index(d) for d in dims]
    for b, name in enumerate(change.POLS[pol]):
        a = np.transpose(v[..., b], order) if 'time' in dims else v[:, :, 0, b]
        ds[name] = (dims, np.ascontiguousarray(a))
    if complex_c12:
        for stem in ('C12', 'C13', 'C23'):
            if stem + '__re' in ds.data_vars:
                ds[stem] = (dims, ds[stem + '__re'].values + 1j * ds[stem + '__im'].values)
                del ds[stem + '__re']
                del ds[stem + '__im']
    if extra:
        ds['mask'] = (dims, np.arange(np.prod([sizes[d] for d in dims])).reshape([sizes[d] for d in dims]) % 3 == 0)
        ds['height'] = (('y', 'x'), np.linspace(0, 1, sizes['y'] * sizes['x']).reshape(sizes['y'], sizes['x']))
    return ds


def _case(pol, shape, seed=0):
    """float32-representable 6-look samples with a bright point target and a step, so float32 and float64 data hold
    the same values."""
    rows, cols, k = shape
    v = series(rows, cols, k, 6, [1.0, 2.0, 0.5][:k] if k <= 3 else [1.0] * k, pol, seed=seed + rows).astype(np.float32)
    v[rows // 2, cols // 3, 0] *= 40.0
    v[:, (2 * cols) // 3:] *= 5.0
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("geometry", ['tiles', 'rows_equal_window', 'cols_equal_window'])
@pytest.mark.parametrize("window", WINDOWS)
@pytest.mark.parametrize("pol", POLS)
def test_kernel_equals_oracle_bitwise(pol, window, geometry):
    ro = _oracle()
    shape = {'tiles': (37, 53, 3), 'rows_equal_window': (window, 19, 1), 'cols_equal_window': (21, window, 2)}[geometry]
    v = _case(pol, shape, seed=window)
    for dtype in (np.float64, np.float32):
        x = v.astype(dtype)
        for looks in (1.0, 4.4):
            got = speckle.refined_lee(x, looks, window, pol)
            want = ro.refined_lee(x, looks, window, pol)
            assert got.dtype == dtype and got.shape == x.shape
            assert np.array_equal(got, want, equal_nan=True), (dtype, looks, np.argwhere(got != want)[:5])


@pytest.mark.gpu
@pytest.mark.parametrize("pol", POLS)
def test_strided_input_bitwise(pol):
    import torch
    v = _case(pol, (37, 53, 4))
    for dtype in (torch.float64, torch.float32):
        t = torch.from_numpy(v).to(dtype).cuda()
        want = speckle.refined_lee(t.cpu().numpy(), 3.0, 11, pol)
        views = [t.permute(3, 0, 1, 2).contiguous().permute(1, 2, 3, 0),          # band-major, like `to_array()`
                 t.permute(2, 0, 1, 3).contiguous().permute(1, 2, 0, 3),          # time-major
                 t.transpose(0, 1).contiguous().transpose(0, 1)]                  # column-major image
        for view in views:
            assert not view.is_contiguous() or pol == 'single'
            out = torch.empty(view.shape, dtype=dtype, device='cuda')
            rc = _lib.lib().ndchg_refined_lee(VP(view.data_ptr()), _lib.i64(view.shape[:3]), _lib.i64(view.stride()),
                                              0 if dtype == torch.float32 else 1, change._POL_CODES[pol], 11, 3.0,
                                              VP(out.data_ptr()), VP(torch.cuda.current_stream().cuda_stream))
            assert rc == 0, _lib.lib().ndchg_last_error()
            assert np.array_equal(out.cpu().numpy(), want, equal_nan=True)


@pytest.mark.gpu
@pytest.mark.parametrize("pol", POLS)
def test_nan_inf_zero_and_constant_samples(pol):
    ro = _oracle()
    v = _case(pol, (37, 53, 5)).astype(np.float64)
    v[5, 6, 0, 0] = np.nan
    v[20, 30, 1, -1] = np.inf
    v[30, 10, 2] = 0.0
    v[0, 52, 2, 0] = -np.inf                                      # in a corner: reflected into the windows
    v[:16, 40:, 3] = np.where(np.isin(np.arange(v.shape[-1]), _diagonal(pol)), 1.0, 0.0)
    v[:, :, 4] = 0.0
    for dtype in (np.float64, np.float32):
        x = v.astype(dtype)
        for window in (7, 15):
            want = ro.refined_lee(x, 2.0, window, pol)
            assert np.isnan(want).any()
            got = speckle.refined_lee(x, 2.0, window, pol)
            assert np.array_equal(got, want, equal_nan=True), (dtype, window)


@pytest.mark.gpu
@pytest.mark.parametrize("window", [7, 15])
def test_large_quad_image_at_tile_seams(window):
    """2048 x 2048 x 3 quad-pol float32: crops of the oracle around tile seams (multiples of 16) agree in their
    interior (a margin of h, where the crop's own reflected edge cannot reach)."""
    ro = _oracle()
    rng = np.random.default_rng(window)
    rows = cols = 2048
    v = rng.gamma(4.0, 0.25, size=(rows, cols, 3, 9)).astype(np.float32)
    v[..., [1, 2, 3, 4, 6, 7]] -= np.float32(1.0)                    # signed off-diagonals
    v[700:900, 1000:1400] *= np.float32(6.0)
    got = speckle.refined_lee(v, 4.0, window, 'quad')
    h = window // 2
    for r0, c0 in ((0, 0), (16 * 43 - 20, 16 * 62 - 20), (880, 1390), (1024 - 24, 2048 - 48), (2048 - 48, 16 * 17 - 9)):
        crop = v[r0:r0 + 48, c0:c0 + 48]
        want = ro.refined_lee(crop, 4.0, window, 'quad')
        assert np.array_equal(got[r0 + h:r0 + 48 - h, c0 + h:c0 + 48 - h], want[h:-h, h:-h]), (r0, c0)


@pytest.mark.gpu
@pytest.mark.parametrize("form", ['pairs', 'complex'])
@pytest.mark.parametrize("dims", [('time', 'y', 'x'), ('y', 'x', 'time'), ('y', 'x')])
@pytest.mark.parametrize("pol", ['dual', 'quad', 'quad_diagonal'])
def test_filter_equals_refined_lee_on_a_dataset(pol, dims, form):
    k = 3 if 'time' in dims else 1
    v = _case(pol, (29, 35, k))
    ds = _dataset(v, pol, dims, complex_c12=form == 'complex', extra=True)
    before = ds.copy(deep=True)
    out = speckle.RefinedLeeFilter(window=11, looks=2.5, pol=pol).apply(ds)
    assert ds.equals(before) and dict(ds.attrs) == dict(before.attrs)
    want = speckle.refined_lee(v, 2.5, 11, pol)
    assert list(out.data_vars) == list(ds.data_vars) and dict(out.attrs) == dict(ds.attrs)
    assert list(out.coords) == list(ds.coords) and all(np.array_equal(out.coords[c], ds.coords[c]) for c in ds.coords)
    for name, var in ds.data_vars.items():
        assert out[name].dims == var.dims and out[name].dtype == var.dtype, name
    for name in ('mask', 'height'):
        assert np.array_equal(out[name].values, ds[name].values)
    order = [dims.index(d) for d in ('y', 'x', 'time') if d in dims]
    for b, band in enumerate(change.POLS[pol]):
        stem, _, part = band.partition('__')
        if form == 'complex' and part:
            got = getattr(out[stem].values, 'real' if part == 're' else 'imag')
        else:
            got = out[band].values
        got = np.transpose(got, order)
        assert np.array_equal(got, want[..., b] if 'time' in dims else want[:, :, 0, b]), band
    same = speckle.refined_lee_filter(ds, window=11, looks=2.5, pol=pol)
    assert same.equals(out)


@pytest.mark.gpu
def test_filter_with_the_time_dim_in_the_middle_and_two_extra_dims():
    v = _case('dual', (24, 26, 6))
    ref = generate_test_dataset(dims={'y': 24, 'band': 2, 'x': 26, 'time': 3}, var=())
    ds = Dataset(coords=ref.coords, attrs=ref.attrs)
    for b, name in enumerate(change.POLS['dual']):
        ds[name] = (('y', 'band', 'x', 'time'), np.ascontiguousarray(v[..., b].reshape(24, 26, 2, 3).transpose(0, 2, 1, 3)))
    out = speckle.refined_lee_filter(ds, looks=3.0)
    want = speckle.refined_lee(v, 3.0, 7, 'dual')
    for b, name in enumerate(change.POLS['dual']):
        assert np.array_equal(out[name].values, want[..., b].reshape(24, 26, 2, 3).transpose(0, 2, 1, 3))


@pytest.mark.gpu
@pytest.mark.parametrize("pol", POLS)
def test_auto_looks_equals_the_enl_it_reports(pol):
    v = _case(pol, (40, 44, 3))
    ds = _dataset(v, pol, complex_c12=True)
    auto = speckle.RefinedLeeFilter(looks='auto', pol=pol).apply(ds)
    E = auto.attrs['enl']
    assert isinstance(E, float) and E == float(np.nanmedian(change.enl_map(v, 7, pol)))
    assert {k: a for k, a in auto.attrs.items() if k != 'enl'} == dict(ds.attrs)
    fixed = speckle.RefinedLeeFilter(looks=E, pol=pol).apply(ds)
    assert 'enl' not in fixed.attrs
    for name in ds.data_vars:
        assert np.array_equal(auto[name].values, fixed[name].values), name


@pytest.mark.gpu
def test_auto_looks_needs_an_estimate():
    v = np.zeros((16, 17, 2, 4), np.float32)                     # every det is 0: no ENL
    with pytest.raises(ValueError, match="could not be estimated"):
        speckle.RefinedLeeFilter(looks='auto').apply(_dataset(v, 'dual'))
