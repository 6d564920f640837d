"""
Change detection, mirroring reference nd/change.py:13-119 (SURVEY.md 8(f) row N4): `ChangeDetection`,
`OmnibusTest(ml, n, alpha).apply(ds)` and the function form `omnibus`.  The tutorial pipeline is
`ds.filter.nlmeans(...)` followed by `ds_nlm.nd.change_omnibus(n=50, alpha=1e-4)` (examples/tutorial_s1.ipynb:133).

Below `_omnibus_change_detection` the reference calls its Cython / GSL extension `_change.change_detection`
(nd/_change.pyx:263-287); here that call goes to the CUDA kernel behind include/ndchg.h (one GPU thread per pixel).
There is no CPU fallback.

Beyond the reference, `pol` selects one of five covariance layouts (`POLS`; include/ndchg.h): dual-pol (the
reference's path, unchanged), single-pol, quad-pol and the intensity-only dual / quad diagonals.  `change_direction`
and `OmnibusTest(..., direction=True)` also say which way each change went (`DIRECTIONS`).  `enl_map`,
`EquivalentLooks` / `equivalent_looks` estimate the equivalent number of looks from the data, and
`OmnibusTest(n='auto')` uses that estimate as the test's number of looks.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .algorithm import Algorithm, wrap_algorithm
from .dataset import DataArray
from .filters import BoxcarFilter, disassemble_complex

__all__ = ['ChangeDetection', 'OmnibusTest', 'omnibus', 'EquivalentLooks', 'equivalent_looks', 'enl_map']

# covariance layout -> the dataset variables stacked on the last axis, in band order
POLS = {
    'dual': ['C11', 'C12__re', 'C12__im', 'C22'],
    'single': ['C11'],
    'quad': ['C11', 'C12__re', 'C12__im', 'C13__re', 'C13__im', 'C22', 'C23__re', 'C23__im', 'C33'],
    'dual_diagonal': ['C11', 'C22'],
    'quad_diagonal': ['C11', 'C22', 'C33'],
}
_POL_CODES = {'dual': 0, 'single': 1, 'quad': 2, 'dual_diagonal': 3, 'quad_diagonal': 4}     # NDCHG_POL_*
_VARS = POLS['dual']
# codes of `change_direction` (NDCHG_DIR_*): the covariance after a change against the mean of the segment before it
DIRECTIONS = {'none': 0, 'increase': 1, 'decrease': 2, 'indefinite': 3}


def _check(rc):
    if rc == 0:
        return
    msg = _lib.lib().ndchg_last_error().decode('utf-8', 'replace')
    if rc == _lib.EDTYPE:
        raise TypeError(msg)
    if rc == _lib.EINVAL:
        raise ValueError(msg)
    raise RuntimeError('ndchg: ' + msg)


def _prepare(values, bands=4):
    values = np.asarray(values)
    if values.ndim != 4 or values.shape[3] != bands:
        raise ValueError('Buffer has wrong number of dimensions (expected (rows, cols, time, %d))' % bands)
    if values.dtype not in (np.float32, np.float64):
        raise TypeError('No matching signature found')
    if not torch.cuda.is_available():
        raise RuntimeError('nd_b200 change detection needs a CUDA device; there is no CPU fallback')
    return values, torch.from_numpy(np.ascontiguousarray(values)).cuda()


def change_detection(values, alpha, n=1, njobs=1):
    """`_change.change_detection(values, alpha, n, njobs)` (nd/_change.pyx:263-287) on the GPU: `values` is
    (rows, cols, time, 4) = [C11, Re C12, Im C12, C22], already multilooked with `n` looks; returns the uint8
    array (rows, cols, time) of detected changes.  `njobs` (OpenMP threads in the reference) is ignored."""
    values, t = _prepare(values)
    res = torch.empty(values.shape[:3], dtype=torch.uint8, device=t.device)
    _check(_lib.lib().ndchg_change_detection(ctypes.c_void_p(t.data_ptr()), _lib.i64(values.shape[:3]), _lib.i64(t.stride()),
                                             0 if values.dtype == np.float32 else 1, ctypes.c_void_p(res.data_ptr()),
                                             float(alpha), int(n), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return res.cpu().numpy()


def omnibus_probability(values, n=1):
    """`single_pixel_omnibus` (nd/_change.pyx:139-160) of every pixel over its whole series."""
    values, t = _prepare(values)
    prob = torch.empty(values.shape[:2], dtype=t.dtype, device=t.device)
    _check(_lib.lib().ndchg_omnibus_probability(ctypes.c_void_p(t.data_ptr()), _lib.i64(values.shape[:3]), _lib.i64(t.stride()),
                                                0 if values.dtype == np.float32 else 1, ctypes.c_void_p(prob.data_ptr()),
                                                int(n), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return prob.cpu().numpy()


def _check_layout(pol):
    if pol not in POLS:
        raise ValueError('unknown covariance layout pol=%r (one of %s)' % (pol, ', '.join(POLS)))


def _check_pol(pol, n):
    _check_layout(pol)
    if n < 1 or (pol == 'quad' and n < 3):
        raise ValueError('pol=%r needs n >= %d looks, got n=%r' % (pol, 3 if pol == 'quad' else 1, n))


def change_detection_pol(values, alpha, n=1, pol='dual'):
    """`change_detection` for the covariance layout `pol` (`POLS`): `values` is (rows, cols, time, bands) with the
    bands of `POLS[pol]` in that order, multilooked with `n` looks (quad-pol needs n >= 3); returns the uint8 array
    (rows, cols, time) of detected changes.  `pol='dual'` is `change_detection`."""
    _check_pol(pol, n)
    values, t = _prepare(values, len(POLS[pol]))
    res = torch.empty(values.shape[:3], dtype=torch.uint8, device=t.device)
    _check(_lib.lib().ndchg_change_detection_pol(ctypes.c_void_p(t.data_ptr()), _lib.i64(values.shape[:3]), _lib.i64(t.stride()),
                                                 0 if values.dtype == np.float32 else 1, _POL_CODES[pol],
                                                 ctypes.c_void_p(res.data_ptr()), float(alpha), int(n),
                                                 ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return res.cpu().numpy()


def omnibus_probability_pol(values, n=1, pol='dual'):
    """`omnibus_probability` for the covariance layout `pol` (see `change_detection_pol`)."""
    _check_pol(pol, n)
    values, t = _prepare(values, len(POLS[pol]))
    prob = torch.empty(values.shape[:2], dtype=t.dtype, device=t.device)
    _check(_lib.lib().ndchg_omnibus_probability_pol(ctypes.c_void_p(t.data_ptr()), _lib.i64(values.shape[:3]), _lib.i64(t.stride()),
                                                    0 if values.dtype == np.float32 else 1, _POL_CODES[pol],
                                                    ctypes.c_void_p(prob.data_ptr()), int(n),
                                                    ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return prob.cpu().numpy()


def change_direction(values, alpha, n=1, pol='dual'):
    """`change_detection_pol` that also classifies every change: returns the uint8 array (rows, cols, time) of
    `DIRECTIONS` codes -- 0 no change, 1 increase (the covariance minus the mean of the segment since the previous
    change is positive definite), 2 decrease (negative definite), 3 indefinite (a mixed change, include/ndchg.h).
    `result != 0` is the change map of `change_detection_pol`; `pol='dual'` walks the reference's dual-pol path."""
    _check_pol(pol, n)
    values, t = _prepare(values, len(POLS[pol]))
    res = torch.empty(values.shape[:3], dtype=torch.uint8, device=t.device)
    _check(_lib.lib().ndchg_change_direction(ctypes.c_void_p(t.data_ptr()), _lib.i64(values.shape[:3]), _lib.i64(t.stride()),
                                             0 if values.dtype == np.float32 else 1, _POL_CODES[pol],
                                             ctypes.c_void_p(res.data_ptr()), float(alpha), int(n),
                                             ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return res.cpu().numpy()


def enl_map(values, window=7, pol='dual'):
    """Equivalent number of looks of every sample (include/ndchg.h, `ndchg_enl`): `values` is (rows, cols, time,
    bands) with the bands of `POLS[pol]`; each time step is estimated over a `window` x `window` neighbourhood (odd,
    3 <= window <= min(rows, cols)).  Returns (rows, cols, time) in the data type: NaN within window // 2 of the
    border and where a window holds a non-finite or non-positive-definite sample, +inf where a window has no
    speckle.  Textured windows bias the estimate low; for a scene ENL take the median over a homogeneous area."""
    _check_layout(pol)
    values = np.asarray(values)
    if isinstance(window, bool) or int(window) != window or window < 3 or window % 2 == 0:
        raise ValueError('the window must be an odd integer >= 3, got %r' % (window,))
    if values.ndim == 4 and window > min(values.shape[:2]):
        raise ValueError('the window (%d) must not exceed the image (%d x %d)' % (window, values.shape[0], values.shape[1]))
    values, t = _prepare(values, len(POLS[pol]))
    enl = torch.empty(values.shape[:3], dtype=t.dtype, device=t.device)
    _check(_lib.lib().ndchg_enl(ctypes.c_void_p(t.data_ptr()), _lib.i64(values.shape[:3]), _lib.i64(t.stride()),
                                0 if values.dtype == np.float32 else 1, _POL_CODES[pol], int(window),
                                ctypes.c_void_p(enl.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return enl.cpu().numpy()


def _stack(ds, pol, ml=None):
    """The variables of layout `pol` (None: the reference's dual-pol variables) as (y, x, time, bands), multilooked
    with an `ml` x `ml` boxcar when `ml` is given."""
    ds_m = ds.copy(deep=True)
    disassemble_complex(ds_m)
    if pol is not None:
        missing = [v for v in POLS[pol] if v not in ds_m.data_vars]
        if missing:
            raise ValueError('pol=%r needs the variables %s (complex, or as __re / __im pairs); missing: %s'
                             % (pol, ', '.join(POLS[pol]), ', '.join(missing)))
    if ml is not None:                                   # multilooking
        ds_m = BoxcarFilter(w=ml).apply(ds_m)
    stack = []
    for v in (_VARS if pol is None else POLS[pol]):
        var = ds_m[v]
        stack.append(np.transpose(var.values, [list(var.dims).index(d) for d in _DIMS]))
    return np.stack(stack, axis=-1)


_DIMS = ('y', 'x', 'time')
_AUTO_WINDOW = 7                                         # window of the ENL estimate behind n='auto'


def _auto_looks(values, pol, ml=None):
    """n='auto': E = the median ENL of `values` over all pixels and steps, times ml**2 when `values` are the data
    before an ml x ml boxcar, and the looks max(floor(E), 1) (3 for quad-pol); the walk takes integer looks.
    With `ml` the estimate is not taken on the multilooked values: neighbouring boxcar outputs share their input
    samples, so a window of them is not N independent samples and the estimator would overstate the looks."""
    enl = enl_map(values, _AUTO_WINDOW, 'dual' if pol is None else pol)
    E = float('nan') if np.isnan(enl).all() else float(np.nanmedian(enl))
    if not np.isfinite(E):
        hint = ("; with ml, single-look data of a full covariance layout have singular samples: leave n out to use "
                "n = ml**2" if ml is not None else "; pass n explicitly")
        raise ValueError("n='auto': the equivalent number of looks could not be estimated from the data (median %r)%s"
                         % (E, hint))
    if ml is not None:
        E *= ml ** 2
    return E, max(int(np.floor(E)), 3 if pol == 'quad' else 1)


class EquivalentLooks(Algorithm):
    """
    Equivalent number of looks of every pixel and time step of a covariance time series (`enl_map`).

    Parameters
    ----------
    window : int, optional
        Side of the square (y, x) window of each estimate, odd and >= 3 (default: 7).
    pol : str, optional (keyword only)
        The covariance layout and the variables it reads, as for `OmnibusTest` (default None: dual-pol C11, C12, C22).

    `apply(ds)` returns a DataArray 'enl' over ('y', 'x', 'time') with the dataset's coords and attrs.  Textured
    areas bias the estimate low: apply it to a homogeneous subset and take the median for a scene ENL.
    """

    def __init__(self, window=7, *, pol=None):
        self.window = window
        self.pol = pol

    def apply(self, ds):
        if self.pol is not None:
            _check_layout(self.pol)
        enl = enl_map(_stack(ds, self.pol), self.window, 'dual' if self.pol is None else self.pol)
        return DataArray(enl, _DIMS, coords={k: c for k, c in ds.coords.items()}, attrs=ds.attrs, name='enl')


equivalent_looks = wrap_algorithm(EquivalentLooks, 'equivalent_looks')


class ChangeDetection(Algorithm):
    njobs = 1

    def __init__(self, njobs=1):
        self.njobs = njobs


def _omnibus_change_detection(ds, alpha=0.01, ml=None, n=1, njobs=1, pol=None, direction=False):
    """Conradsen et al. (2015) omnibus change detection (reference nd/change.py:32-78); `pol` selects the
    covariance layout (`POLS`, None: the reference's dual-pol path); `direction` returns `DIRECTIONS` codes;
    n='auto' estimates the looks of the values the walk reads and records them in the result's attrs."""
    auto = isinstance(n, str)
    if auto and n != 'auto':
        raise ValueError("n must be a number of looks or 'auto', got %r" % (n,))
    if pol is not None:
        if auto:
            _check_layout(pol)
        else:
            _check_pol(pol, ml ** 2 if ml is not None else n)
    values = _stack(ds, pol, ml)
    attrs = ds.attrs
    if auto:
        E, n = _auto_looks(values if ml is None else _stack(ds, pol), pol, ml)
        attrs = dict(ds.attrs, enl=E, looks=n)
    elif ml is not None:
        n = ml ** 2
    dims = _DIMS
    coords = {k: c for k, c in ds.coords.items()}
    if direction:                                        # pol=None: the reference's walk, through the 'dual' entry
        codes = change_direction(values, alpha=alpha, n=n, pol='dual' if pol is None else pol)
        return DataArray(codes, dims, coords=coords, attrs=attrs, name='change_direction')
    if pol is None:
        change = change_detection(values, alpha=alpha, n=n, njobs=njobs)
    else:
        change = change_detection_pol(values, alpha=alpha, n=n, pol=pol)
    return DataArray(np.asarray(change, dtype=bool), dims, coords=coords, attrs=attrs, name='change')


class OmnibusTest(ChangeDetection):
    """
    OmnibusTest (reference nd/change.py:81-116).

    Parameters
    ----------
    ml : int, optional
        Multilooking window size (default: the dataset is already multilooked).
    n : int or 'auto', optional
        The number of looks in `ds`; an integer is ignored if `ml` is given, which uses ml**2 (default: 1).
        'auto' estimates it: E = the median of `enl_map` with a 7 x 7 window over all pixels and steps of `ds`,
        times ml**2 when `ml` is given (the estimate is taken before the boxcar, whose outputs are correlated), then
        n = max(floor(E), 1) (3 for quad-pol); the result's attrs gain 'enl' = E and 'looks' = n.  The estimate
        assumes mostly homogeneous scenes and spatially uncorrelated input pixels: texture biases it low (a
        conservative test); spatially correlated input, e.g. data that were already filtered, biases it high.
    alpha : float (0. ... 1.), optional
        The significance level (default: 0.01).
    pol : str, optional (keyword only)
        The covariance layout and the variables it reads: 'dual' (C11, C12, C22), 'single' (C11), 'quad' (C11,
        C12, C13, C22, C23, C33; needs n >= 3), 'dual_diagonal' (C11, C22) or 'quad_diagonal' (C11, C22, C33).
        Complex off-diagonals may be given as one complex variable or as `__re` / `__im` pairs.  Default None: the
        reference's dual-pol path.
    direction : bool, optional (keyword only)
        If True, `apply` returns uint8 codes named 'change_direction' instead of the boolean 'change': 0 no
        change, 1 increase, 2 decrease, 3 indefinite (`DIRECTIONS`; computed on the multilooked values when `ml`
        is given).  Default False.
    """

    def __init__(self, ml=None, n=1, alpha=0.01, *args, pol=None, direction=False, **kwargs):
        self.ml = ml
        self.n = n
        self.alpha = alpha
        self.pol = pol
        self.direction = direction
        super().__init__(*args, **kwargs)

    def apply(self, ds):
        return _omnibus_change_detection(ds, alpha=self.alpha, ml=self.ml, n=self.n, njobs=self.njobs, pol=self.pol,
                                         direction=self.direction)


omnibus = wrap_algorithm(OmnibusTest, 'omnibus')
