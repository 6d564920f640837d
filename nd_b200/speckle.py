"""
Speckle filtering of covariance time series on the GPU: the refined Lee filter (Lee, Grunes & de Grandi, IEEE TGRS
37(5), 1999) for every covariance layout of `change.POLS`.  `refined_lee` works on a (rows, cols, k, bands) array,
`RefinedLeeFilter` / `refined_lee_filter` on a Dataset.

Each pixel's window is split along the edge its span (total power) shows, and every band is filtered with the same
weight over the half-window on the pixel's side of the edge, so an output is a convex combination of the sample and
a local mean and stays a valid covariance matrix.  The computation is pinned in include/ndchg.h
(`ndchg_refined_lee`); the CUDA kernel behind it has no CPU fallback.  The usual order of work is speckle filtering
first, then `change.OmnibusTest`; `looks='auto'` estimates the filter's number of looks with `change.enl_map`.
"""
import ctypes
import numbers

import numpy as np
import torch

from . import _lib
from .algorithm import Algorithm, wrap_algorithm
from .change import POLS, _POL_CODES, _check, _check_layout, _prepare, enl_map
from .dataset import Dataset

__all__ = ['refined_lee', 'RefinedLeeFilter', 'refined_lee_filter']

WINDOWS = (7, 11, 15)
_AUTO_WINDOW = 7                                         # window of the ENL estimate behind looks='auto'


def _check_window(window):
    if isinstance(window, bool) or not isinstance(window, numbers.Integral) or window not in WINDOWS:
        raise ValueError('the window must be 7, 11 or 15 (4 m + 3), got %r' % (window,))


def _check_looks(looks, auto=False):
    if auto and isinstance(looks, str) and looks == 'auto':
        return
    if isinstance(looks, bool) or not isinstance(looks, numbers.Real) or not np.isfinite(looks) or not looks > 0:
        raise ValueError('the number of looks must be a finite number > 0%s, got %r' % (" or 'auto'" if auto else '', looks))


def refined_lee(values, looks, window=7, pol='dual'):
    """Refined Lee filter of every time step of `values` (include/ndchg.h, `ndchg_refined_lee`): `values` is
    (rows, cols, k, bands), float32 or float64, with the bands of `POLS[pol]` in that order; `looks` is the number
    of looks of the data (real, > 0); `window` is 7, 11 or 15 and at most min(rows, cols).  Image edges are
    scipy's 'reflect'.  Returns the filtered array, same shape and dtype."""
    _check_layout(pol)
    _check_window(window)
    _check_looks(looks)
    values = np.asarray(values)
    if values.ndim == 4 and window > min(values.shape[:2]):
        raise ValueError('the window (%d) must not exceed the image (%d x %d)' % (window, values.shape[0], values.shape[1]))
    values, t = _prepare(values, len(POLS[pol]))
    out = torch.empty(values.shape, dtype=t.dtype, device=t.device)
    _check(_lib.lib().ndchg_refined_lee(ctypes.c_void_p(t.data_ptr()), _lib.i64(values.shape[:3]), _lib.i64(t.stride()),
                                        0 if values.dtype == np.float32 else 1, _POL_CODES[pol], int(window), float(looks),
                                        ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out.cpu().numpy()


def _layout(ds, pol, dims):
    """Where each band of `pol` lives in `ds`: a list of (band, variable, part) with part None (a real variable),
    'real' or 'imag' (of a complex variable), and the layout's common dims."""
    found = []
    for band in POLS[pol]:
        if band in ds.data_vars:
            found.append((band, band, None))
            continue
        stem, _, part = band.partition('__')
        if part and stem in ds.data_vars and np.iscomplexobj(ds[stem].values):
            found.append((band, stem, 'real' if part == 're' else 'imag'))
    missing = [b for b in POLS[pol] if b not in [f[0] for f in found]]
    if missing:
        raise ValueError('pol=%r needs the variables %s (complex, or as __re / __im pairs); missing: %s'
                         % (pol, ', '.join(POLS[pol]), ', '.join(missing)))
    var_dims = {ds[v].dims for _, v, _ in found}
    if len(var_dims) != 1:
        raise ValueError('the variables of pol=%r must share their dims, got %s' % (pol, sorted(var_dims)))
    vdims = var_dims.pop()
    if not set(dims) <= set(vdims):
        raise ValueError('the variables of pol=%r have dims %s, which do not include %s' % (pol, vdims, tuple(dims)))
    return found, vdims


class RefinedLeeFilter(Algorithm):
    """
    Refined Lee speckle filter of a covariance time series (`refined_lee`).

    Parameters
    ----------
    dims : tuple of str, optional
        The two image dimensions (default: ('y', 'x')).  Every other dimension of the layout's variables (time,
        none, or several) is filtered one index at a time.
    window : int, optional
        Side of the square window: 7 (the default, Lee et al.'s), 11 or 15; at most the image size.
    looks : float or 'auto', optional
        The number of looks of the data (real, > 0; default 1).  'auto' estimates it as the median of
        `change.enl_map` with a 7 x 7 window over all pixels and steps (not floored), and the result's attrs gain
        'enl'.  The estimate assumes mostly homogeneous scenes of spatially uncorrelated pixels.
    pol : str, optional (keyword only)
        The covariance layout and the variables it reads, as for `change.OmnibusTest` (default 'dual': C11, C12,
        C22).  Complex off-diagonals may be complex variables or `__re` / `__im` pairs.

    `apply(ds)` returns a new Dataset with the same variables, dims, coords and attrs, the layout's variables
    filtered in their own form (complex stays complex, pairs stay pairs) and every other variable copied unchanged.
    """

    def __init__(self, dims=('y', 'x'), window=7, looks=1, *, pol='dual'):
        self.dims = tuple(dims)
        self.window = window
        self.looks = looks
        self.pol = pol

    def apply(self, ds):
        _check_layout(self.pol)
        _check_window(self.window)
        _check_looks(self.looks, auto=True)
        if len(self.dims) != 2 or self.dims[0] == self.dims[1]:
            raise ValueError('dims must name two different dimensions, got %r' % (self.dims,))
        found, vdims = _layout(ds, self.pol, self.dims)
        rest = [d for d in vdims if d not in self.dims]
        order = [vdims.index(d) for d in self.dims + tuple(rest)]
        bands = []
        for _, v, part in found:
            a = ds[v].values
            a = a if part is None else getattr(a, part)
            bands.append(np.transpose(a, order))
        if len({b.dtype for b in bands}) != 1:
            raise ValueError('the variables of pol=%r must share one data type, got %s'
                             % (self.pol, ', '.join(sorted({str(b.dtype) for b in bands}))))
        shape = bands[0].shape
        values = np.stack(bands, -1).reshape(shape[:2] + (-1, len(bands)))
        attrs = dict(ds.attrs)
        looks = self.looks
        if isinstance(looks, str):
            enl = enl_map(values, _AUTO_WINDOW, self.pol)
            looks = float('nan') if np.isnan(enl).all() else float(np.nanmedian(enl))
            if not np.isfinite(looks):
                raise ValueError("looks='auto': the equivalent number of looks could not be estimated from the data "
                                 "(median %r); pass looks explicitly" % (looks,))
            attrs['enl'] = looks
        filtered = refined_lee(values, looks, self.window, self.pol).reshape(shape + (len(bands),))
        inverse = np.argsort(order)
        out = Dataset(coords={k: c.copy() for k, c in ds.coords.items()}, attrs=attrs)
        for name, var in ds.data_vars.items():
            out.data_vars[name] = var.copy(deep=True)
        for b, (_, v, part) in enumerate(found):
            new = np.ascontiguousarray(np.transpose(filtered[..., b], inverse))
            if part is None:
                out[v] = (vdims, new)
            else:
                getattr(out[v].values, part)[...] = new
        return out


refined_lee_filter = wrap_algorithm(RefinedLeeFilter, 'refined_lee_filter')
