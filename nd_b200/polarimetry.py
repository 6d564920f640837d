"""
Polarimetric decomposition of covariance time series on the GPU: the Cloude-Pottier H / A / alpha eigen-decomposition
(Cloude & Pottier, IEEE TGRS 35(1), 1997) of quad-pol data and Cloude's dual-pol H / alpha (IEEE GRSL 4(2), 2007).
`h_a_alpha` works on a (rows, cols, k, bands) array, `HAAlphaDecomposition` / `h_a_alpha_decomposition` on a Dataset.
The unsupervised H / alpha Wishart classification (Lee et al., IEEE TGRS 37(5), 1999) builds on it: `h_alpha_zones`
cuts the H / alpha plane into the Cloude-Pottier zones, and `wishart_classify` / `WishartClassification` /
`wishart_classification` run k-means with the complex Wishart distance from those zones (or from given labels).

Each sample is decomposed on its own: entropy H (how mixed the scattering is), mean alpha angle (surface, then
dipole / volume, then double bounce as alpha rises from 0 to 90 degrees), anisotropy A (quad only) and the ordered
eigenvalues.  Quad layouts decompose the Pauli coherency matrix T of the lexicographic C3 (what SNAP writes); dual
layouts decompose C2 itself.  The definition is pinned in include/ndchg.h (`ndchg_h_a_alpha`); the CUDA kernel behind
it has no CPU fallback.

The decomposition needs multilooked samples: a single-look full-pol sample is rank 1, so its H is 0.  Multilook
first, e.g. with `filters.BoxcarFilter` or `speckle.RefinedLeeFilter` (which keeps every sample a valid covariance).
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .algorithm import Algorithm, wrap_algorithm
from .change import POLS, _POL_CODES, _check, _check_layout, _prepare
from .dataset import Dataset
from .speckle import _layout

__all__ = ['h_a_alpha', 'HAAlphaDecomposition', 'h_a_alpha_decomposition']

# the outputs of each sample, in order, for the quad and the dual layouts
OUTPUTS = {'quad': ['entropy', 'anisotropy', 'alpha', 'lambda1', 'lambda2', 'lambda3'],
           'dual': ['entropy', 'alpha', 'lambda1', 'lambda2']}


def _outputs(pol):
    return OUTPUTS['quad' if pol.startswith('quad') else 'dual']


def _check_decomposable(pol):
    _check_layout(pol)
    if pol == 'single':
        raise ValueError("pol='single' has no H / A / alpha decomposition (a 1 x 1 matrix has no eigenvectors); "
                         "use 'dual', 'quad', 'dual_diagonal' or 'quad_diagonal'")


def h_a_alpha(values, pol='dual'):
    """H / A / alpha decomposition of every sample of `values` (include/ndchg.h, `ndchg_h_a_alpha`): `values` is
    (rows, cols, k, bands), float32 or float64, with the bands of `POLS[pol]` in that order; `pol` is 'dual',
    'quad', 'dual_diagonal' or 'quad_diagonal'.  Returns (rows, cols, k, n) in the data type: quad layouts
    [H, A, alpha, lambda1, lambda2, lambda3], dual layouts [H, alpha, lambda1, lambda2] (`OUTPUTS`), alpha in
    degrees.  NaN for samples with a non-finite band; H, A and alpha are NaN where every eigenvalue is 0."""
    _check_decomposable(pol)
    values = np.asarray(values)
    if values.ndim == 4 and min(values.shape[:3]) < 1:
        raise ValueError('the H / A / alpha decomposition needs at least 1 pixel and 1 time step, got shape %s'
                         % (values.shape,))
    values, t = _prepare(values, len(POLS[pol]))
    out = torch.empty(values.shape[:3] + (len(_outputs(pol)),), dtype=t.dtype, device=t.device)
    _check(_lib.lib().ndchg_h_a_alpha(ctypes.c_void_p(t.data_ptr()), _lib.i64(values.shape[:3]), _lib.i64(t.stride()),
                                      0 if values.dtype == np.float32 else 1, _POL_CODES[pol],
                                      ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return out.cpu().numpy()


class HAAlphaDecomposition(Algorithm):
    """
    H / A / alpha eigen-decomposition of every sample of a covariance time series (`h_a_alpha`).

    Parameters
    ----------
    pol : str, optional (keyword only)
        The covariance layout and the variables it reads, as for `change.OmnibusTest`: 'dual' (the default: C11,
        C12, C22), 'quad' (C11, C12, C13, C22, C23, C33, the lexicographic C3) or the intensity-only
        'dual_diagonal' / 'quad_diagonal'.  Complex off-diagonals may be complex variables or `__re` / `__im`
        pairs.  'single' has no decomposition.

    `apply(ds)` returns a new Dataset with the variables `entropy`, `anisotropy` (quad layouts only), `alpha`
    (degrees), `lambda1`, `lambda2` (and `lambda3`) over the dims of the layout's variables, which may be any dims
    they share, with the input's coords and attrs.  Other variables are not carried over, and the input is not
    modified.  Multilooking is the caller's: chain `filters.BoxcarFilter` or `speckle.RefinedLeeFilter` first;
    single-look full-pol samples are rank 1, so their H is 0.
    """

    def __init__(self, *, pol='dual'):
        self.pol = pol

    def apply(self, ds):
        _check_decomposable(self.pol)
        found, vdims = _layout(ds, self.pol, ())
        bands = []
        for _, v, part in found:
            a = ds[v].values
            bands.append(a if part is None else getattr(a, part))
        if len({b.dtype for b in bands}) != 1:
            raise ValueError('the variables of pol=%r must share one data type, got %s'
                             % (self.pol, ', '.join(sorted({str(b.dtype) for b in bands}))))
        shape = bands[0].shape
        # every sample is decomposed on its own: all dims are flattened into k
        values = np.stack(bands, -1).reshape(1, 1, -1, len(bands))
        result = h_a_alpha(values, self.pol).reshape(shape + (-1,))
        out = Dataset(coords={k: c.copy() for k, c in ds.coords.items()}, attrs=dict(ds.attrs))
        for q, name in enumerate(_outputs(self.pol)):
            out[name] = (vdims, np.ascontiguousarray(result[..., q]))
        return out


h_a_alpha_decomposition = wrap_algorithm(HAAlphaDecomposition, 'h_a_alpha_decomposition')


# the zone initialisations of `wishart_classify` and their number of classes
INITS = {'h_alpha': 9, 'h_a_alpha': 18}
MAX_CLASSES = 32


def _check_samples(values, what):
    values = np.asarray(values)
    if values.ndim == 4 and min(values.shape[:3]) < 1:
        raise ValueError('%s needs at least 1 pixel and 1 time step, got shape %s' % (what, values.shape))
    return values


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _zones_into(t, pol, anisotropy, zones):
    _check(_lib.lib().ndchg_h_alpha_zones(ctypes.c_void_p(t.data_ptr()), _lib.i64(t.shape[:3]), _lib.i64(t.stride()),
                                          0 if t.dtype == torch.float32 else 1, _POL_CODES[pol], int(anisotropy),
                                          ctypes.c_void_p(zones.data_ptr()), _stream()))


def h_alpha_zones(values, pol='dual', anisotropy=False):
    """Cloude-Pottier zone of every sample of `values` (include/ndchg.h, `ndchg_h_alpha_zones`): `values` as for
    `h_a_alpha`.  Returns the uint8 array (rows, cols, k): 1..9 in Lee et al.'s numbering of the H / alpha plane,
    0 where H or alpha is NaN.  `anisotropy=True` (quad layouts only) adds 9 where A > 0.5 (labels 1..18)."""
    _check_decomposable(pol)
    if anisotropy and not pol.startswith('quad'):
        raise ValueError('anisotropy=True needs a quad layout (pol=%r has no A)' % (pol,))
    values, t = _prepare(_check_samples(values, 'h_alpha_zones'), len(POLS[pol]))
    zones = torch.empty(values.shape[:3], dtype=torch.uint8, device=t.device)
    _zones_into(t, pol, anisotropy, zones)
    return zones.cpu().numpy()


def _check_init(init, pol, shape):
    """The number of classes of `init` and, for a label array, the array as uint8."""
    if isinstance(init, str):
        if init not in INITS:
            raise ValueError("init must be 'h_alpha', 'h_a_alpha' or an integer label array, got %r" % (init,))
        if init == 'h_a_alpha' and not pol.startswith('quad'):
            raise ValueError("init='h_a_alpha' needs a quad layout (pol=%r has no A)" % (pol,))
        return INITS[init], None
    init = np.asarray(init)
    if init.dtype.kind not in 'iub':
        raise TypeError('an init label array must be of an integer type, got %s' % init.dtype)
    if init.shape != tuple(shape):
        raise ValueError('the init label array has shape %s, the samples %s' % (init.shape, tuple(shape)))
    lo, hi = (int(init.min()), int(init.max())) if init.size else (0, 0)
    if lo < 0 or not 1 <= hi <= MAX_CLASSES:
        raise ValueError('init labels must lie in [0, %d] with at least one label > 0, got [%d, %d]' % (MAX_CLASSES, lo, hi))
    return hi, init.astype(np.uint8)


def wishart_classify(values, pol='dual', init='h_alpha', max_iter=10, tol=0.0):
    """Unsupervised Wishart classification of every sample of `values` (include/ndchg.h, `ndchg_wishart_classify`):
    k-means with the complex Wishart distance, with one set of class centres for all pixels and dates.  `values` as
    for `h_a_alpha`.  `init` is 'h_alpha' (the 9 zones of `h_alpha_zones`), 'h_a_alpha' (the 18 zones with the
    anisotropy split, quad layouts only) or a (rows, cols, k) integer array of initial labels 0..K (0 = unlabelled;
    K = its maximum, at most 32) for seeded or supervised starts.  The loop runs at most `max_iter` passes and stops
    once at most `tol` of the valid samples change label.

    Returns `(labels, centres, iterations)`: the uint8 labels (rows, cols, k), 0 for invalid samples (a non-finite
    band, or a trace <= 0); the float64 class centres (K, bands), NaN for empty or singular classes; and the number
    of passes run."""
    _check_decomposable(pol)
    values = _check_samples(values, 'the Wishart classification')
    if values.ndim != 4:
        _prepare(values, len(POLS[pol]))                                # raises the shape error
    K, start = _check_init(init, pol, values.shape[:3])
    if not 0 <= int(max_iter) < 2 ** 32:
        raise ValueError('max_iter must be >= 0, got %r' % (max_iter,))
    if not 0.0 <= float(tol) <= 1.0:
        raise ValueError('tol must be in [0, 1], got %r' % (tol,))
    values, t = _prepare(values, len(POLS[pol]))
    if start is None:
        labels = torch.empty(values.shape[:3], dtype=torch.uint8, device=t.device)
        _zones_into(t, pol, init == 'h_a_alpha', labels)
    else:
        labels = torch.from_numpy(np.ascontiguousarray(start)).to(t.device)
    centres = torch.empty((K, len(POLS[pol])), dtype=torch.float64, device=t.device)
    counts = torch.empty(K, dtype=torch.int64, device=t.device)
    iterations = torch.empty(1, dtype=torch.int32, device=t.device)
    _check(_lib.lib().ndchg_wishart_classify(ctypes.c_void_p(t.data_ptr()), _lib.i64(values.shape[:3]), _lib.i64(t.stride()),
                                             0 if values.dtype == np.float32 else 1, _POL_CODES[pol],
                                             ctypes.c_void_p(labels.data_ptr()), K, int(max_iter), float(tol),
                                             ctypes.c_void_p(centres.data_ptr()), ctypes.c_void_p(counts.data_ptr()),
                                             ctypes.c_void_p(iterations.data_ptr()), _stream()))
    return labels.cpu().numpy(), centres.cpu().numpy(), int(iterations.cpu().numpy().view(np.uint32)[0])


class WishartClassification(Algorithm):
    """
    Unsupervised H / alpha Wishart classification of a covariance time series (`wishart_classify`).

    Parameters (keyword only)
    ----------
    pol : str, optional
        The covariance layout and the variables it reads, as for `HAAlphaDecomposition` (default 'dual').
    init : str or array, optional
        'h_alpha' (the default: the 9 Cloude-Pottier zones), 'h_a_alpha' (18 zones, quad layouts only) or an
        integer array of initial labels over the dims of the layout's variables (0 = unlabelled).
    max_iter : int, optional
        The most k-means passes (default 10).
    tol : float, optional
        Stop once at most this fraction of the valid samples changes label (default 0: until no label changes).

    `apply(ds)` returns a new Dataset with the uint8 variable `label` over the dims of the layout's variables (any
    dims they share; every sample is classified against the same centres, so a label means the same on every date),
    the input's coords and attrs, and `attrs['wishart_centres']` (the (K, bands) float64 centres, in the band order
    of `change.POLS[pol]`) and `attrs['wishart_iterations']`.  The input is not modified.  Multilook first, as for
    `HAAlphaDecomposition`.
    """

    def __init__(self, *, pol='dual', init='h_alpha', max_iter=10, tol=0.0):
        self.pol = pol
        self.init = init
        self.max_iter = max_iter
        self.tol = tol

    def apply(self, ds):
        _check_decomposable(self.pol)
        found, vdims = _layout(ds, self.pol, ())
        bands = []
        for _, v, part in found:
            a = ds[v].values
            bands.append(a if part is None else getattr(a, part))
        if len({b.dtype for b in bands}) != 1:
            raise ValueError('the variables of pol=%r must share one data type, got %s'
                             % (self.pol, ', '.join(sorted({str(b.dtype) for b in bands}))))
        shape = bands[0].shape
        init = self.init
        if not isinstance(init, str):
            init = np.asarray(init)
            if init.shape != shape:
                raise ValueError('the init label array has shape %s, the variables %s' % (init.shape, shape))
            init = init.reshape(1, 1, -1)
        values = np.stack(bands, -1).reshape(1, 1, -1, len(bands))
        labels, centres, iterations = wishart_classify(values, self.pol, init, self.max_iter, self.tol)
        out = Dataset(coords={k: c.copy() for k, c in ds.coords.items()}, attrs=dict(ds.attrs))
        out['label'] = (vdims, labels.reshape(shape))
        out.attrs['wishart_centres'] = centres
        out.attrs['wishart_iterations'] = iterations
        return out


wishart_classification = wrap_algorithm(WishartClassification, 'wishart_classification')
