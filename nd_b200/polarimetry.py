"""
Polarimetric decomposition of covariance time series on the GPU: the Cloude-Pottier H / A / alpha eigen-decomposition
(Cloude & Pottier, IEEE TGRS 35(1), 1997) of quad-pol data and Cloude's dual-pol H / alpha (IEEE GRSL 4(2), 2007).
`h_a_alpha` works on a (rows, cols, k, bands) array, `HAAlphaDecomposition` / `h_a_alpha_decomposition` on a Dataset.

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
