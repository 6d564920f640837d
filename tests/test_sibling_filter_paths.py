"""
Every CUDA kernel of the sibling filters (nd_b200/csrc/ndflt.cu, ndflt_tiled.cuh) on its interior fast path and at
its tile seams, bit for bit against scipy.ndimage (DESIGN.md §10).

`KERNELS` is the table of the kernel instantiations the library holds, written from the template ranges of ndflt.cu.
  * CPU: the table equals the `ndflt::` functions in the built libndnlm.so, so a kernel added without a case here
    fails without a GPU.
  * GPU, one case per table entry: an input that reaches that instantiation equals scipy, and the instantiation's
    name is among the CUDA kernels the profiler recorded.
  * GPU, per kernel family: lengths that are not multiples of the tile, tail tiles, idle threads, extents on which no
    thread is interior, origins at both limits, every mode with a non-zero cval, nearly symmetric weights, footprint
    holes, weights at DBL_EPSILON, strided device tensors.  Every case also checks which family ran.
  * GPU: BoxcarFilter / GaussianFilter on a 256 x 300 x 24 raster, and 64-bit index arithmetic on a tensor of more
    than 2**32 elements.
The bar is np.array_equal in the data's own dtype: the kernels restate scipy's C loops operation by operation.
"""
import os
import re
import shutil
import subprocess
import zlib

import numpy as np
import pytest
import scipy.ndimage as sn

from nd_b200 import _ndimage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "nd_b200", "libndnlm.so")
MODES = ("reflect", "constant", "nearest", "mirror", "wrap")
CVAL = -1.25
FOOTPRINTS_2D = ((3, 3), (3, 5), (5, 3), (5, 5), (7, 7))
DBL_EPS = np.finfo(np.float64).eps


# ---- the table -----------------------------------------------------------------------------------------
def _k(name, *args):
    return "ndflt::%s<%s>" % (name, ",".join(str(a) for a in args))


_T = ("float", "double")
KERNELS = sorted(
    [_k("correlate_1d_slide_kernel", t, sym, s1, 32) for t in _T for sym in (-1, 1) for s1 in range(1, 9)]
    + [_k("correlate_1d_rows_smem_kernel", t, sym, s1) for t in _T for sym in (-1, 1) for s1 in range(1, 9)]
    + [_k("correlate_1d_rows_smem_kernel", t, sym, 0) for t in _T for sym in (-1, 0, 1)]
    + [_k("correlate_1d_rows_kernel", t, sym, 4) for t in _T for sym in (-1, 0, 1)]
    + [_k("correlate_1d_tiled_kernel", t, sym) for t in _T for sym in (-1, 0, 1)]
    + [_k("correlate_1d_kernel", t, sym) for t in _T for sym in (-1, 0, 1)]
    + [_k("correlate_2d_slide_kernel", t, kh, kw, 16) for t in _T for kh, kw in FOOTPRINTS_2D]
    + [_k("correlate_3d_slide_kernel", t, 3, 3, 3, 8) for t in _T]
    + [_k("correlate_nd_tiled_kernel", t) for t in _T]
    + [_k("correlate_nd_kernel", t) for t in _T])


def _normalise(name):
    """'void ndflt::f<float, (int)-1, 4>(ndflt::TileGeom, ...)' -> 'ndflt::f<float,-1,4>'.  cu++filt writes
    `(int)-1`, the profiler's demangler `-1`."""
    name = name.replace("(int)", "").replace(" ", "")
    if name.startswith("void"):
        name = name[len("void"):]
    return name.split("(", 1)[0]


def _parse(entry):
    m = re.fullmatch(r"ndflt::(\w+)<(.*)>", entry)
    args = m.group(2).split(",")
    return m.group(1), (np.float32 if args[0] == "float" else np.float64), [int(a) for a in args[1:]]


def _cuda_tool(name):
    """`name` from the directory of the nvcc that __graft_entry__.build() compiles with."""
    nvcc = shutil.which(os.environ.get("NVCC", "nvcc"))
    if nvcc is None:
        nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    path = os.path.join(os.path.dirname(os.path.realpath(nvcc)), name)
    assert os.path.exists(path), "%s not found next to %s" % (name, nvcc)
    return path


def test_kernel_table_equals_the_functions_in_the_library():
    sass = subprocess.run([_cuda_tool("cuobjdump"), "-sass", LIB], capture_output=True, text=True, check=True).stdout
    mangled = [m.group(1) for m in re.finditer(r"Function : (\S+)", sass)]
    demangled = subprocess.run([_cuda_tool("cu++filt")], input="\n".join(mangled), capture_output=True, text=True,
                               check=True).stdout.splitlines()
    names = sorted(_normalise(n) for n in demangled if "ndflt::" in n)
    assert len(KERNELS) == 104 and len(set(KERNELS)) == 104
    assert names == KERNELS, (sorted(set(names) - set(KERNELS)), sorted(set(KERNELS) - set(names)))


# ---- helpers -------------------------------------------------------------------------------------------
def _rand(shape, dtype, seed):
    return np.random.default_rng(seed).normal(size=shape).astype(dtype)


def _sym_weights(rng, s1, sym, nearly=False):
    """2 s1 + 1 weights, symmetric (sym = 1) or antisymmetric (sym = -1) around an arbitrary centre.  `nearly`: each
    right weight is the next double above its left partner, which scipy's |w_r -+ w_l| <= DBL_EPSILON test still
    calls (anti)symmetric; the arithmetic then uses the left weights only."""
    left = rng.uniform(0.05, 1.0, s1)
    right = np.nextafter(left, 2.0) if nearly else left
    return np.concatenate([left, [rng.uniform(-1.0, 1.0)], sym * right[::-1]])


def _host(family, fn, a, *args, **kw):
    """A case: the _ndimage host function against scipy's function of the same name and arguments."""
    kw.setdefault("cval", CVAL)
    label = "%s %s %s %s %s" % (fn, a.shape, a.dtype, ["%d taps" % np.size(x) if isinstance(x, np.ndarray) else x
                                                      for x in args], {k: v for k, v in kw.items() if k != "cval"})
    return (label, family, lambda: getattr(_ndimage, fn)(a, *args, **kw), lambda: getattr(sn, fn)(a, *args, **kw))


def _device(family, fn, t_in, t_out, *args):
    """A case on CUDA tensors with arbitrary strides (the `*_device` functions); scipy gets the same strided array."""
    label = "%s_device %s strides %s -> %s %s" % (fn, tuple(t_in.shape), t_in.stride(), t_out.stride(), args[1:])

    def run():
        getattr(_ndimage, fn + "_device")(t_in, t_out, *args)
        return t_out.cpu().numpy()

    def ref():
        a = t_in.cpu().numpy()
        if fn == "correlate1d":
            w, axis, origin, mode, cval = args
            return sn.correlate1d(a, w, axis=axis, origin=origin, mode=mode, cval=cval)
        w, origins, mode, cval = args
        return sn.correlate(a, w, origin=origins, mode=mode, cval=cval)
    return label, family, run, ref


def _launched(run):
    """Run `run()` under torch.profiler; returns its result and the normalised names of the ndflt kernels the GPU
    ran.  The kernels come from libndnlm.so, which carries its own static CUDA runtime; CUPTI records kernel
    activity below the runtime, so the profiler sees them like torch's own kernels."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        result = run()
        torch.cuda.synchronize()
    return result, {_normalise(e.name) for e in prof.events() if "ndflt::" in e.name}


def _assert_case(case):
    label, family, run, ref = case
    got, names = _launched(run)
    want = ref()
    assert got.dtype == want.dtype and np.array_equal(got, want), (label, int(np.sum(got != want)), got.size)
    assert any(n.startswith("ndflt::%s<" % family) for n in names), (label, family, sorted(names))


# ---- one case per table entry --------------------------------------------------------------------------
def _table_case(entry):
    family, dtype, p = _parse(entry)
    rng = np.random.default_rng(zlib.crc32(entry.encode()))
    a2 = _rand((100, 40), dtype, 1)
    if family == "correlate_1d_slide_kernel":
        return _host(family, "correlate1d", a2, _sym_weights(rng, p[1], p[0]), axis=0)
    if family == "correlate_1d_rows_smem_kernel":
        w = _sym_weights(rng, p[1] or 12, p[0]) if p[0] else rng.uniform(-1, 1, 10)
        return _host(family, "correlate1d", _rand((30, 300), dtype, 2), w, axis=1)
    if family == "correlate_1d_rows_kernel":
        w = _sym_weights(rng, 65, p[0]) if p[0] else rng.uniform(-1, 1, 130)
        return _host(family, "correlate1d", _rand((20, 150), dtype, 3), w, axis=1)
    if family == "correlate_1d_tiled_kernel":
        w = _sym_weights(rng, 10, p[0]) if p[0] else rng.uniform(-1, 1, 17)
        return _host(family, "correlate1d", a2, w, axis=0)
    if family == "correlate_1d_kernel":
        w = _sym_weights(rng, 512, p[0]) if p[0] else rng.uniform(-1, 1, 1025)
        return _host(family, "correlate1d", a2, w, axis=0)
    if family == "correlate_2d_slide_kernel":
        return _host(family, "correlate", _rand((50, 40), dtype, 4), rng.uniform(-1, 1, (p[0], p[1])))
    if family == "correlate_3d_slide_kernel":
        return _host(family, "correlate", _rand((20, 12, 10), dtype, 5), rng.uniform(-1, 1, (3, 3, 3)))
    if family == "correlate_nd_tiled_kernel":
        return _host(family, "correlate", _rand((40, 30), dtype, 6), rng.uniform(-1, 1, (9, 9)))
    assert family == "correlate_nd_kernel"
    return _host(family, "correlate", _rand((12, 10, 16), dtype, 7), rng.uniform(-1, 1, (5, 7, 11)))


@pytest.mark.gpu
@pytest.mark.parametrize("entry", KERNELS)
def test_each_kernel_instantiation_launches_and_equals_scipy(entry):
    label, family, run, ref = _table_case(entry)
    got, names = _launched(run)
    want = ref()
    assert got.dtype == want.dtype and np.array_equal(got, want), label
    assert entry in names, (label, sorted(names))


# ---- per-family geometry --------------------------------------------------------------------------------
def _slide_cases(dtype):
    """Symmetric / antisymmetric, half-width 1..8, along a slow axis: 32 consecutive rows per thread."""
    fam, rng = "correlate_1d_slide_kernel", np.random.default_rng(10)
    big = _rand((203, 300), dtype, 11)            # 203 rows = 6 x 32 + 11; 300 = 256 + a 44-wide tail tile
    rp2 = _rand((203, 9, 11), dtype, 12)          # inner 99: RP = 2, 58 threads of the CTA idle
    rp21 = _rand((7, 203, 12), dtype, 13)         # along axis 1, outer 7, inner 12: RP = 21
    for s1 in range(1, 9):
        for sym in (1, -1):
            w = _sym_weights(rng, s1, sym)
            for origin in (-s1, 0, s1):
                yield _host(fam, "correlate1d", big, w, axis=0, origin=origin, mode=MODES[(s1 + origin) % 5])
            yield _host(fam, "correlate1d", rp2, w, axis=0, origin=-s1, mode=MODES[s1 % 5])
            yield _host(fam, "correlate1d", rp21, w, axis=1, origin=s1, mode=MODES[(s1 + 2) % 5])
            # 31 + 2 s1 rows: fewer than 32 + 2 s1, so no thread takes the interior variant
            yield _host(fam, "correlate1d", _rand((31 + 2 * s1, 33), dtype, s1), w, axis=0, origin=-s1,
                        mode=MODES[(s1 + 3) % 5])
            yield _host(fam, "correlate1d", big, _sym_weights(rng, s1, sym, nearly=True), axis=0)
    for s1 in (1, 8):
        for sym in (1, -1):
            w = _sym_weights(rng, s1, sym)
            for mode in MODES:
                for origin in (-s1, 0, s1):
                    yield _host(fam, "correlate1d", big, w, axis=0, origin=origin, mode=mode)


def _rows_smem_cases(dtype):
    """Last axis, up to 129 taps: LN lines x CW <= 256 positions per CTA, staged in shared memory."""
    fam, rng = "correlate_1d_rows_smem_kernel", np.random.default_rng(20)
    lines = [_rand((13, 600), dtype, 21),         # column tiles 256 / 256 / 88; 13 lines = 8 + 5 (LN = 8)
             _rand((13, 256), dtype, 22),         # exactly one column tile
             _rand((4, 25, 24), dtype, 23)]       # a time axis: 100 lines, LN = 85 (or 32 at 129 taps)
    for s1 in range(1, 9):
        for sym in (1, -1):
            w = _sym_weights(rng, s1, sym)
            for k, a in enumerate(lines):
                origin = (-s1, 0, s1)[(s1 + k) % 3]
                yield _host(fam, "correlate1d", a, w, axis=-1, origin=origin, mode=MODES[(s1 + k) % 5])
    kernels = [_sym_weights(rng, 12, 1), _sym_weights(rng, 12, -1),      # half-width > 8: <T, +-1, 0>
               _sym_weights(rng, 12, 1, nearly=True), rng.uniform(-1, 1, 10),
               _sym_weights(rng, 64, 1), _sym_weights(rng, 64, -1), rng.uniform(-1, 1, 129)]
    for w in kernels:
        for k, a in enumerate(lines):
            for origin in (-(len(w) // 2), (len(w) - 1) // 2):
                yield _host(fam, "correlate1d", a, w, axis=-1, origin=origin, mode=MODES[(len(w) + k + origin) % 5])
    for w in kernels[-3:]:                        # 129 taps on 24-long lines: repeated reflection
        for mode in MODES:
            yield _host(fam, "correlate1d", lines[2], w, axis=-1, mode=mode)


def _rows_cases(dtype):
    """Last axis, 130..1024 taps: flat thread order, U = 4 outputs per thread."""
    fam, rng = "correlate_1d_rows_kernel", np.random.default_rng(30)
    arrays = [_rand((7, 300), dtype, 31),         # 2100 elements, not a multiple of 1024
              _rand((11, 100), dtype, 32)]        # lines shorter than every kernel here
    kernels = [_sym_weights(rng, 65, 1), _sym_weights(rng, 65, -1), rng.uniform(-1, 1, 130), rng.uniform(-1, 1, 1024)]
    for w in kernels:
        for k, a in enumerate(arrays):
            for origin in (-(len(w) // 2), 0, (len(w) - 1) // 2):
                yield _host(fam, "correlate1d", a, w, axis=1, origin=origin, mode=MODES[(k + origin) % 5])
    for mode in MODES:
        yield _host(fam, "correlate1d", arrays[1], kernels[0], axis=1, mode=mode)
    yield _host(fam, "correlate1d", arrays[0], _sym_weights(rng, 65, -1, nearly=True), axis=1)


def _tiled_1d_cases(dtype):
    """Slow axis, kernels the register window does not take (half-width > 8, or not symmetric)."""
    fam, rng = "correlate_1d_tiled_kernel", np.random.default_rng(40)
    arrays = [(_rand((203, 300), dtype, 41), 0),  # RP = 1, tail tile
              (_rand((203, 9, 11), dtype, 42), 0),  # RP = 2
              (_rand((20, 203, 12), dtype, 43), 1)]  # along x of a (y, x, t) cube: RP = 21
    for k, (a, axis) in enumerate(arrays):
        for sigma in (2.5, 3.0, 8.0):
            for order in (0, 1):
                yield _host(fam, "gaussian_filter1d", a, sigma, axis=axis, order=order, mode=MODES[(k + order) % 5])
        for w in (rng.uniform(-1, 1, 4), rng.uniform(-1, 1, 17), _sym_weights(rng, 10, -1, nearly=True)):
            for origin in (-(len(w) // 2), (len(w) - 1) // 2):
                yield _host(fam, "correlate1d", a, w, axis=axis, origin=origin, mode=MODES[(k + len(w)) % 5])
    w = rng.uniform(-1, 1, 1024)
    for origin in (-512, 0, 511):
        yield _host(fam, "correlate1d", _rand((1100, 3), dtype, 44), w, axis=0, origin=origin, mode=MODES[origin % 5])
        yield _host(fam, "correlate1d", arrays[0][0], w, axis=0, origin=origin, mode=MODES[(origin + 1) % 5])
    for mode in MODES:
        yield _host(fam, "gaussian_filter1d", arrays[1][0], 3.0, axis=0, mode=mode)


def _generic_1d_cases(dtype):
    """The stride-generic 1-D kernel: more than 1024 taps, or arrays that are not C-contiguous."""
    import torch
    fam, rng = "correlate_1d_kernel", np.random.default_rng(50)
    kernels = [_sym_weights(rng, 512, 1), _sym_weights(rng, 512, -1), rng.uniform(-1, 1, 1025)]
    for w in kernels:
        for a, axis in ((_rand((1200, 3), dtype, 51), 0), (_rand((4, 1100), dtype, 52), 1)):
            for origin in (-512, 0, 512):
                yield _host(fam, "correlate1d", a, w, axis=axis, origin=origin, mode=MODES[(origin + axis) % 5])
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    t_in = torch.from_numpy(_rand((10, 16, 12), dtype, 53)).cuda().permute(2, 0, 1)     # (12, 10, 16)
    t_out = torch.empty((16, 12, 10), dtype=tdt, device="cuda").permute(1, 2, 0)
    for w in (_sym_weights(rng, 2, 1), _sym_weights(rng, 3, -1), rng.uniform(-1, 1, 6)):
        for axis in range(3):
            origin = (-(len(w) // 2), 0, (len(w) - 1) // 2)[axis]
            yield _device(fam, "correlate1d", t_in, t_out, w, axis, origin, MODES[(axis + len(w)) % 5], CVAL)


def _slide_2d_cases(dtype):
    """Dense KH x KW footprints: the rows along the tiled axis, the columns along one trailing axis."""
    fam, rng = "correlate_2d_slide_kernel", np.random.default_rng(60)
    yx = _rand((50, 37), dtype, 61)               # 50 rows: 16-row blocks at 0, 16, 32, 48
    cube24, cube32 = _rand((50, 20, 24), dtype, 62), _rand((50, 20, 32), dtype, 63)
    yt = _rand((50, 6, 24), dtype, 64)
    four = _rand((2, 50, 20, 8), dtype, 65)       # outer 2
    for kh, kw in FOOTPRINTS_2D:
        k = rng.uniform(-1, 1, (kh, kw))
        yield _host(fam, "correlate", yx, k)
        yield _host(fam, "correlate", cube24, k[:, :, None], mode="wrap")
        yield _host(fam, "correlate", cube32, k[:, :, None], mode="constant")
        yield _host(fam, "correlate", yt, k[:, None, :], mode="mirror")
        yield _host(fam, "correlate", four, k[None, :, :, None], mode="nearest")
        yield _host(fam, "convolve", cube24, k[:, :, None])
        lim_y, lim_x = (-(kh // 2), (kh - 1) // 2), (-(kw // 2), (kw - 1) // 2)
        for i, oy in enumerate(lim_y):
            for j, ox in enumerate(lim_x):
                yield _host(fam, "correlate", cube24, k[:, :, None], origin=(oy, ox, 0), mode=MODES[2 * i + j])
                yield _host(fam, "correlate", yt, k[:, None, :], origin=(oy, 0, ox), mode=MODES[2 * i + j + 1])
        for mode in MODES:
            yield _host(fam, "correlate", yx, k, origin=(lim_y[1], lim_x[0]), mode=mode)
        hole = k.copy()
        hole[kh // 2, 0] = 0.0                    # not dense any more: the tiled N-D kernel
        yield _host("correlate_nd_tiled_kernel", "correlate", cube24, hole[:, :, None], origin=(lim_y[0], lim_x[1], 0))


def _slide_3d_cases(dtype):
    """Dense 3 x 3 x 3 footprints over the tiled axis and two trailing axes."""
    fam, rng = "correlate_3d_slide_kernel", np.random.default_rng(70)
    k = rng.uniform(-1, 1, (3, 3, 3))
    a3, a4 = _rand((70, 50, 32), dtype, 71), _rand((3, 40, 30, 24), dtype, 72)
    for i, (mode, origin) in enumerate(zip(MODES, ((0, 0, 0), (-1, -1, -1), (1, 1, 1), (1, -1, 0), (-1, 1, 1)))):
        yield _host(fam, "correlate", a3, k, origin=origin, mode=mode)
        yield _host(fam, "correlate", a4, k[None], origin=(0,) + origin, mode=MODES[(i + 1) % 5])
    yield _host(fam, "convolve", a3, k)


def _tiled_nd_cases(dtype):
    """Any footprint of at most 384 taps on C-contiguous arrays, tiled around its slowest axis."""
    fam, rng = "correlate_nd_tiled_kernel", np.random.default_rng(80)
    a3 = _rand((20, 18, 16), dtype, 81)
    k7 = rng.uniform(-1, 1, (7, 7, 7))            # 343 taps
    k9 = rng.uniform(-1, 1, (9, 9))
    k384 = rng.uniform(-1, 1, (8, 8, 6))          # exactly 384 taps
    k448 = rng.uniform(-1, 1, (8, 8, 7))          # 64 weights at or below DBL_EPSILON leave 384 taps
    small = np.array([DBL_EPS, -DBL_EPS, DBL_EPS / 2, 0.0, 1e-300, -1e-20, DBL_EPS * (1 - DBL_EPS / 2), -0.0])
    k448.reshape(-1)[rng.permutation(448)[:64]] = np.resize(small, 64)
    for i, mode in enumerate(MODES):
        yield _host(fam, "correlate", a3, k7, origin=((0, 0, 0), (-3, 3, -3), (3, -3, 3))[i % 3], mode=mode)
        yield _host(fam, "correlate", _rand((60, 50), dtype, 82), k9, origin=((-4, 4), (4, -4), (0, 0))[i % 3], mode=mode)
        yield _host(fam, "correlate", a3, k384, origin=((-4, 3, -3), (3, -4, 2), (0, 0, 0))[i % 3], mode=mode)
        yield _host(fam, "correlate", a3, k448, origin=((-4, 3, 0), (3, -4, 3), (0, 0, -3))[i % 3], mode=mode)
    a4 = _rand((6, 7, 8, 9), dtype, 83)
    for k in (rng.uniform(-1, 1, (3, 3, 3, 3)), rng.uniform(-1, 1, (2, 3, 1, 4))):
        for i, mode in enumerate(MODES):
            yield _host(fam, "correlate", a4, k, origin=((0, -1, 0, -1), (-1, 1, 0, 1))[i % 2], mode=mode)
    yield _host(fam, "convolve", a3, k384)


def _generic_nd_cases(dtype):
    """The stride-generic N-D kernel: more than 384 taps, footprints along the last axis only, strided tensors."""
    import torch
    fam, rng = "correlate_nd_kernel", np.random.default_rng(90)
    k385 = rng.uniform(-1, 1, (5, 7, 11))         # 385 taps
    a = _rand((12, 10, 16), dtype, 91)
    for mode, origin in zip(MODES, ((0, 0, 0), (-2, -3, -5), (2, 3, 5), (-2, 3, 0), (1, -1, 4))):
        yield _host(fam, "correlate", a, k385, origin=origin, mode=mode)
    one = _rand((1000,), dtype, 92)               # 1-D arrays
    for mode in MODES:
        yield _host(fam, "correlate", one, rng.uniform(-1, 1, 7), origin=-3, mode=mode)
        yield _host(fam, "correlate", one, rng.uniform(-1, 1, 4), origin=1, mode=mode)
    tdt = torch.float32 if dtype == np.float32 else torch.float64
    t_in = torch.from_numpy(_rand((10, 16, 12), dtype, 93)).cuda().permute(2, 0, 1)     # (12, 10, 16)
    t_out = torch.empty((16, 12, 10), dtype=tdt, device="cuda").permute(1, 2, 0)
    for i, mode in enumerate(MODES):
        yield _device(fam, "correlate", t_in, t_out, rng.uniform(-1, 1, (3, 3, 3)), [(-1, 0, 1), (0, 0, 0)][i % 2],
                      mode, CVAL)
        yield _device(fam, "correlate", t_in, t_out, rng.uniform(-1, 1, (3, 5, 1)), [0, 2, 0], mode, CVAL)


FAMILIES = {"slide": _slide_cases, "rows_smem": _rows_smem_cases, "rows": _rows_cases, "tiled_1d": _tiled_1d_cases,
            "generic_1d": _generic_1d_cases, "slide_2d": _slide_2d_cases, "slide_3d": _slide_3d_cases,
            "tiled_nd": _tiled_nd_cases, "generic_nd": _generic_nd_cases}


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_family_geometry_equals_scipy(family, dtype):
    for case in FAMILIES[family](dtype):
        _assert_case(case)


# ---- Dataset level ---------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_dataset_boxcar_and_gaussian_on_a_raster_equal_scipy(dtype):
    from nd_b200.dataset import generate_test_dataset
    from nd_b200.filters import BoxcarFilter, GaussianFilter
    ds = generate_test_dataset(dims={'y': 256, 'x': 300, 'time': 24}, dtype=dtype)
    for v in ('C11', 'C22'):
        assert ds[v].dims == ('y', 'x', 'time') and ds[v].values.dtype == dtype
    runs = [(BoxcarFilter(('y', 'x'), w=w), lambda a, w=w: sn.convolve(a, np.ones((w, w, 1)) / w ** 2)) for w in (3, 5, 7)]
    runs.append((BoxcarFilter(('y', 'x', 'time'), w=3), lambda a: sn.convolve(a, np.ones((3, 3, 3)) / 27)))
    runs += [(GaussianFilter(('y', 'x', 'time'), sigma=s), lambda a, s=s: sn.gaussian_filter(a, sigma=s))
             for s in (0.7, 1, 2, 3)]
    for flt, ref in runs:
        res = flt.apply(ds)
        for v in ('C11', 'C22'):
            got, want = res[v].values, ref(ds[v].values)
            assert got.dtype == want.dtype and np.array_equal(got, want), (type(flt).__name__, vars(flt), v)


# ---- index arithmetic above 2**32 elements ----------------------------------------------------------------
@pytest.mark.gpu
def test_index_arithmetic_above_2_to_32_elements():
    """(65537, 256, 256) float32 = 4,295,032,832 elements.  Along the last axis with 131 taps the rows kernel divides
    its flat index by the line length in 64 bits; along the last axis of the transposed view the stride-generic
    kernel decomposes its index in 64 bits.  A 1-D pass depends only on its own line, so sampled lines are compared
    with scipy on those lines alone; lines past element 2**32 (the last plane) are always among them."""
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < 40e9:
        pytest.skip("needs 40 GB of free device memory for two 17.2 GB tensors; %.1f GB free" % (free / 1e9))
    rng = np.random.default_rng(2 ** 32)
    w_sym, w_gen = _sym_weights(rng, 65, 1), rng.uniform(-1, 1, 131)
    ii = torch.from_numpy(np.concatenate([[65536] * 8, rng.integers(0, 65537, 56)])).cuda()
    jj = torch.from_numpy(rng.integers(0, 256, 64)).cuda()
    t = out = view = oview = None
    try:
        t = torch.randn((65537, 256, 256), generator=torch.Generator(device="cuda").manual_seed(0), device="cuda")
        out = torch.empty_like(t)
        assert t.numel() > 2 ** 32
        _, names = _launched(lambda: _ndimage.correlate1d_device(t, out, w_sym, 2))
        assert "ndflt::correlate_1d_rows_kernel<float,1,4>" in names, sorted(names)
        lines, got = t[ii, jj].cpu().numpy(), out[ii, jj].cpu().numpy()
        for k in range(64):
            assert np.array_equal(got[k], sn.correlate1d(lines[k], w_sym, mode="reflect")), ("rows", k)
        view, oview = t.transpose(1, 2), out.transpose(1, 2)          # line (i, j) is t[i, :, j]
        _, names = _launched(lambda: _ndimage.correlate1d_device(view, oview, w_gen, 2, 0, "mirror", CVAL))
        assert "ndflt::correlate_1d_kernel<float,0>" in names, sorted(names)
        lines, got = view[ii, jj].cpu().numpy(), oview[ii, jj].cpu().numpy()
        for k in range(64):
            assert np.array_equal(got[k], sn.correlate1d(lines[k], w_gen, mode="mirror", cval=CVAL)), ("generic", k)
    finally:
        del t, out, view, oview
        torch.cuda.empty_cache()
