#!/usr/bin/env python
"""Timing (GPU) of the H / A / alpha kernel (ndchg_h_a_alpha, include/ndchg.h) on a 1024 x 1024 x 24 cube of 4-look
samples of each decomposable layout, float32 and float64.

CUDA-event time, best of 7 after a warm-up call; before every timed call the L2 is flushed by writing 256 MB.  GB/s
counts the algorithmic bytes: the cube read once and the outputs written once; "HBM bound" is that traffic at 7.7 TB/s.
FP64 work per sample, counted from the kernel's code (an add, subtract or multiply is one operation; divisions,
square roots, hypot, log and acos are counted apart, since each is a sequence of several instructions):
    dual layouts  27 add/mul, 7 div, 1 hypot, 3 sqrt, 2 log, 2 acos
    quad layouts  49 add/mul, 5 div, 3 sqrt, 3 log, 3 acos; each convergence test 19 add/mul; each plane a sweep
                  visits 1 hypot; each rotation (a plane with T[p][q] != 0) 43 add/mul, 5 div, 2 hypot
The counts of tests, planes and rotations of each cube come from `jacobi`, a NumPy replay of the kernel's sweep loop
on 2^16 of its samples.  Usage: dev_haa.py [--out FILE] (default profiles/r8_h_a_alpha.txt)."""
import ctypes, os, sys
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np, torch
from nd_b200 import _lib, change, polarimetry
from dev_chg import cube
from dev_lee import HBM_BYTES_PER_S, card, timed

EPS2 = np.finfo(np.float64).eps ** 2


def jacobi(values, pol):
    """The kernel's Jacobi loop replayed in NumPy on quad-layout samples (n, bands): returns the number of
    convergence tests, sweeps and rotations of each sample, the eigenvalues (unsorted, unclamped) and |V[0][i]|^2."""
    x = np.asarray(values, np.float64)
    x = np.ldexp(x, -np.frexp(np.abs(x).max(-1, keepdims=True))[1] + 1)          # largest band in [1, 2)
    if pol == 'quad':
        c11, c12, c13, c22, c23, c33 = x[:, 0], x[:, 1] + 1j * x[:, 2], x[:, 3] + 1j * x[:, 4], x[:, 5], x[:, 6] + 1j * x[:, 7], x[:, 8]
    else:
        c11, c22, c33 = x[:, 0], x[:, 1], x[:, 2]
        c12 = c13 = c23 = np.zeros(len(x), complex)
    r2 = np.sqrt(0.5)
    d = np.stack([0.5 * (c11 + 2 * c13.real + c33), 0.5 * (c11 - 2 * c13.real + c33), c22], -1)
    u = np.stack([(c12 - c23.conj()) * r2, (c12 + c23.conj()) * r2, 0.5 * (c11 - c33) - 1j * c13.imag], -1)
    v = np.zeros((len(x), 3), complex)
    v[:, 0] = 1.0
    tests, count, rotations = np.zeros((3, len(x)), np.int64)
    live = np.ones(len(x), bool)
    for _ in range(16):
        tests += live
        off = 2.0 * (np.abs(u) ** 2).sum(-1)
        live &= ~(off <= EPS2 * ((d * d).sum(-1) + off))
        if not live.any():
            break
        count += live
        for P, Q in ((0, 1), (0, 2), (1, 2)):
            R = 3 - P - Q
            m = np.abs(u[:, R])
            go = live & (m > 0)
            rotations += go
            ms = np.where(go, m, 1.0)
            ph = np.conj(u[:, R]) / ms
            theta = (d[:, Q] - d[:, P]) / (2.0 * ms)
            t = np.where(theta >= 0, 1.0, -1.0) / (np.abs(theta) + np.hypot(theta, 1.0))
            t = np.where(go, t, 0.0)
            c = 1.0 / np.hypot(t, 1.0)
            s = t * c
            d[:, P] -= t * m
            d[:, Q] += t * m
            u[:, R] = np.where(go, 0.0, u[:, R])
            rp = np.conj(u[:, Q]) if R > P else u[:, Q]
            rq = np.conj(u[:, P]) if R > Q else u[:, P]
            rot = lambda a, b: (c * a - s * (ph * b), s * a + c * (ph * b))
            rp, rq = rot(rp, rq)
            vp, vq = rot(v[:, P], v[:, Q])
            v[:, P], v[:, Q] = np.where(go, vp, v[:, P]), np.where(go, vq, v[:, Q])
            u[:, Q] = np.where(go, np.conj(rp) if R > P else rp, u[:, Q])
            u[:, P] = np.where(go, np.conj(rq) if R > Q else rq, u[:, P])
    return tests, count, rotations, d, np.abs(v) ** 2


def run(pol, dtype, flush, rows=1024, cols=1024, k=24, looks=4):
    v = cube(rows, cols, k, pol, looks, 'flat').to(dtype).contiguous()
    n_out = len(polarimetry.OUTPUTS['quad' if pol.startswith('quad') else 'dual'])
    out = torch.empty((rows, cols, k, n_out), dtype=dtype, device="cuda")
    L = _lib.lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    def call():
        rc = L.ndchg_h_a_alpha(ctypes.c_void_p(v.data_ptr()), _lib.i64(v.shape[:3]), _lib.i64(v.stride()),
                               0 if dtype == torch.float32 else 1, change._POL_CODES[pol], ctypes.c_void_p(out.data_ptr()), st)
        assert rc == 0, L.ndchg_last_error()
    ms = timed(call, flush)
    samples = rows * cols * k
    nbytes = (v.numel() + out.numel()) * v.element_size()
    hbm_ms = nbytes / HBM_BYTES_PER_S * 1e3
    if pol.startswith('quad'):
        sub = v.reshape(-1, v.shape[-1])[:: samples // 65536][:65536].double().cpu().numpy()
        tests, sw, rot = (float(a.mean()) for a in jacobi(sub, pol)[:3])
        addmul, div, hyp = 49 + 19 * tests + 43 * rot, 5 + 5 * rot, 3 * sw + 2 * rot
    else:
        sw = rot = 0.0
        addmul, div, hyp = 27.0, 7.0, 1.0
    line = ("%-13s %s %dx%dx%d: %8.3f ms  %7.1f Msample/s  %7.1f GB/s  HBM bound %6.3f ms (%5.1f %% of the kernel)"
            "  sweeps %4.2f rotations %4.2f  fp64 per sample %5.1f add/mul + %4.1f div + %4.1f hypot:"
            "  %5.2f Top/s add/mul, %5.3f Tdiv/s" % (
                pol, str(dtype)[6:], rows, cols, k, ms, samples / ms / 1e3, nbytes / ms / 1e6, hbm_ms, 100 * hbm_ms / ms,
                sw, rot, addmul, div, hyp, samples * addmul / ms / 1e9, samples * div / ms / 1e9))
    print(line, flush=True)
    del v, out
    torch.cuda.empty_cache()
    return line


if __name__ == "__main__":
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(os.path.dirname(HERE), "profiles", "r8_h_a_alpha.txt")
    head = ["# tools/dev_haa.py on 1 x %s" % card(),
            "# ndchg_h_a_alpha on a 1024 x 1024 x 24 cube of 4-look stationary samples (unit-power independent channels),",
            "# CUDA events, best of 7 after a warm-up, L2 flushed (256 MB written) before every timed call.",
            "# GB/s: cube read once + outputs written once.  HBM bound: those bytes at 7.7 TB/s.  fp64 work per sample",
            "# counted from the kernel's code (tools/dev_haa.py); sweeps / rotations: means over 2^16 samples of the cube,",
            "# from a NumPy replay of the kernel's Jacobi loop.  Besides: 3 sqrt, 3 log, 3 acos (quad); 3 sqrt, 2 log, 2 acos (dual)."]
    for line in head:
        print(line, flush=True)
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    lines = list(head)
    for pol in ('dual', 'quad', 'dual_diagonal', 'quad_diagonal'):
        for dtype in (torch.float32, torch.float64):
            lines.append(run(pol, dtype, flush))
    with open(out, "w") as f:
        f.write("\n".join(lines) + "\n")
