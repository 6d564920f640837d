#!/usr/bin/env python
"""Timing (GPU) of the Wishart classification (ndchg_wishart_classify, include/ndchg.h) on a 1024 x 1024 x 24 cube of
4-look samples drawn from 4 distinct covariances, for each decomposable layout, float32 and float64, K = 9 and 18.

Initial labels: the H / alpha zones (K = 9); K = 18: the H / A / alpha zones for the quad layouts, and for the dual
layouts the zones split in two by the parity of the sample index (cost only: these centres come in near-equal pairs).
CUDA-event time, best of 7 after a warm-up call; before every timed call the L2 is flushed by writing 256 MB.
`call` is a whole call with max_iter = 10, tol = 0; `pass` = (time with max_iter = 5 - time with max_iter = 0) / the
passes run (each pass: the assign kernel over the cube, the fixed-tree reduction and the one-warp centres kernel).
Bounds of one pass:
  HBM   the algorithmic bytes (the cube read once, the labels read once and written once) at 7.7 TB/s;
  FP64  2 K B + K operations per sample, counted from wishart_assign_kernel (a multiply and an add per class and band,
        one compare per class), at 18.5 T operations/s: the 37 TFLOP/s FP64 of the HGX B200 data sheet (one eighth of
        its eight-GPU figure) counts an FMA as two operations, and the pinned distance has no FMA.
Usage: dev_wishart.py [--out FILE] (default profiles/r9_wishart.txt)."""
import ctypes, os, sys
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np, torch
from nd_b200 import _lib, change, polarimetry
from dev_lee import HBM_BYTES_PER_S, card, timed

FP64_OPS_PER_S = 18.5e12
P = {'dual': 2, 'quad': 3, 'dual_diagonal': 2, 'quad_diagonal': 3}


def cube(rows, cols, k, pol, looks=4, centres=4, seed=0):
    """4-look sample covariances drawn from `centres` random well-conditioned covariances, one time step at a time."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    rng = np.random.default_rng(seed)
    p = P[pol]
    sig = []
    for _ in range(centres):
        a = rng.normal(size=(p, p)) + 1j * rng.normal(size=(p, p))
        sig.append(np.linalg.cholesky(a @ a.conj().T + 0.3 * np.eye(p)))
    chol = torch.tensor(np.array(sig), dtype=torch.complex64, device="cuda")
    out = []
    for t in range(k):
        which = torch.randint(0, centres, (rows, cols), device="cuda", generator=g)
        z = torch.randn((rows, cols, looks, p, 2), device="cuda", generator=g) / 2 ** 0.5
        z = torch.einsum('...lj,...ij->...li', torch.complex(z[..., 0], z[..., 1]), chol[which])
        c = torch.einsum('...li,...lj->...ij', z, z.conj()) / looks
        if pol == 'dual':
            b = [c[..., 0, 0].real, c[..., 0, 1].real, c[..., 0, 1].imag, c[..., 1, 1].real]
        elif pol == 'quad':
            b = [c[..., 0, 0].real, c[..., 0, 1].real, c[..., 0, 1].imag, c[..., 0, 2].real, c[..., 0, 2].imag,
                 c[..., 1, 1].real, c[..., 1, 2].real, c[..., 1, 2].imag, c[..., 2, 2].real]
        else:
            b = [c[..., i, i].real for i in range(p)]
        out.append(torch.stack(b, -1))
    return torch.stack(out, 2)


def run(pol, dtype, K, flush, rows=1024, cols=1024, k=24):
    v = cube(rows, cols, k, pol).to(dtype).contiguous()
    B = v.shape[-1]
    L = _lib.lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    zones = torch.empty(v.shape[:3], dtype=torch.uint8, device="cuda")
    quad = pol.startswith('quad')
    rc = L.ndchg_h_alpha_zones(ctypes.c_void_p(v.data_ptr()), _lib.i64(v.shape[:3]), _lib.i64(v.stride()),
                               0 if dtype == torch.float32 else 1, change._POL_CODES[pol], int(K == 18 and quad),
                               ctypes.c_void_p(zones.data_ptr()), st)
    assert rc == 0, L.ndchg_last_error()
    if K == 18 and not quad:
        parity = (torch.arange(zones.numel(), device="cuda") % 2).to(torch.uint8).view(zones.shape)
        zones = torch.where(zones > 0, zones + 9 * parity, zones)
    labels = torch.empty_like(zones)
    centres = torch.empty((K, B), dtype=torch.float64, device="cuda")
    counts = torch.empty(K, dtype=torch.int64, device="cuda")
    its = torch.empty(1, dtype=torch.int32, device="cuda")
    def call(max_iter):
        labels.copy_(zones)
        rc = L.ndchg_wishart_classify(ctypes.c_void_p(v.data_ptr()), _lib.i64(v.shape[:3]), _lib.i64(v.stride()),
                                      0 if dtype == torch.float32 else 1, change._POL_CODES[pol],
                                      ctypes.c_void_p(labels.data_ptr()), K, max_iter, 0.0, ctypes.c_void_p(centres.data_ptr()),
                                      ctypes.c_void_p(counts.data_ptr()), ctypes.c_void_p(its.data_ptr()), st)
        assert rc == 0, L.ndchg_last_error()
    copy_ms = timed(lambda: labels.copy_(zones), flush)
    t0 = timed(lambda: call(0), flush) - copy_ms
    t5 = timed(lambda: call(5), flush) - copy_ms
    passes = int(its.item())
    t10 = timed(lambda: call(10), flush) - copy_ms
    its10 = int(its.item())
    pass_ms = (t5 - t0) / max(passes, 1)
    samples = rows * cols * k
    nbytes = samples * (B * v.element_size() + 2)
    hbm_ms = nbytes / HBM_BYTES_PER_S * 1e3
    ops = 2 * K * B + K
    fp64_ms = samples * ops / FP64_OPS_PER_S * 1e3
    bound, bound_ms = ("FP64", fp64_ms) if fp64_ms > hbm_ms else ("HBM", hbm_ms)
    line = ("%-13s %s K=%2d %dx%dx%d: pass %7.3f ms (%d passes timed)  call(max_iter=10) %7.3f ms (%2d passes)  "
            "iteration 0 %6.3f ms  %6.1f GB/s  fp64 %3d op/sample %5.2f Top/s  HBM bound %6.3f ms  FP64 bound %6.3f ms  "
            "larger: %s, %5.1f %% of the pass" % (
                pol, str(dtype)[6:], K, rows, cols, k, pass_ms, passes, t10, its10, t0, nbytes / pass_ms / 1e6, ops,
                samples * ops / pass_ms / 1e9, hbm_ms, fp64_ms, bound, 100 * bound_ms / pass_ms))
    print(line, flush=True)
    del v, zones, labels
    torch.cuda.empty_cache()
    return line


if __name__ == "__main__":
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(os.path.dirname(HERE), "profiles", "r9_wishart.txt")
    head = ["# tools/dev_wishart.py on 1 x %s" % card(),
            "# ndchg_wishart_classify on a 1024 x 1024 x 24 cube of 4-look samples from 4 distinct covariances; initial",
            "# labels: the H / alpha zones (K = 9), the H / A / alpha zones (quad, K = 18), the zones split by sample parity",
            "# (dual, K = 18).  CUDA events, best of 7 after a warm-up, L2 flushed (256 MB written) before every timed call.",
            "# pass: (call with max_iter = 5 - call with max_iter = 0) / passes run; iteration 0 includes the one host wait.",
            "# GB/s: cube read once + labels read and written once per pass.  HBM bound: those bytes at 7.7 TB/s.  FP64",
            "# bound: 2 K B + K operations per sample at 18.5 T op/s (HGX B200 data sheet, 37 TFLOP/s FP64 with FMA = 2)."]
    for line in head:
        print(line, flush=True)
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    lines = list(head)
    for pol in ('dual', 'quad', 'dual_diagonal', 'quad_diagonal'):
        for dtype in (torch.float32, torch.float64):
            for K in (9, 18):
                lines.append(run(pol, dtype, K, flush))
    with open(out, "w") as f:
        f.write("\n".join(lines) + "\n")
