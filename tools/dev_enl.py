#!/usr/bin/env python
"""Timing (GPU) of the equivalent-number-of-looks kernel (ndchg_enl, include/ndchg.h) on a 1024 x 1024 x 24 cube of
every covariance layout, float32 and float64, windows 7 and 11, next to the omnibus walk (ndchg_change_detection_pol)
on the same cube with the looks that n='auto' would pick, so the cost of n='auto' can be read off.

CUDA-event time, best of 7 after a warm-up call; before every timed call the L2 is flushed by writing 256 MB (the
cube is 0.1-0.9 GB, and single-pol float32 would fit the 126 MB L2).  GB/s counts the algorithmic bytes: the cube
read once and the ENL map written once.  "HBM bound" is that traffic at 7.7 TB/s.
Usage: dev_enl.py [--out FILE] (default profiles/r5_enl.txt)."""
import ctypes, os, sys
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np, torch
from nd_b200 import _lib, change
from dev_chg import card, cube

HBM_BYTES_PER_S = 7.7e12


def timed(call, flush, reps=7):
    call(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e30
    for _ in range(reps):
        flush.zero_()
        e0.record(); call(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def run(pol, dtype, looks, flush, windows=(7, 11), rows=1024, cols=1024, k=24):
    v = cube(rows, cols, k, pol, looks, 'flat').to(dtype).contiguous()
    enl = torch.empty((rows, cols, k), dtype=dtype, device="cuda")
    res = torch.empty((rows, cols, k), dtype=torch.uint8, device="cuda")
    L = _lib.lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    code = 0 if dtype == torch.float32 else 1
    args = (ctypes.c_void_p(v.data_ptr()), _lib.i64(v.shape[:3]), _lib.i64(v.stride()), code, change._POL_CODES[pol])
    lines = []
    for w in windows:
        def call():
            rc = L.ndchg_enl(*args, w, ctypes.c_void_p(enl.data_ptr()), st)
            assert rc == 0, L.ndchg_last_error()
        ms = timed(call, flush)
        E = float(np.nanmedian(enl.cpu().numpy()))
        n = max(int(np.floor(E)), 3 if pol == 'quad' else 1)
        def walk():
            rc = L.ndchg_change_detection_pol(*args, ctypes.c_void_p(res.data_ptr()), 0.99, n, st)
            assert rc == 0, L.ndchg_last_error()
        walk_ms = timed(walk, flush)
        nbytes = v.numel() * v.element_size() + enl.numel() * enl.element_size()
        hbm_ms = nbytes / HBM_BYTES_PER_S * 1e3
        lines.append("%-13s %s %dx%dx%d looks=%d w=%2d: enl %8.3f ms  %7.1f GB/s  HBM bound %6.3f ms (%4.1f %% of the kernel)"
                     "  median ENL %6.2f -> n=%d  walk %7.3f ms  enl / walk %5.2f" % (
                         pol, str(dtype)[6:], rows, cols, k, looks, w, ms, nbytes / ms / 1e6, hbm_ms, 100 * hbm_ms / ms,
                         E, n, walk_ms, ms / walk_ms))
        print(lines[-1], flush=True)
    del v, enl, res
    torch.cuda.empty_cache()
    return lines


if __name__ == "__main__":
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(os.path.dirname(HERE), "profiles", "r5_enl.txt")
    head = ["# tools/dev_enl.py on 1 x %s (card name and power limit read in this run)" % card(),
            "# ndchg_enl on a 1024 x 1024 x 24 cube of 12-look stationary samples (unit-power independent channels),",
            "# CUDA events, best of 7 after a warm-up, L2 flushed (256 MB written) before every timed call.  GB/s: cube",
            "# read once + ENL map written once.  HBM bound: those bytes at 7.7 TB/s.  walk: ndchg_change_detection_pol",
            "# on the same cube, alpha = 0.99, with the looks n = floor(median ENL) that n='auto' picks."]
    for line in head:
        print(line, flush=True)
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    lines = list(head)
    for pol in ('dual', 'single', 'quad', 'dual_diagonal', 'quad_diagonal'):
        for dtype in (torch.float32, torch.float64):
            lines += run(pol, dtype, 12, flush)
    with open(out, "w") as f:
        f.write("\n".join(lines) + "\n")
