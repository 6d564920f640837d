#!/usr/bin/env python
"""Timing (GPU) of the refined Lee filter kernel (ndchg_refined_lee, include/ndchg.h) on a 1024 x 1024 x 24 cube of
every covariance layout, float32 and float64, windows 7, 11 and 15, next to a 7 x 7 boxcar (the sibling-filter
kernel behind BoxcarFilter(w=7)) over the same (rows, cols, k, bands) array as a bandwidth reference.

CUDA-event time, best of 7 after a warm-up call; before every timed call the L2 is flushed by writing 256 MB (the
cube is 0.1-0.9 GB).  GB/s counts the algorithmic bytes: the cube read once and written once; "HBM bound" is that
traffic at 7.7 TB/s.  The kernel's own work per output pixel, from its loops: N^2 (bands + 2) double-precision
shared-memory reads and N^2 (bands + 4) double additions / multiplications (every thread walks the whole window
and keeps the terms inside its mask), plus the staging and the box means.  "smem" is the rate of those reads.
Usage: dev_lee.py [--out FILE] (default profiles/r7_refined_lee.txt)."""
import ctypes, os, subprocess, sys
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy as np, torch
from nd_b200 import _lib, _ndimage, change
from dev_chg import cube

HBM_BYTES_PER_S = 7.7e12


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        info = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        info = "unknown"
    return "%s (nvidia-smi %s: %s)" % (torch.cuda.get_device_name(), q, info or "unknown")


def timed(call, flush, reps=7):
    call(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e30
    for _ in range(reps):
        flush.zero_()
        e0.record(); call(); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best


def run(pol, dtype, looks, flush, windows=(7, 11, 15), rows=1024, cols=1024, k=24):
    v = cube(rows, cols, k, pol, looks, 'flat').to(dtype).contiguous()
    out = torch.empty_like(v)
    L = _lib.lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    B = v.shape[3]
    nbytes = 2 * v.numel() * v.element_size()
    hbm_ms = nbytes / HBM_BYTES_PER_S * 1e3
    box_ms = timed(lambda: _ndimage.correlate_device(v, out, np.ones((7, 7, 1, 1)) / 49.0, [0, 0, 0, 0]), flush)
    lines = []
    for w in windows:
        def call():
            rc = L.ndchg_refined_lee(ctypes.c_void_p(v.data_ptr()), _lib.i64(v.shape[:3]), _lib.i64(v.stride()),
                                     0 if dtype == torch.float32 else 1, change._POL_CODES[pol], w, float(looks),
                                     ctypes.c_void_p(out.data_ptr()), st)
            assert rc == 0, L.ndchg_last_error()
        ms = timed(call, flush)
        outputs = rows * cols * k
        smem_bytes = outputs * w * w * (B + 2) * 8
        flops = outputs * w * w * (B + 4)
        lines.append("%-13s %s %dx%dx%d w=%2d: lee %8.3f ms  %7.1f GB/s  HBM bound %6.3f ms (%5.1f %% of the kernel)"
                     "  smem reads %6.1f TB/s  fp64 %6.2f Top/s  boxcar7 %6.3f ms (lee / boxcar %5.1f)" % (
                         pol, str(dtype)[6:], rows, cols, k, w, ms, nbytes / ms / 1e6, hbm_ms, 100 * hbm_ms / ms,
                         smem_bytes / ms / 1e9, flops / ms / 1e9, box_ms, ms / box_ms))
        print(lines[-1], flush=True)
    del v, out
    torch.cuda.empty_cache()
    return lines


if __name__ == "__main__":
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else os.path.join(os.path.dirname(HERE), "profiles", "r7_refined_lee.txt")
    head = ["# tools/dev_lee.py on 1 x %s" % card(),
            "# ndchg_refined_lee on a 1024 x 1024 x 24 cube of 4-look stationary samples (unit-power independent channels),",
            "# looks = 4, CUDA events, best of 7 after a warm-up, L2 flushed (256 MB written) before every timed call.",
            "# GB/s: cube read once + written once.  HBM bound: those bytes at 7.7 TB/s.  smem reads: N^2 (bands + 2)",
            "# doubles per output.  fp64: N^2 (bands + 4) double operations per output.  boxcar7: the 7 x 7 boxcar",
            "# (ndflt_correlate, as BoxcarFilter(w=7)) over the same array, mode 'reflect'."]
    for line in head:
        print(line, flush=True)
    flush = torch.empty(64 << 20, dtype=torch.float32, device="cuda")
    lines = list(head)
    for pol in ('dual', 'single', 'quad', 'dual_diagonal', 'quad_diagonal'):
        for dtype in (torch.float32, torch.float64):
            lines += run(pol, dtype, 4, flush)
    with open(out, "w") as f:
        f.write("\n".join(lines) + "\n")
