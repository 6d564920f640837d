#!/usr/bin/env python
"""Development timing (GPU) of the omnibus change-detection kernels: Mpixel/s for a (rows, cols, k, bands) cube of
every covariance layout (include/ndchg.h), float32 and float64, with one change per series and without.
`--direction`: the walk alone (ndchg_change_detection_pol) against the walk plus the direction post-pass
(ndchg_change_direction) on the same cube, on series that step up, down and both ways, and on stationary series."""
import ctypes, os, subprocess, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from nd_b200 import _lib, change

P = {'dual': 2, 'single': 1, 'quad': 3, 'dual_diagonal': 2, 'quad_diagonal': 3}

def amplitudes(t, k, p, pattern):
    """Channel amplitudes at step t: 'step' x1.5 from k // 2 on; 'updown' four segments of k // 4 steps -- x1, x1.5
    (increase), x1 (decrease), then channel 0 x1.5 and the others / 1.5 (indefinite; single-pol: increase);
    'flat' x1 throughout."""
    if pattern == 'step':
        return [1.5 if t >= k // 2 else 1.0] * p
    if pattern == 'updown':
        seg = min(4 * t // k, 3)
        return [1.0, 1.5, 1.0][seg:seg + 1] * p if seg < 3 else [1.5] + [1 / 1.5] * (p - 1)
    return [1.0] * p

def cube(rows, cols, k, pol, looks, pattern):
    """n-look sample covariances of independent unit-power channels in the band order of `pol`, generated on the
    GPU one time step at a time, with the channel amplitudes of `amplitudes(t, k, p, pattern)`."""
    g = torch.Generator(device="cuda").manual_seed(0)
    out = []
    for t in range(k):
        z = torch.randn((rows, cols, looks, P[pol], 2), device="cuda", generator=g) / 2 ** 0.5
        if pattern != 'flat':
            z *= torch.tensor(amplitudes(t, k, P[pol], pattern), device="cuda")[:, None]
        z = torch.complex(z[..., 0], z[..., 1])
        c = torch.einsum('...li,...lj->...ij', z, z.conj()) / looks
        if pol == 'dual':
            b = [c[..., 0, 0].real, c[..., 0, 1].real, c[..., 0, 1].imag, c[..., 1, 1].real]
        elif pol == 'quad':
            b = [c[..., 0, 0].real, c[..., 0, 1].real, c[..., 0, 1].imag, c[..., 0, 2].real, c[..., 0, 2].imag,
                 c[..., 1, 1].real, c[..., 1, 2].real, c[..., 1, 2].imag, c[..., 2, 2].real]
        else:
            b = [c[..., i, i].real for i in range(P[pol])]
        out.append(torch.stack(b, -1))
    return torch.stack(out, 2)

def run(rows, cols, k, dtype, pol, looks=50, alpha=0.9999, jumps=True):
    v = cube(rows, cols, k, pol, looks, 'step' if jumps else 'flat').to(dtype).contiguous()
    res = torch.empty((rows, cols, k), dtype=torch.uint8, device="cuda")
    L = _lib.lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    def call():
        rc = L.ndchg_change_detection_pol(ctypes.c_void_p(v.data_ptr()), _lib.i64(v.shape[:3]), _lib.i64(v.stride()),
                                          0 if dtype == torch.float32 else 1, change._POL_CODES[pol],
                                          ctypes.c_void_p(res.data_ptr()), alpha, looks, st)
        assert rc == 0, L.ndchg_last_error()
    call(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e30
    for _ in range(3):
        e0.record(); call(); e1.record(); torch.cuda.synchronize(); best = min(best, e0.elapsed_time(e1))
    nbytes = v.numel() * v.element_size() + res.numel()
    print("%-13s %s %dx%dx%d looks=%d %s: %8.3f ms  %7.1f Mpixel/s  %6.1f GB/s of algorithmic bytes  changes/pixel=%.3f" % (
        pol, str(dtype)[6:], rows, cols, k, looks, "jumps" if jumps else "flat ", best, rows * cols / best / 1e3,
        nbytes / best / 1e6, res.float().sum().item() / (rows * cols)), flush=True)
    del v, res
    torch.cuda.empty_cache()

def run_direction(rows, cols, k, dtype, pol, looks=50, alpha=0.9999, pattern='updown', reps=7):
    v = cube(rows, cols, k, pol, looks, pattern).to(dtype).contiguous()
    walk = torch.empty((rows, cols, k), dtype=torch.uint8, device="cuda")
    codes = torch.empty_like(walk)
    L = _lib.lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    args = lambda out: (ctypes.c_void_p(v.data_ptr()), _lib.i64(v.shape[:3]), _lib.i64(v.stride()),
                        0 if dtype == torch.float32 else 1, change._POL_CODES[pol], ctypes.c_void_p(out.data_ptr()),
                        alpha, looks, st)
    calls = [lambda: L.ndchg_change_detection_pol(*args(walk)), lambda: L.ndchg_change_direction(*args(codes))]
    for call in calls:
        assert call() == 0, L.ndchg_last_error()
    torch.cuda.synchronize()
    assert torch.equal((codes != 0).to(torch.uint8), walk), "direction codes do not mark the walk's changes"
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = [1e30, 1e30]
    for _ in range(reps):                                                        # alternate the two, best of `reps`
        for i, call in enumerate(calls):
            e0.record(); call(); e1.record(); torch.cuda.synchronize(); best[i] = min(best[i], e0.elapsed_time(e1))
    n = float(rows * cols)
    frac = [(codes == c).sum().item() / n for c in (1, 2, 3)]
    print("%-13s %s %dx%dx%d looks=%d %s: walk %8.3f ms  walk+direction %8.3f ms  post-pass %6.3f ms = %5.1f %% of the walk"
          "  changes/pixel=%.3f (increase %.3f, decrease %.3f, indefinite %.3f)" % (
        pol, str(dtype)[6:], rows, cols, k, looks, "jumps" if pattern != 'flat' else "flat ", best[0], best[1],
        best[1] - best[0], 100 * (best[1] - best[0]) / best[0], sum(frac), *frac), flush=True)
    del v, walk, codes
    torch.cuda.empty_cache()

def card():
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        limit = "unknown"
    return "%s, power limit %s" % (torch.cuda.get_device_name(), limit or "unknown")

if __name__ == "__main__":
    print("# %s" % card(), flush=True)
    for pol in ('dual', 'single', 'quad', 'dual_diagonal', 'quad_diagonal'):
        for dtype in (torch.float32, torch.float64):
            for jumps in (True, False):
                if "--direction" in sys.argv:
                    run_direction(1024, 1024, 24, dtype, pol, pattern='updown' if jumps else 'flat')
                else:
                    run(1024, 1024, 24, dtype, pol, jumps=jumps)
