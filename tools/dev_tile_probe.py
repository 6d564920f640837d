#!/usr/bin/env python
"""Tile timeline of the f = 1 tiled NLM kernel (GPU, development only): where the time of one CTA tile goes.

A library built with -DNDNLM_TILE_PROBE=1 has one warp per CTA record clock64() at the phase boundaries of every tile
(nlm_tiled.cuh, slots below).  This tool runs the cfg3 parameters (V = 4, r = (5,5,2), f = 1) on a ROWS x 4096 x 32
cube with NDNLM_PERSIST = 0 and 1 and prints the mean share of each phase in the SM time per tile (the gap between
two tiles on the same SM included).

  python tools/dev_tile_probe.py --build DIR          # compile the probe library into DIR (no GPU needed)
  NDNLM_LIB=DIR/libndnlm.so python tools/dev_tile_probe.py [--rows 600] [--persist 0,1]

Slots: 0 tile start, 1 box landed, 2 / 3 pass barrier entered / left (persistent kernel: 3 = end-of-tile barrier left),
4 box of pass 1 landed, 5 last offset done, 6 epilogue done, 7 SM id.  Cycles are SM clocks.
"""
import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def build(out_dir):
    import __graft_entry__ as g
    os.makedirs(out_dir, exist_ok=True)
    csrc = g.CSRC
    units = [os.path.join(csrc, f) for f in sorted(os.listdir(csrc)) if f.endswith(".cu")]
    flags = g.COMPILE_FLAGS + ["-DNDNLM_TILE_PROBE=1"]
    procs, objs = [], []
    for cu in units:
        obj = os.path.join(out_dir, os.path.basename(cu)[:-3] + ".o")
        objs.append(obj)
        procs.append(subprocess.Popen(["nvcc"] + flags + ["-c", "-o", obj, cu]))
    if any(p.wait() != 0 for p in procs):
        raise SystemExit("nvcc failed")
    lib = os.path.join(out_dir, "libndnlm.so")
    subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", lib] + objs)
    print("built", lib)


def phases(rec, persist):
    import numpy as np
    t = rec[:, :7].astype(np.int64)
    sm = rec[:, 7]
    # SM time per tile: from this tile's start to the start of the next tile on the same SM
    order = np.lexsort((t[:, 0], sm))
    nxt = np.full(len(t), -1, np.int64)
    same = sm[order][1:] == sm[order][:-1]
    nxt[order[:-1][same]] = t[order[1:][same], 0]
    keep = nxt > 0
    t, nxt = t[keep], nxt[keep]
    if persist:
        parts = [("wait for the box", t[:, 1] - t[:, 0]),
                 ("offsets (compute)", t[:, 5] - t[:, 1]),
                 ("end-of-tile barrier + next TMA issue", t[:, 3] - t[:, 5]),
                 ("epilogue", t[:, 6] - t[:, 3]),
                 ("gap to next tile on the SM", nxt - t[:, 6])]
    else:
        parts = [("first box (TMA pass 0)", t[:, 1] - t[:, 0]),
                 ("pass 0 offsets", t[:, 2] - t[:, 1]),
                 ("pass barrier (drain)", t[:, 3] - t[:, 2]),
                 ("second box (TMA pass 1)", t[:, 4] - t[:, 3]),
                 ("pass 1 offsets", t[:, 5] - t[:, 4]),
                 ("epilogue", t[:, 6] - t[:, 5]),
                 ("gap to next CTA on the SM", nxt - t[:, 6])]
    total = (nxt - t[:, 0]).astype(np.float64)
    return parts, total, int(keep.sum())


def main():
    args = sys.argv[1:]
    if args[:1] == ["--build"]:
        build(args[1])
        return
    opts = {"--rows": "600", "--persist": "0,1"}
    for i in range(0, len(args), 2):
        opts[args[i]] = args[i + 1]
    import numpy as np
    import torch
    from nd_b200 import _lib, device
    L = _lib.lib()
    if not hasattr(L, "ndnlm_tile_probe"):
        raise SystemExit("the library at %s was not built with -DNDNLM_TILE_PROBE=1 (see --build)" % _lib.LIB_PATH)
    L.ndnlm_tile_probe.argtypes = [ctypes.c_void_p, ctypes.c_int]
    props = torch.cuda.get_device_properties(0)
    print("device:", props.name, flush=True)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
        print("power limit, SM clock, max SM clock:", q)
    except OSError:
        pass
    shape, r, f = (int(opts["--rows"]), 4096, 32, 4), (5, 5, 2), (1, 1, 1)
    rng = np.random.default_rng(0)
    a = torch.from_numpy(rng.gamma(4.0, 0.25, size=shape).astype(np.float32)).cuda()
    for flag in opts["--persist"].split(","):
        os.environ["NDNLM_PERSIST"] = flag
        plan = device.Plan(shape, r, f, 0.3, 0.6)
        ntiles = int(np.prod([(n + t - 1) // t for n, t in zip(plan.info.n, plan.info.tile)]))
        buf = torch.zeros(ntiles * 8, dtype=torch.int64, device="cuda")
        plan.apply(a)                                   # warm-up
        L.ndnlm_tile_probe(ctypes.c_void_p(buf.data_ptr()), ntiles)
        plan.apply(a)
        torch.cuda.synchronize()
        L.ndnlm_tile_probe(None, 0)
        rec = buf.view(ntiles, 8).cpu().numpy().view(np.uint64)
        parts, total, n = phases(rec, flag != "0")
        print("\nNDNLM_PERSIST=%s  %s  tiles %d (timed %d)  mean SM time per tile %.0f cycles"
              % (flag, plan.kernel_name, ntiles, n, total.mean()))
        for name, d in parts:
            print("  %-40s %10.0f cycles  %6.2f %%" % (name, d.mean(), 100.0 * d.sum() / total.sum()))


if __name__ == "__main__":
    main()
