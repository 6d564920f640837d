#!/usr/bin/env python
"""
bench.py -- NLMeansFilter throughput on B200, one JSON line (driver contract).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--workload cfg3|cfg2|cfg1|cfg4|cfg5] [--rows R] [--semantics as_written|reference_compiled]
                  [--dump-outputs DIR]
  N > 1:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...
  python bench.py --apply-njobs N      single process: NLMeansFilter(...).apply(ds, njobs=N) on a host Dataset

Workloads (BASELINE.json configs):
  cfg3 (default, configs[2])  synthetic SAR-like cube 4096 x 4096 x 32 PER GPU, 4 float32 variables, r=(5,5,2), f=1;
                              device-resident, weak scaling: rank k owns rows [4096 k, 4096 (k+1)).
  cfg2 (configs[1])           synthetic stand-in 1024 x 1024 x 24 (the file is absent from the reference), r=(5,5,1), f=1.
  cfg1 (configs[0])           the reference's own data/slc.data raster (206 x 500, 4 variables; fixture
                              tests/golden/slc_cfg1.npz), r=(3,3), f=1 -- also checked against the reference's output.
  cfg4 (configs[3])           synthetic 16384 x 16384 x 64, 4 variables, r=(7,7,2), f=2: ONE global cube y-sharded over
                              the ranks (strong scaling); each rank streams its shard through the GPU slab by slab
                              (nd_b200.stream.apply_device_streamed) because cube + staged copy + result exceed HBM.
  cfg5 (configs[4])           synthetic 32768 x 32768 x 128, 6 variables, r=(10,10,3), f=2; as cfg4.
  --rows R bounds the rows PER GPU that are actually processed (cfg4 / cfg5: a partial sweep of every shard,
  stated in `config.sweep`; the per-voxel work does not depend on the position in the cube).

Multi-GPU: halo rows r_y+f_y are exchanged between neighbouring ranks with NCCL send/recv before every apply;
there is no other collective on the data path.

A "step" = one pass of the hot path over the rank's rows: (synthesis of the slab for streamed workloads ->)
stage (reflect-pad) -> halo exchange -> nlm kernel -> unstage.  `value` = voxels of all ranks / max-over-ranks time.
`e2e` = the same through the reference-facing entry point `_pixelwise_nlmeans_3d` on pinned HOST arrays (H2D +
kernels + D2H inside the timed region), with the copy-only ceiling of the same pipeline beside it.
`roofline` is for the dominant kernel: algorithmic FP32 flops (SURVEY.md 8(d)) / CUDA-event time of its launches.
`parity` compares sampled sub-cubes of the benchmarked cube (true corner, slab / rank seam, interior) with the oracle
(C restatement pinned bit-exact to the compiled reference) in the same run; above 1e-4 the run fails.
`cpu_baseline` times the reference's own Cython kernel on the host cores on a bounded crop.

--dump-outputs DIR writes what the last timed step computed, the (rows, nx, nt, V) float32 result of each rank, as
DIR/out.npy (DIR/out_rank<k>.npy for N > 1): a (K, V) array of K voxels in memory order, every voxel when the result
fits in 48 MB / N, else a fixed seeded sample (`dump_sample`).  The inputs depend on the arguments only, so two builds
of the project can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg3": dict(rows=4096, nx=4096, nt=32, V=4, r=(5, 5, 2), f=1, sigma=0.25, h=0.5, scaling="weak", mode="resident",
                 roi=(8, 16, 8),
                 text="synthetic SAR-like cube 4096x4096x32 per GPU, 4 float32 variables, r=(5,5,2), f=1 (BASELINE configs[2])"),
    "cfg2": dict(rows=1024, nx=1024, nt=24, V=4, r=(5, 5, 1), f=1, sigma=0.25, h=0.5, scaling="weak", mode="resident",
                 roi=(8, 16, 8),
                 text="synthetic stand-in 1024x1024x24 for the absent s1_kalimantan file, 4 float32 variables, r=(5,5,1), f=1 (BASELINE configs[1])"),
    "cfg1": dict(rows=206, nx=500, nt=1, V=4, r=(3, 3, 0), f=1, sigma=0.01, h=0.05, scaling="weak", mode="resident",
                 roi=(16, 32, 1), real="tests/golden/slc_cfg1.npz",
                 text="the reference's data/slc.data raster 206x500 (C11, C12_real, C12_imag, C22), r=(3,3), f=1, "
                      "sigma=0.01, h=0.05 scaled to the data (BASELINE configs[0])"),
    "cfg4": dict(global_rows=16384, nx=16384, nt=64, V=4, r=(7, 7, 2), f=2, sigma=0.25, h=0.5, scaling="strong",
                 mode="streamed", slab_rows=256, roi=(4, 8, 4),
                 text="synthetic SAR-like cube 16384x16384x64, 4 float32 variables, r=(7,7,2), f=2, y-sharded (BASELINE configs[3])"),
    "cfg5": dict(global_rows=32768, nx=32768, nt=128, V=6, r=(10, 10, 3), f=2, sigma=0.25, h=0.5, scaling="strong",
                 mode="streamed", slab_rows=32, roi=(2, 8, 4),
                 text="synthetic Sentinel-1 C2-like cube 32768x32768x128, 6 float32 covariance components, r=(10,10,3), f=2, y-sharded (BASELINE configs[4])"),
}
METRIC = "NLMeansFilter Mvoxel/s"
UNIT = "Mvoxel/s"
PARITY_TOL = 1e-4
DUMP_BYTES = 48 << 20          # --dump-outputs: all ranks together


def fvec(wl):
    return tuple(wl["f"] if x > 0 else 0 for x in wl["r"])


def dump_sample(shape, world, seed=1234):
    """(y, x, t) coordinates of the voxels --dump-outputs writes of a (ny, nx, nt, V) float32 result, in memory order:
    every voxel when the result fits in DUMP_BYTES / world, else a seeded sample of that many voxels."""
    import numpy as np
    ny, nx, nt, V = shape
    n, k = ny * nx * nt, DUMP_BYTES // world // (4 * V)
    flat = np.arange(n) if n <= k else np.sort(np.random.default_rng(seed).choice(n, k, replace=False))
    y, rest = np.divmod(flat, nx * nt)
    x, t = np.divmod(rest, nt)
    return y, x, t


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm_gbs": float(p.get("hbm_gbs", 6650.0)), "sm_max_mhz": float(p.get("sm_max_mhz", 1965.0)),
                "source": "MEASURED_PEAKS.json"}
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [l.strip().split(", ") for l in open(self.path) if l.strip()]
            os.unlink(self.path)
            sm = sorted(float(r[1]) for r in rows if len(r) >= 8)
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = float(rows[0][2])
                out["power_w_max"] = max(float(r[3]) for r in rows if len(r) >= 8)
                out["samples"] = len(sm)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for i, nm in enumerate(names):
                    if any(r[4 + i].strip().lower() == "active" for r in rows if len(r) >= 8):
                        out["reasons"].append(nm)
        except Exception:
            pass
        return out


# ------------------------------------------------------------------------------------------------
# CPU baseline: the reference's own Cython kernel on the host cores, bounded crop
# ------------------------------------------------------------------------------------------------
def _cpu_crop_job(args):
    """Worker: filter one independent crop with the reference kernel."""
    crop, r, f, sigma, h, which = args
    from oracle import ref
    fn = ref.as_written_patched if which == "as_written" else ref.reference_compiled
    return float(fn(crop, r, f, sigma, h, -1).sum())


def cpu_reference_rate(crop, r, f, sigma, h, which, procs):
    """voxels/s of the reference kernel with `procs` processes, each filtering its own copy-sized crop
    (no overlapping halos between workers: the most favourable way to use all host cores; the
    reference's own njobs mechanism, nd/utils.py:343-401, re-reads r+f buffer rows per worker)."""
    import multiprocessing as mp
    jobs = [(crop, r, f, sigma, h, which)] * procs
    t0 = time.perf_counter()
    if procs == 1:
        sums = [_cpu_crop_job(jobs[0])]
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            sums = pool.map(_cpu_crop_job, jobs)
    dt = time.perf_counter() - t0
    return procs * crop.shape[0] * crop.shape[1] * crop.shape[2] / dt, dt, sums


def _crop_dims(wl, which, seconds):
    """Per-core crop (rows, cols, nt) of the workload for ~`seconds` of reference time.  Every extent is at least
    r+f+1 (below that the reference's single reflection is undefined); the per-voxel cost of the reference does not
    depend on the extents, so a small crop measures the same rate as the full cube.  Sized from the measured cost
    of the reference's loops (~14 ns per patch element as written, ~74 ns per offset for the unmodified binary;
    SURVEY.md 8(a))."""
    r, fv = wl["r"], fvec(wl)
    K = (2 * r[0] + 1) * (2 * r[1] + 1) * (2 * r[2] + 1) - 1
    patch = (2 * fv[0] + 1) * (2 * fv[1] + 1) * (2 * fv[2] + 1)
    per_voxel = K * patch * wl["V"] * 14e-9 if which == "as_written" else K * 74e-9
    nt = min(wl["nt"], max(r[2] + fv[2] + 1, 8 if per_voxel < 2e-3 else 0))
    cols = min(wl["nx"], max(r[1] + fv[1] + 1, 16 if per_voxel < 2e-3 else 0))
    total_rows = wl.get("rows", wl.get("global_rows"))
    rows = int(max(r[0] + fv[0] + 1, min(total_rows, seconds / per_voxel / (cols * nt))))
    return rows, cols, nt


def make_cpu_crop(wl, rows, cols, nt):
    """A (rows, cols, nt, V) float32 crop with the statistics of the synthetic cube (NumPy generator)."""
    import numpy as np
    rng = np.random.default_rng(42)
    a = rng.gamma(4.0, 0.25, size=(rows, cols, nt, wl["V"])).astype(np.float32)
    a[..., 1:3] = rng.normal(0, 0.3, size=a[..., 1:3].shape).astype(np.float32)
    return a


def cpu_baseline(wl, semantics, target_seconds=12.0):
    from oracle import build_ref
    r, sigma, h = wl["r"], wl["sigma"], wl["h"]
    fv = fvec(wl)
    cores = os.cpu_count() or 1
    if not build_ref.built():
        # no compiled reference on this box: fall back to the C port of the oracle (kind "port")
        from oracle import c_port
        crop = make_cpu_crop(wl, *_crop_dims(wl, semantics, target_seconds * cores))
        t0 = time.perf_counter()
        c_port.nlmeans(crop, r, fv, sigma, h, -1, semantics, threads=cores)
        dt = time.perf_counter() - t0
        return {"value": crop[..., 0].size / dt / 1e6, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "%dx%dx%d crop, C port of the oracle with OpenMP" % crop.shape[:3]}
    crop = make_cpu_crop(wl, *_crop_dims(wl, "as_written", target_seconds))
    rate, dt, _ = cpu_reference_rate(crop, r, fv, sigma, h, "as_written", cores)
    rate_c, dt_c, _ = cpu_reference_rate(crop, r, fv, sigma, h, "reference_compiled", cores)
    head = rate if semantics == "as_written" else rate_c
    return {"value": head / 1e6, "unit": UNIT, "cores": cores, "kind": "reference", "semantics": semantics,
            "sample": "%d independent %dx%dx%d crops (V=%d, same r/f/sigma/h as the workload), one per host core; "
                      "as-written = reference .pyx with the three SIZE_TYPE casts (%.1f s), reference_compiled = the "
                      "unmodified binary (%.1f s)" % ((cores,) + crop.shape[:3] + (wl["V"], dt, dt_c)),
            "per_core_value": head / cores / 1e6,
            "as_written_value": rate / 1e6,
            "unmodified_binary_value": rate_c / 1e6,
            "unmodified_binary_note": "unmodified reference binary on the same crop: because of the unsigned-f bug "
                                      "(SURVEY F1) it computes a box mean, not patch distances"}


# ------------------------------------------------------------------------------------------------
# reference arm
# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import build_ref
    wl = WORKLOADS[args.workload]
    r, sigma, h = wl["r"], wl["sigma"], wl["h"]
    fv = fvec(wl)
    cores = os.cpu_count() or 1
    kind = "reference" if build_ref.built() else "port"
    which = args.semantics
    per_step_s = max(2.0, min(8.0, 150.0 / max(args.steps + args.warmup, 1)))
    crop = make_cpu_crop(wl, *_crop_dims(wl, which, per_step_s * (1 if kind == "reference" else cores)))
    rows, cols = crop.shape[:2]
    times = []
    for it in range(args.warmup + args.steps):
        if kind == "reference":
            _, dt, _ = cpu_reference_rate(crop, r, fv, sigma, h, which, cores)
        else:
            from oracle import c_port
            t0 = time.perf_counter()
            c_port.nlmeans(crop, r, fv, sigma, h, -1, which, threads=cores)
            dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    total = sum(times)
    vox = rows * cols * crop.shape[2] * (cores if kind == "reference" else 1)
    value = vox * len(times) / total / 1e6
    sample = ("%s %dx%dx%d crops of the workload (V=%d, same r/f/sigma/h), %s"
              % ("%d independent" % cores if kind == "reference" else "one", rows, cols, crop.shape[2], wl["V"],
                 ("one per host core, reference nd/_filters.pyx (%s)" % ("as-written: three SIZE_TYPE casts"
                                                                         if which == "as_written" else "unmodified binary"))
                 if kind == "reference" else "C port of the oracle with OpenMP on %d threads" % cores))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
            "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "description": wl["text"], "semantics": which},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def bind_to_gpu_cpus(gpu_index):
    """One process per GPU: run on the CPUs that are local to this rank's GPU (NVML's affinity mask), so that the
    pinned host chunk of the e2e leg is allocated on the NUMA node its PCIe link hangs off.  Returns the CPU count
    or None when NVML / the affinity call is unavailable (nothing changes then)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------------
# in-run parity: sampled sub-cubes of the benchmarked cube against the oracle
# ------------------------------------------------------------------------------------------------
def parity_samples(wl, rows_rank0, global_rows, world, seam_rows):
    """ROIs (global coordinates, inside rank 0's processed rows): true corner, slab / rank seams, interior."""
    ry, rx, rt = wl["roi"]
    nx, nt = wl["nx"], wl["nt"]
    ry, rx, rt = min(ry, rows_rank0), min(rx, nx), min(rt, nt)
    out = [("corner", 0, 0, 0)]
    for name, row in seam_rows:
        y0 = min(max(row - ry // 2, 0), rows_rank0 - ry)
        out.append((name, y0, min(nx - rx, (nx // 3) // 2 * 2), max(0, nt - rt)))
    out.append(("interior", max(0, rows_rank0 // 2 - ry // 2), max(0, nx // 2 - rx // 2), max(0, (nt - rt) // 2)))
    seen, res = set(), []
    for name, y0, x0, t0 in out:
        key = (y0, x0, t0)
        if key in seen:
            continue
        seen.add(key)
        res.append({"name": name, "y": (y0, y0 + ry), "x": (x0, x0 + rx), "t": (t0, t0 + rt)})
    return res


def check_parity(wl, samples, gpu_blocks, get_rows, global_rows, semantics):
    """gpu_blocks[i]: NumPy (ry, rx, rt, V) block of the GPU result for samples[i];
    get_rows(ya, yb) -> NumPy (yb-ya, nx, nt, V) input rows (global row indices)."""
    import numpy as np
    from oracle import c_port
    r, fv = wl["r"], fvec(wl)
    pad = [r[k] + fv[k] for k in range(3)]
    nx, nt, V = wl["nx"], wl["nt"], wl["V"]
    worst, rep = 0.0, []
    t_or = time.perf_counter()
    for smp, got in zip(samples, gpu_blocks):
        (y0, y1), (x0, x1), (t0, t1) = smp["y"], smp["x"], smp["t"]
        ya, yb = max(y0 - pad[0], 0), min(y1 + pad[0], global_rows)
        xa, xb = max(x0 - pad[1], 0), min(x1 + pad[1], nx)
        ta, tb = max(t0 - pad[2], 0), min(t1 + pad[2], nt)
        crop = np.ascontiguousarray(get_rows(ya, yb)[:, xa:xb, ta:tb])
        ref = c_port.nlmeans(crop, r, fv, wl["sigma"], wl["h"], -1, semantics, threads=os.cpu_count(),
                             roi=((y0 - ya, y1 - ya), (x0 - xa, x1 - xa), (t0 - ta, t1 - ta)))
        ref = ref[y0 - ya:y1 - ya, x0 - xa:x1 - xa, t0 - ta:t1 - ta]
        err = 0.0
        for v in range(V):
            scale = max(float(np.abs(ref[..., v]).max()), 1e-30)
            err = max(err, float(np.abs(got[..., v].astype(np.float64) - ref[..., v]).max()) / scale)
        if not (np.isfinite(got).all() and np.isfinite(ref).all()):
            err = float("inf")
        rep.append({"name": smp["name"], "y": list(smp["y"]), "x": list(smp["x"]), "t": list(smp["t"]), "err": err,
                    "bitwise_equal_values": int((got == ref).sum()), "values": int(ref.size),
                    "ref_absmax": float(np.abs(ref).max()), "ref_minus_input_absmax":
                    float(np.abs(ref - crop[y0 - ya:y1 - ya, x0 - xa:x1 - xa, t0 - ta:t1 - ta]).max())})
        worst = max(worst, err)
    return {"max_scaled_err": worst, "tolerance": PARITY_TOL, "ok": bool(worst <= PARITY_TOL), "samples": rep,
            "metric": "max_p |out - ref| / max_p |ref_v| per variable over each sub-cube (SURVEY.md 8(d))",
            "oracle": "oracle.c_port (plain-C restatement of nd/_filters.pyx:317-420, pinned bit-exact to the compiled "
                      "reference by tests/test_oracle.py), %s semantics, on crops of the same input with a halo of r+f"
                      % semantics,
            "oracle_seconds": time.perf_counter() - t_or}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from nd_b200 import device
    from nd_b200 import stream as nstream
    from nd_b200._filters import _pixelwise_nlmeans_3d
    from nd_b200.shard import DistributedShard, exchange_halos_dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback")
    # stdout carries exactly ONE JSON line: whatever libraries print on fd 1 meanwhile (NCCL announces its version
    # there) is sent to stderr, and the line is written to the real stdout at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    numa = bind_to_gpu_cpus(local_rank) if world > 1 else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    name = args.workload
    wl = WORKLOADS[name]
    nx, nt, V, r, sigma, h = wl["nx"], wl["nt"], wl["V"], wl["r"], wl["sigma"], wl["h"]
    fv = fvec(wl)
    halo = r[0] + fv[0]
    sem = args.semantics
    streamed = wl["mode"] == "streamed"
    pk = peaks()
    if streamed:
        global_rows = args.global_rows or wl["global_rows"]
        shard_rows = global_rows // world                 # rows of the global cube this rank owns
        ny = min(args.rows, shard_rows) if args.rows else shard_rows    # rows it actually processes
        y_lo = rank * shard_rows
    else:
        ny = args.rows if args.rows else wl["rows"]
        shard_rows = ny
        global_rows = ny * world
        y_lo = rank * ny
    real = None
    if wl.get("real"):
        path = os.path.join(ROOT, wl["real"])
        if os.path.exists(path) and world == 1 and not args.rows:
            real = np.load(path)
    data_kind = "real (reference data/slc.data via tests/golden/slc_cfg1.npz)" if real is not None else "synthetic"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def get_rows(ya, yb):
        """Input rows [ya, yb) of the GLOBAL cube as a NumPy array (synthesised on the device by global index)."""
        if real is not None:
            return real["input"][ya:yb, :, None, :]
        t = torch.empty((yb - ya, nx, nt, V), dtype=torch.float32, device=dev)
        device.synth_cube_into(t, y_offset=ya, seed=42)
        return t.cpu().numpy()

    # ---- parity samples (rank 0 checks its own rows, including the seam with rank 1) ----
    seams = []
    slab_rows = 0
    if streamed:
        # the slab height the streaming layer really uses: the requested one rounded to whole kernel tiles
        slab_rows = nstream.device_slab_rows(ny, (nx, nt, V), wl["r"], fvec(wl), wl["sigma"], wl["h"], -1,
                                             semantics=sem, slab_rows=wl["slab_rows"])
    if streamed and ny > slab_rows:
        seams.append(("slab_seam", slab_rows))
    if world > 1 and ny == shard_rows:
        seams.append(("rank_seam", ny - 1))
    samples = parity_samples(wl, ny, global_rows, world, seams) if rank == 0 else []
    blocks = [None] * len(samples)
    dump = None                    # --dump-outputs: the sampled voxels and, once the last timed step ran, their values
    if args.dump_outputs:
        ys, xs, ts = dump_sample((ny, nx, nt, V), world)
        dump = {"y": ys, "idx": [torch.from_numpy(a).to(dev) for a in (ys, xs, ts)], "last_step": False,
                "values": torch.empty((len(ys), V), dtype=torch.float32, device=dev) if streamed else None}

    kev = []                       # CUDA events around every nlm kernel launch of the timed region
    plan_info = {}
    if not streamed:
        shape = (ny, nx, nt, V)
        if real is not None:
            cube = torch.from_numpy(np.ascontiguousarray(real["input"][:, :, None, :])).to(dev)
        else:
            cube = device.synth_cube(ny, nx, nt, V, y_offset=y_lo, seed=42, device=dev)
        out = torch.empty_like(cube)
        plan = device.Plan(shape, r, fv, sigma, h, -1, semantics=sem)
        shard = DistributedShard(plan, axis=0, rank=rank, world=world)
        plan_info = plan.describe()
        kernel_name, flops_per_voxel = plan.kernel_name, plan.flops_per_voxel

        def step(timed):
            shard.stage(cube)
            shard.exchange()
            if timed:
                e = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                e[0].record()
            shard.run(out)          # C-ordered (y, x, time, 4) float32: the kernels write `out` directly
            if timed:
                e[1].record()
                kev.append(e)
            shard.unstage(out)      # (a no-op then)

        def collect_blocks():
            for i, s in enumerate(samples):
                blocks[i] = out[s["y"][0]:s["y"][1], s["x"][0]:s["x"][1], s["t"][0]:s["t"][1]].cpu().numpy()
        flag_of = lambda: int(shard.flag.item())
    else:
        inner = (nx, nt, V)
        mk = lambda: torch.empty((halo,) + inner, dtype=torch.float32, device=dev)
        send_lo, recv_lo = (mk(), mk()) if rank > 0 else (None, None)
        send_hi, recv_hi = (mk(), mk()) if rank < world - 1 else (None, None)
        own_hi = mk() if ny < shard_rows else None          # partial sweep: the rows above are this rank's own
        state = {"timed": False, "checksum": None, "plan": None}

        def source(lo, hi, dst):
            device.synth_cube_into(dst, y_offset=y_lo + lo, seed=42)

        def sink(lo, hi, res):
            c = res[::max(1, (hi - lo) // 4)].sum(dtype=torch.float64)
            state["checksum"] = c if state["checksum"] is None else state["checksum"] + c
            for i, s in enumerate(samples):
                a, b = max(lo, s["y"][0]), min(hi, s["y"][1])
                if a < b:
                    if blocks[i] is None:
                        blocks[i] = torch.zeros((s["y"][1] - s["y"][0], s["x"][1] - s["x"][0], s["t"][1] - s["t"][0], V),
                                                dtype=torch.float32, device=dev)
                    blocks[i][a - s["y"][0]:b - s["y"][0]] = res[a - lo:b - lo, s["x"][0]:s["x"][1], s["t"][0]:s["t"][1]]
            if dump is not None and dump["last_step"]:          # the slabs are not kept: gather while they pass
                a, b = np.searchsorted(dump["y"], (lo, hi))
                y, x, t = (i[a:b] for i in dump["idx"])
                dump["values"][a:b] = res[y - lo, x, t]

        def on_kernel(before, plan):
            state["plan"] = plan
            if state["timed"]:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                if before:
                    kev.append([e, None])
                else:
                    kev[-1][1] = e

        def step(timed):
            state["timed"] = timed
            # halo rows of the shard edges travel between neighbouring ranks (raw input rows, NCCL send/recv)
            if send_lo is not None:
                device.synth_cube_into(send_lo, y_offset=y_lo, seed=42)
            if send_hi is not None:
                device.synth_cube_into(send_hi, y_offset=y_lo + shard_rows - halo, seed=42)
            if world > 1:
                exchange_halos_dist(send_lo, send_hi, recv_lo, recv_hi, rank, world)
            hi_rows = recv_hi
            if own_hi is not None:
                device.synth_cube_into(own_hi, y_offset=y_lo + ny, seed=42)
                hi_rows = own_hi
            nstream.apply_device_streamed(source, sink, ny, inner, r, fv, sigma, h, -1, semantics=sem,
                                          slab_rows=wl["slab_rows"], lo_rows=recv_lo, hi_rows=hi_rows, on_kernel=on_kernel)

        def collect_blocks():
            for i in range(len(blocks)):
                blocks[i] = blocks[i].cpu().numpy()
        flag_of = lambda: 0

    for _ in range(args.warmup):
        step(False)
    barrier()
    if streamed:
        kernel_name, flops_per_voxel = state["plan"].kernel_name, state["plan"].flops_per_voxel
        plan_info = state["plan"].describe()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = device.launch_count()
    barrier()
    e0.record()
    for i in range(args.steps):
        if dump is not None:
            dump["last_step"] = i == args.steps - 1
        step(True)
    e1.record()
    barrier()
    launches = device.launch_count() - launches0
    ms_total = e0.elapsed_time(e1)
    kernel_ms = sum(a.elapsed_time(b) for a, b in kev) / args.steps
    kernel_launches_per_step = len(kev) // args.steps
    clocks = sampler.stop() if rank == 0 else None
    flag = flag_of()
    if dump is not None:
        if not streamed:
            dump["values"] = out[tuple(dump["idx"])]
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, ("out" if world == 1 else "out_rank%d" % rank) + ".npy"),
                dump["values"].cpu().numpy())
        dump = None

    t = torch.tensor([ms_total, kernel_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, kernel_ms = float(t[0]), float(t[1])
    ms_per_step = ms_total / args.steps
    vox_rank = ny * nx * nt
    value = world * vox_rank / (ms_per_step * 1e-3) / 1e6

    # ---- in-run parity (rank 0) ----
    parity = None
    if rank == 0 and not args.no_parity:
        collect_blocks()
        try:
            parity = check_parity(wl, samples, blocks, get_rows, global_rows, sem)
            if real is not None:           # the whole image against the reference's own output
                key = "out_as_written" if sem == "as_written" else "out_compiled"
                ref_full = real[key][:, :, None, :]
                got = out.cpu().numpy()
                e = max(float(np.abs(got[..., v] - ref_full[..., v]).max() / np.abs(ref_full[..., v]).max()) for v in range(V))
                parity["full_image_vs_reference_output"] = e
                parity["max_scaled_err"] = max(parity["max_scaled_err"], e)
                parity["ok"] = bool(parity["max_scaled_err"] <= PARITY_TOL)
        except Exception as e:                                   # a broken checker must not pass silently
            parity = {"max_scaled_err": None, "tolerance": PARITY_TOL, "ok": False, "error": repr(e)}

    # ---- e2e: the reference-facing entry point on pinned HOST arrays, every step H2D + kernels + D2H ----
    e2e = None
    if not args.no_e2e:
        if not streamed:
            del shard, out, cube
        torch.cuda.empty_cache()
        row_bytes = nx * nt * V * 4
        e2e_rows = ny if not streamed else min(ny, max(4 * halo + 16, (6 << 30) // row_bytes))
        try:
            import psutil
            avail = psutil.virtual_memory().available
            if 2.2 * e2e_rows * row_bytes * max(world, 1) > 0.6 * avail:
                e2e_rows = max(4 * halo + 16, int(0.6 * avail / (2.2 * row_bytes * world)))
        except Exception:
            pass
        # N > 1: like the reference's own njobs mechanism (xr_split, nd/utils.py:305-310) every rank's host
        # chunk carries a buffer of r+f rows of its neighbours; only the interior rows count as work.
        lo_buf = halo if rank > 0 else 0
        hi_buf = halo if rank < world - 1 else 0
        tot_rows = e2e_rows + lo_buf + hi_buf
        h_in = torch.empty((tot_rows, nx, nt, V), dtype=torch.float32, pin_memory=True)
        h_out = torch.empty((tot_rows, nx, nt, V), dtype=torch.float32, pin_memory=True)
        if real is not None:
            h_in.copy_(torch.from_numpy(np.ascontiguousarray(real["input"][:, :, None, :])))
        else:
            chunk = max(1, (1 << 30) // row_bytes)
            for a in range(0, tot_rows, chunk):
                b = min(a + chunk, tot_rows)
                src = torch.empty((b - a, nx, nt, V), dtype=torch.float32, device=dev)
                device.synth_cube_into(src, y_offset=y_lo - lo_buf + a, seed=42)
                h_in[a:b].copy_(src)
                del src
        a_in, a_out = h_in.numpy(), h_out.numpy()
        r3 = np.array(r, dtype=np.uint32)
        f3 = np.array(fv, dtype=np.uint32)
        e2e_steps = max(1, min(args.steps, 3))

        def timed_e2e(fn):
            fn()                                                       # warm-up
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                fn()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt[0])

        dt = timed_e2e(lambda: _pixelwise_nlmeans_3d(a_in, a_out, r3, f3, sigma, h, -1, semantics=sem))
        checksum = float(np.float64(a_out[lo_buf:lo_buf + e2e_rows:max(1, e2e_rows // 64)].sum()))
        ebytes = tot_rows * row_bytes
        e2e = {"value": world * e2e_rows * nx * nt * e2e_steps / dt / 1e6, "unit": UNIT,
               "h2d_bytes_per_step": ebytes, "d2h_bytes_per_step": ebytes, "rows_per_gpu": e2e_rows,
               "steps": e2e_steps, "api": "nd_b200._filters._pixelwise_nlmeans_3d(host arr, host output, r, f, sigma, h, n_eff)",
               "cpus_bound_to_gpu": numa,
               "note": "rank-local host chunk incl. r+f buffer rows of its neighbours (the reference's xr_split rule); "
                       "slab-pipelined H2D / kernels / D2H on three streams; only interior rows are counted",
               "checksum": checksum}
        if nstream.can_pipeline(a_in, a_out) and halo * 8 <= a_in.shape[0] and a_in.nbytes >= (256 << 20):
            # the same slabs, streams and copies without the kernels: the host-memory / PCIe ceiling of this pipeline
            dtc = timed_e2e(lambda: nstream.apply_host_pipelined(a_in, a_out, r, fv, sigma, h, -1, semantics=sem,
                                                                 copy_only=True))
            e2e["host_ceiling_mvoxel_s"] = world * e2e_rows * nx * nt * e2e_steps / dtc / 1e6
            e2e["host_ceiling_gbs_each_way"] = world * ebytes * e2e_steps / dtc / 1e9
            e2e["frac_of_host_ceiling"] = e2e["value"] / e2e["host_ceiling_mvoxel_s"]
            e2e["host_ceiling_note"] = ("copy-only run of the same slab pipeline (H2D + device copy + D2H, no kernels) on "
                                        "all ranks at once: what the host memory system and PCIe allow")

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel ----
    fp32_nominal = 148 * 128 * 2 * pk["sm_max_mhz"] * 1e6 / 1e12           # TFLOP/s, SMs*lanes*2*clock
    try:
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        fp32_nominal = sms * 128 * 2 * pk["sm_max_mhz"] * 1e6 / 1e12
    except Exception:
        pass
    alg_bytes = 8.0 * V * vox_rank
    hbm_view = {"algorithmic_bytes_per_step": alg_bytes, "achieved_gbs": alg_bytes / (kernel_ms * 1e-3) / 1e9,
                "peak_gbs": pk["hbm_gbs"], "frac": alg_bytes / (kernel_ms * 1e-3) / 1e9 / pk["hbm_gbs"]}
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if tj.get("workload") == name and tj.get("rows") == ny and sem == "as_written":
                traffic = tj.get("dram_bytes_per_launch")
                traffic_src = "profiles/traffic.json (static: read from the committed ncu --set full capture %s, not measured in this run)" % tj.get("source", "")
        except Exception:
            pass
    box_mean = sem == "reference_compiled" and any(fv)
    if box_mean:
        # reference_compiled with f > 0 is a reflect box mean (SURVEY.md F1): HBM-bound, 8V bytes per voxel
        roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": hbm_view["achieved_gbs"], "peak": pk["hbm_gbs"],
                    "unit": "GB/s", "frac": hbm_view["frac"], "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": "hbm_gbs (%s)" % pk["source"], "kernel_ms": kernel_ms,
                    "kernel_launches_per_step": kernel_launches_per_step,
                    "algorithmic_bytes_per_voxel": 8 * V}
    else:
        achieved = flops_per_voxel * vox_rank / (kernel_ms * 1e-3) / 1e12
        fp32_measured = device.measure_fp32_peak(0.5)
        roofline = {"bound": "fp32_fma", "kernel": kernel_name, "achieved": achieved, "peak": fp32_nominal,
                    "unit": "TFLOP/s", "frac": achieved / fp32_nominal, "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": "SMs*128*2*sm_max_mhz (%s): nominal FP32 FMA peak, the binding roofline of this path "
                                   "(SURVEY.md 8(d)); no tensor cores" % pk["source"],
                    "kernel_ms": kernel_ms, "kernel_launches_per_step": kernel_launches_per_step,
                    "flops_per_voxel": flops_per_voxel,
                    "fp32_fma_peak_measured_same_run": fp32_measured, "frac_of_measured_fma_peak": achieved / fp32_measured,
                    "hbm": hbm_view}

    cpu = None
    if world == 1 and not args.no_cpu:
        try:
            cpu = cpu_baseline(wl, sem)
        except Exception as e:                                   # never lose the GPU line to the CPU leg
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "unavailable", "sample": repr(e)}

    config = {"workload": name, "description": wl["text"], "rows_per_gpu": ny, "global_shape": [global_rows, nx, nt, V],
              "r": list(r), "f": list(fv), "sigma": sigma, "h": h, "semantics": sem,
              "sharding": ("y-sharded, halo r_y+f_y=%d rows, NCCL send/recv" % halo) if world > 1 else "single GPU",
              "l2": "inputs (%.1f GB per GPU) are larger than L2, no flush needed" % (alg_bytes / 2e9)
                    if alg_bytes / 2 > 126e6 else "input %.1f MB fits in L2 (tiny reference-sized workload)" % (alg_bytes / 2e6),
              "plan": plan_info}
    if streamed:
        config["streaming"] = {"slab_rows": slab_rows, "slabs_per_step": kernel_launches_per_step,
                               "source": "each slab is synthesised on the device by global index inside the timed region",
                               "checksum": float(state["checksum"].item()) if state["checksum"] is not None else None}
        config["sweep"] = {"rows_per_gpu_processed": ny, "rows_per_gpu_total": shard_rows,
                           "fraction": ny / shard_rows,
                           "note": "value counts the processed rows only" if ny < shard_rows else "full shard"}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": data_kind, "config": config,
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "parity": parity,
            "cpu_baseline": cpu, "kernel_flag": flag}
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        sys.stderr.write("PARITY FAILURE: %s\n" % json.dumps(parity))
        return 3
    return 0


# ------------------------------------------------------------------------------------------------
# the Dataset-level public API on N GPUs of one process: NLMeansFilter(...).apply(ds, njobs=N)
# ------------------------------------------------------------------------------------------------
def run_apply_njobs(args):
    import numpy as np
    import torch
    from nd_b200 import device
    from nd_b200.dataset import Dataset
    from nd_b200.filters import NLMeansFilter
    n = args.apply_njobs
    wl = WORKLOADS[args.workload]
    nx, nt, V, r = wl["nx"], wl["nt"], wl["V"], wl["r"]
    ny = (args.rows if args.rows else wl.get("rows", 1024)) * n
    names = ["C11", "C12__re", "C12__im", "C22", "C33", "C13__re"][:V]
    torch.cuda.set_device(0)
    chunk = max(1, (1 << 30) // (nx * nt * V * 4))
    planes = [np.empty((ny, nx, nt), dtype=np.float32) for _ in range(V)]
    for a in range(0, ny, chunk):
        b = min(a + chunk, ny)
        t = device.synth_cube(b - a, nx, nt, V, y_offset=a).cpu().numpy()
        for v in range(V):
            planes[v][a:b] = t[..., v]
    ds = Dataset({nm: (("y", "x", "time"), planes[v]) for v, nm in enumerate(names)},
                 coords={"y": np.arange(ny), "x": np.arange(nx), "time": np.arange(nt)})
    flt = NLMeansFilter(dims=("y", "x", "time"), r=r, sigma=wl["sigma"], h=wl["h"], f=wl["f"])
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        out = flt.apply(ds, njobs=n)
        for d in range(n):
            torch.cuda.synchronize(d)
        if it >= args.warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    line = {"metric": METRIC + " through NLMeansFilter.apply(ds, njobs=N)", "value": ny * nx * nt / dt / 1e6, "unit": UNIT,
            "n_gpus": n, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "global_shape": [ny, nx, nt, V], "api": "nd_b200.filters.NLMeansFilter"
                       "(dims=('y','x','time'), r, sigma, h, f).apply(Dataset, njobs=%d): host Dataset in, host Dataset out" % n},
            "checksum": float(np.float64(out[names[0]].values[::max(1, ny // 64)].sum()))}
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--semantics", default="as_written", choices=["as_written", "reference_compiled"])
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU actually processed (cfg4/cfg5: partial sweep)")
    ap.add_argument("--global-rows", type=int, default=0,
                    help="development: height of the global cube of a streamed workload (default: the configuration's)")
    ap.add_argument("--apply-njobs", type=int, default=0, help="bench NLMeansFilter.apply(ds, njobs=N) in one process")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/*.npy (float32, at most 48 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.apply_njobs or args.impl == "reference"):
        ap.error("--dump-outputs writes the results of --impl ours")
    if args.apply_njobs:
        return run_apply_njobs(args)
    if args.impl == "reference":
        return run_reference(args)
    if WORKLOADS[args.workload]["mode"] != "streamed":
        args.warmup = max(args.warmup, 3)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
