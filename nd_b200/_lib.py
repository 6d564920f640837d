"""
ctypes binding of libndnlm.so (include/ndnlm.h) -- the C-ABI CUDA library that replaces
`nd._filters._pixelwise_nlmeans_3d` (reference nd/_filters.pyx:317-420).

There is NO fallback: if the library has not been built, importing the compute path raises.
Build it with `python -c "import __graft_entry__ as g; g.build()"` (nvcc, sm_100a).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NDNLM_LIB") or os.path.join(_HERE, "libndnlm.so")   # NDNLM_LIB: tuning builds only

OK, EINVAL, EDTYPE, ECUDA, ENOSOLUTION, ERADIUS = 0, -1, -2, -3, -4, -5
WUNDERFLOW = 1
FLAG_NOSOLUTION, FLAG_UNDERFLOW = 1, 2
F32, F64 = 0, 1
AS_WRITTEN, REFERENCE_COMPILED = 0, 1
KERNEL_AUTO, KERNEL_GENERIC, KERNEL_TILED = 0, 1, 2
EDGE_REFLECT, EDGE_HALO, EDGE_SOURCE = 0, 1, 2

SEMANTICS = {"as_written": AS_WRITTEN, "reference_compiled": REFERENCE_COMPILED}
KERNEL_TILED_F64 = 3
KERNELS = {"auto": KERNEL_AUTO, "generic": KERNEL_GENERIC, "tiled": KERNEL_TILED, "tiled64": KERNEL_TILED_F64}

# every symbol include/ndnlm.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "ndnlm_plan_create", "ndnlm_plan_create_roles", "ndnlm_plan_destroy", "ndnlm_plan_info", "ndnlm_stage", "ndnlm_halo_bytes",
    "ndnlm_halo_pack", "ndnlm_halo_unpack", "ndnlm_run", "ndnlm_run_scratch", "ndnlm_scratch_bytes", "ndnlm_unstage", "ndnlm_output_is_native", "ndnlm_workspace_bytes",
    "ndnlm_apply", "ndnlm_synth_cube", "ndnlm_measure_fp32_peak", "ndnlm_launch_count", "ndnlm_last_error", "ndnlm_version",
]
# every symbol include/ndflt.h declares (sibling filters, SURVEY.md 8(f) row N2)
FLT_SYMBOLS = ["ndflt_correlate", "ndflt_correlate1d", "ndflt_launch_count", "ndflt_last_error"]
# every symbol include/ndchg.h declares (omnibus change detection, SURVEY.md 8(f) row N4)
CHG_SYMBOLS = ["ndchg_change_detection", "ndchg_omnibus_probability", "ndchg_change_detection_pol",
               "ndchg_omnibus_probability_pol", "ndchg_change_direction", "ndchg_enl", "ndchg_refined_lee",
               "ndchg_h_a_alpha", "ndchg_last_error"]


class Info(ctypes.Structure):
    _fields_ = [
        ("kernel", ctypes.c_int32),
        ("role_axis", ctypes.c_int32 * 3),
        ("n", ctypes.c_int32 * 3),
        ("pad", ctypes.c_int32 * 3),
        ("padded", ctypes.c_int32 * 3),
        ("vp", ctypes.c_int32),
        ("tile", ctypes.c_int32 * 3),
        ("box", ctypes.c_int32 * 3),
        ("warps", ctypes.c_int32 * 3),
        ("threads", ctypes.c_int32),
        ("grid", ctypes.c_int32),
        ("smem_bytes", ctypes.c_int32),
        ("elem_bytes", ctypes.c_int32),
        ("n_offsets", ctypes.c_int64),
        ("voxels", ctypes.c_int64),
        ("flops_per_voxel", ctypes.c_double),
        ("padded_bytes", ctypes.c_size_t),
        ("out_bytes", ctypes.c_size_t),
        ("kernel_name", ctypes.c_char * 96),
    ]


_lib = None


def lib():
    """Load libndnlm.so (once).  Raises ImportError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "nd_b200: %s is missing -- the CUDA library has not been built and there is no CPU "
            "fallback.  Run `python -c \"import __graft_entry__ as g; g.build()\"`." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i64p, u32p = ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_uint32)
    L.ndnlm_plan_create.argtypes = [ctypes.POINTER(vp), i64p, u32p, u32p, ctypes.c_double, ctypes.c_double,
                                    ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    L.ndnlm_plan_create.restype = ctypes.c_int
    L.ndnlm_plan_create_roles.argtypes = [ctypes.POINTER(vp), i64p, u32p, u32p, ctypes.c_double, ctypes.c_double,
                                          ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                          ctypes.POINTER(ctypes.c_int32)]
    L.ndnlm_plan_create_roles.restype = ctypes.c_int
    L.ndnlm_plan_destroy.argtypes = [vp]
    L.ndnlm_plan_destroy.restype = None
    L.ndnlm_plan_info.argtypes = [vp, ctypes.POINTER(Info)]
    L.ndnlm_plan_info.restype = ctypes.c_int
    L.ndnlm_stage.argtypes = [vp, vp, i64p, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp]
    L.ndnlm_stage.restype = ctypes.c_int
    L.ndnlm_halo_bytes.argtypes = [vp, ctypes.c_int]
    L.ndnlm_halo_bytes.restype = ctypes.c_size_t
    L.ndnlm_halo_pack.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, vp, vp]
    L.ndnlm_halo_pack.restype = ctypes.c_int
    L.ndnlm_halo_unpack.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, vp, vp]
    L.ndnlm_halo_unpack.restype = ctypes.c_int
    L.ndnlm_run.argtypes = [vp, vp, vp, vp, vp]
    L.ndnlm_run.restype = ctypes.c_int
    L.ndnlm_run_scratch.argtypes = [vp, vp, vp, vp, vp, vp]
    L.ndnlm_run_scratch.restype = ctypes.c_int
    L.ndnlm_scratch_bytes.argtypes = [vp]
    L.ndnlm_scratch_bytes.restype = ctypes.c_size_t
    L.ndnlm_unstage.argtypes = [vp, vp, vp, i64p, vp]
    L.ndnlm_unstage.restype = ctypes.c_int
    L.ndnlm_output_is_native.argtypes = [vp, i64p]
    L.ndnlm_output_is_native.restype = ctypes.c_int
    L.ndnlm_workspace_bytes.argtypes = [vp]
    L.ndnlm_workspace_bytes.restype = ctypes.c_size_t
    L.ndnlm_apply.argtypes = [vp, vp, i64p, vp, i64p, vp, vp]
    L.ndnlm_apply.restype = ctypes.c_int
    L.ndnlm_synth_cube.argtypes = [vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32,
                                   ctypes.c_int64, ctypes.c_uint64, vp]
    L.ndnlm_synth_cube.restype = ctypes.c_int
    L.ndnlm_measure_fp32_peak.argtypes = [ctypes.POINTER(ctypes.c_double), ctypes.c_double, ctypes.c_int, vp]
    L.ndnlm_measure_fp32_peak.restype = ctypes.c_int
    L.ndnlm_launch_count.argtypes = []
    L.ndnlm_launch_count.restype = ctypes.c_int64
    L.ndnlm_last_error.argtypes = []
    L.ndnlm_last_error.restype = ctypes.c_char_p
    L.ndnlm_version.argtypes = []
    L.ndnlm_version.restype = ctypes.c_char_p
    dp = ctypes.POINTER(ctypes.c_double)
    L.ndflt_correlate.argtypes = [vp, vp, i64p, i64p, i64p, ctypes.c_int, dp, i64p, i64p, ctypes.c_int, ctypes.c_double, vp]
    L.ndflt_correlate.restype = ctypes.c_int
    L.ndflt_correlate1d.argtypes = [vp, vp, i64p, i64p, i64p, ctypes.c_int, ctypes.c_int, dp, ctypes.c_int64,
                                    ctypes.c_int64, ctypes.c_int, ctypes.c_double, vp]
    L.ndflt_correlate1d.restype = ctypes.c_int
    L.ndflt_launch_count.argtypes = []
    L.ndflt_launch_count.restype = ctypes.c_int64
    L.ndflt_last_error.argtypes = []
    L.ndflt_last_error.restype = ctypes.c_char_p
    L.ndchg_change_detection.argtypes = [vp, i64p, i64p, ctypes.c_int, vp, ctypes.c_double, ctypes.c_uint32, vp]
    L.ndchg_change_detection.restype = ctypes.c_int
    L.ndchg_omnibus_probability.argtypes = [vp, i64p, i64p, ctypes.c_int, vp, ctypes.c_uint32, vp]
    L.ndchg_omnibus_probability.restype = ctypes.c_int
    L.ndchg_change_detection_pol.argtypes = [vp, i64p, i64p, ctypes.c_int, ctypes.c_int, vp, ctypes.c_double,
                                             ctypes.c_uint32, vp]
    L.ndchg_change_detection_pol.restype = ctypes.c_int
    L.ndchg_omnibus_probability_pol.argtypes = [vp, i64p, i64p, ctypes.c_int, ctypes.c_int, vp, ctypes.c_uint32, vp]
    L.ndchg_omnibus_probability_pol.restype = ctypes.c_int
    L.ndchg_change_direction.argtypes = [vp, i64p, i64p, ctypes.c_int, ctypes.c_int, vp, ctypes.c_double, ctypes.c_uint32, vp]
    L.ndchg_change_direction.restype = ctypes.c_int
    L.ndchg_enl.argtypes = [vp, i64p, i64p, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, vp, vp]
    L.ndchg_enl.restype = ctypes.c_int
    L.ndchg_refined_lee.argtypes = [vp, i64p, i64p, ctypes.c_int, ctypes.c_int, ctypes.c_uint32, ctypes.c_double, vp, vp]
    L.ndchg_refined_lee.restype = ctypes.c_int
    L.ndchg_h_a_alpha.argtypes = [vp, i64p, i64p, ctypes.c_int, ctypes.c_int, vp, vp]
    L.ndchg_h_a_alpha.restype = ctypes.c_int
    L.ndchg_last_error.argtypes = []
    L.ndchg_last_error.restype = ctypes.c_char_p
    _lib = L
    return L


def check(rc):
    """Map a C return code onto the exception the reference raises in the same situation."""
    if rc == OK:
        return
    msg = lib().ndnlm_last_error().decode("utf-8", "replace")
    if rc == WUNDERFLOW:
        import warnings
        warnings.warn("ndnlm: " + msg, RuntimeWarning, stacklevel=3)
        return
    if rc == EDTYPE:
        raise TypeError(msg)                      # reference: "No matching signature found"
    if rc == ENOSOLUTION:
        raise ValueError("No solution")           # reference nd/_filters.pyx:310-311
    if rc in (EINVAL, ERADIUS):
        raise ValueError(msg)
    raise RuntimeError("ndnlm: " + msg)


def check_flag(value):
    """The device error flag of ndnlm_run (a bit mask) -> the reference's exception / a warning."""
    value = int(value)
    if value & FLAG_NOSOLUTION:
        raise ValueError("No solution")           # reference nd/_filters.pyx:310-311
    if value & FLAG_UNDERFLOW:
        import warnings
        warnings.warn("ndnlm: at some voxels every neighbour weight is below the float32 range (< 2^-126); they were "
                      "left unfiltered (use float64 data or a larger h)", RuntimeWarning, stacklevel=3)


def i64(values):
    return (ctypes.c_int64 * len(values))(*[int(v) for v in values])


def u32(values):
    return (ctypes.c_uint32 * len(values))(*[int(v) for v in values])
