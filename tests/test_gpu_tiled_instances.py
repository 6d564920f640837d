"""
Every instantiation of the tiled NLM kernel (nd_b200/csrc/nlm_tiled.cuh, listed in instances_g0.inc .. instances_g7.inc)
at geometries that select it, against the C oracle and bit for bit against every sibling instantiation the planner
accepts there.

The planner (configure_tiled in ndnlm.cu) takes the first instantiation whose shared-memory box fits, so the user's
r, f, V, dtype and n_eff decide which one runs; a larger search radius quietly moves a user to a fallback.  `TABLE`
has one entry per instantiation, written from the instantiation macros, with one or two *selecting geometries*
(shape, r, f, n_eff, env) under which the default planner picks exactly that kernel, and the `[passes=N]` count and
`info.tile` it plans there.  Between them the geometries have
  * a tail tile on each of the three axes (an extent that is not a multiple of the tile, with at least one seam),
  * two or more W passes with a short last pass, wherever the instantiation can run several passes by default,
  * a minimal extent r + f = N - 1 on some axis, so that the reflection reaches both ends,
  * V = 3 (one zero lane), V = 5 and 6 (half-group kernels), V = 7 and 8 (two full groups),
  * for the 2-D / batch-axis kernels (f_W = 0) a W extent of 1 and one greater than 1: their W rows per CTA come
    from a divisor search over that extent.
Eight instantiations sit behind an earlier candidate with a strictly smaller box and are never selected by default;
they are `UNREACHABLE` and run only when forced with NDNLM_TILED_VARIANT.

  * CPU: the table equals the nlm_tiled_kernel instantiations in the built libndnlm.so; the planner selects each
    reachable entry at its geometries with the claimed passes and tiles; a search grid selects no unreachable entry.
  * GPU: each reachable entry against the oracle (float64 below 1e-12, float32 below 5e-6), and every other
    instantiation the planner accepts at the same geometry (forced with NDNLM_TILED_VARIANT) equal to it bit for
    bit.  The kernel's sums are direct, in a fixed order, and do not depend on where a tile or a W pass starts, so
    half- and full-group kernels, L = 2 .. 8, every CH, 4 .. 16 warps, double-duty halo warps and persistent CTAs
    must all give the same bits.
"""
import itertools
import os
import re
import shutil
import subprocess
from collections import namedtuple

import numpy as np
import pytest

from helpers import sar_like, scaled_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "nd_b200", "libndnlm.so")
PLANNER_ENV = ("NDNLM_DH", "NDNLM_PERSIST", "NDNLM_TILED_VARIANT")
TOL32 = 5e-6       # the bound test_gpu_parity applies to float64 data on the float32 tiled kernel
TOL64 = 1e-12

# A selecting geometry: the default planner (with `env`, which may only set NDNLM_DH / NDNLM_PERSIST) picks the
# entry's kernel for (shape, r, f, n_eff), in `passes` W passes on tiles of `tile` = (W, R, X) voxels.
G = namedtuple("G", "shape r f passes tile n_eff env")
G.__new__.__defaults__ = (-1.0, None)
UNREACHABLE = namedtuple("UNREACHABLE", "reason")

_FLAGS = {"INST": ("float", "", False, False, False), "INSTH": ("float", "(half)", True, False, False),
          "INST64": ("double", "", False, False, False), "INSTD": ("float", "(dh)", False, True, False),
          "INSTD64": ("double", "(dh)", False, True, False), "INSTP": ("float", "(persist)", False, False, True)}


class E:
    """One TILED_<macro>(NV4, FW, FX, FR, L, NWARPS, CH, NEFF) line of instances_g<group>.inc."""

    def __init__(self, group, macro, nv4, fw, fx, fr, L, nw, ch, neff, geoms):
        self.group, self.macro, self.args = group, macro, (nv4, fw, fx, fr, L, nw, ch, neff)
        t, tag, half, dh, persist = _FLAGS[macro]
        self.dtype = np.float64 if t == "double" else np.float32
        self.unreachable = geoms.reason if isinstance(geoms, UNREACHABLE) else None
        self.geoms = [] if self.unreachable else geoms
        # the kernel_name the planner prints (ndnlm.cu, g_tiled), without its [passes=N]
        self.name = "nlm_tiled<%snv4=%d%s,f=(%d,%d,%d),L=%d,warps=%d%s,ch=%d,neff=%s>" % (
            "double," if t == "double" else "", nv4, "(half)" if half else "", fw, fr, fx, L, nw,
            "" if half else tag, ch, "true" if neff else "false")
        # the kernel function in libndnlm.so (nlm_tiled_kernel<T, NV4, FW, FX, FR, L, NWARPS, CH, NEFF, HALF, DH, PERSIST>)
        self.symbol = "ndnlm::nlm_tiled_kernel<%s,%d,%d,%d,%d,%d,%d,%d,%s>" % (
            t, nv4, fw, fx, fr, L, nw, ch, ",".join("true" if b else "false" for b in (neff, half, dh, persist)))

    def __repr__(self):
        return "g%d:%s%s" % (self.group, self.macro, self.args)


_BEHIND_4W = "behind the 4-warp kernel of the same pattern, whose box is smaller and which retries at the full 227 KB"
TABLE = [
    E(0, "INST", 1, 1, 1, 1, 4, 16, 5, False, [G((21, 5, 33, 3), (6, 3, 1), (1, 1, 1), 2, (14, 4, 30)),
                                               G((8, 5, 5, 4), (6, 3, 1), (1, 1, 1), 2, (14, 4, 30))]),
    E(0, "INST", 1, 1, 1, 1, 4, 16, 5, True, [G((21, 5, 33, 3), (6, 3, 1), (1, 1, 1), 2, (14, 4, 30), 6.0),
                                              G((8, 5, 5, 4), (6, 3, 1), (1, 1, 1), 2, (14, 4, 30), 6.0)]),
    E(1, "INST", 1, 1, 1, 1, 4, 12, 5, False, [G((15, 10, 33, 3), (3, 8, 1), (1, 1, 1), 2, (10, 4, 30)),
                                               G((5, 10, 10, 4), (3, 8, 1), (1, 1, 1), 2, (10, 4, 30))]),
    E(1, "INST", 1, 1, 1, 1, 6, 12, 5, False, UNREACHABLE("behind the L = 4 12-warp kernel, whose box is smaller")),
    E(1, "INST", 1, 1, 1, 1, 4, 8, 5, False, [G((9, 10, 33, 3), (2, 8, 8), (1, 1, 1), 2, (6, 4, 30)),
                                              G((4, 10, 10, 4), (2, 8, 8), (1, 1, 1), 2, (6, 4, 30))]),
    E(1, "INST", 1, 1, 1, 1, 4, 8, 5, True, [G((9, 10, 33, 3), (5, 8, 1), (1, 1, 1), 2, (6, 4, 30), 6.0),
                                             G((7, 10, 10, 4), (5, 8, 1), (1, 1, 1), 2, (6, 4, 30), 6.0)]),
    E(2, "INST", 1, 0, 1, 1, 4, 4, 7, False, [G((6, 7, 33, 3), (5, 1, 1), (0, 1, 1), 2, (4, 4, 30)),
                                              G((3, 5, 61, 4), (0, 1, 1), (0, 1, 1), 1, (2, 4, 60))]),
    E(2, "INST", 1, 0, 1, 1, 4, 4, 7, True, [G((6, 7, 33, 3), (5, 1, 1), (0, 1, 1), 2, (4, 4, 30), 6.0),
                                             G((1, 5, 121, 4), (0, 1, 1), (0, 1, 1), 1, (1, 4, 120), 6.0)]),
    E(2, "INST", 1, 0, 1, 1, 8, 8, 5, False, UNREACHABLE(_BEHIND_4W)),
    E(2, "INST", 1, 0, 1, 1, 8, 8, 5, True, UNREACHABLE(_BEHIND_4W)),
    E(2, "INST", 1, 0, 1, 0, 4, 4, 7, False, [G((6, 5, 33, 3), (3, 4, 1), (0, 0, 1), 2, (4, 4, 30)),
                                              G((3, 5, 61, 4), (0, 4, 1), (0, 0, 1), 1, (2, 4, 60))]),
    E(2, "INST", 1, 0, 1, 0, 8, 8, 5, False, UNREACHABLE(_BEHIND_4W)),
    E(2, "INST", 1, 0, 0, 0, 4, 4, 7, False, [G((6, 5, 35, 3), (3, 4, 1), (0, 0, 0), 2, (4, 4, 32)),
                                              G((1, 5, 129, 4), (0, 4, 1), (0, 0, 0), 1, (1, 4, 128))]),
    E(2, "INST", 1, 0, 0, 0, 8, 8, 5, False, UNREACHABLE(_BEHIND_4W)),
    E(3, "INST", 1, 2, 2, 2, 6, 12, 5, False, [G((12, 10, 31, 3), (1, 7, 1), (2, 2, 2), 2, (8, 6, 28)),
                                               G((4, 10, 10, 4), (1, 7, 1), (2, 2, 2), 2, (8, 6, 28))]),
    E(3, "INST", 1, 2, 2, 2, 4, 12, 5, False, [G((12, 11, 31, 3), (1, 8, 2), (2, 2, 2), 2, (8, 4, 28)),
                                               G((4, 11, 11, 4), (1, 8, 2), (2, 2, 2), 2, (8, 4, 28))]),
    E(3, "INST", 1, 2, 2, 2, 4, 8, 5, False, [G((6, 10, 31, 1), (2, 7, 8), (2, 2, 2), 2, (4, 4, 28)),
                                              G((5, 10, 11, 4), (2, 7, 8), (2, 2, 2), 2, (4, 4, 28))]),
    E(3, "INST", 1, 0, 2, 2, 8, 8, 5, False, [G((12, 9, 31, 3), (5, 6, 1), (0, 2, 2), 2, (8, 8, 28)),
                                              G((1, 17, 113, 4), (0, 6, 1), (0, 2, 2), 1, (1, 16, 112))]),
    E(3, "INST", 1, 2, 2, 2, 4, 12, 5, True, [G((12, 11, 31, 3), (1, 8, 2), (2, 2, 2), 2, (8, 4, 28), 6.0),
                                              G((4, 11, 11, 4), (1, 8, 2), (2, 2, 2), 2, (8, 4, 28), 6.0)]),
    E(3, "INST", 1, 0, 2, 2, 8, 8, 5, True, [G((12, 9, 31, 3), (5, 6, 1), (0, 2, 2), 2, (8, 8, 28), 6.0),
                                             G((1, 17, 113, 4), (0, 6, 1), (0, 2, 2), 1, (1, 16, 112), 6.0)]),
    E(3, "INSTH", 2, 1, 1, 1, 4, 12, 5, False, [G((15, 5, 33, 5), (1, 3, 2), (1, 1, 1), 2, (10, 4, 30)),
                                                G((3, 5, 5, 6), (1, 3, 2), (1, 1, 1), 2, (10, 4, 30))]),
    E(3, "INSTH", 2, 1, 1, 1, 4, 8, 5, False, [G((9, 7, 33, 5), (2, 5, 1), (1, 1, 1), 2, (6, 4, 30)),
                                               G((4, 7, 7, 6), (2, 5, 1), (1, 1, 1), 2, (6, 4, 30))]),
    E(3, "INST", 2, 1, 1, 1, 4, 8, 5, False, [G((9, 5, 33, 7), (4, 3, 1), (1, 1, 1), 2, (6, 4, 30)),
                                              G((6, 5, 5, 8), (4, 3, 1), (1, 1, 1), 2, (6, 4, 30))]),
    E(3, "INSTH", 2, 0, 1, 1, 4, 8, 5, False, [G((12, 5, 33, 5), (5, 3, 1), (0, 1, 1), 2, (8, 4, 30)),
                                               G((3, 5, 121, 6), (0, 3, 1), (0, 1, 1), 1, (2, 4, 120))]),
    E(3, "INST", 2, 0, 1, 1, 4, 8, 5, False, [G((12, 5, 33, 7), (5, 3, 1), (0, 1, 1), 2, (8, 4, 30)),
                                              G((1, 9, 121, 8), (0, 3, 1), (0, 1, 1), 1, (1, 8, 120))]),
    E(4, "INSTH", 2, 2, 2, 2, 4, 12, 3, False, [G((12, 5, 31, 5), (2, 2, 1), (2, 2, 2), 2, (8, 4, 28)),
                                                G((5, 5, 5, 6), (2, 2, 1), (2, 2, 2), 2, (8, 4, 28))]),
    E(4, "INSTH", 2, 2, 2, 2, 4, 8, 4, False, [G((6, 7, 31, 5), (2, 4, 1), (2, 2, 2), 2, (4, 4, 28)),
                                               G((5, 7, 7, 6), (2, 4, 1), (2, 2, 2), 2, (4, 4, 28))]),
    E(4, "INST", 2, 2, 2, 2, 4, 8, 4, False, [G((7, 5, 31, 7), (4, 2, 1), (2, 2, 2), 2, (4, 4, 28)),
                                              G((7, 5, 5, 8), (4, 2, 1), (2, 2, 2), 2, (4, 4, 28))]),
    # one W offset per pass wherever the default planner picks it: no pass is short
    E(4, "INST", 2, 2, 2, 2, 4, 8, 3, False, [G((6, 11, 31, 5), (1, 8, 1), (2, 2, 2), 3, (4, 4, 28)),
                                              G((4, 11, 11, 8), (1, 8, 1), (2, 2, 2), 3, (4, 4, 28))]),
    E(4, "INSTH", 2, 0, 2, 2, 4, 8, 3, False, [G((12, 5, 31, 5), (5, 2, 1), (0, 2, 2), 2, (8, 4, 28)),
                                               G((1, 9, 113, 6), (0, 2, 1), (0, 2, 2), 1, (1, 8, 112))]),
    E(4, "INST", 2, 0, 2, 2, 4, 8, 3, False, [G((12, 5, 31, 7), (5, 2, 1), (0, 2, 2), 2, (8, 4, 28)),
                                              G((1, 9, 113, 8), (0, 2, 1), (0, 2, 2), 1, (1, 8, 112))]),
    E(5, "INST64", 1, 1, 1, 1, 4, 8, 5, False, [G((9, 6, 33, 3), (1, 4, 6), (1, 1, 1), 2, (6, 4, 30)),
                                                G((3, 6, 8, 4), (1, 4, 6), (1, 1, 1), 2, (6, 4, 30))]),
    # one W offset per pass wherever the default planner picks it: no pass is short
    E(5, "INST64", 1, 1, 1, 1, 4, 8, 3, False, [G((9, 10, 33, 3), (1, 8, 1), (1, 1, 1), 3, (6, 4, 30)),
                                                G((3, 10, 10, 4), (1, 8, 1), (1, 1, 1), 3, (6, 4, 30))]),
    E(5, "INST64", 1, 1, 1, 1, 4, 8, 5, True, [G((9, 6, 33, 3), (1, 4, 6), (1, 1, 1), 2, (6, 4, 30), 6.0),
                                               G((3, 6, 8, 4), (1, 4, 6), (1, 1, 1), 2, (6, 4, 30), 6.0)]),
    E(5, "INST64", 1, 0, 1, 1, 4, 4, 7, False, [G((7, 6, 33, 3), (6, 4, 1), (0, 1, 1), 2, (4, 4, 30)),
                                                G((3, 6, 61, 4), (0, 4, 1), (0, 1, 1), 1, (2, 4, 60))]),
    E(5, "INST64", 1, 0, 1, 1, 4, 8, 5, False, UNREACHABLE(_BEHIND_4W)),
    E(5, "INST64", 1, 0, 1, 1, 4, 8, 5, True, [G((12, 5, 33, 3), (5, 3, 1), (0, 1, 1), 2, (8, 4, 30), 6.0),
                                               G((1, 9, 121, 4), (0, 3, 1), (0, 1, 1), 1, (1, 8, 120), 6.0)]),
    E(5, "INST64", 1, 0, 1, 0, 4, 4, 7, False, [G((6, 7, 33, 3), (5, 6, 1), (0, 0, 1), 2, (4, 4, 30)),
                                                G((1, 7, 121, 4), (0, 6, 1), (0, 0, 1), 1, (1, 4, 120))]),
    E(5, "INST64", 1, 0, 1, 0, 4, 8, 5, False, UNREACHABLE(_BEHIND_4W)),
    E(5, "INST64", 1, 0, 0, 0, 4, 4, 7, False, [G((6, 7, 35, 3), (5, 6, 1), (0, 0, 0), 2, (4, 4, 32)),
                                                G((3, 7, 65, 4), (0, 6, 1), (0, 0, 0), 1, (2, 4, 64))]),
    E(5, "INST64", 1, 0, 0, 0, 4, 8, 5, False, UNREACHABLE(_BEHIND_4W)),
    E(5, "INST64", 1, 2, 2, 2, 4, 8, 3, False, [G((6, 9, 31, 3), (1, 6, 1), (2, 2, 2), 2, (4, 4, 28)),
                                                G((4, 9, 9, 4), (1, 6, 1), (2, 2, 2), 2, (4, 4, 28))]),
    E(5, "INST64", 1, 2, 2, 2, 2, 8, 5, False, [G((6, 7, 31, 3), (1, 4, 8), (2, 2, 2), 2, (4, 2, 28)),
                                                G((4, 7, 11, 4), (1, 4, 8), (2, 2, 2), 2, (4, 2, 28))]),
    E(5, "INST64", 1, 0, 2, 2, 4, 8, 3, False, [G((12, 5, 31, 3), (5, 2, 1), (0, 2, 2), 2, (8, 4, 28)),
                                                G((1, 9, 113, 4), (0, 2, 1), (0, 2, 2), 1, (1, 8, 112))]),
    E(6, "INSTD", 1, 2, 2, 2, 6, 12, 5, False, [G((15, 8, 31, 3), (1, 5, 1), (2, 2, 2), 2, (10, 6, 28)),
                                                G((4, 8, 8, 4), (1, 5, 1), (2, 2, 2), 2, (10, 6, 28))]),
    E(6, "INSTD", 1, 2, 2, 2, 4, 12, 5, True, [G((15, 5, 31, 3), (7, 2, 1), (2, 2, 2), 2, (10, 4, 28), 6.0),
                                               G((10, 5, 5, 4), (7, 2, 1), (2, 2, 2), 2, (10, 4, 28), 6.0)]),
    E(6, "INSTD64", 1, 2, 2, 2, 4, 8, 3, False, [G((9, 5, 31, 3), (3, 2, 1), (2, 2, 2), 2, (6, 4, 28)),
                                                 G((6, 5, 5, 4), (3, 2, 1), (2, 2, 2), 2, (6, 4, 28))]),
    E(6, "INSTD64", 1, 1, 1, 1, 4, 8, 5, False, [G((10, 7, 33, 3), (1, 5, 1), (1, 1, 1), 2, (7, 4, 30)),
                                                 G((3, 7, 7, 4), (1, 5, 1), (1, 1, 1), 2, (7, 4, 30))]),
    E(6, "INSTD64", 1, 1, 1, 1, 4, 8, 5, True, [G((10, 7, 33, 3), (1, 5, 1), (1, 1, 1), 2, (7, 4, 30), 6.0),
                                                G((3, 7, 7, 4), (1, 5, 1), (1, 1, 1), 2, (7, 4, 30), 6.0)]),
    E(6, "INSTD", 1, 1, 1, 1, 4, 16, 5, False, [G((22, 7, 33, 3), (2, 5, 1), (1, 1, 1), 2, (15, 4, 30), env={"NDNLM_DH": "1"}),
                                                G((4, 7, 7, 4), (2, 5, 1), (1, 1, 1), 2, (15, 4, 30), env={"NDNLM_DH": "1"})]),
    E(6, "INSTD", 1, 1, 1, 1, 4, 16, 5, True, [G((22, 7, 33, 3), (2, 5, 1), (1, 1, 1), 2, (15, 4, 30), 6.0, {"NDNLM_DH": "1"}),
                                               G((4, 7, 7, 4), (2, 5, 1), (1, 1, 1), 2, (15, 4, 30), 6.0, {"NDNLM_DH": "1"})]),
    # persistent CTAs hold the whole W search range in one box: always one pass
    E(7, "INSTP", 1, 1, 1, 1, 4, 16, 5, False, [G((21, 5, 33, 3), (1, 3, 1), (1, 1, 1), 1, (14, 4, 30)),
                                                G((3, 5, 5, 4), (1, 3, 1), (1, 1, 1), 1, (14, 4, 30))]),
    E(7, "INSTP", 1, 1, 1, 1, 4, 16, 5, True, [G((21, 5, 33, 3), (1, 3, 1), (1, 1, 1), 1, (14, 4, 30), 6.0),
                                               G((3, 5, 5, 4), (1, 3, 1), (1, 1, 1), 1, (14, 4, 30), 6.0)]),
]
REACHABLE = [e for e in TABLE if not e.unreachable]
CASES = [(e, g) for e in REACHABLE for g in e.geoms]


def _case_id(case):
    e, g = case
    return "%s-%s-r%s" % (e.name.replace("nlm_tiled", ""), "x".join(map(str, g.shape)), "".join(map(str, g.r)))


# ---- planning (CPU) -------------------------------------------------------------------------------------
def _plan(dtype, g, monkeypatch, env=None):
    from nd_b200 import device
    for k in PLANNER_ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    return device.Plan(g.shape, g.r, g.f, 0.3, 1.5 if g.n_eff > 0 else 0.6, g.n_eff, dtype=dtype)


def _base(kernel_name):
    return re.sub(r"\[passes=\d+\]$", "", kernel_name)


@pytest.fixture(scope="module")
def variant_index():
    """name -> index of NDNLM_TILED_VARIANT, taken from the planner: each index is forced at the table's geometries
    until one accepts it (never hard-coded; tools/dev_*.py use the same indices)."""
    mp = pytest.MonkeyPatch()
    try:
        index = {}
        for i in range(len(TABLE)):
            for e, g in CASES:
                p = _plan(e.dtype, g, mp, {"NDNLM_TILED_VARIANT": str(i)})
                if p.is_tiled:
                    index.setdefault(_base(p.kernel_name), []).append(i)
                    break
        return index
    finally:
        mp.undo()


def _accepted(e, g, index, monkeypatch):
    """(index, name) of every instantiation the planner accepts at `g` when forced."""
    out = []
    for name, (i,) in sorted(index.items(), key=lambda kv: kv[1]):
        p = _plan(e.dtype, g, monkeypatch, {"NDNLM_TILED_VARIANT": str(i)})
        if p.is_tiled:
            assert _base(p.kernel_name) == name, (i, p.kernel_name, name)
            out.append((i, name))
    return out


def _cuda_tool(name):
    """`name` from the directory of the nvcc that __graft_entry__.build() compiles with."""
    nvcc = shutil.which(os.environ.get("NVCC", "nvcc"))
    if nvcc is None:
        nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    path = os.path.join(os.path.dirname(os.path.realpath(nvcc)), name)
    assert os.path.exists(path), "%s not found next to %s" % (name, nvcc)
    return path


def test_table_equals_the_instantiations_in_the_library():
    sass = subprocess.run([_cuda_tool("cuobjdump"), "-sass", LIB], capture_output=True, text=True, check=True).stdout
    mangled = [m.group(1) for m in re.finditer(r"Function : (\S+)", sass)]
    demangled = subprocess.run([_cuda_tool("cu++filt")], input="\n".join(mangled), capture_output=True, text=True,
                               check=True).stdout.splitlines()
    # 'void ndnlm::nlm_tiled_kernel<float, (int)1, ..., (bool)0>(CUtensorMap_st, ...)' -> 'ndnlm::nlm_tiled_kernel<float,1,...,false>'
    names = sorted(re.sub(r"\(bool\)0", "false", re.sub(r"\(bool\)1", "true", n.replace("(int)", "")))
                   .replace(" ", "")[len("void"):].split("(", 1)[0] for n in demangled if "ndnlm::nlm_tiled_kernel<" in n)
    table = sorted(e.symbol for e in TABLE)
    assert len(set(table)) == len(TABLE) == 53 and len(set(e.name for e in TABLE)) == 53
    assert names == table, (sorted(set(names) - set(table)), sorted(set(table) - set(names)))
    assert sum(1 for e in TABLE if e.unreachable) == 8


def test_variant_index_covers_the_table(variant_index):
    assert sorted(variant_index) == sorted(e.name for e in TABLE)
    assert sorted(i for v in variant_index.values() for i in v) == list(range(len(TABLE)))


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_geometry_selects_its_instantiation(case, monkeypatch):
    e, g = case
    assert set(g.env or {}) <= {"NDNLM_DH", "NDNLM_PERSIST"}
    p = _plan(e.dtype, g, monkeypatch, g.env)
    assert p.kernel_name == "%s[passes=%d]" % (e.name, g.passes)
    assert tuple(p.info.tile) == g.tile
    assert all(g.r[a] + g.f[a] <= g.shape[a] - 1 for a in range(3))


def _geometry_facts(e, g, monkeypatch):
    p = _plan(e.dtype, g, monkeypatch, g.env)
    n, t = list(p.info.n), list(p.info.tile)
    per = p.info.box[0] - p.info.warps[0] + 1                     # W offsets per pass: box rows = CTA rows + per - 1
    return dict(tails=[k for k in range(3) if n[k] > t[k] and n[k] % t[k]],
                short_pass=g.passes > 1 and (2 * g.r[p.roles[0]] + 1) % per != 0,
                minimal=any(g.r[a] + g.f[a] == g.shape[a] - 1 for a in range(3)),
                per=per, w_extent=n[0])


def test_geometries_cover_the_edges(monkeypatch):
    facts = {(repr(e), repr(g)): _geometry_facts(e, g, monkeypatch) for e, g in CASES}
    assert {k for f in facts.values() for k in f["tails"]} == {0, 1, 2}
    assert all(any(facts[repr(e), repr(g)]["minimal"] for g in e.geoms) for e in REACHABLE)
    for e in REACHABLE:
        # a short last pass wherever the kernel runs several passes of more than one W offset by default
        assert e.macro == "INSTP" or any(facts[repr(e), repr(g)]["short_pass"] or facts[repr(e), repr(g)]["per"] == 1
                                         for g in e.geoms), e
        assert any(all(k in facts[repr(e), repr(g)]["tails"] for k in (1, 2)) for g in e.geoms), e
    vs = {g.shape[3] for e, g in CASES}
    assert {3, 5, 6, 7} <= vs
    w2d = {facts[repr(e), repr(g)]["w_extent"] == 1 for e, g in CASES if e.args[1] == 0 and g.r[0] == 0}
    assert w2d == {True, False}


def test_unreachable_entries_are_never_selected_by_default(monkeypatch):
    """A grid over dtype, V, n_eff, patch pattern, radii and the W extent finds no default geometry for any
    UNREACHABLE entry (a few seconds of plan creation).  If the planner changes, this fails."""
    from nd_b200 import device
    for k in PLANNER_ENV:
        monkeypatch.delenv(k, raising=False)
    unreachable = {e.name for e in TABLE if e.unreachable}
    seen = set()
    for dtype, n_eff, V in itertools.product((np.float32, np.float64), (-1.0, 6.0), (1, 3, 4)):
        for fv, rw, rr, rx in itertools.product((0, 1, 2), (0, 1, 2, 3, 5, 8), (0, 1, 2, 3, 5, 8, 10), (1, 2, 3, 5, 8, 12, 16)):
            for f in {(fv, fv, fv), (0, fv, fv), (0, 0, fv)}:
                if rw == 0 and f[0]:
                    continue
                for n0 in ((1, 2, 3, 5, 40) if rw == 0 else (40,)):
                    try:
                        p = device.Plan((n0, 60, 90, V), (rw, rr, rx), f, 0.3, 1.5, n_eff, dtype=dtype)
                    except ValueError:
                        continue
                    seen.add(_base(p.kernel_name))
    assert not seen & unreachable, sorted(seen & unreachable)
    assert len(seen & {e.name for e in REACHABLE}) >= 30        # the grid does reach the rest of the table


def test_every_unreachable_entry_runs_as_a_sibling(variant_index, monkeypatch):
    """Each UNREACHABLE entry is accepted at some selecting geometry, so the sibling test runs it; and the sibling
    pairs span half / full groups, L = 2 .. 8, every CH and 4 .. 16 warps."""
    by_name = {e.name: e for e in TABLE}
    forced = set()
    pairs = set()
    for e, g in CASES:
        for _, name in _accepted(e, g, variant_index, monkeypatch):
            if name != e.name:
                forced.add(name)
                pairs.add((e.args, by_name[name].args, e.macro, by_name[name].macro))
    assert {e.name for e in TABLE if e.unreachable} <= forced
    assert any(("H" in a) != ("H" in b) for _, _, a, b in pairs)                     # half against full group
    assert {x[4] for p in pairs for x in p[:2]} == {2, 4, 6, 8}                      # L
    assert any(x[6] != y[6] for x, y, _, _ in pairs)                                 # CH
    assert {8, 12, 16} <= {x[5] for p in pairs for x in p[:2]}                        # warps


# ---- GPU -----------------------------------------------------------------------------------------------
def _run(e, g, a, monkeypatch, env):
    import torch
    p = _plan(e.dtype, g, monkeypatch, env)
    out = p.apply(torch.from_numpy(a).cuda()).cpu().numpy()
    return out, p.kernel_name


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_instantiation_matches_oracle_and_its_siblings_bitwise(case, c_oracle, variant_index, monkeypatch,
                                                               record_property):
    e, g = case
    a = sar_like(g.shape, seed=sum(g.shape) + 7 * sum(g.r), dtype=e.dtype)
    h = 1.5 if g.n_eff > 0 else 0.6
    out, name = _run(e, g, a, monkeypatch, g.env)
    assert name == "%s[passes=%d]" % (e.name, g.passes)
    assert out.dtype == e.dtype and not np.isnan(out).any()
    ref = c_oracle.nlmeans(a, g.r, g.f, 0.3, h, g.n_eff, threads=8)
    err = scaled_err(out, ref)
    record_property("scaled_err", err)
    assert err < (TOL64 if e.dtype == np.float64 else TOL32), (name, err)
    ran, differ = [], []
    for i, sib in _accepted(e, g, variant_index, monkeypatch):
        if sib == e.name:
            continue
        o, n = _run(e, g, a, monkeypatch, {"NDNLM_TILED_VARIANT": str(i)})
        assert _base(n) == sib
        ran.append(n)
        if not np.array_equal(o, out):
            differ.append((n, int((o != out).sum()), float(np.abs(o.astype(np.float64) - out).max())))
    record_property("siblings", ";".join(ran))
    assert not differ, (name, differ)
