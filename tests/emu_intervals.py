"""ctypes front-end of tests/emu/emu_intervals.cpp: the host emulator with the per-interval mesh error estimate.

TEST HARNESS ONLY.  IntervalEmuEngine is emu_binding.EmuEngine whose mesh error estimate follows a grid's interval
tables (DESIGN.md section 11, "h-refinement") as gelato_eval_mesh_error and gelato_eval_mesh_error_intervals do; every
other entry point is EmuEngine's.
"""
import ctypes
import os
import subprocess

import numpy as np

import emu_binding
from gelato_b200 import engine

LIB = os.path.join(emu_binding.BUILD, "libgelato_emu_intervals.so")
_pd = ctypes.POINTER(ctypes.c_double)


def build(force=False):
    src = os.path.join(emu_binding._HERE, "emu", "emu_intervals.cpp")
    csrc = os.path.join(emu_binding.ROOT, "gelato_b200", "csrc")
    deps = [src, os.path.join(emu_binding._HERE, "emu", "emu.cpp"), os.path.join(emu_binding.ROOT, "include", "gelato_b200.h")] + [
        os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".inc"))]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(f) for f in deps):
        return LIB
    os.makedirs(emu_binding.BUILD, exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-mfma", "-pthread", "-o", LIB, src])
    return LIB


class IntervalEmuEngine(emu_binding.EmuEngine):
    """EmuEngine with engine.Engine's mesh_error and mesh_error_intervals on grids with or without interval tables."""

    def __init__(self, plan, scenario_plans=None):
        super().__init__(plan, scenario_plans=scenario_plans)
        build()
        self.Li = Li = ctypes.CDLL(LIB)
        Li.emu_eval_mesh_error_intervals.argtypes = [ctypes.POINTER(engine.PlanDesc), ctypes.POINTER(engine.ScenarioDesc),
                                                     ctypes.POINTER(engine.MeshGridDesc), _pd, _pd, _pd, ctypes.c_int]
        Li.emu_eval_mesh_error_intervals.restype = ctypes.c_char_p
        self.n_mesh_int = 0

    def set_mesh_grid(self, tables):
        super().set_mesh_grid(tables)
        self.n_mesh_int = engine.grid_intervals(tables)

    def _estimate(self, x, n_scen, per_interval, what):
        x = np.ascontiguousarray(x, dtype=np.float64)
        K = self.n_mesh_int if per_interval else self.plan.S
        out = np.full(n_scen * K * 11, np.nan)
        ptr = out.ctypes.data_as(_pd)
        self._check(self.Li.emu_eval_mesh_error_intervals(ctypes.byref(self.desc), self._sc(), self._grid_ptr(self._grid),
                                                          x.ctypes.data_as(_pd), None if per_interval else ptr,
                                                          ptr if per_interval else None, n_scen), what)
        return out.reshape(K, 11) if n_scen == 1 else out.reshape(n_scen, K, 11)

    def mesh_error(self, x, n_scen=1):
        """engine.Engine.mesh_error: err[S][11], each section's value the max over its intervals."""
        return self._estimate(x, n_scen, False, "gelato_eval_mesh_error")

    def mesh_error_intervals(self, x, n_scen=1):
        """engine.Engine.mesh_error_intervals: err_int[n_int][11]."""
        return self._estimate(x, n_scen, True, "gelato_eval_mesh_error_intervals")
