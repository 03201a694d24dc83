"""The host emulator with the engine's mesh error estimate (TEST HARNESS ONLY; DESIGN.md section 11).

`MeshEmuEngine` is `emu_binding.EmuEngine` plus `set_mesh_grid` / `mesh_error` as `gelato_b200.engine.Engine` has them,
computed by tests/emu/emu_mesh.cpp: the kernels' per-thread code (gelato_b200/csrc/mesh_error.h) compiled with g++.
"""
import ctypes
import os
import subprocess

import numpy as np

import emu_binding
from gelato_b200 import engine

LIB = os.path.join(emu_binding.BUILD, "libgelato_emu_mesh.so")
_pd = ctypes.POINTER(ctypes.c_double)


def build(force=False):
    emu = os.path.join(emu_binding._HERE, "emu")
    src = os.path.join(emu, "emu_mesh.cpp")
    csrc = os.path.join(emu_binding.ROOT, "gelato_b200", "csrc")
    deps = [src, os.path.join(emu, "emu.cpp"), os.path.join(emu_binding.ROOT, "include", "gelato_b200.h")] + [
        os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".inc"))]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(f) for f in deps):
        return LIB
    os.makedirs(emu_binding.BUILD, exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-mfma", "-pthread", "-o", LIB, src])
    return LIB


class MeshEmuEngine(emu_binding.EmuEngine):
    def __init__(self, plan, scenario_plans=None):
        super().__init__(plan, scenario_plans=scenario_plans)
        build()
        self.C = ctypes.CDLL(LIB)
        self.C.emu_mesh_error.argtypes = [ctypes.POINTER(engine.PlanDesc), ctypes.POINTER(engine.ScenarioDesc),
                                          ctypes.POINTER(engine.MeshGridDesc), _pd, _pd, ctypes.c_int]
        self._grid = None

    def set_mesh_grid(self, tables):
        """engine.Engine.set_mesh_grid."""
        self._grid = engine.make_mesh_grid_desc(tables)

    def mesh_error(self, x, n_scen=1, out=None):
        """engine.Engine.mesh_error."""
        assert self._grid is not None, "no mesh grid set"
        x = np.ascontiguousarray(x, dtype=np.float64)
        err = np.full(n_scen * self.plan.S * 11, np.nan)
        rc = self.C.emu_mesh_error(ctypes.byref(self.desc), self._sc(), ctypes.byref(self._grid[0]), x.ctypes.data_as(_pd),
                                   err.ctypes.data_as(_pd), n_scen)
        assert rc == 0, "the plan description failed validate_desc (plan_host.h)"
        return err.reshape(self.plan.S, 11) if n_scen == 1 else err.reshape(n_scen, self.plan.S, 11)
