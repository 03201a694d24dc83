"""ctypes front-end of tests/emu/emu_path.cpp: the host emulator with the path check (TEST HARNESS ONLY).

`PathEmuEngine` is emu_binding.EmuEngine (every evaluation mode, the mesh grid) with `path_check`, the emulator's
counterpart of engine.Engine.path_check (DESIGN.md section 11).  The library is built by __graft_entry__.build().
"""
import ctypes
import os
import subprocess

import numpy as np

import emu_binding
from gelato_b200 import engine

LIB = os.path.join(emu_binding.BUILD, "libgelato_emu_path.so")
_pd = ctypes.POINTER(ctypes.c_double)
_pi32 = ctypes.POINTER(ctypes.c_int32)


def build(force=False):
    emu = os.path.join(emu_binding._HERE, "emu")
    src = os.path.join(emu, "emu_path.cpp")
    csrc = os.path.join(emu_binding.ROOT, "gelato_b200", "csrc")
    deps = [src, os.path.join(emu, "emu.cpp"), os.path.join(emu_binding.ROOT, "include", "gelato_b200.h")] + [
        os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".inc"))]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(f) for f in deps):
        return LIB
    os.makedirs(emu_binding.BUILD, exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-mfma", "-pthread", "-o", LIB, src])
    return LIB


class PathEmuEngine(emu_binding.EmuEngine):
    def __init__(self, plan, scenario_plans=None):
        super().__init__(plan, scenario_plans=scenario_plans)
        build()
        self.Lp = Lp = ctypes.CDLL(LIB)
        assert Lp.emu_unfused_check() == 1
        Lp.emu_eval_path_check.argtypes = [ctypes.POINTER(engine.PlanDesc), ctypes.POINTER(engine.ScenarioDesc),
                                           ctypes.POINTER(engine.MeshGridDesc), _pd, _pd, _pi32, ctypes.c_int]
        Lp.emu_eval_path_check.restype = ctypes.c_char_p

    def path_check(self, x, n_scen=1):
        """engine.Engine.path_check: a call gelato_eval_path_check refuses raises engine.GelatoError with its reason."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        n = n_scen * self.plan.n_aero
        res, at = np.full(n, np.nan), np.full(n, -2, dtype=np.int32)
        why = self.Lp.emu_eval_path_check(ctypes.byref(self.desc), self._sc(),
                                          None if self._grid is None else ctypes.byref(self._grid[0]),
                                          x.ctypes.data_as(_pd), res.ctypes.data_as(_pd), at.ctypes.data_as(_pi32), n_scen)
        if why is not None:
            raise engine.GelatoError("gelato_eval_path_check failed (-1): %s" % why.decode())
        return (res, at) if n_scen == 1 else (res.reshape(n_scen, -1), at.reshape(n_scen, -1))
