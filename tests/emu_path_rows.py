"""ctypes front-end of tests/emu/emu_path_rows.cpp: the host emulator with the path check and the path rows (TEST HARNESS
ONLY).

`PathRowsEmuEngine` is emu_path.PathEmuEngine (every evaluation mode, the mesh grid, the path check) with the path rows
(`set_path_rows`, `path_rows_layout`, `eval_path_rows`), the emulator's counterparts of engine.Engine's (DESIGN.md
section 11), so that GelatoProblem runs with path rows on the CPU tier.  The library is built by
__graft_entry__.build().
"""
import ctypes
import os
import subprocess

import numpy as np

import emu_binding
import emu_path
from gelato_b200 import engine

LIB = os.path.join(emu_binding.BUILD, "libgelato_emu_path_rows.so")
_pd = ctypes.POINTER(ctypes.c_double)
_pi32 = ctypes.POINTER(ctypes.c_int32)
_pi64 = ctypes.POINTER(ctypes.c_int64)


def build(force=False):
    emu = os.path.join(emu_binding._HERE, "emu")
    src = os.path.join(emu, "emu_path_rows.cpp")
    csrc = os.path.join(emu_binding.ROOT, "gelato_b200", "csrc")
    deps = [src, os.path.join(emu, "emu_path.cpp"), os.path.join(emu, "emu.cpp"),
            os.path.join(emu_binding.ROOT, "include", "gelato_b200.h")] + [
        os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".inc"))]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(f) for f in deps):
        return LIB
    os.makedirs(emu_binding.BUILD, exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-mfma", "-pthread", "-o", LIB, src])
    return LIB


class PathRowsEmuEngine(emu_path.PathEmuEngine):
    def __init__(self, plan, scenario_plans=None):
        super().__init__(plan, scenario_plans=scenario_plans)
        build()
        self.Lr = Lr = ctypes.CDLL(LIB)
        assert Lr.emu_unfused_check() == 1
        Lr.emu_path_rows.argtypes = [ctypes.POINTER(engine.PlanDesc), ctypes.POINTER(engine.MeshGridDesc), _pi32, _pi64,
                                     _pi32, _pi32, _pi64]
        Lr.emu_path_rows.restype = ctypes.c_char_p
        Lr.emu_eval_path_rows.argtypes = [ctypes.POINTER(engine.PlanDesc), ctypes.POINTER(engine.ScenarioDesc),
                                          ctypes.POINTER(engine.MeshGridDesc), _pd, _pd, _pd, ctypes.c_int, ctypes.c_int32,
                                          ctypes.c_double]
        Lr.emu_eval_path_rows.restype = ctypes.c_char_p
        self._prow = None  # (grid, layout) of the path rows once set

    # ---- path rows ----
    def set_path_rows(self, tables):
        """engine.Engine.set_path_rows: a grid gelato_plan_set_path_rows refuses raises engine.GelatoError with its
        reason and the previous rows stay."""
        grid = engine.make_mesh_grid_desc(tables)
        self._prow = (grid, self._layout(grid))

    def _layout(self, grid):
        n, v = ctypes.c_int32(0), ctypes.c_int64(0)
        d = ctypes.byref(self.desc)
        why = self.Lr.emu_path_rows(d, ctypes.byref(grid[0]), ctypes.byref(n), ctypes.byref(v), None, None, None)
        if why is not None:
            raise engine.GelatoError("gelato_plan_set_path_rows failed (-1): %s" % why.decode())
        job, l = np.empty(n.value, dtype=np.int32), np.empty(n.value, dtype=np.int32)
        off = np.empty((n.value, 4), dtype=np.int64)
        self.Lr.emu_path_rows(d, ctypes.byref(grid[0]), ctypes.byref(n), ctypes.byref(v), job.ctypes.data_as(_pi32),
                              l.ctypes.data_as(_pi32), off.ctypes.data_as(_pi64))
        return {"n_rows": n.value, "n_vals": v.value, "job": job, "l": l, "off": off}

    def path_rows_layout(self):
        """engine.Engine.path_rows_layout."""
        if self._prow is None:
            raise engine.GelatoError("gelato_plan_path_rows failed (-1): no path rows set (gelato_plan_set_path_rows)")
        return self._prow[1]

    def eval_path_rows(self, x, n_scen=1, jacobian=True, out=None):
        """engine.Engine.eval_path_rows, in the emulator's finite-difference mode (set_fd)."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        self.calls += 1
        grid = None if self._prow is None else self._prow[0]
        lay = self._prow[1] if self._prow is not None else {"n_rows": 0, "n_vals": 0}
        nr, nv = lay["n_rows"], lay["n_vals"]
        if out is not None:
            g = None if out[0] is None else engine._out(out[0], n_scen * nr, "out[0]")
            v = None if out[1] is None else engine._out(out[1], n_scen * nv, "out[1]")
        else:
            g, v = np.full(n_scen * nr, np.nan), (np.full(n_scen * nv, np.nan) if jacobian else None)
        why = self.Lr.emu_eval_path_rows(ctypes.byref(self.desc), self._sc(), None if grid is None else ctypes.byref(grid[0]),
                                         x.ctypes.data_as(_pd), None if g is None else g.ctypes.data_as(_pd),
                                         None if v is None else v.ctypes.data_as(_pd), n_scen, *self._fd)
        if why is not None:
            raise engine.GelatoError("gelato_eval_path_rows failed (-1): %s" % why.decode())
        if n_scen > 1:
            g, v = (None if a is None else a.reshape(n_scen, -1) for a in (g, v))
        return g, v
