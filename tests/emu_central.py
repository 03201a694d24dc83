"""The host emulator with the engine's finite-difference modes (TEST HARNESS ONLY; DESIGN.md H6).

`FdEmuEngine` is `emu_binding.EmuEngine` plus `set_fd` / `fd` as `gelato_b200.engine.Engine` has them: in central mode
every Jacobian it returns (COO, packed, pair, update) comes from tests/emu/emu_central.cpp, which runs the kernels'
per-thread code with +h and -h and averages with jobs.h: fd_central.  In forward mode it is the plain emulator.
"""
import ctypes
import os
import subprocess

import numpy as np

import emu_binding
from gelato_b200 import engine

LIB = os.path.join(emu_binding.BUILD, "libgelato_emu_central.so")
_pd = ctypes.POINTER(ctypes.c_double)


def build(force=False):
    emu = os.path.join(emu_binding._HERE, "emu")
    src = os.path.join(emu, "emu_central.cpp")
    csrc = os.path.join(emu_binding.ROOT, "gelato_b200", "csrc")
    deps = [src, os.path.join(emu, "emu.cpp"), os.path.join(emu_binding.ROOT, "include", "gelato_b200.h")] + [
        os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".inc"))]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(f) for f in deps):
        return LIB
    os.makedirs(emu_binding.BUILD, exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-mfma", "-pthread", "-o", LIB, src])
    return LIB


class FdEmuEngine(emu_binding.EmuEngine):
    def __init__(self, plan, scenario_plans=None):
        super().__init__(plan, scenario_plans=scenario_plans)
        build()
        self.C = ctypes.CDLL(LIB)
        self.C.emu_eval_central.argtypes = [ctypes.POINTER(engine.PlanDesc), ctypes.POINTER(engine.ScenarioDesc), _pd, _pd,
                                            _pd, ctypes.c_int, ctypes.POINTER(ctypes.c_int32), ctypes.c_int, ctypes.c_double]
        self._step = None  # None: forward differences

    def set_fd(self, mode, step=None):
        """engine.Engine.set_fd: "forward" or "central" with step `step` (None: engine.DEFAULT_FD_STEP)."""
        _, h = engine.fd_args(mode, step)
        self._step = h if mode == "central" else None

    @property
    def fd(self):
        return ("forward", float(self.plan.units[5])) if self._step is None else ("central", self._step)

    def _central(self, x, n_scen, scen_ids, packed, pair):
        """(g or None, values) of a central-difference evaluation."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        g = np.full(n_scen * self.plan.n_rows, np.nan) if pair else None
        v = np.full(n_scen * (self.n_pack if packed else self.plan.n_vals), np.nan)
        ids, pids = self._ids(scen_ids)
        rc = self.C.emu_eval_central(ctypes.byref(self.desc), self._sc(), x.ctypes.data_as(_pd),
                                     None if g is None else g.ctypes.data_as(_pd), v.ctypes.data_as(_pd), n_scen, pids,
                                     1 if packed else 0, self._step)
        assert rc == 0, "the plan description failed validate_desc (plan_host.h)"
        if n_scen > 1:
            v = v.reshape(n_scen, -1)
            g = None if g is None else g.reshape(n_scen, -1)
        return g, v

    def eval_jacobian(self, x, n_scen=1, out=None, scen_ids=None):
        if self._step is None:
            return super().eval_jacobian(x, n_scen, out, scen_ids)
        self.launches += 1
        self.calls += 1
        return self._central(x, n_scen, scen_ids, False, False)[1]

    def eval_jacobian_packed(self, x, n_scen=1, scen_ids=None):
        """packed[n_scen][n_pack] of a Jacobian-only evaluation (central mode)."""
        assert self._step is not None
        return self._central(x, n_scen, scen_ids, True, False)[1]

    def eval_pair(self, x, n_scen=1, scen_ids=None, packed=False):
        if self._step is None:
            return super().eval_pair(x, n_scen, scen_ids, packed)
        return self._central(x, n_scen, scen_ids, packed, True)

    def eval_jacobian_update(self, x, out, n_scen=1):
        if self._step is None:
            return super().eval_jacobian_update(x, out, n_scen)
        assert n_scen == 1
        v = self.eval_jacobian(x)
        idx = self.plan.xdep_index()
        out[idx] = v[idx]
        return out

    def eval_pair_update(self, x, g_out, vals_out, n_scen=1):
        if self._step is None:
            return super().eval_pair_update(x, g_out, vals_out, n_scen)
        assert n_scen == 1
        self.launches += 1
        self.calls += 1
        g, v = self._central(x, 1, None, False, True)
        g_out[:] = g
        idx = self.plan.xdep_index()
        vals_out[idx] = v[idx]
        return g_out.reshape(1, -1), vals_out.reshape(1, -1)

    def eval_pair_range(self, x, g, packed, blocks, vacuum):
        if self._step is not None:
            raise ValueError("the range evaluation supports forward differences only")
        return super().eval_pair_range(x, g, packed, blocks, vacuum)
