"""ctypes front-end of tests/emu (the host emulator of the CUDA kernels).

TEST HARNESS ONLY: lets the CPU test tier run the kernels' per-thread code
(gelato_b200/csrc/jobs.h, mesh_error.h) through the same GelatoPlanDesc the GPU library gets, with the settings
gelato_b200.engine.Engine has: the finite-difference mode (DESIGN.md H6), the mesh grid and the grid of the path rows
(DESIGN.md section 11).
"""
import ctypes
import os
import subprocess

import numpy as np

from gelato_b200 import engine

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
BUILD = os.path.join(_HERE, "_build")
LIB = os.path.join(BUILD, "libgelato_emu.so")
_pd = ctypes.POINTER(ctypes.c_double)
_pi32 = ctypes.POINTER(ctypes.c_int32)
_pi64 = ctypes.POINTER(ctypes.c_int64)


def build(force=False):
    src = os.path.join(_HERE, "emu", "emu.cpp")
    csrc = os.path.join(ROOT, "gelato_b200", "csrc")
    deps = [src, os.path.join(ROOT, "include", "gelato_b200.h")] + [
        os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".h", ".inc"))]
    if not force and os.path.exists(LIB) and all(os.path.getmtime(LIB) >= os.path.getmtime(f) for f in deps):
        return LIB
    os.makedirs(BUILD, exist_ok=True)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-mfma", "-pthread", "-o", LIB, src])
    return LIB


class Emulator:
    def __init__(self, plan, scenario_plans=None):
        build()
        self.L = L = ctypes.CDLL(LIB)
        assert L.emu_unfused_check() == 1
        self.plan = plan
        self.desc, self._keep = engine.make_desc(plan)
        self.sc = None
        if scenario_plans is not None:
            self.sc, keep = engine.make_scenario_desc(scenario_plans)
            self._keep += keep
        pdesc, psc, pgrid, c_int = (ctypes.POINTER(engine.PlanDesc), ctypes.POINTER(engine.ScenarioDesc),
                                    ctypes.POINTER(engine.MeshGridDesc), ctypes.c_int)
        L.emu_eval_residuals.argtypes = [pdesc, psc, _pd, _pd, c_int, _pi32]
        L.emu_eval_jacobian.argtypes = [pdesc, psc, _pd, _pd, _pd, c_int, _pi32, c_int, ctypes.c_int32, ctypes.c_double]
        L.emu_eval_pair_range.argtypes = [pdesc, psc, _pd, _pd, _pd] + [c_int] * 5
        L.emu_block_counts.argtypes = [pdesc, ctypes.POINTER(c_int), ctypes.POINTER(c_int)]
        L.emu_packed_map.argtypes = [pdesc, _pi64, _pi64, _pd]
        L.emu_packed_map.restype = ctypes.c_longlong
        L.emu_n_xdep.argtypes = [pdesc]
        L.emu_n_xdep.restype = ctypes.c_longlong
        L.emu_check_mesh_grid.argtypes = [pdesc, pgrid]
        L.emu_eval_mesh_error.argtypes = [pdesc, psc, pgrid, _pd, _pd, c_int]
        L.emu_eval_path_check.argtypes = [pdesc, psc, pgrid, _pd, _pd, _pi32, c_int]
        L.emu_plan_path_rows.argtypes = [pdesc, pgrid, _pi32, _pi64, _pi32, _pi32, _pi64]
        L.emu_eval_path_rows.argtypes = [pdesc, psc, pgrid, _pd, _pd, _pd, c_int, ctypes.c_int32, ctypes.c_double]
        for f in (L.emu_check_mesh_grid, L.emu_eval_mesh_error, L.emu_eval_path_check, L.emu_plan_path_rows,
                  L.emu_eval_path_rows):
            f.restype = ctypes.c_char_p  # NULL or the reason of a refusal
        self.n_pack = int(L.emu_packed_map(ctypes.byref(self.desc), None, None, None))
        self._fd = engine.fd_args("forward")  # (C mode code, step) as gelato_plan_set_fd takes them
        self._grid = None  # the mesh grid once set
        self._prow = None  # (grid, layout) of the path rows once set

    def _sc(self):
        return ctypes.byref(self.sc) if self.sc is not None else None

    @staticmethod
    def _grid_ptr(grid):
        return None if grid is None else ctypes.byref(grid[0])

    @staticmethod
    def _check(why, what):
        """engine._check for the entry points that return NULL or the reason of a refusal: engine.GelatoError as the C
        entry point `what` raises it."""
        if why is not None:
            raise engine.GelatoError("%s failed (-1): %s" % (what, why.decode()))

    @staticmethod
    def _ids(scen_ids):
        if scen_ids is None:
            return None, None
        ids = np.ascontiguousarray(scen_ids, dtype=np.int32)
        return ids, ids.ctypes.data_as(_pi32)

    # ---- settings, as engine.Engine has them ----
    def set_fd(self, mode, step=None):
        """engine.Engine.set_fd: "forward" or "central" with step `step` (None: engine.DEFAULT_FD_STEP)."""
        self._fd = engine.fd_args(mode, step)

    @property
    def fd(self):
        """engine.Engine.fd: (mode, step), forward's step being the plan's dx."""
        code, step = self._fd
        return ("central", step) if code == engine.FD_MODES["central"] else ("forward", float(self.plan.units[5]))

    def set_mesh_grid(self, tables):
        """engine.Engine.set_mesh_grid: a grid gelato_plan_set_mesh_grid refuses raises engine.GelatoError with its
        reason and the previous grid stays."""
        grid = engine.make_mesh_grid_desc(tables)
        self._check(self.L.emu_check_mesh_grid(ctypes.byref(self.desc), ctypes.byref(grid[0])),
                    "gelato_plan_set_mesh_grid")
        self._grid = grid

    def set_path_rows(self, tables):
        """engine.Engine.set_path_rows: a grid gelato_plan_set_path_rows refuses raises engine.GelatoError with its
        reason and the previous rows stay."""
        grid = engine.make_mesh_grid_desc(tables)
        n, v = ctypes.c_int32(0), ctypes.c_int64(0)
        args = (ctypes.byref(self.desc), ctypes.byref(grid[0]), ctypes.byref(n), ctypes.byref(v))
        self._check(self.L.emu_plan_path_rows(*args, None, None, None), "gelato_plan_set_path_rows")
        job, l = np.empty(n.value, dtype=np.int32), np.empty(n.value, dtype=np.int32)
        off = np.empty((n.value, 4), dtype=np.int64)
        self.L.emu_plan_path_rows(*args, job.ctypes.data_as(_pi32), l.ctypes.data_as(_pi32), off.ctypes.data_as(_pi64))
        self._prow = (grid, {"n_rows": n.value, "n_vals": v.value, "job": job, "l": l, "off": off})

    def path_rows_layout(self):
        """engine.Engine.path_rows_layout."""
        if self._prow is None:
            raise engine.GelatoError("gelato_plan_path_rows failed (-1): no path rows set (gelato_plan_set_path_rows)")
        return self._prow[1]

    # ---- evaluations ----
    def eval_residuals(self, x, n_scen=1, scen_ids=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        g = np.full(n_scen * self.plan.n_rows, np.nan)
        ids, pids = self._ids(scen_ids)
        rc = self.L.emu_eval_residuals(ctypes.byref(self.desc), self._sc(), x.ctypes.data_as(_pd), g.ctypes.data_as(_pd), n_scen, pids)
        assert rc == 0, "the plan description failed validate_desc (plan_host.h)"
        return g if n_scen == 1 else g.reshape(n_scen, -1)

    def _jacobian(self, x, n_scen, scen_ids, packed, pair):
        """(g or None, COO or packed values) of one evaluation in the current finite-difference mode."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        g = np.full(n_scen * self.plan.n_rows, np.nan) if pair else None
        v = np.full(n_scen * (self.n_pack if packed else self.plan.n_vals), np.nan)
        ids, pids = self._ids(scen_ids)
        rc = self.L.emu_eval_jacobian(ctypes.byref(self.desc), self._sc(), x.ctypes.data_as(_pd),
                                      None if g is None else g.ctypes.data_as(_pd), v.ctypes.data_as(_pd), n_scen, pids,
                                      1 if packed else 0, *self._fd)
        assert rc == 0, "the plan description failed validate_desc (plan_host.h)"
        if n_scen > 1:
            v = v.reshape(n_scen, -1)
            g = None if g is None else g.reshape(n_scen, -1)
        return g, v

    def eval_jacobian(self, x, n_scen=1, scen_ids=None):
        return self._jacobian(x, n_scen, scen_ids, False, False)[1]

    def eval_jacobian_packed(self, x, n_scen=1, scen_ids=None):
        """packed[n_scen][n_pack] of a Jacobian-only evaluation."""
        return self._jacobian(x, n_scen, scen_ids, True, False)[1]

    def eval_pair(self, x, n_scen=1, scen_ids=None, packed=False):
        """(g, vals or packed) of a pair evaluation: defects from the Jacobian blocks' centre columns."""
        return self._jacobian(x, n_scen, scen_ids, packed, True)

    def packed_map(self):
        """(full_slot, src, sgn): vals[full_slot] = sgn * packed[src] (plan_host.h: build_packed_layout)."""
        n = int(self.L.emu_n_xdep(ctypes.byref(self.desc)))
        full, src, sgn = np.empty(n, dtype=np.int64), np.empty(n, dtype=np.int64), np.empty(n)
        self.L.emu_packed_map(ctypes.byref(self.desc), full.ctypes.data_as(_pi64), src.ctypes.data_as(_pi64),
                              sgn.ctypes.data_as(_pd))
        return full, src, sgn

    def mesh_error(self, x, n_scen=1):
        """engine.Engine.mesh_error: a call gelato_eval_mesh_error refuses raises engine.GelatoError with its reason."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        err = np.full(n_scen * self.plan.S * 11, np.nan)
        self._check(self.L.emu_eval_mesh_error(ctypes.byref(self.desc), self._sc(), self._grid_ptr(self._grid),
                                               x.ctypes.data_as(_pd), err.ctypes.data_as(_pd), n_scen),
                    "gelato_eval_mesh_error")
        return err.reshape(self.plan.S, 11) if n_scen == 1 else err.reshape(n_scen, self.plan.S, 11)

    def path_check(self, x, n_scen=1):
        """engine.Engine.path_check: a call gelato_eval_path_check refuses raises engine.GelatoError with its reason."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        n = n_scen * self.plan.n_aero
        res, at = np.full(n, np.nan), np.full(n, -2, dtype=np.int32)
        self._check(self.L.emu_eval_path_check(ctypes.byref(self.desc), self._sc(), self._grid_ptr(self._grid),
                                               x.ctypes.data_as(_pd), res.ctypes.data_as(_pd), at.ctypes.data_as(_pi32),
                                               n_scen), "gelato_eval_path_check")
        return (res, at) if n_scen == 1 else (res.reshape(n_scen, -1), at.reshape(n_scen, -1))

    def eval_path_rows(self, x, n_scen=1, jacobian=True, out=None):
        """engine.Engine.eval_path_rows, in the emulator's finite-difference mode (set_fd)."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        grid, lay = self._prow if self._prow is not None else (None, {"n_rows": 0, "n_vals": 0})
        nr, nv = lay["n_rows"], lay["n_vals"]
        if out is not None:
            g = None if out[0] is None else engine._out(out[0], n_scen * nr, "out[0]")
            v = None if out[1] is None else engine._out(out[1], n_scen * nv, "out[1]")
        else:
            g, v = np.full(n_scen * nr, np.nan), (np.full(n_scen * nv, np.nan) if jacobian else None)
        self._check(self.L.emu_eval_path_rows(ctypes.byref(self.desc), self._sc(), self._grid_ptr(grid),
                                              x.ctypes.data_as(_pd), None if g is None else g.ctypes.data_as(_pd),
                                              None if v is None else v.ctypes.data_as(_pd), n_scen, *self._fd),
                    "gelato_eval_path_rows")
        if n_scen > 1:
            g, v = (None if a is None else a.reshape(n_scen, -1) for a in (g, v))
        return g, v

    # ---- one problem sharded over ranks (gelato_b200/batch.py: ShardedProblem) ----
    def block_counts(self):
        """(blocks of a pair evaluation, vacuum dynamics nodes): the two ranges a rank's share is cut from."""
        nb, nv = ctypes.c_int(0), ctypes.c_int(0)
        self.L.emu_block_counts(ctypes.byref(self.desc), ctypes.byref(nb), ctypes.byref(nv))
        return nb.value, nv.value

    def eval_pair_range(self, x, g, packed, blocks, vacuum):
        """The packed pair evaluation restricted to blocks [b0, b1) and vacuum nodes [v0, v1), written into the
        caller's g[n_rows] / packed[n_pack] (what gelato_eval_pair_packed_range_dev launches)."""
        if self.fd[0] != "forward":
            raise ValueError("the range evaluation supports forward differences only")
        x = np.ascontiguousarray(x, dtype=np.float64)
        assert g.dtype == np.float64 and g.flags.c_contiguous and g.size == self.plan.n_rows
        assert packed.dtype == np.float64 and packed.flags.c_contiguous and packed.size == self.n_pack
        rc = self.L.emu_eval_pair_range(ctypes.byref(self.desc), self._sc(), x.ctypes.data_as(_pd), g.ctypes.data_as(_pd),
                                        packed.ctypes.data_as(_pd), 1, blocks[0], blocks[1] - blocks[0], vacuum[0],
                                        vacuum[1] - vacuum[0])
        assert rc == 0


class EmuEngine(Emulator):
    """The emulator behind the Engine interface GelatoProblem uses (CPU test tier only)."""

    def __init__(self, plan, scenario_plans=None):
        super().__init__(plan, scenario_plans=scenario_plans)
        self.launches = self.calls = 0

    def eval_residuals(self, x, n_scen=1, out=None, scen_ids=None):
        self.launches += 1
        self.calls += 1
        return super().eval_residuals(x, n_scen, scen_ids)

    def eval_jacobian(self, x, n_scen=1, out=None, scen_ids=None):
        self.launches += 1
        self.calls += 1
        return super().eval_jacobian(x, n_scen, scen_ids)

    def eval_path_rows(self, x, n_scen=1, jacobian=True, out=None):
        self.calls += 1
        return super().eval_path_rows(x, n_scen, jacobian, out)

    # update mode as the drop-in's default `sens` uses it: one output buffer kept across calls
    class _HostArray:
        def __init__(self, n):
            self.array = np.empty(int(n))

        def free(self):
            self.array = None

    def alloc_output(self, n):
        return EmuEngine._HostArray(n)

    def jacobian_template(self, out, n_scen=1):
        assert n_scen == 1
        out[:] = self.plan.vals_template
        return out

    def eval_jacobian_update(self, x, out, n_scen=1):
        assert n_scen == 1
        v = self.eval_jacobian(x)
        idx = self.plan.xdep_index()
        out[idx] = v[idx]  # only the x-dependent slots move, as on the device
        return out

    def eval_pair_update(self, x, g_out, vals_out, n_scen=1):
        assert n_scen == 1
        self.launches += 1
        self.calls += 1
        g, v = self.eval_pair(x)
        g_out[:] = g
        idx = self.plan.xdep_index()
        vals_out[idx] = v[idx]
        return g_out.reshape(1, -1), vals_out.reshape(1, -1)

    def close(self):
        pass
