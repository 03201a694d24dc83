"""Oracle-side result-table user constraints (TEST INFRASTRUCTURE ONLY).

`table_rows_at` is the function a gelato_b200.plan.TableAtEvent stands for, written the way a GELATO user would write
it in user_constraints.py: read the event's first node from xdict, call the result table's per-node body
(oracle_leaves.cpp: output_row, the oracle's restatement of output_result.py:130-261) and return column / scale -
offset.  The oracle's jac_fd then runs over it like over any user function.  `group_rows_at` concatenates the rows of
several such functions -- a user_constraints.py whose function returns them all.
"""
import ctypes

import numpy as np

from oracle import output as oracle_output
from oracle import user_builtin

_P = ctypes.POINTER(ctypes.c_double)


def output_row(leaves, mass, pos, vel, quat, t, thrust, area, nozzle, wind, ca, lat0, lon0):
    """The 34 columns of one node (oracle.output.KERNEL_COLUMNS order)."""
    a = [np.ascontiguousarray(v, dtype=np.float64) for v in (mass, pos, vel, quat, t, thrust, area, nozzle)]
    wind = np.ascontiguousarray(wind, dtype=np.float64)
    ca = np.ascontiguousarray(ca, dtype=np.float64)
    out = np.empty(len(oracle_output.KERNEL_COLUMNS))
    p = lambda v: v.ctypes.data_as(_P)  # noqa: E731
    leaves.lib.o_output_rows(ctypes.c_int(1), *[p(v) for v in a], p(wind), ctypes.c_int(wind.shape[0]), p(ca),
                             ctypes.c_int(ca.shape[0]), ctypes.c_double(lat0), ctypes.c_double(lon0), p(out))
    return out


def table_rows_at(leaves, event_name, rows):
    """rows: [(column, scale, offset)] -> user function of (xdict, pdict, unitdict, condition)."""
    cols = [oracle_output.KERNEL_COLUMNS.index(c) for c, _, _ in rows]

    def user(xdict, pdict, unitdict, condition):
        i = pdict["event_index"][event_name]
        a2 = pdict["ps_params"].index_start_u(i) + i
        prm = pdict["params"][i]
        out = output_row(leaves, xdict["mass"][a2: a2 + 1] * unitdict["mass"],
                         xdict["position"][a2 * 3: (a2 + 1) * 3] * unitdict["position"],
                         xdict["velocity"][a2 * 3: (a2 + 1) * 3] * unitdict["velocity"],
                         xdict["quaternion"][a2 * 4: (a2 + 1) * 4], xdict["t"][i: i + 1] * unitdict["t"],
                         [prm["thrust"]], [prm["reference_area"]], [prm["nozzle_area"]], pdict["wind_table"],
                         pdict["ca_table"], pdict["LaunchCondition"]["lat"], pdict["LaunchCondition"]["lon"])
        vals = [(out[c] / scale) - offset for c, (_, scale, offset) in zip(cols, rows)]
        return vals[0] if len(vals) == 1 else np.array(vals)

    return user


def group_rows_at(leaves, parts):
    """parts: [("orbit" | "table", event_name, rows)] -> ONE user function returning all their rows in order."""
    fns = [(user_builtin.orbit_rows_at if kind == "orbit" else table_rows_at)(leaves, ev, rows) for kind, ev, rows in parts]

    def user(xdict, pdict, unitdict, condition):
        vals = np.concatenate([np.atleast_1d(f(xdict, pdict, unitdict, condition)) for f in fns])
        return vals[0] if vals.size == 1 else vals

    return user
