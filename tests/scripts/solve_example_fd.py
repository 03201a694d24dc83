#!/usr/bin/env python
"""The shipped example solved by the redsqp stand-in (NOT IPOPT) with the Jacobian in a chosen finite-difference mode
(DESIGN.md H6), once on the CPU oracle's callbacks (tests/central_oracle.py) and once on the CUDA callbacks
(GelatoProblem(derivative=...)): same solver, same problem, same start.  Prints one JSON line per arm in the fields of
tests/scripts/solve_example.py, which runs the same solve with forward differences, then whether the iterates of the two
arms are identical.

    python tests/scripts/solve_example_fd.py [--arm cpu|gpu|both] [--derivative central|forward] [--fd-step 1e-6]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers  # noqa: E402
from gelato_b200 import nlpshim, problem  # noqa: E402


def run(arm, derivative, fd_step, maxiter):
    from gelato_b200 import redsqp
    from oracle import leaves, user_builtin

    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    if arm == "cpu":
        from central_oracle import CentralOracleNLP

        O = CentralOracleNLP(p, u, c, "gmath", "seqfma", user_eq=user_builtin.perigee_ratio_at(Lg, helpers.USER_EVENT),
                             derivative=derivative, fd_step=fd_step)
        objfunc, sens = O.objfunc, (lambda x, f=None: O.sens(x))
    else:
        from gelato_b200 import callbacks

        prob = callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT), coord=Lg.coordinate_c,
                                       derivative=derivative, fd_step=fd_step)
        objfunc, sens = prob.objfunc, prob.sens
    opt = nlpshim.attach_structure(nlpshim.register(objfunc, sens, helpers.copy_x(x0), c), p)
    sol = redsqp.ReducedSQP({"max_iter": maxiter})(opt, sens=sens)
    out = {
        "arm": arm, "derivative": derivative, "fd_step": fd_step, "solver": "redsqp (NOT IPOPT)",
        "penalty_levels": sol.penalty_levels, "optimality": sol.optimality, "nodes": int(p["N"]), "nit": sol.nit,
        "status": sol.status, "message": sol.message, "obj": float(sol.fStar), "constr_violation": sol.constr_violation,
        "payload_kg": float(sol.xStar["mass"][0] * u["mass"]),
        "event_times_s": [float(v) for v in sol.xStar["t"] * u["t"]],
        "optTime": sol.optTime, "userObjTime": sol.userObjTime, "userObjCalls": sol.userObjCalls,
        "userSensTime": sol.userSensTime, "userSensCalls": sol.userSensCalls,
    }
    return out, problem.xdict_to_vector(sol.xStar)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--arm", default="both", choices=["cpu", "gpu", "both"])
    ap.add_argument("--derivative", default="central", choices=["forward", "central"])
    ap.add_argument("--fd-step", type=float, default=None, help="central step (default: engine.DEFAULT_FD_STEP)")
    ap.add_argument("--maxiter", type=int, default=1800)
    a = ap.parse_args()
    res = {}
    for arm in (["cpu", "gpu"] if a.arm == "both" else [a.arm]):
        res[arm] = run(arm, a.derivative, a.fd_step, a.maxiter)
        print(json.dumps(res[arm][0]), flush=True)
    if len(res) == 2:
        xa, xb = res["cpu"][1], res["gpu"][1]
        print(json.dumps({"max_abs_diff_x": float(np.max(np.abs(xa - xb))), "identical_iterates": bool(np.array_equal(xa, xb))}))


if __name__ == "__main__":
    main()
