#!/usr/bin/env python
"""The shipped example re-solved with path rows (DESIGN.md section 11) on the GPU: GelatoProblem(..., path_grid=
mesh.grid_tables(ps)) -- Q-alpha enforced at the default grid's test points between the nodes as "ineqcon_path" --
solved by the redsqp stand-in (NOT IPOPT) from the example solution on the CUDA callbacks.  Records, before and after:
the minimum of the aero node rows and of the path rows, and the path check on a dense grid (m = --dense test points per
section, separate from the path rows' grid); after: the solver's status, iterations, payload and wall time.  One JSON
line per stage, with the card's name and power limit.

    python tests/scripts/path_rows_example.py [--dense 64] [--maxiter 1800] [--out profiles/r07a_path_rows_example.jsonl]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

import mesh_refine_example as mre  # noqa: E402  (also puts the repository and tests/ on sys.path)
import helpers  # noqa: E402
from gelato_b200 import callbacks, mesh, nlpshim, problem  # noqa: E402

AERO_KEYS = ("ineqcon_alpha", "ineqcon_q", "ineqcon_qalpha")


def stage(name, prob, x, dense, extra):
    """The rows the solver holds and the path check on the dense grid at x."""
    f, _ = prob.objfunc(x)
    node = min(float(np.min(f[k])) for k in AERO_KEYS if f[k] is not None)
    pc = prob.path_check(x)
    rec = dict(extra, stage=name, node_rows_min=node, path_rows_min=float(np.min(f["ineqcon_path"])),
               path_rows=int(np.size(f["ineqcon_path"])), dense_grid_m=dense,
               dense_path_check=[{"constraint": k, "event": ev, "residual": r, "time_s": t} for (k, ev), (r, t) in pc.items()])
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dense", type=int, default=64)
    ap.add_argument("--maxiter", type=int, default=1800)
    ap.add_argument("--out", default=os.path.join(mre.ROOT, "profiles", "r07a_path_rows_example.jsonl"))
    a = ap.parse_args()
    from gelato_b200 import redsqp
    from oracle import leaves

    Lg = leaves.get("gmath")
    info = mre.gpu_info()
    p, u, c, _ = helpers.example_problem(coord=Lg.coordinate_c)
    prob = callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT), coord=Lg.coordinate_c,
                                   path_grid=mesh.grid_tables(p["ps_params"]))
    prob._mesh_grid = mesh.grid_tables(p["ps_params"], m=a.dense)  # path_check on the dense grid
    prob.engine.set_mesh_grid(prob._mesh_grid)
    P = prob.plan
    x_sol = problem.vector_to_xdict(np.load(os.path.join(helpers.GOLDEN, "example_solution.npz"))["x"], P.M, P.N, P.S)
    lines = [stage("example solution", prob, x_sol, a.dense,
                   dict(info, payload_kg=float(x_sol["mass"][0] * u["mass"])))]
    opt = nlpshim.attach_structure(nlpshim.register(prob.objfunc, prob.sens, helpers.copy_x(x_sol), c), p)
    t0 = time.perf_counter()
    sol = redsqp.ReducedSQP({"max_iter": a.maxiter})(opt, sens=prob.sens)
    wall = time.perf_counter() - t0
    lines.append(stage("re-solved with path rows", prob, sol.xStar, a.dense, dict(
        info, solver="redsqp (NOT IPOPT)", status=sol.status, message=sol.message, nit=sol.nit,
        optimality=sol.optimality, constr_violation=sol.constr_violation, wall_s=wall,
        payload_kg=float(sol.xStar["mass"][0] * u["mass"]), payload_kg_before=float(x_sol["mass"][0] * u["mass"]))))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
            print(json.dumps(rec), flush=True)
    prob.close()


if __name__ == "__main__":
    sys.exit(main())
