#!/usr/bin/env python
"""Mesh refinement of the shipped example on the GPU (DESIGN.md section 11): the collocation error estimate of the
converged example solution (tests/golden/example_solution.npz), one p-refinement at --tol, the solution transferred
onto the refined mesh and estimated again; with --solve the refined problem is re-solved by the redsqp stand-in (NOT
IPOPT) from the transferred point and estimated a third time.  One JSON line per stage, with the card's name and power
limit.

    python tests/scripts/mesh_refine_example.py [--tol 1e-6] [--n-max 30] [--solve] [--out profiles/r04a_mesh_refine_example.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers  # noqa: E402
from gelato_b200 import callbacks, mesh, nlpshim, problem  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.splitlines()[0].split(",")
    return {"gpu": q[0].strip(), "power_limit": q[1].strip()}


def stage(name, prob, x, p, extra=None):
    t0 = time.perf_counter()
    err = prob.mesh_error(x)
    ms = (time.perf_counter() - t0) * 1e3
    rec = {"stage": name, "nodes": int(p["N"]), "host_call_ms": ms,
           "sections": [{"event": k, "n": int(p["ps_params"].nodes(i)), "err_max": float(np.max(v)),
                         "worst_component": int(np.argmax(v))} for i, (k, v) in enumerate(err.items())],
           "err_max": float(max(np.max(v) for v in err.values()))}
    rec.update(extra or {})
    return rec, err


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tol", type=float, default=1e-6)
    ap.add_argument("--n-max", type=int, default=30)
    ap.add_argument("--solve", action="store_true")
    ap.add_argument("--maxiter", type=int, default=1800)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04a_mesh_refine_example.jsonl"))
    a = ap.parse_args()
    from oracle import leaves

    Lg = leaves.get("gmath")
    info = gpu_info()
    user = callbacks.PerigeeAtEvent(helpers.USER_EVENT)
    p, u, c, _ = helpers.example_problem(coord=Lg.coordinate_c)
    prob = callbacks.GelatoProblem(p, u, c, user_eq=user, coord=Lg.coordinate_c)
    P = prob.plan
    x_sol = problem.vector_to_xdict(np.load(os.path.join(helpers.GOLDEN, "example_solution.npz"))["x"], P.M, P.N, P.S)
    lines = []
    rec, err = stage("example solution", prob, x_sol, p, info)
    lines.append(rec)
    inp = helpers.example_inputs()
    inp["events"], report = mesh.refine_nodes(inp["events"], err, a.tol, a.n_max)
    p2, u2, c2, _ = problem.problem_from_inputs(inp, coord=Lg.coordinate_c)
    x2 = mesh.transfer(x_sol, p["ps_params"], p2["ps_params"])
    prob2 = callbacks.GelatoProblem(p2, u2, c2, user_eq=user, coord=Lg.coordinate_c)
    rec, _ = stage("transferred", prob2, x2, p2, dict(info, tol=a.tol, n_max=a.n_max,
                                                       refinement=[r._asdict() for r in report]))
    lines.append(rec)
    if a.solve:
        from gelato_b200 import redsqp

        opt = nlpshim.attach_structure(nlpshim.register(prob2.objfunc, prob2.sens, helpers.copy_x(x2), c2), p2)
        sol = redsqp.ReducedSQP({"max_iter": a.maxiter})(opt, sens=prob2.sens)
        rec, _ = stage("re-solved", prob2, sol.xStar, p2, dict(
            info, solver="redsqp (NOT IPOPT)", status=sol.status, message=sol.message, nit=sol.nit,
            optimality=sol.optimality, constr_violation=sol.constr_violation,
            payload_kg=float(sol.xStar["mass"][0] * u2["mass"]),
            payload_kg_before=float(x_sol["mass"][0] * u["mass"])))
        lines.append(rec)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
            print(json.dumps({k: v for k, v in rec.items() if k not in ("sections", "refinement")}), flush=True)
    prob.close()
    prob2.close()


if __name__ == "__main__":
    main()
