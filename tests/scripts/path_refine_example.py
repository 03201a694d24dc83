#!/usr/bin/env python
"""The path check in a refinement of the shipped example on the GPU (DESIGN.md section 11): every stage of
mesh_refine_example.py --solve (the example solution, one p-refinement at --tol by the estimate alone, the transferred
point, its re-solve by the redsqp stand-in, NOT IPOPT) with, per stage, the aero constraints between the nodes
(GelatoProblem.path_check) next to their node rows; then a second round refined by the estimate and the path residuals
together (refine_nodes(..., path=..., path_tol=--path-tol)), transferred, re-solved and checked again.  Its record says
whether each section ends at or above -path_tol.  One JSON line per stage, with the card's name and power limit.

    python tests/scripts/path_refine_example.py [--tol 1e-6] [--n-max 30] [--path-tol 1e-3]
        [--out profiles/r06a_path_refine_example.jsonl]
"""
import argparse
import json
import os
import sys

import numpy as np

import mesh_refine_example as mre  # noqa: E402  (also puts the repository and tests/ on sys.path)
import helpers  # noqa: E402
from gelato_b200 import callbacks, mesh, nlpshim, problem  # noqa: E402

AERO_KEYS = ("ineqcon_alpha", "ineqcon_q", "ineqcon_qalpha")


def node_rows(plan, g, key, name):
    """objfunc's rows of the aero job `key` over the section of event `name` (what the solver holds >= 0)."""
    kind, i = AERO_KEYS.index(key), plan.p["event_index"][name]
    r0 = 0
    for k, sec, nk, _ in plan.aero_i32:
        if k == kind and sec == i:
            return np.atleast_1d(g[key])[r0:r0 + nk]
        if k == kind:
            r0 += nk
    raise KeyError((key, name))


def stage(name, prob, x, p, extra=None):
    """mesh_refine_example.stage plus the path check: (record, estimate, path check)."""
    rec, err = mre.stage(name, prob, x, p, extra)
    pc = prob.path_check(x)
    g = prob.plan.split_residuals(prob.residuals(prob.pack(x)))
    rec["path"] = [{"constraint": key, "event": ev, "n": int(p["ps_params"].nodes(p["event_index"][ev])),
                    "residual_between_nodes": r, "time_s": t_s,
                    "residual_at_nodes": float(np.min(node_rows(prob.plan, g, key, ev)))}
                   for (key, ev), (r, t_s) in pc.items()]
    return rec, err, pc


def resolve(prob, x, c, p, u, maxiter):
    from gelato_b200 import redsqp

    opt = nlpshim.attach_structure(nlpshim.register(prob.objfunc, prob.sens, helpers.copy_x(x), c), p)
    sol = redsqp.ReducedSQP({"max_iter": maxiter})(opt, sens=prob.sens)
    return sol, dict(solver="redsqp (NOT IPOPT)", status=sol.status, message=sol.message, nit=sol.nit,
                     optimality=sol.optimality, constr_violation=sol.constr_violation,
                     payload_kg=float(sol.xStar["mass"][0] * u["mass"]))


def refined(inp, events, x, ps_old, user, Lg):
    """(problem, GelatoProblem, transferred x) of the inputs with `events`."""
    inp["events"] = events
    p2, u2, c2, _ = problem.problem_from_inputs(inp, coord=Lg.coordinate_c)
    prob2 = callbacks.GelatoProblem(p2, u2, c2, user_eq=user, coord=Lg.coordinate_c)
    return (p2, u2, c2), prob2, mesh.transfer(x, ps_old, p2["ps_params"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tol", type=float, default=1e-6)
    ap.add_argument("--n-max", type=int, default=30)
    ap.add_argument("--path-tol", type=float, default=1e-3)
    ap.add_argument("--maxiter", type=int, default=1800)
    ap.add_argument("--out", default=os.path.join(mre.ROOT, "profiles", "r06a_path_refine_example.jsonl"))
    a = ap.parse_args()
    from oracle import leaves

    Lg = leaves.get("gmath")
    info = mre.gpu_info()
    user = callbacks.PerigeeAtEvent(helpers.USER_EVENT)
    p, u, c, _ = helpers.example_problem(coord=Lg.coordinate_c)
    prob = callbacks.GelatoProblem(p, u, c, user_eq=user, coord=Lg.coordinate_c)
    P = prob.plan
    x_sol = problem.vector_to_xdict(np.load(os.path.join(helpers.GOLDEN, "example_solution.npz"))["x"], P.M, P.N, P.S)
    probs, lines = [prob], []
    rec, err, _ = stage("example solution", prob, x_sol, p, info)
    lines.append(rec)
    # round 1: the estimate alone, as mesh_refine_example.py --solve
    inp = helpers.example_inputs()
    events, report = mesh.refine_nodes(inp["events"], err, a.tol, a.n_max)
    (p2, u2, c2), prob2, x2 = refined(inp, events, x_sol, p["ps_params"], user, Lg)
    probs.append(prob2)
    rec, _, _ = stage("transferred", prob2, x2, p2, dict(info, tol=a.tol, n_max=a.n_max,
                                                          refinement=[r._asdict() for r in report]))
    lines.append(rec)
    sol, extra = resolve(prob2, x2, c2, p2, u2, a.maxiter)
    rec, err2, pc2 = stage("re-solved", prob2, sol.xStar, p2, dict(
        info, payload_kg_before=float(x_sol["mass"][0] * u["mass"]), **extra))
    lines.append(rec)
    # round 2: the estimate and the path residuals
    events, report = mesh.refine_nodes(inp["events"], err2, a.tol, a.n_max, path=pc2, path_tol=a.path_tol)
    (p3, u3, c3), prob3, x3 = refined(inp, events, sol.xStar, p2["ps_params"], user, Lg)
    probs.append(prob3)
    sol3, extra = resolve(prob3, x3, c3, p3, u3, a.maxiter)
    rec, _, pc3 = stage("path round re-solved", prob3, sol3.xStar, p3, dict(
        info, tol=a.tol, n_max=a.n_max, path_tol=a.path_tol, refinement=[r._asdict() for r in report], **extra))
    rec["path_min"] = float(min(r for r, _ in pc3.values()))
    rec["above_minus_path_tol"] = {ev: bool(r >= -a.path_tol) for (_, ev), (r, _) in pc3.items()}
    lines.append(rec)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
            print(json.dumps({k: v for k, v in rec.items() if k not in ("sections", "refinement")}), flush=True)
    for pr in probs:
        pr.close()


if __name__ == "__main__":
    sys.exit(main())
