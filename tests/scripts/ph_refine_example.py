#!/usr/bin/env python
"""ph-refinement rounds of the shipped example on the GPU (DESIGN.md section 11).  From the converged example solution
(tests/golden/example_solution.npz), each round estimates the collocation error per LGR interval
(GelatoProblem.mesh_error_intervals), applies refine_nodes(..., n_min, n_max) with the path check as `path` (a raised
degree up to n_max, else a split into intervals of n_min nodes), transfers the solution onto the new mesh and re-solves
it with the redsqp stand-in (NOT IPOPT) on the CUDA callbacks, optionally with path rows (--path-rows: the aero limits
as NLP rows at the n_k + 1 test points of every interval).  It stops when every interval is at or below --tol and no
path residual is below -path_tol, or after --rounds.  One JSON line per stage: nodes and intervals per section, the
largest estimate per section, the path check on a dense grid (--dense test points per interval), and the solver's
status, iterations, payload and wall time, with the card's name and power limit.

    python tests/scripts/ph_refine_example.py [--tol 1e-6] [--n-min 4] [--n-max 12] [--rounds 4] [--path-rows]
        [--out profiles/r09a_ph_refine_example.jsonl]
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


def dense_path_check(prob, x, m):
    """GelatoProblem.path_check on a grid of m test points per interval; the default grid is set back afterwards."""
    default = prob._default_mesh_grid()
    prob._mesh_grid = mesh.grid_tables(prob.plan.ps, m=m)
    prob.engine.set_mesh_grid(prob._mesh_grid)
    try:
        return prob.path_check(x)
    finally:
        prob._mesh_grid = default
        prob.engine.set_mesh_grid(default)


def stage(name, prob, x, p, dense, extra):
    """(record, per-interval estimate, path check on the default grid)"""
    ps = p["ps_params"]
    err = prob.mesh_error_intervals(x)
    pc = prob.path_check(x)
    pd = dense_path_check(prob, x, dense)
    rec = {"stage": name, "nodes": int(p["N"]),
           "intervals": int(sum(len(ps.intervals(i)[0]) for i in range(ps.num_sections()))),
           "sections": [{"event": k, "n": int(ps.nodes(i)), "intervals": list(ps.intervals(i)[0]),
                         "err_max": float(np.max(v))} for i, (k, v) in enumerate(err.items())],
           "err_max": float(max(np.max(v) for v in err.values())),
           "path_dense": [{"constraint": key, "event": ev, "residual": r, "time_s": t} for (key, ev), (r, t) in pd.items()],
           "path_dense_min": float(min([r for r, _ in pd.values()] or [np.inf]))}
    rec.update(extra)
    return rec, err, pc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tol", type=float, default=1e-6)
    ap.add_argument("--n-min", type=int, default=4)
    ap.add_argument("--n-max", type=int, default=12)
    ap.add_argument("--path-tol", type=float, default=1e-3)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--path-rows", action="store_true")
    ap.add_argument("--dense", type=int, default=40)
    ap.add_argument("--maxiter", type=int, default=1800)
    ap.add_argument("--out", default=os.path.join(mre.ROOT, "profiles", "r09a_ph_refine_example.jsonl"))
    a = ap.parse_args()
    from gelato_b200 import redsqp
    from oracle import leaves

    Lg = leaves.get("gmath")
    info = mre.gpu_info()
    user = callbacks.PerigeeAtEvent(helpers.USER_EVENT)
    inp = helpers.example_inputs()
    p, u, c, _ = helpers.example_problem(coord=Lg.coordinate_c)
    prob = callbacks.GelatoProblem(p, u, c, user_eq=user, coord=Lg.coordinate_c)
    P = prob.plan
    x = problem.vector_to_xdict(np.load(os.path.join(helpers.GOLDEN, "example_solution.npz"))["x"], P.M, P.N, P.S)
    events = inp["events"]
    rec, err, pc = stage("example solution", prob, x, p, a.dense, dict(info, round=0))
    lines = [rec]
    print(json.dumps({k: v for k, v in rec.items() if k not in ("sections", "path_dense")}), flush=True)
    for rnd in range(1, a.rounds + 1):
        t_ev = np.asarray(x["t"]) * u["t"]
        events, report = mesh.refine_nodes(events, err, a.tol, a.n_max, path=pc, path_tol=a.path_tol, n_min=a.n_min,
                                           t_events=t_ev)
        if all(r.n_new == r.n_old and r.split == 1 for r in report):
            lines[-1]["converged"] = True
            break
        inp2 = dict(inp, events=events)
        p2, u2, c2, _ = problem.problem_from_inputs(inp2, coord=Lg.coordinate_c)
        x2 = mesh.transfer(x, p["ps_params"], p2["ps_params"])
        prob.close()
        path_grid = mesh.grid_tables(p2["ps_params"]) if a.path_rows else None
        prob = callbacks.GelatoProblem(p2, u2, c2, user_eq=user, coord=Lg.coordinate_c, path_grid=path_grid)
        opt = nlpshim.attach_structure(nlpshim.register(prob.objfunc, prob.sens, helpers.copy_x(x2), c2), p2)
        t0 = time.perf_counter()
        sol = redsqp.ReducedSQP({"max_iter": a.maxiter})(opt, sens=prob.sens)
        wall = time.perf_counter() - t0
        x, p, u = sol.xStar, p2, u2
        rec, err, pc = stage("round %d re-solved" % rnd, prob, x, p, a.dense, dict(
            info, round=rnd, tol=a.tol, n_min=a.n_min, n_max=a.n_max, path_tol=a.path_tol, path_rows=a.path_rows,
            refinement=[r._asdict() for r in report], solver="redsqp (NOT IPOPT)", status=sol.status,
            message=sol.message, nit=sol.nit, optimality=sol.optimality, constr_violation=sol.constr_violation,
            payload_kg=float(x["mass"][0] * u["mass"]), wall_s=wall))
        lines.append(rec)
        print(json.dumps({k: v for k, v in rec.items() if k not in ("sections", "path_dense", "refinement")}), flush=True)
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")
    prob.close()


if __name__ == "__main__":
    sys.exit(main())
