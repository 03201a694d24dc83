#!/usr/bin/env python
"""Re-solve the shipped example with a result-table user constraint (DESIGN.md section 10 "a16"): from the recorded
solution (tests/golden/example_solution.npz), gelato_b200/redsqp.py (the host stand-in solver, not IPOPT) with the
example's PerigeeAtEvent("IIP_END") and an inequality TableAtEvent that is active there -- the altitude at the first
node of SEIG (second-stage ignition) at least `--margin` above its value in the recorded solution:

    ineqcon_user = altitude(SEIG) / h_rec - (1 + margin) >= 0

The arms run the same solve on the oracle's callbacks (tests/table_oracle.py through oracle.nlp) and on the CUDA
callbacks (GelatoProblem; "emu": the host emulator of the kernels), recording every decision vector the solver
evaluates.  Prints one JSON line per arm (status, iterations, payload, the constraint's value and the result table's
altitude at that node) and the largest |dx| between the arms' iterates.

    python tests/scripts/user_table_example.py --arm both [--margin 0.01] [--out profiles/r11c_user_table_example.jsonl]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
EVENT = "SEIG"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--arm", choices=["oracle", "cuda", "emu", "both"], default="both")
    ap.add_argument("--margin", type=float, default=0.01)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import helpers
    import table_oracle
    from gelato_b200 import callbacks, nlpshim, output, problem, redsqp
    from gelato_b200 import plan as gplan
    from oracle import leaves, nlp, user_builtin

    Lg = leaves.get("gmath")
    p, u, c, _ = problem.problem_from_inputs(helpers.variant_inputs("example"), coord=Lg.coordinate_c, factor=1, max_nodes=20)
    rec = np.load(os.path.join(ROOT, "tests", "golden", "example_solution.npz"))
    xs = problem.vector_to_xdict(rec["x"], p["M"], p["N"], p["num_sections"])
    i = p["event_index"][EVENT]
    row = p["ps_params"].index_start_u(i) + i

    def table_altitude(x):
        """the result table's altitude at the event's first node (the oracle's output_row, which the kernels match)"""
        prm = p["params"][i]
        cols = table_oracle.output_row(Lg, x["mass"][row: row + 1] * u["mass"], x["position"][3 * row: 3 * row + 3] * u["position"],
                                       x["velocity"][3 * row: 3 * row + 3] * u["velocity"], x["quaternion"][4 * row: 4 * row + 4],
                                       x["t"][i: i + 1] * u["t"], [prm["thrust"]], [prm["reference_area"]], [prm["nozzle_area"]],
                                       p["wind_table"], p["ca_table"], p["LaunchCondition"]["lat"], p["LaunchCondition"]["lon"])
        return float(cols[output.KERNEL_COLUMNS.index("altitude")])

    h_rec = table_altitude(xs)
    rows = [("altitude", h_rec, 1.0 + a.margin)]
    arms = ["oracle", "cuda"] if a.arm == "both" else [a.arm]
    out, paths = [], {}
    for arm in arms:
        if arm == "oracle":
            O = nlp.OracleNLP(p, u, c, "gmath", "seqfma", user_eq=user_builtin.perigee_ratio_at(Lg, helpers.USER_EVENT),
                              user_ineq=table_oracle.table_rows_at(Lg, EVENT, rows))
            objfunc, sens, close = (lambda x: O.objfunc(x)), (lambda x, f=None: O.sens(x)), (lambda: None)
        else:
            kw = {}
            if arm == "emu":
                import emu_table

                kw["engine_factory"] = emu_table.TableEmuEngine
            prob = callbacks.GelatoProblem(p, u, c, user_eq=callbacks.PerigeeAtEvent(helpers.USER_EVENT),
                                           user_ineq=gplan.TableAtEvent(EVENT, rows), coord=Lg.coordinate_c, **kw)
            objfunc, sens, close = prob.objfunc, prob.sens, prob.close
        seen = []

        def rec_objfunc(x, objfunc=objfunc, seen=seen):
            seen.append(problem.xdict_to_vector(x).copy())
            return objfunc(x)

        opt = nlpshim.register(rec_objfunc, sens, helpers.copy_x(xs), c)
        sol = redsqp.ReducedSQP({"phase1_evals": 0, "penalty0": float(rec["multiplier"]) / 10.0 ** 0.5, "penalty_levels": 2,
                                 "level_iter": 50, "max_iter": 300})(opt, sens=sens)
        f, _ = objfunc(helpers.copy_x(sol.xStar))
        doc = {"arm": arm, "status": int(sol.status), "iterations": int(sol.nit),
               "constr_violation": float(sol.constr_violation),
               "payload_kg": float(sol.xStar["mass"][0] * u["mass"]), "payload_rec_kg": float(rec["payload_kg"]),
               "altitude_rec_m": h_rec, "altitude_bound_m": h_rec * (1.0 + a.margin),
               "ineqcon_user": float(f["ineqcon_user"]), "table_altitude_m": table_altitude(sol.xStar),
               "evaluations": len(seen)}
        out.append(doc)
        paths[arm] = seen
        print(json.dumps(doc))
        close()
    if len(arms) == 2:
        A, B = paths[arms[0]], paths[arms[1]]
        dx = max(float(np.max(np.abs(x - y))) for x, y in zip(A, B)) if len(A) == len(B) else float("inf")
        doc = {"iterates": [len(A), len(B)], "max_abs_dx": dx}
        out.append(doc)
        print(json.dumps(doc))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write("".join(json.dumps(d) + "\n" for d in out))


if __name__ == "__main__":
    main()
