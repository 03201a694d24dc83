#!/usr/bin/env python
"""Device time of the per-interval mesh error estimate and of a pair step on a composite mesh (DESIGN.md section 11),
at the benchmark workload: 128 dispersed scenarios of the example x15 (bench.load_workload's inputs and perturbation).
Two meshes of the same node counts: the benchmark's, and the same with two sections split into LGR intervals
(ZEROLIFT_START 10 | 10, ZEROLIFT_START__1 7 | 7 | 6).  Alternated in one process, each call bracketed by CUDA events on
the launch stream after a 256 MiB write that evicts L2:
    mesh_error_dev on the single-interval grid | mesh_error_dev and mesh_error_intervals_dev on the composite grid |
    the packed pair step on the unsplit mesh | the packed pair step on the composite mesh.
Writes one JSON document with the card's name, power limit and max SM clock.

    python tests/scripts/mesh_interval_timing.py [--reps 200] [--out profiles/r09b_mesh_interval_timing.json]
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

SPLITS = {"ZEROLIFT_START": [10, 10], "ZEROLIFT_START__1": [7, 7, 6]}


def workload(B, factor, split):
    """plans and perturbed decision vectors of bench.load_workload, with SPLITS applied when `split`"""
    import bench
    from gelato_b200 import plan as gplan
    from gelato_b200 import problem, scenarios

    scen = scenarios.disperse(bench.workload_inputs("example"), B, seed=20260117)
    plans, xs = [], []
    for k in range(B):
        inp = copy.deepcopy(scen[k])
        inp["events"], inp["settings"]["FlightConstraint"] = problem.refine_events(
            inp["events"], inp["settings"]["FlightConstraint"], factor, 20)
        for e in inp["events"]:
            if split and e["name"] in SPLITS:
                assert e["num_nodes"] == sum(SPLITS[e["name"]])
                e["mesh_intervals"] = SPLITS[e["name"]]
        p, u, c, x0 = problem.problem_from_inputs(inp)
        rng = np.random.default_rng(1000 + k)
        x = {key: v + (0.0 if key == "t" else 1e-3) * rng.uniform(-1.0, 1.0, v.shape) for key, v in x0.items()}
        plans.append(gplan.CompiledPlan(p, u, c, user_eq=gplan.PerigeeAtEvent(bench.USER_EVENT)))
        xs.append(problem.xdict_to_vector(x))
    return plans, np.stack(xs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--scenarios", type=int, default=128)
    ap.add_argument("--factor", type=int, default=15)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09b_mesh_interval_timing.json"))
    a = ap.parse_args()
    import torch

    from gelato_b200 import engine, mesh

    if not torch.cuda.is_available():
        raise SystemExit("mesh_interval_timing.py: no CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.splitlines()[0].split(",")
    B = a.scenarios
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    side = {}
    for name, split in (("plain", False), ("split", True)):
        plans, X = workload(B, a.factor, split)
        P = plans[0]
        E = engine.Engine(P, device=0, scenario_plans=plans)
        tabs = mesh.grid_tables(P.ps)
        E.set_mesh_grid(tabs)
        n_pack = int(E.L.gelato_plan_n_pack(E.h))
        side[name] = {"P": P, "E": E, "tabs": tabs, "x": torch.from_numpy(X).cuda(),
                      "err": torch.empty((B, P.S, 11), dtype=torch.float64, device="cuda"),
                      "err_int": torch.empty((B, E.n_mesh_int, 11), dtype=torch.float64, device="cuda"),
                      "g": torch.empty((B, P.n_rows), dtype=torch.float64, device="cuda"),
                      "pk": torch.empty((B, n_pack), dtype=torch.float64, device="cuda")}
    pl, sp = side["plain"], side["split"]
    assert (pl["P"].n_vals, pl["P"].n_rows) == (sp["P"].n_vals, sp["P"].n_rows)
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")
    calls = {
        "mesh_error_dev_single": lambda: pl["E"].mesh_error_dev(pl["x"].data_ptr(), pl["err"].data_ptr(), B, st.cuda_stream),
        "mesh_error_dev_composite": lambda: sp["E"].mesh_error_dev(sp["x"].data_ptr(), sp["err"].data_ptr(), B,
                                                                   st.cuda_stream),
        "mesh_error_intervals_dev_composite": lambda: sp["E"].mesh_error_intervals_dev(
            sp["x"].data_ptr(), sp["err_int"].data_ptr(), B, st.cuda_stream),
        "pair_packed_dev_unsplit": lambda: pl["E"].eval_pair_packed_dev(pl["x"].data_ptr(), pl["g"].data_ptr(),
                                                                        pl["pk"].data_ptr(), B, st.cuda_stream),
        "pair_packed_dev_composite": lambda: sp["E"].eval_pair_packed_dev(sp["x"].data_ptr(), sp["g"].data_ptr(),
                                                                          sp["pk"].data_ptr(), B, st.cuda_stream),
    }
    for fn in calls.values():  # warm-up: module load, scratch allocation
        for _ in range(5):
            fn()
    st.synchronize()
    times = {k: [] for k in calls}
    for r in range(a.reps):
        for name, fn in calls.items():
            flush.fill_(float(r))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            fn()
            e1.record(st)
            times[name].append((e0, e1))
    st.synchronize()
    res = {}
    for name, evs in times.items():
        ms = np.array([s.elapsed_time(e) for s, e in evs])
        res[name] = {"median_ms": float(np.median(ms)), "p10_ms": float(np.percentile(ms, 10)),
                     "p90_ms": float(np.percentile(ms, 90)), "min_ms": float(ms.min())}
    ei = sp["err_int"].cpu().numpy()
    doc = {"gpu": q[0].strip(), "power_limit": q[1].strip(), "clocks_max_sm": q[2].strip(),
           "workload": "example x%d, %d dispersed scenarios, N=%d, S=%d; composite: %s as LGR intervals, %d intervals"
                       % (a.factor, B, pl["P"].N, pl["P"].S, SPLITS, sp["E"].n_mesh_int),
           "test_points": {k: int(v["tabs"]["m"].sum()) for k, v in side.items()},
           "l2": "256 MiB write before every timed call (inputs and scratch read from HBM)",
           "timing": "CUDA events around each call on the launch stream, %d calls each, all entries alternating" % a.reps,
           "results": res,
           "err_int_max_over_batch": float(np.max(ei)), "err_int_finite": bool(np.isfinite(ei).all())}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))
    for v in side.values():
        v["E"].close()


if __name__ == "__main__":
    main()
