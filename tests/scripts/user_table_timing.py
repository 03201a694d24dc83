#!/usr/bin/env python
"""Device time of the result-table user constraints (DESIGN.md section 10 "a16") in the packed pair step, at the
benchmark workload: 128 dispersed scenarios of the example x15 (bench.load_workload's inputs and perturbation).  Two
plans of the same problem: the benchmark's (PerigeeAtEvent at IIP_END), and the same with a 3-row TableAtEvent at
FAIRING in the equality group and a 1-row TableAtEvent at KICKTURN in the inequality group.  gelato_eval_pair_packed_dev
of the two alternated in one process, each call bracketed by CUDA events on the launch stream after a 256 MiB write
that evicts L2.  Writes one JSON document with the card's name, power limit and max SM clock.

    python tests/scripts/user_table_timing.py [--reps 300] [--out profiles/r11b_user_table_timing.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

EQ_TABLE = ("FAIRING", [("altitude", 1e5, 1.0), ("dynamic_pressure", 1e3, 0.0), ("flightpath_vel_inertial_geocentric", 1.0, 0.0)])
INEQ_TABLE = ("KICKTURN", [("AOA_total", 5.0, 0.0)])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=300)
    ap.add_argument("--scenarios", type=int, default=128)
    ap.add_argument("--factor", type=int, default=15)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11b_user_table_timing.json"))
    a = ap.parse_args()
    import torch

    import bench
    from gelato_b200 import engine
    from gelato_b200 import plan as gplan

    if not torch.cuda.is_available():
        raise SystemExit("user_table_timing.py: no CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.splitlines()[0].split(",")
    B = a.scenarios
    plans, X, probs = bench.load_workload("example", a.factor, B, 0, B)
    tplans = [gplan.CompiledPlan(p, u, c, user_eq=[gplan.PerigeeAtEvent(bench.USER_EVENT), gplan.TableAtEvent(*EQ_TABLE)],
                                 user_ineq=gplan.TableAtEvent(*INEQ_TABLE)) for p, u, c, _ in probs]
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    xd = torch.from_numpy(X).cuda()
    side = {}
    for name, ps in (("benchmark_plan", plans), ("with_table_jobs", tplans)):
        E = engine.Engine(ps[0], device=0, scenario_plans=ps)
        side[name] = {"E": E, "P": ps[0], "g": torch.empty((B, ps[0].n_rows), dtype=torch.float64, device="cuda"),
                      "pk": torch.empty((B, E.n_pack), dtype=torch.float64, device="cuda")}
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")

    def call(s):
        return lambda: s["E"].eval_pair_packed_dev(xd.data_ptr(), s["g"].data_ptr(), s["pk"].data_ptr(), B, st.cuda_stream)

    calls = {k: call(v) for k, v in side.items()}
    for fn in calls.values():  # warm-up: module load
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
    # the rows the two plans share come out the same
    t, b = side["with_table_jobs"], side["benchmark_plan"]
    gt, gb = t["g"].cpu().numpy(), b["g"].cpu().numpy()
    r_eq = t["P"].group_rows["eqcon_user"][0]
    same_before = bool(np.array_equal(gt[:, : r_eq + 1], gb[:, : r_eq + 1], equal_nan=True))
    doc = {"gpu": q[0].strip(), "power_limit": q[1].strip(), "clocks_max_sm": q[2].strip(),
           "workload": "example x%d, %d dispersed scenarios, N=%d, S=%d" % (a.factor, B, b["P"].N, b["P"].S),
           "table_jobs": {"eqcon_user": [bench.USER_EVENT + " perigee", EQ_TABLE], "ineqcon_user": [INEQ_TABLE]},
           "l2": "256 MiB write before every timed call",
           "timing": "CUDA events around each gelato_eval_pair_packed_dev call on the launch stream, %d calls each, "
                     "the two plans alternating" % a.reps,
           "results": res,
           "added_ms_median": res["with_table_jobs"]["median_ms"] - res["benchmark_plan"]["median_ms"],
           "rows_before_the_user_group_identical": same_before}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))
    for v in side.values():
        v["E"].close()


if __name__ == "__main__":
    main()
