#!/usr/bin/env python
"""Device time of the path check at the benchmark workload (DESIGN.md section 11): 128 dispersed scenarios of the
example x15 (N = 990), loaded by bench.load_workload, on the default mesh grid.  gelato_eval_path_check_dev (two
launches) and gelato_eval_mesh_error_dev (the estimate on the same grid, for scale) are timed alternately in the same
process, each call bracketed by CUDA events on the launch stream.  L2: a 256 MiB write before every timed call evicts
the working set, so every call reads its inputs from HBM.  Writes one JSON document with the card's name, power limit
and max SM clock.

    python tests/scripts/path_check_timing.py [--reps 200] [--out profiles/r06b_path_check_timing.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--scenarios", type=int, default=128)
    ap.add_argument("--factor", type=int, default=15)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06b_path_check_timing.json"))
    a = ap.parse_args()
    import torch

    import bench
    from gelato_b200 import engine, mesh

    if not torch.cuda.is_available():
        raise SystemExit("path_check_timing.py: no CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.splitlines()[0].split(",")
    B = a.scenarios
    plans, X, _ = bench.load_workload("example", a.factor, B, 0, B)
    P = plans[0]
    E = engine.Engine(P, device=0, scenario_plans=plans)
    tabs = mesh.grid_tables(P.ps)
    E.set_mesh_grid(tabs)
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    xd = torch.from_numpy(X).cuda()
    rd = torch.empty((B, P.n_aero), dtype=torch.float64, device="cuda")
    ad = torch.empty((B, P.n_aero), dtype=torch.int32, device="cuda")
    ed = torch.empty((B, P.S, 11), dtype=torch.float64, device="cuda")
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")
    calls = {"path_check_dev": lambda: E.path_check_dev(xd.data_ptr(), rd.data_ptr(), ad.data_ptr(), B, st.cuda_stream),
             "mesh_error_dev": lambda: E.mesh_error_dev(xd.data_ptr(), ed.data_ptr(), B, st.cuda_stream)}
    for fn in calls.values():  # warm-up: module load, scratch allocation
        for _ in range(5):
            fn()
    st.synchronize()
    times = {k: [] for k in calls}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(2 * a.reps)]
    k = 0
    for _ in range(a.reps):
        for name, fn in calls.items():
            flush.fill_(float(k))
            ev[k][0].record(st)
            fn()
            ev[k][1].record(st)
            times[name].append(ev[k])
            k += 1
    st.synchronize()
    res = {}
    for name, evs in times.items():
        ms = np.array([s.elapsed_time(e) for s, e in evs])
        res[name] = {"median_ms": float(np.median(ms)), "p10_ms": float(np.percentile(ms, 10)),
                     "p90_ms": float(np.percentile(ms, 90)), "min_ms": float(ms.min())}
    r = rd.cpu().numpy()
    full = P.aero_i32[:, 2] > 1
    n_pts = int(sum(tabs["m"][i] for i in P.aero_i32[full, 1]))
    doc = {"gpu": q[0].strip(), "power_limit": q[1].strip(), "clocks_max_sm": q[2].strip(),
           "workload": "example x%d, %d dispersed scenarios (bench.load_workload), N=%d, S=%d, aero jobs=%d "
                       "(over a whole section: %d), their test points=%d, aero evaluations per call=%d"
                       % (a.factor, B, P.N, P.S, P.n_aero, int(full.sum()), n_pts, B * n_pts),
           "l2": "256 MiB write before every timed call (inputs and scratch read from HBM)",
           "timing": "CUDA events around each call on the launch stream, %d calls each, the two entries alternating"
                     % a.reps,
           "launches_per_call": {"path_check_dev": 2, "mesh_error_dev": 2},
           "results": res, "ratio_median": res["path_check_dev"]["median_ms"] / res["mesh_error_dev"]["median_ms"],
           "res_min_over_batch": float(np.min(r[:, full])), "res_nan": bool(np.isnan(r).any())}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))
    E.close()


if __name__ == "__main__":
    main()
