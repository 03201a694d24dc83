#!/usr/bin/env python
"""Device time of the mesh error estimate at the benchmark workload (DESIGN.md section 11): 128 dispersed scenarios
of the example x15 (N = 990), loaded by bench.load_workload.  gelato_eval_mesh_error_dev (two launches) and
gelato_eval_residuals_dev (the objfunc kernel, for scale) are timed alternately in the same process, each call
bracketed by CUDA events on the launch stream.  L2: a 256 MiB write before every timed call evicts the working set
(x 11 MB, the estimate's point scratch 23 MB), so every call reads its inputs from HBM.  Writes one JSON document
with the card's name and power limit.

    python tests/scripts/mesh_error_timing.py [--reps 200] [--out profiles/r04b_mesh_error_timing.json]
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04b_mesh_error_timing.json"))
    a = ap.parse_args()
    import torch

    import bench
    from gelato_b200 import engine, mesh

    if not torch.cuda.is_available():
        raise SystemExit("mesh_error_timing.py: no CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.splitlines()[0].split(",")
    B = a.scenarios
    plans, X, _ = bench.load_workload("example", a.factor, B, 0, B)
    P = plans[0]
    E = engine.Engine(P, device=0, scenario_plans=plans)
    E.set_mesh_grid(mesh.grid_tables(P.ps))
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    xd = torch.from_numpy(X).cuda()
    ed = torch.empty((B, P.S, 11), dtype=torch.float64, device="cuda")
    gd = torch.empty((B, P.n_rows), dtype=torch.float64, device="cuda")
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")
    calls = {"mesh_error_dev": lambda: E.mesh_error_dev(xd.data_ptr(), ed.data_ptr(), B, st.cuda_stream),
             "residuals_dev": lambda: E.eval_residuals_dev(xd.data_ptr(), gd.data_ptr(), B, st.cuda_stream)}
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
    err = ed.cpu().numpy()
    n_pts = int(sum(P.ps.nodes(i) + 1 for i in range(P.S)))
    doc = {"gpu": q[0].strip(), "power_limit": q[1].strip(), "clocks_max_sm": q[2].strip(),
           "workload": "example x%d, %d dispersed scenarios (bench.load_workload), N=%d, S=%d, test points=%d"
                       % (a.factor, B, P.N, P.S, n_pts),
           "l2": "256 MiB write before every timed call (inputs and scratch read from HBM)",
           "timing": "CUDA events around each call on the launch stream, %d calls each, the two entries alternating"
                     % a.reps,
           "launches_per_call": {"mesh_error_dev": 2, "residuals_dev": 1},
           "results": res, "ratio_median": res["mesh_error_dev"]["median_ms"] / res["residuals_dev"]["median_ms"],
           "err_max_over_batch": float(np.max(err)), "err_finite": bool(np.isfinite(err).all())}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))
    E.close()


if __name__ == "__main__":
    main()
