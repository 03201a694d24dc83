#!/usr/bin/env python
"""Device time of the path rows at the benchmark workload (DESIGN.md section 11): 128 dispersed scenarios of the
example x15 (N = 990), loaded by bench.load_workload, with path rows on the default grid (n + 1 points per section).
gelato_eval_path_rows_dev residual-only, with the forward Jacobian and with the central Jacobian, and
gelato_eval_pair_packed_dev (one pair step of the NLP, for scale) are timed alternately in the same process, each call
bracketed by CUDA events on the launch stream.  L2: a 256 MiB write before every timed call evicts the working set.
The aero evaluations per call are counted from shapes.  Writes one JSON document with the card's name, power limit
and max SM clock.

    python tests/scripts/path_rows_timing.py [--reps 200] [--out profiles/r07b_path_rows_timing.json]
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07b_path_rows_timing.json"))
    a = ap.parse_args()
    import torch

    import bench
    from gelato_b200 import engine, mesh

    if not torch.cuda.is_available():
        raise SystemExit("path_rows_timing.py: no CUDA device")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.splitlines()[0].split(",")
    B = a.scenarios
    plans, X, _ = bench.load_workload("example", a.factor, B, 0, B)
    P = plans[0]
    E = engine.Engine(P, device=0, scenario_plans=plans)
    E.set_path_rows(mesh.grid_tables(P.ps))
    lay = E.path_rows_layout()
    nr, nv = lay["n_rows"], lay["n_vals"]
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    xd = torch.from_numpy(X).cuda()
    gd = torch.empty((B, nr), dtype=torch.float64, device="cuda")
    vd = torch.empty((B, nv), dtype=torch.float64, device="cuda")
    g_main = torch.empty((B, P.n_rows), dtype=torch.float64, device="cuda")
    pk = torch.empty((B, E.n_pack), dtype=torch.float64, device="cuda")
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device="cuda")
    x, g, v, s = xd.data_ptr(), gd.data_ptr(), vd.data_ptr(), st.cuda_stream

    def path(jac, mode):
        def call():
            E.eval_path_rows_dev(x, g, v if jac else None, B, s)
        return (mode, call)

    calls = {"path_rows_dev residual-only": path(False, "forward"), "path_rows_dev forward": path(True, "forward"),
             "path_rows_dev central": path(True, "central"),
             "pair_packed_dev forward": ("forward", lambda: E.eval_pair_packed_dev(x, g_main.data_ptr(), pk.data_ptr(), B, s))}
    for mode, fn in calls.values():  # warm-up: module load, scratch allocation
        E.set_fd(mode)
        for _ in range(5):
            fn()
    st.synchronize()
    times = {k: [] for k in calls}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(len(calls) * a.reps)]
    k = 0
    for _ in range(a.reps):
        for name, (mode, fn) in calls.items():
            E.set_fd(mode)  # host-side flag only; no device work
            flush.fill_(float(k))
            ev[k][0].record(st)
            fn()
            ev[k][1].record(st)
            times[name].append(ev[k])
            k += 1
    st.synchronize()
    res = {}
    for name, evs in times.items():
        ms = np.array([e0.elapsed_time(e1) for e0, e1 in evs])
        res[name] = {"median_ms": float(np.median(ms)), "p10_ms": float(np.percentile(ms, 10)),
                     "p90_ms": float(np.percentile(ms, 90)), "min_ms": float(ms.min())}
    kinds = P.aero_i32[lay["job"], 0]
    lanes = int(np.sum(np.where(kinds == 1, 8, 12)))  # quotient lanes per scenario: max-q rows have no quaternion lanes
    doc = {"gpu": q[0].strip(), "power_limit": q[1].strip(), "clocks_max_sm": q[2].strip(),
           "workload": "example x%d, %d dispersed scenarios (bench.load_workload), N=%d, S=%d, path rows=%d on the "
                       "default grid, row values=%d per scenario" % (a.factor, B, P.N, P.S, nr, nv),
           "aero_evaluations_per_call": {"residual-only": B * nr, "forward": B * (nr + lanes),
                                         "central": B * (nr + 2 * lanes)},
           "l2": "256 MiB write before every timed call (inputs read from HBM)",
           "timing": "CUDA events around each call on the launch stream, %d calls each, the entries alternating" % a.reps,
           "results": res,
           "ratio_median_to_pair": {k: res[k]["median_ms"] / res["pair_packed_dev forward"]["median_ms"] for k in res},
           "g_min_over_batch": float(gd.min().item()), "nan": bool(torch.isnan(vd).any().item() or torch.isnan(gd).any().item())}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))
    E.close()


if __name__ == "__main__":
    main()
