#!/usr/bin/env python
"""Device time of one pair step (objfunc + sens of the batch: gelato_eval_pair_packed_dev) in forward and in central
finite-difference mode (DESIGN.md H6), at bench.py's workload (example x15, N = 990, 128 dispersed scenarios).

Same measurement as bench.py's headline: CUDA events around each step on the launch stream, L2 flushed between steps
(256 MiB write, outside the events).  The two modes alternate in rounds inside one process, so drifting clocks or a
neighbour on the machine hit both alike; the card's name and power limit are read in the same run.

    python tests/scripts/fd_modes_timing.py [--rounds 5] [--steps 20] [--out fd_modes_timing.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], text=True)
        return dict(zip(q.split(","), [v.strip() for v in out.strip().split(",")]))
    except (OSError, subprocess.CalledProcessError) as e:
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scenarios", type=int, default=128)
    ap.add_argument("--step", type=float, default=None, help="central step (default: engine.DEFAULT_FD_STEP)")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import torch

    import bench
    from gelato_b200 import engine

    if not torch.cuda.is_available():
        raise SystemExit("fd_modes_timing.py: no CUDA device")
    variant, factor, _ = bench.WORKLOADS["example_x15"]
    B = a.scenarios
    plans, X, _ = bench.load_workload(variant, factor, B, 0, B)
    P = plans[0]
    E = engine.Engine(P, scenario_plans=plans)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    st = stream.cuda_stream
    xd = torch.from_numpy(X).cuda()
    gd = torch.empty((B, P.n_rows), dtype=torch.float64, device="cuda")
    pd = torch.empty((B, E.n_pack), dtype=torch.float64, device="cuda")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def step():
        E.eval_pair_packed_dev(xd.data_ptr(), gd.data_ptr(), pd.data_ptr(), B, st)

    def timed():
        for _ in range(a.warmup):
            step()
            flush.zero_()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
        torch.cuda.synchronize()
        l0 = E.launches
        for e0, e1 in evs:
            e0.record()
            step()
            e1.record()
            flush.zero_()
        torch.cuda.synchronize()
        return [e0.elapsed_time(e1) for e0, e1 in evs], (E.launches - l0) // a.steps

    modes = {"forward": None, "central": a.step}
    ms = {m: [] for m in modes}
    launches = {}
    for _ in range(a.rounds):
        for m, h in modes.items():
            E.set_fd(m, h)
            t, launches[m] = timed()
            ms[m] += t
    E.set_fd("central", a.step)
    res = {
        "what": "pair step (gelato_eval_pair_packed_dev), CUDA events per step, L2 flushed between steps, modes alternated",
        "card": card(), "torch_device": torch.cuda.get_device_name(0),
        "workload": "example x15 (N = %d, n_pack = %d), %d dispersed scenarios" % (P.N, E.n_pack, B),
        "central_step": E.fd[1], "rounds": a.rounds, "steps_per_round": a.steps,
        "median_ms": {m: float(np.median(v)) for m, v in ms.items()},
        "min_ms": {m: float(np.min(v)) for m, v in ms.items()},
        "launches_per_step": launches,
    }
    res["central_over_forward"] = res["median_ms"]["central"] / res["median_ms"]["forward"]
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(dict(res, samples_ms=ms), f, indent=1)


if __name__ == "__main__":
    main()
