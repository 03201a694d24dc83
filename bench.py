#!/usr/bin/env python
"""Benchmark of the NLP-callback hot path (BASELINE.json metric: FD-Jacobian +
residual leaf evaluations per second; callback pairs per second; batched NLP solves
per hour).

Workloads (`--workload`, BASELINE.json `configs`):
  example_x15      configs[1] (default): the shipped example refined to ~1 000 LGR nodes
                   (x15 -> N = 990 in 53 sections of <= 20 nodes); one STEP = one `objfunc`
                   + one `sens` over a batch of 128 dispersed launch scenarios per GPU (mass /
                   thrust / wind perturbations, each scenario its own decision vector; 8 GPUs =
                   the 1 024 scenarios of configs[3]).
  three_stage_250  configs[2]: three stages, 250 sections, N = 4 836; 32 scenarios per GPU.
  sweep_1e2 .. sweep_1e5
                   configs[4]: ONE NLP (no batching) of 132 / 990 / 9 900 / 99 000 nodes.
An "eval" is one physics-leaf evaluation at one (node x perturbation column): see
CompiledPlan.eval_counts / DESIGN.md.

  value   device-resident: x already in HBM, outputs stay in HBM, CUDA events.  A step is ONE pair
          evaluation (gelato_eval_pair_packed_dev) = ONE launch of the Jacobian kernel, whose blocks
          also write objfunc's rows (dynamics defects from the centre columns, aero / event rows from
          one more column at the pristine state, linear rows as blocks of their own).
  e2e     the same step through the host-buffer C-ABI call (gelato_eval_pair_packed): x from
          page-locked host memory -> device, the kernels, g and the packed Jacobian values back
          into host buffers as contiguous copies, wall clock.
  solves  after the timed steps (not inside them): `--solve-scenarios` dispersed scenarios of the shipped
          example per GPU (default 4; 0 = skip) solved from the reference's initial guess by the host-side
          stand-in solver gelato_b200/redsqp.py (NOT IPOPT) on the CUDA callbacks, one worker process each;
          `solves_per_hour` = converged solves of all ranks / wall time (max over ranks).  The reference arm
          solves the same scenarios on the CPU oracle's callbacks.
Multi-GPU: scenarios are independent NLPs; each rank owns `--scenarios` of them
(weak scaling), no data-path collective (DESIGN.md "multi-GPU").

`--impl reference` times the CPU path instead: the reference's own C++ physics
(oracle/_ref: /root/reference/src compiled against oracle/ref_shim in the build
container; falls back to the bit-identical oracle restatement if that file is
absent) under oracle/nlp.py, the numpy port of the reference's lib/con_*.py
(the reference's Python files themselves do not travel to the GPU box), the
scenarios of a step spread over all host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fd_jacobian_plus_residual_evals_per_s"
UNIT = "evals/s"
INPUTS = os.path.join(ROOT, "tests", "golden", "example_inputs.json")
USER_EVENT = "IIP_END"

# algorithmic FP64 work per leaf evaluation (DESIGN.md "roofline"): elementary ops (+ - * / sqrt)
# counted 1 each, sin/cos/exp = 40, atan2/acos/asin = 60, pow = 120
FLOPS = {"air": 1000.0, "noair": 70.0, "quat": 20.0, "aero": 800.0, "evt": 400.0}

# name -> (variant, mesh factor, default scenarios per GPU)
WORKLOADS = {
    "example_x15": ("example", 15, 128),
    "three_stage_250": ("three_stage", 62, 32),
    "sweep_1e2": ("example", 2, 1),
    "sweep_1e3": ("example", 15, 1),
    "sweep_1e4": ("example", 150, 1),
    "sweep_1e5": ("example", 1500, 1),
}
REFERENCE_SCEN_CAP = 128  # scenarios per step of the CPU arm (a bounded sample of a multi-GPU step)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gelato", choices=["gelato", "reference"])
    ap.add_argument("--workload", default="example_x15", choices=sorted(WORKLOADS))
    ap.add_argument("--scenarios", type=int, default=0,
                    help="dispersed scenarios per GPU in one step (0 = the workload's default; 128 x 8 GPUs = the 1 024 "
                         "scenarios of BASELINE.json configs[3])")
    ap.add_argument("--factor", type=int, default=0, help="override the workload's mesh refinement factor")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="budget of each cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sustained-seconds", type=float, default=2.0, help="length of the back-to-back device leg")
    ap.add_argument("--preheat-seconds", type=float, default=0.5,
                    help="untimed run of the timed launches right before the timed steps (the clocks are sampled over it)")
    ap.add_argument("--e2e-slices", type=int, default=0, help="pipeline slices of the end-to-end leg (0 = library default)")
    ap.add_argument("--solve-mode", default="processes", choices=["processes", "threads"],
                    help="--solve-scenarios: one worker process per scenario (default; the solver's host side is the cost), or "
                         "host threads behind the coalescing server")
    ap.add_argument("--solve-procs", type=int, default=0, help="worker processes per rank (0: host cores / ranks)")
    ap.add_argument("--solve-scenarios", type=int, default=4,
                    help="also solve this many dispersed scenarios of the shipped example per GPU to convergence "
                         "(batched NLP solves per hour, BASELINE.json metric iii; 0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned to its caller for rank 0's scenarios "
                         "(residuals.npy: scenarios x residual rows; jacobian_packed.npy: scenarios x packed Jacobian "
                         "values) as float64 arrays under DIR, at most 64 MB in all (beyond that, the columns of a "
                         "fixed seeded sample), so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "gelato":
        ap.error("--dump-outputs: only the GPU arm (--impl gelato) returns its outputs to this process")
    variant, factor, scen = WORKLOADS[a.workload]
    a.variant = variant
    a.factor = a.factor or factor
    a.scenarios = a.scenarios or scen
    return a


def workload_inputs(variant):
    from gelato_b200 import problem

    inp = problem.load_inputs_json(INPUTS)
    if variant == "three_stage":
        problem.three_stage_inputs(inp)
    return inp


def load_workload(variant, factor, n_scen_total, first, count, coord=None):
    """Plans and decision vectors of scenarios [first, first+count)."""
    from gelato_b200 import plan as gplan
    from gelato_b200 import problem, scenarios

    scen = scenarios.disperse(workload_inputs(variant), n_scen_total, seed=20260117)
    plans, xs, probs = [], [], []
    for k in range(first, first + count):
        p, u, c, x0 = problem.problem_from_inputs(scen[k], coord=coord, factor=factor, max_nodes=20)
        rng = np.random.default_rng(1000 + k)
        x = {key: v + (0.0 if key == "t" else 1e-3) * rng.uniform(-1.0, 1.0, v.shape) for key, v in x0.items()}
        plans.append(gplan.CompiledPlan(p, u, c, user_eq=gplan.PerigeeAtEvent(USER_EVENT), coord=coord))
        xs.append(problem.xdict_to_vector(x))
        probs.append((p, u, c, x))
    return plans, np.stack(xs), probs


def config_of(args, P, world):
    """The `config` object of the JSON line -- identical for both arms."""
    ec = P.eval_counts()
    return {"workload": "%s (%s x%d, N=%d, sections of <= 20 nodes)" % (args.workload, args.variant, args.factor, P.N),
            "scenarios_per_gpu": args.scenarios, "nodes": P.N, "sections": P.S, "n_vars": P.n_vars, "n_rows": P.n_rows,
            "n_vals": int(P.n_vals), "evals_per_scenario_step": ec["objfunc"] + ec["sens"],
            "parallelism": "scenarios x%d" % world,
            "step": "objfunc + sens of every scenario of the batch at its own decision vector",
            "l2": "flushed between timed steps (256 MiB write); per-step CUDA events on the launch stream"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks and throttle reasons DURING the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))
        except Exception:
            pass

    def summary(self, t0=None, t1=None):
        sm, smax, reasons, power = [], 0.0, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, r in list(self.rows):
            if (t0 is not None and t < t0) or (t1 is not None and t > t1):
                continue
            try:
                sm.append(float(r[0]))
                smax = max(smax, float(r[1]))
                power.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except (ValueError, IndexError):
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None,
                "power_w": float(np.median(power)) if power else None, "reasons": sorted(reasons), "samples": len(sm)}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        return self.summary()


def ncu_traffic(kernel, grid_blocks):
    """DRAM bytes (read + write) per launch of `kernel` from the committed `ncu --set full` capture
    (profiles/traffic.json, written by tools/ncu_summary.py), if it was taken on this launch geometry."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        e = json.load(open(path))[kernel]
        if int(e["grid"].strip("()").split(",")[0]) == int(grid_blocks):
            return e["dram_bytes_per_launch"], "profiles/" + e["source"]
    except (OSError, KeyError, ValueError):
        pass
    return None, None


DUMP_BYTES = 64 * 1000 * 1000  # files, .npy headers included
DUMP_SEED = 20260119


def dump_outputs(out_dir, arrays):
    """Write each (scenarios x n) device tensor of `arrays` as out_dir/<name>.npy in float64.  If together they pass
    DUMP_BYTES, the larger ones keep only the columns of a sample drawn with DUMP_SEED (sorted, the same in every
    run) so that the total fits; the smaller ones are written whole."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    left, todo = DUMP_BYTES, sorted(arrays.items(), key=lambda kv: kv[1].numel())
    for i, (name, a) in enumerate(todo):
        keep = min(a.shape[1], (left // (len(todo) - i) - 4096) // (8 * a.shape[0]))
        if keep < a.shape[1]:
            cols = np.sort(np.random.default_rng(DUMP_SEED).choice(a.shape[1], keep, replace=False))
            a = a.index_select(1, torch.from_numpy(cols).to(a.device))
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, a.to(torch.float64).cpu().numpy())
        left -= os.path.getsize(path)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------
# CPU legs (oracle port of the reference's callbacks)
# ---------------------------------------------------------------------------
_CPU_CACHE = {}


def _cpu_problem(variant, factor, n_total, k, flav):
    """The oracle's callbacks and the decision vector of scenario k (built once per worker process)."""
    key = (variant, factor, n_total, k, flav)
    if key not in _CPU_CACHE:
        from oracle import leaves, nlp, user_builtin

        plans, X, probs = load_workload(variant, factor, n_total, k, 1)
        p, u, c, x = probs[0]
        L = leaves.get(flav)
        _CPU_CACHE[key] = (nlp.OracleNLP(p, u, c, flav, "numpy", user_eq=user_builtin.perigee_ratio_at(L, USER_EVENT)), x)
    return _CPU_CACHE[key]


def _cpu_worker(args):
    """objfunc + sens of the scenarios `ks`, `reps` times; returns the seconds spent in the callbacks."""
    variant, factor, n_total, ks, reps, flav = args
    if isinstance(ks, int):
        ks = [ks]
    todo = [_cpu_problem(variant, factor, n_total, k, flav) for k in ks]
    t0 = time.perf_counter()
    for _ in range(reps):
        for O, x in todo:
            xa = {key: v.copy() for key, v in x.items()}
            f, _ = O.objfunc(xa)
            O.sens(xa)
    return time.perf_counter() - t0


def _ref_solve_one(args):
    """One dispersed scenario of the shipped example solved by gelato_b200/redsqp.py on the CPU ORACLE's callbacks (the
    reference arm of the solves-per-hour figure: same solver, same problems as the GPU arm's solve leg)."""
    n_total, k, flav, iters = args
    from gelato_b200 import nlpshim, problem, redsqp, scenarios
    from oracle import leaves, nlp, user_builtin

    scen = scenarios.disperse(workload_inputs("example"), n_total, seed=20260117)
    p, u, c, x0 = problem.problem_from_inputs(scen[k])
    O = nlp.OracleNLP(p, u, c, flav, "numpy", user_eq=user_builtin.perigee_ratio_at(leaves.get(flav), USER_EVENT))
    sens = lambda x, f=None: O.sens(x)  # noqa: E731
    s = redsqp.ReducedSQP({"max_iter": iters})(nlpshim.register(lambda x: O.objfunc(x), sens, x0, c), sens=sens)
    return {"status": int(s.status), "nit": int(s.nit), "payload_kg": float(s.xStar["mass"][0] * u["mass"]),
            "optTime": float(s.optTime), "userObjTime": float(s.userObjTime), "userSensTime": float(s.userSensTime),
            "constr_violation": float(s.constr_violation)}


def reference_solves(args, world, flav):
    """Solves per hour of the CPU arm: the scenarios the GPU arm's solve leg solves, on the oracle's callbacks, one
    worker process per scenario over the host cores."""
    import multiprocessing as mp

    total = args.solve_scenarios * world
    nw = max(1, min(total, os.cpu_count() or 1))
    t0 = time.perf_counter()
    with mp.get_context("spawn").Pool(nw) as pool:
        res = pool.map(_ref_solve_one, [(total, k, flav, 1800) for k in range(total)], chunksize=1)
    wall = time.perf_counter() - t0
    ok = sum(1 for r in res if r["status"] in (0, 3))
    return {"solver": "gelato_b200/redsqp.py on the CPU oracle's callbacks (%s) -- NOT IPOPT" % CPU_DESC[flav],
            "scenarios_total": total, "converged_total": ok, "worker_processes": nw, "wall_s": wall,
            "runs_per_hour": total / wall * 3600.0, "solves_per_hour": ok / wall * 3600.0,
            "statuses": [r["status"] for r in res], "major_iterations": [r["nit"] for r in res],
            "payload_kg": [r["payload_kg"] for r in res], "optTime_mean_s": float(np.mean([r["optTime"] for r in res])),
            "userObjTime_mean_s": float(np.mean([r["userObjTime"] for r in res])),
            "userSensTime_mean_s": float(np.mean([r["userSensTime"] for r in res]))}


def cpu_flavour():
    """Physics leaves of the CPU arm: the reference's own C++ (oracle/_ref, built where the
    reference tree is mounted and shipped with the snapshot) when present, else the
    bit-identical hand-written restatement on glibc."""
    from oracle import leaves

    return "ref" if leaves.ref_available() else "libm"


CPU_DESC = {"ref": "the reference's own C++ leaves (oracle/_ref) under oracle/nlp.py, the numpy port of lib/con_*.py",
            "libm": "oracle/nlp.py port on the oracle's own libm leaves (bit-identical to the reference's C++, lighter call layer)"}


def cpu_baseline(args, evals_per_scen, nodes):
    """One host core, one scenario of the workload, objfunc+sens repeated for ~budget seconds -- on the reference's own
    C++ leaves (the headline figure) and on the oracle's restatement of them (4-5x faster per leaf call)."""
    out = None
    for flav in ([cpu_flavour()] + (["libm"] if cpu_flavour() == "ref" else [])):
        t1 = _cpu_worker((args.variant, args.factor, 1, 0, 1, flav))  # also warms imports / builds
        reps = int(max(2, min(50, args.cpu_seconds / max(t1, 1e-3))))
        dt = _cpu_worker((args.variant, args.factor, 1, 0, reps, flav))
        leg = {"value": evals_per_scen * reps / dt, "unit": UNIT, "cores": 1, "kind": "port", "leaves": flav,
               "pairs_per_s": reps / dt,
               "sample": "%d x (objfunc+sens) of 1 scenario of the workload (N=%d nodes), %s, %.3f s per pair"
                         % (reps, nodes, CPU_DESC[flav], dt / reps)}
        if out is None:
            out = leg
        else:
            out["libm_leaves"] = leg
    return out


def run_reference(args):
    """The reference's CPU path on all host cores.  Honours --steps / --warmup / --scenarios: a step is objfunc + sens
    of the step's scenarios (at most REFERENCE_SCEN_CAP of them: a bounded sample of a multi-GPU step), spread over a
    pool of one worker per host core."""
    import multiprocessing as mp

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1
    plans, _, _ = load_workload(args.variant, args.factor, 1, 0, 1)
    P = plans[0]
    ec = P.eval_counts()
    evals_per_scen = ec["objfunc"] + ec["sens"]
    n_step = min(args.scenarios * world, REFERENCE_SCEN_CAP)
    flav = cpu_flavour()
    nw = min(cores, n_step)
    # one single-process executor per worker, so that scenario k always lands in the process that has already set its
    # problem up (the reference sets a problem up once per solve, not once per callback)
    from concurrent.futures import ProcessPoolExecutor

    ctx = mp.get_context("spawn")
    workers = [ProcessPoolExecutor(1, mp_context=ctx) for _ in range(nw)]
    tasks = [(args.variant, args.factor, n_step, list(range(w, n_step, nw)), 1, flav) for w in range(nw)]

    def step():
        for f in [workers[w].submit(_cpu_worker, tasks[w]) for w in range(nw)]:
            f.result()

    step()  # problem set-up and imports in every worker (not a timed or counted step)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    for w in workers:
        w.shutdown()
    value = evals_per_scen * n_step * args.steps / dt
    sample = ("each step = objfunc+sens of %d dispersed scenarios of the workload%s, spread over %d worker processes (one per "
              "host core; every problem set up once, before the warm-up), %s"
              % (n_step, "" if n_step == args.scenarios * world else " (of the %d of a step of the GPU arm)" % (args.scenarios * world),
                 nw, CPU_DESC[flav]))
    solves = None
    if args.solve_scenarios > 0:
        try:
            solves = reference_solves(args, world, flav)
        except Exception as exc:
            solves = {"error": "%s: %s" % (type(exc).__name__, exc), "solves_per_hour": None}
    print(json.dumps({
        "solves": solves, "solves_per_hour": solves.get("solves_per_hour") if solves else None,
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(args, P, world),
        "pairs_per_s": n_step * args.steps / dt,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": nw, "kind": "port", "leaves": flav,
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def run_gelato(args):
    import torch
    import torch.distributed as dist

    from gelato_b200 import engine
    from gelato_b200 import scenarios as gscen

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the GPU arm has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    B = args.scenarios
    own = gscen.partition(B * world, world, rank)
    plans, X, probs = load_workload(args.variant, args.factor, B * world, own.start, len(own))
    P = plans[0]
    E = engine.Engine(P, device=local, scenario_plans=plans if B > 1 else None)
    E.set_update_slices(args.e2e_slices)
    ec = P.eval_counts()
    evals_step_rank = (ec["objfunc"] + ec["sens"]) * B
    n_pack = E.n_pack
    # a dedicated non-default stream: the C ABI reads stream 0 as "the plan's own stream", and the
    # CUDA events below must sit on the stream the kernels are launched on
    tstream = torch.cuda.Stream()
    torch.cuda.set_stream(tstream)
    st = tstream.cuda_stream
    assert st != 0

    xd = torch.from_numpy(X).cuda()
    gd = torch.full((B, P.n_rows), float("nan"), dtype=torch.float64, device="cuda")
    pd = torch.full((B, n_pack), float("nan"), dtype=torch.float64, device="cuda")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    W = max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_events(launch, n_ev=2):
        """W warm-up steps, then args.steps steps bracketed by CUDA events on the launch stream, L2 flushed between
        steps (outside the brackets); returns the summed milliseconds."""
        for _ in range(W):
            launch()
            flush.zero_()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(args.steps)]
        barrier()
        for k in range(args.steps):
            evs[k][0].record()
            launch()
            evs[k][1].record()
            flush.zero_()
        barrier()
        return sum(e[0].elapsed_time(e[1]) for e in evs)

    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)

    # ---- the headline: objfunc + sens of the batch as ONE pair evaluation, packed Jacobian output ----
    # K timed steps last a few milliseconds, less than one nvidia-smi sample: the same launches run for 0.5 s right
    # before them (untimed, on top of the W warm-up steps) and the clocks are read over that run plus the timed steps
    t_dev0 = time.perf_counter()
    while time.perf_counter() - t_dev0 < args.preheat_seconds:
        for _ in range(50):
            E.eval_pair_packed_dev(xd.data_ptr(), gd.data_ptr(), pd.data_ptr(), B, st)
        torch.cuda.synchronize()
    launches0 = E.launches
    dev_ms = timed_events(lambda: E.eval_pair_packed_dev(xd.data_ptr(), gd.data_ptr(), pd.data_ptr(), B, st))
    t_dev1 = time.perf_counter()
    launches = (E.launches - launches0) * args.steps // (args.steps + W)
    clocks = sampler.summary(t_dev0 + 0.1, t_dev1 + 0.05)
    clocks["window"] = "0.5 s of the timed launches run immediately before the timed steps, and the timed steps"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"residuals": gd, "jacobian_packed": pd})

    # ---- each kernel alone (CUDA events around the single launch, L2 flushed): the roofline's kernel is the heavy one ----
    vd = torch.empty((B, P.n_vals), dtype=torch.float64, device="cuda")
    E.fill_template(vd.data_ptr(), B, st)
    gsep = torch.full((B, P.n_rows), float("nan"), dtype=torch.float64, device="cuda")
    gp = gd.data_ptr()
    jac_ms = timed_events(lambda: E.launch_kernel_dev(1, xd.data_ptr(), pd.data_ptr(), B, True, st)) / args.steps
    kblk_ms = timed_events(lambda: E.launch_kernel_dev(6, xd.data_ptr(), pd.data_ptr(), B, True, st, gp)) / args.steps
    kvac_ms = timed_events(lambda: E.launch_kernel_dev(5, xd.data_ptr(), pd.data_ptr(), B, True, st, gp)) / args.steps \
        if ec["noair_nodes"] else 0.0
    res_ms = timed_events(lambda: E.launch_kernel_dev(0, xd.data_ptr(), gsep.data_ptr(), B, False, st)) / args.steps
    # the two callbacks as separate device calls with the reference's COO layout (what a per-callback driver gets)
    sep_ms = timed_events(lambda: (E.eval_residuals_dev(xd.data_ptr(), gsep.data_ptr(), B, st),
                                   E.eval_jacobian_dev(xd.data_ptr(), vd.data_ptr(), B, st)))
    # the pair evaluation must reproduce them bit for bit
    full, src, sgn = E.packed_map()
    assert torch.equal(gsep, gd), "pair and separate evaluations disagree (residual rows)"
    v_host = vd.cpu().numpy()
    pk_host = pd.cpu().numpy()
    assert np.array_equal(v_host[:, full], sgn * pk_host[:, src]), "packed and COO Jacobian values disagree"

    # ---- sustained: back-to-back pair evaluations for >= N seconds, no flush, one event pair around all of them ----
    n_sus = max(args.steps, int(args.sustained_seconds / max(dev_ms / args.steps * 1e-3, 1e-6)))
    barrier()
    t_s0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_sus):
        E.eval_pair_packed_dev(xd.data_ptr(), gd.data_ptr(), pd.data_ptr(), B, st)
    e1.record()
    barrier()
    t_s1 = time.perf_counter()
    sus_ms = e0.elapsed_time(e1)
    sus_clocks = sampler.summary(t_s0 + 0.2, t_s1)

    # ---- end to end through the host-buffer C ABI (what a batched driver calls) ----
    px, pg, pp = engine.PinnedArray(X.size), engine.PinnedArray(B * P.n_rows), engine.PinnedArray(B * n_pack)
    px.array[:] = X.ravel()
    pg.array[:] = np.nan
    pp.array[:] = np.nan

    def timed_wall(step):
        for _ in range(W):
            step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        barrier()
        return time.perf_counter() - t0

    e2e_s = timed_wall(lambda: E.eval_pair_packed(px.array, B, g_out=pg.array, packed_out=pp.array))
    assert np.array_equal(pg.array.reshape(B, -1), gd.cpu().numpy()), "host and device paths disagree"
    assert np.array_equal(pp.array.reshape(B, -1), pk_host), "host and device paths disagree"
    # the reference's layout through the same boundary: COO values in a page-locked buffer kept across calls
    # (update mode: x-dependent slots scattered into place) and the plain full copy
    pv = engine.PinnedArray(B * P.n_vals)
    E.jacobian_template(pv.array, B)
    e2e_upd_s = timed_wall(lambda: E.eval_pair_update(px.array, pg.array, pv.array, B))
    assert np.array_equal(pv.array.reshape(B, -1), v_host), "host and device paths disagree"
    e2e_full_s = timed_wall(lambda: (E.eval_residuals(px.array, B, out=pg.array), E.eval_jacobian(px.array, B, out=pv.array)))

    # ---- FP64 issue peaks, with the clocks they were measured at ----
    t_p0 = time.perf_counter()
    peaks = [engine.fp64_peak(local) for _ in range(6)]
    t_p1 = time.perf_counter()
    fma_tf, nofma_tf = max(p[0] for p in peaks), max(p[1] for p in peaks)
    peak_clocks = sampler.summary(t_p0, t_p1)
    sampler.stop()

    t = torch.tensor([dev_ms, e2e_s * 1e3, kblk_ms, kvac_ms, res_ms, e2e_full_s * 1e3, sep_ms, e2e_upd_s * 1e3, sus_ms / n_sus,
                      jac_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, kblk_ms, kvac_ms, res_ms, e2e_full_ms, sep_ms, e2e_upd_ms, sus_step_ms, jac_ms = [float(v) for v in t.cpu()]

    if rank == 0:
        peak_hbm, peak_src = measured_peaks()
        K = args.steps
        rate = lambda ms_total: evals_step_rank * world * K / (ms_total * 1e-3)  # noqa: E731
        # the dominant kernel of the timed step: k_jacobian as a pair evaluation launches it (air dynamics nodes, aero rows
        # with their pristine column, fallback nodes, event rows, linear rows; the vacuum nodes are k_jacobian_noair's)
        n_air_fd, n_gen = ec["air_fd_nodes"], ec["air_nodes"] - ec["air_fd_nodes"]
        flops_jac = B * (FLOPS["air"] * (14 * n_air_fd + 9 * n_gen) + FLOPS["quat"] * 7 * ec["air_free_nodes"]
                         + FLOPS["aero"] * (ec["aero_jac_evals"] + ec["aero_rows"]) + FLOPS["evt"] * (ec["evt_jac_evals"] + ec["evt_jobs"]))
        bytes_jac = B * (P.n_vars + n_pack + P.n_rows) * 8.0  # reads x once, writes every packed value and residual row once
        traffic, traffic_src = ncu_traffic("k_jacobian", E.n_jac_blocks_pair * B)
        ach_tf = flops_jac / (kblk_ms * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": rate(dev_ms), "unit": UNIT,
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": dev_ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_of(args, P, world),
            "pairs_per_s": B * world * K / (dev_ms * 1e-3),
            "clocks": clocks,
            "e2e": {"value": rate(e2e_ms), "unit": UNIT, "ms_per_step": e2e_ms / K, "pairs_per_s": B * world * K / (e2e_ms * 1e-3),
                    "h2d_bytes_per_step": int(X.size * 8), "d2h_bytes_per_step": int(B * (P.n_rows + n_pack) * 8),
                    "mode": "gelato_eval_pair_packed: page-locked host buffers; x up, one pair evaluation per slice of 16 "
                            "scenarios, g and the %d independent x-dependent Jacobian values per scenario (of %d x-dependent, "
                            "%d total COO slots) down as contiguous copies" % (n_pack, int(P.n_xdep), int(P.n_vals)),
                    "coo_update_mode": {"value": rate(e2e_upd_ms), "ms_per_step": e2e_upd_ms / K,
                                        "d2h_bytes_per_step": int(B * (P.n_rows + P.n_xdep) * 8),
                                        "note": "the reference's COO layout in a host buffer kept across calls; x-dependent "
                                                "slots scattered into place (gelato_eval_pair_update)"},
                    "coo_full_copy": {"value": rate(e2e_full_ms), "ms_per_step": e2e_full_ms / K,
                                      "d2h_bytes_per_step": int(B * (P.n_rows + P.n_vals) * 8)}},
            "gpu_launches": int(launches),
            "sustained": {"value": evals_step_rank * world / (sus_step_ms * 1e-3), "ms_per_step": sus_step_ms, "steps": n_sus,
                          "seconds": sus_ms * 1e-3, "clocks": sus_clocks,
                          "note": "back-to-back pair evaluations, no L2 flush, one CUDA-event pair around all of them"},
            "kernels": {"k_jacobian_ms": kblk_ms, "k_jacobian_noair_ms": kvac_ms, "pair_step_ms": dev_ms / K,
                        "sens_only_ms": jac_ms, "k_residuals_ms": res_ms,
                        "note": "CUDA events around single launches, L2 flushed between them.  The timed step (pair_step) "
                                "launches k_jacobian (block kernel) and k_jacobian_noair (vacuum nodes, one thread each) on "
                                "two streams; k_jacobian_ms / k_jacobian_noair_ms: each alone, as that step launches them "
                                "(objfunc's rows written too).  sens_only: the same two kernels without objfunc's rows (one "
                                "`sens`); k_residuals: one `objfunc` on its own",
                        "separate_calls_coo_ms_per_step": sep_ms / K, "separate_calls_coo_value": rate(sep_ms)},
            "roofline": {"kernel": "k_jacobian", "bound": "fp64",
                         "achieved": ach_tf, "peak": nofma_tf, "unit": "TFLOP/s",
                         "frac": (ach_tf / nofma_tf) if nofma_tf else None,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "algorithmic_flops_per_launch": flops_jac,
                         "peak_source": "gelato_fp64_peak on this device in this run: unfused DMUL+DADD issue rate (fused "
                                        "multiply-add is off by the bit-parity contract); best of 6",
                         "peak_measurement": {"dmul_dadd_tflops": nofma_tf, "dfma_tflops": fma_tf, "clocks": peak_clocks},
                         "frac_of_dfma_peak": (ach_tf / fma_tf) if fma_tf else None,
                         "hbm": {"bound": "hbm", "achieved": bytes_jac / (kblk_ms * 1e-3) / 1e9,
                                 "peak": peak_hbm, "unit": "GB/s", "frac": bytes_jac / (kblk_ms * 1e-3) / 1e9 / peak_hbm,
                                 "algorithmic_bytes_per_launch": bytes_jac, "peak_source": peak_src,
                                 "note": "the step's own bytes (x read once, every packed value and residual row written once); "
                                         "the path is FP64-issue bound, ~15 flop per byte"}},
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, ec["objfunc"] + ec["sens"], P.N)
        if args.solve_scenarios > 0:
            line["solves"] = None  # filled below by every rank's solve leg
    sol = None
    if args.solve_scenarios > 0:
        sol = run_solves(args, world, rank, local)
        if rank == 0:
            line["solves"] = sol
            line["solves_per_hour"] = sol.get("solves_per_hour")
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_solves(args, world, rank, local):
    """Batched solver runs per hour: `--solve-scenarios` dispersed scenarios of the shipped example per GPU, each run by
    gelato_b200/redsqp.py (NOT IPOPT: state elimination + penalty continuation on the dependent terminal row; converged =
    its status 0 or 3, see solve_batch.py) on the CUDA callbacks -- one worker process per scenario by default, since the
    solver's host side is what a batch of solves has to share.  `solves_per_hour` stays null unless every run converged."""
    import torch
    import torch.distributed as dist

    from gelato_b200 import solve_batch

    try:
        if args.solve_mode == "processes":
            res = solve_batch.solve_dispersed_processes(workload_inputs("example"), args.solve_scenarios * world, world, rank, device=local,
                                                        processes=args.solve_procs or None)
        else:  # one process per GPU, a host thread per scenario, callbacks coalesced into batched launches (server.py)
            res = solve_batch.solve_dispersed(workload_inputs("example"), args.solve_scenarios * world, world, rank, device=local)
    except Exception as exc:  # the collectives below still have to be entered by every rank
        res = {"error": "%s: %s" % (type(exc).__name__, exc), "wall_s": float("inf"), "converged": 0}
    t = torch.tensor([res["wall_s"]], dtype=torch.float64, device="cuda")
    n_ok = torch.tensor([res["converged"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(n_ok, op=dist.ReduceOp.SUM)
    wall = float(t.item())
    total = args.solve_scenarios * world
    res.update({"scenarios_total": total, "converged_total": int(n_ok.item()), "wall_s_max_over_ranks": wall,
                "runs_per_hour": total / wall * 3600.0,
                "solves_per_hour": int(n_ok.item()) / wall * 3600.0 if wall > 0 and wall != float("inf") else None,
                "solves_per_hour_note": "CONVERGED solves (status 0 or 3) of all ranks / wall time (max over ranks); runs that did not "
                                        "converge cost time and count nothing"})
    return res


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gelato(args)


if __name__ == "__main__":
    main()
