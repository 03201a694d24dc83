#!/usr/bin/env python
"""Step sweep of the central-difference Jacobian (DESIGN.md H6) on the CPU oracle: no GPU needed.

The shipped example at x0 + 1e-3 U(-1, 1) (helpers.perturbed), gmath leaves, sequential-FMA D.X; the yardstick is
helpers.true_jacobian (4th-order central differences of objfunc).  For every Jacobian block whose values depend on the
step, the max and rms distance to the derivative of the forward mode (the plan's dx = 1e-8) and of the central mode at
each step.  The default step is the one with the smallest geometric mean over those blocks of (central rms / forward
rms): one scalar for every block, so it trades the blocks that want a smaller step (the position columns of the
air-dependent rows: density ~ exp(-altitude / 7 km)) against the rest.

    python tests/scripts/fd_step_sweep.py [--steps 1e-5,3e-6,1e-6,3e-7,1e-7] [--out sweep.json]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers  # noqa: E402


def oracle(p, u, c, derivative="forward", fd_step=None):
    from central_oracle import CentralOracleNLP
    from oracle import leaves, user_builtin

    Lg = leaves.get("gmath")
    return CentralOracleNLP(p, u, c, "gmath", "seqfma", user_eq=user_builtin.perigee_ratio_at(Lg, helpers.USER_EVENT),
                            derivative=derivative, fd_step=fd_step)


def sweep(steps, seed=7):
    """{"fd_blocks": [...], "forward": {block: (max, rms)}, "central": {step: {block: (max, rms)}}, "choice": step}."""
    from oracle import leaves

    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    x = helpers.perturbed(x0, seed=seed)
    row0, J, col0 = helpers.true_jacobian(oracle(p, u, c).objfunc, x)

    def errors(O):
        s, _ = O.sens(helpers.copy_x(x))
        return s, helpers.derivative_errors(s, row0, J, col0)

    def stats(e):
        return (float(e.max()), float(np.sqrt(np.mean(np.square(e))))) if e.size else (0.0, 0.0)

    s_fwd, e_fwd = errors(oracle(p, u, c))
    fs_fwd = helpers.flatten_sens(s_fwd)
    res = {"forward": {k: stats(e) for k, e in e_fwd.items()}, "central": {}, "fd_blocks": []}
    fd = set()
    for h in steps:
        s, e = errors(oracle(p, u, c, "central", h))
        for k, (_, _, d, _) in helpers.flatten_sens(s).items():
            if not np.array_equal(np.asarray(d).view(np.int64), np.asarray(fs_fwd[k][2]).view(np.int64)):
                fd.add(k)
        res["central"][repr(h)] = {k: stats(v) for k, v in e.items()}
    res["fd_blocks"] = sorted(k for k in fd if k in e_fwd and res["forward"][k][1] > 0.0)
    score = {}
    for h in steps:
        r = [res["central"][repr(h)][k][1] / res["forward"][k][1] for k in res["fd_blocks"]]
        score[repr(h)] = float(np.exp(np.mean(np.log(np.maximum(r, 1e-300)))))
    res["geomean_rms_ratio"] = score
    res["choice"] = float(min(score, key=score.get))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", default="1e-5,3e-6,1e-6,3e-7,1e-7")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    steps = [float(v) for v in a.steps.split(",")]
    res = sweep(steps)
    w = max(len(k) for k in res["fd_blocks"])
    print("max |error| / rms error against the 4th-order derivative, per block whose values depend on the step")
    print("%-*s  %-21s" % (w, "block", "forward dx=1e-8") + "".join("  %-21s" % ("central h=%g" % h) for h in steps))
    for k in res["fd_blocks"]:
        line = "%-*s  %9.2e / %9.2e" % ((w, k) + tuple(res["forward"][k]))
        for h in steps:
            line += "  %9.2e / %9.2e" % tuple(res["central"][repr(h)][k])
        print(line)
    print("geometric mean over these blocks of central rms / forward rms: " +
          ", ".join("h=%g: %.3g" % (h, res["geomean_rms_ratio"][repr(h)]) for h in steps))
    print("choice: h = %g" % res["choice"])
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
