"""Regenerates the golden fixtures in this folder.  Run ONLY in the container
that holds the reference at /root/reference (it is not available on the GPU box):

    python tests/golden/make_golden.py

What it writes
  example_inputs.json   the shipped example's inputs (settings JSON, events / wind /
                        CA tables, the columns of the initial-trajectory table the
                        initial guess reads) re-serialised by gelato_b200.problem.
  example_reference.npz decision vectors x0 (initial guess) and x1 (x0 + 1e-3 noise) and,
                        for each, every `funcs` entry and every Jacobian block returned by
                        the REFERENCE'S OWN Python layer (/root/reference/lib/con_*.py and the
                        objfunc / sens bodies of Trajectory_Optimization.py, imported where
                        they lie) running on the reference's own C++ physics
                        (/root/reference/src/*.cpp|hpp compiled where they lie against the minimal
                        Eigen / pybind11 stand-in of oracle/ref_shim -- the image has no Eigen3,
                        /root/reference/CMakeLists.txt:13 -- and loaded through oracle/leaves.py).  Also `jn/...`: per Jacobian
                        slot, how far the reference's own value moves when every input is nudged
                        by one ulp (64 random draws) -- its finite-difference noise floor.
  bench_reference.npz   the same (x1 only) for the BENCHMARK workload: the example refined x15 into sections
                        of <= 20 nodes (N = 990, 13 507 variables, 571 254 Jacobian values), so that the
                        configuration bench.py times is pinned to the reference directly.
  example_gmath.npz     the same quantities from oracle/nlp.py with the gmath leaves and
                        sequential-FMA D.X -- the flavour the CUDA kernels must match
                        bit for bit on any machine.
  psparams.npz          tau and D of the reference's PSparams for n = 2..24.
  example_output_result.npz
                        every column of the table the reference's own output_result function
                        (/root/reference/output_result.py:37-263, imported where it lies, on the reference's
                        C++ leaves) produces for x0 and x1.
  example_trajectory_kinematics.npz
                        the 67 rows of /root/reference/example/example-trajectory_init.csv: state (t, position,
                        velocity, quaternion) and the derived columns a former output_result wrote next to it
                        (latitude, longitude, altitude, apogee / perigee altitude, inclination, IIP, total angle
                        of attack) -- the only known answers the reference ships for the physics leaves.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import helpers  # noqa: E402
import refharness  # noqa: E402
from gelato_b200 import problem  # noqa: E402
from oracle import leaves  # noqa: E402


NOISE_DRAWS = 64


def savez_lzma(path, **arrays):
    """np.savez with LZMA compression, which np.load reads as it reads any .npz: bench_reference.npz stays under 1 MB
    this way (np.savez_compressed's deflate leaves it at 1.1 MB)."""
    import io
    import zipfile

    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_LZMA) as zf:
        for k, v in arrays.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(v), allow_pickle=False)
            zf.writestr(k + ".npy", buf.getvalue())


def pack(prefix, f, s, out):
    for k, v in helpers.flatten_funcs(f).items():
        out["%s/f/%s" % (prefix, k)] = v
    for k, (r, c, d, shape) in helpers.flatten_sens(s).items():
        out["%s/j/%s/data" % (prefix, k)] = d
        out["%s/j/%s/shape" % (prefix, k)] = np.array(shape, dtype=np.int64)
        if r is not None:
            out["%s/j/%s/rows" % (prefix, k)] = r
            out["%s/j/%s/cols" % (prefix, k)] = c
    out["%s/none_f" % prefix] = np.array([k for k, v in f.items() if v is None])
    out["%s/none_j" % prefix] = np.array([k for k, v in s.items() if v is None])


def reference_record(name, x, objfunc, sens, out):
    """x, every funcs entry, every Jacobian block and the per-slot noise floor of the reference's callbacks."""
    out["%s/x" % name] = problem.xdict_to_vector(x)
    xa = helpers.copy_x(x)
    f, fail = objfunc(xa)
    assert fail is False
    s, fail = sens(xa, f)
    pack(name, f, s, out)
    # FD noise floor of the reference itself: its Jacobian re-evaluated with every input moved
    # by one ulp in a random direction; per slot, the largest change over the draws
    base = helpers.flatten_sens(s)
    noise = {k: np.zeros_like(v[2], dtype=np.float64) for k, v in base.items()}
    rng = np.random.default_rng(11)
    for _ in range(NOISE_DRAWS):
        xn = {k: np.nextafter(v, np.where(rng.random(v.shape) < 0.5, -np.inf, np.inf)) for k, v in x.items()}
        fn, _ = objfunc(xn)
        sn, _ = sens(xn, fn)
        for k, v in helpers.flatten_sens(sn).items():
            noise[k] = np.maximum(noise[k], np.abs(v[2] - base[k][2]))
    for k, v in noise.items():
        out["%s/jn/%s" % (name, k)] = v


def main():
    assert refharness.available(), "/root/reference is required"
    inp = problem.read_inputs(os.path.join(refharness.REF, "example", "example-settings.json"))
    problem.dump_inputs_json(inp, helpers.INPUTS)

    # ---- the reference's own Python layer on the reference's own C++ leaves (oracle/_ref:
    #      /root/reference/src compiled against oracle/ref_shim; bit-identical to the oracle's
    #      libm flavour, tests/test_oracle_vs_refcpp.py) -----------------------------------
    L = leaves.get("ref")
    pdict, unitdict, condition = refharness.reference_setup(L)
    objfunc, sens = refharness.reference_callbacks(L, pdict, unitdict, condition)
    p, u, c, x0 = helpers.example_problem()
    x1 = helpers.perturbed(x0)
    out = {}
    for name, x in (("x0", x0), ("x1", x1)):
        reference_record(name, x, objfunc, sens, out)
    np.savez_compressed(os.path.join(HERE, "example_reference.npz"), **out)

    # ---- the same at the benchmark workload (bench.py: factor 15, sections of <= 20 nodes) ----
    pb, ub, cb, xb0 = problem.problem_from_inputs(helpers.example_inputs(), factor=15, max_nodes=20)
    objfunc_b, sens_b = refharness.reference_callbacks(L, pb, ub, cb)
    out = {}
    reference_record("x1", helpers.perturbed(xb0), objfunc_b, sens_b, out)
    savez_lzma(os.path.join(HERE, "bench_reference.npz"), **out)

    # ---- gmath / sequential-FMA flavour of the oracle ---------------------
    Lg = leaves.get("gmath")
    p, u, c, x0 = helpers.example_problem(coord=Lg.coordinate_c)
    O = helpers.oracle_nlp(p, u, c, "gmath", "seqfma")
    out = {}
    for name, x in (("x0", x0), ("x1", helpers.perturbed(x0))):
        out["%s/x" % name] = problem.xdict_to_vector(x)
        xa = helpers.copy_x(x)
        f, _ = O.objfunc(xa)
        s, _ = O.sens(xa)
        pack(name, f, s, out)
    np.savez_compressed(os.path.join(HERE, "example_gmath.npz"), **out)

    # ---- the known answers the reference ships: kinematic columns of its example trajectory table ----
    import csv

    with open(os.path.join(refharness.REF, "example", "example-trajectory_init.csv")) as fh:
        rows = list(csv.DictReader(fh))

    def col(*names):
        return np.array([[float(r[n]) if r[n] != "" else np.nan for n in names] for r in rows])

    np.savez_compressed(
        os.path.join(HERE, "example_trajectory_kinematics.npz"),
        t=col("time")[:, 0], pos=col("pos_ECI_X", "pos_ECI_Y", "pos_ECI_Z"), vel=col("vel_ECI_X", "vel_ECI_Y", "vel_ECI_Z"),
        quat=col("quat_ECI2BODY_0", "quat_ECI2BODY_1", "quat_ECI2BODY_2", "quat_ECI2BODY_3"),
        lat=col("lat")[:, 0], lon=col("lon")[:, 0], altitude=col("altitude")[:, 0],
        apogee=col("altitude_apogee")[:, 0], perigee=col("altitude_perigee")[:, 0], inclination=col("inclination")[:, 0],
        lat_iip=col("lat_IIP")[:, 0], lon_iip=col("lon_IIP")[:, 0], aoa_deg=col("AOA_total")[:, 0])

    # ---- the reference's own output_result table of the two decision vectors --------------------
    out_fn = refharness.reference_output_result(L)
    tab = {}
    for name, x in (("x0", x0), ("x1", x1)):
        tx, tu = refharness.result_times(x, pdict, unitdict)
        df = out_fn(helpers.copy_x(x), unitdict, tx, tu, pdict)
        tab["%s/columns" % name] = np.array(list(df.columns))
        for c in df.columns:
            v = np.asarray(df[c].values)
            tab["%s/%s" % (name, c)] = v if v.dtype.kind in "fiub" else np.array([str(e) for e in v])
    np.savez_compressed(os.path.join(HERE, "example_output_result.npz"), **tab)

    # ---- reference PSparams ------------------------------------------------
    ns = refharness.load(L)
    ps_out = {}
    for n in range(2, 25):
        ps = ns["PSparams"]([n])
        ps_out["tau_%d" % n] = ps.tau(0)
        ps_out["D_%d" % n] = ps.D(0)
    np.savez_compressed(os.path.join(HERE, "psparams.npz"), **ps_out)
    for f in sorted(os.listdir(HERE)):
        print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()
