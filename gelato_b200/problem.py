"""Problem set-up: settings JSON + CSV tables -> (pdict, unitdict, condition, xdict0).

Host-side, runs once per problem.  Produces exactly the dictionaries the
reference's callbacks take (/root/reference/Trajectory_Optimization.py:49-177:
wind table :55-59, events -> per-section params :78-121, PSparams :132, launch
state :140-149, units :153-165, dx :167, condition :169-177) and the initial
guess interpolated from a trajectory table
(/root/reference/initialize.py:322-413), so that a user of the reference can feed
the same files.  No pandas / pyoptsparse dependency.

Also holds the synthetic mesh generators the benchmarks use (SURVEY.md 8(d):
C2 refined example, C5 node sweep).
"""
import copy
import csv
import json
import math
import os

import numpy as np

from . import hostmath
from .psparams import PSparams, check_intervals

G0 = 9.80665


def _read_csv(path):
    with open(path, newline="") as f:
        rows = list(csv.reader(f))
    header = [h.strip() for h in rows[0]]
    body = [[c.strip() for c in r] for r in rows[1:] if len(r) and any(c.strip() for c in r)]
    return header, body


def read_wind_table(path):
    """[altitude, wind_n, wind_e] rows (reference :55-59)."""
    header, body = _read_csv(path)
    a = np.array([[float(c) for c in r] for r in body])
    ia, isp, idir = header.index("altitude[m]"), header.index("wind_speed[m/s]"), header.index("direction[deg]")
    wind_n = a[:, isp] * -np.cos(np.radians(a[:, idir]))
    wind_e = a[:, isp] * -np.sin(np.radians(a[:, idir]))
    return np.ascontiguousarray(np.column_stack((a[:, ia], wind_n, wind_e)))


def read_ca_table(path):
    """[mach, CA] rows (reference :61-62)."""
    _, body = _read_csv(path)
    return np.ascontiguousarray(np.array([[float(c) for c in r] for r in body]))


def read_events(path):
    """List of event records with the reference's column names and types."""
    header, body = _read_csv(path)
    events = []
    for r in body:
        d = dict(zip(header, r))
        ev = {
            "name": d["name"],
            "time": float(d["time"]),
            "time_ref": d["time_ref"] if d["time_ref"] != "" else float("nan"),
            "rocketStage": int(d["rocketStage"]),
            "engineOn": d["engineOn"].lower() == "true",
            "thrust": float(d["thrust"]),
            "nozzle_area": float(d["nozzle_area"]),
            "attitude": d["attitude"],
            "pitchrate_init": float(d["pitchrate_init"]),
            "yawrate_init": float(d["yawrate_init"]),
            "num_nodes": int(d["num_nodes"]),
        }
        # optional: the LGR intervals of a composite section, ';'-separated (DESIGN.md section 11)
        if d.get("mesh_intervals", "") != "":
            ev["mesh_intervals"] = [int(v) for v in d["mesh_intervals"].split(";")]
        if d.get("mesh_breaks", "") != "":
            ev["mesh_breaks"] = [float(v) for v in d["mesh_breaks"].split(";")]
        events.append(ev)
    return events


def read_trajectory(path):
    header, body = _read_csv(path)
    cols = {}
    for j, h in enumerate(header):
        try:
            cols[h] = np.array([float(r[j]) if r[j] != "" else np.nan for r in body])
        except ValueError:
            cols[h] = [r[j] for r in body]
    return cols


def event_intervals(e):
    """None or (counts, breaks) of an event record's optional `mesh_intervals` / `mesh_breaks` (PSparams), validated
    against its `num_nodes`; ValueError names the event."""
    if "mesh_intervals" not in e:
        if "mesh_breaks" in e:
            raise ValueError("event %s: mesh_breaks without mesh_intervals" % e["name"])
        return None
    try:
        return check_intervals(int(e["num_nodes"]), e["mesh_intervals"], e.get("mesh_breaks"))
    except (TypeError, ValueError) as exc:
        raise ValueError("event %s: %s" % (e["name"], exc)) from None


def build_problem(settings, events, wind_table, ca_table, coord=None):
    """(pdict, unitdict, condition) from already-parsed inputs.

    `coord` supplies geodetic2ecef / ecef2eci / vel_ecef2eci / quat_eci2nedg /
    quat_from_euler / quatmult for the launch state (default: hostmath)."""
    coord = coord or hostmath
    settings = copy.deepcopy(settings)
    events = copy.deepcopy(events)
    stages = settings["RocketStage"]
    launch = settings["LaunchCondition"]
    names = [e["name"] for e in events]
    num_sections = len(events) - 1

    for k, e in enumerate(events):
        e["timeduration"] = (events[k + 1]["time"] - e["time"]) if k + 1 < len(events) else 9000.0
        e["timeFinishAt"] = e["time"] + e["timeduration"]
        e["mass_jettison"] = 0.0
    for stage in stages.values():
        if stage["separation_at"] in names:
            events[names.index(stage["separation_at"])]["mass_jettison"] = stage["mass_dry"]
        if stage.get("dropMass") is not None:
            for item in stage["dropMass"].values():
                if item["separation_at"] in names:
                    events[names.index(item["separation_at"])]["mass_jettison"] = item["mass"]
    for e in events:
        stage = stages[str(e["rocketStage"])]
        e["massflow"] = 0.0
        e["reference_area"] = stage["reference_area"]
        e["hold_pitch"] = False
        e["hold_yaw"] = False
        if e["engineOn"]:
            e["massflow"] = e["thrust"] / stage["Isp_vac"] / G0

    pdict = settings
    pdict["params"] = events
    pdict["event_index"] = {e["name"]: i for i, e in enumerate(events)}
    nodes = [e["num_nodes"] for e in events[:-1]]
    N = int(sum(nodes))
    pdict["ps_params"] = PSparams(nodes, [event_intervals(e) for e in events[:-1]])
    pdict["wind_table"] = np.ascontiguousarray(wind_table, dtype=np.float64)
    pdict["ca_table"] = np.ascontiguousarray(ca_table, dtype=np.float64)
    pdict["N"] = N
    pdict["M"] = N + num_sections
    pdict["num_sections"] = num_sections
    pdict["dx"] = 1.0e-8

    t_init = 0.0
    site_ecef = np.asarray(coord.geodetic2ecef(launch["lat"], launch["lon"], launch["altitude"]))
    r_init = np.asarray(coord.ecef2eci(site_ecef, t_init))
    v_init = np.asarray(coord.vel_ecef2eci(np.zeros(3), site_ecef, t_init))
    quat_init = np.asarray(
        coord.quatmult(coord.quat_eci2nedg(r_init, t_init), coord.quat_from_euler(launch["flight_azimuth_init"], 90.0, 0.0))
    )
    m_init = sum(s["mass_dry"] + s["mass_propellant"] for s in stages.values())
    if settings["OptimizationMode"] != "Payload":
        m_init += settings["mass_payload"]

    unitdict = {"mass": m_init, "position": 6378137, "velocity": 1000.0, "u": 1.0, "t": events[-1]["time"]}

    condition = {**settings["TerminalCondition"], **settings["FlightConstraint"]}
    condition["init"] = {
        "mass": m_init,
        "position": r_init,
        "velocity": v_init,
        "quaternion": quat_init,
        "u": np.zeros(2),
    }
    condition["flight_azimuth_init"] = launch["flight_azimuth_init"]
    condition["OptimizationMode"] = settings["OptimizationMode"]
    return pdict, unitdict, condition


def load_problem(settings_path, coord=None):
    """Read a reference-format settings JSON (paths relative to its folder)."""
    base = os.path.dirname(os.path.abspath(settings_path))
    with open(settings_path) as f:
        settings = json.load(f)
    wind = read_wind_table(os.path.join(base, settings["Wind file"]))
    ca = read_ca_table(os.path.join(base, settings["CA file"]))
    events = read_events(os.path.join(base, settings["Event setting file"]))
    pdict, unitdict, condition = build_problem(settings, events, wind, ca, coord)
    xdict = None
    traj = settings.get("Initial trajectory file")
    if traj is not None:
        xdict = initial_guess_from_table(read_trajectory(os.path.join(base, traj)), pdict, unitdict)
    return pdict, unitdict, condition, xdict


TRAJ_COLUMNS = (
    "time mass pos_ECI_X pos_ECI_Y pos_ECI_Z vel_ECI_X vel_ECI_Y vel_ECI_Z quat_ECI2BODY_0 quat_ECI2BODY_1 "
    "quat_ECI2BODY_2 quat_ECI2BODY_3 rate_BODY_Y rate_BODY_Z"
).split()


def read_inputs(settings_path):
    """All inputs of a reference-format problem as one plain dictionary
    {"settings", "events", "wind_table", "ca_table", "trajectory"}."""
    base = os.path.dirname(os.path.abspath(settings_path))
    with open(settings_path) as f:
        settings = json.load(f)
    inp = {
        "settings": settings,
        "events": read_events(os.path.join(base, settings["Event setting file"])),
        "wind_table": read_wind_table(os.path.join(base, settings["Wind file"])),
        "ca_table": read_ca_table(os.path.join(base, settings["CA file"])),
        "trajectory": None,
    }
    if settings.get("Initial trajectory file") is not None:
        traj = read_trajectory(os.path.join(base, settings["Initial trajectory file"]))
        inp["trajectory"] = {k: np.asarray(traj[k], dtype=np.float64) for k in TRAJ_COLUMNS}
    return inp


def dump_inputs_json(inp, path):
    """Freeze `read_inputs` output into one JSON file (floats round-trip exactly)."""
    def ev(e):
        e = dict(e)
        if isinstance(e["time_ref"], float):  # NaN = free event time
            e["time_ref"] = None
        return e

    doc = {
        "settings": inp["settings"],
        "events": [ev(e) for e in inp["events"]],
        "wind_table": np.asarray(inp["wind_table"]).tolist(),
        "ca_table": np.asarray(inp["ca_table"]).tolist(),
        "trajectory": None if inp["trajectory"] is None else {k: np.asarray(v).tolist() for k, v in inp["trajectory"].items()},
    }
    with open(path, "w") as f:
        json.dump(doc, f, indent=0, sort_keys=False)


def load_inputs_json(path):
    with open(path) as f:
        doc = json.load(f)
    for e in doc["events"]:
        if e["time_ref"] is None:
            e["time_ref"] = float("nan")
    doc["wind_table"] = np.array(doc["wind_table"], dtype=np.float64)
    doc["ca_table"] = np.array(doc["ca_table"], dtype=np.float64)
    if doc["trajectory"] is not None:
        doc["trajectory"] = {k: np.array(v, dtype=np.float64) for k, v in doc["trajectory"].items()}
    return doc


def problem_from_inputs(inp, coord=None, factor=1, max_nodes=20):
    """(pdict, unitdict, condition, xdict0) from a `read_inputs` dictionary;
    factor > 1 refines the mesh with `refine_events` (C2)."""
    settings = copy.deepcopy(inp["settings"])
    events = copy.deepcopy(inp["events"])
    if factor != 1:
        events, fc = refine_events(events, settings["FlightConstraint"], factor, max_nodes)
        settings["FlightConstraint"] = fc
    pdict, unitdict, condition = build_problem(settings, events, inp["wind_table"], inp["ca_table"], coord)
    xdict = None
    if inp.get("trajectory") is not None:
        xdict = initial_guess_from_table(inp["trajectory"], pdict, unitdict)
    return pdict, unitdict, condition, xdict


def _interp_extrap(tq, t, y):
    """Piecewise-linear interpolation with linear extrapolation (the behaviour of
    scipy interp1d(fill_value="extrapolate") the reference uses)."""
    t = np.asarray(t, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    idx = np.clip(np.searchsorted(t, tq, side="right") - 1, 0, len(t) - 2)
    slope = (y[idx + 1] - y[idx]) / (t[idx + 1] - t[idx])[(...,) + (None,) * (y.ndim - 1)]
    return y[idx] + slope * (tq - t[idx])[(...,) + (None,) * (y.ndim - 1)]


def section_time_grids(pdict):
    """(control-node times, state-node times) in seconds from the event table."""
    tc, tx = [], []
    for i in range(pdict["num_sections"]):
        to = pdict["params"][i]["time"]
        tf = pdict["params"][i]["timeFinishAt"]
        tau = pdict["ps_params"].tau(i)
        tc.append(tau * (tf - to) / 2.0 + (tf + to) / 2.0)
        tx.append(np.hstack((-1.0, tau)) * (tf - to) / 2.0 + (tf + to) / 2.0)
    return np.concatenate(tc), np.concatenate(tx)


def initial_guess_from_table(traj, pdict, unitdict):
    """Decision vector by interpolating a trajectory table onto the LGR mesh
    (reference: initialize.py:322-413).  Key order = pyoptsparse's run-time order."""
    tc, tx = section_time_grids(pdict)
    t_ref = traj["time"]

    def col(names):
        return np.column_stack([traj[n] for n in names])

    xdict = {}
    xdict["mass"] = (_interp_extrap(tx, t_ref, traj["mass"]) / unitdict["mass"]).ravel()
    xdict["position"] = (
        _interp_extrap(tx, t_ref, col(["pos_ECI_X", "pos_ECI_Y", "pos_ECI_Z"])) / unitdict["position"]
    ).ravel()
    xdict["velocity"] = (
        _interp_extrap(tx, t_ref, col(["vel_ECI_X", "vel_ECI_Y", "vel_ECI_Z"])) / unitdict["velocity"]
    ).ravel()
    xdict["quaternion"] = _interp_extrap(
        tx, t_ref, col(["quat_ECI2BODY_0", "quat_ECI2BODY_1", "quat_ECI2BODY_2", "quat_ECI2BODY_3"])
    ).ravel()
    xdict["u"] = (_interp_extrap(tc, t_ref, col(["rate_BODY_Y", "rate_BODY_Z"])) / unitdict["u"]).ravel()
    xdict["t"] = np.array([e["time"] for e in pdict["params"]]) / unitdict["t"]
    return {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in xdict.items()}


# ---------------------------------------------------------------------------
# synthetic meshes (SURVEY.md 8(d))
# ---------------------------------------------------------------------------


def refine_events(events, condition_src, factor, max_nodes=20):
    """Multiply every section's node count by `factor` and cut it into
    time-chained sub-sections of at most `max_nodes` nodes (C2, split variant).

    Returns (events, FlightConstraint) where per-section flight constraints
    ("all"-range ones) are replicated onto the sub-sections.  Sub-sections keep
    the parent's stage/engine/attitude; their start times are pinned to the
    parent's reference event, exactly like hand-written intermediate events."""
    out = []
    fc = copy.deepcopy(condition_src)
    for k, e in enumerate(events):
        if k == len(events) - 1:
            out.append(copy.deepcopy(e))
            break
        total = e["num_nodes"] * factor
        nsub = max(1, math.ceil(total / max_nodes))
        base, extra = divmod(total, nsub)
        t0, t1 = e["time"], events[k + 1]["time"]
        for s in range(nsub):
            ev = copy.deepcopy(e)
            ev["num_nodes"] = base + (1 if s < extra else 0)
            if s > 0:
                ev["name"] = "%s__%d" % (e["name"], s)
                ev["time"] = t0 + (t1 - t0) * s / nsub
                # chained to the parent event so the NLP keeps the split fixed
                ev["time_ref"] = e["name"]
                if ev["attitude"] in ("kick-turn", "pitch", "pitch-yaw"):
                    ev["attitude"] = "same-rate"
                for key in ("AOA_max", "dynamic_pressure_max", "Q_alpha_max"):
                    if e["name"] in fc.get(key, {}) and fc[key][e["name"]]["range"] == "all":
                        fc[key][ev["name"]] = copy.deepcopy(fc[key][e["name"]])
            out.append(ev)
    return out, fc


def load_refined_example(example_dir, factor, max_nodes=20, coord=None):
    """The shipped example refined to factor x its node count (C2)."""
    spath = os.path.join(example_dir, "example-settings.json")
    with open(spath) as f:
        settings = json.load(f)
    wind = read_wind_table(os.path.join(example_dir, settings["Wind file"]))
    ca = read_ca_table(os.path.join(example_dir, settings["CA file"]))
    events = read_events(os.path.join(example_dir, settings["Event setting file"]))
    events2, fc = refine_events(events, settings["FlightConstraint"], factor, max_nodes)
    settings["FlightConstraint"] = fc
    pdict, unitdict, condition = build_problem(settings, events2, wind, ca, coord)
    traj = read_trajectory(os.path.join(example_dir, settings["Initial trajectory file"]))
    xdict = initial_guess_from_table(traj, pdict, unitdict)
    return pdict, unitdict, condition, xdict


def xdict_to_vector(xdict):
    """Concatenate in the decision-vector order mass|position|velocity|quaternion|u|t
    (reference: Trajectory_Optimization.py:318-352)."""
    return np.concatenate([np.asarray(xdict[k], dtype=np.float64).ravel() for k in VAR_ORDER])


def vector_to_xdict(x, M, N, S):
    sizes = [M, 3 * M, 3 * M, 4 * M, 2 * N, S + 1]
    out, o = {}, 0
    for k, s in zip(VAR_ORDER, sizes):
        out[k] = x[o : o + s]
        o += s
    return out


VAR_ORDER = ("mass", "position", "velocity", "quaternion", "u", "t")


def three_stage_inputs(inp):
    """BASELINE.json configs[2]: the shipped example with a third stage (coast, burn, coast) appended after
    SEP2.  `inp` is a `read_inputs` dictionary; modified in place and returned."""
    s = inp["settings"]
    s["RocketStage"]["3"] = {"mass_dry": 150.0, "mass_propellant": 600.0, "dropMass": {}, "Isp_vac": 320.0,
                             "reference_area": 0.0, "ignition_at": "TEIG", "cutoff_at": "TECO",
                             "separation_at": "SEP3"}
    ev = inp["events"]
    base = dict(ev[-1])
    ev[-2]["rocketStage"] = 3  # SEP2 starts the third stage's coast
    ev.pop()  # SIMEND is re-appended last

    def event(name, time, ref, on, thrust, att, nodes, pr=0.0):
        e = dict(base)
        e.update(name=name, time=time, time_ref=ref, rocketStage=3, engineOn=on, thrust=thrust, attitude=att,
                 pitchrate_init=pr, yawrate_init=0.0, num_nodes=nodes)
        return e

    ev += [event("TEIG", 640.0, "SEP2", True, 5000.0, "pitch-yaw", 7, -0.02),
           event("TECO", 700.0, float("nan"), False, 0.0, "hold", 3),
           event("SEP3", 720.0, "TECO", False, 0.0, "hold", 2),
           event("SIMEND", 725.0, "SEP3", False, 0.0, "hold", 2)]
    return inp
