"""ctypes binding of libgelato_b200.so (the C ABI in include/gelato_b200.h).

This is the thin layer that stands where the reference's five pybind11 modules
stood (/root/reference/src/pybind_*.cpp): Python hands the engine a decision
vector, the engine runs ONE fused CUDA kernel and hands back the whole residual
vector or the whole Jacobian value vector.

There is no CPU path: if the shared library is missing or no CUDA device is
present, construction raises.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# GELATO_B200_LIB: an alternative build of the same library (kernel tuning experiments, tools/ab_bench.sh)
LIB_PATH = os.environ.get("GELATO_B200_LIB") or os.path.join(CSRC, "libgelato_b200.so")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-fmad=false", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]

# Finite-difference modes of the Jacobian (include/gelato_b200.h: gelato_plan_set_fd; DESIGN.md H6)
FD_MODES = {"forward": 0, "central": 1}
# default step of central differences: the step sweep of profiles/r03a_fd_step_sweep.txt (DESIGN.md H6)
DEFAULT_FD_STEP = 1e-6

_c_d = ctypes.c_double
_pd = ctypes.POINTER(ctypes.c_double)
_pi32 = ctypes.POINTER(ctypes.c_int32)
_pi64 = ctypes.POINTER(ctypes.c_int64)
_pu8 = ctypes.POINTER(ctypes.c_uint8)


class GelatoError(RuntimeError):
    pass


class PlanDesc(ctypes.Structure):
    """GelatoPlanDesc (include/gelato_b200.h)."""

    _fields_ = [
        ("n_sections", ctypes.c_int32), ("n_nodes", ctypes.c_int32), ("n_rows", ctypes.c_int32),
        ("n_vals", ctypes.c_int64), ("payload_mode", ctypes.c_int32),
        ("sec_i32", _pi32), ("sec_i64", _pi64), ("sec_f64", _pd),
        ("d_pool", _pd), ("d_pool_len", ctypes.c_int64), ("tau_pool", _pd), ("tau_pool_len", ctypes.c_int64),
        ("wind", _pd), ("n_wind", ctypes.c_int32), ("ca", _pd), ("n_ca", ctypes.c_int32),
        ("unit_mass", _c_d), ("unit_pos", _c_d), ("unit_vel", _c_d), ("unit_u", _c_d), ("unit_t", _c_d), ("dx", _c_d),
        ("n_lin", ctypes.c_int32), ("lin_i32", _pi32), ("lin_f64", _pd),
        ("n_aero", ctypes.c_int32), ("aero_i32", _pi32), ("aero_i64", _pi64), ("aero_f64", _pd), ("rc_aero", _pu8),
        ("n_evt", ctypes.c_int32), ("evt_i32", _pi32), ("evt_i64", _pi64), ("evt_f64", _pd),
        ("vals_template", _pd),
        ("xdep_idx", _pi64), ("n_xdep", ctypes.c_int64),
        ("n_tab", ctypes.c_int32), ("tab_i32", _pi32), ("tab_f64", _pd), ("n_tab_rows", ctypes.c_int32),
        ("tab_col", _pi32), ("tab_aux", _pi64), ("tab_sf", _pd),
    ]


class ScenarioDesc(ctypes.Structure):
    """GelatoScenarioDesc (include/gelato_b200.h)."""

    _fields_ = [("n_scen", ctypes.c_int32), ("sec_f64", _pd), ("wind", _pd), ("unit_mass", _pd), ("lin_const", _pd),
                ("vals_template", _pd)]


class MeshGridDesc(ctypes.Structure):
    """GelatoMeshGridDesc (include/gelato_b200.h)."""

    _fields_ = [("m", _pi32), ("off", _pi64), ("pool", _pd), ("pool_len", ctypes.c_int64), ("n_int", _pi32),
                ("int_m", _pi32), ("int_base", _pi32)]


def _ptr(arr, typ):
    if arr is None or arr.size == 0:
        return ctypes.cast(None, typ)
    return arr.ctypes.data_as(typ)


def _out(arr, n, what):
    """A caller-supplied output buffer the C side will write n doubles into: it must be a writeable,
    C-contiguous float64 array of exactly that size (anything else would be written through a wrong
    pointer or stride -- memory corruption instead of an exception)."""
    if not isinstance(arr, np.ndarray) or arr.dtype != np.float64 or not arr.flags.c_contiguous or not arr.flags.writeable:
        raise ValueError("%s must be a writeable C-contiguous float64 numpy array" % what)
    if arr.size != n:
        raise ValueError("%s has %d entries, expected %d" % (what, arr.size, n))
    return arr


def make_desc(plan):
    """CompiledPlan -> (PlanDesc, keepalive list of the arrays it points into)."""
    keep = []

    def c(a, dt):
        a = np.ascontiguousarray(a, dtype=dt)
        keep.append(a)
        return a

    d = PlanDesc()
    d.n_sections, d.n_nodes, d.n_rows, d.n_vals = plan.S, plan.N, plan.n_rows, plan.n_vals
    d.payload_mode = plan.payload_mode
    d.sec_i32 = _ptr(c(plan.sec_i32, np.int32), _pi32)
    d.sec_i64 = _ptr(c(plan.sec_i64, np.int64), _pi64)
    d.sec_f64 = _ptr(c(plan.sec_f64, np.float64), _pd)
    d.d_pool = _ptr(c(plan.d_pool, np.float64), _pd)
    d.d_pool_len = plan.d_pool.size
    d.tau_pool = _ptr(c(plan.tau_pool, np.float64), _pd)
    d.tau_pool_len = plan.tau_pool.size
    d.wind = _ptr(c(plan.wind, np.float64), _pd)
    d.n_wind = plan.wind.shape[0]
    d.ca = _ptr(c(plan.ca, np.float64), _pd)
    d.n_ca = plan.ca.shape[0]
    d.unit_mass, d.unit_pos, d.unit_vel, d.unit_u, d.unit_t, d.dx = plan.units
    d.n_lin = plan.n_lin
    d.lin_i32 = _ptr(c(plan.lin_i32, np.int32), _pi32)
    d.lin_f64 = _ptr(c(plan.lin_f64, np.float64), _pd)
    d.n_aero = plan.n_aero
    d.aero_i32 = _ptr(c(plan.aero_i32, np.int32), _pi32)
    d.aero_i64 = _ptr(c(plan.aero_i64, np.int64), _pi64)
    d.aero_f64 = _ptr(c(plan.aero_f64, np.float64), _pd)
    d.rc_aero = _ptr(c(plan.rc_aero, np.uint8), _pu8)
    d.n_evt = plan.n_evt
    d.evt_i32 = _ptr(c(plan.evt_i32, np.int32), _pi32)
    d.evt_i64 = _ptr(c(plan.evt_i64, np.int64), _pi64)
    d.evt_f64 = _ptr(c(plan.evt_f64, np.float64), _pd)
    d.vals_template = _ptr(c(plan.vals_template, np.float64), _pd)
    xdep = c(plan.xdep_index(), np.int64)
    d.xdep_idx = _ptr(xdep, _pi64)
    d.n_xdep = xdep.size
    d.n_tab, d.n_tab_rows = plan.n_tab, plan.n_tab_rows
    d.tab_i32 = _ptr(c(plan.tab_i32, np.int32), _pi32)
    d.tab_f64 = _ptr(c(plan.tab_f64, np.float64), _pd)
    d.tab_col = _ptr(c(plan.tab_col, np.int32), _pi32)
    d.tab_aux = _ptr(c(plan.tab_aux, np.int64), _pi64)
    d.tab_sf = _ptr(c(plan.tab_sf, np.float64), _pd)
    return d, keep


def make_scenario_desc(plans):
    """Per-scenario blocks from a list of CompiledPlans that share one structure
    (same mesh, same constraint rows) and differ in section parameters, wind
    table, mass unit and the constants derived from them."""
    base = plans[0]
    for p in plans[1:]:
        if (p.n_rows, p.n_vals, p.n_lin, p.n_evt, p.n_aero, p.wind.shape) != (
                base.n_rows, base.n_vals, base.n_lin, base.n_evt, base.n_aero, base.wind.shape):
            raise ValueError("scenario plans must share the problem structure")
        # what is NOT carried per scenario is evaluated with the base plan's copy: it must be the same everywhere
        shared = ("sec_i32", "sec_i64", "d_pool", "tau_pool", "ca", "lin_i32", "aero_i32", "aero_i64", "aero_f64",
                  "rc_aero", "evt_i32", "evt_i64", "evt_f64", "tab_i32", "tab_f64", "tab_col", "tab_aux", "tab_sf")
        for name in shared:
            a, b = getattr(base, name, None), getattr(p, name, None)
            if a is None and b is None:
                continue
            if a is None or b is None or not np.array_equal(np.asarray(a), np.asarray(b)):
                raise ValueError("scenario plans differ in `%s`, which is shared by every scenario of a batch "
                                 "(per scenario: section parameters, wind table, mass unit, linear-row constants)" % name)
        if not np.array_equal(np.asarray(base.units)[1:], np.asarray(p.units)[1:]):
            raise ValueError("scenario plans differ in a unit other than the mass unit")
        if not np.array_equal(np.asarray(base.lin_f64)[:, :2], np.asarray(p.lin_f64)[:, :2]) or \
                not np.array_equal(np.asarray(base.lin_f64)[:, 3:], np.asarray(p.lin_f64)[:, 3:]):
            raise ValueError("scenario plans differ in linear-row coefficients other than the constant")
    keep = []

    def stack(get):
        a = np.ascontiguousarray(np.stack([np.asarray(get(p), dtype=np.float64) for p in plans]))
        keep.append(a)
        return a

    sc = ScenarioDesc()
    sc.n_scen = len(plans)
    sc.sec_f64 = _ptr(stack(lambda p: p.sec_f64), _pd)
    sc.wind = _ptr(stack(lambda p: p.wind), _pd)
    sc.unit_mass = _ptr(stack(lambda p: p.units[0]), _pd)
    sc.lin_const = _ptr(stack(lambda p: p.lin_f64[:, 2]), _pd)
    sc.vals_template = _ptr(stack(lambda p: p.vals_template), _pd)
    return sc, keep


def make_mesh_grid_desc(tables):
    """{"m", "off", "pool"} and optionally {"n_int", "int_m", "int_base"} (gelato_b200/mesh.py: grid_tables) ->
    (MeshGridDesc, keepalive list)."""
    m = np.ascontiguousarray(tables["m"], dtype=np.int32)
    off = np.ascontiguousarray(tables["off"], dtype=np.int64)
    pool = np.ascontiguousarray(tables["pool"], dtype=np.float64)
    d = MeshGridDesc()
    d.m, d.off, d.pool, d.pool_len = _ptr(m, _pi32), _ptr(off, _pi64), _ptr(pool, _pd), pool.size
    keep = [m, off, pool]
    if "n_int" in tables:
        iv = [np.ascontiguousarray(tables[k], dtype=np.int32) for k in ("n_int", "int_m", "int_base")]
        d.n_int, d.int_m, d.int_base = (_ptr(a, _pi32) for a in iv)
        keep += iv
    return d, keep


def grid_intervals(tables):
    """The number of intervals of a mesh grid: sum(n_int), or one per section without interval tables."""
    return int(np.sum(tables["n_int"])) if "n_int" in tables else len(tables["m"])


def build_library(force=False, verbose=False, out=None, extra=()):
    """Compile csrc/gelato_b200.cu for sm_100a into csrc/libgelato_b200.so (in tree).
    `out` / `extra`: another output path and extra nvcc flags (tuning variants)."""
    src = os.path.join(CSRC, "gelato_b200.cu")
    srcs = [src, os.path.join(CSRC, "leaf_api.cu")]
    if out is not None:
        subprocess.check_call(["nvcc"] + NVCC_FLAGS + list(extra) + ["-o", out] + srcs)
        return out
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".inc"))]
    deps.append(os.path.join(INCLUDE, "gelato_b200.h"))
    if not force and os.path.exists(LIB_PATH) and all(os.path.getmtime(LIB_PATH) >= os.path.getmtime(f) for f in deps):
        return LIB_PATH
    cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH] + srcs
    subprocess.check_call(cmd)
    return LIB_PATH


_lib = None


def load_library():
    """dlopen the engine and declare the prototypes of include/gelato_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GelatoError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the callback evaluations)" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp = ctypes.c_void_p
    L.gelato_last_error.restype = ctypes.c_char_p
    L.gelato_device_count.restype = ctypes.c_int
    L.gelato_plan_create.argtypes = [ctypes.POINTER(PlanDesc), ctypes.c_int, ctypes.POINTER(vp)]
    L.gelato_plan_set_scenarios.argtypes = [vp, ctypes.POINTER(ScenarioDesc)]
    L.gelato_plan_destroy.argtypes = [vp]
    L.gelato_plan_n_vars.argtypes = [vp]
    L.gelato_plan_n_vars.restype = ctypes.c_int32
    L.gelato_plan_n_rows.argtypes = [vp]
    L.gelato_plan_n_rows.restype = ctypes.c_int32
    L.gelato_plan_n_vals.argtypes = [vp]
    L.gelato_plan_n_vals.restype = ctypes.c_int64
    L.gelato_plan_launch_count.argtypes = [vp]
    L.gelato_plan_launch_count.restype = ctypes.c_int64
    L.gelato_plan_set_fd.argtypes = [vp, ctypes.c_int32, _c_d]
    L.gelato_plan_get_fd.argtypes = [vp, _pi32, _pd]
    L.gelato_eval_residuals.argtypes = [vp, _pd, _pd, ctypes.c_int32]
    L.gelato_plan_set_mesh_grid.argtypes = [vp, ctypes.POINTER(MeshGridDesc)]
    L.gelato_eval_mesh_error.argtypes = [vp, _pd, _pd, ctypes.c_int32]
    L.gelato_eval_mesh_error_dev.argtypes = [vp, vp, vp, ctypes.c_int32, vp]
    L.gelato_eval_mesh_error_intervals.argtypes = [vp, _pd, _pd, ctypes.c_int32]
    L.gelato_eval_mesh_error_intervals_dev.argtypes = [vp, vp, vp, ctypes.c_int32, vp]
    L.gelato_eval_path_check.argtypes = [vp, _pd, _pd, _pi32, ctypes.c_int32]
    L.gelato_eval_path_check_dev.argtypes = [vp, vp, vp, vp, ctypes.c_int32, vp]
    L.gelato_plan_set_path_rows.argtypes = [vp, ctypes.POINTER(MeshGridDesc)]
    L.gelato_plan_path_rows.argtypes = [vp, _pi32, _pi64, _pi32, _pi32, _pi64]
    L.gelato_eval_path_rows.argtypes = [vp, _pd, _pd, _pd, ctypes.c_int32]
    L.gelato_eval_path_rows_dev.argtypes = [vp, vp, vp, vp, ctypes.c_int32, vp]
    L.gelato_eval_jacobian.argtypes = [vp, _pd, _pd, ctypes.c_int32]
    L.gelato_eval_residuals_ids.argtypes = [vp, _pd, _pd, ctypes.c_int32, _pi32]
    L.gelato_eval_jacobian_ids.argtypes = [vp, _pd, _pd, ctypes.c_int32, _pi32]
    L.gelato_eval_residuals_dev.argtypes = [vp, vp, vp, ctypes.c_int32, vp]
    L.gelato_eval_jacobian_dev.argtypes = [vp, vp, vp, ctypes.c_int32, vp]
    L.gelato_fill_template.argtypes = [vp, vp, ctypes.c_int32, vp]
    L.gelato_plan_n_blocks.argtypes = [vp, ctypes.c_int]
    L.gelato_plan_n_blocks.restype = ctypes.c_int32
    L.gelato_plan_n_xdep.argtypes = [vp]
    L.gelato_plan_n_xdep.restype = ctypes.c_int64
    L.gelato_jacobian_template.argtypes = [vp, _pd, ctypes.c_int32]
    L.gelato_eval_jacobian_update.argtypes = [vp, _pd, _pd, ctypes.c_int32]
    L.gelato_eval_pair_update.argtypes = [vp, _pd, _pd, _pd, ctypes.c_int32]
    L.gelato_eval_pair_dev.argtypes = [vp, vp, vp, vp, ctypes.c_int32, vp]
    L.gelato_eval_pair_packed_dev.argtypes = [vp, vp, vp, vp, ctypes.c_int32, vp]
    L.gelato_eval_pair_packed_range_dev.argtypes = [vp, vp, vp, vp, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                    ctypes.c_int32, vp]
    L.gelato_plan_n_pack.argtypes = [vp]
    L.gelato_plan_n_pack.restype = ctypes.c_int64
    L.gelato_plan_packed_map.argtypes = [vp, _pi64, _pi64, _pd]
    L.gelato_eval_pair_packed.argtypes = [vp, _pd, _pd, _pd, ctypes.c_int32]
    L.gelato_eval_jacobian_packed.argtypes = [vp, _pd, _pd, ctypes.c_int32]
    L.gelato_eval_pair_packed_ids.argtypes = [vp, _pd, _pd, _pd, ctypes.c_int32, _pi32]
    L.gelato_set_host_threads.argtypes = [vp, ctypes.c_int32]
    L.gelato_set_update_zero_copy.argtypes = [vp, ctypes.c_int32]
    L.gelato_set_update_slices.argtypes = [vp, ctypes.c_int32]
    L.gelato_probe_update.argtypes = [vp, _pd, ctypes.c_int32, ctypes.c_int, ctypes.POINTER(ctypes.c_float)]
    L.gelato_pack_xdep_dev.argtypes = [vp, vp, vp, ctypes.c_int32, vp]
    L.gelato_host_alloc.argtypes = [ctypes.c_size_t, ctypes.POINTER(vp)]
    L.gelato_host_free.argtypes = [vp]
    L.gelato_time_kernel.argtypes = [vp, ctypes.c_int, vp, vp, ctypes.c_int32, ctypes.c_int,
                                     ctypes.POINTER(ctypes.c_float)]
    L.gelato_launch_kernel_dev.argtypes = [vp, ctypes.c_int, vp, vp, vp, ctypes.c_int32, ctypes.c_int32, vp]
    L.gelato_selftest_unfused.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
    L.gelato_fp64_peak.argtypes = [ctypes.c_int, _pd, _pd]
    i32 = ctypes.c_int32
    L.gelato_leaf_dynamics_velocity.argtypes = [ctypes.c_int, i32, _pd, _pd, _pd, _pd, _pd, _pd, _pd, i32, _pd, i32, _pd, _pd]
    L.gelato_leaf_dynamics_velocity_noair.argtypes = [ctypes.c_int, i32, _pd, _pd, _pd, _pd, _pd, _pd]
    L.gelato_leaf_dynamics_quaternion.argtypes = [ctypes.c_int, i32, _pd, _pd, _c_d, _pd]
    L.gelato_leaf_aero.argtypes = [ctypes.c_int, i32, i32, _pd, _pd, _pd, _pd, _pd, i32, _pd]
    L.gelato_leaf_eci2geodetic.argtypes = [ctypes.c_int, i32, _pd, _pd, _pd]
    L.gelato_leaf_gravity.argtypes = [ctypes.c_int, i32, _pd, _pd]
    L.gelato_leaf_iip.argtypes = [ctypes.c_int, i32, _pd, _pd, i32, _pd]
    L.gelato_leaf_atmosphere.argtypes = [ctypes.c_int, i32, _pd, _pd]
    L.gelato_leaf_output_table.argtypes = [ctypes.c_int, i32] + [_pd] * 9 + [i32, _pd, i32, _c_d, _c_d, _pd]
    L.gelato_leaf_coordinate.argtypes = [ctypes.c_int, i32, i32, _pd, i32, _pd, i32, _pd, _pd]
    L.gelato_init_rocket_simulation.argtypes = [ctypes.c_int, i32, _pd, _pd, ctypes.POINTER(ctypes.c_int32), i32, _pd, i32,
                                                _pd, i32, _pd, i32, ctypes.POINTER(ctypes.c_int64), _c_d, _pd, i32, _c_d, _pd, _pd]
    _lib = L
    return L


EXPORTS = (
    "gelato_last_error gelato_device_count gelato_plan_create gelato_plan_set_scenarios gelato_plan_destroy "
    "gelato_plan_n_vars gelato_plan_n_rows gelato_plan_n_vals gelato_plan_launch_count gelato_eval_residuals "
    "gelato_eval_jacobian gelato_eval_residuals_ids gelato_eval_jacobian_ids gelato_eval_residuals_dev gelato_eval_jacobian_dev gelato_time_kernel "
    "gelato_selftest_unfused gelato_fp64_peak gelato_fill_template gelato_host_alloc gelato_host_free "
    "gelato_eval_pair_update gelato_eval_pair_dev gelato_plan_n_blocks gelato_plan_n_xdep gelato_set_update_zero_copy gelato_set_update_slices gelato_probe_update gelato_jacobian_template gelato_eval_jacobian_update gelato_set_host_threads "
    "gelato_eval_pair_packed_dev gelato_plan_n_pack gelato_plan_packed_map gelato_eval_pair_packed gelato_eval_jacobian_packed "
    "gelato_eval_pair_packed_ids gelato_launch_kernel_dev "
    "gelato_pack_xdep_dev gelato_leaf_dynamics_velocity gelato_leaf_dynamics_velocity_noair "
    "gelato_leaf_dynamics_quaternion gelato_leaf_aero gelato_leaf_eci2geodetic gelato_leaf_gravity gelato_leaf_iip "
    "gelato_leaf_atmosphere gelato_leaf_output_table gelato_init_rocket_simulation gelato_leaf_coordinate "
    "gelato_eval_pair_packed_range_dev gelato_plan_set_fd gelato_plan_get_fd "
    "gelato_plan_set_mesh_grid gelato_eval_mesh_error gelato_eval_mesh_error_dev "
    "gelato_eval_mesh_error_intervals gelato_eval_mesh_error_intervals_dev "
    "gelato_eval_path_check gelato_eval_path_check_dev "
    "gelato_plan_set_path_rows gelato_plan_path_rows gelato_eval_path_rows gelato_eval_path_rows_dev"
).split()


def fd_args(mode, step=None):
    """("forward" | "central", step or None) -> (C mode code, step): what gelato_plan_set_fd accepts, else ValueError.
    The step of forward mode is the plan's dx and is ignored."""
    if mode not in FD_MODES:
        raise ValueError("derivative mode must be one of %s, not %r" % (sorted(FD_MODES), mode))
    if mode == "forward":
        return FD_MODES[mode], 0.0
    step = DEFAULT_FD_STEP if step is None else step
    if isinstance(step, bool) or not isinstance(step, (int, float)) or not 0.0 < float(step) <= 1e-3:
        raise ValueError("the central-difference step must be a number in (0, 1e-3], not %r" % (step,))
    return FD_MODES[mode], float(step)


def _check(L, rc, what):
    if rc != 0:
        raise GelatoError("%s failed (%d): %s" % (what, rc, L.gelato_last_error().decode()))


class Engine:
    """One plan handle on one GPU.  Not thread-safe (one CUDA stream per handle)."""

    def __init__(self, plan, device=0, scenario_plans=None):
        self.L = L = load_library()
        self.plan = plan
        self.device = device
        desc, self._keep = make_desc(plan)
        h = ctypes.c_void_p()
        _check(L, L.gelato_plan_create(ctypes.byref(desc), device, ctypes.byref(h)), "gelato_plan_create")
        self.h = h
        self.n_scen_cfg = 1
        self.calls = 0  # evaluation calls made through this handle (a call launches one to three kernels)
        if scenario_plans is not None:
            sc, keep = make_scenario_desc(scenario_plans)
            _check(L, L.gelato_plan_set_scenarios(self.h, ctypes.byref(sc)), "gelato_plan_set_scenarios")
            self.n_scen_cfg = len(scenario_plans)
        self.n_jac_blocks = L.gelato_plan_n_blocks(h, 1)
        self.n_res_blocks = L.gelato_plan_n_blocks(h, 0)
        self.n_jac_heavy = L.gelato_plan_n_blocks(h, 2)
        self.n_jac_light = L.gelato_plan_n_blocks(h, 3)
        self.n_jac_blocks_pair = L.gelato_plan_n_blocks(h, 4)
        self.n_vacuum_nodes = L.gelato_plan_n_blocks(h, 5)
        self.n_vars = L.gelato_plan_n_vars(h)
        self.n_rows = L.gelato_plan_n_rows(h)
        self.n_vals = L.gelato_plan_n_vals(h)
        assert self.n_vars == plan.n_vars and self.n_rows == plan.n_rows and self.n_vals == plan.n_vals
        self._prow = None  # the path-row layout (path_rows_layout), read once per grid
        self.n_mesh_int = 0  # intervals of the mesh grid once set (mesh_error_intervals)
        ok = ctypes.c_int(0)
        _check(L, L.gelato_selftest_unfused(device, ctypes.byref(ok)), "gelato_selftest_unfused")
        if not ok.value:
            raise GelatoError("libgelato_b200.so was built with fused multiply-add; rebuild with -fmad=false")

    def close(self):
        if getattr(self, "h", None):
            self.L.gelato_plan_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self):
        return int(self.L.gelato_plan_launch_count(self.h))

    def set_fd(self, mode, step=None):
        """Finite-difference mode of every Jacobian this handle returns: "forward" (default; the plan's dx, the
        reference's values bit for bit) or "central" with step `step` (None: DEFAULT_FD_STEP).  DESIGN.md H6."""
        code, step = fd_args(mode, step)
        _check(self.L, self.L.gelato_plan_set_fd(self.h, code, step), "gelato_plan_set_fd")

    @property
    def fd(self):
        """(mode, step): the current finite-difference mode and its step (forward: the plan's dx)."""
        m, h = ctypes.c_int32(0), ctypes.c_double(0.0)
        _check(self.L, self.L.gelato_plan_get_fd(self.h, ctypes.byref(m), ctypes.byref(h)), "gelato_plan_get_fd")
        return {v: k for k, v in FD_MODES.items()}[m.value], h.value

    # ---- mesh error estimate (DESIGN.md section 11) ----
    def set_mesh_grid(self, tables):
        """The test grid of the mesh error estimate: {"m", "off", "pool"} as gelato_b200.mesh.grid_tables builds it."""
        desc, _keep = make_mesh_grid_desc(tables)
        _check(self.L, self.L.gelato_plan_set_mesh_grid(self.h, ctypes.byref(desc)), "gelato_plan_set_mesh_grid")
        self.n_mesh_int = grid_intervals(tables)

    def mesh_error(self, x, n_scen=1, out=None):
        """err[S][11] (n_scen > 1: [n_scen][S][11]) of the decision vectors x[n_scen][n_vars]: per section and state
        component (mass | position 3 | velocity 3 | quaternion 4) the collocation error estimate between the nodes."""
        x = self._x(x, n_scen)
        self.calls += 1
        n = n_scen * self.plan.S * 11
        err = _out(out, n, "out") if out is not None else np.empty(n)
        _check(self.L, self.L.gelato_eval_mesh_error(self.h, _ptr(x, _pd), _ptr(err, _pd), n_scen), "gelato_eval_mesh_error")
        return err.reshape(self.plan.S, 11) if n_scen == 1 else err.reshape(n_scen, self.plan.S, 11)

    def mesh_error_dev(self, x_ptr, err_ptr, n_scen=1, stream=None):
        _check(self.L, self.L.gelato_eval_mesh_error_dev(self.h, x_ptr, err_ptr, n_scen, stream), "gelato_eval_mesh_error_dev")

    def mesh_error_intervals(self, x, n_scen=1, out=None):
        """err_int[n_int][11] (n_scen > 1: [n_scen][n_int][11]): the estimate of every LGR interval of the mesh grid, the
        intervals of section 0 first (one per section on a grid without interval tables)."""
        x = self._x(x, n_scen)
        self.calls += 1
        n = n_scen * self.n_mesh_int * 11
        err = _out(out, n, "out") if out is not None else np.empty(n)
        _check(self.L, self.L.gelato_eval_mesh_error_intervals(self.h, _ptr(x, _pd), _ptr(err, _pd), n_scen),
               "gelato_eval_mesh_error_intervals")
        return err.reshape(self.n_mesh_int, 11) if n_scen == 1 else err.reshape(n_scen, self.n_mesh_int, 11)

    def mesh_error_intervals_dev(self, x_ptr, err_ptr, n_scen=1, stream=None):
        _check(self.L, self.L.gelato_eval_mesh_error_intervals_dev(self.h, x_ptr, err_ptr, n_scen, stream),
               "gelato_eval_mesh_error_intervals_dev")

    def path_check(self, x, n_scen=1, out=None):
        """(res, at) of the decision vectors x[n_scen][n_vars], [n_aero] each (n_scen > 1: [n_scen][n_aero]), in the
        plan's aero-job order: per aero job the smallest residual 1 - f / limit over the test points of its section on
        the mesh grid, and the index of that test point (an "initial" job: +inf and -1).  out: (res float64, at int32)
        buffers of n_scen * n_aero entries (page-locked ones are DMA'd directly)."""
        x = self._x(x, n_scen)
        self.calls += 1
        n = n_scen * self.plan.n_aero
        if out is not None:
            res, at = _out(out[0], n, "out[0]"), out[1]
            if not isinstance(at, np.ndarray) or at.dtype != np.int32 or not at.flags.c_contiguous or at.size != n:
                raise ValueError("out[1] must be a C-contiguous int32 numpy array of %d entries" % n)
        else:
            res, at = np.empty(n), np.empty(n, dtype=np.int32)
        _check(self.L, self.L.gelato_eval_path_check(self.h, _ptr(x, _pd), _ptr(res, _pd), _ptr(at, _pi32), n_scen),
               "gelato_eval_path_check")
        return (res, at) if n_scen == 1 else (res.reshape(n_scen, -1), at.reshape(n_scen, -1))

    def path_check_dev(self, x_ptr, res_ptr, at_ptr, n_scen=1, stream=None):
        _check(self.L, self.L.gelato_eval_path_check_dev(self.h, x_ptr, res_ptr, at_ptr, n_scen, stream),
               "gelato_eval_path_check_dev")

    # ---- path rows (DESIGN.md section 11) ----
    def set_path_rows(self, tables):
        """The grid of the path rows ({"m", "off", "pool"} as gelato_b200.mesh.grid_tables builds it), separate from the
        mesh grid: the aero constraints become NLP rows at its test points (include/gelato_b200.h)."""
        desc, _keep = make_mesh_grid_desc(tables)
        _check(self.L, self.L.gelato_plan_set_path_rows(self.h, ctypes.byref(desc)), "gelato_plan_set_path_rows")
        self._prow = None

    def path_rows_layout(self):
        """{"n_rows", "n_vals", "job" int32[n_rows], "l" int32[n_rows], "off" int64[n_rows][4]}: the rows (aero job,
        test point) and where each row's position | velocity | quaternion (-1: none) | t entries start in the values of
        one scenario (gelato_plan_path_rows; read once per grid)."""
        if self._prow is None:
            L, n, v = self.L, ctypes.c_int32(0), ctypes.c_int64(0)
            _check(L, L.gelato_plan_path_rows(self.h, ctypes.byref(n), ctypes.byref(v), None, None, None),
                   "gelato_plan_path_rows")
            job, l = np.empty(n.value, dtype=np.int32), np.empty(n.value, dtype=np.int32)
            off = np.empty((n.value, 4), dtype=np.int64)
            _check(L, L.gelato_plan_path_rows(self.h, ctypes.byref(n), ctypes.byref(v), _ptr(job, _pi32), _ptr(l, _pi32),
                                              _ptr(off, _pi64)), "gelato_plan_path_rows")
            self._prow = {"n_rows": n.value, "n_vals": v.value, "job": job, "l": l, "off": off}
        return self._prow

    def eval_path_rows(self, x, n_scen=1, jacobian=True, out=None):
        """(g [n_rows], vals [n_vals] or None) of the decision vectors x[n_scen][n_vars] (n_scen > 1: [n_scen][...]):
        the path rows' values and, with `jacobian`, their Jacobian values in the current finite-difference mode.
        out: (g, vals) float64 buffers to write into instead, page-locked ones DMA'd directly; a None entry is not
        computed (`jacobian` is then not read)."""
        x = self._x(x, n_scen)
        self.calls += 1
        lay = self.path_rows_layout()
        nr, nv = lay["n_rows"], lay["n_vals"]
        if out is not None:  # a None entry: that output is not computed
            g = None if out[0] is None else _out(out[0], n_scen * nr, "out[0]")
            v = None if out[1] is None else _out(out[1], n_scen * nv, "out[1]")
        else:
            g, v = np.empty(n_scen * nr), (np.empty(n_scen * nv) if jacobian else None)
        _check(self.L, self.L.gelato_eval_path_rows(self.h, _ptr(x, _pd), _ptr(g, _pd), _ptr(v, _pd), n_scen),
               "gelato_eval_path_rows")
        if n_scen > 1:
            g, v = (None if a is None else a.reshape(n_scen, -1) for a in (g, v))
        return g, v

    def eval_path_rows_dev(self, x_ptr, g_ptr, vals_ptr, n_scen=1, stream=None):
        _check(self.L, self.L.gelato_eval_path_rows_dev(self.h, x_ptr, g_ptr, vals_ptr, n_scen, stream),
               "gelato_eval_path_rows_dev")

    # ---- host-buffer calls (what objfunc / sens use) --------------------
    def _x(self, x, n_scen):
        x = np.ascontiguousarray(x, dtype=np.float64)
        if x.size != n_scen * self.n_vars:
            raise ValueError("x has %d entries, expected %d x %d" % (x.size, n_scen, self.n_vars))
        return x

    def eval_residuals(self, x, n_scen=1, out=None, scen_ids=None):
        """scen_ids: batch slot k uses the parameter blocks of configured scenario scen_ids[k]."""
        x = self._x(x, n_scen)
        self.calls += 1
        g = _out(out, n_scen * self.n_rows, "out") if out is not None else np.empty(n_scen * self.n_rows)
        if scen_ids is None:
            _check(self.L, self.L.gelato_eval_residuals(self.h, _ptr(x, _pd), _ptr(g, _pd), n_scen), "gelato_eval_residuals")
        else:
            ids = np.ascontiguousarray(scen_ids, dtype=np.int32)
            assert ids.size == n_scen
            _check(self.L, self.L.gelato_eval_residuals_ids(self.h, _ptr(x, _pd), _ptr(g, _pd), n_scen, _ptr(ids, _pi32)),
                   "gelato_eval_residuals_ids")
        return g if n_scen == 1 else g.reshape(n_scen, self.n_rows)

    def eval_jacobian(self, x, n_scen=1, out=None, scen_ids=None):
        x = self._x(x, n_scen)
        self.calls += 1
        v = _out(out, n_scen * self.n_vals, "out") if out is not None else np.empty(n_scen * self.n_vals)
        if scen_ids is None:
            _check(self.L, self.L.gelato_eval_jacobian(self.h, _ptr(x, _pd), _ptr(v, _pd), n_scen), "gelato_eval_jacobian")
        else:
            ids = np.ascontiguousarray(scen_ids, dtype=np.int32)
            assert ids.size == n_scen
            _check(self.L, self.L.gelato_eval_jacobian_ids(self.h, _ptr(x, _pd), _ptr(v, _pd), n_scen, _ptr(ids, _pi32)),
                   "gelato_eval_jacobian_ids")
        return v if n_scen == 1 else v.reshape(n_scen, self.n_vals)

    # ---- update mode: one persistent host buffer per batch, only x-dependent slots cross PCIe ----
    def jacobian_template(self, out, n_scen=1):
        """Fill out[n_scen * n_vals] with the constant Jacobian slots (once per buffer)."""
        _out(out, n_scen * self.n_vals, "out")
        _check(self.L, self.L.gelato_jacobian_template(self.h, _ptr(out, _pd), n_scen), "gelato_jacobian_template")
        return out

    def eval_jacobian_update(self, x, out, n_scen=1):
        """Rewrite the x-dependent slots of `out` (a buffer initialised by jacobian_template or
        holding an earlier result); afterwards `out` equals what eval_jacobian returns."""
        x = self._x(x, n_scen)
        self.calls += 1
        _out(out, n_scen * self.n_vals, "out")
        _check(self.L, self.L.gelato_eval_jacobian_update(self.h, _ptr(x, _pd), _ptr(out, _pd), n_scen),
               "gelato_eval_jacobian_update")
        return out if n_scen == 1 else out.reshape(n_scen, self.n_vals)

    def eval_pair_update(self, x, g_out, vals_out, n_scen=1):
        """objfunc + sens of the same decision vectors in one call (x uploaded once, the two kernels
        concurrent); g_out is filled whole, vals_out updated as by eval_jacobian_update."""
        x = self._x(x, n_scen)
        self.calls += 1
        _out(g_out, n_scen * self.n_rows, "g_out")
        _out(vals_out, n_scen * self.n_vals, "vals_out")
        _check(self.L, self.L.gelato_eval_pair_update(self.h, _ptr(x, _pd), _ptr(g_out, _pd), _ptr(vals_out, _pd), n_scen),
               "gelato_eval_pair_update")
        return g_out.reshape(n_scen, self.n_rows), vals_out.reshape(n_scen, self.n_vals)

    # ---- packed mode: the independent x-dependent values only, contiguous; the consumer gathers ----
    @property
    def n_pack(self):
        return int(self.L.gelato_plan_n_pack(self.h))

    def packed_map(self):
        """(full_slot, src, sgn): vals[full_slot] = sgn * packed[src] for the x-dependent COO slots."""
        n = int(self.L.gelato_plan_n_xdep(self.h))
        full, src, sgn = np.empty(n, dtype=np.int64), np.empty(n, dtype=np.int64), np.empty(n)
        _check(self.L, self.L.gelato_plan_packed_map(self.h, _ptr(full, _pi64), _ptr(src, _pi64), _ptr(sgn, _pd)),
               "gelato_plan_packed_map")
        return full, src, sgn

    def eval_pair_packed(self, x, n_scen=1, g_out=None, packed_out=None, scen_ids=None):
        """objfunc + sens of the same decision vectors: (g[n_scen][n_rows], packed[n_scen][n_pack])."""
        x = self._x(x, n_scen)
        self.calls += 1
        g = _out(g_out, n_scen * self.n_rows, "g_out") if g_out is not None else np.empty(n_scen * self.n_rows)
        pk = _out(packed_out, n_scen * self.n_pack, "packed_out") if packed_out is not None else np.empty(n_scen * self.n_pack)
        if scen_ids is None:
            _check(self.L, self.L.gelato_eval_pair_packed(self.h, _ptr(x, _pd), _ptr(g, _pd), _ptr(pk, _pd), n_scen),
                   "gelato_eval_pair_packed")
        else:
            ids = np.ascontiguousarray(scen_ids, dtype=np.int32)
            assert ids.size == n_scen
            _check(self.L, self.L.gelato_eval_pair_packed_ids(self.h, _ptr(x, _pd), _ptr(g, _pd), _ptr(pk, _pd), n_scen,
                                                              _ptr(ids, _pi32)), "gelato_eval_pair_packed_ids")
        if n_scen == 1:
            return g, pk
        return g.reshape(n_scen, self.n_rows), pk.reshape(n_scen, self.n_pack)

    def eval_jacobian_packed(self, x, n_scen=1, packed_out=None):
        x = self._x(x, n_scen)
        self.calls += 1
        pk = _out(packed_out, n_scen * self.n_pack, "packed_out") if packed_out is not None else np.empty(n_scen * self.n_pack)
        _check(self.L, self.L.gelato_eval_jacobian_packed(self.h, _ptr(x, _pd), _ptr(pk, _pd), n_scen),
               "gelato_eval_jacobian_packed")
        return pk if n_scen == 1 else pk.reshape(n_scen, self.n_pack)

    def eval_pair_packed_dev(self, x_ptr, g_ptr, packed_ptr, n_scen=1, stream=None):
        _check(self.L, self.L.gelato_eval_pair_packed_dev(self.h, x_ptr, g_ptr, packed_ptr, n_scen, stream),
               "gelato_eval_pair_packed_dev")

    def eval_pair_packed_range_dev(self, x_ptr, g_ptr, packed_ptr, blocks, vacuum, n_scen=1, stream=None):
        """The pair evaluation restricted to blocks [blocks[0], blocks[1]) and vacuum nodes [vacuum[0], vacuum[1])
        (one problem sharded over GPUs); n_jac_blocks_pair / n_vacuum_nodes give the totals."""
        _check(self.L, self.L.gelato_eval_pair_packed_range_dev(self.h, x_ptr, g_ptr, packed_ptr, n_scen, blocks[0],
                                                                blocks[1] - blocks[0], vacuum[0], vacuum[1] - vacuum[0], stream),
               "gelato_eval_pair_packed_range_dev")

    def eval_pair_dev(self, x_ptr, g_ptr, vals_ptr, n_scen=1, stream=None):
        _check(self.L, self.L.gelato_eval_pair_dev(self.h, x_ptr, g_ptr, vals_ptr, n_scen, stream), "gelato_eval_pair_dev")

    def set_update_zero_copy(self, on=True):
        _check(self.L, self.L.gelato_set_update_zero_copy(self.h, 1 if on else 0), "gelato_set_update_zero_copy")

    def probe_update(self, vals, n_scen, reps=10):
        """Device times (ms) of the transfer pieces of update mode (measurement only; tools/e2e_probe.py)."""
        out = (ctypes.c_float * 6)()
        _check(self.L, self.L.gelato_probe_update(self.h, vals.ctypes.data_as(_pd), n_scen, reps, out), "gelato_probe_update")
        return dict(zip(("copies_2d", "zero_copy", "both", "pack_and_copy", "contiguous_all", "residual_copy"), list(out)))

    def set_update_slices(self, n):
        _check(self.L, self.L.gelato_set_update_slices(self.h, int(n)), "gelato_set_update_slices")

    def set_host_threads(self, n):
        _check(self.L, self.L.gelato_set_host_threads(self.h, int(n)), "gelato_set_host_threads")

    # ---- device-resident calls (raw device pointers, e.g. torch .data_ptr()) ----
    def eval_residuals_dev(self, x_ptr, g_ptr, n_scen=1, stream=None):
        _check(self.L, self.L.gelato_eval_residuals_dev(self.h, x_ptr, g_ptr, n_scen, stream), "gelato_eval_residuals_dev")

    def fill_template(self, vals_ptr, n_scen=1, stream=None):
        """Write the constant Jacobian entries into a device buffer (once per buffer)."""
        _check(self.L, self.L.gelato_fill_template(self.h, vals_ptr, n_scen, stream), "gelato_fill_template")

    def eval_jacobian_dev(self, x_ptr, vals_ptr, n_scen=1, stream=None):
        _check(self.L, self.L.gelato_eval_jacobian_dev(self.h, x_ptr, vals_ptr, n_scen, stream), "gelato_eval_jacobian_dev")

    def pack_xdep_dev(self, vals_ptr, packed_ptr, n_scen=1, stream=None):
        _check(self.L, self.L.gelato_pack_xdep_dev(self.h, vals_ptr, packed_ptr, n_scen, stream), "gelato_pack_xdep_dev")

    def launch_kernel_dev(self, which, x_ptr, out_ptr, n_scen=1, packed=False, stream=None, g_ptr=None):
        """Enqueue ONE kernel (0 residual, 2 heavy Jacobian, 3 light Jacobian, 4 non-dynamics residual blocks) on
        `stream` (measurement helper); g_ptr: a Jacobian kernel also writes the pair evaluation's defect rows."""
        _check(self.L, self.L.gelato_launch_kernel_dev(self.h, which, x_ptr, out_ptr, g_ptr, n_scen, 1 if packed else 0, stream),
               "gelato_launch_kernel_dev")

    def time_kernel(self, which, x_ptr, out_ptr, n_scen=1, reps=10):
        """Average duration [ms] of `reps` back-to-back launches (0 residual kernel, 1 Jacobian evaluation,
        2 heavy Jacobian kernel alone, 3 light Jacobian kernel alone), CUDA events on the launch stream."""
        ms = ctypes.c_float(0)
        _check(self.L, self.L.gelato_time_kernel(self.h, which, x_ptr, out_ptr, n_scen, reps, ctypes.byref(ms)),
               "gelato_time_kernel")
        return float(ms.value)


class PinnedArray:
    """A page-locked float64 host array (gelato_host_alloc) the engine DMAs directly."""

    def __init__(self, n):
        self.L = load_library()
        self.ptr = ctypes.c_void_p()
        _check(self.L, self.L.gelato_host_alloc(max(8, int(n) * 8), ctypes.byref(self.ptr)), "gelato_host_alloc")
        self.array = np.frombuffer((ctypes.c_double * int(n)).from_address(self.ptr.value), dtype=np.float64)

    def free(self):
        if self.ptr:
            self.array = None
            self.L.gelato_host_free(self.ptr)
            self.ptr = None


def fp64_peak(device=0):
    """(TFLOP/s with DFMA, TFLOP/s with separate DMUL+DADD) measured on the device."""
    L = load_library()
    a, b = ctypes.c_double(0), ctypes.c_double(0)
    _check(L, L.gelato_fp64_peak(device, ctypes.byref(a), ctypes.byref(b)), "gelato_fp64_peak")
    return a.value, b.value
