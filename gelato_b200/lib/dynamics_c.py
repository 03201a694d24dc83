"""dynamics_c (/root/reference/src/pybind_dynamics.cpp:108-114) on the GPU: same names, same arguments."""
import numpy as np

from ._leaf import arr, call, ptr


def dynamics_velocity(mass_e, pos_eci_e, vel_eci_e, quat_eci2body, t, param, wind_table, CA_table, units):
    """pybind_dynamics.cpp:30-71 -- acceleration / unit_vel for n nodes, (n, 3)."""
    m = arr(mass_e).ravel()
    n = m.size
    pos, vel, quat = arr(pos_eci_e, (n, 3)), arr(vel_eci_e, (n, 3)), arr(quat_eci2body, (n, 4))
    tt, prm, un = arr(t).ravel(), arr(param).ravel(), arr(units).ravel()
    wind, ca = arr(wind_table, (-1, 3)), arr(CA_table, (-1, 2))  # the row counts go to the C ABI
    out = np.empty((n, 3))
    call("gelato_leaf_dynamics_velocity", n, ptr(m), ptr(pos), ptr(vel), ptr(quat), ptr(tt), ptr(prm), ptr(wind),
         wind.shape[0], ptr(ca), ca.shape[0], ptr(un), ptr(out))
    return out


def dynamics_velocity_NoAir(mass_e, pos_eci_e, quat_eci2body, param, units):
    """pybind_dynamics.cpp:73-92."""
    m = arr(mass_e).ravel()
    n = m.size
    pos, quat = arr(pos_eci_e, (n, 3)), arr(quat_eci2body, (n, 4))
    prm, un = arr(param).ravel(), arr(units).ravel()
    out = np.empty((n, 3))
    call("gelato_leaf_dynamics_velocity_noair", n, ptr(m), ptr(pos), ptr(quat), ptr(prm), ptr(un), ptr(out))
    return out


def dynamics_quaternion(quat_eci2body, u_e, unit_u):
    """pybind_dynamics.cpp:94-106."""
    quat = arr(quat_eci2body).reshape(-1, 4)
    n = quat.shape[0]
    u = arr(u_e, (n, 2))
    out = np.empty((n, 4))
    call("gelato_leaf_dynamics_quaternion", n, ptr(quat), ptr(u), float(unit_u), ptr(out))
    return out
