"""utils_c (/root/reference/src/pybind_utils.cpp:28-48) on the GPU: the aero-constraint leaves, wind_ned and the
two-plane angle of attack.  Dimensional inputs, t in seconds, as in wrapper_utils.hpp:82-206.  (haversine is not
offered: no call site in the reference's live code.)"""
import numpy as np

from ._leaf import arr, call, ptr


def _aero(kind, pos, vel, quat, t, wind):
    pos = arr(pos).reshape(-1, 3)
    n = pos.shape[0]
    vel = arr(vel, (n, 3))
    q = arr(quat, (n, 4)) if quat is not None else None
    tt = arr(t).ravel()
    w = arr(wind, (-1, 3))
    out = np.empty(n)
    call("gelato_leaf_aero", kind, n, ptr(pos), ptr(vel), ptr(q), ptr(tt), ptr(w), w.shape[0], ptr(out))
    return out


def angle_of_attack_all_array_rad(pos_eci, vel_eci, quat, t, wind):
    return _aero(0, pos_eci, vel_eci, quat, t, wind)


def dynamic_pressure_array_pa(pos_eci, vel_eci, t, wind):
    return _aero(1, pos_eci, vel_eci, None, t, wind)


def q_alpha_array_pa_rad(pos_eci, vel_eci, quat, t, wind):
    return _aero(2, pos_eci, vel_eci, quat, t, wind)


def angle_of_attack_all_rad(pos_eci, vel_eci, quat, t, wind):
    return float(_aero(0, pos_eci, vel_eci, quat, [t], wind)[0])


def dynamic_pressure_pa(pos_eci, vel_eci, t, wind):
    return float(_aero(1, pos_eci, vel_eci, None, [t], wind)[0])


def q_alpha_pa_rad(pos_eci, vel_eci, quat, t, wind):
    return float(_aero(2, pos_eci, vel_eci, quat, [t], wind)[0])


def angle_of_attack_ab_array_rad(pos_eci, vel_eci, quat, t, wind):
    """wrapper_utils.hpp:150-161 -> (n, 2): pitch-plane and yaw-plane angles of the air-relative velocity in body axes."""
    pos = arr(pos_eci).reshape(-1, 3)
    n = pos.shape[0]
    w = arr(wind, (-1, 3))
    out = np.empty((n, 2))
    call("gelato_leaf_aero", 3, n, ptr(pos), ptr(arr(vel_eci, (n, 3))), ptr(arr(quat, (n, 4))), ptr(arr(t).ravel()), ptr(w),
         w.shape[0], ptr(out))
    return out


def angle_of_attack_ab_rad(pos_eci, vel_eci, quat, t, wind):
    """wrapper_utils.hpp:125-148"""
    return angle_of_attack_ab_array_rad(pos_eci, vel_eci, quat, [t], wind)[0]


def wind_ned(altitude_m, wind):
    """wrapper_utils.hpp:82-87 -> (north, east, 0) wind at an altitude (or (n, 3) for n altitudes)."""
    alt = arr(altitude_m).ravel()
    w = arr(wind, (-1, 3))
    out = np.empty((alt.size, 3))
    call("gelato_leaf_aero", 4, alt.size, ptr(None), ptr(None), ptr(None), ptr(alt), ptr(w), w.shape[0], ptr(out))
    return out[0] if np.ndim(altitude_m) == 0 else out


def haversine(lon1, lat1, lon2, lat2, r, fn=None):
    """Great-circle distance on a sphere of radius r, angles in degrees (pybind_utils.cpp:29, wrapper_utils.hpp:37-49)."""
    from .coordinate_c import _haversine

    return _haversine(lon1, lat1, lon2, lat2, r, fn=fn)
