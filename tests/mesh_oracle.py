"""The mesh error estimate on the CPU oracle (TEST INFRASTRUCTURE ONLY; DESIGN.md section 11).

A numpy restatement of gelato_b200/csrc/mesh_error.h on top of `oracle.nlp.OracleNLP` built with dot="seqfma": the
interpolations and the integral are `o_seqfma_matmul` products (fused multiply-add chains, ascending index, from 0.0),
the right-hand sides are the oracle's own leaves (`dynamics_velocity`, `dynamics_velocity_NoAir`,
`dynamics_quaternion`) with the operations of its collocation defects.  With the gmath flavour it agrees with the
kernels bit for bit.
"""
import numpy as np


def section_rhs(O, i, Xl, Ul, tau_t, to, tf):
    """rh[M][11]: the right-hand-side term of each state component of section i at the test points, as the oracle's
    eq_dyn_* form it at the nodes (engine-off mass and held attitude: 0)."""
    u, prm = O.u, O.p["params"][i]
    ut, dt = u["t"], tf - to
    M = Xl.shape[0]
    rh = np.zeros((M, 11))
    if prm["engineOn"]:
        rh[:, 0] = -prm["massflow"] / u["mass"] * dt * ut / 2.0
    rh[:, 1:4] = Xl[:, 4:7] * u["velocity"] * dt * ut / 2.0 / u["position"]
    t_l = tau_t * dt / 2 + (tf + to) / 2
    f = O._rhs_vel(i, Xl[:, 0], Xl[:, 1:4], Xl[:, 4:7], Xl[:, 7:11], t_l, O._units3())
    rh[:, 4:7] = f * dt * ut / 2.0
    if not O._holds(i):
        rh[:, 7:11] = O.dyn.dynamics_quaternion(Xl[:, 7:11], Ul, u["u"]) * dt * ut / 2.0
    return rh


def section_states(O, x, i):
    """(X[n+1][11], U[n][2]) of section i of the decision dictionary x."""
    ua, ub, xa, xb, n = O.ps.get_index(i)
    X = np.column_stack((x["mass"][xa:xb], x["position"].reshape(-1, 3)[xa:xb], x["velocity"].reshape(-1, 3)[xa:xb],
                         x["quaternion"].reshape(-1, 4)[xa:xb]))
    return X, x["u"].reshape(-1, 2)[ua:ub]


def unpack(tables, i, n):
    """(tau_t, P, Q, I) of section i from the pool of gelato_b200.mesh.grid_tables."""
    M, o = int(tables["m"][i]), int(tables["off"][i])
    pool = tables["pool"]
    tau_t = pool[o:o + M]
    o += M
    P = pool[o:o + M * (n + 1)].reshape(M, n + 1)
    o += M * (n + 1)
    Q = pool[o:o + M * n].reshape(M, n)
    o += M * n
    return tau_t, P, Q, pool[o:o + M * M].reshape(M, M)


def mesh_error(O, x, tables):
    """err[S][11] of the decision dictionary x on the test grid `tables`."""
    err = np.empty((O.S, 11))
    t = x["t"]
    for i in range(O.S):
        n = O.ps.nodes(i)
        tau_t, P, Q, I = unpack(tables, i, n)
        X, U = section_states(O, x, i)
        Xl, Ul = O._dot(P, X), O._dot(Q, U)
        rh = section_rhs(O, i, Xl, Ul, tau_t, t[i], t[i + 1])
        Xh = X[0] + O._dot(I, rh)
        err[i] = np.max(np.abs(Xh - Xl), axis=0) / (1.0 + np.max(np.abs(Xl), axis=0))
    return err
